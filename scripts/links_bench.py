"""Cost of row links (`BatchedPredPreyGrass.track_links()`, include/ppg.h ppg_track_links) on the flagship workloads
(bench.py's configurations: BASE 4096, ADD 16384, ECO 16384, STAG 8192 envs at caps 160+640).

For each config two handles of the same config are created in one process, one with links switched on before its first
reset and one without, both pre-rolled (random actions, auto-reset) to the steady-state population; then ms per step of the
random rollout of each, alternated over several windows (CUDA events around `--steps` steps), and the bytes of the link
state.  Prints one JSON document (also written to --out) with the GPU name and power limit (nvidia-smi query only).

    python scripts/links_bench.py --out profiles/links_b200.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from scripts.world_state_bench import CONFIGS, make_cfg, timed  # noqa: E402


def measure(name, preroll, steps, windows):
    import torch

    from predpreygrass_b200.batched import BatchedPredPreyGrass

    variant, mode, B, cap = CONFIGS[name]
    cfg = make_cfg(variant, mode, cap)
    off, on = BatchedPredPreyGrass(cfg, B), BatchedPredPreyGrass(cfg, B)
    on.track_links()
    for g in (off, on):
        g.reset()
        for _ in range(preroll):
            g.step(*g.random_actions(7))
    torch.cuda.synchronize()

    def rollout(g):
        return lambda: g.step(*g.random_actions(7))

    ms_off, ms_on = [], []
    for _ in range(windows):  # alternated: both arms see the same kind of population and the same machine state
        ms_off.append(timed(rollout(off), steps) / steps)
        ms_on.append(timed(rollout(on), steps) / steps)
    err = int(on.links_error().item())
    linked = sum(int((p[:n] >= 0).sum()) for p, n in zip(on.prev_row(), on.out.counts()))
    rows = sum(on.out.counts())
    table_words = sum(B << max(1, (2 * c - 1).bit_length()) for c in cap)
    state_bytes = sum(on.row_capacity) * 4 + table_words * 4 + 2 * B * 16
    for g in (off, on):
        g.close()
    best_off, best_on = min(ms_off), min(ms_on)
    return {"envs": B, "cap_live": list(cap), "preroll_steps": preroll, "steps_per_window": steps,
            "ms_per_step_off": best_off, "ms_per_step_on": best_on, "ms_per_step_off_windows": ms_off, "ms_per_step_on_windows": ms_on,
            "links_cost_us_per_step": (best_on - best_off) * 1e3, "links_share_of_step": (best_on - best_off) / best_off,
            "rows_last_output": rows, "linked_rows_last_output": linked, "link_error_bits": err, "link_state_bytes": state_bytes}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", nargs="+", default=list(CONFIGS), choices=list(CONFIGS))
    ap.add_argument("--preroll", type=int, default=300)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--windows", type=int, default=4)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("links_bench.py measures on a CUDA device; there is none")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1], "configs": {}}
    for name in args.configs:
        r = measure(name, args.preroll, args.steps, args.windows)
        res["configs"][name] = r
        print(name, json.dumps(r), flush=True)
    doc = json.dumps(res, indent=1)
    print(doc)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(doc + "\n")


if __name__ == "__main__":
    main()
