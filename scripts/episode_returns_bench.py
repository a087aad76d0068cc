"""Cost of episode-return tracking (`BatchedPredPreyGrass.track_returns()`, include/ppg.h ppg_track_returns) on the
flagship workloads (bench.py's configurations).

For each config two handles of the same config are created in one process, one with tracking switched on before its first
reset and one without, both pre-rolled (random actions, auto-reset) to the steady-state population; then
  * ms per step of the random rollout of each, alternated over several windows (CUDA events around `--steps` steps),
  * us per episode_stats_device() call (CUDA events around `--calls` back-to-back calls after warm-up),
  * the bytes of the tracking state (row columns, per-agent tables, per-env state).
Prints one JSON document (also written to --out) with the GPU name and power limit (nvidia-smi query only).

    python scripts/episode_returns_bench.py --out profiles/episode_returns_b200.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from scripts.world_state_bench import CONFIGS, make_cfg, timed  # noqa: E402


def measure(name, preroll, steps, windows, calls):
    import torch

    from predpreygrass_b200.batched import BatchedPredPreyGrass

    variant, mode, B, cap = CONFIGS[name]
    cfg = make_cfg(variant, mode, cap)
    off, on = BatchedPredPreyGrass(cfg, B), BatchedPredPreyGrass(cfg, B)
    on.track_returns()
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
    for _ in range(20):
        on.episode_stats_device()
    ms_calls = [timed(on.episode_stats_device, calls) for _ in range(3)]
    metrics = on.episode_metrics()
    rows = sum(on.out.counts())
    state_bytes = (sum(on.row_capacity) * 12 + B * 12 * (cfg.n_possible[0] + cfg.n_possible[1]) + B * (16 + 1 + 16 * 8))
    for g in (off, on):
        g.close()
    best_off, best_on = min(ms_off), min(ms_on)
    return {"envs": B, "cap_live": list(cap), "preroll_steps": preroll, "steps_per_window": steps,
            "ms_per_step_off": best_off, "ms_per_step_on": best_on, "ms_per_step_off_windows": ms_off, "ms_per_step_on_windows": ms_on,
            "tracking_cost_us_per_step": (best_on - best_off) * 1e3, "tracking_share_of_step": (best_on - best_off) / best_off,
            "rows_last_output": rows, "us_per_episode_stats_call": min(ms_calls) / calls * 1e3,
            "tracking_state_bytes": state_bytes, "num_episodes": metrics["num_episodes"],
            "episode_return_mean": metrics["episode_return_mean"], "episode_len_mean": metrics["episode_len_mean"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", nargs="+", default=list(CONFIGS), choices=list(CONFIGS))
    ap.add_argument("--preroll", type=int, default=300)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--windows", type=int, default=4)
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("episode_returns_bench.py measures on a CUDA device; there is none")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1], "configs": {}}
    for name in args.configs:
        r = measure(name, args.preroll, args.steps, args.windows, args.calls)
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
