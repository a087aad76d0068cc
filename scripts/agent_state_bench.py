#!/usr/bin/env python
"""Cost of one agent_state() call (include/ppg.h ppg_agent_state) next to the step of the same handle.

For each of bench.py's configurations (BASE at 4096 envs; its `configs` runs ADD 16384, ECO 16384 and STAG 8192 envs at caps
160 + 640; one handle each): pre-roll the envs to their steady-state population with random actions, then in one process
  - time `--steps` steps of random actions with CUDA events (the step time, agent_state not called),
  - time `--repeats` agent_state() calls on the last output, each between its own pair of CUDA events,
  - and again `--steps` steps, so a drift of the card between the two step windows shows,
and report the median call time, its share of the step time, and the bytes the call moves, counted from the row and list
counts: per env the flags, row offsets and list lengths; per list entry of an env that continues the entry's row, id,
position, energy and the variant's extra columns plus the row id it is matched against; per row the sentinels of every
column, and the columns again for a present row; per grass patch its position and energy read and written.  The list
lengths are taken from env_count (live agents; ECO carcasses still in the list are not counted, so ECO's bytes are a slight
underestimate).  The card's name and power limit are read in the same run.
Usage: python scripts/agent_state_bench.py [--out FILE] [--preroll 300] [--steps 100] [--repeats 200]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# bytes per element of each per-species column: (read from the list, written per row)
COL_BYTES = {"present": (0, 1), "pos": (2, 8), "energy": (8, 8), "age": (2, 4), "trait": (8, 8), "facing": (1, 1), "acc": (8, 8)}


def card():
    import torch

    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["nvidia_smi"] = q
    except Exception as e:  # noqa: BLE001
        info["nvidia_smi"] = f"unavailable: {e}"
    return info


def bytes_moved(env, st):
    """(read, written) bytes of the last agent_state() call, from the output's counts (one host synchronisation)"""
    import torch

    from predpreygrass_b200.batched import agent_state_columns

    cols = agent_state_columns(env.cfg)
    o = env.out
    n = o.counts()
    cont = (o.env_flags & 3) == 0
    listed = (o.env_count.to(torch.int64) * cont[:, None]).sum(0).tolist()
    present = [int(st.present[s][: n[s]].sum()) for s in range(2)]
    B, ng = env.n_envs, env.cfg.n_grass
    rd = B * (1 + 2 * (8 + 4 + 4 + 2)) + int(cont.sum()) * ng * (2 + 8)
    wr = B * ng * (8 + 8)
    for s in range(2):
        per_entry = 4 + 2 + 4 + sum(COL_BYTES[c][0] for c in cols if cols[c][s])  # ag_prow, ag_id, row_agent, the columns
        per_row = sum(COL_BYTES[c][1] for c in cols if cols[c][s])
        rd += listed[s] * per_entry
        wr += (n[s] + present[s]) * per_row
    return rd, wr, n, present


def time_steps(env, steps):
    import torch

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        env.step(*env.random_actions(7))
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def measure(name, argv, preroll, steps, repeats):
    import torch

    import bench
    from predpreygrass_b200.batched import BatchedPredPreyGrass

    args = bench.parse(argv)
    cfg = bench.build_config(args, seed=12345)
    env = BatchedPredPreyGrass(cfg, args.envs)
    try:
        env.reset()
        for _ in range(preroll):
            env.step(*env.random_actions(7))
        torch.cuda.synchronize()
        ms_step_a = time_steps(env, steps)
        st = env.agent_state()  # warm-up: allocates the buffers, loads the kernel
        torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(repeats)]
        for a, b in ev:
            a.record()
            env.agent_state()
            b.record()
        torch.cuda.synchronize()
        us = sorted(1000.0 * a.elapsed_time(b) for a, b in ev)
        rd, wr, n, present = bytes_moved(env, st)
        ms_step_b = time_steps(env, steps)
        med = us[len(us) // 2]
        ms_step = 0.5 * (ms_step_a + ms_step_b)
        return {
            "config": name, "variant": args.variant, "reward_mode": args.reward_mode, "envs": args.envs, "cap_live": list(args.cap),
            "rows": list(n), "present_rows": present,
            "us_agent_state_median": med, "us_agent_state_min": us[0], "us_agent_state_max": us[-1], "repeats": repeats,
            "us_per_step": 1000.0 * ms_step, "us_per_step_before": 1000.0 * ms_step_a, "us_per_step_after": 1000.0 * ms_step_b,
            "share_of_step": med / (1000.0 * ms_step),
            "bytes_read": rd, "bytes_written": wr, "bytes_per_row": (rd + wr) / max(1, n[0] + n[1]),
            "achieved_GBps": (rd + wr) / (med * 1e-6) / 1e9,
        }
    finally:
        env.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--preroll", type=int, default=300)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--repeats", type=int, default=200)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("agent_state_bench.py needs a CUDA device")
    from predpreygrass_b200.build import build

    build()
    res = {"card": card(), "runs": []}
    for name, argv in (("base 4096", ["--envs", "4096"]),
                       ("add 16384", ["--reward-mode", "additive", "--envs", "16384"]),
                       ("eco 16384", ["--variant", "eco", "--envs", "16384"]),
                       ("stag 8192", ["--variant", "stag", "--envs", "8192", "--cap", "160", "640"])):
        r = measure(name, argv, args.preroll, args.steps, args.repeats)
        print(json.dumps(r), flush=True)
        res["runs"].append(r)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()
