#!/usr/bin/env python
"""Cost of GAE on the device (include/ppg.h ppg_gae, connector.RolloutBuffer) next to the steps it covers.

For each configuration (bench.py's BASE at 4096 envs with T = 64 and T = 128; its ECO configuration at 16384 envs and its
STAG configuration at 8192 envs, the env counts of bench.py's `configs` runs, with T = 64; one handle each):
pre-roll the envs to their steady-state population with random actions, then in one process
  - time T steps of random actions with CUDA events (the rollout's step time, no recording),
  - record T+1 outputs into a RolloutBuffer, timing every record() call with CUDA events around it on the stream,
  - time `--repeats` compute() calls (one ppg_gae launch each) with CUDA events,
and report the times and their shares of the step time.  The card's name and power limit are read in the same run.
Usage: python scripts/gae_bench.py [--out FILE] [--preroll 300] [--repeats 50]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


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


def measure(variant, envs, T, preroll, repeats, keep_obs):
    import torch

    import bench
    from predpreygrass_b200.batched import BatchedPredPreyGrass
    from predpreygrass_b200.connector import RolloutBuffer

    args = bench.parse(["--variant", variant, "--envs", str(envs)])
    cfg = bench.build_config(args, seed=12345)
    env = BatchedPredPreyGrass(cfg, args.envs)
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    try:
        env.reset()
        for _ in range(preroll):
            env.step(*env.random_actions(7))
        torch.cuda.synchronize()
        # T steps, no recording
        e0, e1 = ev(), ev()
        e0.record()
        for _ in range(T):
            env.step(*env.random_actions(7))
        e1.record()
        torch.cuda.synchronize()
        ms_steps = e0.elapsed_time(e1)
        # T+1 recorded outputs
        buf = RolloutBuffer(env, T, keep_obs=keep_obs)
        rec = []
        rows = 0
        for t in range(T + 1):
            n = env.out.counts()
            rows += n[0] + n[1]
            vals = tuple(torch.zeros(n[s], device=env.device) for s in range(2))
            acts = tuple(env.actions[s][: n[s]] for s in range(2))
            a, b = ev(), ev()
            a.record()
            buf.record(vals, actions=acts if t < T else None)
            b.record()
            rec.append((a, b))
            if t < T:
                env.step(*env.random_actions(7))
        torch.cuda.synchronize()
        ms_record = [a.elapsed_time(b) for a, b in rec]
        buf.compute(0.99, 0.95)  # warm-up launch
        cols = buf.columns()
        n_tr = sum(int(c["advantages"].shape[0]) for c in cols.values())
        del cols
        starts, ends = [ev() for _ in range(repeats)], [ev() for _ in range(repeats)]
        for k in range(repeats):
            starts[k].record()
            buf.compute(0.99, 0.95)
            ends[k].record()
        torch.cuda.synchronize()
        ms_gae = sorted(s.elapsed_time(e) for s, e in zip(starts, ends))
        med = ms_gae[len(ms_gae) // 2]
        rec_mean = sum(ms_record[:T]) / T
        return {
            "variant": variant, "envs": args.envs, "cap_live": list(args.cap), "T": T, "keep_obs": keep_obs,
            "rows_per_output_mean": rows / (T + 1), "transitions": n_tr,
            "ms_per_step": ms_steps / T, "ms_T_steps": ms_steps,
            "ms_gae_median": med, "ms_gae_min": ms_gae[0], "ms_gae_max": ms_gae[-1], "gae_repeats": repeats,
            "gae_share_of_T_steps": med / ms_steps,
            "ms_record_per_step_mean": rec_mean, "record_share_of_step": rec_mean / (ms_steps / T),
        }
    finally:
        env.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--preroll", type=int, default=300)
    ap.add_argument("--repeats", type=int, default=50)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("gae_bench.py needs a CUDA device")
    from predpreygrass_b200.build import build

    build()
    res = {"card": card(), "runs": []}
    # observation rows are kept where they fit comfortably (BASE); ECO and STAG record the small columns only
    for variant, envs, T, keep_obs in (("base", 4096, 64, True), ("base", 4096, 64, False), ("base", 4096, 128, True),
                                       ("eco", 16384, 64, False), ("stag", 8192, 64, False)):
        r = measure(variant, envs, T, args.preroll, args.repeats, keep_obs)
        print(json.dumps(r), flush=True)
        res["runs"].append(r)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()
