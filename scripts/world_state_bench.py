"""Cost of `BatchedPredPreyGrass.world_state()` (ppg_world_state) on the flagship workloads.

For each config: the handle is pre-rolled (random actions, auto-reset) to the steady-state population, then
  * us per world_state() call over all envs (CUDA events around >= 200 back-to-back calls after warm-up),
  * bytes written (B*C*G*G*4) and image bytes read (B * image size), the resulting GB/s, and that rate as a fraction of
    the write-only (fill_) and read+write (copy_) rates of 2 GiB buffers measured in the same process (scripts/write_peak.py),
  * ms per step of the random rollout with and without one world_state() per step (alternated, device-timed),
  * whether the output fits the 126 MB L2 (consecutive calls rewrite the same buffer).
Prints one JSON document (also written to --out) with the GPU name and power limit (nvidia-smi query only).

    python scripts/world_state_bench.py --out profiles/world_state_b200.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

L2_BYTES = 126e6
CONFIGS = {  # name: (variant, reward mode, envs, cap_live) — bench.py's default caps
    "base": ("base", "sparse", 4096, (32, 128)),
    "add": ("base", "additive", 16384, (32, 128)),
    "eco": ("eco", "sparse", 16384, (32, 96)),
    "stag": ("stag", "sparse", 8192, (160, 640)),
}


def make_cfg(variant, mode, cap):
    from predpreygrass_b200 import config as cf

    if variant == "stag":
        return cf.make_config(cf.STAG_CONFIG, variant=cf.VARIANT_STAG, cap_live=cap, seed=1)
    if variant == "eco":
        return cf.make_config(cf.ECO_CONFIG, variant=cf.VARIANT_ECO, cap_live=cap, seed=1)
    return cf.make_config(cf.BASE_CONFIG, reward_mode=mode, cap_live=cap, seed=1)


def image_bytes(cfg):
    """bytes of one env image as ppg_create lays it out (csrc/ppg_api.cu): header, value tables, row descriptors, owner
    maps, wall table — what ppg_world_state_kernel reads per env"""
    eco, stag = cfg.variant == 1, cfg.variant == 2
    G, cap, ng = cfg.grid_size, (cfg.cap_live[0], cfg.cap_live[1]), cfg.n_grass
    off = [(cfg.obs_range[s] - 1) // 2 for s in range(2)]
    P = max(off)
    PH = max(2 * off[0], off[1]) if stag else P
    PS = G + PH
    align = lambda v, a: (v + a - 1) // a * a  # noqa: E731
    CH = align(P + (G + P + PH) * PS + P, 4)
    mb = 1 if cap[0] <= 253 and cap[1] <= 253 and ng <= 253 else 2
    o = 0

    def take(n, a):
        nonlocal o
        o = align(o, a)
        r = o
        o += n
        return r

    take(4 * 16, 16)
    vt0 = take(4 * (cap[0] + 2), 16)
    take(4 * (cap[1] + 1), 4)
    take(4 * (ng + 1), 4)
    for s in range(2):
        take(4 * cap[s] if (eco or stag) else 0, 4)
    for s in range(2):
        take(2 * cap[s], 2)
    need = (cfg.n_initial[0] + cfg.n_initial[1] + ng) * 4
    if o - vt0 < need:
        take(need - (o - vt0), 1)
    take(mb * CH, 16)
    take(mb * CH, 4)
    take(mb * CH, 4)
    take(mb * CH if stag else 0, 4)
    take(4 * (cap[0] + 2), 4)
    return align(o, 16)


def timed(fn, n):
    import torch

    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)  # ms


def peaks():
    """write-only and read+write HBM rates of 2 GiB buffers (scripts/write_peak.py), best of 10"""
    import torch

    x = torch.empty(1 << 29, dtype=torch.float32, device="cuda")
    y = torch.empty_like(x)
    nbytes = x.numel() * 4
    fill = min(timed(lambda: x.fill_(1.0), 1) for _ in range(10))
    copy = min(timed(lambda: y.copy_(x), 1) for _ in range(10))
    del x, y
    torch.cuda.empty_cache()
    return {"fill_GBps": nbytes / fill / 1e6, "copy_GBps": 2 * nbytes / copy / 1e6}


def measure(name, preroll, calls, steps):
    import torch

    from predpreygrass_b200.batched import BatchedPredPreyGrass

    variant, mode, B, cap = CONFIGS[name]
    cfg = make_cfg(variant, mode, cap)
    g = BatchedPredPreyGrass(cfg, B)
    g.reset()

    def step():
        g.step(*g.random_actions(7))

    for _ in range(preroll):
        step()
    for _ in range(20):
        g.world_state()
    torch.cuda.synchronize()
    ms_calls = [timed(g.world_state, calls) for _ in range(3)]
    us_call = min(ms_calls) / calls * 1e3
    C, G = cfg.num_obs_channels, cfg.grid_size
    written, img = B * C * G * G * 4, image_bytes(cfg)
    read = B * img

    def step_ws():
        step()
        g.world_state()

    ms_step, ms_step_ws = [], []
    for _ in range(2):  # alternated: the rollout keeps evolving, both arms see the same kind of population
        ms_step.append(timed(step, steps) / steps)
        ms_step_ws.append(timed(step_ws, steps) / steps)
    st = g.stats()
    g.close()
    return {"envs": B, "cap_live": list(cap), "channels": C, "grid": G, "preroll_steps": preroll, "timed_calls": calls,
            "us_per_call": us_call, "us_per_call_batches": [m / calls * 1e3 for m in ms_calls],
            "bytes_written": written, "image_bytes_per_env": img, "image_bytes_read": read,
            "GBps_written": written / us_call / 1e3, "GBps_read_plus_written": (written + read) / us_call / 1e3,
            "output_fits_L2": written < L2_BYTES,
            "ms_per_step": min(ms_step), "ms_per_step_with_world_state": min(ms_step_ws),
            "ms_per_step_runs": ms_step, "ms_per_step_with_world_state_runs": ms_step_ws, "rollout_steps_timed": steps,
            "world_state_share_of_step": us_call / 1e3 / min(ms_step), "status_envs": st["status_envs"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", nargs="+", default=list(CONFIGS), choices=list(CONFIGS))
    ap.add_argument("--preroll", type=int, default=300)
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("world_state_bench.py measures on a CUDA device; there is none")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1], "peaks": peaks(), "configs": {}}
    for name in args.configs:
        r = measure(name, args.preroll, args.calls, args.steps)
        r["fraction_of_fill"] = r["GBps_written"] / res["peaks"]["fill_GBps"]
        r["fraction_of_copy"] = r["GBps_read_plus_written"] / res["peaks"]["copy_GBps"]
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
