#!/usr/bin/env python
"""bench.py — agent-steps/s (incl. observation generation) of the batched PredPreyGrass env step.

Contract (driver): `python bench.py --gpus N --steps K --warmup W [--impl reference]`, for N > 1
launched under torchrun (one rank per GPU).  Prints ONE JSON line on rank 0.

A "step" is one lockstep `step()` of every env instance the rank owns (BASELINE configs[1]:
base_environment, 4096 envs per GPU, uniform random actions from the device-side Philox action
generator, auto-reset).  Before the W warm-up steps every env is PRE-ROLLED `--preroll` untimed steps
(default 300) so that the timed region sees the steady-state population the metric is quoted on
(~35 live agents per env for BASE; a fresh reset has 14) — SURVEY §8d "warm-up 200 steps".

`value` = agent-steps/s over all ranks with everything resident in HBM; `e2e` = the same through
`ppg_step_host` (actions from pinned host memory, whole row batch copied back to pinned host memory
every step); `e2e_device_policy` = the zero-copy consumer path (a torch policy reads the row batch in
place and writes the actions in place: `predpreygrass_b200.connector`).  `roofline` is the DOMINANT
kernel by bytes, `ppg_obs_kernel` (> 85 % of the bytes of a step): the observation-row bytes it wrote
(counted on the device) over its CUDA-event duration against MEASURED_PEAKS.json; `roofline.whole_step`
relates ALL algorithmic bytes of a step (SURVEY §8d) to the measured `ms_per_step`.  `cpu_baseline` is
the CPU oracle (a C port of the reference's Python step; the Python reference itself cannot travel to
the GPU box) on host cores.  `configs` holds short runs of BASELINE configs[2..4] (ADD 16384 envs,
ECO 16384 envs, STAG 8192 envs per GPU); at N > 1 `allreduce_us` is the median latency of the one
collective of the path (the statistics all-reduce, SURVEY §8e).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "agent_steps_per_s_incl_obs"
UNIT = "agent-steps/s"
_REAL_STDOUT = 1
S_AGENT = 42  # bytes of per-agent state + io per agent-step (SURVEY §8d): pos 2 + energy 8 + id 4 (read+write = 28), action 4, reward 4 + flags 2 + id 4
L2_BYTES = 126e6

DEFAULT_CAPS = {"base": [32, 128], "eco": [32, 96], "eco_rich": [256, 512], "stag": [160, 640],
                "cadence": [32, 96], "metabolic": [32, 96], "investment": [32, 96], "cooperation": [32, 96]}
ECO_FAMILY = ("eco", "cadence", "metabolic", "investment", "cooperation")


def parse(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--preroll", type=int, default=300,
                    help="untimed steps before the warm-up that bring every env to its steady-state population")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=4096, help="env instances per GPU (BASELINE configs[1])")
    ap.add_argument("--groups", type=int, default=None,
                    help="env groups per GPU stepped on their own CUDA streams (software pipelining: the latency-bound step "
                         "kernel of one group runs under the bandwidth-bound observation kernel of the other); default per variant")
    ap.add_argument("--variant", default="base", choices=["base", "stag"] + list(ECO_FAMILY),
                    help="base: BASELINE configs[1]/[2] (base_environment family); eco: configs[3] (eco_evolutionary, speed trait); "
                         "stag: configs[4] (stag_hunt_forward_view_nature_nurture, team capture); cadence / metabolic / investment / "
                         "cooperation: the other heritable-trait variants of north_star")
    ap.add_argument("--eco-rich", action="store_true", help="eco: reproduction-heavy override (thresholds 8/5, grass regrowth 0.3)")
    ap.add_argument("--seasonal", action="store_true", help="base: base_environment_seasonal config (square-wave grass regrowth)")
    ap.add_argument("--reward-mode", default="sparse")
    ap.add_argument("--cap", type=int, nargs=2, default=None)
    ap.add_argument("--e2e-steps", type=int, default=30)
    ap.add_argument("--cpu-envs", type=int, default=2048, help="envs of the cpu_baseline sample of the GPU arm")
    ap.add_argument("--cpu-steps", type=int, default=200, help="timed steps of the cpu_baseline sample (after as many untimed ones)")
    ap.add_argument("--ref-envs", type=int, default=None, help="reference arm: envs stepped (default: --envs, the labelled workload)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the short runs of BASELINE configs[2..4]")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the row batch of the last timed step as DIR/<name>.npy (rank 0; see dump_outputs)")
    args = ap.parse_args(argv)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.cap is None:
        # slot capacity per env and species: large enough that no env of the rollout ever fills it (`status_envs` 0 —
        # a full list would suppress births the reference allows); measured maxima: BASE 26 / 83, ECO 13 / 65,
        # ECO reproduction-heavy 222 / 416+, STAG 127 / 416+ (scripts/status_diag.py)
        args.cap = DEFAULT_CAPS["eco_rich" if (args.variant == "eco" and args.eco_rich) else args.variant]
    args.groups_explicit = args.groups is not None or "PPG_BENCH_GROUPS" in os.environ
    if args.groups is None:
        # measured (profiles/r02_summary.md): two groups win where each group still fills the GPU's 2960 step-kernel warps
        # (16384-env configs of the base / eco families: +8..12 %), lose at 4096 envs (-20 %) and for STAG (-3 %)
        auto = 2 if (args.variant != "stag" and args.envs >= 8192 and args.envs % 2 == 0) else 1
        args.groups = int(os.environ.get("PPG_BENCH_GROUPS", auto))
    return args


def workload_name(args):
    pre = f"pre-rolled {args.preroll} untimed steps to the steady-state population"
    if args.variant == "stag":
        return (f"stag_hunt_forward_view_nature_nurture default config_env, {args.envs} envs per GPU, uniform random actions "
                f"(predators [9, 2], prey 9), auto-reset, Philox facing/trait/capture draws, {pre}")
    if args.variant in ECO_FAMILY:
        name = {"eco": "eco_evolutionary", "cadence": "eco_evolutionary_cadence", "metabolic": "eco_evolutionary_metabolic_rate",
                "investment": "eco_evolutionary_investment", "cooperation": "eco_evolutionary_cooperation"}[args.variant]
        return (f"{name} default config_env{' + reproduction-heavy override' if args.eco_rich else ''}, {args.envs} envs per GPU, "
                f"uniform random actions ({n_actions(args)}), auto-reset, Philox trait/mutation draws, {pre}")
    name = "base_environment_seasonal" if getattr(args, "seasonal", False) else "base_environment"
    return f"{name} default config_env, {args.envs} envs per GPU, uniform random actions, auto-reset, reward={args.reward_mode}, {pre}"


def config_block(args):
    """static description of the workload: identical in the GPU arm and the reference arm"""
    return {"workload": workload_name(args), "envs_per_gpu": args.envs, "cap_live": list(args.cap), "preroll_steps": args.preroll,
            "l2": "no explicit flush: every step rewrites the handle's observation-row buffers (same addresses every step) with the "
                  "bytes given in l2_note; when that exceeds the 126 MB L2 the row stream cannot stay cache-resident",
            "state": "fp64 energies in HBM, fp32 observations/rewards out"}


def build_config(args, **kw):
    from predpreygrass_b200 import config as cf

    if args.variant == "stag":
        return cf.make_config(cf.STAG_CONFIG, variant=cf.VARIANT_STAG, cap_live=tuple(args.cap), **kw)
    if args.variant in ECO_FAMILY:
        d = dict(cf.ECO_CONFIG if args.variant == "eco" else cf.TRAIT_CONFIGS[args.variant])
        if args.eco_rich:
            d.update(energy_gain_per_step_grass=0.3, prey_creation_energy_threshold=5.0, predator_creation_energy_threshold=8.0,
                     energy_loss_per_step_predator=0.1, n_possible_predators=8000, n_possible_prey=24000)
        return cf.make_config(d, variant=cf.VARIANT_ECO, cap_live=tuple(args.cap), **kw)
    if getattr(args, "seasonal", False):
        return cf.make_config(cf.SEASONAL_CONFIG, reward_mode=args.reward_mode, cap_live=tuple(args.cap), **kw)
    return cf.make_config(cf.BASE_CONFIG, reward_mode=args.reward_mode, cap_live=tuple(args.cap), **kw)


def n_actions(args):
    return 25 if args.variant == "eco" else 9  # the trait variants have action_range 3 (MR:203-210, CAD config)


def action_pools(args, n, rng):
    """host-side random actions (numpy int32) for n rows per species; STAG predators carry the join_hunt bit (include/ppg.h)"""
    import numpy as np

    a0 = rng.integers(0, n_actions(args), size=n, dtype=np.int32)
    a1 = rng.integers(0, n_actions(args), size=n, dtype=np.int32)
    if args.variant == "stag":
        a0 = a0 | (rng.integers(0, 2, size=n, dtype=np.int32) << 8)
    return a0, a1


class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index), "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def cpu_oracle_rate(args, n_envs, threads, steps, untimed):
    """agent-steps/s of the CPU oracle (C port of the reference step) on `threads` host threads: `untimed` steps first
    (population build-up), then `steps` timed ones."""
    import numpy as np

    from oracle.oracle import Oracle

    cfg = build_config(args, seed=12345)
    o = Oracle(cfg, n_envs, threads=threads)
    o.reset()
    rng = np.random.default_rng(0)
    pool0, pool1 = action_pools(args, n_envs * (args.cap[0] + args.cap[1]) + 16, rng)

    def run(k):
        t = 0.0
        for _ in range(k):
            t0 = time.perf_counter()
            o.step(pool0, pool1)  # any action value is valid for any row; sampling is not timed
            t += time.perf_counter() - t0
        return t

    run(untimed)
    s0 = o.stats()
    dt = run(steps)
    s1 = o.stats()
    o.close()
    agent_steps = int(s1[1] - s0[1])
    env_steps = int(s1[0] - s0[0])
    return agent_steps / dt, env_steps / dt, dt, agent_steps / max(env_steps, 1)


def main_reference(args, rank):
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    n_envs = args.ref_envs or args.envs
    W = max(3, args.warmup)
    rate, env_rate, dt, live = cpu_oracle_rate(args, n_envs, threads, args.steps, args.preroll + W)
    sample = (f"{n_envs} envs x {args.steps} timed steps of the same workload after {args.preroll} pre-roll + {W} warm-up steps, "
              f"{threads} threads (envs partitioned over threads)")
    cfgb = config_block(args)
    if n_envs != args.envs:
        cfgb["reference_sample_envs"] = n_envs
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": W, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": cfgb,
        "note": "reference arm = CPU oracle (C port of the reference's Python step; the Python reference cannot travel to the GPU box)",
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "env_steps_per_s": env_rate, "mean_live_agents_per_env": live, "gpu_launches": 0,
    }
    emit(line)


def emit(line):
    """the ONE JSON line of the contract, on the process's real stdout"""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


def load_peak():
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(peaks["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    except Exception:
        return 6650.0, "fallback 6650 GB/s (of fallback)"


DUMP_BYTES = 64 << 20


def dump_outputs(pipe, out_dir, stats):
    """Writes what the timed path handed out in its last step, as out_dir/<name>.npy (integers as float64, observations and
    rewards as float32), so that two builds run with the same arguments can be compared array for array:

      stats                                 the statistics vector of the timed steps (config.STAT_NAMES)
      env_flags, env_status, env_step, env_count
      {pred,prey}_old_off, _new_off, _new_cnt  row offsets per env (new_off is 0 where new_cnt is 0, as include/ppg.h leaves it undefined)
      {pred,prey}_row_index                 which valid rows the per-row arrays below hold
      {pred,prey}_obs, _reward, _row_env, _row_agent, _flags

    With several env groups every array is the concatenation of the groups' arrays in group order (offsets and row_env stay
    relative to the group), and a row index counts the valid rows of all groups in that order.  When the valid rows do not fit
    in DUMP_BYTES, the per-row arrays hold a sample: a sorted draw without replacement from a fixed-seed generator."""
    import numpy as np
    import torch

    outs = [e.out for e in pipe.envs]
    f64 = lambda ts: torch.cat([t.to(torch.float64) for t in ts]).cpu().numpy()  # noqa: E731
    arrays = {"stats": stats.to(torch.float64).cpu().numpy()}
    for name in ("env_flags", "env_status", "env_step", "env_count"):
        arrays[name] = f64([getattr(o, name) for o in outs])
    for s, sp in enumerate(("pred", "prey")):
        arrays[f"{sp}_old_off"] = f64([o.old_off[s] for o in outs])
        arrays[f"{sp}_new_off"] = f64([torch.where(o.new_cnt[s] > 0, o.new_off[s], 0) for o in outs])
        arrays[f"{sp}_new_cnt"] = f64([o.new_cnt[s] for o in outs])
    budget = (DUMP_BYTES - sum(a.nbytes for a in arrays.values())) // 2  # per species
    for s, sp in enumerate(("pred", "prey")):
        n = [o.counts()[s] for o in outs]
        total = sum(n)
        row_bytes = 4 * pipe.C * pipe.R[s] ** 2 + 4 + 4 * 8  # obs + reward (f32), row index, env, agent, flags (f64)
        m = min(total, budget // row_bytes)
        idx = np.arange(total) if m == total else np.sort(np.random.default_rng(s).choice(total, m, replace=False))
        parts = {k: [] for k in ("obs", "reward", "row_env", "row_agent", "flags")}
        first = 0
        for o, k in zip(outs, n):
            sel = idx[(idx >= first) & (idx < first + k)] - first
            sel = torch.from_numpy(sel).to(o.obs[s].device)
            for name in parts:
                parts[name].append(getattr(o, name)[s].index_select(0, sel))
            first += k
        arrays[f"{sp}_row_index"] = idx.astype(np.float64)
        arrays[f"{sp}_obs"] = torch.cat(parts["obs"]).cpu().numpy()
        arrays[f"{sp}_reward"] = torch.cat(parts["reward"]).cpu().numpy()
        for name in ("row_env", "row_agent", "flags"):
            arrays[f"{sp}_{name}"] = f64(parts[name])
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return sorted(arrays)


class Rollout:
    """`groups` handles of envs / groups env instances each, every group on its own CUDA stream."""

    def __init__(self, args, rank, local_rank, envs, groups):
        import torch

        from predpreygrass_b200.pipelined import PipelinedPredPreyGrass

        self.args, self.torch = args, torch
        self.envs, self.groups = envs, groups
        self.pipe = PipelinedPredPreyGrass(lambda base, **kw: build_config(args, seed=1000, env_index_base=rank * envs + base, **kw),
                                           envs, groups=groups, device=local_rank)
        self.pipe.reset()

    def run(self, k):
        self.pipe.rollout_random(k, 4242)

    def stats(self):
        return self.pipe.stats_device().clone()

    def launches(self):
        return self.pipe.launch_count()

    def close(self):
        self.pipe.close()


def measure(args, rank, local_rank, world, K, W, full):
    """one workload on this rank's GPU -> dict (device-timed, max over ranks)"""
    import numpy as np
    import torch
    import torch.distributed as dist

    from predpreygrass_b200.config import STAT_NAMES

    dev = torch.device("cuda", local_rank)
    ro = Rollout(args, rank, local_rank, args.envs, args.groups)
    pipe = ro.pipe
    cfg = pipe.cfg

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ro.run(args.preroll)  # untimed: population build-up
    ro.run(W)
    torch.cuda.synchronize()
    stats0 = ro.stats()
    launches0 = ro.launches()
    sampler = ClockSampler(local_rank)
    if full:
        sampler.start()
        time.sleep(0.25)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    pipe.fork(ev0)   # ev0 on the current stream; every group stream waits for it
    t_host = time.perf_counter()
    ro.run(K)
    t_host = time.perf_counter() - t_host  # host time to ISSUE the timed region's launches (no synchronisation inside)
    pipe.join(ev1)   # the current stream waits for every group stream; ev1 after that
    barrier()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if full else None
    launches = ro.launches() - launches0
    stats1 = ro.stats()
    if full and args.dump_outputs and rank == 0:
        dump_outputs(pipe, args.dump_outputs, stats1 - stats0)
    d = (stats1 - stats0).to(torch.float64)  # this rank's env/agent steps, rows, births... in the timed region
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        # the one collective of this path: the small all-reduce of episode/population statistics
        dist.all_reduce(d, op=dist.ReduceOp.SUM)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    tot = dict(zip(STAT_NAMES, d.tolist()))
    value = tot["agent_steps"] / (ms_max * 1e-3)
    env_rate = tot["env_steps"] / (ms_max * 1e-3)
    row_bytes = [4 * pipe.C * cfg.obs_range[s] ** 2 for s in range(2)]
    s_agent = S_AGENT + (20 if args.variant != "base" else 0)  # + trait 8 (read+write 16), age 2+2 (SURVEY §8d)
    # algorithmic bytes of the timed region, per step of one rank (SURVEY §8d)
    obs_bytes_t = (tot["rows_pred"] * row_bytes[0] + tot["rows_prey"] * row_bytes[1]) / K / world
    alg_bytes_t = obs_bytes_t + (tot["agent_steps"] * s_agent + tot["env_steps"] * (cfg.n_grass * 16 + 64)) / K / world
    peak, peak_source = load_peak()

    # ---- per-kernel timing: CUDA events recorded by the library on the launching stream around each of the step's kernels
    # (kernels back to back, no overlap, one group after the other: a kernel's time is its own)
    KR = min(K, 200)
    sk0 = ro.stats()
    torch.cuda.synchronize()
    step_ms_sum, obs_ms_sum = pipe.profile_rollout(KR, 4242)
    sk1 = ro.stats()
    kd = dict(zip(STAT_NAMES, (sk1 - sk0).tolist()))
    step_ms, obs_ms = step_ms_sum / KR, obs_ms_sum / KR  # per lockstep step of ALL the rank's envs (sum over the groups' launches)
    obs_bytes = (kd["rows_pred"] * row_bytes[0] + kd["rows_prey"] * row_bytes[1]) / KR
    alg_bytes = obs_bytes + (kd["agent_steps"] * s_agent + kd["env_steps"] * (cfg.n_grass * 16 + 64)) / KR
    step_kernel = "ppg_step_stag_kernel" if args.variant == "stag" else "ppg_step_eco_kernel" if args.variant in ECO_FAMILY else "ppg_step_base_kernel"
    live = tot["agent_steps"] / max(tot["env_steps"], 1.0)
    traffic, traffic_note = None, "no ncu capture of this workload at this population under profiles/traffic.json"
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(f"{args.variant}_{args.envs}_g{args.groups}", {})
        # only a capture of the same workload at the same population says anything about this run
        if tj and abs(tj.get("mean_live_agents_per_env", 0.0) - live) <= 0.1 * live:
            traffic = tj.get("dram_bytes_per_launch")
            traffic_note = tj.get("source")
    except Exception:
        pass
    achieved = obs_bytes / (obs_ms * 1e-3) / 1e9 if obs_ms > 0 else 0.0  # bytes of all the groups' launches over their summed durations
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_note": traffic_note,
                "kernel": "ppg_obs_kernel", "kernel_ms": obs_ms / args.groups, "launches_per_step": args.groups,
                "algorithmic_bytes_per_launch": obs_bytes / args.groups,
                "step_kernel": step_kernel, "step_kernel_ms": step_ms / args.groups,
                "whole_step": {"ms": ms_max / K, "algorithmic_bytes": alg_bytes_t,
                               "achieved": alg_bytes_t / (ms_max / K * 1e-3) / 1e9,
                               "frac": alg_bytes_t / (ms_max / K * 1e-3) / 1e9 / peak,
                               "note": "all algorithmic bytes of a step (SURVEY §8d) over the measured ms_per_step of the timed region"},
                "kernels_back_to_back": {"ms": step_ms + obs_ms, "frac": alg_bytes / ((step_ms + obs_ms) * 1e-3) / 1e9 / peak},
                "peak_source": peak_source}
    res = {"value": value, "ms_per_step": ms_max / K, "env_steps_per_s": env_rate, "mean_live_agents_per_env": live,
           "roofline": roofline, "gpu_launches": int(launches), "clocks": clocks, "tot": tot, "host_issue_ms_per_step": 1e3 * t_host / K,
           "l2_note": "%.0f MB of observation rows per step and GPU (%s the 126 MB L2), written to the same buffers every step"
                      % (obs_bytes_t / 1e6, "more than" if obs_bytes_t > L2_BYTES else "LESS than")}

    if full and not args.no_e2e:
        # ---- e2e through the C-ABI with host buffers (rank-local rate, summed over ranks); group 0's handle owns all envs of
        # this leg when groups == 1, else every group is stepped through its own ppg_step_host call
        res["e2e"] = pipe.bench_host(args.e2e_steps, lambda n: action_pools(args, n, np.random.default_rng(1)), row_bytes, barrier, world, dev)
        res["e2e"]["unit"] = UNIT
        res["e2e_device_policy"] = pipe.bench_device_policy(min(K, 100), barrier, world, dev)
        res["e2e_device_policy"]["unit"] = UNIT
    if world > 1 and full:
        # latency of the statistics all-reduce (128 bytes), median of 100, CUDA events on the current stream
        sv = pipe.stats_device()
        for _ in range(10):
            dist.all_reduce(sv, op=dist.ReduceOp.SUM)
        lat = []
        for _ in range(100):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            dist.all_reduce(sv, op=dist.ReduceOp.SUM)
            b.record()
            b.synchronize()
            lat.append(a.elapsed_time(b) * 1e3)
        res["allreduce_us"] = statistics.median(lat)
    res["status_envs"] = pipe.stats()["status_envs"]
    ro.close()
    return res


def main():
    args = parse()
    # libraries print to stdout behind Python's back (NCCL: "NCCL version ..."): everything but the JSON line goes to stderr
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return main_reference(args, rank)

    import torch
    import torch.distributed as dist

    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    bound = 0
    if world > 1 and os.environ.get("PPG_BENCH_BIND", "1") != "0":
        from predpreygrass_b200.sharding import bind_to_gpu_locality

        bound = bind_to_gpu_locality(local_rank)  # pinned e2e buffers on the GPU's own NUMA node
        print(f"[bench] rank {rank}: bound to {bound} cores next to GPU {local_rank}", file=sys.stderr)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W, K = max(3, args.warmup), args.steps

    res = measure(args, rank, local_rank, world, K, W, full=True)

    # ---- short runs of the other BASELINE configs (value + roofline each; same pre-roll, 50 timed steps)
    others = None
    if not args.no_configs and args.variant == "base" and args.reward_mode == "sparse" and not args.seasonal and args.envs == 4096:
        others = {}
        for name, extra in (("configs[2] dense_rewards_additive 16384 envs", ["--reward-mode", "additive", "--envs", "16384"]),
                            ("configs[3] eco_evolutionary 16384 envs", ["--variant", "eco", "--envs", "16384"]),
                            ("configs[4] stag_hunt 8192 envs per GPU", ["--variant", "stag", "--envs", "8192"])):
            a2 = parse(extra + ["--preroll", str(args.preroll), "--no-e2e", "--no-cpu"] + (["--groups", str(args.groups)] if args.groups_explicit else []))
            try:
                r2 = measure(a2, rank, local_rank, world, 50, 5, full=False)
                others[name] = {"value": r2["value"], "unit": UNIT, "ms_per_step": r2["ms_per_step"], "envs_per_gpu": a2.envs,
                                "cap_live": a2.cap, "groups": a2.groups, "mean_live_agents_per_env": r2["mean_live_agents_per_env"],
                                "obs_kernel_frac": r2["roofline"]["frac"], "whole_step_frac": r2["roofline"]["whole_step"]["frac"],
                                "obs_kernel_ms": r2["roofline"]["kernel_ms"], "step_kernel_ms": r2["roofline"]["step_kernel_ms"],
                                "status_envs": r2["status_envs"], "steps": 50, "warmup": 5}
            except Exception as ex:  # a config that fails must not take the headline line with it
                others[name] = {"error": repr(ex)[:300]}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        threads = os.cpu_count() or 1
        r, er, dt, live = cpu_oracle_rate(args, args.cpu_envs, threads, args.cpu_steps, args.cpu_steps)
        cpu = {"value": r, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"{args.cpu_envs} envs x {args.cpu_steps} timed steps of the same workload ({dt:.1f} s) after {args.cpu_steps} untimed ones "
                         f"({live:.1f} live agents per env), oracle/ C port of the reference step, {threads} threads"}

    if rank == 0:
        cfgb = config_block(args)
        line = {
            "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": cfgb, "groups": args.groups, "host_cores_bound": bound, "l2_note": res["l2_note"],
            # launch chain between steps (include/ppg.h ppg_set_pdl_chain): off unless PPG_PDL_CHAIN=1, and never used with env groups
            "launch_chain": "on" if (args.groups == 1 and os.environ.get("PPG_PDL_CHAIN", "0") not in ("", "0")) else "off",
            "env_steps_per_s": res["env_steps_per_s"],
            "mean_live_agents_per_env": res["mean_live_agents_per_env"],
            "roofline": res["roofline"], "cpu_baseline": cpu, "e2e": res.get("e2e"), "e2e_device_policy": res.get("e2e_device_policy"),
            "gpu_launches": res["gpu_launches"], "host_issue_ms_per_step": res["host_issue_ms_per_step"],
            "clocks": res["clocks"], "status_envs": res["status_envs"],
        }
        if "allreduce_us" in res:
            line["allreduce_us"] = res["allreduce_us"]
        if others is not None:
            line["configs"] = others
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
