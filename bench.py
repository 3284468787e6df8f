"""bench.py -- env-steps/sec of the env.step hot path (random actions), contract per the round driver.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--env ID] [--envs-per-gpu E] [--impl reference] [--dump-outputs DIR]

Own arm: one "step" = ONE control step (10 physics substeps + obs/reward/done/auto-reset) of every env on
every rank.  `value` = env-steps/s with actions already resident in HBM; `e2e` = the same through
MyoVecEnv.step_host (pinned host action -> H2D, step, D2H of obs/reward/done inside the timed region).
Reference arm (--impl reference): the reference's CPU implementation of the path on the host cores.  MuJoCo
is not installable here (no network, not in /opt/wheelhouse), so this is the CPU oracle port
(oracle/libmyo_oracle.so) -- labelled kind="port".
Each env differs (per-env random state and actions); the working set lives in shared memory and the HBM traffic per
step is the compulsory state/action/obs I/O (8 MB for 4096 hand envs, smaller than L2), so L2 is evicted between
timed steps by a 192 MiB write inside the timed region (config.l2; --no-l2-flush turns it off; it costs < 1 %).
--dump-outputs DIR writes what env.step returned in the last timed step (see dump_outputs); the inputs are seeded, so two builds
run with the same arguments can be compared output for output.
The benchmark runs from the tree as build() left it and writes nothing into it: what it compiles goes to a temporary directory.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the tree may be read-only; leave no __pycache__ behind either

DEFAULT_ENV = "myoHandPoseRandom-v0"       # BASELINE.json target config (configs[2]; 23 dof / 39 muscles), 4096 envs/GPU
# algorithmic bytes per env-step (SURVEY.md section 8d, A_io): action f32 + state f64 in/out + obs f32 + reward/done
A_IO = {"myoElbowPose1D6MRandom-v0": 24 + 2 * (8 * 8) + 36 + 5, "myoHandPoseRandom-v0": 156 + 2 * (85 * 8) + 432 + 5,
        "myoHandObjHoldRandom-v0": 156 + 2 * (98 * 8) + 364 + 5 + 36, "myoFatiLegWalk-v0": 320 + 2 * (149 * 8) + 2 * (240 * 8) + 1612 + 5,
        "myoLegWalk-v0": 320 + 2 * (149 * 8) + 1612 + 5,
        "myoHandReachRandom-v0": 156 + 2 * (85 * 8) + 460 + 5 + 120}        # (+ 15 target coordinates f64)
A_OBS = {"myoElbowPose1D6MRandom-v0": 9, "myoHandPoseRandom-v0": 108, "myoHandObjHoldRandom-v0": 91, "myoFatiLegWalk-v0": 403, "myoLegWalk-v0": 403, "myoHandReachRandom-v0": 115}


def usable_cores():
    """Host cores this process may actually use: the scheduler affinity mask capped by the cgroup CPU quota
    (os.cpu_count() reports the machine, not the lease: round 1's arm forked 128 workers onto ~15 cores)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    try:                                     # cgroup v2
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:                                 # cgroup v1
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    if quota is not None:
        n = max(1, min(n, int(quota + 0.5)))
    return n


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region: NVML polled from a thread every 10 ms (the timed region of the default run is
    only ~0.1 s, shorter than nvidia-smi's start-up); falls back to an `nvidia-smi -lms` child when NVML cannot be loaded."""
    _BITS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))      # nvmlClocksThrottleReason* / ClocksEventReason*

    def __init__(self, index=0):
        self.rows, self.proc, self.index, self.h, self.run, self.thread, self.max_mhz = [], None, index, None, False, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else index
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.h = None

    def _poll(self):
        nv = self.nv
        while self.run:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    bits = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((mhz, bits))
            except Exception:
                pass
            time.sleep(0.010)

    def start(self):
        if self.h is not None:
            self.run = True
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.h is not None:
            self.run = False
            if self.thread:
                self.thread.join(timeout=1.0)
            sm = sorted(r[0] for r in self.rows)
            reasons = sorted(name for name, bit in self._BITS if any(r[1] & bit for r in self.rows))
            return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons, "samples": len(sm), "source": "nvml"}
        if self.proc:
            self.proc.terminate()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def _cpu_worker(args):
    """One host core: a single env stepped in a loop (reference protocol:
    /root/reference/benchmarks/mjx_benchmark_baseline.py:8-25 -- gym.make, reset, timeit(env.step(random action)))."""
    env_id, budget_s, seed, u01 = (tuple(args) + (False,))[:4]          # budget_s: wall-clock seconds of stepping (a bounded sample; the oracle's rate varies 10x with the contact load)
    import numpy as np
    from myosuite_b200 import assets, blob, vec_env
    from oracle import env_oracle
    from oracle.oracle_py import Oracle
    steps, kw, _ = vec_env.env_spec(env_id)
    m = assets.load(vec_env._MODEL_OF_XML[kw["model_path"]])
    o = Oracle(*blob.pack(m))
    rng = np.random.default_rng(seed)
    q = m.qpos0.copy()
    t0 = time.perf_counter()
    pose = "Pose" in env_id
    s = 0
    while time.perf_counter() - t0 < budget_s:
        if s % steps == 0:
            o.reset()
            if pose:
                for j in range(m.njnt):
                    if m.jnt_type[j] != 0:
                        q[m.jnt_qposadr[j]] = rng.uniform(*m.jnt_range[j])
                o.set(qpos=q)
            elif "Walk" in env_id:
                o.set(qpos=m.key_qpos[2], qvel=m.key_qvel[2])
        env_oracle.env_step(o, rng.uniform(0, 1, m.nu) if u01 else rng.uniform(-1, 1, m.nu), 10)
        if pose:
            env_oracle.pose_obs(o.f("qpos"), o.f("qvel"), o.f("act"), q, 0.02)
        else:
            o.forward()          # the reference's extra mj_forward for the observed data (robot.py:607)
        s += 1
    return s, time.perf_counter() - t0


def cpu_baseline(env_id, budget_s, threads=1, u01=False):
    """(env-steps/s, total steps) of `threads` independent single-env loops of the oracle port, one process per host core, each stepping
    for budget_s seconds of wall clock; the rate is total steps / the slowest worker's loop time (process start-up and model load excluded)."""
    if threads == 1:
        n, t = _cpu_worker((env_id, budget_s, 0, u01))
        return n / t, n
    import multiprocessing as mp
    with mp.get_context("fork").Pool(threads) as pool:
        res = pool.map(_cpu_worker, [(env_id, budget_s, i, u01) for i in range(threads)])
    return sum(r[0] for r in res) / max(r[1] for r in res), sum(r[0] for r in res)


MUJOCO_PUBLISHED = {"myoHandPoseRandom-v0": "reference's own CPU MuJoCo single-env figure on the hand model (myoHandReachRandom, derived from its plot): ~1.9 k env-steps/s on 1 core (BASELINE.md section 1)",
                    "myoElbowPose1D6MRandom-v0": "reference's own CPU MuJoCo single-env figure on this model (derived from its plot): ~10 k env-steps/s on 1 core (BASELINE.md section 1)"}


def reference_arm(args, W):
    """bench.py --impl reference: the CPU implementation of the path on the box's host cores.  MuJoCo is not installable here, so this is
    the oracle PORT (kind = "port"), built -O3 -march=native on this machine, one single-env loop per usable core."""
    from oracle import oracle_py
    os.environ["MYO_ORACLE_LIB"] = oracle_py.build_native()        # inherited by the forked workers
    thr = usable_cores()
    budget = float(os.environ.get("MYO_BENCH_CPU_BUDGET_S", 8.0))      # bounded sample: every usable core steps its own env for 8 s
    u01 = args.actions == "u01"
    t0 = time.perf_counter()
    v, total = cpu_baseline(args.env, budget, threads=thr, u01=u01)
    ms = (time.perf_counter() - t0) * 1e3
    per_thread = max(total // thr, 1)
    sample = "%d threads x %.0f s of stepping = %d env-steps of %s (1 env each, random actions %s, reset every episode); machine has %d CPUs, affinity/cgroup leave %d" % (
        thr, budget, total, args.env, "U(0,1)" if u01 else "U[-1,1]", os.cpu_count() or 0, thr)
    line = {"impl": "reference", "metric": "env-steps/sec (random actions, 4096 envs/GPU)", "value": v, "unit": "env-steps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": W, "ms_per_step": ms / max(per_thread, 1), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "%s, frame_skip 10, random actions %s, reset every episode; CPU arm: one single-env loop of the oracle port (gcc -O3 -march=native) per usable host core"
                                   % (args.env, "U(0,1)" if u01 else "U[-1,1]"),
                       "note": "the port is NOT MuJoCo; " + MUJOCO_PUBLISHED.get(args.env, "no published MuJoCo figure for this env")},
            "cpu_baseline": {"value": v, "unit": "env-steps/s", "cores": thr, "per_core": v / thr, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


DUMP_LIMIT = 64 * 10 ** 6          # bytes written by --dump-outputs in all


def dump_outputs(out_dir, step_result, seed=0):
    """Write what env.step returned (obs, reward, done, truncated and the arrays of its info dict) as <out_dir>/<name>.npy, float32 arrays
    as they are and every other dtype as float64 (exact for these integer flags and counters).  When the rows of all envs exceed
    DUMP_LIMIT, a fixed seeded sample of env rows, the same for every array, is written instead, with the env ids in env_index.npy."""
    import numpy as np
    obs, reward, done, truncated, info = step_result
    arrays = {"obs": obs, "reward": reward, "done": done, "truncated": truncated, **info}
    arrays = {k: v.detach().cpu().numpy() for k, v in arrays.items()}
    arrays = {k: v if v.dtype in (np.float32, np.float64) else v.astype(np.float64) for k, v in arrays.items()}
    n = len(obs)
    row_bytes = sum(v.nbytes for v in arrays.values()) // n
    budget = DUMP_LIMIT - 128 * (len(arrays) + 1)          # a .npy header is 128 bytes
    if n * row_bytes > budget:
        keep = np.sort(np.random.default_rng(seed).choice(n, budget // (row_bytes + 8), replace=False))
        arrays = {k: v[keep] for k, v in arrays.items()}
        arrays["env_index"] = keep.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--env", default=DEFAULT_ENV)
    ap.add_argument("--envs-per-gpu", type=int, default=4096)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--actions", default="u11", choices=["u11", "u01"], help="u11: U[-1,1] = action_space.sample() (default); u01: U(0,1), the reference benchmark's protocol (benchmarks/mjx_benchmark_baseline.py:15)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip config.extra (the other BASELINE configs, the U(0,1) variant, the sustained run)")
    ap.add_argument("--no-l2-flush", action="store_true", help="do not evict L2 between timed steps (default: a 192 MiB write per step)")
    ap.add_argument("--maxcon", type=int, default=0, help="contact capacity per env (0 = library default 32); experiments only")
    ap.add_argument("--barrier-mode", type=int, default=0)
    ap.add_argument("--lockstep-groups", type=int, default=0)
    ap.add_argument("--solver-tolerance", type=float, default=0.0, help="Newton stop (scaled gradient); 0 = library default")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what env.step returned in the last one as DIR/<name>.npy "
                                                          "(rank 0's envs; a fixed sample of envs above 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    W = max(args.warmup, 3)

    if args.impl == "reference":
        if rank == 0:
            reference_arm(args, W)
        return

    import torch
    import torch.distributed as dist
    from myosuite_b200 import abi, vec_env
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    if not os.path.exists(abi.lib_path()):
        raise SystemExit("bench.py: %s is missing -- build it first (python __graft_entry__.py)" % abi.lib_path())
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    # L2 (126 MB) is evicted between timed steps by writing a 192 MiB buffer: step k+1 reads the state step k wrote from HBM, not from L2
    flush_buf = None if args.no_l2_flush else torch.empty(192 << 20, dtype=torch.uint8, device=dev)

    def flush_l2(i):
        if flush_buf is not None:
            flush_buf.fill_(i & 1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(*ms):
        t = torch.tensor(list(ms), device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t]

    def make(env_id, n):
        env = vec_env.MyoVecEnv(env_id, n, device=local_rank, seed=0, env_offset=rank * n, barrier_mode=args.barrier_mode, lockstep_groups=args.lockstep_groups, solver_tolerance=args.solver_tolerance, maxcon=args.maxcon)
        env.reset(seed=0)
        return env

    def rings(env, u01):
        gen = torch.Generator(device=dev).manual_seed(1234 + rank + (7777 if u01 else 0))
        # a ring of pre-generated random action batches: U[-1,1] = the action_space.sample() distribution; U(0,1) = the reference benchmark's
        return [(torch.rand(env.num_envs, env.act_dim, device=dev, generator=gen) * (1 if u01 else 2) - (0 if u01 else 1)) for _ in range(16)]

    def timed(env, ring, steps, warm, flush=True, host=False):
        """ms for `steps` control steps of every env on this rank (CUDA events on the launching stream), max over ranks; launches issued;
        what the last step returned."""
        step = env.step_host if host else env.step
        for i in range(warm):
            step(ring[i % 16])
        barrier()
        l0 = env.batch.launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            if flush:
                flush_l2(i)
            last = step(ring[i % 16])
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))[0], env.batch.launches - l0, last

    n = args.envs_per_gpu
    env = make(args.env, n)
    nu = env.act_dim
    ring = rings(env, args.actions == "u01")
    ring_host = [r.cpu().pin_memory() for r in ring]
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms, launches, last = timed(env, ring, args.steps, W)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)          # before the runs below step the same envs further
    ms_e2e, _, _ = timed(env, ring_host, args.steps, 3, host=True)        # end to end through the public API with host buffers
    clocks = sampler.stop() if rank == 0 else None
    # the one collective of the path: gather finished-episode returns at rollout end (SURVEY.md section 8e), timed on its own
    allgather_us = None
    if world > 1:
        gathered = torch.empty(world * n, device=dev, dtype=torch.float32)
        dist.all_gather_into_tensor(gathered, env.t["last_return"])        # warm-up (communicator set-up)
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record(); dist.all_gather_into_tensor(gathered, env.t["last_return"]); g1.record()
        barrier()
        allgather_us = max_over_ranks(g0.elapsed_time(g1))[0] * 1e3
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))

    def roofline(env_id, n_env, ms_total, n_steps):
        # dominant kernel = the env-step kernel, launched once per control step; its launch duration is bounded above by the timed region
        # per step (which also holds the one-CTA regroup kernel, 0.2 %, and the L2 flush, 1 %: profiles/r02_launches_timed_region.csv)
        aio = A_IO.get(env_id, 0)
        achieved = aio * n_env / (ms_total * 1e-3 / max(n_steps, 1)) / 1e9
        traffic = None
        for tf in ("r02_traffic.json", "r01_traffic.json"):
            f = os.path.join(ROOT, "profiles", tf)
            if os.path.exists(f):
                traffic = json.load(open(f)).get(env_id)
                break
        return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "note": "fused step is issue/latency bound, not HBM bound (SURVEY 8d): algorithmic bytes %d B/env-step; peak = %s" % (aio, "measured" if peaks else "fallback")}

    extra = {}
    if not args.no_extra:
        # (a) sustained: >= 1 s and >= 1 full episode, so that TimeLimit truncation and the in-kernel auto-reset fire inside the timed region
        per = ms / max(args.steps, 1)
        ks = max(int(1000.0 / max(per, 1e-3)) + 1, (env.max_episode_steps or 100) + 10)
        ms_s, _, _ = timed(env, ring, ks, 0, flush=False)
        extra["sustained"] = {"steps": ks, "value": world * n * ks / (ms_s * 1e-3), "ms_per_step": ms_s / ks, "l2": "not flushed", "episodes_finished_per_env": float(env.t["episode_count"].double().mean().item()) - 1.0}
        # (b) the reference benchmark's action protocol, U(0,1)
        if args.actions == "u11":
            ms_u, _, _ = timed(env, rings(env, True), 30, 3)
            extra["actions_u01"] = {"steps": 30, "value": world * n * 30 / (ms_u * 1e-3), "ms_per_step": ms_u / 30}
        overflow_frac = float((env.t["overflow"] != 0).double().mean().item())
        del env
        # (c) the other BASELINE.json configs (2, 4, 5), measured outside the headline region
        # ... and myoHandReachRandom-v0: the env the reference's own published hand benchmark plot is drawn on (BASELINE.md section 1; SURVEY 8f-1)
        for eid, ne, st in (("myoElbowPose1D6MRandom-v0", 4096, 100), ("myoFatiLegWalk-v0", 2048, 30), ("myoHandObjHoldRandom-v0", 2048, 40), ("myoHandReachRandom-v0", 4096, 40)):
            if eid == args.env:
                continue
            e2 = make(eid, ne)
            ms2, l2, _ = timed(e2, rings(e2, False), st, 3)
            extra[eid] = {"envs_per_gpu": ne, "steps": st, "value": world * ne * st / (ms2 * 1e-3), "ms_per_step": ms2 / st, "roofline": roofline(eid, ne, ms2, st)}
            del e2
    else:
        overflow_frac = float((env.t["overflow"] != 0).double().mean().item())
    if rank == 0:
        total = world * n * args.steps
        value, e2e = total / (ms * 1e-3), total / (ms_e2e * 1e-3)
        line = {"metric": "env-steps/sec (random actions, 4096 envs/GPU)", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
                "warmup": W, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic", "impl": "b200",
                "config": {"workload": "%s, %d envs/GPU, frame_skip 10, random actions %s, auto-reset" % (args.env, n, "U(0,1)" if args.actions == "u01" else "U[-1,1]"),
                           "l2": ("not flushed (--no-l2-flush)" if args.no_l2_flush else "flushed between timed steps: a 192 MiB write per step inside the timed region (inputs, 8 MB of state per step, are smaller than L2)"), "parallelism": "env-sharded x%d, no data-path collective" % world,
                           "contact_overflow_env_fraction": overflow_frac, "rollout_end_allgather_us": allgather_us, "extra": extra},
                "e2e": {"value": e2e, "unit": "env-steps/s", "h2d_bytes_per_step": world * n * nu * 4, "d2h_bytes_per_step": world * n * (max(A_OBS.get(args.env, 0), 0) * 4 + 4 + 1)},      # whole job, like `value`
                "gpu_launches": int(launches),
                "roofline": roofline(args.env, n, ms, args.steps),
                "clocks": clocks}
        if not args.no_cpu_baseline and world == 1:      # the CPU leg is an N = 1 figure (rank 0 only); at N > 1 the other ranks would just wait for it
            from oracle import oracle_py
            os.environ["MYO_ORACLE_LIB"] = oracle_py.build_native()
            t0 = time.perf_counter()
            v, nst = cpu_baseline(args.env, float(os.environ.get("MYO_BENCH_CPU_BUDGET_S", 10.0)), threads=1, u01=args.actions == "u01")         # bounded sample: 10 s of single-thread stepping
            line["cpu_baseline"] = {"value": v, "unit": "env-steps/s", "cores": 1, "kind": "port",
                                    "sample": "%d env-steps of %s, 1 env, 1 thread (%.1f s), oracle port built -O3 -march=native; not MuJoCo: %s" % (nst, args.env, time.perf_counter() - t0, MUJOCO_PUBLISHED.get(args.env, "no published figure"))}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
