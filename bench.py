"""
bench.py -- env-steps/sec of the batched random-action LocoEnv.step() rollout (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--envs 4096] [--task UnitreeA1.simple]
  python bench.py --impl reference ...      # the CPU restatement of the reference loop on the host cores
  python bench.py --dump-outputs DIR ...    # also write the last timed step's outputs of every workload as DIR/*.npy

Headline workload (BASELINE.json configs[1]): UnitreeA1.simple, 4096 envs per GPU, actions ~ U(-1,1)^12, auto-reset
from the mini-dataset table; a "step" is one LocoEnv.step() of the whole batch (= 10 MuJoCo sub-steps per env).
The same JSON line carries, under "configs", the other single-box BASELINE configs measured the same way in the same
run: HumanoidTorque.run @ 4096 envs/GPU (config 3) and the mixed Atlas.walk + Talos.walk batch with domain randomisation
@ 1024 + 1024 envs/GPU (config 4: two engines, each spread over all SMs, back to back).  One JSON line on stdout (rank 0).  DESIGN.md "Measurement" explains every field.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault("LOCO_MUJOCO_B200_FORCE_BUNDLED", "1")     # the GPU box has no reference checkout
# (set before CUDA initialises) one hardware work queue per stream: with the default of 8, two of a mixed batch's streams can
# alias to one queue, which serialises the members' kernels (config 4: 3.0 instead of 2.5 ms per step); the package sets it too
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

METRIC = "env-steps/sec (batched random-action rollout)"


def algo_bytes(eng):
    """Algorithmic HBM bytes of one env-step (SURVEY 8(d), DESIGN.md section 4): read qpos, qvel, warmstart (3 nv floats) and
    the action (nu floats), write the same state back plus obs (D floats), reward (4 B) and done (1 B).
    UnitreeA1 633, HumanoidTorque 657, Atlas 549, Talos 621."""
    return 4 * (6 * eng.nq + eng.action_dim + eng.obs_dim + 1) + 1

# Per-launch figures of step_kernel from the committed ncu captures of the CURRENT build (profiles/README.md, round 2):
# DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum, `--set full`) and FP32 flops per env-step
# (2*FFMA + FMUL + FADD thread instructions / envs).  None = not captured for that robot.
NCU = json.load(open(os.path.join(ROOT, "profiles", "ncu_constants.json"))) \
    if os.path.exists(os.path.join(ROOT, "profiles", "ncu_constants.json")) else {}
PREROLL = 40          # untimed steps after the mass reset, so that the timed window sees the stationary episode-age mix
# array bytes --dump-outputs writes at most (the whole dump, .npy headers included, stays under 64 MB); past it every member
# keeps the same seeded fraction of its envs
DUMP_BYTES = 60 * 1024 * 1024


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=200)
    p.add_argument("--warmup", type=int, default=20)
    p.add_argument("--envs", type=int, default=4096, help="envs per GPU")
    p.add_argument("--task", default="UnitreeA1.simple")
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--cpu-seconds", type=float, default=12.0, help="target duration of the cpu_baseline sample")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-configs", action="store_true", help="headline workload only (skip configs 3 and 4)")
    p.add_argument("--no-flush", action="store_true", help="diagnostic: do not flush L2 between timed steps")
    p.add_argument("--no-gather", action="store_true", help="N>1: skip the rollout all-gather (it is on by default)")
    p.add_argument("--gather-chunk", type=int, default=0, help="steps per gathered rollout chunk (default: 32, or K/2)")
    p.add_argument("--dr-pool", default=None, help="npz with a domain-randomisation parameter pool (key `pool`)")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write obs / reward / done / next_obs of the last timed step of every workload member (rank 0) "
                        "as DIR/<workload>.<task>.<array>.npy, float32")
    return p.parse_args()


def dump_outputs(out_dir, outputs):
    """outputs: {prefix: (obs, reward, done, next_obs) numpy arrays of one member}. Writes float32 .npy files; when they
    would exceed DUMP_BYTES in all, every member keeps a fixed, seeded sample of its envs, listed in <prefix>.env_index.npy."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    total = sum(x.size * 4 for arrays in outputs.values() for x in arrays)
    # a sample also writes its env indices (8 bytes per kept env), so the fraction is taken of the total including them
    frac = 1.0 if total <= DUMP_BYTES else DUMP_BYTES / (total + sum(8 * len(a[0]) for a in outputs.values()))
    for prefix, arrays in outputs.items():
        arrays = [np.asarray(x, dtype=np.float32) for x in arrays]
        n = len(arrays[0])
        if frac < 1.0:
            idx = np.sort(np.random.RandomState(0).choice(n, max(1, int(n * frac)), replace=False))
            arrays = [x[idx] for x in arrays]
            np.save(os.path.join(out_dir, prefix + ".env_index.npy"), idx.astype(np.float64))
        for name, x in zip(("obs", "reward", "done", "next_obs"), arrays):
            np.save(os.path.join(out_dir, "%s.%s.npy" % (prefix, name)), x)


# ----------------------------------------------------------------------------------------------------------------------
# host side: core accounting and the CPU arm
# ----------------------------------------------------------------------------------------------------------------------
def host_cores():
    """(threads to use, description): the affinity mask, capped by the cgroup CPU quota if there is one."""
    try:
        aff = len(os.sched_getaffinity(0))
    except Exception:
        aff = os.cpu_count() or 1
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        pass
    n = aff if quota is None else max(1, min(aff, int(quota + 0.5)))
    return n, {"affinity_cpus": aff, "cgroup_quota_cpus": quota}


_NATIVE = {}


def oracle_lib(native=True):
    """ctypes handle of the CPU restatement.  native=True: rebuilt HERE with -O3 -march=native into a temp dir (the
    portable -O2 build that travels with the repo is what the parity tests use); falls back to the portable build."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_binding
    key = "native" if native else "portable"
    if key in _NATIVE:
        return _NATIVE[key]
    so, flags = os.path.join(ROOT, "oracle", "liblocosim_ref.so"), "-O2"
    if not os.path.exists(so):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle")], stdout=subprocess.DEVNULL)
    if native:
        try:
            out = os.path.join(tempfile.mkdtemp(prefix="locosim_native_"), "liblocosim_ref_native.so")
            subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "native", "OUT=" + out],
                                  stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            so, flags = out, "-O3 -march=native"
        except Exception:
            pass
    _NATIVE[key] = (oracle_binding.load(so), flags)
    return _NATIVE[key]


def cpu_rollout(env, seconds, threads, min_steps=1024):
    """Time the CPU restatement (oracle/locosim_ref.c: same LocoEnv.step contract, same random-action law, auto-reset) on
    `threads` pinned host threads, 4 envs per thread, >= `min_steps` steps per env (>= 4096 env-steps per thread);
    returns a cpu_baseline dict.  A 1-thread run of the same length gives the per-core rate."""
    import ctypes
    import numpy as np
    from loco_mujoco_b200 import modelpack
    o, flags = oracle_lib()
    lib = o.lib
    vp, ip = ctypes.c_void_p, ctypes.c_int
    lib.ref_rollout_ex.restype = ctypes.c_long
    lib.ref_rollout_ex.argtypes = [vp, ip, vp, ip, vp, ip, vp, ip, ip, ip, ip, ctypes.c_ulonglong, vp, vp, ip, vp]
    mi, mr = [np.ascontiguousarray(x) for x in modelpack.pack(env._model)]
    ti, tr = [np.ascontiguousarray(x) for x in env.task_spec().pack()]
    P = lambda a: a.ctypes.data_as(vp)

    def run(n_envs, n_steps, nthreads, seed):
        stats = np.zeros(4)
        resets = ctypes.c_long(0)
        n = lib.ref_rollout_ex(P(mi), len(mi), P(mr), len(mr), P(ti), len(ti), P(tr), len(tr), n_envs, n_steps, nthreads,
                               seed, None, ctypes.byref(resets), 1, P(stats))
        return n, resets.value, stats

    n1, _, s1 = run(4, 256, 1, 1)                       # calibration = the single-thread rate
    rate1 = n1 / s1[0]
    steps = max(min_steps, int(rate1 * seconds / 4))
    n, resets, st = run(4 * threads, steps, threads, 2)
    value = n / st[0]
    nsub = env.task_spec().n_substeps
    return {"value": value, "unit": "env-steps/s", "cores": threads, "kind": "port",
            "effective_cores": round(st[1] / st[0], 2), "pinned_cpus": int(st[3]),
            "single_thread_env_steps_per_s": round(rate1, 1), "us_per_mj_step_per_thread": round(1e6 * st[1] / (n * nsub), 2),
            "parallel_efficiency": round(value / (rate1 * threads), 3), "build": flags,
            "sample": "%d envs x %d steps on %d pinned threads (%d env-steps per thread), %.1f s wall, %.1f CPU-s, %d resets; "
                      "fp64 C restatement of the reference loop (oracle/locosim_ref.c), NOT MuJoCo 2.3.7 itself"
                      % (4 * threads, steps, threads, 4 * steps, st[0], st[1], resets)}


def reference_importable():
    """Can the real reference loop run here?  (It needs mujoco==2.3.7 + mushroom_rl; neither is in this image.)"""
    import importlib.util
    return all(importlib.util.find_spec(m) is not None for m in ("mujoco", "mushroom_rl"))


# ----------------------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 6:
                    self.rows.append(parts)
            except Exception:
                pass
            self._stop_evt.wait(0.1)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=3)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        import statistics
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


# ----------------------------------------------------------------------------------------------------------------------
# one workload = a list of members (task, envs, kwargs) stepped together on one GPU
# ----------------------------------------------------------------------------------------------------------------------
class Workload:
    def __init__(self, name, members, rank, world, local, pools=None):
        import torch
        from loco_mujoco_b200.parallel import MixedBatch
        self.name, self.members, self.world = name, members, world
        self.dev = torch.device("cuda", local)
        per_gpu = sum(n for _, n, _ in members)
        self.batch = MixedBatch([(t + ".real", n, dict(kw, debug=True, copy_outputs=False)) for t, n, kw in members],
                                device="cuda:%d" % local, seed=0, env_id_offset=rank * per_gpu)
        self.engines = self.batch.engines
        for eng, pool in zip(self.engines, pools or [None] * len(members)):
            if pool is not None:
                eng.set_param_pool(pool)
        self.N = per_gpu
        self.torch = torch

    def counters(self):
        c = [e.counters() for e in self.engines]
        return {"resets": int(sum(x[:, 1].sum().item() for x in c)), "nonfinite": int(sum(x[:, 4].sum().item() for x in c))}

    def launches(self):
        return sum(e.launches for e in self.engines)

    def named_outputs(self, tag):
        """{"<tag>.<task>": (obs, reward, done, next_obs)} of the last step that `measure` timed."""
        return {"%s.%s" % (tag, t): o for (t, _, _), o in zip(self.members, self.last_outputs)}

    def step(self, acts, packed=None):
        if len(self.engines) == 1:
            return [self.engines[0].step(acts[0], auto_reset=True, packed=None if packed is None else packed[0])]
        return self.batch.step(acts, packed)

    def measure(self, a, rank, gather, sampler_index=None):
        """Device-resident throughput (value), optional chunked rollout all-gather, then the end-to-end leg."""
        import torch
        import torch.distributed as dist
        from loco_mujoco_b200.parallel import RolloutGather, aggregate_throughput
        torch_, dev, world = torch, self.dev, self.world
        K, W = a.steps, a.warmup
        total = PREROLL + W + K
        self.batch.reset()
        gen = torch.Generator(device=dev).manual_seed(1234 + rank)
        actions = [torch.rand((total, e.n_envs, e.action_dim), device=dev, generator=gen) * 2 - 1 for e in self.engines]
        flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
        chunk = a.gather_chunk or (32 if K >= 64 else max(1, K // 2))
        rg = [RolloutGather(e.packed_bytes, chunk, dev) for e in self.engines] if gather else None

        def barrier():
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()

        def one_step(k):
            out = self.step([x[k] for x in actions], None if rg is None else [g.slot() for g in rg])
            if rg is not None:
                for g in rg:
                    g.advance()
            return out

        for k in range(PREROLL + W):
            one_step(k)
        if rg is not None:
            for g in rg:
                g.finish()
        barrier()
        c0, l0 = self.counters(), self.launches()
        g0 = sum(g.n_gathers for g in rg) if rg is not None else 0
        sampler = ClockSampler(sampler_index) if sampler_index is not None else None
        if sampler:
            sampler.start()
        ev = lambda: torch.cuda.Event(enable_timing=True)
        t_start, t_end = ev(), ev()
        f0, f1 = [ev() for _ in range(K)], [ev() for _ in range(K)]
        s0, s1 = [ev() for _ in range(K)], [ev() for _ in range(K)]
        t_start.record()
        for k in range(K):
            f0[k].record()
            if not a.no_flush:
                flush.fill_(k & 0xff)
            f1[k].record()
            s0[k].record()
            last = one_step(PREROLL + W + k)
            s1[k].record()
        if rg is not None:
            for g in rg:
                g.finish()                      # the compute stream waits for the last chunk's gather: inside the timing
        t_end.record()
        barrier()
        clocks = sampler.stop() if sampler else None
        if a.dump_outputs:                      # per member (obs, reward, done, next_obs) of the last timed step
            self.last_outputs = [tuple(x.cpu().numpy() for x in r) for r in last]
        span = t_start.elapsed_time(t_end)
        flush_ms = sum(x.elapsed_time(y) for x, y in zip(f0, f1))
        kernel_ms = sum(x.elapsed_time(y) for x, y in zip(s0, s1))
        ms = span - flush_ms                    # everything between the first launch and the last gather, minus the L2 flushes
        t = torch.tensor([ms, kernel_ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, kernel_ms = float(t[0]), float(t[1])
        c1 = self.counters()
        res = {"value": world * self.N * K / (ms / 1e3), "ms_per_step": ms / K, "kernel_ms_per_step": kernel_ms / K,
               "gpu_launches": self.launches() - l0, "resets_in_run": c1["resets"] - c0["resets"],
               "nonfinite_in_run": c1["nonfinite"] - c0["nonfinite"], "clocks": clocks}
        if rg is not None:
            res["gather"] = {"chunk_steps": chunk, "collectives_in_run": sum(g.n_gathers for g in rg) - g0,
                             "nvlink_bytes_received_per_step_per_gpu": sum(g.bytes_received_per_chunk() for g in rg) // chunk,
                             "collective": "all_gather_into_tensor of [chunk, N, obs|reward|done] per member on a side stream, "
                                           "double buffered, overlapped with the next chunk"}
        return res

    def measure_e2e(self, a):
        """Same metric through the public LocoEnv API with HOST buffers: per step one H2D of the step's actions (pinned),
        LocoEnv.step, one D2H of (obs, reward, done) and one D2H of next_obs (the observation a host policy acts on after
        the in-kernel auto-reset), then a sync."""
        import torch
        import torch.distributed as dist
        from loco_mujoco_b200.parallel import aggregate_throughput
        dev, K = self.dev, a.steps
        envs = self.batch.envs
        gen = torch.Generator().manual_seed(4321 + int(os.environ.get("RANK", "0")))
        h_act = [(torch.rand((K, e.n_envs, e.action_dim), generator=gen) * 2 - 1).pin_memory() for e in self.engines]
        d_act = [torch.empty((e.n_envs, e.action_dim), dtype=torch.float32, device=dev) for e in self.engines]
        h_out = [torch.empty_like(e.packed_out, device="cpu").pin_memory() for e in self.engines]
        h_nxt = [torch.empty_like(e.next_obs, device="cpu").pin_memory() for e in self.engines]
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k in range(K):
            for i, env in enumerate(envs):
                d_act[i].copy_(h_act[i][k], non_blocking=True)
            if len(envs) == 1:
                envs[0].step(d_act[0])
            else:
                self.batch.step(d_act)
            for i, e in enumerate(self.engines):
                h_out[i].copy_(e.packed_out, non_blocking=True)
                h_nxt[i].copy_(e.next_obs, non_blocking=True)
            torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        e2e, _ = aggregate_throughput(self.N * K, dt, device=dev)
        return {"value": e2e, "unit": "env-steps/s",
                "h2d_bytes_per_step": sum(e.n_envs * e.action_dim * 4 for e in self.engines),
                "d2h_bytes_per_step": sum(e.packed_bytes + e.n_envs * e.obs_dim * 4 for e in self.engines)}

    def roofline(self, res, peak, which, fp32_peak):
        """HBM roofline of step_kernel: algorithmic bytes of one launch / its launch time (CUDA events around the step
        on the launching stream); per member for a mixed batch the figures are summed (the kernels overlap)."""
        algo = sum(algo_bytes(e) * e.n_envs for e in self.engines)
        dr_extra = sum(4 * e.lib.locosim_param_pool_row_len(e.h) * e.n_envs for e, (_, _, kw) in zip(self.engines, self.members)
                       if kw.get("domain_randomization_config"))
        sec = res["kernel_ms_per_step"] / 1e3
        achieved = (algo + dr_extra) / sec / 1e9
        traffic = flops = None
        if all(t.split(".")[0] in NCU for t, _, _ in self.members):
            traffic = sum(NCU[t.split(".")[0]]["dram_bytes_per_env_step"] * n for t, n, _ in self.members)
            flops = sum(NCU[t.split(".")[0]]["fp32_flops_per_env_step"] * n for t, n, _ in self.members)
        r = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
             "traffic_unit": "DRAM bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum, profiles/ncu_constants.json)",
             "peak_source": which, "algorithmic_bytes_per_launch": algo + dr_extra,
             "algorithmic_bytes_per_env_step": {t: algo_bytes(e) for (t, _, _), e in zip(self.members, self.engines)},
             "note": "compute/latency-bound by design: the state stays in shared memory across the 10 sub-steps (DESIGN.md); "
                     "the HBM fraction is low on purpose, the FP32 figure below is the relevant utilisation"}
        if flops is not None and fp32_peak:
            tf = flops / sec / 1e12
            r["fp32"] = {"achieved_tflops": tf, "peak_tflops": fp32_peak, "frac": tf / fp32_peak,
                         "peak_source": "measured (locosim_measure_fp32_peak: register-only FMA chains on all SMs)",
                         "flops_per_launch": flops}
        return r


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from loco_mujoco_b200 import LocoEnv
    env = LocoEnv.make(a.task + ".real", debug=True)
    threads, core_info = host_cores()
    # every "step" is a bounded sample of the workload; the whole run is sized to ~2.5 minutes whatever K and W are
    per_step = max(1.0, min(20.0, 150.0 / max(1, a.steps + a.warmup)))
    samples = []
    for k in range(a.warmup + a.steps):
        c = cpu_rollout(env, per_step, threads)
        if k >= a.warmup:
            samples.append(c)
    vals = sorted(s["value"] for s in samples)
    value = vals[len(vals) // 2]                          # median of the timed samples
    rep = min(samples, key=lambda s: abs(s["value"] - value))
    rep = dict(rep, value=value, host=core_info, samples_min_max=[vals[0], vals[-1]],
               real_reference_importable=reference_importable())
    cfg = workload_config(a.task, a.envs)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": a.gpus,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * a.envs / value, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg, "cpu_baseline": rep,
            "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def workload_config(task, envs):
    return {"workload": "%s random-action rollout, %d envs/GPU, 10 substeps/step, auto-reset from mini dataset" % (task, envs),
            "envs_per_gpu": envs, "task": task, "action_law": "U(-1,1)",
            "l2": "L2 flushed (256 MiB write) between timed steps, flush time subtracted (CUDA events)",
            "preroll": "%d untimed steps after the mass reset before --warmup (stationary episode ages)" % PREROLL}


def main():
    a = parse()
    if a.impl == "reference":
        return run_reference(a)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    import numpy as np
    import torch
    import torch.distributed as dist
    from loco_mujoco_b200 import engine as _engine
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, which = json.load(open(peaks_path))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, which = 6650.0, "fallback (B200_PROFILING.md)"
    fp32_peak = _engine.measure_fp32_peak(local)

    # ---- headline: BASELINE config 2 ----
    pools = [np.load(a.dr_pool)["pool"]] if a.dr_pool else None
    head = Workload(a.task, [(a.task, a.envs, {})], rank, world, local, pools)
    gather = world > 1 and not a.no_gather
    res = head.measure(a, rank, gather, sampler_index=local)
    dumps = head.named_outputs("head") if a.dump_outputs else {}
    res_nog = head.measure(a, rank, False) if gather else None
    e2e = head.measure_e2e(a)
    line = None
    if rank == 0:
        cfg = workload_config(a.task, a.envs)
        if a.dr_pool:
            cfg["domain_randomization"] = "parameter pool %s" % os.path.basename(a.dr_pool)
        line = {"metric": METRIC, "value": res["value"], "unit": "env-steps/s", "n_gpus": world, "steps": a.steps,
                "warmup": a.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg, "clocks": res["clocks"],
                "gpu_launches": res["gpu_launches"], "e2e": e2e,
                "roofline": head.roofline(res, peak, which, fp32_peak),
                "resets_in_run": res["resets_in_run"], "nonfinite_in_run": res["nonfinite_in_run"],
                "kernel_ms_per_step": res["kernel_ms_per_step"], "launch_info": head.engines[0].launch_info(),
                "physics_substeps_per_s": res["value"] * 10}
        if gather:
            line["gather"] = dict(res["gather"], value_without_gather=res_nog["value"],
                                  cost_frac=1.0 - res["value"] / res_nog["value"])
    del head
    torch.cuda.empty_cache()

    # ---- the other single-box BASELINE configs, same method, same run ----
    configs = []
    if not a.no_configs:
        dr = lambda robot: "domain_randomization_%s.yaml" % robot
        plan = [("config 3: HumanoidTorque.run, 4096 envs/GPU (reference default TargetVelocityReward(2.5); the reference has "
                 "no mocap-tracking reward, SURVEY F7)", [("HumanoidTorque.run", 4096, {})]),
                ("config 4: Atlas.walk + Talos.walk mixed batch with domain randomisation, 1024 + 1024 envs/GPU, two engines, "
                 "each spread over all SMs, launched back to back (shipped YAMLs, pre-built seeded pools: tools/build_dr_pools.py)",
                 [("Atlas.walk", 1024, {"domain_randomization_config": dr("atlas")}),
                  ("Talos.walk", 1024, {"domain_randomization_config": dr("talos")})])]
        for name, members in plan:
            wl = Workload(name, members, rank, world, local)
            r = wl.measure(a, rank, gather)
            if a.dump_outputs:
                dumps.update(wl.named_outputs(name.split(":")[0].replace(" ", "")))
            e = wl.measure_e2e(a)
            extra = {}
            if members[0][0].startswith("HumanoidTorque") and len(members) == 1:
                # the same workload without the bone-against-bone (mesh-mesh, mjc_Convex / MPR) candidate pairs: separates the
                # engine's speed from the cost of that part of the narrow phase (round 1 had no such pairs at all)
                wl2 = Workload(name, [(t, n, dict(kw, convex_collisions=False)) for t, n, kw in members], rank, world, local)
                r2 = wl2.measure(a, rank, False)
                extra = {"value_without_convex_pairs": r2["value"], "kernel_ms_per_step_without_convex_pairs": r2["kernel_ms_per_step"]}
                del wl2
                torch.cuda.empty_cache()
            if rank == 0:
                c = {"workload": name, "value": r["value"], "unit": "env-steps/s", "ms_per_step": r["ms_per_step"],
                     "kernel_ms_per_step": r["kernel_ms_per_step"], "e2e": e, "roofline": wl.roofline(r, peak, which, fp32_peak),
                     "resets_in_run": r["resets_in_run"], "nonfinite_in_run": r["nonfinite_in_run"],
                     "gpu_launches": r["gpu_launches"], "envs_per_gpu": wl.N,
                     "launch_info": [x.launch_info() for x in wl.engines]}
                if gather:
                    c["gather"] = r["gather"]
                c.update(extra)
                configs.append(c)
            del wl
            torch.cuda.empty_cache()

    if rank == 0:
        line["configs"] = configs
        if not a.no_cpu_baseline and world == 1:      # reported at N=1 only
            from loco_mujoco_b200 import LocoEnv
            threads, core_info = host_cores()
            cpu = cpu_rollout(LocoEnv.make(a.task + ".real", debug=True), a.cpu_seconds, threads)
            cpu["host"] = core_info
            cpu["real_reference_importable"] = reference_importable()
            line["cpu_baseline"] = cpu
        else:
            line["cpu_baseline"] = None
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, dumps)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
