#!/usr/bin/env python
"""bench.py -- drone-steps/s of the fused Physics.DYN control tick on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    torchrun --nproc-per-node N ... bench.py --gpus N ...      (one rank per GPU, weak scaling)

Workload (config.workload): BASELINE configs[2] -- MultiHoverAviary, 65536 drones per GPU as 32768 two-drone
aviaries, act=RPM (A=4), action buffer B=15 (obs 72 floats), 240 Hz physics / 30 Hz control (S=8 substeps per
step), random actions in [-1,1], SAME_STEP autoreset (an RL rollout).  One "step" = one env.step() = one launch of
the fused kernel over all 65536 drones of the rank.  The working set of one batch (42 MB) fits the 126 MB L2, so the
timed loop rotates over R independent batches (R x 42 MB > L2): every launch finds its inputs in HBM.

One JSON line; `value` = device-resident steps (actions already in HBM; after W warm-up steps exactly K steps are timed
in one window, the slowest rank's window counts, per-rank values alongside), `e2e` = the same
steps through the NumPy API (pinned H2D of the actions + D2H of obs/reward/flags/terminal observations inside the timed
region) with the pinned D2H copy rate measured in the same run (`pcie_frac`), `roofline` = algorithmic bytes of the step
kernel / its launch period in the timed window (`frac`, back-to-back launches overlap through programmatic dependent
launch) and / its duration alone on an idle GPU with a cold L2 (`frac_isolated`), against MEASURED_PEAKS.json;
`cpu_baseline` = the float64 NumPy oracle on a bounded sample on this host.

--dump-outputs DIR writes what the last timed step returned (rank 0) as DIR/<name>.npy: obs [E, D, 72], reward [E],
terminated / truncated / final_obs_mask [E] (as float32), and final_obs [E, D, 72], the terminal observation of every
aviary that finished in that step and zeros for the others, so every array has the same shape in every run.  Actions come
from a seeded generator and the step count is fixed by W and K, so two builds run with the same arguments can be compared
array for array.
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
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

DRONES_PER_GPU = 65536
D = 2                    # drones per aviary (learn.py DEFAULT_AGENTS)
A, B, S = 4, 15, 8       # action width, action-buffer length, substeps per control tick
OBS_DIM = 12 + A * B
# ALGORITHMIC bytes per drone-step (SURVEY.md 8d, W-RL(A=4,B=15)): state 52 r + 52 w, action 16 r, history 4*A*(B-1) r,
# obs 4*(12+B*A) w, per-aviary counter/reward/flags (4 r + 4+4+2 w) counted per drone as in the survey = 646 B
ALG_BYTES = 52 + 52 + 4 * A + 4 * A * (B - 1) + 4 + 4 * OBS_DIM + 4 + 2 + 4
METRIC = "drone-steps/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batches", type=int, default=8, help="independent 65536-drone batches rotated through (L2 defeat)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


def bind_to_gpu_numa(local):
    """Pins this process to the cores next to its GPU (sysfs local_cpulist of the PCI device) BEFORE any pinned memory is
    allocated, so the staging buffers are first-touched on the GPU's NUMA node.  Returns a short description or None."""
    try:
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[local]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else local
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,pci.bus_id", "--format=csv,noheader"], capture_output=True, text=True, timeout=20).stdout
        bus = None
        for line in out.strip().splitlines():
            i, b = [c.strip() for c in line.split(",")]
            if int(i) == phys:
                bus = b
        if bus is None:
            return None
        dom, rest = bus.split(":", 1)
        path = "/sys/bus/pci/devices/%s:%s/local_cpulist" % (dom[-4:].lower(), rest.lower())
        cpus = set()
        for part in open(path).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return "gpu %d (%s) -> %d cores %s" % (phys, bus, len(cpus), open(path).read().strip())
    except Exception:
        return None


# ---------------------------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md recipe)
# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------
# CPU legs: the float64 NumPy oracle (port of the reference's DYN path), never the product
# ---------------------------------------------------------------------------------------------------------------
def _oracle_worker(args):
    n_envs, steps, seed = args
    import numpy as np
    from oracle.dyn_oracle import OracleAviary
    env = OracleAviary("multihover", n_envs, D, act="rpm")
    env.reset()
    rng = np.random.default_rng(seed)
    acts = rng.uniform(-1, 1, (steps, n_envs, D, A)).astype(np.float32)
    t0 = time.perf_counter()
    for t in range(steps):
        obs, rew, term, trunc = env.step(acts[t])
        done = term | trunc
        if done.any():
            env.reset(mask=done)
    return time.perf_counter() - t0


def cpu_baseline_single(n_envs=2048, steps=1000):
    """Bounded sample on one core: 4096 drones x `steps` control ticks of the same workload."""
    dt = _oracle_worker((n_envs, steps, 0))
    return {"value": n_envs * D * steps / dt, "unit": METRIC, "cores": 1, "kind": "port",
            "sample": "%d drones x %d steps (S=%d) of the bench workload, float64 NumPy oracle, %.1f s" % (n_envs * D, steps, S, dt)}


def reference_arm(a):
    """--impl reference: the reference's CPU implementation of the path.  The reference is pure Python and cannot travel
    to the GPU box, so this is the oracle port (batched float64 NumPy restatement pinned to the reference by
    tests/golden), fanned out over every host core; each step is a bounded sample of the workload."""
    import multiprocessing as mp
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    per_proc_envs = 2048                      # 4096 drones per process per step
    steps, warm = max(1, min(a.steps, 500)), max(1, min(a.warmup, 5))
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        pool.map(_oracle_worker, [(per_proc_envs, warm, 100 + i) for i in range(cores)])
        t0 = time.perf_counter()
        pool.map(_oracle_worker, [(per_proc_envs, steps, i) for i in range(cores)])
        wall = time.perf_counter() - t0
    drones = per_proc_envs * D * cores
    val = drones * steps / wall
    sample = "%d processes x %d drones x %d steps (S=%d), float64 NumPy oracle port" % (cores, per_proc_envs * D, steps, S)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": METRIC, "n_gpus": a.gpus, "steps": steps, "warmup": warm,
        "ms_per_step": 1e3 * wall / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(a, drones),
        "cpu_baseline": {"value": val, "unit": METRIC, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": METRIC, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def step_outputs(result):
    """Device copies of what one vector-API step returned, taken before later steps reuse its buffers."""
    import torch
    obs, rew, term, trunc, info = result
    out = {"obs": obs.clone(), "reward": rew.clone(), "terminated": term.clone(), "truncated": trunc.clone()}
    if "final_obs" in info:
        mask = info["_final_obs"]
        out["final_obs_mask"], out["final_obs"] = mask.clone(), torch.where(mask[:, None, None], info["final_obs"], 0.0)
    return out


def dump_outputs(directory, outputs):
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, t in outputs.items():
        x = t.cpu().numpy()
        np.save(os.path.join(directory, name + ".npy"), x if x.dtype in (np.float32, np.float64) else x.astype(np.float32))


def workload_config(a, drones_per_step):
    return {"workload": "MultiHoverAviary x %d aviaries x %d drones (=%d drones per GPU), act=RPM (A=4), action buffer B=15, obs 72 f32, "
                        "pyb 240 Hz / ctrl 30 Hz (S=8), random actions, SAME_STEP autoreset [BASELINE configs[2]]" % (DRONES_PER_GPU // D, D, DRONES_PER_GPU),
            "drones_per_gpu": DRONES_PER_GPU, "drones_per_step": drones_per_step, "substeps_per_step": S, "obs_dim": OBS_DIM,
            "parallelism": "env-sharded x%d (no collective on the step path)" % a.gpus,
            "l2": "%d rotating independent batches x 42 MB > 126 MB L2 (no flush kernel in the timed region)" % a.batches}


# ---------------------------------------------------------------------------------------------------------------
def main():
    a = parse()
    if a.impl == "reference":
        reference_arm(a)
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    numa = bind_to_gpu_numa(local)
    import numpy as np
    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL may print its version banner on stdout when the first communicator is created: keep stdout for the one
        # JSON line by pointing fd 1 at stderr while the process group comes up
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            warm = torch.zeros(1, device=dev)
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    from gym_pybullet_drones_b200.envs import MultiHoverAviary
    from gym_pybullet_drones_b200.utils.enums import ActionType, Physics

    E = DRONES_PER_GPU // D
    R = a.batches
    envs = [MultiHoverAviary(num_drones=D, physics=Physics.DYN, act=ActionType.RPM, num_envs=E, device=dev,
                             autoreset="same_step", host_copy=False) for _ in range(R)]
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    # uniform[-1, 1) actions, a fresh draw every step: K_ACT action tensors per batch, cycled (8 x 16 x 1 MB)
    K_ACT = 16
    acts = [[torch.rand((E, D, A), device=dev, generator=gen) * 2 - 1 for _ in range(K_ACT)] for _ in range(R)]
    for e in envs:
        e.reset()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def all_max(x):
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_gather_f(x):
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        if world == 1:
            return [float(x)]
        out = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(out, t)
        return [float(o.item()) for o in out]

    def run(n, k0=0):
        res = None
        for k in range(k0, k0 + n):
            i = k % R
            res = envs[i].step(acts[i][(k // R) % K_ACT])
        return res

    # ---- device-resident throughput: one window of exactly K steps, barrier + sync on both sides, max over ranks ----
    run(max(a.warmup, 3))
    k0 = a.warmup
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        barrier()
        ev0.record()
        last = run(a.steps, k0)
        ev1.record()
        barrier()
        my_ms = ev0.elapsed_time(ev1)
        outputs = step_outputs(last) if a.dump_outputs and rank == 0 else None
        k0 += a.steps
        # keep the sampler over a little more load so short runs still see clocks under load
        t_end = time.time() + 0.6
        while time.time() < t_end:
            run(50)
        torch.cuda.synchronize()
    ms_window = all_max(my_ms)
    value = DRONES_PER_GPU * world * a.steps / (ms_window * 1e-3)
    per_rank = all_gather_f(DRONES_PER_GPU * a.steps / (my_ms * 1e-3))

    # ---- roofline of the step kernel: launch period in the timed loop (pipelined) and duration alone (isolated, cold L2) ----
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
    kern_ms = my_ms / a.steps                                 # back-to-back launches of only this kernel: launch period
    scrub = torch.empty(192 << 20, dtype=torch.uint8, device=dev)
    iso = []
    for k in range(40):
        scrub.fill_(k & 255)                                  # evict the 126 MB L2
        torch.cuda.synchronize()
        ev0.record()
        envs[k % R].step(acts[k % R][k % K_ACT])
        ev1.record()
        torch.cuda.synchronize()
        iso.append(ev0.elapsed_time(ev1))
    del scrub
    iso_ms = statistics.median(iso)
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "r02_step_traffic.json")))["dram_bytes_per_launch"]
    except Exception:
        pass
    alg = ALG_BYTES * DRONES_PER_GPU
    roofline = {"bound": "hbm", "achieved": alg / (kern_ms * 1e-3) / 1e9, "peak": peak_gbs, "unit": "GB/s",
                "frac": alg / (kern_ms * 1e-3) / 1e9 / peak_gbs, "frac_isolated": alg / (iso_ms * 1e-3) / 1e9 / peak_gbs,
                "traffic": traffic, "kernel": "step_fast_kernel<A=4,task,reset,rpy_f32>", "kernel_ms": kern_ms, "kernel_ms_isolated": iso_ms,
                "alg_bytes_per_drone_step": ALG_BYTES, "alg_bytes_per_launch": alg,
                "timing": "frac: CUDA events around the %d back-to-back launches of the timed window / count (launch period; neighbours overlap "
                          "through programmatic dependent launch); frac_isolated: median of events around single launches after a sync and a "
                          "192 MB L2 scrub (includes ~2 us of event/launch gap); traffic: ncu dram__bytes_read+write per launch (profiles/)" % a.steps,
                "peak_source": "MEASURED_PEAKS.json (of measured)" if peaks else "fallback 6.65 TB/s (of fallback)"}

    # ---- end to end through the NumPy API: page-locked ndarray actions in, ndarrays out, every copy inside step() ----
    h_acts = []
    for xs in acts:
        row = []
        for x in xs:
            t = torch.empty(x.shape, dtype=torch.float32).pin_memory()
            t.copy_(x)
            row.append(t.numpy())
        h_acts.append(row)
    e2e_steps = max(10, min(a.steps, 200))
    for k in range(5):
        envs[k % R].step(h_acts[k % R][k % K_ACT])
    barrier()
    n_fin_tot = 0
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        i = k % R
        obs, rew, term, trunc, info = envs[i].step(h_acts[i][(k // R) % K_ACT])
        n_fin_tot += info["final_obs"].shape[0] if "final_obs" in info else 0
    barrier()
    e2e_s = all_max(time.perf_counter() - t0)
    e2e_val = DRONES_PER_GPU * world * e2e_steps / e2e_s
    n_fin = n_fin_tot / e2e_steps
    h2d = DRONES_PER_GPU * A * 4
    d2h = int(DRONES_PER_GPU * OBS_DIM * 4 + E * (4 + 1 + 1 + 1) + n_fin * (D * OBS_DIM * 4 + 8) + 4)
    # the link itself, same process, same pinned memory: one 19 MB device -> pinned host copy, repeated
    hbuf = torch.empty((DRONES_PER_GPU, OBS_DIM), dtype=torch.float32).pin_memory()
    dbuf = envs[0]._obs_buf[0]
    for _ in range(3):
        hbuf.copy_(dbuf, non_blocking=True)
    barrier()
    t0 = time.perf_counter()
    for _ in range(20):
        hbuf.copy_(dbuf, non_blocking=True)
    torch.cuda.synchronize()
    pcie_gbs = 20 * hbuf.numel() * 4 / (time.perf_counter() - t0) / 1e9
    e2e_gbs = (h2d + d2h) * e2e_steps / (e2e_s) / 1e9 if world == 1 else (h2d + d2h) / (DRONES_PER_GPU / (e2e_val / world)) / 1e9
    e2e = {"value": e2e_val, "unit": METRIC, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
           "ms_per_step": 1e3 * e2e_s / e2e_steps, "d2h_gbs": d2h / (e2e_s / e2e_steps) / 1e9, "pcie_d2h_gbs_measured": pcie_gbs,
           "pcie_frac": d2h / (e2e_s / e2e_steps) / 1e9 / pcie_gbs, "terminal_obs_aviaries_per_step": n_fin, "numa_binding": numa,
           "api": "MultiHoverAviary.step(page-locked ndarray) -> ndarrays (qs_step_host: H2D actions, tick, device-side compaction of the "
                  "finished aviaries, D2H obs/reward/flags + their terminal observations; the batch is cut into chunks of whole warps whose "
                  "observation copies run under the next chunk's H2D + tick; host_copy=False)"}
    del hbuf
    # the same loop with the chunk count of qs_step_host's H2D -> tick -> D2H pipeline forced (QS_HOST_CHUNKS is read per call;
    # 1 = one copy up, one launch, one copy down); the headline above is the library default
    try:
        sweep = {}
        old_env = os.environ.get("QS_HOST_CHUNKS")
        n_sw = max(10, min(a.steps, 100))
        for c in (1, 2, 4, 8):
            os.environ["QS_HOST_CHUNKS"] = str(c)
            for k in range(4):
                envs[k % R].step(h_acts[k % R][k % K_ACT])
            barrier()
            t0 = time.perf_counter()
            for k in range(n_sw):
                envs[k % R].step(h_acts[k % R][(k // R) % K_ACT])
            barrier()
            sw = all_max(time.perf_counter() - t0)
            sweep[str(c)] = {"ms_per_step": 1e3 * sw / n_sw, "value": DRONES_PER_GPU * world * n_sw / sw}
        if old_env is None:
            del os.environ["QS_HOST_CHUNKS"]
        else:
            os.environ["QS_HOST_CHUNKS"] = old_env
        e2e["host_chunks_sweep"] = sweep
    except Exception as ex:  # noqa: BLE001
        e2e["host_chunks_sweep"] = {"error": repr(ex)}
    # the same loop with host_obs="head": only the 12-float kinematic head of every observation crosses PCIe (the rest of a KIN
    # observation is the action history the caller supplied itself) -- reported next to the headline e2e, never instead of it
    try:
        henv = [MultiHoverAviary(num_drones=D, physics=Physics.DYN, act=ActionType.RPM, num_envs=E, device=dev, autoreset="same_step",
                                 host_copy=False, host_obs="head") for _ in range(2)]
        for e in henv:
            e.reset()
        for k in range(4):
            henv[k & 1].step(h_acts[k % R][k % K_ACT])
        barrier()
        t0 = time.perf_counter()
        for k in range(e2e_steps):
            henv[k & 1].step(h_acts[k % R][(k // R) % K_ACT])
        barrier()
        hs = all_max(time.perf_counter() - t0)
        e2e["head_only_mode"] = {"value": DRONES_PER_GPU * world * e2e_steps / hs, "ms_per_step": 1e3 * hs / e2e_steps,
                                 "d2h_bytes_per_step_obs": DRONES_PER_GPU * 12 * 4,
                                 "note": "extra: MultiHoverAviary(host_obs='head').step(ndarray) returns [E, D, 12] heads; terminal observations still travel in full"}
        del henv
    except Exception as ex:  # pragma: no cover
        e2e["head_only_mode"] = {"error": repr(ex)}

    extras = {} if a.no_extras else run_extras(a, envs, acts, gen, dev, world, R, peak_gbs, barrier)

    if rank == 0:
        out = {
            "metric": METRIC, "value": value, "unit": METRIC, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms_window / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(a, DRONES_PER_GPU * world),
            "clocks": clk.summary(),
            "e2e": e2e,
            "gpu_launches": a.steps,
            "per_rank_value": per_rank,
            "roofline": roofline,
            "substeps_per_s": value * S,
            "state_storage": "f64 planes (pos, quat, vel, body rates), f32 observations/actions; arithmetic f64",
            "extras": extras,
        }
        if world == 1 and not a.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline_single()
        print(json.dumps(out))
    if outputs is not None:
        dump_outputs(a.dump_outputs, outputs)
    if world > 1:
        dist.destroy_process_group()


def run_extras(a, envs, acts, gen, dev, world, R, peak_gbs, barrier):
    """Reported next to the headline, never instead of it."""
    import torch
    from gym_pybullet_drones_b200.envs import HoverAviary, MultiHoverAviary
    from gym_pybullet_drones_b200.utils.enums import ActionType, Physics
    extras = {}

    def timed(fn, n, reps=3):
        best = 1e30
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            fn(n)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1) / n)
        return best

    K_ACT = len(acts[0])

    def run(n):
        for k in range(n):
            envs[k % R].step(acts[k % R][(k // R) % K_ACT])

    try:   # the same launches replayed from a CUDA graph: no per-step host work
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            run(2 * R)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        with torch.cuda.graph(g):
            run(2 * R)                      # two ticks per batch: the obs double buffers end where they started
        for _ in range(3):
            g.replay()
        gms = timed(lambda n: [g.replay() for _ in range(n)], 40) / (2 * R)
        extras["cuda_graph_replay"] = {"ms_per_step": gms, "value": DRONES_PER_GPU * world / (gms * 1e-3), "unit": METRIC,
                                       "hbm_frac": ALG_BYTES * DRONES_PER_GPU / (gms * 1e-3) / 1e9 / peak_gbs}
    except Exception as ex:  # pragma: no cover
        extras["cuda_graph_replay"] = {"error": repr(ex)}
        torch.cuda.synchronize()
    # the same kernel at sizes where several waves overlap load, compute and store (working set > L2)
    sweep = {}
    if world == 1:
        for n in (262144, 1048576):
            try:
                big = [MultiHoverAviary(num_drones=D, physics=Physics.DYN, act=ActionType.RPM, num_envs=n // D, device=dev, autoreset="same_step") for _ in range(2)]
                ba = torch.rand((n // D, D, A), device=dev, generator=gen) * 2 - 1
                for b in big:
                    b.reset()
                bms = timed(lambda m: [big[k & 1].step(ba) for k in range(m)], 60)
                sweep[str(n)] = {"ms_per_step": bms, "value": n / (bms * 1e-3), "hbm_frac": ALG_BYTES * n / (bms * 1e-3) / 1e9 / peak_gbs}
                del big, ba
            except Exception as ex:  # pragma: no cover
                sweep[str(n)] = {"error": repr(ex)}
        extras["drones_per_launch_sweep"] = sweep
    # learn.py's default action type: ONE_D_RPM (A=1, obs 27 floats): 286 algorithmic bytes per drone-step
    try:
        e1 = [MultiHoverAviary(num_drones=D, physics=Physics.DYN, act=ActionType.ONE_D_RPM, num_envs=DRONES_PER_GPU // D, device=dev, autoreset="same_step") for _ in range(R)]
        a1 = [torch.rand((DRONES_PER_GPU // D, D, 1), device=dev, generator=gen) * 2 - 1 for _ in range(R)]
        for e in e1:
            e.reset()
        ms1 = timed(lambda m: [e1[k % R].step(a1[k % R]) for k in range(m)], 400)
        alg1 = 52 + 52 + 4 + 4 * 14 + 4 + 4 * 27 + 4 + 2 + 4
        extras["one_d_rpm_65536"] = {"ms_per_step": ms1, "value": DRONES_PER_GPU / (ms1 * 1e-3), "alg_bytes_per_drone_step": alg1,
                                     "hbm_frac": alg1 * DRONES_PER_GPU / (ms1 * 1e-3) / 1e9 / peak_gbs}
        del e1, a1
    except Exception as ex:  # pragma: no cover
        extras["one_d_rpm_65536"] = {"error": repr(ex)}
    # two of the rotating batches in flight at once (even batches on one stream, odd ones on another)
    try:
        if R % 2 == 0:
            s_even, s_odd = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
            cur = torch.cuda.current_stream(dev)

            def run2(n):
                s_even.wait_stream(cur)
                s_odd.wait_stream(cur)
                for k in range(n):
                    i = k % R
                    with torch.cuda.stream(s_even if (i & 1) == 0 else s_odd):
                        envs[i].step(acts[i][(k // R) % K_ACT])
                cur.wait_stream(s_even)
                cur.wait_stream(s_odd)

            run2(64)
            ms2 = timed(run2, 400)
            extras["two_batches_in_flight"] = {"ms_per_step": ms2, "value": DRONES_PER_GPU * world / (ms2 * 1e-3), "unit": METRIC,
                                               "hbm_frac": ALG_BYTES * DRONES_PER_GPU / (ms2 * 1e-3) / 1e9 / peak_gbs,
                                               "note": "same launches, even/odd batches on two streams (rank-local)"}
    except Exception as ex:  # pragma: no cover
        extras["two_batches_in_flight"] = {"error": repr(ex)}
        torch.cuda.synchronize()
    # fused multi-tick rollout (qs_rollout): T ticks per launch, device-generated uniform actions, obs written as [T,N,72]
    try:
        T = 32
        ro = None
        for k in range(3):
            ro = envs[0].rollout(num_steps=T, seed=7, out=ro)
        hold = [ro]

        def roll(n):
            for k in range(n):
                hold[0] = envs[k % R].rollout(num_steps=T, seed=7, out=hold[0])

        rms = timed(roll, 20) / T
        extras["fused_rollout_T32"] = {"ms_per_step": rms, "value": DRONES_PER_GPU * world / (rms * 1e-3), "unit": METRIC,
                                       "hbm_frac_algorithmic": ALG_BYTES * DRONES_PER_GPU / (rms * 1e-3) / 1e9 / peak_gbs,
                                       "note": "qs_rollout: 32 control ticks per launch, state in registers, history in a sliding shared-memory window; "
                                               "per tick only the obs rows/reward/flags are written (the 646 B algorithmic figure counts traffic the fusion removes)"}
        del ro, hold
    except Exception as ex:  # pragma: no cover
        extras["fused_rollout_T32"] = {"error": repr(ex)}
    # policy + env in ONE launch: the SB3-MlpPolicy-shaped actor (+ critic) evaluated inside qs_rollout every tick
    try:
        from gym_pybullet_drones_b200.policy import MlpPolicy
        T = 16
        for name, critic in (("actor_only", False), ("actor_critic", True)):
            pol = MlpPolicy.random(D * OBS_DIM, D * A, seed=3, critic=critic, device=dev)
            noise = torch.randn((T, DRONES_PER_GPU // D, D * A), device=dev, generator=gen)
            hold = [envs[0].rollout(policy=pol, noise=noise)]

            def prol(n):
                for k in range(n):
                    hold[0] = envs[k % R].rollout(policy=pol, noise=noise, out=hold[0])

            pms = timed(prol, 10) / T
            macs = (D * OBS_DIM * 64 + 64 * 64 + 64 * D * A) + ((D * OBS_DIM * 64 + 64 * 64 + 64) if critic else 0)
            extras["policy_rollout_" + name] = {"ms_per_tick": pms, "value": DRONES_PER_GPU * world / (pms * 1e-3), "unit": METRIC,
                                                 "mlp_gflop_per_tick_fp32_equiv": 2e-9 * macs * (DRONES_PER_GPU // D), "mlp_tflops_fp32_equiv": 2 * macs * (DRONES_PER_GPU // D) / (pms * 1e-3) / 1e12,
                                                 "note": "qs_rollout(policy=MlpPolicy %d-64-64-%d%s): evaluated inside the rollout kernel on the tensor cores (mma.sync m16n8k16 F16, two-term operand split = fp32-level accuracy, 3 mma per fp32-equivalent block), T=%d ticks per launch" % (D * OBS_DIM, D * A, " + critic" if critic else "", T)}
            del hold, noise, pol
    except Exception as ex:  # pragma: no cover
        extras["policy_rollout"] = {"error": repr(ex)}
        torch.cuda.synchronize()
    # BASELINE configs[1]: 4096 x HoverAviary with the embedded DSLPIDControl (act=PID): per-launch (launch-latency bound) and
    # through the fused rollout, where the launch cost is paid once per 32 ticks
    try:
        pe = HoverAviary(physics=Physics.DYN, act=ActionType.PID, num_envs=4096, device=dev, autoreset="same_step")
        pa = torch.rand((4096, 1, 3), device=dev, generator=gen) * torch.tensor([1.0, 1.0, 1.0], device=dev) + torch.tensor([-0.5, -0.5, 0.5], device=dev)
        pe.reset()
        msp = timed(lambda m: [pe.step(pa) for _ in range(m)], 400)
        pacts = pa.unsqueeze(0).expand(32, -1, -1, -1).contiguous()
        ro = pe.rollout(pacts)
        hold = [ro]

        def proll(n):
            for _ in range(n):
                hold[0] = pe.rollout(pacts, out=hold[0])

        msr = timed(proll, 20) / 32
        algp = 598
        extras["config2_hover_pid_4096"] = {"per_launch_ms": msp, "per_launch_value": 4096 / (msp * 1e-3),
                                            "rollout_T32_ms_per_tick": msr, "rollout_value": 4096 / (msr * 1e-3),
                                            "alg_bytes_per_drone_step": algp, "rollout_hbm_frac": algp * 4096 / (msr * 1e-3) / 1e9 / peak_gbs,
                                            "note": "2.4 MB per tick: launch-latency bound, not a bandwidth number"}
        del pe, ro, hold
    except Exception as ex:  # pragma: no cover
        extras["config2_hover_pid_4096"] = {"error": repr(ex)}
    tiny = MultiHoverAviary(num_drones=D, physics=Physics.DYN, act=ActionType.RPM, num_envs=64, device=dev, autoreset="same_step")
    ta = torch.zeros((64, D, A), device=dev)
    tiny.reset()
    for _ in range(200):
        tiny.step(ta)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(2000):
        tiny.step(ta)
    torch.cuda.synchronize()
    extras["host_us_per_step_call"] = (time.perf_counter() - t0) / 2000 * 1e6
    return extras


if __name__ == "__main__":
    main()
