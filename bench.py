#!/usr/bin/env python
"""bench.py — differentiable world-steps/s (fwd+bwd) of the batched Atlas timestep.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B] [--dump-outputs DIR]
  torchrun --nproc-per-node N bench.py --gpus N ...         (one rank per GPU; batch shards, no data-path collective)

--dump-outputs DIR writes what the last timed step returned to a caller of the headline path (next state, gradient w.r.t. the state,
gradient w.r.t. the action; rank 0's shard) as DIR/<name>.npy, float32.  The inputs are seeded, so two builds can be compared output for
output.  Above 64 MB in all, a fixed seeded sample of worlds (rows) is written instead.

Headline workload (BASELINE.json configs[1]): Atlas humanoid (33 DoF, 28 moving bodies), contact-free, batch 4096 per GPU,
one step = forward kernel + backward kernel over the whole batch, synthetic seeded inputs.
`extra.legs` (every world size; each with its own value / roofline / e2e): configs[2] half-cheetah + ground (4096/GPU), configs[3]
Atlas + ground contact (8192/GPU), configs[4] 64-step Atlas + ground rollout with backprop through the horizon (1024/GPU, the
scalar loss all-reduced over NCCL).  Contact legs step FRESH states: x_{t+1} is the engine's own x_t -> step, LCP cache flowing.
`value`   : worlds*steps / device time, inputs resident in HBM (rotating buffer sets larger than L2).
`e2e`     : same metric through the C-ABI host entry points (host buffers, H2D/D2H inside the timed region).
`roofline`: HBM roofline of the dominant kernel from the algorithmic bytes of SURVEY §8(d) (see DESIGN.md).
`cpu_baseline`: the fp64 oracle port timed on this box's host cores on a bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ATLAS = os.path.join(ROOT, "tests", "golden", "models", "atlas.json")
METRIC = "differentiable world-steps/sec (fwd+bwd), batched Atlas"
UNIT = "world-steps/s"


def make_inputs(raw, B, seed):
    """SURVEY §8(d) config 2: root rot ~N(0,0.1), root pos ~U(-0.1,0.1), joints ~U(-pi/8,pi/8), qdot ~U(-pi/4,pi/4),
    tau = 0 on the root, U(-50,50) elsewhere."""
    rng = np.random.default_rng(seed)
    n, na = raw.ndof, len(raw.action_map)
    q = rng.uniform(-np.pi / 8, np.pi / 8, (B, n))
    q[:, 0:3] = rng.normal(0, 0.1, (B, 3))
    q[:, 3:6] = rng.uniform(-0.1, 0.1, (B, 3))
    q = np.clip(q, np.maximum(raw.pos_lo, -10), np.minimum(raw.pos_hi, 10))
    v = rng.uniform(-np.pi / 4, np.pi / 4, (B, n))
    tau = rng.uniform(-50, 50, (B, n))
    tau[:, :6] = 0.0
    a = tau[:, raw.action_map]
    g = rng.normal(size=(B, 2 * n))
    return (np.concatenate([q, v], 1).astype(np.float32), a.astype(np.float32), g.astype(np.float32))


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.rows = []
        self.stop_flag = False
        self.gpu = gpu_index
        self.proc = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
                if self.stop_flag:
                    break
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc:
            try:
                self.proc.terminate()
            except Exception:
                pass
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for k, nm in enumerate(names):
                    if r[2 + k].lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


_CPU_STATE = {}


def _cpu_worker_init(raw_json):
    from oracle.binding import OracleWorld
    import nimblephysics_b200 as nb

    raw = nb.RawModel.from_json(raw_json)
    _CPU_STATE["raw"] = raw
    _CPU_STATE["ow"] = OracleWorld(raw)  # one World per worker, like MultiShot.cpp:66-70


def _cpu_worker_run(job):
    seed, lo, hi, total = job
    raw, ow = _CPU_STATE["raw"], _CPU_STATE["ow"]
    s, a, g = make_inputs(raw, total, seed)
    s64, a64, g64 = s.astype(np.float64), a.astype(np.float64), g.astype(np.float64)
    t0 = time.perf_counter()
    for w in range(lo, hi):
        ow.step(s64[w], a64[w])
        ow.backprop(s64[w], a64[w], g64[w])
    return time.perf_counter() - t0



def bind_to_gpu_numa(local_rank):
    """Pin this rank (and therefore the first-touch placement of its pinned host buffers) to the NUMA node its GPU hangs off:
    the e2e path streams host memory over PCIe, and 8 unpinned ranks on a 2-socket box cross the inter-socket link."""
    try:
        out = subprocess.run(["nvidia-smi", f"--id={local_rank}", "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=10).stdout.strip()
        bdf = out.lower()
        if bdf.count(":") == 2 and len(bdf.split(":")[0]) == 8:
            bdf = bdf[4:]  # 00000000:17:00.0 -> 0000:17:00.0
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        if node < 0:
            return None
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus += list(range(int(lo), int(hi or lo) + 1))
        os.sched_setaffinity(0, set(cpus))
        return {"numa_node": node, "cpus": len(cpus)}
    except Exception:
        return None


def probe_reference():
    """BASELINE.md §3 step 1: is the real reference importable (a driver-provided install under baseline/_ref/ or site-packages)?
    Returns the module or None.  It cannot be built in the authoring container (needs Eigen, ccd, assimp, boost, ...)."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if os.path.isdir(ref_dir) and ref_dir not in sys.path:
        sys.path.insert(0, ref_dir)
    try:
        import nimblephysics  # noqa: F401

        return nimblephysics
    except Exception:
        return None


def time_real_reference(nimble, seconds=3.0):
    """forwardPass + backpropState of the real reference on Atlas (python/nimblephysics_benchmarks/atlas_bench.py:12-27), one
    process; returns world-steps/s or None when its data files are missing."""
    try:
        world = nimble.simulation.World()
        world.setGravity([0, -9.81, 0])
        base = os.path.dirname(nimble.__file__)
        atlas = world.loadSkeleton(os.path.join(base, "models", "atlas", "atlas_v3_no_head.urdf"))
        world.setTimeStep(1e-3)
        n = world.getNumDofs()
        rng = np.random.default_rng(0)
        g = rng.normal(size=2 * n)
        t0 = time.perf_counter(); k = 0
        while time.perf_counter() - t0 < seconds:
            world.setPositions(rng.uniform(-0.3, 0.3, n)); world.setVelocities(rng.uniform(-1, 1, n))
            snap = nimble.neural.forwardPass(world)
            lw = nimble.neural.LossGradient(); lw.lossWrtPosition = g[:n]; lw.lossWrtVelocity = g[n:]
            out = nimble.neural.LossGradient()
            snap.backprop(world, out, lw)
            k += 1
        return k / (time.perf_counter() - t0)
    except Exception:
        return None

def _cpu_worker_init_contact(raw_json, name):
    from oracle.binding import OracleContactWorld
    import nimblephysics_b200 as nb

    raw = nb.RawModel.from_json(raw_json)
    _CPU_STATE["craw"], _CPU_STATE["cname"] = raw, name
    _CPU_STATE["cow"] = OracleContactWorld(raw)


def _cpu_worker_run_contact(job):
    from tests.util import contact_inputs

    seed, lo, hi, total = job
    raw, ow, name = _CPU_STATE["craw"], _CPU_STATE["cow"], _CPU_STATE["cname"]
    s, a = contact_inputs(raw, name, total, seed=seed)
    g = np.random.default_rng(seed).normal(size=s.shape)
    t0 = time.perf_counter()
    for w in range(lo, hi):
        ow.step_contact(s[w].astype(np.float64), a[w].astype(np.float64))
        ow.backprop_contact(s[w].astype(np.float64), a[w].astype(np.float64), g[w])
    return time.perf_counter() - t0


def cpu_contact_baseline(raw, name, procs, n_worlds):
    """fp64 oracle port (step with the contact stage + backprop) on `procs` host processes -> world-steps/s"""
    import multiprocessing as mp

    pool = mp.get_context("fork").Pool(procs, initializer=_cpu_worker_init_contact, initargs=(raw.to_json(), name))
    per = (n_worlds + procs - 1) // procs
    jobs = [(77, k * per, min(n_worlds, (k + 1) * per), n_worlds) for k in range(procs) if k * per < n_worlds]
    pool.map(_cpu_worker_run_contact, jobs[: max(1, len(jobs) // 4)])  # warm-up
    busy = pool.map(_cpu_worker_run_contact, jobs)
    pool.close(); pool.join()
    return n_worlds / (sum(busy) / len(busy)) if busy else None


class CpuReference:
    """Times the fp64 oracle (forward + backprop per world) on `procs` host processes (one World each)."""

    def __init__(self, raw, procs):
        import multiprocessing as mp

        self.procs = procs
        self.pool = mp.get_context("fork").Pool(procs, initializer=_cpu_worker_init, initargs=(raw.to_json(),))
        self.run(procs * 2)  # warm-up: library load, page faults

    def run(self, n_worlds, seed=1234):
        per = (n_worlds + self.procs - 1) // self.procs
        jobs = [(seed, k * per, min(n_worlds, (k + 1) * per), n_worlds) for k in range(self.procs)]
        t0 = time.perf_counter()
        busy = self.pool.map(_cpu_worker_run, jobs)
        wall = time.perf_counter() - t0
        # throughput of the pool = worlds / (sum of busy time / processes): the mean load per core.  (max(busy) measured the one
        # straggler a fork()ed pool of 128 always has and moved 6x between boxes; the wall clock includes input synthesis.)
        dt = sum(busy) / max(len(busy), 1)
        return n_worlds / dt, dt, wall

    def close(self):
        self.pool.close()
        self.pool.join()



ALG_BYTES = {"atlas_ground": 4 * (10 * 33 + 3 * 33) + 12 * 24, "half_cheetah": 4 * (10 * 9 + 3 * 9) + 12 * 12}  # SURVEY §8(d): 52 n + 12 m_max


def contact_leg(nb, torch, name, B, K, W, dev, dist, rank, world_size, peak, cpu_rate):
    """fwd+bwd world-steps/s of a model with the contact / boxed-LCP stage, stepping FRESH states: x_{t+1} = step(x_t) with the LCP
    cache flowing, every step back-propagated with a random upstream gradient (configs[2] / configs[3])."""
    from nimblephysics_b200 import _cabi
    from tests.util import contact_inputs

    raw = nb.RawModel.load(os.path.join(ROOT, "tests", "golden", "models", f"{name}.json"))
    world = nb.World.from_raw(raw)
    s, a = contact_inputs(raw, name, B, seed=7 + rank)
    x0 = torch.tensor(s, device=dev); at = torch.tensor(a, device=dev); g = torch.randn(B, 2 * raw.ndof, device=dev)
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def barrier():
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    fwd_ms, bwd_ms = [], []

    def step(x, timed):
        xi = x.detach().requires_grad_(True); ai = at.detach().requires_grad_(True)
        if timed:
            e0, e1, e2 = ev(), ev(), ev(); e0.record()
        out = nb.timestep(world, xi, ai)
        if timed:
            e1.record()
        out.backward(g)
        if timed:
            e2.record(); fwd_ms.append((e0, e1)); bwd_ms.append((e1, e2))
        return out.detach()

    nb.reset_contact_cache(world)
    x = x0
    for _ in range(W):
        x = step(x, False)
    barrier()
    l0 = _cabi.lib().nb2_launch_count()
    t0, t1 = ev(), ev()
    t0.record()
    for _ in range(K):
        x = step(x, True)
    t1.record()
    barrier()
    ms = t0.elapsed_time(t1)
    launches = _cabi.lib().nb2_launch_count() - l0
    c = world._lcp_cache
    st, mm = c["status"], c["m"]
    frac = lambda bit: float(((st & bit) > 0).float().mean())
    stats = {"mean_lcp_rows": float(mm.float().mean()), "frac_shortcircuit": frac(1), "frac_dantzig": frac(2), "frac_pgs": frac(8), "frac_friction_dropped": frac(16)}
    # sustained: >= 0.5 s of timed work, states re-seeded every 32 steps so that the robot does not leave the contact regime
    n_sus = max(K, int(np.ceil(650.0 / max(ms / K, 1e-3))))
    barrier()
    u0, u1 = ev(), ev()
    u0.record()
    for i in range(n_sus):
        if i % 32 == 0:
            x = x0; nb.reset_contact_cache(world)
        x = step(x, False)
    u1.record()
    barrier()
    sus_ms = u0.elapsed_time(u1)
    sticky = nb.check_contact_status(world)
    # e2e: the public call with pinned HOST tensors (H2D of state / action, D2H of the next state and of the gradients inside)
    hs = torch.tensor(s).pin_memory(); ha = torch.tensor(a).pin_memory(); hg = torch.randn(B, 2 * raw.ndof).pin_memory()
    e2e_steps = max(3, K // 4)

    xi = hs.requires_grad_(True); ai = ha.requires_grad_(True)   # pinned leaves, allocated once (cudaHostAlloc costs milliseconds)

    def e2e_step():
        xi.grad = None; ai.grad = None
        nb.timestep(world, xi, ai).backward(hg)
        return xi.grad

    for _ in range(3):
        e2e_step()
    barrier()
    w0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    barrier()
    e2e_ms = 1e3 * (time.perf_counter() - w0)
    t = torch.tensor([ms, sus_ms, e2e_ms], device=dev, dtype=torch.float64)
    if dist:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, sus_ms, e2e_ms = t.tolist()
    value = B * world_size * K / (ms * 1e-3)
    alg = ALG_BYTES[name]
    achieved = (value / world_size) * alg / 1e9
    traffic = None
    if name == "atlas_ground" and B == 8192:  # the ncu capture behind profiles/dram_traffic.json is this workload at this batch (sum of the 5 kernels of a step)
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "dram_traffic.json")))
            traffic = float(sum(tj[k] for k in ("k_cbuild", "k_csolve<0>", "k_csolve<1>", "k_capply", "k_cstep_bwd")))
        except Exception:
            traffic = None
    n, na = raw.ndof, len(raw.action_map)
    leg = {"workload": f"{name}: fwd+bwd step with the contact / boxed-LCP stage, batch={B}/GPU, fresh states (x_t+1 = step(x_t), LCP cache flowing)",
           "value": value, "unit": UNIT, "n_gpus": world_size, "steps": K, "warmup": W, "ms_per_step": ms / K,
           "sustained": {"value": B * world_size * n_sus / (sus_ms * 1e-3), "steps": n_sus, "timed_region_s": sus_ms * 1e-3},
           "kernel_ms": {"forward (build + solve x2 + apply)": float(np.mean([a_.elapsed_time(b_) for a_, b_ in fwd_ms])),
                         "backward (k_cstep_bwd)": float(np.mean([a_.elapsed_time(b_) for a_, b_ in bwd_ms]))},
           "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                        "algorithmic_bytes_per_world_step": alg, "algorithmic_bytes_per_step": alg * B,
                        "note": "latency / instruction-issue bound fp64 kernels (profiles/r02_*): the HBM fraction is reported as asked"},
           "e2e": {"value": B * world_size * e2e_steps / (e2e_ms * 1e-3), "unit": UNIT, "steps": e2e_steps,
                   "h2d_bytes_per_step": int(4 * B * (2 * n + na + 2 * n)), "d2h_bytes_per_step": int(4 * B * (2 * n + 2 * n + na)),
                   "path": "nimblephysics_b200.timestep() with pinned host tensors (copies inside the timed region)"},
           "gpu_launches": int(launches), "branch_stats_last_step": stats, "sticky_status": int(sticky)}
    if cpu_rate is not None:
        leg["cpu_baseline"] = cpu_rate
    return leg


def rollout_leg(nb, torch, B, T, reps, dev, dist, rank, world_size):
    """configs[4]: T-step rollout of Atlas + ground, loss = sum |x_T|^2 over ALL worlds (all-reduced over NCCL), backprop to x_0 and
    every tau_t through the whole horizon.  One host sync per rollout (the sticky contact status)."""
    from nimblephysics_b200.rollout import sharded_trajectory_loss
    from tests.util import contact_inputs

    raw = nb.RawModel.load(os.path.join(ROOT, "tests", "golden", "models", "atlas_ground.json"))
    world = nb.World.from_raw(raw)
    Bg = B * world_size
    s, _ = contact_inputs(raw, "atlas_ground", Bg, seed=11)
    rng = np.random.default_rng(12)
    na = len(raw.action_map)
    acts_np = rng.uniform(-20, 20, (T, Bg, na)).astype(np.float32)
    acts_np[:, :, :6] = 0.0
    x0 = torch.tensor(s, device=dev)                                  # the GLOBAL batch: sharded_trajectory_loss takes this rank's slice
    acts = [torch.tensor(acts_np[t], device=dev) for t in range(T)]
    loss_fn = lambda xT: (xT * xT).sum()

    def run(k=0):
        nb.reset_contact_cache(world)
        total, gx0, gacts = sharded_trajectory_loss(world, x0, acts, loss_fn, rank, world_size, checkpoint_every=k)  # all-reduces the scalar loss (NCCL)
        return total, gx0

    def timed(k):
        run(k); run(k)
        if dist:
            dist.barrier()
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            total, gx0 = run(k)
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / reps], device=dev, dtype=torch.float64)
        if dist:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), total, gx0, torch.cuda.max_memory_allocated(dev) / 2 ** 30

    ms, total, gx0, peak_gb = timed(0)
    ms_k, total_k, gx0_k, peak_gb_k = timed(8)
    sticky = nb.check_contact_status(world)
    return {"workload": f"64-step Atlas + ground rollout, backprop through the horizon, batch={B}/GPU (BASELINE configs[4])", "horizon": T,
            "value": Bg * T / (ms * 1e-3), "unit": UNIT, "n_gpus": world_size, "ms_per_rollout_fwd_bwd": ms, "rollouts_timed": reps,
            "driver": "nb2_rollout_forward_contact + nb2_rollout_backward_contact (one C call per direction, no host sync inside the horizon)",
            "loss": float(total), "loss_finite": bool(torch.isfinite(total)), "grad_finite": bool(torch.isfinite(gx0).all()),
            "collective": "all_reduce(SUM) of the scalar loss over %d rank(s)" % world_size, "sticky_status": int(sticky),
            "peak_memory_gb": peak_gb, "tape_bytes_per_gpu": nb.rollout_tape_bytes(world, B, T, 0),
            "checkpoint_every_8": {"value": Bg * T / (ms_k * 1e-3), "ms_per_rollout_fwd_bwd": ms_k, "peak_memory_gb": peak_gb_k,
                                   "tape_bytes_per_gpu": nb.rollout_tape_bytes(world, B, T, 8),
                                   "same_bits_as_full_tape": bool(torch.equal(gx0, gx0_k) and float(total) == float(total_k))}}

DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, arrays):
    """arrays: name -> [B, k] host array, one row per world.  Writes DIR/<name>.npy (float32); above DUMP_BYTES in all, the same
    seeded sample of rows from every array."""
    B = next(iter(arrays.values())).shape[0]
    per_world = sum(4 * a.shape[1] for a in arrays.values())
    keep = min(B, (DUMP_BYTES - 4096) // per_world)
    rows = np.arange(B) if keep == B else np.sort(np.random.default_rng(0).choice(B, keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a[rows], dtype=np.float32))


_REAL_STDOUT = None


def emit(obj):
    """The ONE JSON line of the contract goes to the process's original stdout; everything else any library prints
    (NCCL's version banner, torch warnings) was routed to stderr at start-up."""
    line = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, line)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)  # fd-level: also catches output of native libraries
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=4096, help="worlds per GPU")
    ap.add_argument("--precision", default="fp32", choices=["fp32", "fp64"])
    ap.add_argument("--lanes", type=int, default=0, help="threads cooperating on one world (0 = library picks from the batch size)")
    ap.add_argument("--no-extra", action="store_true", help="skip the cpu_baseline / e2e-independent extra contact legs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step of the GPU headline path as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs covers the GPU headline path (--impl ours) only")

    rank = int(os.environ.get("RANK", "0"))
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    import nimblephysics_b200 as nb

    raw = nb.RawModel.load(ATLAS)
    n, na = raw.ndof, len(raw.action_map)
    bytes_fwd = 4 * (2 * n + na + 2 * n)           # read state+action, write next state
    bytes_bwd = 4 * ((2 * n + na) + 2 * n + (2 * n + na))  # re-read inputs, read dL/dx', write grads
    config = {"workload": "Atlas (atlas_v3 URDF, 33 DoF, 28 moving bodies) contact-free Featherstone step fwd+bwd, "
                          f"batch={args.batch}/GPU, dt=1e-3, y-up gravity (BASELINE configs[1])",
              "global_batch": args.batch * max(world_size, 1), "parallelism": f"batch-sharded x{max(world_size,1)} (no data-path collective)",
              "l2_policy": "rotating buffer sets > L2 (126 MB)", "precision_inside_kernels": args.precision}

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        cores = os.cpu_count() or 1
        sample = max(cores * 32, 256)
        config = dict(config, precision_inside_kernels="fp64 (CPU)")
        real = probe_reference()
        if real is not None:
            rv = time_real_reference(real, seconds=max(3.0, 0.2 * args.steps))
            if rv is not None:
                v = rv * cores
                emit(({"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                       "ms_per_step": 1e3 * args.batch / v, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                       "data": "synthetic", "config": config,
                       "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "reference",
                                        "sample": f"nimblephysics forwardPass + backprop on Atlas: {rv:.1f} steps/s on one core x {cores} cores"},
                       "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
                return
        ref = CpuReference(raw, cores)
        for _ in range(max(args.warmup, 1)):
            ref.run(sample)
        tot_t, tot_n = 0.0, 0
        for _ in range(args.steps):
            _, dt, _ = ref.run(sample)
            tot_t += dt
            tot_n += sample
        ref.close()
        v = tot_n / tot_t
        emit(({
            "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{sample} Atlas worlds per step (fwd + backprop each), {cores} host processes, one oracle World per process; "
                                       "fp64 restatement of dart/{dynamics,neural}, NOT the reference binary (it cannot be built here)"},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    # ------------------------------------------------------------------ our arm (GPU)
    cpu_baseline = None
    cpu_contact = {}
    if world_size == 1 and not args.no_extra:  # timed BEFORE CUDA is initialised so the forked workers never inherit a CUDA context
        cores = os.cpu_count() or 1
        sample = max(cores * 16, 128)
        ref = CpuReference(raw, cores)
        v, dt, _ = ref.run(sample)
        ref.close()
        cpu_baseline = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": f"{sample} Atlas worlds (fwd + backprop each), mean busy time {dt:.2f} s per process on {cores} host processes; fp64 "
                                  "oracle (restatement of dart/{dynamics,neural}, not the reference binary)"}
        real = probe_reference()
        if real is not None:
            rv = time_real_reference(real)
            if rv is not None:
                cpu_baseline = {"value": rv * cores, "unit": UNIT, "cores": cores, "kind": "reference",
                                "sample": f"nimblephysics forwardPass + backprop on Atlas, one process for 3 s ({rv:.1f} steps/s) x {cores} cores "
                                          "(one World per core like MultiShot.cpp:66-70)", "port_value": v}
        for cname in ("half_cheetah", "atlas_ground"):
            try:
                craw = nb.RawModel.load(os.path.join(ROOT, "tests", "golden", "models", f"{cname}.json"))
                nw = max(cores * 2, 64)
                cv = cpu_contact_baseline(craw, cname, cores, nw)
                cpu_contact[cname] = {"value": cv, "unit": UNIT, "cores": cores, "kind": "port",
                                      "sample": f"{nw} worlds, step with the contact stage + backprop (dual-number Jacobians), fp64 oracle on {cores} processes"}
            except Exception as ex:
                cpu_contact[cname] = {"error": repr(ex)}
    import torch

    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    numa = bind_to_gpu_numa(local_rank)  # before the pinned buffers are allocated: they are first-touched on this node
    torch.cuda.set_device(local_rank)
    dist = None
    if world_size > 1:
        import torch.distributed as dist_mod

        dist_mod.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist = dist_mod
    dev = torch.device("cuda", local_rank)
    from nimblephysics_b200 import _cabi
    from nimblephysics_b200.engine import FP32, FP64

    prec = FP64 if args.precision == "fp64" else FP32
    B = args.batch
    dm = nb.DeviceModel.from_raw(raw)
    if args.lanes:
        dm.set_lanes(args.lanes)
    lanes_used = {"fwd": dm.lanes_for(B, False, prec), "bwd": dm.lanes_for(B, True, prec)}
    per_set = 4 * B * (2 * n * 4 + 2 * na + dm.saved_words * (2 if prec == FP64 else 1))
    nsets = max(2, int(np.ceil(160e6 / per_set)))
    sets = []
    for k in range(nsets):
        s, a, g = make_inputs(raw, B, 1234 + 1000 * rank + k)
        sets.append(dict(s=torch.tensor(s, device=dev), a=torch.tensor(a, device=dev), g=torch.tensor(g, device=dev),
                         nxt=torch.empty((B, 2 * n), device=dev), saved=torch.empty((dm.saved_words, B), device=dev, dtype=torch.float64 if prec == FP64 else torch.float32),
                         gs=torch.empty((B, 2 * n), device=dev), ga=torch.empty((B, na), device=dev)))
    stream = torch.cuda.current_stream().cuda_stream

    def fwd(d):
        dm.forward_device(B, d["s"].data_ptr(), d["a"].data_ptr(), d["nxt"].data_ptr(), d["saved"].data_ptr(), stream, prec)

    def bwd(d):
        dm.backward_device(B, d["s"].data_ptr(), d["a"].data_ptr(), d["saved"].data_ptr(), d["g"].data_ptr(),
                           d["gs"].data_ptr(), d["ga"].data_ptr(), stream, prec)

    def barrier():
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        fwd(sets[i % nsets]); bwd(sets[i % nsets])
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    # keep the GPU busy (untimed) while the clock sampler starts: an idle gap right before a timed region of a few milliseconds would make it
    # measure the clock ramp, not the kernels
    t_busy = time.perf_counter()
    k = 0
    while time.perf_counter() - t_busy < 0.3:
        d = sets[k % nsets]; k += 1
        fwd(d); bwd(d)
        if k % 64 == 0:
            torch.cuda.synchronize()
    l0 = _cabi.lib().nb2_launch_count()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t0.record()
    for i in range(args.steps):   # the timed region: exactly K steps, two events around it
        d = sets[(args.warmup + i) % nsets]
        fwd(d); bwd(d)
    t1.record()
    barrier()
    launches = _cabi.lib().nb2_launch_count() - l0
    total_ms = t0.elapsed_time(t1)
    # the passes below reuse these buffers: keep the last timed step's outputs now
    last = None
    if args.dump_outputs:
        d = sets[(args.warmup + args.steps - 1) % nsets]
        last = {"next_state": d["nxt"].cpu().numpy(), "grad_state": d["gs"].cpu().numpy(), "grad_action": d["ga"].cpu().numpy()}
    # per-kernel times from a separate instrumented pass (an event after every launch), outside the timed region
    ne = min(args.steps, 50)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * ne + 1)]
    ev[0].record()
    for i in range(ne):
        d = sets[i % nsets]
        fwd(d); ev[2 * i + 1].record()
        bwd(d); ev[2 * i + 2].record()
    torch.cuda.synchronize()
    fwd_ms = float(np.mean([ev[2 * i].elapsed_time(ev[2 * i + 1]) for i in range(ne)]))
    bwd_ms = float(np.mean([ev[2 * i + 1].elapsed_time(ev[2 * i + 2]) for i in range(ne)]))
    # sustained: the same loop for >= 0.5 s of timed work (the K-step region above is a few milliseconds long)
    n_sus = max(args.steps, int(np.ceil(650.0 / max(total_ms / args.steps, 1e-3))))
    barrier()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    for i in range(n_sus):
        d = sets[i % nsets]
        fwd(d); bwd(d)
    s1.record()
    barrier()
    sus_ms = s0.elapsed_time(s1)
    time.sleep(0.2)
    clocks = sampler.finish()

    # ---- e2e through the C-ABI host entry points (pinned host buffers; copies inside the timed region)
    hs, ha, hg = make_inputs(raw, B, 99 + rank)
    pin = lambda x: torch.from_numpy(x).pin_memory()
    hs_t, ha_t, hg_t = pin(hs), pin(ha), pin(hg)
    o_n, o_gs, o_ga = (torch.empty((B, 2 * n)).pin_memory(), torch.empty((B, 2 * n)).pin_memory(), torch.empty((B, na)).pin_memory())
    e2e_steps = max(5, args.steps // 2)

    def e2e_step():
        dm.forward_host(hs_t.numpy(), ha_t.numpy(), True, prec, out=o_n.numpy())
        dm.backward_host(hg_t.numpy(), prec, out_state=o_gs.numpy(), out_action=o_ga.numpy())

    tw = time.perf_counter()
    while time.perf_counter() - tw < 0.25:  # untimed: the clock sampler's shutdown and the pinned allocations above left the GPU idle
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    barrier()
    e2e_ms = 1e3 * (time.perf_counter() - t0)

    # ---- the other BASELINE configs, at EVERY world size (the batch shards; the rollout leg all-reduces its loss over NCCL)
    extra = {"legs": {}}
    if numa is not None:
        extra["numa_binding"] = numa
    if not args.no_extra:
        peak_hbm = 6650.0
        try:
            peak_hbm = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", peak_hbm))
        except Exception:
            pass
        for cname, cB, label in (("half_cheetah", 4096, "half_cheetah_ground_fwd_bwd (configs[2])"), ("atlas_ground", 8192, "atlas_ground_fwd_bwd (configs[3])")):
            try:
                extra["legs"][label] = contact_leg(nb, torch, cname, cB, max(args.steps, 8), max(args.warmup, 3), dev, dist, rank, world_size, peak_hbm,
                                                   cpu_contact.get(cname))
            except Exception as ex:  # never let a leg break the headline line
                extra["legs"][label] = {"error": repr(ex)}
        try:
            extra["legs"]["atlas_ground_rollout64 (configs[4])"] = rollout_leg(nb, torch, 1024, 64, 6, dev, dist, rank, world_size)
        except Exception as ex:
            extra["legs"]["atlas_ground_rollout64 (configs[4])"] = {"error": repr(ex)}
        # contact-free 64-step rollout through the fused entry points (nb2_rollout_forward / nb2_rollout_backward)
        try:
            from nimblephysics_b200.rollout import rollout_fused

            fworld = nb.World.from_raw(raw)
            fworld._contacts_disabled = True
            Tf = 64
            rngf = np.random.default_rng(21 + rank)
            uf = rngf.uniform(-20, 20, (Tf, B, na)).astype(np.float32)
            uf[:, :, :6] = 0.0
            xf0 = sets[0]["s"].clone().requires_grad_(True)
            uft = torch.tensor(uf, device=dev, requires_grad=True)

            def runf():
                tr = rollout_fused(fworld, xf0, uft)
                (tr[-1] * tr[-1]).sum().backward()

            runf(); runf()
            barrier()
            q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            q0.record()
            for _ in range(8):
                runf()
            q1.record()
            barrier()
            tq = torch.tensor([q0.elapsed_time(q1) / 8], device=dev, dtype=torch.float64)
            if dist:
                dist.all_reduce(tq, op=dist.ReduceOp.MAX)
            msf = float(tq[0])
            extra["legs"]["atlas_rollout64_contact_free"] = {"batch_per_gpu": B, "horizon": Tf, "ms_per_rollout_fwd_bwd": msf, "n_gpus": world_size,
                                                             "value": B * world_size * Tf / (msf * 1e-3), "unit": UNIT}
        except Exception as ex:
            extra["legs"]["atlas_rollout64_contact_free"] = {"error": repr(ex)}

    t_total = torch.tensor([total_ms, e2e_ms, sus_ms], device=dev, dtype=torch.float64)
    if dist:
        dist.all_reduce(t_total, op=dist.ReduceOp.MAX)
    total_ms, e2e_ms, sus_ms = t_total.tolist()
    value = B * world_size * args.steps / (total_ms * 1e-3)
    e2e_value = B * world_size * e2e_steps / (e2e_ms * 1e-3)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        dom, dom_ms, dom_bytes = ("k_step_bwd", bwd_ms, bytes_bwd) if bwd_ms >= fwd_ms else ("k_step_fwd", fwd_ms, bytes_fwd)
        achieved = dom_bytes * B / (dom_ms * 1e-3) / 1e9
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "dram_traffic.json"))).get(dom)
        except Exception:
            pass
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world_size, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32" if prec == FP32 else "f64", "data": "synthetic", "config": config,
            "kernel_ms": {"k_step_fwd": fwd_ms, "k_step_bwd": bwd_ms, "note": "separate instrumented pass with an event after every launch (about +3 us per launch); the timed region has two events"}, "lanes_per_world": lanes_used,
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic,
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s",
                         "algorithmic_bytes_per_world": {"k_step_fwd": bytes_fwd, "k_step_bwd": bytes_bwd, "step": bytes_fwd + bytes_bwd},
                         "note": "path is FP32-latency bound, not HBM bound (DESIGN.md §roofline): the HBM fraction is reported as asked"},
            "e2e": {"value": e2e_value, "unit": UNIT,
                    "h2d_bytes_per_step": int(4 * B * (2 * n + na + 2 * n)), "d2h_bytes_per_step": int(4 * B * (2 * n + 2 * n + na)),
                    "steps": e2e_steps, "path": "nb2_step_forward_host + nb2_step_backward_host (pinned host buffers)"},
            "sustained": {"value": B * world_size * n_sus / (sus_ms * 1e-3), "steps": n_sus, "timed_region_s": sus_ms * 1e-3},
            "gpu_launches": int(launches), "clocks": clocks, "extra": extra,
        }
        if cpu_baseline is not None:
            out["cpu_baseline"] = cpu_baseline
        if last is not None:
            dump_outputs(args.dump_outputs, last)
        emit(out)
    if dist:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
