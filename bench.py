#!/usr/bin/env python
"""bench.py -- geometry-energy + gradient iterations/sec at 64 tet-spheres x 4096 tets per GPU.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR

--dump-outputs DIR writes what the last timed step computed, as a caller of tsb_energy_grad receives it:
DIR/energy.npy (float32 [3]: total, smoothness, barrier) and DIR/grad.npy (float32 [n,3]); under torchrun
every rank writes its own, suffixed _rank<r>.  The inputs depend on the arguments only, so two builds run
with the same arguments can be compared file by file.

A *step* is ONE launch of the fused energy+gradient kernel (tsb_energy_grad) over one synthetic pack
of 64 tet-spheres x 4096 tets (BASELINE.json metric; the kernel-only form of configs[2], whose
rasterizer/trainer dependencies are absent -- SURVEY.md F7).  Weak scaling: every rank owns its own
64-sphere pack (spheres share nothing, so there is no data-path collective); the scalar energies are
all-reduced asynchronously once per graph replay, off the critical path.  Before timing, multi-rank runs
check the sharded product path (tssplat_b200.sharding.ShardedEnergy) against a single-GPU evaluation.

Timing rules honoured: W >= 3 warm-up steps; the timed steps rotate over R distinct packs whose
combined footprint exceeds the 126 MB L2, so every step streams its plan data from HBM; CUDA events
on the launching stream, barrier + synchronize on both sides, max over ranks; SM clocks and
throttle reasons sampled through NVML during the timed region.

The reference arm and the cpu_baseline run a CPU *restatement* of the reference's math (the
reference extension needs libpgo + cuSPARSE + a GPU and ships no CPU path: SURVEY.md F2/F4): the
matrix-free C oracle (oracle/tet_energy_oracle.c, OpenMP, pinned threads), in its fastest build for
this host (fp32 arithmetic like the reference when the host has AVX2+FMA, else the portable fp64
build).  The slower "vanilla PyTorch" restatement of the reference's SpMV pipeline
(oracle/torch_energy.py) is timed too and reported in `extras`.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import sys
import threading
import time

try:      # before anything can start an OpenMP region: OMP_PROC_BIND narrows the main thread's mask to its own place
    _AFFINITY0 = frozenset(os.sched_getaffinity(0))
except Exception:
    _AFFINITY0 = None

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
if "reference" in sys.argv:       # CPU arm only: pin the OpenMP threads (must be set before libgomp loads).  The GPU arm runs
    os.environ.setdefault("OMP_PROC_BIND", "close")     # its cpu_baseline leg in a child process instead: binding would
    os.environ.setdefault("OMP_PLACES", "cores")        # confine this process (and the plan builder's threads) to one core

SPHERES, TETS = 64, 4096
METRIC = "geometry_energy_grad_iters_per_sec_64x4k"
UNIT = "iters/s"
N_ROTATE = 8           # distinct packs per rank; 8 x ~23 MB of plan data > 126 MB L2
ORDER = 2
DUMP_BYTES = 64 << 20  # --dump-outputs budget over all ranks; a larger gradient is written as a seeded row sample
KERNEL_SOURCES = ("tssplat_b200/csrc/tsb_kernels.cu", "tssplat_b200/csrc/tsb_plan.cpp", "tssplat_b200/csrc/tsb_plan.h")


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def kernel_hash() -> str:
    h = hashlib.sha1()
    for f in KERNEL_SOURCES:
        h.update(open(os.path.join(ROOT, f), "rb").read())
    return h.hexdigest()[:16]


def _traffic():
    """DRAM bytes per launch from the committed `ncu --set full` capture; only trusted when it was taken
    on exactly these kernel / plan sources (stamped with their hash), else null."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        d = json.load(open(p))
        if d.get("kernel_hash") == kernel_hash():
            return float(d["dram_bytes_per_step"]), d.get("source", "")
        return None, f"stale: profiles/traffic.json was captured on kernel {d.get('kernel_hash')}, this is {kernel_hash()}"
    except Exception:
        return None, "no capture"


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40,
                 "sw_thermal_slowdown": 0x20, "hw_power_brake_slowdown": 0x80}
        while not self._halt.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                break
            time.sleep(0.001)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        return {"sm_mhz": (float(np.median(self.samples)) if self.samples else None),
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ---- CPU arms ------------------------------------------------------------------------------------------
def _host_threads():
    """Hardware threads this process was given at start-up (NOT the current mask: once libgomp has bound the
    main thread to its place, sched_getaffinity reports that one core only)."""
    return len(_AFFINITY0) if _AFFINITY0 else (os.cpu_count() or 1)


def _c_oracle(pack, variant=""):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from _helpers import COracle
    return COracle(pack.verts, pack.tets, variant=variant)


def _cpu_variants():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from _helpers import host_has_avx2_fma
    return ["fast32", "fast", ""] if host_has_avx2_fma() else [""]


def _calibrate(pack, x, c1, c2):
    """Fastest (build, thread count) of the CPU port on this host: >= 10 repetitions per candidate."""
    avail = _host_threads()
    best = None
    for variant in _cpu_variants():
        co = _c_oracle(pack, variant)
        for th in sorted({t for t in (4, 8, 16, 32, 64, 96, avail) if t <= avail}):
            co.energy_grad(x, c1, c2, ORDER, nthreads=th)
            ts = []
            for _ in range(10):
                t0 = time.perf_counter()
                co.energy_grad(x, c1, c2, ORDER, nthreads=th)
                ts.append(time.perf_counter() - t0)
            dt = float(np.median(ts))
            if best is None or dt < best[0]:
                best = (dt, variant, th, co)
    return best


def _time_cpu(co, x, c1, c2, threads, min_seconds, min_steps):
    """Per-step times of the CPU port: at least min_steps steps and min_seconds of work."""
    ts = []
    t_start = time.perf_counter()
    while len(ts) < min_steps or time.perf_counter() - t_start < min_seconds:
        t0 = time.perf_counter()
        co.energy_grad(x, c1, c2, ORDER, nthreads=threads)
        ts.append(time.perf_counter() - t0)
        if time.perf_counter() - t_start > 60.0:
            break
    return np.asarray(ts)


def _variant_name(v):
    return {"fast32": "fp32 arithmetic (the reference's precision), -O3 AVX2+FMA", "fast": "fp64, -O3 AVX2+FMA",
            "": "fp64, portable -O2"}[v]


def run_reference(args):
    """CPU arm: the oracle port on the host cores (rank 0 only), all the OpenMP threads it can use."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from tssplat_b200.mesh import make_pack, perturb
    pack = make_pack(SPHERES, TETS, seed=0, unique=8)
    x = perturb(pack, sigma_rel=0.02, seed=0)
    c1, c2 = 2e-4 / SPHERES, 2e-4
    dt0, variant, cores, co = _calibrate(pack, x, c1, c2)
    for _ in range(max(args.warmup, 3)):
        co.energy_grad(x, c1, c2, ORDER, nthreads=cores)
    ts = _time_cpu(co, x, c1, c2, cores, min_seconds=args.min_seconds, min_steps=max(200, min(args.steps, 2000)))
    dt = float(np.median(ts))
    value = 1.0 / dt
    sample = (f"{len(ts)} energy+gradient iterations of the full {SPHERES}-sphere pack ({SPHERES * TETS} tets), median step time "
              f"(p10 {np.percentile(ts, 10) * 1e3:.2f} ms, p90 {np.percentile(ts, 90) * 1e3:.2f} ms); matrix-free C port "
              f"(oracle/tet_energy_oracle.c), {_variant_name(variant)}, OpenMP {cores} threads pinned "
              f"(fastest of the builds/thread counts tried, {_host_threads()} available)")
    out = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
           "steps": int(len(ts)), "warmup": max(args.warmup, 3), "ms_per_step": dt * 1e3,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32" if variant == "fast32" else "f64",
           "data": "synthetic",
           "config": {"workload": f"{SPHERES} tet-spheres x {TETS} tets, energy+gradient, CPU port of the reference's "
                                  "math (the reference itself needs libpgo + a GPU)", "spheres_per_gpu": SPHERES,
                      "total_spheres": SPHERES, "tets_per_sphere": TETS, "order": ORDER,
                      "x": "rest + N(0,(0.02 h)^2), no inverted tets"},
           "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))


# ---- GPU arm ---------------------------------------------------------------------------------------------
def dump_outputs(out_dir, energy, grad, suffix="", budget=DUMP_BYTES):
    """energy[3] and grad[n,3] (host float32) as out_dir/energy<suffix>.npy and grad<suffix>.npy.  A gradient larger
    than the budget keeps a fixed, seeded, sorted sample of its rows, the same one for every build."""
    os.makedirs(out_dir, exist_ok=True)
    if grad.nbytes + energy.nbytes > budget:
        keep = (budget - energy.nbytes) // grad[0].nbytes
        grad = grad[np.sort(np.random.default_rng(0).choice(len(grad), keep, replace=False))]
    np.save(os.path.join(out_dir, f"energy{suffix}.npy"), energy)
    np.save(os.path.join(out_dir, f"grad{suffix}.npy"), grad)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4000)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--spheres-per-gpu", type=int, default=SPHERES,
                    help="weak scaling (default): spheres owned by every rank")
    ap.add_argument("--total-spheres", type=int, default=0,
                    help="strong scaling: total spheres split sphere-per-rank (BASELINE configs[3], [4])")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--min-seconds", type=float, default=2.0, help="CPU arm: minimum timed duration")
    ap.add_argument("--no-extras", action="store_true", help="skip the size sweep / trainer-loop / strong-scaling extras")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the energy and gradient of the last timed step to DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    from tssplat_b200 import _capi
    from tssplat_b200 import tet_spheres_ext as ext
    from tssplat_b200.energies import SmoothnessBarrierEnergy, SmoothnessBarrierFunc
    from tssplat_b200.mesh import make_pack, perturb
    from tssplat_b200.sharding import ShardedEnergy, partition_spheres

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: tssplat_b200 has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lib = _capi.lib

    # ---- multi-rank: the sharded product path must reproduce a single-GPU evaluation --------------------
    shard_check = None
    if world > 1:
        chk = make_pack(4 * world, 1024, seed=5)
        xc = perturb(chk, sigma_rel=0.35, seed=2)
        se = ShardedEnergy(chk, rank, world, device=dev)
        lo, hi = se.sphere_range
        v0, v1 = int(chk.vert_offsets[lo]), int(chk.vert_offsets[hi])
        e_sh, g_sh = se.energy_grad(torch.from_numpy(xc[v0:v1]).to(dev), 1e-4, 2e-4, 2)
        se.wait()
        full = ext.TetSpheres(chk.verts.reshape(-1), chk.tets.reshape(-1), device=dev)
        e_f, g_f = full.energy_grad(torch.from_numpy(xc).to(dev), 1e-4, 2e-4, 2)
        torch.cuda.synchronize()
        ok = (abs(float(e_sh[0]) - float(e_f[0])) <= 2e-5 * abs(float(e_f[0])) and
              float((g_sh - g_f[v0:v1]).norm()) <= 2e-5 * float(g_f[v0:v1].norm()))
        flag = torch.tensor([1.0 if ok else 0.0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if float(flag.item()) != 1.0:
            raise SystemExit("ShardedEnergy check failed: sharded energy/gradient differ from the single-GPU result")
        shard_check = "ShardedEnergy (NCCL) == single-GPU evaluation: sum-energy and per-rank gradient slices within 2e-5"
        del se, full

    # ---- inputs: R distinct packs per rank, resident in HBM ---------------------------------------
    strong = args.total_spheres > 0
    if strong:
        lo, hi = partition_spheres([TETS] * args.total_spheres, world)[rank]
        n_sph = hi - lo
    else:
        n_sph = args.spheres_per_gpu
    total_spheres = args.total_spheres if strong else n_sph * world
    c1, c2 = 2e-4 / total_spheres, 2e-4
    packs, handles, xs, create_main = [], [], [], []
    L2_BYTES = 126e6
    n_rotate = None
    i = 0
    while n_rotate is None or i < n_rotate:
        pk = make_pack(n_sph, TETS, seed=1000 * rank + 17 * i, unique=8)
        packs.append(pk)
        t_c = time.perf_counter()
        handles.append(ext.TetSpheres(pk.verts.reshape(-1), pk.tets.reshape(-1)))
        create_main.append(time.perf_counter() - t_c)
        xs.append(torch.from_numpy(perturb(pk, sigma_rel=0.02, seed=i)).to(dev))
        if n_rotate is None:   # enough distinct packs that one rotation streams > 1.5 x L2 through the GPU
            n_rotate = int(min(64, max(2, -(-1.5 * L2_BYTES // handles[0].info["stream_bytes"]))))
            n_rotate = max(n_rotate, N_ROTATE if n_sph <= 128 else 2)
        i += 1
    n = handles[0].n
    info = handles[0].info
    b_alg = float(np.mean([pk.algorithmic_bytes() for pk in packs]))
    footprint = sum(h.info["stream_bytes"] for h in handles)
    energies = torch.zeros((n_rotate, 3), device=dev)
    grads = [torch.empty((h.n, 3), device=dev) for h in handles]
    stream = torch.cuda.Stream(device=dev)
    comm = torch.cuda.Stream(device=dev)

    def launch(i, st, hs=handles, x_=xs, en=energies, gr=grads, c1_=None):
        rc = lib.tsb_energy_grad(hs[i]._h, x_[i].data_ptr(), c1 if c1_ is None else c1_, c2, ORDER, 1.0, None,
                                 en[i].data_ptr(), gr[i].data_ptr(), st)
        if rc != 0:
            raise RuntimeError(_capi.last_error(hs[i]._h))

    def graph_of(fn, count):
        with torch.cuda.stream(stream):
            for k in range(min(count, 3)):
                fn(k)
            stream.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=stream):
                for k in range(count):
                    fn(k)
            g.replay()
            stream.synchronize()
        return g

    with torch.cuda.stream(stream):
        for w in range(args.warmup):
            launch(w % n_rotate, stream.cuda_stream)
        stream.synchronize()
    # one replay = `rounds` passes over the rotating packs (~1 ms of device work), so that neither the replay call
    # nor, under torchrun, the once-per-replay scalar all-reduce is what the host has to keep up with
    rounds = int(max(1, min(args.steps // n_rotate, 96 // n_rotate if n_sph <= 128 else 1)))
    graph_len = rounds * n_rotate
    graph = graph_of(lambda k: launch(k % n_rotate, stream.cuda_stream), graph_len)

    def timed_region(steps):
        """Exactly `steps` steps; returns seconds (device time, this rank)."""
        reps, rem = divmod(steps, graph_len)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        with torch.cuda.stream(stream):
            ev0.record(stream)
            for _ in range(reps):
                graph.replay()
                if world > 1:       # scalar loss all-reduce, once per replay, on the side stream
                    comm.wait_stream(stream)
                    with torch.cuda.stream(comm):
                        dist.all_reduce(energies, op=dist.ReduceOp.SUM, async_op=True)
            for i in range(rem):
                launch(i % n_rotate, stream.cuda_stream)
            stream.wait_stream(comm)
            ev1.record(stream)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        return ev0.elapsed_time(ev1) * 1e-3

    timed_region(min(args.steps, 3 * graph_len))                      # settle clocks / NCCL
    sampler = ClockSampler(local_rank)
    sampler.start()
    t_local = timed_region(args.steps)
    clocks = sampler.stop()
    if args.dump_outputs:       # before anything else launches on these buffers
        rem = args.steps % graph_len
        last = (rem - 1 if rem else graph_len - 1) % n_rotate          # pack of the last timed step
        dump_outputs(args.dump_outputs, energies[last].cpu().numpy(), grads[last].cpu().numpy(),
                     f"_rank{rank}" if world > 1 else "", DUMP_BYTES // world)
    t_all = torch.tensor([t_local], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_all, op=dist.ReduceOp.MAX)
    t = float(t_all.item())
    ms_per_step = t / args.steps * 1e3
    # weak: every rank steps its own pack -> aggregate pack-iterations/s; strong: all ranks together
    # advance ONE pack of total_spheres per step.  Reported in units of the 64-sphere metric pack.
    value = args.steps / t * (total_spheres / SPHERES)

    def time_graph(g, per_replay, min_replays=3, budget_s=0.25):
        with torch.cuda.stream(stream):
            g.replay(); stream.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream); g.replay(); e1.record(stream); stream.synchronize()
            one = max(e0.elapsed_time(e1) * 1e-3, 1e-6)
            reps = int(max(min_replays, min(2000, budget_s / one)))
            e0.record(stream)
            for _ in range(reps):
                g.replay()
            e1.record(stream)
            stream.synchronize()
        return e0.elapsed_time(e1) * 1e-3 / (reps * per_replay)

    # ---- warm-L2 variant (one pack replayed): explains the launch-latency floor ---------------
    g1 = graph_of(lambda k: launch(0, stream.cuda_stream), n_rotate)
    warm_ms = time_graph(g1, n_rotate) * 1e3

    # ---- end to end with HOST buffers: (1) through the C-ABI host entry point, (2) through the
    # reference-facing autograd surface (SmoothnessBarrierEnergy) -- copies inside the timed region
    x_host = xs[0].cpu().pin_memory()
    g_host = torch.empty((n, 3), dtype=torch.float32).pin_memory()
    e_host = torch.empty(3, dtype=torch.float32).pin_memory()

    def timed_e2e(step_fn, steps):
        for _ in range(5):
            step_fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ee0, ee1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ee0.record()
        for _ in range(steps):
            step_fn()
        ee1.record()
        torch.cuda.synchronize()
        te = torch.tensor([ee0.elapsed_time(ee1) * 1e-3], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        return world * steps / float(te.item())

    e2e_scale = (n_sph / SPHERES) if not strong else (total_spheres / SPHERES) / world
    e2e_steps = int(min(args.steps, 1000))
    e2e_value = e2e_scale * timed_e2e(lambda: ext.energy_grad_host(handles[0], x_host, c1, c2, ORDER, 1.0, e_host, g_host), e2e_steps)

    eng = SmoothnessBarrierEnergy.__new__(SmoothnessBarrierEnergy)
    torch.nn.Module.__init__(eng)
    from types import SimpleNamespace
    eng.tet_sp, eng.FLAGS = handles[0], SimpleNamespace(smooth_eng_coeff=c1, barrier_coeff=c2, increase_order_iter=10 ** 9)
    eng.smooth_eng_func = SmoothnessBarrierFunc
    tet_v = torch.nn.Parameter(torch.empty((n, 3), device=dev))
    e0_host = torch.empty((), dtype=torch.float32).pin_memory()

    def autograd_step():
        tet_v.grad = None
        with torch.no_grad():
            tet_v.copy_(x_host, non_blocking=True)                   # H2D of this step's input
        e = eng(tet_v, 0, c1, c2)                                     # forward (fused launch)
        e.backward()                                                  # backward (cached gradient)
        g_host.copy_(tet_v.grad, non_blocking=True)                  # D2H of the result
        e0_host.copy_(e.detach(), non_blocking=True)

    e2e_autograd = e2e_scale * timed_e2e(autograd_step, int(min(args.steps, 500)))

    class _Floor(torch.autograd.Function):       # what torch.autograd costs when forward/backward launch nothing
        @staticmethod
        def forward(ctx, x, e, g):
            ctx.g = g
            return e[0]

        @staticmethod
        def backward(ctx, go):
            return ctx.g, None, None

    e_pre, g_pre = torch.zeros(3, device=dev), torch.zeros((n, 3), device=dev)

    def floor_step():
        tet_v.grad = None
        with torch.no_grad():
            tet_v.copy_(x_host, non_blocking=True)
        e = _Floor.apply(tet_v, e_pre, g_pre)
        e.backward()
        g_host.copy_(tet_v.grad, non_blocking=True)
        e0_host.copy_(e.detach(), non_blocking=True)

    autograd_floor = e2e_scale * timed_e2e(floor_step, int(min(args.steps, 500)))

    # ---- extras ------------------------------------------------------------------------------------------
    extras = {"e2e_autograd_surface_iters_per_s": e2e_autograd,
              "e2e_autograd_surface_note": "pinned host x -> H2D -> SmoothnessBarrierEnergy.forward/backward "
                                           "(torch.autograd.Function) -> D2H grad+energy",
              "e2e_autograd_torch_floor_iters_per_s": autograd_floor,
              "e2e_autograd_torch_floor_note": "the same step with a torch.autograd.Function that launches nothing: the ceiling "
                                               "torch's Python autograd machinery and the three copy_ calls leave for this surface",
              "tsb_create_seconds_64_spheres": float(np.median(create_main)),
              "tsb_create_note": "setup (SURVEY 8 f3): host plan build on all cores + upload, median over the rotating packs; "
                                 "the 1024-sphere figure is in config4_1024_spheres_one_gpu",
              "warm_l2_ms_per_step": warm_ms, "warm_l2_iters_per_s": 1e3 / warm_ms,
              "stream_bytes_per_step": int(info["stream_bytes"])}
    if shard_check:
        extras["sharded_path_check"] = shard_check
    peak, peak_src = _peaks()

    create_s = {}
    extras_1sphere_us = None

    def one_pack_rate(S, seed):
        """us/step of one S-sphere pack on this GPU (graph replay; > L2 when S >= 512)."""
        pk = make_pack(S, TETS, seed=seed, unique=8)
        t_c = time.perf_counter()
        h = ext.TetSpheres(pk.verts.reshape(-1), pk.tets.reshape(-1))
        torch.cuda.synchronize()
        create_s[S] = time.perf_counter() - t_c
        xx = [torch.from_numpy(perturb(pk, sigma_rel=0.02, seed=0)).to(dev)]
        en = torch.zeros((1, 3), device=dev)
        gr = [torch.empty((h.n, 3), device=dev)]
        reps = 4 if S >= 512 else 16
        g = graph_of(lambda k: launch(0, stream.cuda_stream, [h], xx, en, gr, 2e-4 / S), reps)
        sec = time_graph(g, reps)
        return sec, pk.algorithmic_bytes(), h.info

    if not args.no_extras and not strong and n_sph == SPHERES:
        if world == 1:
            try:      # single process: an extra that fails is reported, the headline line still prints
                sec1, _, _ = one_pack_rate(1, 7000)
                extras_1sphere_us = sec1 * 1e6
                sec, b16, _ = one_pack_rate(16, 7001)
                extras["config1_16_spheres"] = {"us_per_step": sec * 1e6, "iters_per_s": 1.0 / sec, "hbm_frac_by_B_alg": b16 / sec / 1e9 / peak,
                                                "note": "BASELINE configs[1]: 16 tet-spheres, fused kernel only, fp32, 1 GPU (L2-resident)"}
                sec, b1k, inf = one_pack_rate(1024, 7002)
                extras["config4_1024_spheres_one_gpu"] = {"us_per_step": sec * 1e6, "algorithmic_GBps": b1k / sec / 1e9,
                                                          "hbm_frac_by_B_alg": b1k / sec / 1e9 / peak,
                                                          "plan_stream_GBps": inf["stream_bytes"] / sec / 1e9,
                                                          "tsb_create_seconds": create_s.get(1024),
                                                          "note": "BASELINE configs[4] pack (1024 spheres, 4.2 M tets) on ONE GPU: "
                                                                  "306 MB of plan data per step, HBM-streaming regime"}
            except Exception as ex:  # pragma: no cover
                extras["size_sweep_error"] = repr(ex)
            try:
                sys.path.insert(0, os.path.join(ROOT, "tools"))
                from energy_only_loop import run as loop_run
                loop_run(spheres=SPHERES, iters=30)
                rate, le0, le1 = loop_run(spheres=SPHERES, iters=600)
                extras["config2_energy_only_trainer_loop"] = {
                    "iters_per_s": rate, "reg_loss_first": le0, "reg_loss_last": le1,
                    "note": "BASELINE configs[2] substitute (rasterizer/data deps absent, SURVEY F7): trainer.py:71-132 minus the "
                            "renderer -- coefficient scheduler + autograd surface + AdamUniform(grad_limit) + cosine LR, wall clock"}
            except Exception as ex:  # pragma: no cover
                extras["config2_energy_only_trainer_loop"] = {"error": repr(ex)}
        else:
            # strong scaling lines (BASELINE configs[3] / [4]): total spheres fixed, sharded sphere-per-rank
            for total in (256, 1024):
                lo2, hi2 = partition_spheres([TETS] * total, world)[rank]
                pk = make_pack(hi2 - lo2, TETS, seed=9000 + 31 * rank + total, unique=8)
                h = ext.TetSpheres(pk.verts.reshape(-1), pk.tets.reshape(-1))
                xx = [torch.from_numpy(perturb(pk, sigma_rel=0.02, seed=0)).to(dev)]
                en = torch.zeros((1, 3), device=dev)
                gr = [torch.empty((h.n, 3), device=dev)]
                reps = 8
                g = graph_of(lambda k: launch(0, stream.cuda_stream, [h], xx, en, gr, 2e-4 / total), reps)
                dist.barrier()
                sec = time_graph(g, reps)
                ts_ = torch.tensor([sec], device=dev, dtype=torch.float64)
                dist.all_reduce(ts_, op=dist.ReduceOp.MAX)
                extras[f"strong_scaling_{total}_spheres"] = {
                    "us_per_step_max_over_ranks": float(ts_.item()) * 1e6, "pack_iters_per_s": 1.0 / float(ts_.item()),
                    "spheres_per_rank": hi2 - lo2,
                    "note": f"BASELINE configs[{3 if total == 256 else 4}]: {total} spheres split sphere-per-rank over {world} GPUs, "
                            "one fused launch per rank per step, graph replay (compare with the single-GPU time of the same pack)"}
                del h, g

    if rank == 0:
        achieved = b_alg / (t / args.steps) / 1e9                   # GB/s per GPU, whole step (one launch)
        traffic, traffic_src = _traffic()
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if strong else "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{n_sph} tet-spheres x {TETS} tets per GPU ({total_spheres} in total), ONE fused energy+grad "
                                   "launch per step; kernel-only form of BASELINE configs[2] (rasterizer deps absent); value is "
                                   "in 64-sphere-pack iterations/s",
                       "spheres_per_gpu": n_sph, "total_spheres": total_spheres, "tets_per_sphere": TETS, "vertices": int(n), "order": ORDER,
                       "x": "rest + N(0,(0.02 h)^2), no inverted tets", "parallelism": f"sphere-per-rank x{world}",
                       "l2": f"inputs larger than L2: rotating {n_rotate} distinct packs, {footprint / 1e6:.0f} MB "
                             "of per-step data > 126 MB L2",
                       "grid": int(info["grid"]), "warps_per_cta": int(info["warps_per_cta"]), "segments": int(info["n_segments"]),
                       "graph": f"CUDA graph of {graph_len} steps ({rounds} passes over the {n_rotate} packs) replayed"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "algorithmic_bytes_per_step": b_alg, "plan_stream_bytes_per_step": int(info["stream_bytes"]),
                         "note": "achieved = B_alg (24V+68T per sphere, SURVEY 8d) / CUDA-event step time of the single fused launch; "
                                 "the streamed-operator formulation actually moves plan_stream_bytes_per_step"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(n * 12),
                    "d2h_bytes_per_step": int(n * 12 + 12), "steps": e2e_steps,
                    "path": "C-ABI tsb_energy_grad_host: pinned host x -> H2D (two alternating internal streams, double-buffered) -> fused launch -> "
                            "D2H grad + energy[3]"},
            "gpu_launches": int(args.steps),
            "clocks": clocks,
            "extras": extras,
        }
        if world == 1 and not args.no_cpu_baseline and n_sph == SPHERES:
            x0 = xs[0].cpu().numpy()
            # the CPU port, timed in a child process (pinned OpenMP threads, all host cores): `--impl reference` itself
            import subprocess
            env = {k: v for k, v in os.environ.items() if k not in ("OMP_NUM_THREADS",)}
            try:
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--min-seconds", "10"],
                                   capture_output=True, text=True, env=env, timeout=600)
                out["cpu_baseline"] = json.loads(r.stdout.strip().splitlines()[-1])["cpu_baseline"]
            except Exception as ex:      # keep the GPU line: time the port in this process instead (threads not pinned)
                dt0, variant, cores, co = _calibrate(packs[0], x0, c1, c2)
                ts = _time_cpu(co, x0, c1, c2, cores, min_seconds=10.0, min_steps=200)
                out["cpu_baseline"] = {"value": 1.0 / float(np.median(ts)), "unit": UNIT, "cores": cores, "kind": "port",
                                       "sample": f"{len(ts)} energy+gradient iterations of the full 64-sphere pack, median step; "
                                                 f"matrix-free C port, {_variant_name(variant)}, OpenMP {cores} threads, NOT pinned "
                                                 f"(the pinned child process failed: {type(ex).__name__})"}
            if not args.no_extras:
                try:
                    # the reference-shaped "vanilla PyTorch" pipeline (SpMV GTLTLG, SpMV G, autograd), best thread count
                    from oracle.torch_energy import time_fwd_bwd
                    best, ns, avail = None, 2, _host_threads()
                    sub = packs[0].slice_spheres(0, ns)
                    v1 = int(packs[0].vert_offsets[ns])
                    for th in sorted({min(avail, 8), min(avail, 32), avail}):
                        tt_, _, _ = time_fwd_bwd(sub.verts, sub.tets, x0[:v1], c1, c2, ORDER, iters=4, warmup=1, threads=th)
                        if best is None or tt_ < best[0]:
                            best = (tt_, th)
                    # BASELINE configs[0]: ONE tet-sphere, vanilla-PyTorch forward+backward on the host cores, beside the fused
                    # launch on the same sphere
                    one = packs[0].slice_spheres(0, 1)
                    v0 = int(packs[0].vert_offsets[1])
                    t1s, _, _ = time_fwd_bwd(one.verts, one.tets, x0[:v0], c1, c2, ORDER, iters=20, warmup=3, threads=best[1])
                    s16 = packs[0].slice_spheres(0, 16)
                    v16 = int(packs[0].vert_offsets[16])
                    t16s, _, _ = time_fwd_bwd(s16.verts, s16.tets, x0[:v16], c1, c2, ORDER, iters=20, warmup=3, threads=best[1])
                    cpu_model = ""
                    try:
                        with open("/proc/cpuinfo") as f:
                            cpu_model = next((ln.split(":", 1)[1].strip() for ln in f if ln.startswith("model name")), "")
                    except OSError:
                        pass
                    out["extras"]["host"] = {"cpu_model": cpu_model, "os_cpu_count": os.cpu_count(), "threads_available": avail}
                    if "config1_16_spheres" in out["extras"]:
                        out["extras"]["config1_16_spheres"]["vanilla_torch_cpu_ms_per_fwd_bwd"] = t16s * 1e3
                        out["extras"]["config1_16_spheres"]["vanilla_torch_cpu_threads"] = best[1]
                    out["extras"]["config0_1_sphere"] = {
                        "vanilla_torch_cpu_ms_per_fwd_bwd": t1s * 1e3, "threads": best[1],
                        "b200_fused_launch_us": extras_1sphere_us,
                        "note": "BASELINE configs[0]: 1 tet-sphere x 4096 tets; torch sparse fp32 + autograd restatement of the "
                                "reference's SpMV pipeline on the CPU vs ONE fused energy+grad launch (graph replay)"}
                    out["extras"]["cpu_torch_restatement_iters_per_s"] = 1.0 / (best[0] * SPHERES / ns)
                    out["extras"]["cpu_torch_restatement_note"] = (f"torch sparse fp32 + autograd restatement of the reference's SpMV "
                                                                   f"pipeline, {ns} of {SPHERES} spheres extrapolated, best of thread "
                                                                   f"counts -> {best[1]} threads")
                except Exception as ex:      # extras never cost the headline line
                    out["extras"]["cpu_torch_restatement_error"] = f"{type(ex).__name__}: {ex}"
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
