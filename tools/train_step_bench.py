"""Energy-only trainer loop, eager Python (the loop of tools/energy_only_loop.py: SmoothnessBarrierEnergy + AdamUniform
+ CosineAnnealingLR, one autograd step per iteration) against GeometryStep.run (tsb_train_step: the same step as
captured CUDA graphs of device-scheduled launches), in one process, timed with CUDA events and alternated A/B.

    python tools/train_step_bench.py [--spheres 64 1024] [--iters 1500] [--reps 3] [--out FILE.json]

64 x 4096 spheres keep the step's working set (23 MB of plan data plus x, grad and the moments) in the 126 MB L2 from
one step to the next (L2-warm); 1024 x 4096 (16 times as much) streams it from HBM every step (HBM-cold).  Prints
it/s and us/step of both loops, the loss after the last step of each, and the GPU's name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tssplat_b200.energies import SmoothnessBarrierEnergy  # noqa: E402
from tssplat_b200.mesh import make_pack, perturb  # noqa: E402
from tssplat_b200.optimizer import AdamUniform  # noqa: E402
from tssplat_b200.train_step import GeometryStep  # noqa: E402


def gpu_identity():
    """Name and power limit of cuda:0 (a read-only nvidia-smi query)."""
    out = {"name": torch.cuda.get_device_name(0), "power_limit": "unknown"}
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        if r.returncode == 0 and r.stdout.strip():
            name, power, clk = (s.strip() for s in r.stdout.strip().splitlines()[0].split(","))
            out.update(name=name, power_limit=power, max_sm_clock=clk)
    except (OSError, subprocess.TimeoutExpired):
        pass
    return out


def bench(spheres, iters, reps):
    pack = make_pack(spheres, 4096, seed=0, unique=8)
    flags = dict(smooth_eng_coeff=2e-4 / spheres, barrier_coeff=2e-4, increase_order_iter=1000)   # as energy_only_loop
    opt_kw = dict(grad_limit=True, grad_limit_values=[0.01, 0.01], grad_limit_iters=[1500], lr=0.2)
    x0 = torch.from_numpy(perturb(pack, sigma_rel=0.35, seed=1)).cuda()
    eng = SmoothnessBarrierEnergy(pack.verts, pack.tets, flags)
    tet_v = torch.nn.Parameter(x0.clone())
    xg = x0.clone()
    gs = GeometryStep(eng, xg, iters, lr_scheduler=lambda o: torch.optim.lr_scheduler.CosineAnnealingLR(o, T_max=iters),
                      **opt_kw)

    def eager():                                     # tools/energy_only_loop.py:27-43, same pieces
        tet_v.data.copy_(x0)
        opt = AdamUniform([tet_v], **opt_kw)
        sched = torch.optim.lr_scheduler.CosineAnnealingLR(opt, T_max=iters)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for it in range(iters):
            c1, c2 = eng.coeff_scheduler(it)
            reg_loss = eng(tet_v, it, c1, c2)
            opt.zero_grad(set_to_none=True)
            reg_loss.backward()
            opt.step()
            sched.step()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) * 1e-3, float(reg_loss.detach())

    def graphed():
        xg.copy_(x0)
        gs.reset()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        gs.run(iters)
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) * 1e-3, float(gs.history()[-1, 0])

    eager()                                          # warm-up: module loads, autograd, the graphs' capture
    graphed()
    t_e, t_g, l_e, l_g = [], [], [], []
    for _ in range(reps):                            # alternated A/B
        t, loss = eager()
        t_e.append(t)
        l_e.append(loss)
        t, loss = graphed()
        t_g.append(t)
        l_g.append(loss)
    me, mg = float(np.median(t_e)), float(np.median(t_g))
    return {
        "spheres": spheres, "tets_per_sphere": 4096, "vertices": int(pack.n), "iters": iters, "reps": reps,
        "cache_state": "L2-warm" if spheres <= 64 else "HBM-cold",
        "eager_it_s": iters / me, "eager_us_per_step": me / iters * 1e6, "eager_seconds": t_e,
        "graph_it_s": iters / mg, "graph_us_per_step": mg / iters * 1e6, "graph_seconds": t_g,
        "speedup": me / mg, "eager_last_loss": l_e[-1], "graph_last_loss": l_g[-1],
        "eager_last_loss_per_rep": l_e, "graph_last_loss_per_rep": l_g,
        "graph_steps": gs.graph_steps, "mode_global": int(eng.tet_sp.info["mode_global"]),
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--spheres", type=int, nargs="+", default=[64, 1024])
    ap.add_argument("--iters", type=int, default=1500)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the results as JSON to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("train_step_bench needs a CUDA device")
    gpu = gpu_identity()
    print(f"GPU: {gpu['name']}, power limit {gpu['power_limit']}")
    rows = []
    for s in args.spheres:
        r = bench(s, args.iters, args.reps)
        rows.append(r)
        print(f"{s:5d} spheres x 4096 ({r['cache_state']}): eager {r['eager_it_s']:8.0f} it/s ({r['eager_us_per_step']:6.1f} us/step) | "
              f"GeometryStep.run {r['graph_it_s']:8.0f} it/s ({r['graph_us_per_step']:6.1f} us/step) | x{r['speedup']:.2f} | "
              f"last loss eager {r['eager_last_loss']:.6g} graph {r['graph_last_loss']:.6g}", flush=True)
    res = {"gpu": gpu, "results": rows}
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
