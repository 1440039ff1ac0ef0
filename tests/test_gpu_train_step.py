"""GPU tests of the graph-replayable training step (tsb_train_step, tssplat_b200.train_step.GeometryStep): pinned to
the reference's own AdamUniform trajectory, against the eager Python loop (SmoothnessBarrierEnergy + AdamUniform +
LR scheduler) in staged and global-gather mode, graph replay against eager stepping bitwise, and its interplay with
the autograd surface and its errors."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from _helpers import GOLDEN, COracle
from tssplat_b200.mesh import make_pack, perturb

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mods():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from tssplat_b200 import _capi, train_step
    from tssplat_b200.energies import SmoothnessBarrierEnergy
    from tssplat_b200.optimizer import AdamUniform
    return _capi, train_step, SmoothnessBarrierEnergy, AdamUniform


def _cosine(T):
    return lambda o: torch.optim.lr_scheduler.CosineAnnealingLR(o, T, eta_min=1e-4)


def _python_loop(Energy, AdamUniform, verts, tets, flags, x0, n_steps, W, opt_kw, T):
    """What trainer.py:71-133 does around the energy, with loss = reg_loss + (x * W).sum() as the image term."""
    eng = Energy(verts, tets, flags)
    x = torch.nn.Parameter(torch.from_numpy(x0).cuda())
    opt = AdamUniform([x], **opt_kw)
    sched = _cosine(T)(opt)
    regs = []
    for it in range(n_steps):
        c1, c2 = eng.coeff_scheduler(it)
        reg = eng(x, it, c1, c2)
        loss = reg + (x * W).sum() if W is not None else reg
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        sched.step()
        regs.append(reg.detach().clone())
    torch.cuda.synchronize()
    return x.detach(), torch.stack(regs).cpu().numpy().astype(np.float64), opt.state[x]


def _compare_with_python_loop(mods, verts, tets, x0, n_steps, order_iter, opt_kw, graph_steps=32, min_replays=1):
    _capi, ts, Energy, AdamUniform = mods
    flags = dict(smooth_eng_coeff=2e-4 / 4, barrier_coeff=2e-4, increase_order_iter=order_iter)
    W = (torch.randn(x0.shape, generator=torch.Generator().manual_seed(5)) * 1e-3).cuda()   # fixed linear image loss
    x_py, regs, st_py = _python_loop(Energy, AdamUniform, verts, tets, flags, x0, n_steps, W, opt_kw, n_steps)

    eng = Energy(verts, tets, flags)
    x = torch.from_numpy(x0).cuda()
    gs = ts.GeometryStep(eng, x, n_steps, lr_scheduler=_cosine(n_steps), graph_steps=graph_steps, **opt_kw)
    gs.run(n_steps, grad_ext=W)
    torch.cuda.synchronize()
    assert len(gs._graphs) >= min_replays
    hist = gs.history().cpu().numpy().astype(np.float64)
    assert hist.shape == (n_steps, 4) and gs.state["step"] == n_steps
    rel = np.abs(hist[:, 0] - regs) / np.abs(regs)
    assert rel.max() <= 1e-5, (rel.max(), int(rel.argmax()))
    disp = float((x_py - torch.from_numpy(x0).cuda()).abs().max())
    drift = float((x - x_py).abs().max())
    assert drift <= 1e-4 * disp, (drift, disp)
    assert not gs.schedule_overrun()
    return gs, eng, x


def test_pinned_to_reference_adam_uniform(mods):
    """c1 = c2 = 0 and the fixture's gradients as grad_ext: the trajectory of the reference's own utils/optimizer.py
    AdamUniform (tests/golden/make_ref_fixtures.py), eagerly and through one-step graph replays."""
    _capi, ts, Energy, _ = mods
    fix = np.load(os.path.join(GOLDEN, "ref_fixtures.npz"))
    lr, b1, b2, m0, m1, it = (float(v) for v in fix["adam/hyper"])
    base = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1]], dtype=np.float32)
    verts = np.concatenate([base + np.float32(3 * i) for i in range(150)])          # 150 disjoint tets, 600 vertices
    tets = np.arange(600, dtype=np.int32).reshape(150, 4)
    assert verts.shape == fix["adam/p0"].shape
    eng = Energy(verts, tets, dict(smooth_eng_coeff=0.0, barrier_coeff=0.0, increase_order_iter=1000))
    kw = dict(lr=lr, betas=(b1, b2), grad_limit=True, grad_limit_values=[m0, m1], grad_limit_iters=[int(it)])
    grads = [torch.from_numpy(g).cuda() for g in fix["adam/grads"]]
    for mode in ("eager", "graph"):
        x = torch.from_numpy(fix["adam/p0"]).cuda()
        gs = ts.GeometryStep(eng, x, len(grads), graph_steps=1, **kw)
        buf = torch.empty_like(x)
        for k, g in enumerate(grads):
            if mode == "eager":
                gs.step(grad_ext=g)
            else:
                buf.copy_(g)                                  # the captured buffer, rewritten between runs
                gs.run(1, grad_ext=buf)
            want = torch.from_numpy(fix["adam/traj"][k]).cuda()
            assert torch.allclose(x, want, rtol=2e-5, atol=2e-6), (mode, k)
        assert torch.allclose(gs.state["g1"], torch.from_numpy(fix["adam/g1"]).cuda(), rtol=1e-5, atol=1e-7)
        assert torch.allclose(gs.state["g2"], torch.from_numpy(fix["adam/g2"]).cuda(), rtol=1e-5, atol=1e-9)
        assert torch.all(gs.history()[:, 0] == 0)                                   # c1 = c2 = 0
        if mode == "graph":
            assert len(gs._graphs) == 1


def test_against_eager_python_loop_across_order_switch(mods):
    """4 x 1024 pack with inverted tets (barrier active), 120 steps crossing the order switch at iteration 60 and the
    grad_limit switch at 40, CosineAnnealingLR, a linear image term: graph replays + eager remainder vs the Python loop."""
    pack = make_pack(4, 1024, seed=1)
    x0 = perturb(pack, sigma_rel=0.35, seed=1)
    kw = dict(lr=0.2, grad_limit=True, grad_limit_values=[0.01, 0.005], grad_limit_iters=[40])
    gs, _, _ = _compare_with_python_loop(mods, pack.verts, pack.tets, x0, 120, 60, kw, min_replays=2)
    assert set(gs.orders.tolist()) == {2, 4}


def test_graph_replay_equals_eager_bitwise(mods):
    """No inverted tets (no barrier atomics): graph replays and eager steps give bitwise the same x, g1, g2 and
    history; work is left zeroed and the counter equals the steps taken; step 1 (m = 1) equals one step of the Python
    loop bitwise."""
    _capi, ts, Energy, AdamUniform = mods
    pack = make_pack(4, 1024, seed=2)
    x0 = perturb(pack, sigma_rel=0.02, seed=2)
    flags = dict(smooth_eng_coeff=2e-4 / 4, barrier_coeff=2e-4, increase_order_iter=30)
    kw = dict(lr=0.2, grad_limit=True, grad_limit_values=[0.01, 0.005], grad_limit_iters=[20])
    n = 75
    eng = Energy(pack.verts, pack.tets, flags)
    xa, xb = torch.from_numpy(x0).cuda(), torch.from_numpy(x0).cuda()
    a = ts.GeometryStep(eng, xa, n, lr_scheduler=_cosine(n), graph_steps=8, **kw)
    b = ts.GeometryStep(eng, xb, n, lr_scheduler=_cosine(n), graph_steps=8, **kw)
    for _ in range(n):
        a.step()
    b.run(n)
    torch.cuda.synchronize()
    assert len(b._graphs) == 2
    assert torch.equal(xa, xb) and torch.equal(a.state["g1"], b.state["g1"]) and torch.equal(a.state["g2"], b.state["g2"])
    assert torch.equal(a.history(), b.history())
    assert not torch.equal(xa, torch.from_numpy(x0).cuda())
    for s in (a, b):
        assert torch.all(s._work == 0) and int(s._step.item()) == n and s.state["step"] == n
    # step 1 against the eager Python loop
    x_py, regs, st_py = _python_loop(Energy, AdamUniform, pack.verts, pack.tets, flags, x0, 1, None, kw, n)
    xc = torch.from_numpy(x0).cuda()
    c = ts.GeometryStep(eng, xc, n, lr_scheduler=_cosine(n), **kw)
    c.step()
    torch.cuda.synchronize()
    assert torch.equal(xc, x_py) and torch.equal(c.state["g1"], st_py["g1"]) and torch.equal(c.state["g2"], st_py["g2"])
    assert float(c.history()[0, 0]) == float(regs[0]) and float(c.history()[0, 3]) == 1.0


def test_global_gather_mode(mods):
    """The reference's a.veg (4500 vertices in one component: the kernel's global-gather mode) against the Python loop."""
    d = np.load(os.path.join(GOLDEN, "a_veg_mesh.npz"))
    verts, tets = d["verts"].astype(np.float32), d["tets"].astype(np.int32)
    x0 = perturb(verts, tets, 0.35, 1)
    kw = dict(lr=0.2, grad_limit=True, grad_limit_values=[0.01, 0.005], grad_limit_iters=[3])
    gs, eng, _ = _compare_with_python_loop(mods, verts, tets, x0, 12, 6, kw, graph_steps=4, min_replays=2)
    assert eng.tet_sp.info["mode_global"] == 1


def test_autograd_surface_after_run_and_errors(mods):
    """After run(): forward + backward of SmoothnessBarrierEnergy on the moved x agree with the fp64 C oracle, also for
    a forward taken before the run (no stale cached gradient).  Running past n_steps raises; tsb_train_step rejects bad
    arguments with TSB_E_INVALID; a device counter past the schedule changes nothing and raises the flag."""
    _capi, ts, Energy, _ = mods
    pack = make_pack(2, 1024, seed=3)
    x0 = perturb(pack, sigma_rel=0.3, seed=4)
    flags = dict(smooth_eng_coeff=2e-4 / 2, barrier_coeff=2e-4, increase_order_iter=1000)
    eng = Energy(pack.verts, pack.tets, flags)
    x = torch.nn.Parameter(torch.from_numpy(x0).cuda())
    gs = ts.GeometryStep(eng, x.data, 10, lr=0.2, graph_steps=2)
    c1, c2 = eng.coeff_scheduler(5)
    e_before = eng(x, 5, c1, c2)                                 # caches the gradient at x0
    gs.run(5)
    e_before.backward()                                          # must not hand back the gradient at x0
    e_after = eng(x, 5, c1, c2)
    g_before = x.grad.clone()
    x.grad = None
    e_after.backward()
    torch.cuda.synchronize()
    x_np = x.detach().cpu().numpy()
    assert not np.array_equal(x_np, x0)
    eo, _, go = COracle(pack.verts, pack.tets).energy_grad(x_np, c1, c2, 2)
    assert abs(float(e_after.detach()) - eo) <= 1e-5 * abs(eo)
    for g in (g_before, x.grad):
        assert np.linalg.norm(g.cpu().numpy().astype(np.float64) - go) <= 1e-5 * np.linalg.norm(go)

    gs.run(5)
    with pytest.raises(RuntimeError):
        gs.step()
    with pytest.raises(RuntimeError):
        gs.run(1)
    with pytest.raises(ValueError):
        gs.run(-1)
    with pytest.raises(RuntimeError):
        ts.GeometryStep(eng, torch.zeros(7, device="cuda"), 5)
    with pytest.raises(RuntimeError):
        ts.GeometryStep(eng, x.data, 5).step(grad_ext=torch.zeros(3, device="cuda"))
    torch.cuda.synchronize()
    assert gs.state["step"] == 10 and int(gs._step.item()) == 10 and not gs.schedule_overrun()

    # the C ABI: argument checks, then a counter past the schedule
    lib, h, st = _capi.lib, eng.tet_sp._h, gs._st
    stream = torch.cuda.current_stream().cuda_stream
    xp = x.data.data_ptr()
    assert lib.tsb_train_step(None, xp, None, 1.0, 1.0, 2, C.byref(st), stream) == _capi.TSB_E_INVALID
    assert lib.tsb_train_step(h, None, None, 1.0, 1.0, 2, C.byref(st), stream) == _capi.TSB_E_INVALID
    assert lib.tsb_train_step(h, xp, None, 1.0, 1.0, 2, None, stream) == _capi.TSB_E_INVALID
    assert lib.tsb_train_step(h, xp, None, 1.0, 1.0, 3, C.byref(st), stream) == _capi.TSB_E_INVALID
    for field, val in (("n_steps", 0), ("beta1", 1.0), ("beta2", -0.5), ("work", None), ("schedule", None)):
        bad = _capi.tsb_train_state_t.from_buffer_copy(st)
        setattr(bad, field, val)
        assert lib.tsb_train_step(h, xp, None, 1.0, 1.0, 2, C.byref(bad), stream) == _capi.TSB_E_INVALID, field
    before = [t.clone() for t in (x.data, gs.state["g1"], gs.state["g2"], gs._history)]
    assert lib.tsb_train_step(h, xp, None, 1.0, 1.0, 2, C.byref(st), stream) == _capi.TSB_OK
    torch.cuda.synchronize()
    after = (x.data, gs.state["g1"], gs.state["g2"], gs._history)
    assert all(torch.equal(u, v) for u, v in zip(before, after))
    assert gs.schedule_overrun() and int(gs._step.item()) == 10
