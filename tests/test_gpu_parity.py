"""GPU parity tests (run with -m gpu on a B200): the CUDA path, called through the C ABI, against
the fp64 C oracle, the committed golden fixtures and size-independent properties.

Tolerance: BASELINE.json's north_star asks for outputs within 1e-5 relative (fp32) of the
reference; here relative energy error <= 1e-5 and relative gradient L2 error <= 1e-5 against the
fp64 restatement (the reference itself cannot run here; parity vs its binary is unpinned)."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from _helpers import GOLDEN, COracle
from tssplat_b200.mesh import concat_spheres, make_pack, make_tet_sphere, perturb

pytestmark = pytest.mark.gpu
REL = 1e-5


@pytest.fixture(scope="module")
def ext():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from tssplat_b200 import tet_spheres_ext
    return tet_spheres_ext


def _check(ext, verts, tets, x_np, c1, c2, order, gradH=1.0, scale=0, rel=REL, **kw):
    sp = ext.TetSpheres(np.ascontiguousarray(verts, dtype=np.float32).reshape(-1),
                        np.ascontiguousarray(tets, dtype=np.int32).reshape(-1), laplacian_scale=scale, **kw)
    x = torch.from_numpy(np.asarray(x_np, dtype=np.float32)).cuda()
    e, g = sp.energy_grad(x, c1, c2, order, gradH)
    torch.cuda.synchronize()
    eo, terms, go = COracle(verts, tets, scale).energy_grad(x_np, c1, c2, order, gradH=gradH)
    e = e.cpu().numpy().astype(np.float64)
    g = g.cpu().numpy().astype(np.float64)
    assert not np.isnan(g).any()
    assert abs(e[0] - eo) <= rel * max(abs(eo), 1e-30), (e[0], eo)
    assert abs(e[1] - terms[0]) <= rel * max(abs(terms[0]), 1e-30)
    assert abs(e[2] - terms[1]) <= rel * max(abs(terms[1]), 1e-30)
    assert np.linalg.norm(g - go) <= rel * np.linalg.norm(go), np.linalg.norm(g - go) / np.linalg.norm(go)
    return sp, e, g


VARIANTS = [dict(), dict(warps_per_cta=8), dict(force_global=True), dict(warps_per_cta=8, force_global=True),
            dict(ring_slots=4)]


@pytest.mark.parametrize("kw", VARIANTS, ids=lambda k: "-".join(f"{a}{b}" for a, b in k.items()) or "default")
@pytest.mark.parametrize("sig,order", [(0.02, 2), (0.35, 2), (0.35, 4)])
def test_parity_small_pack(ext, kw, sig, order):
    """Every kernel variant (16 / 8 warps per CTA, components staged in shared memory / global gathers)."""
    pack = make_pack(3, 1024, seed=1)
    _check(ext, pack.verts, pack.tets, perturb(pack, sigma_rel=sig, seed=1), 2e-4 / 3, 2e-4, order, gradH=0.7, **kw)


def test_parity_coefficient_range_and_scale(ext):
    """c multipliers 1 and 16 (energies/smooth_barrier.py:50-54) and the scaled Laplacian."""
    pack = make_pack(2, 1500, seed=4)                     # ragged: 1500 is not a block multiple
    x = perturb(pack, sigma_rel=0.35, seed=3)
    for m in (1.0, 16.0):
        _check(ext, pack.verts, pack.tets, x, 2e-4 / 2 * m, 2e-4 * m, 2)
    _check(ext, pack.verts, pack.tets, x, 1e-3, 1e-3, 4, scale=1)


def test_parity_16_spheres(ext):
    """BASELINE.json configs[1]: 16 tet-spheres, fused energy+grad kernel only, fp32."""
    pack = make_pack(16, 4096, seed=0, unique=4)
    for sig, order in ((0.02, 2), (0.35, 4)):
        _check(ext, pack.verts, pack.tets, perturb(pack, sigma_rel=sig, seed=1), 2e-4 / 16, 2e-4, order)


def test_golden_fixtures(ext):
    gold = np.load(os.path.join(GOLDEN, "golden_energy.npz"))
    d = np.load(os.path.join(GOLDEN, "a_veg_mesh.npz"))
    pk = make_pack(3, 1024, seed=1)
    meshes = {"a_veg": (d["verts"], d["tets"]), "pack3x1024": (pk.verts.astype(np.float64), pk.tets)}
    cases = {"benign_o2": (0.02, 0, 2, 2e-4, 2e-4, 1.0), "inverted_o2": (0.35, 1, 2, 3.2e-3, 3.2e-3, 0.5),
             "inverted_o4": (0.35, 1, 4, 2e-4, 2e-4, 1.0)}
    for mname, (v, t) in meshes.items():
        for cname, (sig, seed, order, c1, c2, gh) in cases.items():
            x = perturb(v, t, sig, seed)
            _, e, g = _check(ext, v, t, x, c1, c2, order, gradH=gh)
            k = f"{mname}/{cname}"
            assert e[0] == pytest.approx(float(gold[k + "/energy"]), rel=REL)
            assert np.linalg.norm(g) == pytest.approx(float(gold[k + "/grad_l2"]), rel=REL)
            samp = g[:: max(1, len(g) // 64)][:64]
            assert np.abs(samp - gold[k + "/grad_sample"]).max() <= 1e-5 * np.abs(gold[k + "/grad_sample"]).max()


def test_known_answers(ext):
    v, t = make_tet_sphere(1003, 512)
    v = v.astype(np.float32)
    sp = ext.TetSpheres(v.reshape(-1), t.reshape(-1))

    def run(x, c1=1.0, c2=1.0, order=2):
        e, g = sp.energy_grad(torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).cuda(), c1, c2, order)
        return e.cpu().numpy().astype(np.float64), g.cpu().numpy()
    e, g = run(v)                                          # rest state
    assert abs(e[0]) < 1e-7 and np.abs(g).max() < 1e-4
    A = np.array([[1.1, 0.2, 0.0], [0.0, 0.9, 0.1], [0.1, 0.0, 1.2]])
    e, _ = run(v.astype(np.float64) @ A.T + 0.3)           # affine map: L F = 0, det > 0
    assert abs(e[0]) < 1e-6 * len(t)
    xr = v * np.array([1, 1, -1], dtype=np.float32)        # reflection: det F = -1 in every tet
    for order in (2, 4):
        e, _ = run(xr, 1.0, 0.25, order)
        assert e[2] == pytest.approx(len(t), rel=1e-5) and e[0] == pytest.approx(0.25 * len(t), rel=1e-5)


def test_tiny_and_unreferenced(ext):
    v1 = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1], [9, 9, 9]], dtype=np.float32)  # vertex 4 unused
    t1 = np.array([[0, 1, 2, 3]], dtype=np.int32)
    x = v1 * np.array([1, 1, -1.5], dtype=np.float32)
    sp, e, g = _check(ext, v1, t1, x, 1.0, 1.0, 2)
    assert e[1] == 0.0 and e[2] == pytest.approx(2.25, rel=1e-6) and np.all(g[4] == 0.0)
    v2 = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1], [1, 1, 1]], dtype=np.float32)
    t2 = np.array([[0, 1, 2, 3], [1, 3, 2, 4]], dtype=np.int32)
    _check(ext, v2, t2, perturb(v2, t2, 0.3, 1), 0.7, 0.3, 2)


def test_deterministic_and_reentrant_handles(ext):
    """No inverted tet: every gradient row has one writer and the energies are folded in a fixed order, so
    results are bitwise repeatable.  With inverted tets the barrier gradient arrives through
    red.global.add.f32 (BASELINE north_star: "per-vertex atomic scatter-add"): repeatable to rounding only."""
    pack = make_pack(4, 2048, seed=6)
    a = ext.TetSpheres(pack.verts.reshape(-1), pack.tets.reshape(-1))
    b = ext.TetSpheres(pack.verts.reshape(-1), pack.tets.reshape(-1), warps_per_cta=8)
    x = torch.from_numpy(perturb(pack, sigma_rel=0.02, seed=5)).cuda()
    e1, g1 = a.energy_grad(x, 1e-4, 2e-4, 2)
    eb, gb = b.energy_grad(x, 1e-4, 2e-4, 2)
    e2, g2 = a.energy_grad(x, 1e-4, 2e-4, 2)
    torch.cuda.synchronize()
    assert float(e1[2]) == 0.0                                            # no inverted tet
    assert torch.equal(g1, g2) and torch.equal(e1, e2)                  # bitwise repeatable
    assert torch.allclose(g1, gb, rtol=1e-4, atol=1e-7)                  # other work split: same answer
    xi = torch.from_numpy(perturb(pack, sigma_rel=0.35, seed=5)).cuda()
    e3, g3 = a.energy_grad(xi, 1e-4, 2e-4, 2)
    e4, g4 = a.energy_grad(xi, 1e-4, 2e-4, 2)
    torch.cuda.synchronize()
    assert float(e3[2]) > 0.0 and torch.equal(e3, e4)                    # energies: fixed order even with inversions
    assert float((g3 - g4).norm()) <= 1e-6 * float(g3.norm())
    del a, b


def test_autograd_surface(ext):
    """The reference's Python surface: SmoothnessBarrierEnergy / SmoothnessBarrierFunc
    (energies/smooth_barrier.py:9-67) as trainer.py / tetmesh_geometry.py use it."""
    from tssplat_b200.energies import SmoothnessBarrierEnergy
    pack = make_pack(3, 1024, seed=2)
    flags = dict(smooth_eng_coeff=2e-4 / 3, barrier_coeff=2e-4, increase_order_iter=1000)
    eng = SmoothnessBarrierEnergy(pack.verts, pack.tets, flags)
    x_np = perturb(pack, sigma_rel=0.35, seed=2)
    orc = COracle(pack.verts, pack.tets)
    for it in (10, 1500):                                    # order 2, then order 4 (smooth_barrier.py:61-63)
        tet_v = torch.nn.Parameter(torch.from_numpy(x_np).cuda())
        c1, c2 = eng.coeff_scheduler(it)
        e = eng(tet_v, it, c1, c2)
        assert e.dim() == 0 and e.is_cuda
        loss = 3.0 * e + 1.0                                 # grad_output = 3 arrives as a CUDA scalar
        loss.backward()
        order = 4 if it > 1000 else 2
        eo, _, go = orc.energy_grad(x_np, c1, c2, order, gradH=3.0)
        assert float(e.detach()) == pytest.approx(eo, rel=REL)
        g = tet_v.grad.cpu().numpy().astype(np.float64)
        assert tet_v.grad.shape == (pack.n, 3) and np.linalg.norm(g - go) <= REL * np.linalg.norm(go)
    # stale-cache protection: modify x in place between forward and backward -> backward recomputes
    tet_v = torch.nn.Parameter(torch.from_numpy(x_np).cuda())
    e = eng(tet_v, 10, 1e-4, 2e-4)
    with torch.no_grad():
        tet_v.mul_(1.0)                                      # bumps the version counter
    g_direct = ext.backward(torch.tensor(1.0), tet_v, eng.tet_sp, 1e-4, 2e-4, 2)   # CPU grad_output, like the reference
    _, _, go = orc.energy_grad(x_np, 1e-4, 2e-4, 2)
    assert np.linalg.norm(g_direct.cpu().numpy() - go) <= REL * np.linalg.norm(go)
    # reference-style CPU scalar on request; no-grad forward skips the gradient
    ext.return_cpu_scalar = True
    try:
        with torch.no_grad():
            e_cpu = ext.forward(tet_v.detach(), eng.tet_sp, 1e-4, 2e-4, 2)
        assert not e_cpu.is_cuda and e_cpu.dim() == 0
    finally:
        ext.return_cpu_scalar = False
    assert ext.random_x(eng.tet_sp).shape == (pack.n, 3)


def test_host_buffer_entry_point(ext):
    """tsb_energy_grad_host: host x in, host energy/grad out, async on the current stream."""
    pack = make_pack(3, 1024, seed=5)
    x_np = perturb(pack, sigma_rel=0.35, seed=4)
    sp = ext.TetSpheres(pack.verts.reshape(-1), pack.tets.reshape(-1))
    x_host = torch.from_numpy(x_np).pin_memory()
    g_host = torch.empty((pack.n, 3), dtype=torch.float32).pin_memory()
    e_host = torch.empty(3, dtype=torch.float32).pin_memory()
    ext.energy_grad_host(sp, x_host, 1e-4, 2e-4, 4, 0.5, e_host, g_host)
    torch.cuda.synchronize()
    eo, terms, go = COracle(pack.verts, pack.tets).energy_grad(x_np, 1e-4, 2e-4, 4, gradH=0.5)
    assert float(e_host[0]) == pytest.approx(eo, rel=REL) and float(e_host[2]) == pytest.approx(terms[1], rel=REL)
    assert np.linalg.norm(g_host.numpy() - go) <= REL * np.linalg.norm(go)
    ext.energy_grad_host(sp, x_host, 1e-4, 2e-4, 4, 0.5, e_host, None)          # energy only
    torch.cuda.synchronize()
    assert float(e_host[0]) == pytest.approx(eo, rel=REL)
    with pytest.raises(RuntimeError):
        ext.energy_grad_host(sp, x_host[:-1], 1e-4, 2e-4, 4, 0.5, e_host, g_host)
    # pageable host buffers (no device alias for the energy, staged copies) give the same answer
    x_pg, g_pg, e_pg = torch.from_numpy(x_np.copy()), torch.zeros((pack.n, 3)), torch.zeros(3)
    ext.energy_grad_host(sp, x_pg, 1e-4, 2e-4, 4, 0.5, e_pg, g_pg)
    torch.cuda.synchronize()
    assert float(e_pg[0]) == pytest.approx(float(e_host[0]), rel=1e-6)
    assert (g_pg - g_host).norm() <= 1e-6 * g_host.norm()      # inverted tets: atomics, equal to rounding
    # a pipelined burst of calls with different inputs: every call's outputs belong to its own input
    xs = [torch.from_numpy(perturb(pack, sigma_rel=0.01 * (i + 1), seed=10 + i)).pin_memory() for i in range(6)]
    gs = [torch.empty((pack.n, 3)).pin_memory() for _ in xs]
    es = [torch.empty(3).pin_memory() for _ in xs]
    for xi, gi, ei in zip(xs, gs, es):
        ext.energy_grad_host(sp, xi, 1e-4, 2e-4, 2, 1.0, ei, gi)
    torch.cuda.synchronize()
    for xi, gi, ei in zip(xs, gs, es):
        e1, g1 = sp.energy_grad(xi.cuda(), 1e-4, 2e-4, 2)
        assert float(ei[0]) == pytest.approx(float(e1[0]), rel=1e-6)
        assert (gi - g1.cpu()).norm() <= 1e-6 * g1.norm().cpu()


def test_construct_from_veg_file(ext, tmp_path):
    """TetSpheres(filename) (tet_spheres.cpp:108-117,233) without libpgo: the .veg reader feeds tsb_create."""
    from tssplat_b200.mesh import save_veg
    v, t = make_tet_sphere(1007, 300)
    path = str(tmp_path / "sphere.veg")
    save_veg(path, v, t)
    sp = ext.TetSpheres(path)
    assert sp.n == len(v) and sp.nele == len(t)
    x_np = perturb(v, t, 0.3, 2)
    e, g = sp.energy_grad(torch.from_numpy(x_np).cuda(), 1e-3, 1e-3, 2)
    eo, _, go = COracle(v.astype(np.float32), t).energy_grad(x_np, 1e-3, 1e-3, 2)
    assert float(e[0]) == pytest.approx(eo, rel=REL)
    assert np.linalg.norm(g.cpu().numpy() - go) <= REL * np.linalg.norm(go)


def test_error_behaviour(ext):
    v, t = make_tet_sphere(1005, 128)
    sp = ext.TetSpheres(v.astype(np.float32).reshape(-1), t.reshape(-1))
    x = torch.from_numpy(v.astype(np.float32)).cuda()
    with pytest.raises(RuntimeError, match="order"):
        sp.energy_grad(x, 1.0, 1.0, 3)
    with pytest.raises(RuntimeError):
        sp.energy_grad(x.double(), 1.0, 1.0, 2)
    with pytest.raises(RuntimeError):
        sp.energy_grad(x.cpu(), 1.0, 1.0, 2)
    with pytest.raises(RuntimeError):
        sp.energy_grad(x[:-1], 1.0, 1.0, 2)
    with pytest.raises(RuntimeError, match="zero rest volume"):
        ext.TetSpheres(np.zeros(12, dtype=np.float32), np.array([0, 1, 2, 3], dtype=np.int32))
    with pytest.raises(RuntimeError):
        ext.TetSpheres(v.astype(np.float64).reshape(-1), t.reshape(-1))           # wrong dtype


def test_full_size_properties_64_spheres(ext):
    """BASELINE.json's headline size (64 x 4096 tets): oracle parity plus properties that do not
    need an oracle -- rigid-motion invariance, zero net force per sphere, block-diagonality."""
    pack = make_pack(64, 4096, seed=0, unique=8)
    x_np = perturb(pack, sigma_rel=0.35, seed=1)
    c1, c2 = 2e-4 / 64, 2e-4
    sp, e, g = _check(ext, pack.verts, pack.tets, x_np, c1, c2, 2)
    # zero net force on every sphere (translation invariance)
    for s in range(pack.num_spheres):
        v0, v1 = pack.vert_offsets[s], pack.vert_offsets[s + 1]
        assert np.abs(g[v0:v1].sum(axis=0)).max() <= 2e-4 * np.abs(g[v0:v1]).sum(axis=0).max()
    # rigid motion leaves the energy unchanged and rotates the gradient
    q, _ = np.linalg.qr(np.random.default_rng(0).normal(size=(3, 3)))
    if np.linalg.det(q) < 0:
        q[:, 0] = -q[:, 0]
    xr = (x_np.astype(np.float64) @ q.T + np.array([0.3, -0.2, 0.1])).astype(np.float32)
    e2, g2 = sp.energy_grad(torch.from_numpy(xr).cuda(), c1, c2, 2)
    assert float(e2[0]) == pytest.approx(e[0], rel=2e-5)
    g2 = g2.cpu().numpy().astype(np.float64)
    assert np.linalg.norm(g2 - g @ q.T) <= 5e-5 * np.linalg.norm(g)
    # block-diagonality: spheres 10..13 as their own handle give the same gradient slice
    sub = pack.slice_spheres(10, 14)
    v0, v1 = int(pack.vert_offsets[10]), int(pack.vert_offsets[14])
    sps = ext.TetSpheres(sub.verts.reshape(-1), sub.tets.reshape(-1))
    es, gs = sps.energy_grad(torch.from_numpy(x_np[v0:v1]).cuda(), c1, c2, 2)
    assert np.linalg.norm(gs.cpu().numpy() - g[v0:v1]) <= 2e-5 * np.linalg.norm(g[v0:v1])


def test_large_pack_properties_256_spheres(ext):
    """BASELINE configs[3] size on one GPU (256 spheres, 1.05 M tets): parity with the C oracle and
    the oracle-free invariants, on a pack where every persistent CTA walks several components."""
    pack = make_pack(256, 4096, seed=3, unique=8)
    x_np = perturb(pack, sigma_rel=0.35, seed=2)
    c1, c2 = 2e-4 / 256, 2e-4
    sp, e, g = _check(ext, pack.verts, pack.tets, x_np, c1, c2, 4)
    assert sp.info["n_segments"] >= 256 and sp.info["mode_global"] == 0
    x2 = torch.from_numpy(x_np).cuda()
    e2, g2 = sp.energy_grad(x2, c1, c2, 4)
    assert float((torch.from_numpy(g.astype(np.float32)).cuda() - g2).norm()) <= 1e-6 * float(g2.norm())
    forces = np.add.reduceat(g, pack.vert_offsets[:-1].astype(np.int64), axis=0)  # net force per sphere
    scale = np.add.reduceat(np.abs(g), pack.vert_offsets[:-1].astype(np.int64), axis=0)
    assert np.all(np.abs(forces) <= 3e-4 * scale.max(axis=1, keepdims=True))


def test_grad_limit_and_adam_uniform(ext):
    from tssplat_b200 import _capi
    torch.manual_seed(0)
    g = torch.randn(1000, 3, device="cuda") * 0.01
    ref = g.clone()
    ext.grad_limit(g, 0.5, 0.05)                                            # below threshold: untouched
    assert torch.equal(g, ref)
    ext.grad_limit(g, 0.001, 0.05)                                          # scale so that max|g| = s
    assert float(g.abs().max()) == pytest.approx(0.05, rel=1e-6)
    assert torch.allclose(g, ref * (0.05 / ref.abs().max()), rtol=1e-6)
    # AdamUniform.step (utils/optimizer.py:37-89) restated in torch vs the two-launch CUDA version
    n = 5000
    p = torch.randn(n, 3, device="cuda")
    p_ref, g1r, g2r = p.clone(), torch.zeros_like(p), torch.zeros_like(p)
    g1, g2, work = torch.zeros_like(p), torch.zeros_like(p), torch.zeros(4, device="cuda")
    lr, b1, b2, limit = 0.2, 0.9, 0.999, 0.01
    st = torch.cuda.current_stream().cuda_stream
    for step in range(1, 6):
        grad = torch.randn(n, 3, device="cuda") * (0.1 if step != 3 else 10.0)
        g1r.mul_(b1).add_(grad, alpha=1 - b1)
        g2r.mul_(b2).add_(grad.square(), alpha=1 - b2)
        m1, m2 = g1r / (1 - b1 ** step), g2r / (1 - b2 ** step)
        gr = m1 / (1e-8 + m2.sqrt().max())
        s = gr.abs().max()
        if s > limit:
            gr = gr * (limit / s)
        p_ref.sub_(gr, alpha=lr)
        rc = _capi.lib.tsb_adam_uniform_step(p.data_ptr(), grad.data_ptr(), g1.data_ptr(), g2.data_ptr(), p.numel(),
                                             lr, b1, b2, step, limit, work.data_ptr(), st)
        assert rc == 0
    torch.cuda.synchronize()
    assert torch.allclose(p, p_ref, rtol=1e-5, atol=1e-7) and torch.allclose(g1, g1r, rtol=1e-5, atol=1e-6)
    assert torch.allclose(g2, g2r, rtol=1e-5, atol=1e-8)
    assert torch.all(work == 0)


def test_adam_uniform_optimizer_class(ext):
    """tssplat_b200.optimizer.AdamUniform (drop-in for utils/optimizer.py) against a torch restatement
    of the reference's step, incl. the grad_limit schedule, and a short energy-only descent."""
    from tssplat_b200.optimizer import AdamUniform
    torch.manual_seed(1)
    p = torch.nn.Parameter(torch.randn(2000, 3, device="cuda"))
    ref = p.detach().clone()
    g1r, g2r = torch.zeros_like(ref), torch.zeros_like(ref)
    opt = AdamUniform([p], grad_limit=True, grad_limit_values=[0.05, 0.01], grad_limit_iters=[3], lr=0.2)
    lr, b1, b2 = 0.2, 0.9, 0.999
    ptr, cc = 0, 0
    for step in range(1, 7):
        grad = torch.randn_like(ref) * (5.0 if step % 2 else 0.01)
        p.grad = grad.clone()
        opt.step()
        g1r.mul_(b1).add_(grad, alpha=1 - b1)
        g2r.mul_(b2).add_(grad.square(), alpha=1 - b2)
        gr = (g1r / (1 - b1 ** step)) / (1e-8 + (g2r / (1 - b2 ** step)).sqrt().max())
        m = [0.05, 0.01][ptr]
        if ptr < 1 and cc >= 3:
            ptr += 1
        s = gr.abs().max()
        if s > m:
            gr = gr * (m / s)
        ref.sub_(gr, alpha=lr)
        cc += 1
    torch.cuda.synchronize()
    assert torch.allclose(p.detach(), ref, rtol=1e-5, atol=1e-6)
    # descent: the loop the trainer runs around the energy must decrease it
    import os, sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    from energy_only_loop import run
    rate, e0, e1 = run(spheres=2, iters=60)
    assert e1 < 0.5 * e0 and np.isfinite(e1)


def test_bench_input_and_config4_parity(ext):
    """The headline bench input (64 x 4096, sigma = 0.02 h, order 2) and BASELINE configs[4] (1024 spheres,
    4.2 M tets, one GPU) against the fp64 C oracle."""
    pack = make_pack(64, 4096, seed=0, unique=8)
    _check(ext, pack.verts, pack.tets, perturb(pack, sigma_rel=0.02, seed=0), 2e-4 / 64, 2e-4, 2)
    big = make_pack(1024, 4096, seed=0, unique=8)
    sp, e, g = _check(ext, big.verts, big.tets, perturb(big, sigma_rel=0.35, seed=3), 2e-4 / 1024, 2e-4, 2)
    assert sp.info["n_components"] == 1024


def test_bench_dump_outputs(ext, tmp_path):
    """bench.py --dump-outputs: the energy and gradient of the last timed step (one step: the first pack), equal to the
    fp64 C oracle on that pack's input, bitwise the same in a second run, and exactly --steps timed launches."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    S = 64                                                             # bench.py's default pack
    for run in ("a", "b"):
        cmd = [sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", "1", "--warmup", "3",
               "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / run)]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-2000:]
        d = json.loads(r.stdout.strip().splitlines()[-1])
        assert d["steps"] == 1 and d["gpu_launches"] == 1
    e, g = np.load(tmp_path / "a" / "energy.npy"), np.load(tmp_path / "a" / "grad.npy")
    assert e.dtype == np.float32 and e.shape == (3,) and g.dtype == np.float32
    assert np.array_equal(e, np.load(tmp_path / "b" / "energy.npy")) and np.array_equal(g, np.load(tmp_path / "b" / "grad.npy"))
    pack = make_pack(S, 4096, seed=0, unique=8)                       # bench.py: rank 0, pack 0
    x_np = perturb(pack, sigma_rel=0.02, seed=0)
    eo, terms, go = COracle(pack.verts, pack.tets).energy_grad(x_np, 2e-4 / S, 2e-4, 2)
    assert g.shape == (pack.n, 3)
    assert abs(float(e[0]) - eo) <= REL * abs(eo) and abs(float(e[1]) - terms[0]) <= REL * abs(terms[0])
    assert np.linalg.norm(g.astype(np.float64) - go) <= REL * np.linalg.norm(go)


def test_reference_pinned_barrier_and_F(ext):
    """Fixtures computed by the reference's own compute_G_matrix (geometry/mesh_utils.py:38-69, imported by
    tests/golden/make_ref_fixtures.py): the kernel's barrier sum equals sum max(-det F_ref, 0)^p."""
    fix = np.load(os.path.join(GOLDEN, "ref_fixtures.npz"))
    d = np.load(os.path.join(GOLDEN, "a_veg_mesh.npz"))
    pk = make_pack(3, 1024, seed=1)
    for name, (v, t) in {"a_veg": (d["verts"].astype(np.float32), d["tets"]), "pack3x1024": (pk.verts, pk.tets)}.items():
        sp = ext.TetSpheres(np.ascontiguousarray(v, dtype=np.float32).reshape(-1), np.ascontiguousarray(t, dtype=np.int32).reshape(-1))
        for case in ("benign", "inverted"):
            x = torch.from_numpy(fix[f"{name}/{case}/x"]).cuda()
            for order in (2, 4):
                e, _ = sp.energy_grad(x, 1.0, 1.0, order, want_grad=False)
                want = float(fix[f"{name}/{case}/barrier_o{order}"])
                assert float(e[2]) == pytest.approx(want, rel=REL, abs=1e-30), (name, case, order)


def test_adam_uniform_matches_reference_class(ext):
    """tssplat_b200.optimizer.AdamUniform and tsb_adam_uniform_step against a trajectory produced by the
    reference's own utils/optimizer.py AdamUniform (fixture: tests/golden/make_ref_fixtures.py)."""
    from tssplat_b200.optimizer import AdamUniform
    fix = np.load(os.path.join(GOLDEN, "ref_fixtures.npz"))
    lr, b1, b2, m0, m1, it = (float(v) for v in fix["adam/hyper"])
    p = torch.nn.Parameter(torch.from_numpy(fix["adam/p0"]).cuda())
    opt = AdamUniform([p], grad_limit=True, grad_limit_values=[m0, m1], grad_limit_iters=[int(it)], lr=lr, betas=(b1, b2))
    for k, g in enumerate(fix["adam/grads"]):
        p.grad = torch.from_numpy(g).cuda()
        opt.step()
        want = torch.from_numpy(fix["adam/traj"][k]).cuda()
        assert torch.allclose(p.detach(), want, rtol=2e-5, atol=2e-6), k
    st = opt.state[p]
    assert torch.allclose(st["g1"], torch.from_numpy(fix["adam/g1"]).cuda(), rtol=1e-5, atol=1e-7)
    assert torch.allclose(st["g2"], torch.from_numpy(fix["adam/g2"]).cuda(), rtol=1e-5, atol=1e-9)


def test_surface_gather_and_vertex_normals(ext):
    """tssplat_b200.surface (tsb_surface_*): forward against normals produced by the reference's own
    _compute_vertex_normal body (fixture), forward + backward against the fp64 torch restatement."""
    from oracle.surface_normals import vertex_normals
    from tssplat_b200.mesh import surface_vf
    from tssplat_b200.surface import SurfaceForwardData, SurfaceNormals
    fix = np.load(os.path.join(GOLDEN, "ref_fixtures.npz"))
    d = np.load(os.path.join(GOLDEN, "a_veg_mesh.npz"))
    pk = make_pack(3, 1024, seed=1)
    for name, t in {"a_veg": d["tets"], "pack3x1024": pk.tets}.items():
        sv, sf = surface_vf(t)
        x_np = fix[name + "/inverted/x"]
        surf = SurfaceNormals(sv, sf, len(x_np))
        tet_v = torch.nn.Parameter(torch.from_numpy(x_np).cuda())
        v_pos, v_nrm = surf(tet_v)
        assert torch.equal(v_pos.detach().cpu(), torch.from_numpy(x_np)[torch.from_numpy(sv)])
        assert np.abs(v_nrm.detach().cpu().numpy() - fix[name + "/v_nrm"]).max() < 2e-6
        # backward: a generic scalar of both outputs
        torch.manual_seed(3)
        wp, wn = torch.randn(len(sv), 3), torch.randn(len(sv), 3)
        (v_pos * wp.cuda()).sum().add((v_nrm * wn.cuda()).sum()).backward()
        x64 = torch.from_numpy(x_np).double().requires_grad_(True)
        p64, n64 = vertex_normals(x64, torch.from_numpy(sv), torch.from_numpy(sf))
        ((p64 * wp.double()).sum() + (n64 * wn.double()).sum()).backward()
        g, go = tet_v.grad.cpu().double(), x64.grad
        assert float((g - go).norm()) <= 1e-5 * float(go.norm())
        assert torch.all(g[np.setdiff1d(np.arange(len(x_np)), sv)] == 0)               # interior vertices: no gradient
        v2, n2 = surf.forward(tet_v)
        assert torch.equal(n2, v_nrm.detach())                                          # bitwise repeatable
        fd = SurfaceForwardData(tet_v, surf, torch.from_numpy(sf).cuda())
        assert torch.equal(fd._compute_vertex_normal().detach(), n2) and fd.t_pos_idx.shape == (len(sf), 3)
    # degenerate fallback: a face of zero area gives (0, 0, 1)
    sv0 = np.array([0, 1, 2], dtype=np.int32)
    flat = SurfaceNormals(sv0, np.array([[0, 1, 2]], dtype=np.int32), 3)
    _, n0 = flat.forward(torch.zeros(3, 3, device="cuda"))
    assert torch.equal(n0.cpu(), torch.tensor([[0.0, 0.0, 1.0]] * 3))


def test_amips_term_default_off(ext):
    """a15: the AMIPS term BASELINE.json names.  The reference has none (SURVEY.md F1), so the checks are the
    fp64 restatements (oracle/tet_energy_oracle.{py,c}), the known answers and "c3 = 0 changes nothing"."""
    pack = make_pack(3, 1024, seed=8)
    v, t = pack.verts, pack.tets
    sp = ext.TetSpheres(v.reshape(-1), t.reshape(-1), enable_amips=True)
    plain = ext.TetSpheres(v.reshape(-1), t.reshape(-1))
    orc = COracle(v, t)
    for sig, order in ((0.05, 2), (0.2, 4)):
        x_np = perturb(pack, sigma_rel=sig, seed=4)
        x = torch.from_numpy(x_np).cuda()
        e, g = sp.energy_grad(x, 2e-4, 3e-4, order, 0.8, c3=1e-4)
        eo, terms, go = orc.energy_grad_ex(x_np, 2e-4, 3e-4, 1e-4, order, gradH=0.8)
        e, g = e.cpu().numpy().astype(np.float64), g.cpu().numpy().astype(np.float64)
        assert e[3] == pytest.approx(terms[2], rel=2e-5) and e[0] == pytest.approx(eo, rel=2e-5)
        assert np.linalg.norm(g - go) <= 2e-5 * np.linalg.norm(go)
        # c3 = 0 on the AMIPS-enabled handle == the plain handle, bit for bit (no inverted tets at sigma 0.05)
        e0, g0 = sp.energy_grad(x, 2e-4, 3e-4, order, 0.8)
        e1, g1 = plain.energy_grad(x, 2e-4, 3e-4, order, 0.8)
        assert torch.equal(e0, e1) and (sig > 0.1 or torch.equal(g0, g1))
    rest = torch.from_numpy(v).cuda()
    e, g = sp.energy_grad(rest, 0.0, 0.0, 2, c3=1.0)                       # rest state: minimum, zero gradient
    assert abs(float(e[3])) < 1e-3 and float(g.abs().max()) < 1e-3
    with pytest.raises(RuntimeError, match="enable_amips"):
        plain.energy_grad(rest, 1.0, 1.0, 2, c3=0.5)


def test_handles_with_different_staging_sizes_coexist(ext):
    """The dynamic shared-memory opt-in is per kernel, not per handle: a small-staging handle created after a
    large one must not shrink it (bench.py keeps 8 packs alive)."""
    big = make_pack(2, 4096, seed=31)
    small = make_pack(3, 512, seed=32)
    a = ext.TetSpheres(big.verts.reshape(-1), big.tets.reshape(-1))
    b = ext.TetSpheres(small.verts.reshape(-1), small.tets.reshape(-1))
    assert a.info["smem_bytes"] > b.info["smem_bytes"]
    xa = torch.from_numpy(perturb(big, sigma_rel=0.3, seed=1)).cuda()
    e, g = a.energy_grad(xa, 1e-4, 2e-4, 2)
    eo, _, go = COracle(big.verts, big.tets).energy_grad(xa.cpu().numpy(), 1e-4, 2e-4, 2)
    assert float(e[0]) == pytest.approx(eo, rel=REL) and np.linalg.norm(g.cpu().numpy() - go) <= REL * np.linalg.norm(go)


def test_surface_extraction_on_gpu_matches_reference(ext):
    """tsb_surface_extract (radix sorts + select + scan on the device) against fixtures produced by the reference's own
    get_surface_vf (geometry/mesh_utils.py:5-35, via tests/golden/make_ref_fixtures.py) and against the numpy
    restatement: identical vertex list, identical triangles in identical order and orientation."""
    from tssplat_b200.mesh import surface_vf, surface_vf_gpu
    fix = np.load(os.path.join(GOLDEN, "ref_fixtures.npz"))
    d = np.load(os.path.join(GOLDEN, "a_veg_mesh.npz"))
    pk = make_pack(3, 1024, seed=1)
    for name, t in {"a_veg": d["tets"], "pack3x1024": pk.tets}.items():
        sv, sf = surface_vf_gpu(t)
        assert np.array_equal(sv, fix[name + "/surface_vid"]) and np.array_equal(sf, fix[name + "/surface_f"])
    # a large pack (64 x 4096), unused vertex ids, a face shared by three tets (dropped like the reference drops it)
    big = make_pack(64, 4096, seed=3, unique=4)
    sv, sf = surface_vf_gpu(big.tets, big.n)
    sv0, sf0 = surface_vf(big.tets)
    assert np.array_equal(sv, sv0) and np.array_equal(sf, sf0)
    odd = np.array([[0, 1, 2, 3], [0, 1, 2, 4], [0, 1, 2, 9], [5, 6, 7, 9]], dtype=np.int32)
    sv, sf = surface_vf_gpu(odd, 12)
    sv0, sf0 = surface_vf(odd)
    assert np.array_equal(sv, sv0) and np.array_equal(sf, sf0)
    sv, sf = surface_vf_gpu(np.zeros((0, 4), dtype=np.int32), 5)
    assert len(sv) == 0 and sf.shape == (0, 3)
    with pytest.raises(RuntimeError, match="out of range"):
        surface_vf_gpu(np.array([[0, 1, 2, 7]], dtype=np.int32), 4)


def test_native_autograd_bridge_matches_python_function(ext):
    """csrc/torch_binding.cpp (C++ torch::autograd::Function over the C ABI) against the Python Function: same
    energies, same gradients, same cache semantics (single use, recompute after parameters changed), CUDA and host
    grad_output; and against the oracle."""
    from tssplat_b200 import energies, native_autograd
    from tssplat_b200.optimizer import AdamUniform
    if not native_autograd.available():
        pytest.skip("C++ autograd bridge not built (python -c 'import __graft_entry__ as g; g.build()')")
    pack = make_pack(3, 1024, seed=7)
    x_np = perturb(pack, sigma_rel=0.35, seed=3)
    eng = energies.SmoothnessBarrierEnergy(pack.verts, pack.tets, dict(smooth_eng_coeff=1e-4, barrier_coeff=2e-4, increase_order_iter=10))
    oracle = COracle(pack.verts, pack.tets)
    try:
        for it, order in ((0, 2), (11, 4)):
            res = {}
            for native in (True, False):
                energies.use_native_autograd = native
                x = torch.from_numpy(x_np).cuda().requires_grad_(True)
                e = eng(x, it, 1e-4, 2e-4)
                (e * 0.5).backward()                                  # CUDA grad_output 0.5
                res[native] = (float(e.detach()), x.grad.clone())
            assert res[True][0] == res[False][0]
            assert (res[True][1] - res[False][1]).norm() <= 1e-6 * res[False][1].norm()
            eo, _, go = oracle.energy_grad(x_np, 1e-4, 2e-4, order, gradH=0.5)
            assert res[True][0] == pytest.approx(eo, rel=REL)
            assert np.linalg.norm(res[True][1].cpu().numpy() - go) <= REL * np.linalg.norm(go)
        energies.use_native_autograd = True
        # flat [3n] input keeps its shape; host-scalar grad_output; second backward recomputes (single-use cache)
        x = torch.from_numpy(x_np.reshape(-1)).cuda().requires_grad_(True)
        e = eng(x, 0, 1e-4, 2e-4)
        g1, = torch.autograd.grad(e, x, grad_outputs=torch.tensor(2.0), retain_graph=True)
        g2, = torch.autograd.grad(e, x, grad_outputs=torch.tensor(2.0, device="cuda"))
        _, _, go = oracle.energy_grad(x_np, 1e-4, 2e-4, 2, gradH=2.0)
        assert g1.shape == x.shape and (g1 - g2).norm() <= 1e-6 * g1.norm()
        assert np.linalg.norm(g1.cpu().numpy().reshape(-1, 3) - go) <= REL * np.linalg.norm(go)
        # parameters changed behind autograd's back between forward and backward: the gradient is recomputed at the new x
        p = torch.nn.Parameter(torch.from_numpy(x_np).cuda())
        opt = AdamUniform([p], lr=0.01)
        e = eng(p, 0, 1e-4, 2e-4)
        p.grad = torch.ones_like(p)
        opt.step()                                                    # p.data moved, p._version did not
        p.grad = None
        e.backward()
        _, _, go = oracle.energy_grad(p.detach().cpu().numpy(), 1e-4, 2e-4, 2)
        assert np.linalg.norm(p.grad.cpu().numpy() - go) <= REL * np.linalg.norm(go)
        # errors surface as exceptions
        with pytest.raises(RuntimeError):
            eng(torch.zeros(5, device="cuda", requires_grad=True), 0, 1e-4, 2e-4)
        # the graph keeps the handle alive: backward after the energy module is gone
        import gc
        eng2 = energies.SmoothnessBarrierEnergy(pack.verts, pack.tets, dict(smooth_eng_coeff=1e-4, barrier_coeff=2e-4, increase_order_iter=10))
        x = torch.from_numpy(x_np).cuda().requires_grad_(True)
        loss = eng2(x, 0, 1e-4, 2e-4) * 3.0
        del eng2
        gc.collect()
        loss.backward()
        _, _, go = oracle.energy_grad(x_np, 1e-4, 2e-4, 2, gradH=3.0)
        assert np.linalg.norm(x.grad.cpu().numpy() - go) <= REL * np.linalg.norm(go)
    finally:
        energies.use_native_autograd = True


def test_randomised_ragged_meshes_on_gpu(ext):
    """The kernel on random ragged, relabelled, interleaved multi-component meshes (unreferenced vertices, components
    of very different sizes) in every variant, against the fp64 C oracle."""
    from test_host_logic import _ragged_mesh
    for seed in range(8):
        rng = np.random.default_rng(100 + seed)
        V, T = _ragged_mesh(rng, int(rng.integers(1, 7)), 1200)
        orc = COracle(V, T)
        for kw in ({}, {"warps_per_cta": 8}, {"force_global": True}):
            sp = ext.TetSpheres(V.reshape(-1), T.reshape(-1), **kw)
            for sig, order in ((0.03, 2), (0.4, 4)):
                x_np = (V + rng.normal(0, sig * 0.2, V.shape)).astype(np.float32)
                e, g = sp.energy_grad(torch.from_numpy(x_np).cuda(), 3e-4, 2e-4, order, 1.3)
                eo, _, go = orc.energy_grad(x_np, 3e-4, 2e-4, order, gradH=1.3)
                assert float(e[0]) == pytest.approx(eo, rel=REL, abs=1e-12), (seed, kw, sig)
                assert np.linalg.norm(g.cpu().numpy() - go) <= REL * max(np.linalg.norm(go), 1e-12), (seed, kw, sig)


def test_thousands_of_tiny_components(ext):
    """2600 twelve-tet components: more segments per CTA (18) than the shared-memory segment table holds (16), many
    staging hand-overs per CTA, every variant."""
    pk = make_pack(2600, 12, seed=3, unique=6)
    orc = COracle(pk.verts, pk.tets)
    rng = np.random.default_rng(0)
    for kw in ({}, {"warps_per_cta": 8}, {"force_global": True}):
        sp = ext.TetSpheres(pk.verts.reshape(-1), pk.tets.reshape(-1), **kw)
        for sig, order in ((0.02, 2), (0.3, 4)):
            x_np = (pk.verts + rng.normal(0, sig, pk.verts.shape)).astype(np.float32)
            e, g = sp.energy_grad(torch.from_numpy(x_np).cuda(), 2e-4, 3e-4, order)
            eo, _, go = orc.energy_grad(x_np, 2e-4, 3e-4, order)
            assert float(e[0]) == pytest.approx(eo, rel=REL), (kw, sig)
            assert np.linalg.norm(g.cpu().numpy() - go) <= REL * np.linalg.norm(go), (kw, sig)
