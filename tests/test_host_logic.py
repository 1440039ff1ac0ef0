"""CPU tests of the product's host logic: the C-ABI library loads and exports what the header
declares, the tile plan is consistent (re-enacted in numpy against the oracle), mesh helpers,
error paths, and loud failure without a GPU."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from _helpers import GOLDEN, ROOT, COracle, build_host_plan, emulate_kernel
from tssplat_b200 import _capi
from tssplat_b200.mesh import (concat_spheres, connected_components, load_veg, make_pack, make_tet_sphere, perturb,
                               save_veg)


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "tssplat_b200.h")).read()
    declared = set(re.findall(r"\b(tsb_[a-z_0-9]+)\s*\(", hdr))
    assert declared == set(_capi.EXPORTED_SYMBOLS)
    for sym in declared:
        assert hasattr(_capi.lib, sym), sym


def test_info_struct_matches_header():
    hdr = open(os.path.join(ROOT, "include", "tssplat_b200.h")).read()
    body = hdr[hdr.index("typedef struct {\n  int32_t n;"):hdr.index("} tsb_info_t;")]
    fields = re.findall(r"int(?:32|64)_t\s+([a-z_]+);", body)
    assert fields == [f for f, _ in _capi.tsb_info_t._fields_]


PLAN_VARIANTS = [dict(nw=16, grid=148), dict(nw=8, grid=5), dict(nw=16, grid=7, force_global=1),
                 dict(nw=8, grid=3, vh_cap=100, area_cap=300),        # components staged in the "whole area" mode
                 dict(nw=16, grid=1), dict(nw=8, grid=296)]


@pytest.mark.parametrize("kw", PLAN_VARIANTS, ids=lambda k: "-".join(f"{a}{b}" for a, b in k.items()))
def test_plan_reenactment_matches_oracle(kw):
    """The product's plan builder (operator rows, bank-aware placement, segments, warp streams) walked in
    numpy exactly as the kernel walks it, against the fp64 C oracle."""
    pack = make_pack(3, 768, seed=2)
    plan = build_host_plan(pack.verts, pack.tets, **kw)
    assert plan["n_components"] == 3 and plan["mode_global"] == kw.get("force_global", 0)
    orc = COracle(pack.verts, pack.tets)
    for sig, order in ((0.02, 2), (0.35, 4)):
        x = perturb(pack, sigma_rel=sig, seed=1)
        E, es, eb, g = emulate_kernel(plan, x, 2e-4, 3e-4, order, gradH=0.7)
        Eo, terms, go = orc.energy_grad(x, 2e-4, 3e-4, order, gradH=0.7)
        assert E == pytest.approx(Eo, rel=2e-6)          # fp32 operator entries, fp64 arithmetic
        assert es == pytest.approx(terms[0], rel=2e-6) and eb == pytest.approx(terms[1], rel=2e-6, abs=1e-300)
        assert np.linalg.norm(g - go) <= 2e-6 * np.linalg.norm(go)


def test_plan_operator_is_the_reference_matrix():
    """The streamed rows are M = G^T L^T L G (tet_spheres.cpp:148) minus its diagonal: rebuild M from the
    stream and compare with the scipy operator of the oracle, entry by entry."""
    from oracle.tet_energy_oracle import ReferenceEnergyOracle
    v, t = make_tet_sphere(1201, 300)
    plan = build_host_plan(v, t, nw=8, grid=3)
    M = ReferenceEnergyOracle(v.astype(np.float32), t).M.tocsr()[0::3, :][:, 0::3].toarray()
    n = len(v)
    R = np.zeros((n, n))
    x = np.zeros((n, 3), dtype=np.float32)
    X = v.astype(np.float32)
    for j in range(n):                                  # column j of the operator = gradient for u = e_j (x-coordinate)
        x[:] = X
        x[j, 0] += 1.0
        _, _, _, g = emulate_kernel(plan, x, 1.0, 0.0, 2)
        R[:, j] = g[:, 0]
    assert np.abs(R - M).max() <= 2e-6 * np.abs(M).max()
    assert np.abs(R.sum(axis=1)).max() <= 1e-4 * np.abs(M).max()        # zero row sums (difference form)


def test_plan_bank_placement_and_slot_colouring():
    """Bank-aware staging: positions are a permutation, every row's columns are spread over the 8 bank
    groups, and the slot assignment keeps the quarter-warp gathers (nearly) conflict free."""
    pack = make_pack(4, 2048, seed=5)
    plan = build_host_plan(pack.verts, pack.tets, nw=16, grid=37)
    assert plan["gather_wf"] <= 1.15 * plan["gather_wf_ideal"]
    for sg in plan["segs"]:
        pos = plan["pos16"][sg["x4off"]:sg["x4off"] + sg["nv"]]
        assert len(set(pos.tolist())) == sg["nv"] and pos.max() < sg["npos"] <= sg["nv"] + 64
        assert np.bincount(pos % 8, minlength=8).min() >= sg["nv"] // 8 - 8


def test_plan_laplacian_scale_and_unreferenced_vertices():
    v, t = make_tet_sphere(1201, 300)
    v = np.concatenate([v, [[5.0, 5.0, 5.0], [6.0, 6.0, 6.0]]])          # two vertices no tet uses
    plan = build_host_plan(v, t, nw=8, grid=4, laplacian_scale=1)
    assert sorted(plan["orphans"].tolist()) == [len(v) - 2, len(v) - 1]
    x = perturb(v, t, 0.3, 7)
    E, _, _, g = emulate_kernel(plan, x, 1e-3, 1e-3, 2)
    Eo, _, go = COracle(v, t, 1).energy_grad(x, 1e-3, 1e-3, 2)
    assert E == pytest.approx(Eo, rel=2e-6)
    assert np.all(g[-2:] == 0.0) and np.all(go[-2:] == 0.0)
    assert np.linalg.norm(g - go) <= 2e-6 * np.linalg.norm(go)


def test_plan_noncontiguous_components():
    """Two spheres whose vertices are interleaved in the caller's numbering (vlist path)."""
    pk = make_pack(2, 400, seed=11)
    n = pk.n
    perm = np.random.default_rng(0).permutation(n)                        # new id of old vertex
    verts = np.empty_like(pk.verts)
    verts[perm] = pk.verts
    tets = perm[pk.tets].astype(np.int32)
    plan = build_host_plan(verts, tets, nw=8, grid=6)
    assert plan["contiguous"] == 0 and plan["n_components"] == 2
    x = perturb(verts, tets, 0.3, 3)
    E, _, _, g = emulate_kernel(plan, x, 1e-3, 2e-3, 4)
    Eo, _, go = COracle(verts, tets).energy_grad(x, 1e-3, 2e-3, 4)
    assert E == pytest.approx(Eo, rel=2e-6) and np.linalg.norm(g - go) <= 2e-6 * np.linalg.norm(go)


def test_plan_real_mesh_a_veg():
    """The reference's only in-tree mesh (tssplat_ext/a.veg, 4500 vertices in one component): too large to
    stage in shared memory, so it runs in the global-gather mode."""
    d = np.load(os.path.join(GOLDEN, "a_veg_mesh.npz"))
    plan = build_host_plan(d["verts"], d["tets"], nw=16, grid=148)
    assert plan["mode_global"] == 1
    x = perturb(d["verts"], d["tets"], 0.35, 1)
    E, es, eb, g = emulate_kernel(plan, x, 3.2e-3, 3.2e-3, 2, gradH=0.5)
    gold = np.load(os.path.join(GOLDEN, "golden_energy.npz"))
    assert E == pytest.approx(float(gold["a_veg/inverted_o2/energy"]), rel=2e-6)
    assert np.linalg.norm(g) == pytest.approx(float(gold["a_veg/inverted_o2/grad_l2"]), rel=2e-6)


def test_tiny_meshes():
    """One tet (no neighbours: smoothness identically 0) and two tets sharing a face."""
    v1 = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1]], dtype=np.float64)
    t1 = np.array([[0, 1, 2, 3]], dtype=np.int32)
    x = (v1 * np.array([1, 1, -1.5])).astype(np.float32)
    E, es, eb, g = emulate_kernel(build_host_plan(v1, t1, nw=8, grid=2), x, 1.0, 1.0, 2)
    assert es == 0.0 and eb == pytest.approx(1.5 ** 2)
    v2 = np.concatenate([v1, [[1.0, 1.0, 1.0]]])
    t2 = np.array([[0, 1, 2, 3], [1, 3, 2, 4]], dtype=np.int32)             # positive orientation
    x2 = perturb(v2, t2, 0.3, 1)
    E2, _, _, g2 = emulate_kernel(build_host_plan(v2, t2, nw=8, grid=2), x2, 0.7, 0.3, 2)
    Eo, _, go = COracle(v2, t2).energy_grad(x2, 0.7, 0.3, 2)
    assert E2 == pytest.approx(Eo, rel=1e-5) and np.abs(g2 - go).max() < 1e-5 * np.abs(go).max()


def _plan_error(v, t):
    with pytest.raises(RuntimeError) as ei:
        build_host_plan(np.asarray(v, dtype=np.float64), np.asarray(t, dtype=np.int32), nw=8, grid=4)
    return str(ei.value)


def test_plan_rejects_bad_meshes():
    v = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1], [1, 1, 1]], dtype=np.float64)
    assert "out of range" in _plan_error(v, [[0, 1, 2, 7]])
    assert "zero rest volume" in _plan_error(np.zeros((4, 3)), [[0, 1, 2, 3]])
    assert "repeats a vertex" in _plan_error(v, [[0, 1, 1, 3]])
    three = [[0, 1, 2, 3], [0, 2, 1, 4], [0, 1, 2, 4]]                     # face (0,1,2) used three times
    vv = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1], [0, 0, -1]], dtype=np.float64)
    assert "non-manifold" in _plan_error(vv, three)


def test_bad_plan_configuration():
    v, t = make_tet_sphere(1202, 64)
    with pytest.raises(RuntimeError):
        build_host_plan(v, t, nw=64, grid=4)            # more warps than the kernel variants have
    with pytest.raises(RuntimeError):
        build_host_plan(v, t, nw=8, grid=0)


def test_veg_round_trip(tmp_path):
    v, t = make_tet_sphere(1203, 200)
    p = str(tmp_path / "m.veg")
    save_veg(p, v, t)
    v2, t2 = load_veg(p)
    assert np.array_equal(t, t2) and np.abs(v - v2).max() < 1e-14
    # the reference's own file (a verbatim excerpt of tssplat_ext/a.veg) reads as the committed a.veg arrays
    va, ta = load_veg(os.path.join(GOLDEN, "a_veg_excerpt.veg"))
    d = np.load(os.path.join(GOLDEN, "a_veg_mesh.npz"))
    inside = d["tets"].max(axis=1) < len(va)
    assert len(va) == 1000 and len(ta) == 133
    assert np.array_equal(ta, d["tets"][inside]) and np.array_equal(va, d["verts"][:len(va)])


def test_surface_extraction_matches_reference_get_surface_vf():
    """tssplat_b200.mesh.surface_vf against fixtures produced by the reference's own get_surface_vf
    (geometry/mesh_utils.py:5-35, imported by tests/golden/make_ref_fixtures.py): identical vertex list,
    identical triangles in identical order and orientation."""
    from tssplat_b200.mesh import surface_vf
    fix = np.load(os.path.join(GOLDEN, "ref_fixtures.npz"))
    d = np.load(os.path.join(GOLDEN, "a_veg_mesh.npz"))
    pk = make_pack(3, 1024, seed=1)
    for name, t in {"a_veg": d["tets"], "pack3x1024": pk.tets}.items():
        sv, sf = surface_vf(t)
        assert np.array_equal(sv, fix[name + "/surface_vid"]) and np.array_equal(sf, fix[name + "/surface_f"])
    sv, sf = surface_vf(d["tets"])
    assert len(sv) == 973 and len(sf) == 1942                      # SURVEY 8c: a.veg surface


def test_npy_sphere_export_round_trip(tmp_path):
    from tssplat_b200.mesh import load_npy_spheres, save_npy_spheres
    pk = make_pack(3, 256, seed=12)
    files = save_npy_spheres(pk, str(tmp_path), "final")
    assert len(files) == 2 + 2 * 3
    e1 = np.load(str(tmp_path / "final_sp1_elem.npy"))
    assert e1.min() == 0 and e1.max() == pk.vert_offsets[2] - pk.vert_offsets[1] - 1     # sphere-local indices
    back = load_npy_spheres(str(tmp_path), "final")
    assert np.array_equal(back.verts, pk.verts) and np.array_equal(back.tets, pk.tets)
    assert np.array_equal(back.vert_offsets, pk.vert_offsets)
    assert np.array_equal(np.load(str(tmp_path / "final_vtx.npy")), pk.verts)


def test_synthetic_pack_properties():
    from oracle.tet_energy_oracle import face_adjacency
    from tssplat_b200.mesh import _signed_volumes
    pk = make_pack(4, 512, seed=9)
    assert pk.nele == 4 * 512 and pk.num_spheres == 4
    assert np.all(_signed_volumes(pk.verts.astype(np.float64), pk.tets.astype(np.int64)) > 0)
    face_adjacency(pk.tets)                                                # manifold (raises otherwise)
    lab = connected_components(pk.n, pk.tets)
    for s in range(4):
        assert len(set(lab[pk.vert_offsets[s]:pk.vert_offsets[s + 1]].tolist())) == 1
    assert len(set(lab.tolist())) == 4
    assert pk.algorithmic_bytes() == 24 * pk.n + 68 * pk.nele            # BASELINE.md section 3
    sub = pk.slice_spheres(1, 3)
    assert sub.nele == 1024 and sub.tets.min() == 0 and sub.tets.max() == sub.n - 1


def test_product_fails_loudly_without_gpu():
    import torch
    from tssplat_b200 import tet_spheres_ext as ext
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    v, t = make_tet_sphere(1204, 64)
    with pytest.raises(RuntimeError, match="CUDA"):
        ext.TetSpheres(v.astype(np.float32).reshape(-1), t.reshape(-1))
    h = C.c_void_p()
    vf = np.ascontiguousarray(v, dtype=np.float32)
    rc = _capi.lib.tsb_create(vf.ctypes.data, t.ctypes.data, len(v), len(t), None, 0, C.byref(h))
    assert rc == _capi.TSB_E_CUDA and not h.value                           # no CPU fallback
    with pytest.raises(RuntimeError):
        ext.TetSpheres(np.zeros(9), np.zeros(4, dtype=np.int32))            # wrong dtype (float64)


def test_drop_in_import_and_scheduler():
    """`from tet_spheres import tet_spheres_ext` (energies/smooth_barrier.py:6) and the coefficient
    scheduler / order switch (energies/smooth_barrier.py:47-66)."""
    import math
    from tet_spheres import tet_spheres_ext
    for name in ("TetSpheres", "forward", "backward", "random_x", "grad_limit"):
        assert hasattr(tet_spheres_ext, name)
    from tssplat_b200.energies import SmoothnessBarrierEnergy
    eng = SmoothnessBarrierEnergy.__new__(SmoothnessBarrierEnergy)
    from types import SimpleNamespace
    eng.FLAGS = SimpleNamespace(smooth_eng_coeff=2e-4 / 64, barrier_coeff=2e-4, increase_order_iter=1000)
    assert eng.coeff_scheduler(0) == pytest.approx((2e-4 / 64, 2e-4))
    c1, c2 = eng.coeff_scheduler(600)
    m = 2 ** (4 * abs(math.sin(600 / 2400 * math.pi)))
    assert c1 == pytest.approx(2e-4 / 64 * m) and c2 == pytest.approx(2e-4 * m)
    assert eng.coeff_scheduler(5000) == pytest.approx((2e-4 / 64 * 16, 2e-4 * 16))


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the GPU arm): one JSON line with the contract's
    keys, the same metric/unit as the GPU arm, e2e == value with zero copy bytes, no GPU launches.  Under torchrun only
    rank 0 prints."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "3", "--min-seconds", "0.2"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "dtype", "data",
              "config", "cpu_baseline", "e2e", "impl"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "geometry_energy_grad_iters_per_sec_64x4k" and d["unit"] == "iters/s"
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["steps"] >= 200
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_bench_dump_outputs_writes_a_fixed_sample_within_budget(tmp_path):
    """bench.py's --dump-outputs writer: float32 arrays as given, and a gradient over the byte budget becomes the same
    seeded sample of its rows every time."""
    import bench
    e = np.array([1.0, 2.0, 3.0], dtype=np.float32)
    g = np.arange(3000, dtype=np.float32).reshape(1000, 3)
    bench.dump_outputs(str(tmp_path / "all"), e, g)
    assert np.array_equal(np.load(tmp_path / "all" / "energy.npy"), e)
    assert np.array_equal(np.load(tmp_path / "all" / "grad.npy"), g)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), e, g, "_rank1", budget=1212)
    s = np.load(tmp_path / "a" / "grad_rank1.npy")
    assert s.dtype == np.float32 and s.shape == (100, 3) and s.nbytes + e.nbytes <= 1212
    assert np.array_equal(s, np.load(tmp_path / "b" / "grad_rank1.npy"))
    rows = s[:, 0].astype(np.int64) // 3
    assert np.all(np.diff(rows) > 0) and np.array_equal(s, g[rows])


def test_native_autograd_bridge_builds_and_binds():
    """The C++ autograd bridge (csrc/torch_binding.cpp) compiles with the image's g++ against this torch, loads, and
    takes the C entry points from the already loaded library (no GPU needed for any of that)."""
    from tssplat_b200 import native_autograd
    so = native_autograd.build()
    assert so and os.path.exists(so)
    assert native_autograd.available()
    mod = native_autograd.module()
    for name in ("bind", "state_new", "state_free", "note_parameters_changed", "energy"):
        assert hasattr(mod, name)
    mod.note_parameters_changed()


def _ragged_mesh(rng, n_comp, max_tets):
    """Components = connected chunks of tet-spheres (ragged boundaries), vertex ids shuffled over a range with
    gaps (unreferenced vertices), tets of different components interleaved."""
    verts, tets = [], []
    for c in range(n_comp):
        v, t = make_tet_sphere(1300 + int(rng.integers(0, 50)), int(rng.integers(24, max_tets)))
        keep = t[: int(rng.integers(max(4, len(t) // 3), len(t) + 1))]          # a prefix of the generator's order stays face-connected
        used = np.unique(keep)
        remap = -np.ones(len(v), dtype=np.int64)
        remap[used] = np.arange(len(used))
        verts.append(v[used] + rng.normal(0, 3.0, 3))
        tets.append(remap[keep])
    off = np.cumsum([0] + [len(v) for v in verts])
    V = np.concatenate(verts)
    T = np.concatenate([t + off[i] for i, t in enumerate(tets)])
    n_total = len(V) + int(rng.integers(0, 6))                                  # extra unreferenced vertices
    perm = rng.permutation(n_total)
    Vp = rng.normal(0, 1, (n_total, 3))
    Vp[perm[: len(V)]] = V
    Tp = perm[T]
    Tp = Tp[rng.permutation(len(Tp))]
    return Vp.astype(np.float32), Tp.astype(np.int32)


def test_plan_randomised_ragged_meshes_match_oracle():
    """Property test of the host plan builder + stream format: for random ragged, relabelled, interleaved
    multi-component meshes and random launch shapes, the numpy walk of the plan equals the fp64 C oracle."""
    from hypothesis import HealthCheck, given, settings, strategies as st

    @settings(max_examples=25, deadline=None, suppress_health_check=list(HealthCheck), derandomize=True)
    @given(seed=st.integers(0, 10 ** 6), n_comp=st.integers(1, 5), nw=st.sampled_from([8, 16]), grid=st.integers(1, 9),
           force_global=st.sampled_from([0, 1]), scale=st.sampled_from([0, 1]))
    def run(seed, n_comp, nw, grid, force_global, scale):
        rng = np.random.default_rng(seed)
        V, T = _ragged_mesh(rng, n_comp, 400)
        if len(np.unique(T)) < 4:
            return
        plan = build_host_plan(V, T, nw=nw, grid=grid, force_global=force_global, laplacian_scale=scale)
        orc = COracle(V, T, scale)
        for sig, order in ((0.03, 2), (0.4, 4)):
            x = (V + rng.normal(0, sig * 0.2, V.shape)).astype(np.float32)
            E, es, eb, g = emulate_kernel(plan, x, 3e-4, 2e-4, order, gradH=1.3)
            Eo, terms, go = orc.energy_grad(x, 3e-4, 2e-4, order, gradH=1.3)
            assert E == pytest.approx(Eo, rel=5e-6, abs=1e-12)
            assert np.linalg.norm(g - go) <= 5e-6 * max(np.linalg.norm(go), 1e-12)
    run()


def test_plan_thousands_of_tiny_components():
    """2600 twelve-tet components on 148 CTAs: up to 18 segments per CTA (more than the kernel's 16-entry
    shared-memory segment table, so the global fallback path of the headers is part of the plan's contract)."""
    pk = make_pack(2600, 12, seed=3, unique=6)
    plan = build_host_plan(pk.verts, pk.tets, nw=16, grid=148)
    cs = plan["cta_seg"].reshape(-1, 2)
    assert plan["n_components"] == 2600 and (cs[:, 1] - cs[:, 0]).max() > 16
    x = (pk.verts + np.random.default_rng(0).normal(0, 0.05, pk.verts.shape)).astype(np.float32)
    E, _, _, g = emulate_kernel(plan, x, 2e-4, 3e-4, 2)
    Eo, _, go = COracle(pk.verts, pk.tets).energy_grad(x, 2e-4, 3e-4, 2)
    assert E == pytest.approx(Eo, rel=2e-6) and np.linalg.norm(g - go) <= 2e-6 * np.linalg.norm(go)
