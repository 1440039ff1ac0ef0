"""Generates the committed golden fixtures from the original project's ``tssplat_ext/a.veg``:

    python tests/golden/make_golden.py <original project>/tssplat_ext/a.veg

* ``a_veg_mesh.npz``  -- the reference's only in-tree tet mesh (``tssplat_ext/a.veg``: 4500 verts,
  22120 tets) converted to arrays, so the tests can use it without the original project.
* ``a_veg_excerpt.veg`` -- the first 1000 vertex lines of ``a.veg`` and the element lines among them, verbatim,
  with the header counts adjusted: a small sample of the reference's own file for the ``.veg`` reader.
* ``golden_energy.npz`` -- energies and gradient checksums produced by the fp64 sparse-operator
  oracle (``oracle/tet_energy_oracle.py``, restating ``tet_spheres_cuda.cu:118-263``) on seeded
  inputs.  The reference ships NO golden vectors for this path and cannot be built here (libpgo),
  so these are oracle-generated: they pin the oracle against regressions and pin the CUDA path to
  the oracle; parity against the reference binary itself stays UNPINNED (DESIGN.md).
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle.tet_energy_oracle import ReferenceEnergyOracle  # noqa: E402
from tssplat_b200.mesh import load_veg, make_pack, perturb  # noqa: E402

CASES = [  # (name, sigma_rel, seed, order, c1, c2, gradH)
    ("benign_o2", 0.02, 0, 2, 2e-4, 2e-4, 1.0),
    ("inverted_o2", 0.35, 1, 2, 3.2e-3, 3.2e-3, 0.5),
    ("inverted_o4", 0.35, 1, 4, 2e-4, 2e-4, 1.0),
]


def run(mesh_name, verts, tets, out):
    orc = ReferenceEnergyOracle(verts, tets)
    for name, sig, seed, order, c1, c2, gh in CASES:
        x = perturb(verts, tets, sig, seed) if not hasattr(verts, "verts") else None
        sm, bar = orc.energy_terms(x, order)
        g = orc.backward(gh, x, c1, c2, order)
        key = f"{mesh_name}/{name}"
        out[key + "/energy"] = np.float64(orc.forward(x, c1, c2, order))
        out[key + "/smooth"] = np.float64(sm)
        out[key + "/barrier"] = np.float64(bar)
        out[key + "/grad_l2"] = np.float64(np.linalg.norm(g))
        out[key + "/grad_sum"] = g.sum(axis=0)
        out[key + "/grad_sample"] = g[:: max(1, len(g) // 64)][:64].copy()
        out[key + "/inverted_fraction"] = np.float64(orc.inverted_fraction(x))
        print(key, float(out[key + "/energy"]), float(out[key + "/inverted_fraction"]))


def write_veg_excerpt(src, dst, n_verts=1000):
    """Vertex lines 1..n_verts of ``src`` and the element lines whose four vertices are among them, verbatim."""
    lines = open(src).read().splitlines()
    iv, ie = lines.index("*VERTICES"), lines.index("*ELEMENTS")
    assert lines[ie + 1] == "TET" and int(lines[iv + 1].split()[0]) >= n_verts
    ne = int(lines[ie + 2].split()[0])
    elems = [ln for ln in lines[ie + 3:ie + 3 + ne] if max(int(s) for s in ln.split()[1:5]) <= n_verts]
    with open(dst, "w") as f:
        f.write("\n".join([lines[0], f"# {n_verts} vertices, {len(elems)} elements", "", "*VERTICES", f"{n_verts} 3 0 0",
                           *lines[iv + 2:iv + 2 + n_verts], "", "*ELEMENTS", "TET", f"{len(elems)} 4 0", *elems,
                           *lines[ie + 3 + ne:]]) + "\n")


if __name__ == "__main__":
    write_veg_excerpt(sys.argv[1], os.path.join(HERE, "a_veg_excerpt.veg"))
    v, t = load_veg(sys.argv[1])
    np.savez_compressed(os.path.join(HERE, "a_veg_mesh.npz"), verts=v.astype(np.float64), tets=t.astype(np.int32))
    out = {}
    run("a_veg", v, t, out)
    pk = make_pack(3, 1024, seed=1)
    run("pack3x1024", pk.verts.astype(np.float64), pk.tets, out)
    np.savez_compressed(os.path.join(HERE, "golden_energy.npz"), **out)
