"""Generator of tests/golden/c2f_grid.npz (CONTAINER ONLY: needs /root/reference): the grid the REFERENCE's own
Seg3dLossless class (MCAcc/seg3d_lossless.py:233-428, imported unmodified through oracle/refload.py) returns on the CPU for
the analytic three-sphere query function and the anisotropic pyramid of tests/test_c2f_cpu.py, and of
tests/golden/c2f_lattice.npz: the lattice geometry the same instance computes (spacing_{x,y,z}, b{x,y,z}).

    python tests/golden/make_golden_c2f.py            # writes the fixtures
    python tests/golden/make_golden_c2f.py --check    # verifies the committed fixtures bit for bit (no write)
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import refload  # noqa: E402
from test_c2f_cpu import KW, sphere_query  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "c2f_grid.npz")
OUT_LATTICE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "c2f_lattice.npz")
LATTICE = ("spacing_x", "spacing_y", "spacing_z", "bx", "by", "bz")


def main():
    torch.set_num_threads(8)
    ns = refload.load()
    eng = ns.MCAcc.Seg3dLossless(sphere_query, **KW)
    with torch.no_grad():
        grid = eng.forward()[0, 0].numpy()
    lattice = {k: np.float64(getattr(eng, k)) for k in LATTICE}
    if "--check" in sys.argv:
        gold = np.load(OUT)["grid"]
        assert np.array_equal(grid, gold), "committed c2f_grid.npz differs from the reference class's output"
        gold = np.load(OUT_LATTICE)
        assert all(gold[k] == v for k, v in lattice.items()), "committed c2f_lattice.npz differs from the reference class"
        print("c2f_grid.npz, c2f_lattice.npz == reference Seg3dLossless output, bit for bit", grid.shape)
        return
    np.savez_compressed(OUT, grid=grid)
    np.savez(OUT_LATTICE, **lattice)
    print("wrote", OUT, grid.shape, OUT_LATTICE)


if __name__ == "__main__":
    main()
