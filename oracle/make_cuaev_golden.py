"""Generate tests/golden/ref_cuaev_water*.npz: the reference's OWN CUDA AEV kernels (cuAEV) on seeded water boxes.

TEST INFRASTRUCTURE ONLY; needs a GPU and oracle/_ref/cuaev.so (oracle/build_ref.sh).  For each box of
``synthetic.water_box(molecules, seed=0)`` it hands the pair list of ``torchani_b200.neighbors.CellList`` to the
reference's half-neighbour-list entry point (csrc/cuaev.cpp:204-223, driven as aev/_computer.py:365-407 does) and
stores

* ``aev``: rows ``rows`` of the reference's float32 AEVs (a seeded sample of 128 atoms, to keep the fixture small),
* ``grad``: the reference's gradient of ``(aev * g).sum()`` with respect to the coordinates, where
  ``g = torch.randn(aev.shape, generator=torch.Generator().manual_seed(5))``,
* ``shape``: the shape of the full AEV tensor.

tests/test_gpu_reference_cuaev.py compares the project's AEV kernels against these.

Usage:  python oracle/make_cuaev_golden.py [--out DIR]      (default DIR: tests/golden)
"""
from __future__ import annotations

import argparse
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
ROWS = 128


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "tests", "golden"))
    args = ap.parse_args()
    from torchani_b200 import neighbors, synthetic
    from torchani_b200.engine import constants_2x

    so = os.path.join(HERE, "_ref", "cuaev.so")
    torch.ops.load_library(so)
    dev = torch.device("cuda", 0)
    consts = constants_2x()
    f32 = dict(dtype=torch.float32, device=dev)
    comp = torch.classes.cuaev.CuaevComputer(
        consts.rcr, consts.rca, torch.tensor([consts.eta_r], **f32), torch.tensor(consts.shf_r, **f32),
        torch.tensor([consts.eta_a], **f32), torch.tensor([consts.zeta], **f32), torch.tensor(consts.shf_a, **f32),
        torch.tensor(consts.shf_z, **f32), consts.num_species, True)
    os.makedirs(args.out, exist_ok=True)
    for molecules in (333, 3333):
        _, idx, coords, cell, pbc = synthetic.water_box(molecules, seed=0)
        idx_d = idx.to(dev)
        c = coords.to(dev).requires_grad_(True)
        nb = neighbors.CellList()(consts.rcr, idx_d, c.detach(), cell.to(dev), pbc.to(dev))
        aev = torch.ops.cuaev.run_with_half_nbrlist(c, idx_d.to(torch.int32), nb.indices.to(torch.int32),
                                                    nb.diff_vectors.contiguous(), nb.distances.contiguous(), comp)
        g = torch.randn(aev.shape, generator=torch.Generator().manual_seed(5)).to(dev)
        (grad,) = torch.autograd.grad(aev, c, g)
        n = aev.shape[1]
        rows = np.sort(np.random.default_rng(0).choice(n, ROWS, replace=False))
        path = os.path.join(args.out, f"ref_cuaev_water{n}.npz")
        np.savez_compressed(path, rows=rows, aev=aev[0].detach().cpu().numpy()[rows], grad=grad.cpu().numpy(),
                            shape=np.array(aev.shape))
        print(f"{path}: {n} atoms, {int(nb.indices.shape[1])} pairs, {os.path.getsize(path)} bytes")


if __name__ == "__main__":
    main()
