"""Our AEV kernels against the REFERENCE'S OWN CUDA kernels (cuAEV).

The AEVs and the force-side gradient of the reference's half-neighbour-list path (csrc/cuaev.cpp:204-223) on seeded
water boxes are stored in tests/golden/ref_cuaev_water*.npz (oracle/make_cuaev_golden.py, run on a B200 with the
reference's kernels compiled for sm_100 by oracle/build_ref.sh); the first test checks ours against them.  The
second test runs the reference's compiled cell list and cuAEV binaries (oracle/_ref, git-ignored) beside ours and
records their times; it is skipped where those binaries are absent.
"""
import json
import os

import numpy as np
import pytest
import torch

from helpers import GOLD, ROOT

pytestmark = pytest.mark.gpu
# one copy per process: the staged reference package (oracle/_ref/torchani, used by the drop-in tests) loads its own
# cuaev.so / cell_list.so; registering a second copy of the same torch classes aborts the interpreter
_STAGED = os.path.join(ROOT, "oracle", "_ref", "torchani")
REF_SO = os.path.join(_STAGED, "cuaev.so") if os.path.exists(os.path.join(_STAGED, "cuaev.so")) else \
    os.path.join(ROOT, "oracle", "_ref", "cuaev.so")


def _reference_computer(consts, dev):
    if not os.path.exists(REF_SO):
        pytest.skip("oracle/_ref/cuaev.so has not been built (oracle/build_ref.sh needs /root/reference)")
    try:
        torch.ops.load_library(REF_SO)
        f32 = dict(dtype=torch.float32, device=dev)
        return torch.classes.cuaev.CuaevComputer(
            consts.rcr, consts.rca, torch.tensor([consts.eta_r], **f32), torch.tensor(consts.shf_r, **f32),
            torch.tensor([consts.eta_a], **f32), torch.tensor([consts.zeta], **f32), torch.tensor(consts.shf_a, **f32),
            torch.tensor(consts.shf_z, **f32), consts.num_species, True)
    except Exception as exc:  # ABI / driver mismatch on this box: not a failure of the product
        pytest.skip(f"the reference cuAEV extension does not load here: {exc}")


def _time_ms(fn, reps=20, warm=5):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


@pytest.mark.parametrize("molecules", [333, 3333])
def test_aev_and_gradient_match_the_reference_cuda_kernels(molecules):
    from torchani_b200 import synthetic
    from torchani_b200.aev import AEVComputer
    dev = torch.device("cuda", 0)
    gold = np.load(os.path.join(GOLD, f"ref_cuaev_water{3 * molecules}.npz"))
    rows = torch.from_numpy(gold["rows"]).to(dev)
    aev_ref = torch.from_numpy(gold["aev"]).to(dev)
    g_ref = torch.from_numpy(gold["grad"]).to(dev)
    _, idx, coords, cell, pbc = synthetic.water_box(molecules, seed=0)
    idx_d, cell_d, pbc_d = idx.to(dev), cell.to(dev), pbc.to(dev)
    ours = AEVComputer.like_2x().to(dev)
    c_our = coords.to(dev).requires_grad_(True)
    aev_our = ours(idx_d, c_our, cell_d, pbc_d)
    assert tuple(aev_our.shape) == tuple(gold["shape"])
    err = (aev_our[0, rows] - aev_ref).abs()
    # two float32 GPU implementations of the same formulas (the reference with -use_fast_math)
    assert bool((err <= 5e-5 * aev_ref.abs() + 5e-5).all()), float(err.max())
    g = torch.randn(aev_our.shape, generator=torch.Generator().manual_seed(5)).to(dev)
    (g_our,) = torch.autograd.grad(aev_our, c_our, g)
    scale = float(g_ref.abs().max())
    assert float((g_our - g_ref).abs().max()) <= 5e-4 * scale, (float((g_our - g_ref).abs().max()), scale)


def test_reference_gpu_path_pieces_beside_ours():
    """The stages of the reference's GPU path on the same box and inputs: its C++/ATen cell list
    (csrc/cell_list.cpp, built into oracle/_ref), its cuAEV kernels and the BmmEnsemble network path (restated with
    torch.baddbmm in oracle/gpu_baseline.py).  Checks that they agree with ours and records their times."""
    if os.environ.get("ANI_B200_REF_PATH_TEST", "0") == "0":
        pytest.skip("measurement of the reference's GPU path pieces: set ANI_B200_REF_PATH_TEST=1 to run it")
    from torchani_b200 import models, neighbors, synthetic
    from torchani_b200.engine import constants_2x
    import oracle.gpu_baseline as gb
    dev = torch.device("cuda", 0)
    consts = constants_2x()
    comp = _reference_computer(consts, dev)
    cl_so = os.path.join(_STAGED, "cell_list.so")
    if not os.path.exists(cl_so):
        cl_so = os.path.join(ROOT, "oracle", "_ref", "cell_list.so")
    if not os.path.exists(cl_so):
        pytest.skip("oracle/_ref/cell_list.so has not been built")
    try:
        torch.ops.load_library(cl_so)
    except Exception as exc:
        pytest.skip(f"the reference cell_list extension does not load here: {exc}")
    z, idx, coords, cell, pbc = synthetic.water_box(3333, seed=0)
    idx_d, c_d, cell_d, pbc_d = idx.to(dev), coords.to(dev), cell.to(dev), pbc.to(dev)

    # ---- neighbour stage: reference op vs our CellList (same pair set)
    def ref_list():
        return torch.ops.cell_list.cell_list(consts.rcr, idx_d, c_d, cell_d, pbc_d)

    try:
        r_idx, r_dist, _ = ref_list()
    except Exception as exc:   # the reference's op is the yardstick here, not the thing under test
        pytest.skip(f"the reference cell_list op does not run on this box: {exc}")
    ours_nb = neighbors.CellList()(consts.rcr, idx_d, c_d, cell_d, pbc_d)
    # pairs exactly at the cutoff round differently in the two float32 distance computations (first run on a
    # B200: 284 110 pairs from the reference op, 284 111 from ours, out of 284 k)
    n_ref, n_our = r_idx.shape[1], ours_nb.indices.shape[1]
    assert abs(n_ref - n_our) <= 3, (n_ref, n_our)
    k = min(n_ref, n_our)
    assert float((torch.sort(r_dist)[0][:k] - torch.sort(ours_nb.distances)[0][:k]).abs().max()) < 1e-3
    t_list_ref = _time_ms(ref_list, reps=5, warm=2)
    t_list_ours = _time_ms(lambda: neighbors.CellList()(consts.rcr, idx_d, c_d, cell_d, pbc_d), reps=5, warm=2)

    # ---- AEV stage: the reference's cuAEV kernels (given pair list -> AEV -> gradient) vs our AEV module (which
    #      builds its bucket grid inside the call); module-level API on both sides, dense 1008-wide AEV written
    from torchani_b200.aev import AEVComputer
    c_ref, c_our = c_d.clone().requires_grad_(True), c_d.clone().requires_grad_(True)
    ij32, sp32 = ours_nb.indices.to(torch.int32), idx_d.to(torch.int32)
    diff, dist = ours_nb.diff_vectors.contiguous(), ours_nb.distances.contiguous()
    ours = AEVComputer.like_2x().to(dev)
    g = torch.randn((1, 9999, 1008), generator=torch.Generator().manual_seed(5)).to(dev)

    def ref_forward():
        return torch.ops.cuaev.run_with_half_nbrlist(c_ref, sp32, ij32, diff, dist, comp)

    def ref_fwd_bwd():
        torch.autograd.grad(ref_forward(), c_ref, g)

    def our_fwd_bwd():
        torch.autograd.grad(ours(idx_d, c_our, cell_d, pbc_d), c_our, g)

    with torch.no_grad():
        t_aev_ref = _time_ms(ref_forward)
        t_aev_ours = _time_ms(lambda: ours(idx_d, c_our, cell_d, pbc_d))
    t_aev_ref_fb, t_aev_ours_fb = _time_ms(ref_fwd_bwd), _time_ms(our_fwd_bwd)

    # ---- networks: BmmEnsemble restated (cuBLAS) vs our tensor-core ensemble on the same AEVs
    weights = synthetic.make_weights(models.SYMBOLS_2X, synthetic.DIMS_2X, 1008, 8, seed=1234)
    model = models.from_weight_lists("2x", weights, device=dev, periodic_table_index=False)
    aev = model.aev_computer(idx_d, c_d, cell_d, pbc_d).detach()
    bmm = gb.BmmNetworks(weights, models.SYMBOLS_2X, dev)
    idx_list = bmm.make_idx_list(idx_d)
    times = {}
    for tf32 in (False, True):
        torch.backends.cuda.matmul.allow_tf32 = tf32
        a_ref = aev.clone().requires_grad_(True)
        e_ref = bmm.energy(idx_d, a_ref, idx_list)
        (g_ref,) = torch.autograd.grad(e_ref.sum(), a_ref)
        if not tf32:
            a_our = aev.clone().requires_grad_(True)
            e_our = model.neural_networks(idx_d, a_our)
            (g_our,) = torch.autograd.grad(e_our.sum(), a_our)
            assert abs(float(e_our[0]) - float(e_ref[0])) < 1e-5 * abs(float(e_ref[0])) + 5e-3   # fp32 sums of 1e4 terms
            assert float((g_our - g_ref).abs().max()) < 1e-5 + 1e-3 * float(g_ref.abs().max())

        def fwd_bwd():
            a = aev.clone().requires_grad_(True)
            torch.autograd.grad(bmm.energy(idx_d, a, idx_list).sum(), a)

        times["tf32" if tf32 else "fp32"] = _time_ms(fwd_bwd, reps=10, warm=3)
    torch.backends.cuda.matmul.allow_tf32 = False
    rec = {"atoms": 9999, "reference_cell_list_ms": t_list_ref, "ours_cell_list_module_ms": t_list_ours,
           "reference_cuaev_forward_ms": t_aev_ref, "reference_cuaev_forward_backward_ms": t_aev_ref_fb,
           "ours_aev_module_forward_ms": t_aev_ours, "ours_aev_module_forward_backward_ms": t_aev_ours_fb,
           "bmm_ensemble_port_fwd_bwd_fp32_ms": times["fp32"], "bmm_ensemble_port_fwd_bwd_tf32_ms": times["tf32"],
           "note": "reference cell list = torch.ops.cell_list.cell_list built from the reference's csrc/cell_list.cpp; "
                   "network path = BmmEnsemble (nn/_infer.py:61-216) restated with torch.baddbmm (cuBLAS), forward + "
                   "backward to the AEVs.  Ours inside the fused step: prepare 0.04 ms, six tensor-core GEMMs 0.23 ms."}
    print("reference GPU path pieces:", json.dumps(rec))
    out_dir = os.path.join(ROOT, "gpurun_out")
    if os.path.isdir(out_dir):
        with open(os.path.join(out_dir, "ref_gpu_path_timing.json"), "w") as fh:
            json.dump(rec, fh)
