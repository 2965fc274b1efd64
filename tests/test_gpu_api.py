"""GPU tests of the drop-in modules (interfaces of torchani.neighbors / AEVComputer / nn / ANI)."""
import os

import numpy as np
import pytest
import torch

import oracle.ani_oracle as orc
from helpers import (AEV_ATOL, AEV_RTOL, E_ATOL, E_RTOL, F_ATOL, assert_close, golden_inputs, load_golden,
                     oracle_model)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _pairs_sorted(indices, distances):
    lo = np.minimum(indices[0], indices[1])
    hi = np.maximum(indices[0], indices[1])
    order = np.lexsort((distances, hi, lo))
    return lo[order], hi[order], distances[order]


@pytest.mark.parametrize("name", ["water30_pbc_ani2x", "benzene_pbc_ani2x", "randbatch_ani2x", "kat2x5_ani2x"])
def test_neighborlists_match_reference_pairs(name):
    from torchani_b200.neighbors import AllPairs, CellList
    rec = load_golden(name)
    species, coords, cell, pbc = golden_inputs(rec, torch.float32)
    nl = CellList() if species.shape[0] == 1 else AllPairs()
    args = [species.to(DEV), coords.to(DEV), None if cell is None else cell.to(DEV),
            None if pbc is None else pbc.to(DEV)]
    nb = nl(5.1, *args)
    assert nb.indices.shape == (2, int(rec["num_pairs"])) and nb.indices.dtype == torch.int64
    lo, hi, d = _pairs_sorted(nb.indices.cpu().numpy(), nb.distances.cpu().numpy())
    glo, ghi, gd = _pairs_sorted(rec["pairs"], rec["distances"])
    assert (lo == glo).all() and (hi == ghi).all()
    assert np.abs(d - gd).max() < 5e-6
    assert torch.allclose(nb.diff_vectors.norm(dim=-1), nb.distances, atol=1e-6)
    # autograd edge to coords like neighbors.py:107-112
    c = args[1].clone().requires_grad_(True)
    nb = nl(5.1, args[0], c, args[2], args[3])
    (g,) = torch.autograd.grad(nb.distances.sum(), c)
    assert bool(torch.isfinite(g).all()) and float(g.abs().max()) > 0


def test_verlet_cell_list_matches_cell_list():
    """neighbors.VerletCellList: cached pairs within cutoff + skin, re-screened every call; the pair set
    must equal a fresh CellList at every step, and the cache must be rebuilt after a large move."""
    from torchani_b200 import neighbors
    rec = load_golden("water30_pbc_ani2x")
    species, coords, cell, pbc = golden_inputs(rec, torch.float32)
    sp, c, cell_d, pbc_d = species.to(DEV), coords.to(DEV), cell.to(DEV), pbc.to(DEV)
    vl, cl = neighbors.VerletCellList(skin=0.6), neighbors.CellList()
    g = torch.Generator(device="cpu").manual_seed(3)

    def canon(nb):
        i = nb.indices.cpu().numpy()
        d = nb.distances.detach().cpu().numpy()
        lo, hi = np.minimum(i[0], i[1]), np.maximum(i[0], i[1])
        order = np.lexsort((np.round(d, 4), hi, lo))
        return lo[order], hi[order], d[order]

    for it in range(8):
        c = c + (torch.randn(c.shape, generator=g) * 0.03).to(DEV)
        a, b = canon(vl(5.1, sp, c, cell_d, pbc_d)), canon(cl(5.1, sp, c, cell_d, pbc_d))
        assert a[0].shape == b[0].shape and (a[0] == b[0]).all() and (a[1] == b[1]).all()
        assert np.abs(a[2] - b[2]).max() < 1e-5
    assert 1 <= vl.rebuilds < 8
    before = vl.rebuilds
    c = c.clone()
    c[0, 4] += torch.tensor([1.5, 0.0, 0.0], device=DEV)
    a, b = canon(vl(5.1, sp, c, cell_d, pbc_d)), canon(cl(5.1, sp, c, cell_d, pbc_d))
    assert vl.rebuilds == before + 1 and (a[0] == b[0]).all() and (a[1] == b[1]).all()
    c2 = c.clone().requires_grad_(True)
    nb = vl(5.1, sp, c2, cell_d, pbc_d)
    (gr,) = torch.autograd.grad(nb.distances.sum(), c2)            # autograd edge to the coordinates
    assert gr.shape == c2.shape and bool(torch.isfinite(gr).all())
    with pytest.raises(ValueError):
        neighbors.VerletCellList(skin=0.0)


def test_neighborlist_validation():
    from torchani_b200.neighbors import CellList
    nl = CellList()
    sp = torch.zeros(1, 4, dtype=torch.long, device=DEV)
    co = torch.rand(1, 4, 3, device=DEV)
    with pytest.raises(ValueError):
        nl(5.1, sp, co, None, torch.tensor([False, False, False], device=DEV))
    with pytest.raises(ValueError):
        nl(5.1, sp, co, torch.eye(3, device=DEV), None)
    with pytest.raises(ValueError):
        nl(-1.0, sp, co)
    with pytest.raises(RuntimeError, match="too small"):
        nl(5.1, sp, co, torch.eye(3, device=DEV) * 3.0, torch.tensor([True, True, True], device=DEV))
    with pytest.raises(ValueError):
        nl(5.1, sp.cpu(), co.cpu())


@pytest.mark.parametrize("name", ["water30_pbc_ani2x", "randbatch_ani2x", "ch4_ani1x"])
def test_aev_computer_forward_backward(name):
    from torchani_b200.aev import AEVComputer
    rec = load_golden(name)
    species, coords, cell, pbc = golden_inputs(rec, torch.float32)
    aevc = (AEVComputer.like_2x() if rec["kind"] == "2x" else AEVComputer.like_1x()).to(DEV)
    c = coords.to(DEV).requires_grad_(True)
    aev = aevc(species.to(DEV), c, None if cell is None else cell.to(DEV), None if pbc is None else pbc.to(DEV))
    assert aev.shape == (*species.shape, aevc.out_dim)
    # oracle AEV + a random linear functional of it for the backward check
    spec = orc.aev_spec_2x() if rec["kind"] == "2x" else orc.aev_spec_1x()
    c64 = coords.double().requires_grad_(True)
    nb = orc.neighborlist(rec["neighborlist"], spec.rcr, species, c64, None if cell is None else cell.double(), pbc)
    ref = orc.aev_from_neighbors(spec, species, nb)
    assert_close("aev", aev.detach().cpu().numpy(), ref.detach().numpy(), AEV_RTOL, AEV_ATOL)
    w = torch.randn(ref.shape, generator=torch.Generator().manual_seed(3), dtype=torch.float64) * 1e-2
    (g_ref,) = torch.autograd.grad((ref * w).sum(), c64)
    (g,) = torch.autograd.grad((aev * w.float().to(DEV)).sum(), c)
    assert_close("dL/dcoords", g.cpu().numpy(), g_ref.numpy(), 1e-4, 2e-5)
    # padding rows are exactly zero
    pad = (species == -1)
    if bool(pad.any()):
        assert float(aev.detach().cpu()[pad].abs().max()) == 0.0


def test_ensemble_forward_on_given_aevs():
    from torchani_b200 import models
    rec = load_golden("randbatch_ani2x")
    species, coords, _, _ = golden_inputs(rec, torch.float32)
    om = oracle_model("2x", torch.float32)
    model = models.from_weight_lists("2x", om.weights, device=DEV)
    ens = model.neural_networks
    aev_ref = torch.tensor(rec["aev"], dtype=torch.float32)
    a = aev_ref.to(DEV).requires_grad_(True)
    e = ens(species.to(DEV), a)
    assert e.shape == (species.shape[0],)
    assert_close("molecular NN energies", e.detach().cpu().numpy(), rec["energy_nn"], 1e-5, 2e-6)
    e_at = ens(species.to(DEV), a, atomic=True)
    assert_close("atomic", e_at.detach().cpu().numpy(), rec["member_atomic"].mean(0), E_RTOL, E_ATOL)
    e_mem = ens(species.to(DEV), a, atomic=True, ensemble_values=True)
    assert_close("member atomic", e_mem.detach().cpu().numpy(), rec["member_atomic"], E_RTOL, E_ATOL)
    # backward-to-input vs oracle autograd
    a64 = torch.tensor(rec["aev"]).requires_grad_(True)
    m64 = oracle_model("2x", torch.float64)
    e64 = orc.ensemble_atomic_energies(m64.symbols, m64.weights, species, a64).mean(0).sum()
    (g_ref,) = torch.autograd.grad(e64, a64)
    (g,) = torch.autograd.grad(e.sum(), a)
    assert_close("dE/dAEV", g.cpu().numpy(), g_ref.numpy(), 1e-4, 1e-7)
    # set_active_members
    ens.set_active_members([0, 5])
    e2 = ens(species.to(DEV), a.detach(), atomic=True)
    assert_close("active members", e2.cpu().numpy(), rec["member_atomic"][[0, 5]].mean(0), E_RTOL, E_ATOL)
    ens.set_active_members(list(range(8)))
    # a single ANINetworks member == that member of the ensemble (tests/test_ensemble.py:22-37)
    e_m3 = ens[3](species.to(DEV), a.detach(), atomic=True)
    assert_close("member 3", e_m3.cpu().numpy(), rec["member_atomic"][3], E_RTOL, E_ATOL)


@pytest.mark.parametrize("name", ["water30_pbc_ani2x", "kat2x5_ani2x", "small264_nopbc_ani2x"])
def test_ani_model_energy_and_autograd_forces(name):
    """models.ANI2x-style call: energies = model((Z, coords), cell, pbc).energies; F = -dE/dx."""
    from torchani_b200 import models
    rec = load_golden(name)
    species, coords, cell, pbc = golden_inputs(rec, torch.float32)
    om = oracle_model("2x", torch.float32)
    model = models.from_weight_lists("2x", om.weights, device=DEV, periodic_table_index=True)
    znum = torch.tensor([orc.ATOMIC_NUMBERS[s] for s in orc.SYMBOLS_2X])
    z = torch.where(species >= 0, znum[species.clamp(min=0)], torch.full_like(species, -1))
    c = coords.to(DEV).requires_grad_(True)
    cell_d = None if cell is None else cell.to(DEV)
    pbc_d = None if pbc is None else pbc.to(DEV)
    out = model((z.to(DEV), c), cell_d, pbc_d)
    assert out.species.cpu().tolist() == species.tolist()
    (g,) = torch.autograd.grad(out.energies.sum(), c)
    assert_close("forces", -g.cpu().numpy(), rec["forces"], 0.0, F_ATOL)
    sae = orc.self_energies(orc.SYMBOLS_2X, orc.GSAES_WB97X_631GD, species, torch.float64).sum(-1).numpy()
    assert_close("energies", out.energies.detach().cpu().numpy(), rec["energy_nn"] + sae, 2e-7, 1e-5)
    e64 = model.energies_f64((z.to(DEV), coords.to(DEV)), cell_d, pbc_d)
    assert_close("energies f64", e64.cpu().numpy(), rec["energy_nn"] + sae, 0.0, 1e-5)
    at = model((z.to(DEV), coords.to(DEV)), cell_d, pbc_d, atomic=True).energies
    assert at.shape == species.shape
    ev = model((z.to(DEV), coords.to(DEV)), cell_d, pbc_d, ensemble_values=True).energies
    assert ev.shape == (8, species.shape[0])
    assert_close("ensemble mean", ev.mean(0).cpu().numpy(), rec["energy_nn"] + sae, 2e-7, 1e-5)
    e2, f2 = model.energies_and_forces(z.to(DEV), coords.to(DEV), cell_d, pbc_d)
    assert_close("forces (direct)", f2.cpu().numpy(), rec["forces"], 0.0, F_ATOL)
    with pytest.raises(ValueError):
        model((torch.full_like(z, 15).to(DEV), c), cell_d, pbc_d)  # phosphorus is not an ANI-2x element


def test_ani_model_member_forces_qbc_and_neighbor_entry():
    """arch.py:354-576: members_forces / energies_qbcs / atomic_stdev / force_qbc and the
    compute_from_neighbors entry point of the model, against per-member oracle runs."""
    from torchani_b200 import models, neighbors
    rec = load_golden("water30_pbc_ani2x")
    species, coords, cell, pbc = golden_inputs(rec, torch.float32)
    om = oracle_model("2x", torch.float32)
    o64 = oracle_model("2x", torch.float64, "cell_list")
    model = models.from_weight_lists("2x", om.weights, device=DEV, periodic_table_index=True)
    znum = torch.tensor([orc.ATOMIC_NUMBERS[s] for s in orc.SYMBOLS_2X])
    z = znum[species].to(DEV)
    c, cell_d, pbc_d = coords.to(DEV), cell.to(DEV), pbc.to(DEV)
    sf = model.members_forces((z, c), cell_d, pbc_d)
    assert sf.energies.shape == (8, 1) and sf.forces.shape == (8, 1, species.shape[1], 3)
    for m in (0, 5):
        ref = orc.compute(o64, species, coords.double(), cell.double(), pbc, members=[m])
        assert abs(float(sf.energies[m, 0]) - float(ref["energy"][0])) < 5e-3      # float32 at |E| ~ 760 Ha
        assert_close(f"member {m} forces", sf.forces[m].cpu().numpy(), ref["forces"].numpy(), 0.0, F_ATOL)
    assert_close("mean of member forces", sf.forces.mean(0).cpu().numpy(), rec["forces"], 0.0, F_ATOL)
    assert list(model.neural_networks.active_members_idxs) == list(range(8))       # restored
    ev = model((z, c), cell_d, pbc_d, ensemble_values=True).energies
    q = model.energies_qbcs((z, c), cell_d, pbc_d)
    assert_close("qbc", q.qbcs.cpu().numpy(), (ev.std(0) / np.sqrt(species.shape[1])).cpu().numpy(), 1e-6, 1e-9)
    st = model.atomic_stdev((z, c), cell_d, pbc_d)
    ref_std = np.std(rec["member_atomic"], axis=0, ddof=1)
    assert_close("atomic stdev", st.stdev_atomic_energies.cpu().numpy(), ref_std, 1e-3, 1e-6)
    fq = model.force_qbc((z, c), cell_d, pbc_d)
    mags = sf.forces.norm(dim=-1)
    assert_close("force magnitudes", fq.magnitudes.cpu().numpy(), mags.mean(0).cpu().numpy(), 1e-6, 1e-9)
    assert fq.relative_stdev.shape == mags.shape[1:] and bool((fq.relative_range > 0).all())
    # neighbour-list entry point of the model: a list built with a LARGER cutoff is narrowed down first
    idx = model.species_converter(z)
    nl = neighbors.CellList()(6.0, idx, c, cell_d, pbc_d)
    e_nb = model.compute_from_neighbors(idx, c, nl)
    sae = float(orc.self_energies(orc.SYMBOLS_2X, orc.GSAES_WB97X_631GD, species, torch.float64).sum())
    assert abs(float(e_nb[0]) - (float(rec["energy_nn"][0]) + sae)) < 5e-3
    e_at = model.compute_from_neighbors(idx, c, nl, atomic=True)
    assert e_at.shape == species.shape


@pytest.mark.parametrize("name", ["water30_pbc_ani2x", "water999_pbc_ani2x"])
def test_stress_from_the_force_kernel(name):
    """ase.py:164-173: stress = virial / volume.  The GPU accumulates the f-dot-r virial in the force
    kernel; the oracle differentiates the energy with respect to a strain of coordinates and cell."""
    from torchani_b200 import models
    rec = load_golden(name)
    species, coords, cell, pbc = golden_inputs(rec, torch.float32)
    om = oracle_model("2x", torch.float32)
    model = models.from_weight_lists("2x", om.weights, device=DEV, periodic_table_index=True)
    znum = torch.tensor([orc.ATOMIC_NUMBERS[s] for s in orc.SYMBOLS_2X])
    e, f, stress = model.energies_forces_stress(znum[species].to(DEV), coords.to(DEV), cell.to(DEV), pbc.to(DEV))
    # the strain derivative of the reference needs wrapped atoms (map_to_central uses a detached cell)
    c64, cell64 = coords.double(), cell.double()
    wrapped = c64 - torch.floor(c64 @ torch.linalg.inv(cell64)) @ cell64
    ref = orc.compute(oracle_model("2x", torch.float64, "cell_list"), species, wrapped, cell64, pbc, stress=True)
    assert_close("forces", f.cpu().numpy(), ref["forces"].numpy(), 0.0, F_ATOL)
    s_gpu, s_ref = stress.cpu().numpy(), ref["stress"].numpy()
    assert np.abs(s_gpu - s_gpu.T).max() < 1e-7
    assert_close("stress", s_gpu, s_ref, 1e-4, 1e-8)     # |stress| ~ 2e-4 Ha/A^3
    fix = np.load(os.path.join(os.path.dirname(__file__), "golden", "stress_pbc_ani2x.npz"))
    if name in fix.files:                                # the reference's own f-dot-r stress (make_golden.py --stress)
        assert_close("stress vs reference", s_gpu, fix[name], 1e-4, 1e-8)


def test_host_calculator_matches_oracle_and_repeats():
    """calculator.HostCalculator (counterpart of ase.py:75-173): host positions in, host E/F out;
    repeated calls replay the captured CUDA graph and must keep giving the oracle's answer."""
    from torchani_b200 import models
    from torchani_b200.calculator import HostCalculator
    rec = load_golden("water30_pbc_ani2x")
    species, coords, cell, pbc = golden_inputs(rec, torch.float32)
    om = oracle_model("2x", torch.float32)
    model = models.from_weight_lists("2x", om.weights, device=DEV, periodic_table_index=True)
    znum = torch.tensor([orc.ATOMIC_NUMBERS[s] for s in orc.SYMBOLS_2X])
    calc = HostCalculator(model, znum[species[0]].numpy(), cell.numpy(), pbc=True)
    sae = float(orc.self_energies(orc.SYMBOLS_2X, orc.GSAES_WB97X_631GD, species, torch.float64).sum())
    for it in range(6):  # eager x3, capture, replay, replay
        e, f = calc.calculate(coords[0].numpy())
        assert abs(e - (float(rec["energy_nn"][0]) + sae)) < 1e-5
        assert_close("forces", f, rec["forces"][0], 0.0, F_ATOL)
    # moved atoms: the replayed graph must see the new positions
    moved = coords[0].numpy().copy()
    moved[3] += np.array([0.05, -0.02, 0.01], dtype=np.float32)
    e2, f2 = calc.calculate(moved)
    ref = orc.compute(oracle_model("2x", torch.float64, "cell_list"), species, torch.tensor(moved).double().unsqueeze(0),
                      cell.double(), pbc)
    assert abs(e2 - float(ref["energy"][0])) < 1e-5
    assert_close("forces moved", f2, ref["forces"][0].numpy(), 0.0, F_ATOL)
    calc.check_status()


def test_host_calculator_verlet_skin_reuse():
    """HostCalculator(skin=...): the bucket grid of an earlier step is reused while the atoms stay inside
    their skin/2 spheres (VerletCellList semantics, neighbors.py:759-884) -- every step must still give
    the answer of a fresh grid; a jump beyond skin/2 is detected and the step redone."""
    from torchani_b200 import models
    from torchani_b200.calculator import HostCalculator
    rec = load_golden("water30_pbc_ani2x")
    species, coords, cell, pbc = golden_inputs(rec, torch.float32)
    om = oracle_model("2x", torch.float32)
    model = models.from_weight_lists("2x", om.weights, device=DEV, periodic_table_index=True)
    znum = torch.tensor([orc.ATOMIC_NUMBERS[s] for s in orc.SYMBOLS_2X])
    z = znum[species[0]].numpy()
    try:
        calc = HostCalculator(model, z, cell.numpy(), pbc=True, skin=0.4)
        o64 = oracle_model("2x", torch.float64, "cell_list")
        rng = np.random.default_rng(7)
        vel = rng.normal(scale=0.006, size=(species.shape[1], 3)).astype(np.float32)   # Angstrom per step
        pos = coords[0].numpy().copy()
        for it in range(40):
            pos = pos + vel
            e, f = calc.calculate(pos)
            if it % 4 == 0 or it > 36:
                ref = orc.compute(o64, species, torch.tensor(pos).double().unsqueeze(0), cell.double(), pbc)
                assert abs(e - float(ref["energy"][0])) < 1e-5, (it, e)
                assert_close(f"forces step {it}", f, ref["forces"][0].numpy(), 0.0, F_ATOL)
        assert calc.rebuilds >= 2 and calc.rebuilds < 30, calc.rebuilds       # reused most steps, rebuilt some
        before = calc.redone
        pos[5] += np.array([0.9, 0.0, -0.4], dtype=np.float32)                 # far beyond skin / 2
        e, f = calc.calculate(pos)
        assert calc.redone == before + 1 or not calc._have_grid or calc.rebuilds > 0
        ref = orc.compute(o64, species, torch.tensor(pos).double().unsqueeze(0), cell.double(), pbc)
        assert abs(e - float(ref["energy"][0])) < 1e-5
        assert_close("forces after jump", f, ref["forces"][0].numpy(), 0.0, F_ATOL)
        calc.check_status()
    finally:
        model.engine(DEV).skin = 0.0


@pytest.mark.parametrize("name", ["water30_pbc_ani2x", "randbatch_ani2x"])
def test_compute_from_neighbors_split_api(name):
    """The reference's split call: neighbors = nl(cutoff, idxs, coords, cell, pbc);
    aevs = aevc.compute_from_neighbors(idxs, coords, neighbors)  (aev/_computer.py:251-272)."""
    from torchani_b200.aev import AEVComputer
    from torchani_b200.neighbors import AllPairs, CellList, discard_outside_cutoff
    rec = load_golden(name)
    species, coords, cell, pbc = golden_inputs(rec, torch.float32)
    aevc = AEVComputer.like_2x().to(DEV)
    nl = CellList() if species.shape[0] == 1 else AllPairs()
    c = coords.to(DEV).requires_grad_(True)
    cell_d = None if cell is None else cell.to(DEV)
    pbc_d = None if pbc is None else pbc.to(DEV)
    nb = nl(5.1, species.to(DEV), c, cell_d, pbc_d)
    aev = aevc.compute_from_neighbors(species.to(DEV), c, nb)
    assert_close("aev", aev.detach().cpu().numpy(), rec["aev"], AEV_RTOL, AEV_ATOL)
    fused = aevc(species.to(DEV), c.detach(), cell_d, pbc_d)
    assert float((fused - aev.detach()).abs().max()) < 2e-5
    w = torch.randn(aev.shape, generator=torch.Generator().manual_seed(5)).to(DEV) * 1e-2
    (g1,) = torch.autograd.grad((aev * w).sum(), c)
    c2 = coords.to(DEV).requires_grad_(True)
    (g2,) = torch.autograd.grad((aevc(species.to(DEV), c2, cell_d, pbc_d) * w).sum(), c2)
    assert float((g1 - g2).abs().max()) < 2e-5
    # a filtered list (here: a larger cutoff list narrowed back) is honoured as given
    nb_big = nl(6.0, species.to(DEV), coords.to(DEV), cell_d, pbc_d)
    aev2 = aevc.compute_from_neighbors(species.to(DEV), coords.to(DEV), discard_outside_cutoff(nb_big, 5.1))
    assert float((aev2 - aev.detach()).abs().max()) < 2e-5


def test_weight_packing_kernel_matches_the_python_tiler():
    """ani_b200_pack_b_operand (the library's own model-pack kernel) against engine.tile_b_operand (the python
    statement of the tiled B operand layout, itself checked on the CPU in tests/test_host_logic.py): every operand
    of every species byte for byte, incl. hidden widths that need zero padding (ANI-1x carbon: 144, 112)."""
    from torchani_b200 import _lib
    from torchani_b200.engine import PackedNetworks, tile_b_operand
    dev = torch.device("cuda", 0)
    P2 = 2 * _lib.operand_format().parts
    for kind, in_dim, members in (("2x", 1008, 3), ("1x", 384, 2)):
        m = oracle_model(kind, members=members)
        w = [[wm[s] for s in m.symbols] for wm in m.weights]
        nets = PackedNetworks(w, in_dim, dev)
        src, dst = nets._keep[:2]
        torch.cuda.synchronize()
        M, ldx = nets.num_members, nets.ldx
        pad = lambda v: (v + 31) // 32 * 32  # noqa: E731
        for s, sym in enumerate(m.symbols):
            q, sp = nets._plan[s], nets.model.sp[s]
            h1, h2, h3 = nets.dims[s]
            p1, p2, p3 = pad(h1), pad(h2), pad(h3)
            assert (sp.h1, sp.h2, sp.h3) == (p1, p2, p3)
            Wp = []
            for k, (po, pi) in enumerate(((p1, ldx), (p2, p1), (p3, p2))):
                layer = []
                for mem in range(M):
                    z = torch.zeros(po, pi)
                    wt = m.weights[mem][sym][k][0].float()
                    z[:wt.shape[0], :wt.shape[1]] = wt
                    layer.append(z)
                Wp.append(layer)
            sc = list(sp.w_scale)
            w1n = torch.cat(Wp[0], 0)
            expect = {
                "d_f1": torch.cat([tile_b_operand(x, sc[0]) for x in Wp[0]]),
                "d_f2": torch.cat([tile_b_operand(x, sc[1]) for x in Wp[1]]),
                "d_f3": torch.cat([tile_b_operand(x, sc[2]) for x in Wp[2]]),
                "d_b3": torch.cat([tile_b_operand(x.t().contiguous(), sc[2]) for x in Wp[2]]),
                "d_b2": torch.cat([tile_b_operand(x.t().contiguous(), sc[1]) for x in Wp[1]]),
                "d_b1": tile_b_operand(w1n.t().contiguous(), sc[0]),
            }
            for name, ref in expect.items():
                ref_bytes = ref.view(torch.uint8).reshape(-1)
                got = dst[q[name]: q[name] + ref_bytes.numel()].cpu()
                assert torch.equal(got, ref_bytes), (kind, sym, name)
            b4 = src[q["s_b4"]: q["s_b4"] + M].cpu()
            assert torch.equal(b4, torch.stack([m.weights[mem][sym][3][1].float().view(()) for mem in range(M)]))
        assert P2 in (4, 6)
        nets.set_active_members([0, 1])
        assert list(nets.model.member_scale)[:2] == [0.5, 0.5]
        with pytest.raises(IndexError):
            nets.set_active_members([7])


def test_model_level_calls_raise_device_side_conditions():
    """The public model paths read the device status word (one 4-byte copy): a periodic cell thinner than the
    cutoff raises the reference's RuntimeError (neighbors.py:402-403), more neighbours than nbr_cap raises instead
    of returning energies of a truncated list."""
    from torchani_b200 import models, synthetic
    w = synthetic.make_weights(models.SYMBOLS_2X, synthetic.DIMS_2X, 1008, 2, seed=1)
    model = models.from_weight_lists("2x", w, device=DEV, periodic_table_index=False)
    z, idx, coords, cell, pbc = synthetic.water_box(20, seed=2)          # L = 8.4 A
    thin = cell.clone()
    thin[2, 2] = 4.0                                                       # thinner than Rcr = 5.1 A
    args = ((idx.to(DEV), coords.to(DEV)), thin.to(DEV), pbc.to(DEV))
    with pytest.raises(RuntimeError, match="Cell is too small"):
        model(*args)
    with pytest.raises(RuntimeError, match="Cell is too small"):
        model.energies_and_forces(idx.to(DEV), coords.to(DEV), thin.to(DEV), pbc.to(DEV))
    # the status word is cleared by the raise: the next (valid) call works
    out = model((idx.to(DEV), coords.to(DEV)), cell.to(DEV), pbc.to(DEV))
    assert bool(torch.isfinite(out.energies).all())
    # neighbour overflow: 200 atoms inside a 3 A ball, nbr_cap = 128
    g = torch.Generator().manual_seed(0)
    blob = (torch.rand(1, 200, 3, generator=g) * 3.0).to(DEV)
    sp = torch.zeros(1, 200, dtype=torch.long, device=DEV)
    with pytest.raises(RuntimeError, match="nbr_cap"):
        model((sp, blob))
    # an engine on cuda:0 launches on cuda:0 whatever the current device is (device guard)
    if torch.cuda.device_count() > 1:
        with torch.cuda.device(1):
            out2 = model((idx.to(DEV), coords.to(DEV)), cell.to(DEV), pbc.to(DEV))
        assert torch.equal(out2.energies, out.energies)


def test_packed_weights_follow_in_place_edits():
    """In-place parameter edits (no invalidate_packed() call) and self-energy edits reach the kernels."""
    from torchani_b200 import models, synthetic
    w = synthetic.make_weights(models.SYMBOLS_2X, synthetic.DIMS_2X, 1008, 2, seed=1)
    model = models.from_weight_lists("2x", w, device=DEV, periodic_table_index=False)
    _, idx, coords, cell, pbc = synthetic.water_box(20, seed=2)
    args = ((idx.to(DEV), coords.to(DEV)), cell.to(DEV), pbc.to(DEV))
    e0 = float(model(*args).energies[0])
    with torch.no_grad():
        model.neural_networks.members[0].atomics["H"].final_layer.bias.add_(0.5)     # 40 H atoms, 2 members
    e1 = float(model(*args).energies[0])
    assert abs((e1 - e0) - 0.5 * 40 / 2) < 2e-3
    with torch.no_grad():
        model.energy_shifter.self_energies[3] += 1.0                                    # 20 O atoms
    e2 = float(model(*args).energies[0])
    assert abs((e2 - e1) - 20.0) < 2e-3
    model.energy_shifter._enabled = False
    e3 = float(model(*args).energies[0])
    assert abs(e3) < 50.0 and abs(e3 - e2) > 1e3


def test_operand_range_falls_back_to_the_bf16x3_build():
    """Weights scaled so that layer-1 activations leave the range of the 2 x fp16 operand pieces (|value| >= 1023):
    the device raises ANI_STATUS_OPERAND_RANGE, the model switches to the 3 x bfloat16 build of the library (both
    builds are loaded side by side) and redoes the step; the results agree with the float64 oracle."""
    import warnings
    from torchani_b200 import _lib, models
    if not _lib.available("bf16x3"):
        pytest.skip("libani_b200_bf16x3.so has not been built")
    om = oracle_model("2x", torch.float64, members=2)
    scaled = []
    for wm in om.weights:
        per = {}
        for s, layers in wm.items():
            (w1, b1), rest = layers[0], layers[1:]
            # x 30000 into layer 1, x 1/30000 on layer 2's input side: activations of layer 1 reach ~1e4-1e5
            (w2, b2) = rest[0]
            per[s] = [(w1 * 30000.0, b1 * 30000.0), (w2 / 30000.0, b2)] + list(rest[1:])
        scaled.append(per)
    om_scaled = om._replace(weights=scaled)
    rec = load_golden("water30_pbc_ani2x")
    species, coords, cell, pbc = golden_inputs(rec, torch.float64)
    ref = orc.compute(om_scaled, species, coords, cell, pbc)
    w32 = [{s: [(w.float(), b.float()) for w, b in layers] for s, layers in wm.items()} for wm in scaled]
    model = models.from_weight_lists("2x", w32, device=DEV, periodic_table_index=False)
    assert model.neural_networks._variant == ""
    c = coords.float().to(DEV)
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        e, f = model.energies_and_forces(species.to(DEV), c, cell.float().to(DEV), pbc.to(DEV))
    assert any("bfloat16" in str(w.message) for w in caught)
    assert model.neural_networks._variant == "bf16x3" and model.engine(torch.device(DEV)).variant == "bf16x3"
    scale = float(ref["forces"].abs().max())
    assert float((f.cpu().double() - ref["forces"]).abs().max()) < 1e-4 * max(1.0, scale)
    assert abs(float(e[0]) - float(ref["energy"][0])) < 1e-5 * abs(float(ref["energy"][0])) + 1e-3
    # the module-level container path falls back the same way
    model2 = models.from_weight_lists("2x", w32, device=DEV, periodic_table_index=False)
    aev = model2.aev_computer(species.to(DEV), c, cell.float().to(DEV), pbc.to(DEV))
    with warnings.catch_warnings(record=True):
        warnings.simplefilter("always")
        e2 = model2.neural_networks(species.to(DEV), aev)
    assert model2.neural_networks._variant == "bf16x3"
    assert abs(float(e2[0]) - float(ref["energy_nn"][0])) < 1e-5 * abs(float(ref["energy_nn"][0])) + 1e-3


def test_partial_pbc_and_periodic_batches_match_the_oracle():
    """`all_pairs` generality (neighbors.py:187-275): PBC in only some directions (slab: image shifts along the
    periodic lattice vectors only) and a batch of conformers in one shared periodic cell."""
    from torchani_b200 import models, neighbors
    rec = load_golden("water30_pbc_ani2x")
    species, coords, cell, _ = golden_inputs(rec, torch.float64)
    om = oracle_model("2x", torch.float64, "all_pairs")
    w32 = [{s: [(w.float(), b.float()) for w, b in layers] for s, layers in wm.items()} for wm in om.weights]
    model = models.from_weight_lists("2x", w32, device=DEV, periodic_table_index=False)
    sp_d, cell_d = species.to(DEV), cell.float().to(DEV)
    # --- slab: periodic in x and y only
    for flags in ([True, True, False], [False, True, False]):
        pbc = torch.tensor(flags)
        ref = orc.compute(om, species, coords, cell, pbc)
        c = coords.float().to(DEV).requires_grad_(True)
        e = model((sp_d, c), cell_d, pbc.to(DEV)).energies
        (g,) = torch.autograd.grad(e.sum(), c)
        assert abs(float(e[0]) - float(ref["energy"][0])) < 5e-3, flags
        assert_close(f"forces pbc={flags}", -g.cpu().numpy(), ref["forces"].numpy(), 0.0, F_ATOL)
        aev = model.aev_computer(sp_d, coords.float().to(DEV), cell_d, pbc.to(DEV))
        assert_close(f"aev pbc={flags}", aev.cpu().numpy(), ref["aev"].numpy(), AEV_RTOL, AEV_ATOL)
        nb = neighbors.AllPairs()(5.1, sp_d, coords.float().to(DEV), cell_d, pbc.to(DEV))
        assert nb.indices.shape[1] == int(ref["num_pairs"])
    # --- periodic batch: two conformers, one cell
    pbc = torch.tensor([True, True, True])
    co2 = torch.cat([coords, coords + 0.05 * torch.randn(coords.shape, generator=torch.Generator().manual_seed(3),
                                                         dtype=torch.float64)])
    sp2 = torch.cat([species, species])
    refs = [orc.compute(om, sp2[k:k + 1], co2[k:k + 1], cell, pbc) for k in range(2)]
    c = co2.float().to(DEV).requires_grad_(True)
    e = model((sp2.to(DEV), c), cell_d, pbc.to(DEV)).energies
    assert e.shape == (2,)
    (g,) = torch.autograd.grad(e.sum(), c)
    for k in range(2):
        assert abs(float(e[k]) - float(refs[k]["energy"][0])) < 5e-3
        assert_close("forces batch", -g[k:k + 1].cpu().numpy(), refs[k]["forces"].numpy(), 0.0, F_ATOL)
    nb = neighbors.AllPairs()(5.1, sp2.to(DEV), co2.float().to(DEV), cell_d, pbc.to(DEV))
    assert nb.indices.shape[1] == int(refs[0]["num_pairs"]) + int(refs[1]["num_pairs"])
    assert int(nb.indices.max()) >= 30      # indices into the flattened (C * A) atoms


def test_periodic_cell_thinner_than_the_cutoff_all_pairs_semantics():
    """neighbors.py:245-275: `all_pairs` pairs every atom with several lattice images when the cell is thinner than
    the cutoff (a cell list raises instead).  Here: a supercell of translation-equivalent copies."""
    from torchani_b200 import models
    from torchani_b200.aev import AEVComputer
    om = oracle_model("2x", torch.float64, "all_pairs", members=2)
    w32 = [{s: [(w.float(), b.float()) for w, b in layers] for s, layers in wm.items()} for wm in om.weights]
    g = torch.Generator().manual_seed(4)
    species = torch.tensor([[3, 0, 0, 1, 0, 2]])
    cell = torch.tensor([[4.2, 0.0, 0.0], [0.3, 3.9, 0.0], [0.0, 0.2, 9.0]], dtype=torch.float64)   # two thin directions
    frac = torch.rand(1, 6, 3, generator=g, dtype=torch.float64)
    coords = frac @ cell
    pbc = torch.tensor([True, True, True])
    ref = orc.compute(om, species, coords, cell, pbc)
    model = models.from_weight_lists("2x", w32, device=DEV, neighborlist="all_pairs", periodic_table_index=False)
    c = coords.float().to(DEV).requires_grad_(True)
    e = model((species.to(DEV), c), cell.float().to(DEV), pbc.to(DEV)).energies
    (gr,) = torch.autograd.grad(e.sum(), c)
    assert abs(float(e[0]) - float(ref["energy"][0])) < 2e-3
    assert_close("forces", -gr.cpu().numpy(), ref["forces"].numpy(), 0.0, F_ATOL)
    at = model((species.to(DEV), coords.float().to(DEV)), cell.float().to(DEV), pbc.to(DEV), atomic=True).energies
    assert at.shape == (1, 6)
    aev = AEVComputer.like_2x(neighborlist="all_pairs").to(DEV)(species.to(DEV), coords.float().to(DEV),
                                                               cell.float().to(DEV), pbc.to(DEV))
    assert_close("aev", aev.cpu().numpy(), ref["aev"].numpy(), AEV_RTOL, AEV_ATOL)
    # the cell-list flavour keeps the reference's error
    strict = models.from_weight_lists("2x", w32, device=DEV, neighborlist="cell_list", periodic_table_index=False)
    with pytest.raises(RuntimeError, match="too small"):
        strict((species.to(DEV), coords.float().to(DEV)), cell.float().to(DEV), pbc.to(DEV))


def test_bench_dump_outputs(tmp_path):
    """bench.py --dump-outputs: the last timed step of both timed paths, written as .npy, is the energy and force
    of the seeded workload (checked against the float64 oracle), and --steps is the number of timed steps."""
    import json
    import subprocess
    import sys
    from helpers import ROOT
    out = tmp_path / "dump"
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "water1k", "--molecules", "100",
                          "--steps", "2", "--warmup", "3", "--cpu-steps", "0", "--dump-outputs", str(out)],
                         capture_output=True, text=True, timeout=600, cwd=str(tmp_path))
    assert res.returncode == 0, res.stderr[-3000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["config"]["atoms"] == 300
    d = {p.stem: np.load(p) for p in out.glob("*.npy")}
    assert sorted(d) == ["e2e_energies", "e2e_forces", "energies", "grad"]
    assert d["energies"].dtype == np.float64 and d["energies"].shape == (1,)
    assert d["grad"].dtype == np.float32 and d["grad"].shape == (1, 300, 3)
    assert d["e2e_energies"].dtype == np.float64 and d["e2e_forces"].dtype == np.float32
    from torchani_b200 import synthetic
    _, idx, coords, cell, pbc = synthetic.water_box(100, seed=0)
    ref = orc.compute(oracle_model("2x", torch.float64), idx, coords.double(), cell.double(), pbc)
    assert abs(float(d["energies"][0]) - float(ref["energy"][0])) < 5e-3             # float32 total
    assert_close("forces", -d["grad"], ref["forces"].numpy(), 0.0, F_ATOL)
    assert abs(float(d["e2e_energies"][0]) - float(ref["energy"][0])) < 5e-3
    assert_close("e2e forces", d["e2e_forces"], ref["forces"][0].numpy(), 0.0, F_ATOL)
