"""The resident-chain MLP kernel (csrc/gemm_resident.cuh) against the other two schedules of the same step.

A CTA runs one (row tile, member) chain at a time with the layer-to-layer operands in shared memory; the arithmetic,
the operand split and the K order of every accumulator are those of the chained launches, so results agree with them
to rounding (the layer-1 backward's split-K REDs into dE/dAEV are the only sums whose order varies) -- the bars of
test_gpu_parity.py::test_dataflow_mlp_launch_matches_the_chained_launches."""
import pytest
import torch

from helpers import oracle_model

pytestmark = pytest.mark.gpu

ARMS = {   # name -> (ANI_B200_MLP_FUSED, ANI_B200_MLP_RESIDENT)
    "chained": ("0", "0"),
    "dataflow": ("1", "0"),
    "resident": ("1", "1"),
}


@pytest.fixture(scope="module")
def nets():
    from torchani_b200.engine import PackedNetworks, constants_1x, constants_2x
    dev = torch.device("cuda:0")
    out = {}
    for kind, consts in (("2x", constants_2x()), ("1x", constants_1x())):
        m = oracle_model(kind)
        out[kind] = (consts, PackedNetworks([[wm[s] for s in m.symbols] for wm in m.weights], consts.out_dim, dev),
                     [m.sae[s] for s in m.symbols])
    return out


def engine(nets, kind, arm, monkeypatch):
    """A fresh engine per arm: its CUDA graphs are captured with that arm's kernel."""
    from torchani_b200.engine import Engine
    fused, resident = ARMS[arm]
    monkeypatch.setenv("ANI_B200_MLP_RESIDENT", resident)
    monkeypatch.delenv("ANI_B200_MLP_CHAIN", raising=False)
    consts, pn, sae = nets[kind]
    eng = Engine(consts, pn, sae)
    eng.mlp_mode = fused
    return eng


def run_arms(nets, kind, system, monkeypatch, want_grad=True, steps=5):
    """Per arm: the first (eager) step and the last one (CUDA-graph replay)."""
    sp, co, ce = system
    out = {}
    for arm in ARMS:
        eng = engine(nets, kind, arm, monkeypatch)
        assert eng.mlp_schedule(sp.numel(), eng.workspace(*sp.shape).rows_cap) == arm
        res = []
        for i in range(steps):
            r = eng.step(sp, co, ce, want_grad)
            if i in (0, steps - 1):
                res.append((r.energies.clone(), r.grad.clone() if want_grad else None, r.member_atomic.clone()))
        eng.check_status()
        out[arm] = res
    return out


def assert_agree(a, b, n_atoms, want_grad=True):
    assert float((a[0] - b[0]).abs().max()) < 1e-6 * max(1, n_atoms)
    if want_grad:
        assert float((a[1] - b[1]).abs().max()) < 2e-6
    assert float((a[2] - b[2]).abs().max()) < 1e-6


def water(n_mol, seed=17):
    from torchani_b200 import synthetic
    d = torch.device("cuda:0")
    _, idx, coords, cell, _ = synthetic.water_box(n_mol, seed=seed)
    return idx.to(d), coords.to(d), cell.to(d)


@pytest.mark.parametrize("n_mol", [20, 333, 3333])
def test_resident_mlp_matches_the_other_schedules_on_water(nets, n_mol, monkeypatch):
    """Fewer chains than SMs, about two per SM, and four or five per SM; eager steps and graph replays."""
    out = run_arms(nets, "2x", water(n_mol), monkeypatch)
    for k in (0, 1):
        assert_agree(out["resident"][k], out["chained"][k], 3 * n_mol)
        assert_agree(out["resident"][k], out["dataflow"][k], 3 * n_mol)


def test_resident_mlp_on_five_elements(nets, monkeypatch):
    """H C N O S: twenty live AEV column blocks, so the layer-1 backward of a chain runs three dE/dAEV column tiles."""
    from torchani_b200 import synthetic
    d = torch.device("cuda:0")
    _, idx, coords, cell, _ = synthetic.protein_in_water(12001, seed=3)
    assert set(idx.unique().tolist()) == {0, 1, 2, 3, 4}
    out = run_arms(nets, "2x", (idx.to(d), coords.to(d), cell.to(d)), monkeypatch)
    for k in (0, 1):
        assert_agree(out["resident"][k], out["chained"][k], idx.numel())


def test_resident_mlp_ani1x(nets, monkeypatch):
    """ANI-1x: hidden widths 160 / 144 / 128 / 112 / 96, padded to multiples of 32 (smaller resident image)."""
    out = run_arms(nets, "1x", water(700, seed=4), monkeypatch)
    for k in (0, 1):
        assert_agree(out["resident"][k], out["chained"][k], 2100)


def test_resident_mlp_energies_only(nets, monkeypatch):
    """want_backward = 0: a chain stops at the head."""
    out = run_arms(nets, "2x", water(1500, seed=6), monkeypatch, want_grad=False)
    for k in (0, 1):
        assert_agree(out["resident"][k], out["chained"][k], 4500, want_grad=False)


def test_resident_mlp_members_forces(nets, monkeypatch):
    """want_backward = 2 (Engine.step_members): one dE_m/dAEV slab per member, plain stores."""
    sp, co, ce = water(900, seed=8)
    out = {}
    for arm in ("dataflow", "resident"):
        eng = engine(nets, "2x", arm, monkeypatch)
        e_m, g_m = eng.step_members(sp, co, ce, True)
        eng.check_status()
        out[arm] = (e_m.clone(), g_m.clone())
    assert float((out["resident"][0] - out["dataflow"][0]).abs().max()) < 1e-6 * 2700
    # one member per slab: no split-K sum, so the same bar as the summed gradient
    assert float((out["resident"][1] - out["dataflow"][1]).abs().max()) < 2e-6


def test_resident_mlp_eight_shards_sum_to_the_whole(nets, monkeypatch):
    """Sharded row ranges: what eight ranks compute adds up to the single-GPU step."""
    sp, co, ce = water(3333, seed=9)
    eng = engine(nets, "2x", "resident", monkeypatch)
    whole = eng.step(sp, co, ce, True)
    e0, g0 = float(whole.energies[0]), whole.grad.clone()
    parts_e, parts_g = 0.0, torch.zeros_like(g0)
    for r in range(8):
        rr = eng.step(sp, co, ce, True, shard=(r, 8))
        parts_e += float(rr.energies[0])
        parts_g += rr.grad
    eng.check_status()
    assert abs(parts_e - e0) < 1e-5
    assert float((parts_g - g0).abs().max()) < 2e-5
