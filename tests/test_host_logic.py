"""Host-side logic that needs no GPU: weight packing, constants, module trees / state dicts,
species conversion, sharding arithmetic and the 2-rank (gloo) reduction of partial results."""
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import oracle.ani_oracle as orc
from helpers import ROOT, golden_inputs, load_golden, oracle_model


def test_constants_match_oracle_spec():
    from torchani_b200.engine import constants_1x, constants_2x
    for mine, ref in ((constants_2x(), orc.aev_spec_2x()), (constants_1x(), orc.aev_spec_1x())):
        assert mine.out_dim == ref.out_dim and mine.radial_len == ref.radial_len
        assert mine.shf_r == ref.shf_r and mine.shf_a == ref.shf_a and mine.shf_z == ref.shf_z
        st = mine.to_struct()
        assert st.eta_r == np.float32(ref.eta_r) and st.zeta == np.float32(ref.zeta)
        assert abs(st.cos_z[0] - math.cos(np.float32(ref.shf_z[0]))) < 1e-7
    assert constants_2x().out_dim == 1008 and constants_1x().out_dim == 384


def test_unsupported_configurations_are_rejected_loudly():
    from torchani_b200.engine import constants_2x
    with pytest.raises(ValueError):
        constants_2x()._replace(shf_a=(0.9, 1.0, 1.1)).to_struct()
    with pytest.raises(ValueError):
        constants_2x()._replace(cutoff_fn="triweight").to_struct()
    from torchani_b200.aev import AEVComputer
    with pytest.raises(ValueError):
        AEVComputer.like_2x(strategy="pyaev")
    with pytest.raises(ValueError):
        AEVComputer.like_2x().set_strategy("cuaev")
    from torchani_b200.nn import AtomicNetwork
    with pytest.raises(ValueError):
        AtomicNetwork((1008, 256, 192, 160, 1), activation="gelu")


def _piece_to_f32(u16, parts):
    if parts == 2:
        return u16.view(np.float16).astype(np.float32)
    return (u16.astype(np.uint32) << 16).view(np.float32)


def _untile(t, n, k):
    """Inverse of engine.tile_b_operand (numpy, element-wise from the documented layout of
    include/ani_b200.h): returns the 16-bit pieces (still scaled) as float32 arrays."""
    from torchani_b200._lib import operand_format
    P = operand_format().parts
    kp = (k + 31) // 32 * 32
    nkb = kp // 32
    t = t.view(torch.int16).numpy().view(np.uint16)
    parts = [np.zeros((n, kp), np.float32) for _ in range(P)]
    for r in range(n):
        n0 = r // 256 * 256
        bn = min(256, n - n0)
        rr = r - n0
        for kb in range(nkb):
            for ch in range(4):
                # element offsets: n tile base, K-block base (P pieces of bn x 32), 8-row group, row, swizzled chunk
                base = n0 * nkb * 32 * P + kb * bn * 32 * P + (rr // 8) * 256 + (rr % 8) * 32 + ((ch ^ ((rr >> 1) & 3)) * 8)
                for p in range(P):
                    parts[p][r, kb * 32 + ch * 8: kb * 32 + ch * 8 + 8] = _piece_to_f32(
                        t[base + p * bn * 32: base + p * bn * 32 + 8], P)
    return parts


def test_weight_packing_layout():
    from torchani_b200._lib import operand_format
    from torchani_b200.engine import tile_a_operand, tile_b_operand, untile_a_operand, weight_scale
    P = operand_format().parts
    # the tiled / split / swizzled B operand round-trips and the pieces add up to scale * x
    b = torch.randn(288, 40, generator=torch.Generator().manual_seed(0))
    sc = weight_scale([b])
    assert sc == (1.0 if P == 3 else 2.0 ** np.floor(np.log2(16384.0 / float(b.abs().max()))))
    parts = _untile(tile_b_operand(b, sc), 288, 40)
    assert parts[0].shape == (288, 64)                                # K padded to a multiple of 32
    total = sum(q.astype(np.float64) for q in parts)[:, :40] / sc
    # 3 x bf16: 24 significant bits; 2 x fp16: 22 bits, absolute floor 2^-25 / scale (half subnormals)
    tol = np.abs(b.numpy()) * (2.0 ** -24 if P == 3 else 2.0 ** -22) + (0.0 if P == 3 else 2.0 ** -25 / sc)
    assert (np.abs(total - b.numpy()) <= tol).all()
    assert float(np.abs(parts[0][:, 40:]).max()) == 0.0
    step = 2.0 ** -8 if P == 3 else 2.0 ** -11
    for k in range(1, P):
        assert np.abs(parts[k]).max() <= np.abs(b.numpy()).max() * sc * step ** k
    # A operand: tile / untile round trip
    x = torch.randn(256, 96, generator=torch.Generator().manual_seed(1))
    back = untile_a_operand(tile_a_operand(x), 256, 96)
    assert float((back - x).abs().max()) <= float(x.abs().max()) * 2.0 ** -22
    # (the device-side packer ani_b200_pack_b_operand is compared with this tiler byte for byte in
    # tests/test_gpu_api.py::test_weight_packing_kernel_matches_the_python_tiler)


def test_model_tree_and_reference_state_dict_keys():
    from torchani_b200 import models
    m = models.ANI2x(seed=1)
    keys = set(m.state_dict().keys())
    assert "neural_networks.members.7.atomics.Cl.final_layer.bias" in keys
    assert "neural_networks.members.0.atomics.H.layers.0.weight" in keys
    assert m.aev_computer.out_dim == 1008 and len(m) == 8
    assert sum(p.numel() for p in m.neural_networks.members[0].parameters()) == 1713223  # SURVEY 8
    # the reference's key names (arch.py:278-290) load
    sd = {}
    for k, v in m.state_dict().items():
        k = k.replace("aev_computer.", "potentials.nnp.aev_computer.") if k.startswith("aev_computer.") else k
        k = k.replace("neural_networks.", "potentials.nnp.neural_networks.") if k.startswith("neural_networks.") else k
        sd[k] = v.clone()
    m2 = models.ANI2x(seed=2)
    m2.load_state_dict(sd)
    a = m.neural_networks.members[3].atomics["O"].layers[1].weight
    b = m2.neural_networks.members[3].atomics["O"].layers[1].weight
    assert torch.equal(a, b)
    sub = m[2]
    assert len(sub) == 1 and sub.neural_networks.num_species == 7


def test_species_converter_and_self_energy():
    from torchani_b200.models import SelfEnergy
    from torchani_b200.nn import SpeciesConverter
    conv = SpeciesConverter(["H", "C", "N", "O"])
    z = torch.tensor([[6, 1, 1, 1, 1], [7, 1, 1, 1, -1]])
    assert conv(z).tolist() == [[1, 0, 0, 0, 0], [2, 0, 0, 0, -1]]
    with pytest.raises(ValueError):
        conv(torch.tensor([[16, 1]]))
    sae = SelfEnergy.with_gsaes(["H", "C", "N", "O"])
    e = sae(conv(z))
    assert abs(float(e[1]) - (-54.5732825 - 3 * 0.4993212)) < 1e-9


def test_shard_bounds_cover_everything():
    from torchani_b200.parallel import shard_bounds
    for n in (1, 7, 999, 9999):
        for world in (1, 2, 3, 8):
            spans = [shard_bounds(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))


_GLOO_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from torchani_b200.parallel import allreduce_partials, shard_bounds
dist.init_process_group("gloo", rank=int(os.environ["RANK"]), world_size=int(os.environ["WORLD_SIZE"]))
r, w = dist.get_rank(), dist.get_world_size()
torch.manual_seed(0)
full_grad = torch.randn(3, 10, 3)
full_e = torch.randn(3, dtype=torch.float64)
lo, hi = shard_bounds(30, r, w)
mask = torch.zeros(30); mask[lo:hi] = 1
part_grad = (full_grad.view(30, 3) * mask.view(-1, 1)).view(3, 10, 3)
part_e = full_e * (1.0 / w)
grad, e = allreduce_partials(part_grad, part_e)
assert torch.allclose(grad.float(), full_grad, atol=1e-6), "gradient all-reduce wrong"
assert torch.allclose(e, full_e, atol=1e-12)
dist.destroy_process_group()
print("ok", r)
'''


def test_two_rank_gloo_allreduce_of_partials(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_GLOO_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29631", WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, str(script), ROOT], env=dict(env, RANK=str(r)),
                              stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True) for r in range(2)]
    for p in procs:
        out, err = p.communicate(timeout=120)
        assert p.returncode == 0, err
        assert "ok" in out


def test_synthetic_generators_agree_with_the_oracle_copies():
    from torchani_b200 import synthetic
    a = synthetic.water_box(20, seed=3)
    b = orc.water_box(20, seed=3)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    sa, ca = synthetic.conformer_batch(5, seed=2)
    sb, cb = orc.conformer_batch(5, seed=2)
    assert torch.equal(sa, sb) and torch.equal(ca, cb)
    wa = synthetic.make_weights(("H", "O"), synthetic.DIMS_2X, 1008, 2, seed=9)
    wb = orc.make_weights(("H", "O"), orc.DIMS_2X, 1008, 2, seed=9)
    assert torch.equal(wa[1]["O"][2][0], wb[1]["O"][2][0])


def test_operand_format_and_weight_scales():
    """The GEMM operand format of the loaded build and the per-tensor power-of-two weight scales."""
    from torchani_b200 import _lib
    from torchani_b200.engine import weight_scale
    fmt = _lib.operand_format()
    assert fmt.parts in (2, 3)
    if fmt.parts == 2:
        assert fmt.value_scale == 64.0 and fmt.grad_scale == 4096.0
        assert weight_scale([torch.full((4, 4), 0.03)]) == 4096.0            # capped at 2^12
        assert weight_scale([torch.full((4, 4), 100.0)]) == 128.0            # 100 * 128 < 2^14 <= 100 * 256
        assert weight_scale([torch.zeros(2, 2)]) == 4096.0
        with pytest.raises(ValueError):
            weight_scale([torch.tensor([[float("nan")]])])
    else:
        assert fmt.value_scale == 1.0 and weight_scale([torch.ones(2, 2)]) == 1.0


def test_neighborlist_table_and_verlet_arguments():
    from torchani_b200 import neighbors
    assert isinstance(neighbors._parse_neighborlist("verlet_cell_list"), neighbors.VerletCellList)
    assert isinstance(neighbors._parse_neighborlist("adaptive"), neighbors.AdaptiveList)
    with pytest.raises(ValueError):
        neighbors.VerletCellList(skin=-1.0)
    with pytest.raises(ValueError):
        neighbors._parse_neighborlist("octree")


def test_oracle_stress_is_the_strain_derivative():
    """oracle stress (ase.py:110-121,170-173, 'scaling'): symmetric for wrapped atoms and equal to the
    finite-difference strain derivative of the energy."""
    rec = load_golden("water30_pbc_ani2x")
    sp, co, cell, pbc = golden_inputs(rec, torch.float64)
    co = co - torch.floor(co @ torch.linalg.inv(cell)) @ cell
    m = oracle_model("2x", torch.float64, "cell_list", members=2)
    out = orc.compute(m, sp, co, cell, pbc, stress=True)
    s = out["stress"]
    assert float((s - s.T).abs().max()) < 1e-12
    eps = 1e-5
    sc = torch.eye(3, dtype=torch.float64)
    sc[0, 1] += eps
    ep = float(orc.compute(m, sp, co @ sc, cell @ sc, pbc, forces=False)["energy_nn"][0])
    sc[0, 1] -= 2 * eps
    em = float(orc.compute(m, sp, co @ sc, cell @ sc, pbc, forces=False)["energy_nn"][0])
    assert abs((ep - em) / (2 * eps) / float(torch.det(cell)) - float(s[0, 1])) < 1e-9


def test_bench_reference_arm_line(tmp_path):
    """bench.py --impl reference: one JSON line with the contract's keys (tiny box so that it runs in seconds)."""
    import json
    import subprocess
    import sys
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--molecules", "20",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=300, cwd=str(tmp_path))
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    import oracle.ref_torchani as rt
    staged = rt.available()
    # the real reference where it is available, else the CPU port of its algorithm
    assert d["impl"] == "reference" and d["cpu_baseline"]["kind"] == ("reference" if staged else "port")
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["cpu_baseline"]["cores"] >= 1 and d["config"]["atoms"] == 60


def test_species_major_staging_arithmetic():
    """The index arithmetic of k_aev_forward_cta's staging (csrc/aev.cu, steps (b)-(d)) restated in numpy:
    from the 27 species-sorted candidate ranges, counts per (species, range) -> exclusive prefix in species-major
    order -> adj[s][o] = off[s][o] - (candidates of lower species in range o) -> place = adj + offset in range.
    The places must be a permutation that groups the candidates by species and keeps range-major order inside a
    species; the windowed scan must visit every species segment exactly once and report the right segment ends."""
    rng = np.random.default_rng(11)
    S, R, CAP = 7, 27, 64          # a small window capacity forces several staging windows
    for trial in range(20):
        lens = rng.integers(0, 9, size=R)
        lens[rng.integers(0, R, size=5)] = 0
        species = [np.sort(rng.integers(0, S, size=n)) for n in lens]       # every range is species-sorted
        r_off = np.concatenate([[0], np.cumsum(lens)])
        T = int(r_off[-1])
        cnt = np.zeros((S, R), dtype=int)
        for o in range(R):
            for sp in species[o]:
                cnt[sp, o] += 1
        off = np.concatenate([[0], np.cumsum(cnt.reshape(-1))])            # q = s * R + o
        adj = np.zeros((S, R), dtype=int)
        for o in range(R):
            lower = 0
            for s in range(S):
                adj[s, o] = off[s * R + o] - lower
                lower += cnt[s, o]
        dest, sp_of, key = np.zeros(T, dtype=int), np.zeros(T, dtype=int), []
        for t in range(T):
            o = int(np.searchsorted(r_off, t, side="right") - 1)
            while lens[o] == 0:                                             # (the kernel's search never lands here)
                o += 1
            k = t - r_off[o]
            sp = species[o][k]
            dest[t], sp_of[t] = adj[sp, o] + k, sp
            key.append((sp, o, k))
        assert sorted(dest.tolist()) == list(range(T))                      # a permutation
        order = np.argsort(dest)
        assert [key[i] for i in order] == sorted(key)                       # species-major, then range, then offset
        # windows of CAP places: the segment of species s inside window [F0, F0 + CAP) is [max(F0, a), min(F0 + CAP, b))
        seen = np.zeros(T, dtype=int)
        seg_end = np.zeros(S + 1, dtype=int)
        count = 0
        for F0 in range(0, max(T, 1), CAP):
            for s in range(S):
                a, b = max(F0, off[s * R]), min(F0 + CAP, off[(s + 1) * R])
                for p in range(a, b):
                    seen[p] += 1
                    count += 1
                if off[(s + 1) * R] >= F0:                                  # the rule that fixed the benzene case
                    seg_end[s + 1] = count
        assert (seen == 1).all()
        assert seg_end[1:].tolist() == [int(off[(s + 1) * R]) for s in range(S)]


def _column_live(c, mask, S, n_shf_r, angular_sub, out_dim, pad):
    """Python statement of aev_column_live (csrc/cells.cu): internal column c of the tiled AEV operand -- radial block,
    `pad` never-written columns, angular block of `angular_sub` columns per element pair (row-major upper triangle)."""
    RL = S * n_shf_r
    if c < RL:
        return bool((mask >> (c // n_shf_r)) & 1)
    c -= pad
    if c < RL or c >= out_dim:
        return False
    s1, rem = 0, (c - RL) // angular_sub
    while rem >= S - s1:
        rem -= S - s1
        s1 += 1
    return bool((mask >> s1) & 1) and bool((mask >> (s1 + rem)) & 1)


def test_aligned_angular_block_live_blocks():
    """ani_aev_params::ang_pad: with the angular block of ANI-2x on a 32-column boundary every element pair fills exactly
    one 32-column GEMM block.  Live blocks for water / H C N O S, reference order vs internal order; the padded layout
    still fits ldx = 1024 and maps every reference column to a distinct internal column."""
    S, nR, sub, out_dim, ldx = 7, 16, 32, 1008, 1024
    pad = (-S * nR) % 32
    assert pad == 16 and out_dim + pad == ldx

    def live_blocks(mask, pad):
        return [b for b in range(ldx // 32) if any(_column_live(c, mask, S, nR, sub, out_dim, pad) for c in range(32 * b, 32 * b + 32))]

    water = (1 << 0) | (1 << 3)                         # H, O of (H, C, N, O, S, F, Cl)
    hcnos = (1 << 0) | (1 << 1) | (1 << 2) | (1 << 3) | (1 << 4)
    assert len(live_blocks(water, 0)) == 8 and len(live_blocks(water, pad)) == 5
    assert len(live_blocks(hcnos, pad)) == 3 + 15       # radial blocks {0, 1, 2} + one block per element pair
    assert len(live_blocks(hcnos, pad)) < len(live_blocks(hcnos, 0))
    internal = [c if c < S * nR else c + pad for c in range(out_dim)]   # what PackedNetworks / the AEV kernels apply
    assert len(set(internal)) == out_dim and max(internal) < ldx
    assert all(_column_live(ci, 0x7f, S, nR, sub, out_dim, pad) for ci in internal)
    assert not any(_column_live(c, 0x7f, S, nR, sub, out_dim, pad) for c in range(S * nR, S * nR + pad))


def test_chain_walk_covers_every_unit_once_in_dependency_order():
    """Python statement of ChainWalk (csrc/gemm_chain.cuh): CTA c runs rounds of D chains, inside a round unit-major and
    chain-minor.  Every (chain, unit) is visited exactly once by exactly one CTA, a chain's units appear in order in its
    CTA's sequence, and with D >= 2 full slots a unit's predecessor is at least D - 1 units back (what the shared-memory
    barriers and the lagged publication of finished units rely on)."""
    def walk(G, c, D, U, num_chains):
        out, rnd = [], 0
        while c + G * D * rnd < num_chains:
            for u in range(U):
                for j in range(D):
                    chain = c + G * D * rnd + G * j
                    if chain < num_chains:
                        out.append((j, chain, u))
            rnd += 1
        return out

    for G, D, U, num_chains in ((148, 3, 6, 632), (148, 1, 6, 72), (4, 2, 8, 11), (148, 8, 6, 3200), (5, 4, 3, 5)):
        seen = {}
        for c in range(G):
            seq = walk(G, c, D, U, num_chains)
            pos = {}
            for k, (slot, chain, u) in enumerate(seq):
                assert (chain, u) not in seen
                seen[(chain, u)] = c
                pos[(chain, u)] = k
                if u > 0:
                    assert pos[(chain, u - 1)] < k                       # producer first, same CTA
            # the device picks the interleave depth so that rounds are equally deep (k_mlp_chain)
        assert len(seen) == num_chains * U
        per_cta = -(-num_chains // G)
        rounds = -(-per_cta // 8)
        assert 1 <= -(-per_cta // rounds) <= 8


def test_row_tile_windows_partition_the_tiles():
    """build_tile_map (csrc/gemm_tc.cuh): window w of W takes tiles [first + n w / W, first + n (w + 1) / W) of every
    species -- a partition, whatever the counts."""
    for counts in ((53, 27), (1, 0, 3), (7,), (400, 0, 0, 13, 2)):
        for W in (1, 2, 3, 4, 16):
            first = np.concatenate([[0], np.cumsum(counts)])
            taken = []
            for w in range(W):
                for s, n in enumerate(counts):
                    lo, hi = first[s] + n * w // W, first[s] + n * (w + 1) // W
                    taken += list(range(lo, hi))
            assert sorted(taken) == list(range(sum(counts)))
