"""Host side of the fused hot path: owns the device workspaces (the C-ABI never allocates) and
sequences the kernels of ``libani_b200.so`` on the current CUDA stream.

One step  =  bucket grid -> species layout -> fused neighbour search + AEV -> ensemble MLP
forward + backward-to-AEV -> AEV backward (dE/dcoords) -> energy reduction.  No host
synchronisation happens inside a step; device-side error conditions accumulate in a status
word that is checked when results are read (``Engine.check_status``).

PyTorch is used only for device memory, streams and (in ``parallel.py``) torch.distributed.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import typing as tp

import numpy as np
import torch
from torch import Tensor

from . import _lib
from ._lib import AEVParams, Grid, MLPModel, check, ptr

TILE = _lib.ANI_TILE_ROWS


def _f32(v: float) -> float:
    return float(np.float32(v))


class AEVConstants(tp.NamedTuple):
    """The numbers that define an ANI AEV (see aev/_computer.py:499-600 in the reference)."""

    num_species: int
    rcr: float
    rca: float
    eta_r: float
    shf_r: tp.Tuple[float, ...]
    eta_a: float
    zeta: float
    shf_a: tp.Tuple[float, ...]
    shf_z: tp.Tuple[float, ...]
    cutoff_fn: str = "cosine"

    @property
    def radial_len(self) -> int:
        return self.num_species * len(self.shf_r)

    @property
    def angular_len(self) -> int:
        return self.num_species * (self.num_species + 1) // 2 * len(self.shf_a) * len(self.shf_z)

    @property
    def out_dim(self) -> int:
        return self.radial_len + self.angular_len

    def to_struct(self) -> AEVParams:
        if self.cutoff_fn not in ("cosine", "smooth"):
            raise ValueError(f"cutoff function {self.cutoff_fn!r} is not supported by the B200 kernels")
        if (len(self.shf_a), len(self.shf_z)) not in ((8, 4), (4, 8)):
            raise ValueError("the B200 AEV kernels need ShfA x ShfZ = 8x4 (ANI-2x) or 4x8 (ANI-1x)")
        if len(self.shf_r) > _lib.ANI_MAX_SHFR or self.num_species > _lib.ANI_MAX_SPECIES:
            raise ValueError("too many radial shifts / species for the B200 kernels")
        p = AEVParams()
        p.rcr, p.rca = self.rcr, self.rca
        # the reference keeps eta/zeta/shifts as float32 buffers (aev/_terms.py:153-156,288-292)
        p.eta_r, p.eta_a, p.zeta = _f32(self.eta_r), _f32(self.eta_a), _f32(self.zeta)
        p.n_shf_r, p.n_shf_a, p.n_shf_z = len(self.shf_r), len(self.shf_a), len(self.shf_z)
        p.num_species = self.num_species
        p.cutoff_kind = 0 if self.cutoff_fn == "cosine" else 1
        for k, v in enumerate(self.shf_r):
            p.shf_r[k] = _f32(v)
        for k, v in enumerate(self.shf_a):
            p.shf_a[k] = _f32(v)
        for k, v in enumerate(self.shf_z):
            p.cos_z[k] = math.cos(_f32(v))
            p.sin_z[k] = math.sin(_f32(v))
        return p


def _linspace(start: float, stop: float, steps: int) -> tp.Tuple[float, ...]:
    return tuple(start + ((stop - start) / steps) * j for j in range(steps))  # utils.py:101-107


def constants_2x(num_species: int = 7, cutoff_fn: str = "cosine") -> AEVConstants:
    a0 = math.pi / 4 / 2
    return AEVConstants(num_species, 5.1, 3.5, 19.7, _linspace(0.8, 5.1, 16), 12.5, 14.1,
                        _linspace(0.8, 3.5, 8), _linspace(a0, math.pi + a0, 4), cutoff_fn)


def constants_1x(num_species: int = 4, cutoff_fn: str = "cosine") -> AEVConstants:
    a0 = math.pi / 8 / 2
    return AEVConstants(num_species, 5.2, 3.5, 16.0, _linspace(0.9, 5.2, 16), 8.0, 32.0,
                        _linspace(0.9, 3.5, 4), _linspace(a0, math.pi + a0, 8), cutoff_fn)


def _split(x: Tensor, scale: float = 1.0, variant: tp.Optional[str] = None) -> tp.List[Tensor]:
    """x (float32) -> the 16-bit pieces of ``scale * x`` in the library's operand format
    (``_lib.operand_format``): two IEEE half pieces or three bfloat16 pieces, each rounded to
    nearest, ``scale * x = p1 + p2 (+ p3)``."""
    fmt = _lib.operand_format(variant)
    dt = torch.float16 if fmt.parts == 2 else torch.bfloat16
    r = x.to(torch.float32) * scale
    out = []
    for _ in range(fmt.parts):
        p = r.to(dt)
        out.append(p)
        r = r - p.to(torch.float32)
    return out


def weight_scale(ws: tp.Sequence[Tensor], variant: tp.Optional[str] = None) -> float:
    """Power-of-two operand scale for a group of weight matrices (half pieces: the largest
    |scale * w| stays below 2^14, the scale below 2^12; bfloat16 pieces need none)."""
    if _lib.operand_format(variant).parts != 2:
        return 1.0
    top = max(float(w.abs().max()) for w in ws)
    if not math.isfinite(top):
        raise ValueError("network weights contain inf/NaN")
    if top == 0.0:
        return 4096.0
    return float(min(4096.0, max(1.0, 2.0 ** math.floor(math.log2(16384.0 / top)))))


def _swizzle_index(device) -> Tensor:
    """idx[row in 8-row group][position] = the 16-byte chunk stored at that position (SWIZZLE_64B)."""
    rows = torch.arange(8, device=device).view(8, 1)
    pos = torch.arange(4, device=device).view(1, 4)
    return pos ^ ((rows >> 1) & 3)


def tile_b_operand(b: Tensor, scale: float = 1.0, variant: tp.Optional[str] = None) -> Tensor:
    """``B[N][K]`` (float32, K-major, N % 32 == 0) -> the "tiled B operand" byte layout of
    include/ani_b200.h: K zero-padded to 32, the 16-bit pieces of ``scale * B``,
    [n tile of 256 rows][k block of 32][p1 bn x 64 B | p2 (| p3)] with every 8-row group in tcgen05
    SWIZZLE_64B order.  Returned as a flat 16-bit tensor."""
    n, k = b.shape
    assert n % 32 == 0, "rows of a B operand must come in groups of 32"
    kp = (k + 31) // 32 * 32
    nkb = kp // 32
    bp = torch.zeros(n, kp, dtype=torch.float32, device=b.device)
    bp[:, :k] = b
    pieces = _split(bp, scale, variant)
    src_chunk = _swizzle_index(b.device)
    out = []
    for n0 in range(0, n, 256):
        bn = min(256, n - n0)
        parts = []
        idx = src_chunk.view(1, 1, 8, 4, 1).expand(nkb, bn // 8, 8, 4, 8)
        for part in pieces:
            x = part[n0:n0 + bn].view(bn // 8, 8, nkb, 4, 8)           # [group][row][kb][chunk][8]
            x = x.permute(2, 0, 1, 3, 4)                                # [kb][group][row][chunk][8]
            parts.append(torch.gather(x, 3, idx).reshape(nkb, bn * 32))
        out.append(torch.stack(parts, 1).reshape(-1))                  # [kb][piece][bn*32]
    return torch.cat(out).contiguous()


def tile_a_operand(x: Tensor, scale: tp.Optional[float] = None, variant: tp.Optional[str] = None) -> Tensor:
    """Plain ``[rows][cols]`` float32 (rows % 128 == 0, cols % 32 == 0) -> flat "tiled operand"
    (A-operand form of include/ani_b200.h; ``scale`` defaults to the library's value scale).
    Plumbing for the API paths that receive plain AEVs."""
    rows, cols = x.shape
    assert rows % 128 == 0 and cols % 32 == 0
    nkb = cols // 32
    if scale is None:
        scale = _lib.operand_format(variant).value_scale
    idx = _swizzle_index(x.device).view(1, 1, 1, 8, 4, 1).expand(rows // 128, nkb, 16, 8, 4, 8)
    parts = []
    for part in _split(x.contiguous().to(torch.float32), scale, variant):
        v = part.view(rows // 128, 16, 8, nkb, 4, 8).permute(0, 3, 1, 2, 4, 5)   # [rt][kb][grp][row][ch][8]
        parts.append(torch.gather(v, 4, idx).reshape(rows // 128, nkb, 4096))
    return torch.stack(parts, 2).reshape(-1).contiguous()                          # [rt][kb][piece][4096]


def untile_a_operand(t: Tensor, rows: int, cols: int, scale: tp.Optional[float] = None,
                     variant: tp.Optional[str] = None) -> Tensor:
    """Inverse of ``tile_a_operand`` (returns (p1 + p2 (+ p3)) / scale as plain float32 ``[rows][cols]``)."""
    fmt = _lib.operand_format(variant)
    if scale is None:
        scale = fmt.value_scale
    nkb = cols // 32
    P = fmt.parts
    dt = torch.float16 if P == 2 else torch.bfloat16
    v = t.view(dt).view(rows // 128, nkb, P, 16, 8, 4, 8)                        # [rt][kb][piece][grp][row][pos][8]
    idx = _swizzle_index(t.device).view(1, 1, 1, 1, 8, 4, 1).expand(rows // 128, nkb, P, 16, 8, 4, 8)
    w = torch.gather(v.to(torch.float32), 5, idx).flip(2).sum(2) / scale           # [rt][kb][grp][row][ch][8]
    return w.permute(0, 2, 3, 1, 4, 5).reshape(rows, cols).contiguous()


def operand_buffer(rows: int, cols: int, device, variant: tp.Optional[str] = None) -> Tensor:
    """Zeroed storage of a tiled operand matrix with ``rows x cols`` values."""
    fmt = _lib.operand_format(variant)
    return torch.zeros(rows, fmt.parts * cols, dtype=torch.float16 if fmt.parts == 2 else torch.bfloat16,
                       device=device)


class PackedNetworks:
    """Device-resident, kernel-layout copy of an ensemble of per-element MLPs (``dims`` keeps the
    true layer widths, the kernel model the widths padded to multiples of 32).

    ``weights[member][species_index] = [(W [out,in], b [out]) x 4]`` in ``torch.nn.Linear``
    layout (nn/_core.py:117-149).  All members must share the layer widths of a species.
    """

    def __init__(self, weights: tp.Sequence[tp.Sequence[tp.Sequence[tp.Tuple[Tensor, Tensor]]]],
                 in_dim: int, device: torch.device, celu_alpha: float = 0.1, variant: tp.Optional[str] = None,
                 radial_len: int = 0):
        """``radial_len`` (number of radial AEV columns, S * len(ShfR)) > 0 and not a multiple of 32: the angular block
        of the layer-1 operands starts at the next 32-column boundary (``col_pad`` zero columns in between) if that
        still fits the padded width -- every element pair then fills exactly one 32-column GEMM block, and the
        block-sparse layer 1 skips more (water: 5 live blocks instead of 8).  The AEV kernels write / read the same
        internal order (``ani_aev_params::ang_pad``); plain AEV rows keep the reference's order."""
        self.device = torch.device(device)
        self.variant = variant or ""   # build of the library (operand format) these operands are packed for
        M = len(weights)
        S = len(weights[0])
        if not (1 <= M <= _lib.ANI_MAX_MEMBERS) or not (1 <= S <= _lib.ANI_MAX_SPECIES):
            raise ValueError("unsupported number of ensemble members / species")
        self.num_members, self.num_species, self.in_dim = M, S, in_dim
        self.ldx = (in_dim + 31) // 32 * 32
        self.radial_len = int(radial_len)
        self.col_pad = (-self.radial_len) % 32 if 0 < self.radial_len < in_dim else 0
        if in_dim + self.col_pad > self.ldx or os.environ.get("ANI_B200_ALIGN_ANGULAR", "1") == "0":
            self.col_pad = 0
        self.celu_alpha = celu_alpha
        self.dims: tp.List[tp.Tuple[int, int, int]] = []
        self._keep: tp.List[Tensor] = []
        self.model = MLPModel()
        mdl = self.model
        mdl.num_species, mdl.num_members, mdl.in_dim, mdl.ldx = S, M, in_dim, self.ldx
        mdl.celu_alpha = celu_alpha
        # Weights are gathered on the HOST into one flat float32 buffer (zero-padded to 32-column blocks),
        # uploaded with a single copy and re-laid out into the tiled B operands by this library's own
        # ani_b200_pack_b_operand kernel: no ATen kernel touches them (one launch per operand kind).
        pad = lambda v: (v + 31) // 32 * 32  # noqa: E731
        P2 = 2 * _lib.operand_format(self.variant).parts          # bytes per operand element
        plan = []                                     # per species: sizes, scales, source / destination offsets
        src_off = 0
        dst_off = 0

        def take_src(count: int) -> int:
            nonlocal src_off
            o = src_off
            src_off += (count + 63) // 64 * 64         # 256-byte aligned float32 blocks
            return o

        def take_dst(nbytes: int) -> int:
            nonlocal dst_off
            o = dst_off
            dst_off += (nbytes + 1023) // 1024 * 1024
            return o

        host_w = []
        for s in range(S):
            layers0 = weights[0][s]
            if len(layers0) != 4:
                raise ValueError("the B200 MLP kernels support exactly 3 hidden layers + 1 output")
            h1, h2, h3 = (int(layers0[k][0].shape[0]) for k in range(3))
            if int(layers0[3][0].shape[0]) != 1:
                raise ValueError("out_dim != 1 is not supported")
            if layers0[0][0].shape[1] != in_dim:
                raise ValueError("first layer width does not match the AEV length")
            self.dims.append((h1, h2, h3))
            W = [[weights[m][s][k][0].detach().to("cpu", torch.float32) for m in range(M)] for k in range(4)]
            Bv = [[weights[m][s][k][1].detach().to("cpu", torch.float32) for m in range(M)] for k in range(4)]
            for m in range(M):
                if tuple(W[0][m].shape) != (h1, in_dim) or tuple(W[1][m].shape) != (h2, h1) \
                        or tuple(W[2][m].shape) != (h3, h2) or tuple(W[3][m].shape) != (1, h3):
                    raise ValueError("all ensemble members must share the layer widths of an element")
            host_w.append((W, Bv))
            p1, p2, p3 = pad(h1), pad(h2), pad(h3)
            sc = [weight_scale(W[k], self.variant) for k in range(3)]   # one scale per layer, shared by W and W^T
            plan.append(dict(
                h=(h1, h2, h3), p=(p1, p2, p3), sc=sc,
                s_w1=take_src(M * p1 * self.ldx), s_w2=take_src(M * p2 * p1), s_w3=take_src(M * p3 * p2),
                s_b1=take_src(M * p1), s_b2=take_src(M * p2), s_b3=take_src(M * p3), s_w4=take_src(M * p3),
                s_b4=take_src(M),
                d_f1=take_dst(M * p1 * self.ldx * P2), d_f2=take_dst(M * p2 * p1 * P2), d_f3=take_dst(M * p3 * p2 * P2),
                d_b3=take_dst(M * p2 * p3 * P2), d_b2=take_dst(M * p1 * p2 * P2), d_b1=take_dst(self.ldx * M * p1 * P2)))
        host = torch.zeros(src_off, dtype=torch.float32)   # zero weights and biases in the padding:
        for s in range(S):                                   # CELU(0) = 0 meets zero weights: results unchanged
            (W, Bv), q = host_w[s], plan[s]
            (h1, h2, h3), (p1, p2, p3) = q["h"], q["p"]
            w1 = host[q["s_w1"]:q["s_w1"] + M * p1 * self.ldx].view(M, p1, self.ldx)
            w2 = host[q["s_w2"]:q["s_w2"] + M * p2 * p1].view(M, p2, p1)
            w3 = host[q["s_w3"]:q["s_w3"] + M * p3 * p2].view(M, p3, p2)
            b1 = host[q["s_b1"]:q["s_b1"] + M * p1].view(M, p1)
            b2 = host[q["s_b2"]:q["s_b2"] + M * p2].view(M, p2)
            b3 = host[q["s_b3"]:q["s_b3"] + M * p3].view(M, p3)
            w4 = host[q["s_w4"]:q["s_w4"] + M * p3].view(M, p3)
            b4 = host[q["s_b4"]:q["s_b4"] + M]
            for m in range(M):
                if self.col_pad:   # internal column order: radial | col_pad zeros | angular
                    RLc = self.radial_len
                    w1[m, :h1, :RLc] = W[0][m][:, :RLc]
                    w1[m, :h1, RLc + self.col_pad:in_dim + self.col_pad] = W[0][m][:, RLc:]
                else:
                    w1[m, :h1, :in_dim] = W[0][m]
                w2[m, :h2, :h1] = W[1][m]
                w3[m, :h3, :h2] = W[2][m]
                b1[m, :h1], b2[m, :h2], b3[m, :h3] = Bv[0][m], Bv[1][m], Bv[2][m]
                w4[m, :h3] = W[3][m].view(-1)
                b4[m] = Bv[3][m].view(())
        with torch.cuda.device(self.device):
            src = host.pin_memory().to(self.device, non_blocking=True)
            dst = torch.empty(dst_off, dtype=torch.uint8, device=self.device)
            st = torch.cuda.current_stream(self.device).cuda_stream
            L = _lib.lib(self.variant)
            sp0, dp0 = src.data_ptr(), dst.data_ptr()
            for s in range(S):
                q = plan[s]
                (p1, p2, p3), sc = q["p"], q["sc"]
                ldx_ = self.ldx
                jobs = [   # (src, n, k, ld_src, transpose, scale, batch, src stride, dst, dst stride in bytes)
                    (q["s_w1"], p1, ldx_, ldx_, 0, sc[0], M, p1 * ldx_, q["d_f1"], p1 * ldx_ * P2),      # per member [h1][ldx]
                    (q["s_w2"], p2, p1, p1, 0, sc[1], M, p2 * p1, q["d_f2"], p2 * p1 * P2),              # per member [h2][h1]
                    (q["s_w3"], p3, p2, p2, 0, sc[2], M, p3 * p2, q["d_f3"], p3 * p2 * P2),              # per member [h3][h2]
                    (q["s_w3"], p2, p3, p2, 1, sc[2], M, p3 * p2, q["d_b3"], p2 * p3 * P2),              # W3^T [h2][h3]
                    (q["s_w2"], p1, p2, p1, 1, sc[1], M, p2 * p1, q["d_b2"], p1 * p2 * P2),              # W2^T [h1][h2]
                    (q["s_w1"], ldx_, M * p1, ldx_, 1, sc[0], 1, 0, q["d_b1"], 0),                       # W1^T [ldx][M*h1]
                ]
                for (so, n_, k_, ld_, tr, scale, batch, sstr, do, dstr) in jobs:
                    check(L.ani_b200_pack_b_operand(sp0 + 4 * so, n_, k_, ld_, tr, scale, batch, sstr, dp0 + do, dstr, st),
                          "pack_b_operand")
                spm = mdl.sp[s]
                spm.h1, spm.h2, spm.h3 = p1, p2, p3
                for k in range(3):
                    spm.w_scale[k] = sc[k]
                spm.w_scale[3] = 1.0
                for name, off in (("b1", q["s_b1"]), ("b2", q["s_b2"]), ("b3", q["s_b3"]), ("w4", q["s_w4"]),
                                  ("b4", q["s_b4"])):
                    setattr(spm, name, sp0 + 4 * off)
                for name, off in (("t_f1", q["d_f1"]), ("t_f2", q["d_f2"]), ("t_f3", q["d_f3"]), ("t_b3", q["d_b3"]),
                                  ("t_b2", q["d_b2"]), ("t_b1", q["d_b1"])):
                    setattr(spm, name, dp0 + off)
        # scratch of the per-step compaction of the layer-1 backward operands (live AEV column blocks only; as large
        # as those operands together; ani_mlp_model::b1_compact)
        b1c = torch.empty(sum(self.ldx * (M * q["p"][0] // 32) * 32 * P2 for q in plan), dtype=torch.uint8,
                          device=self.device)
        mdl.b1_compact = b1c.data_ptr()
        self._keep = [src, dst, b1c]
        self._plan = plan
        mdl.h1_max = max(q["p"][0] for q in plan)
        mdl.h2_max = max(q["p"][1] for q in plan)
        mdl.h3_max = max(q["p"][2] for q in plan)
        self.set_active_members(list(range(M)))

    def set_active_members(self, idxs: tp.Sequence[int]) -> None:
        """nn/_core.py:99-110: the ensemble output is the mean over the active members."""
        for i in idxs:
            if not 0 <= i < self.num_members:
                raise IndexError(f"Idx {i} should be 0 <= idx < {self.num_members}")
        self.active = list(idxs)
        # captured CUDA graphs bake the member scales in: they are keyed by this tuple (Engine.run)
        self.active_key = tuple(self.active)
        for m in range(_lib.ANI_MAX_MEMBERS):
            self.model.member_scale[m] = (1.0 / len(self.active)) if m in self.active else 0.0

    @property
    def ld(self) -> tp.Tuple[int, int, int]:
        M = self.num_members
        return M * self.model.h1_max, M * self.model.h2_max, M * self.model.h3_max

    def flops_per_atom(self, species_index: int, backward: bool = True) -> float:
        h1, h2, h3 = self.dims[species_index]
        macs = self.in_dim * h1 + h1 * h2 + h2 * h3 + h3
        return 2.0 * macs * self.num_members * (2 if backward else 1)


class Workspace:
    """All device buffers for one (n_conf, n_per_conf) problem shape."""

    def __init__(self, n_conf: int, n_per_conf: int, num_species: int, ldx: int, ld: tp.Tuple[int, int, int],
                 num_members: int, nbr_cap: int, device: torch.device, owned_cap: tp.Optional[int] = None,
                 variant: tp.Optional[str] = None):
        n = n_conf * n_per_conf
        self.n, self.n_conf, self.n_per_conf = n, n_conf, n_per_conf
        owned = n if owned_cap is None else min(n, owned_cap)
        self.rows_cap = (owned + num_species * (TILE - 1) + TILE - 1) // TILE * TILE
        self.max_bins = max(64, n + 2) if n_conf == 1 else n_conf + 2
        i32 = dict(dtype=torch.int32, device=device)
        f32 = dict(dtype=torch.float32, device=device)
        self.grid = torch.zeros(C.sizeof(Grid) // 4, **i32)
        # What a host-driven loop moves per step lives in TWO contiguous blocks, so that calculator.HostCalculator needs one
        # H2D and one D2H copy (each copy is a node of the captured graph with its own DMA set-up latency):
        #   in_block  f32: [cell 9 | pad to 16 | coords 3 n]
        #   out_block u8 : [energies f64 x n_conf | status i32 | pad to 16 B | grad f32 x 3 n]
        self.in_block = torch.zeros(16 + 3 * n, **f32)
        self._out_grad_off = (8 * n_conf + 4 + 15) // 16 * 16
        self.out_block = torch.zeros(self._out_grad_off + 12 * n, dtype=torch.uint8, device=device)
        self.status = self.out_block[8 * n_conf: 8 * n_conf + 4].view(torch.int32)
        self.bin_start = torch.zeros(self.max_bins + 2, **i32)
        self.sorted_orig = torch.zeros(n, **i32)
        self.orig_to_sorted = torch.zeros(n, **i32)
        self.spos = torch.zeros(n, 4, **f32)
        self.sbin = torch.zeros(n, **i32)
        self.scratch = torch.zeros(3 * n + self.max_bins + 2 + (n // 256 + 3) * 8 + 64, **i32)
        self.row_of = torch.zeros(n, **i32)
        self.row_atom = torch.zeros(self.rows_cap, **i32)
        self.tile_species = torch.zeros(self.rows_cap // TILE, **i32)
        self.layout_info = torch.zeros(16, **i32)
        self.aev_blocks = torch.zeros(ldx // 32 + 3, **i32)   # [count, ids..., element mask, changed flag]
        self.n_blocks = ldx // 32
        self.bucket_ranges = torch.zeros((self.max_bins - 1) * 27 * 8, **f32) if n_conf == 1 else None
        # per-bucket species offsets (ani_b200_prepare_step -> ani_b200_aev_forward): i32[max_bins][8].  Experiment
        # (ANI_B200_AEV_BSS=1): lets the AEV forward skip its candidate-counting pass; measured on B200 it is 2 us
        # SLOWER at 10 k atoms (64.2 vs 62.4 us) -- the table row is one more dependent global load at the head of
        # every CTA and the per-warp prefixes cost what the two saved barriers bought -- so it is off
        self.bucket_species = (torch.zeros(self.max_bins * 8, **i32)
                               if n_conf == 1 and os.environ.get("ANI_B200_AEV_BSS", "0") != "0" else None)
        self.nbr_cap = nbr_cap
        self.nbr_cnt = torch.zeros(n, **i32)
        self.nbr_list = torch.zeros(n * nbr_cap, **i32)
        # x / act*: "tiled operand" form (16-bit pieces of every value); dx: plain float32 rows
        self.x = operand_buffer(self.rows_cap, ldx, device, variant)
        self.dx = torch.zeros(self.rows_cap, ldx, **f32)
        self.act1 = operand_buffer(self.rows_cap, ld[0], device, variant)
        self.act2 = operand_buffer(self.rows_cap, ld[1], device, variant)
        self.act3 = operand_buffer(self.rows_cap, ld[2], device, variant)
        self.e_member = torch.zeros(num_members, self.rows_cap, **f32)
        self.mlp_sync = torch.zeros(6 * (self.rows_cap // TILE) + 8, **i32)   # data-flow counters of ani_b200_mlp_step
        self.species_i32 = torch.zeros(n, **i32)
        self.coords = self.in_block[16:].view(n, 3)
        self.cell = self.in_block[:9]
        self.grad = self.out_block[self._out_grad_off:].view(torch.float32).view(n, 3)
        self.atomic = torch.zeros(n, **f32)
        self.member_atomic = torch.zeros(num_members, n, **f32)
        self.energies = self.out_block[:8 * n_conf].view(torch.float64)
        # where the step's kernels ACCUMULATE forces / conformer energies: these buffers, or -- multi-GPU,
        # parallel.ShardedEngine.attach -- partial-sum buffers in peer-mapped memory whose reduction over the
        # ranks (reducer.launch, the last launch of the step) lands in `grad` / `energies`
        self.grad_ptr = self.grad.data_ptr()
        self.energies_ptr = self.energies.data_ptr()
        self.reducer: tp.Any = None
        # distinct elements seen at graph-capture time (0 = not known): sizes the shared-memory gradient
        # table of the AEV backward kernel; the results never depend on it (Engine.note_composition)
        self.max_elements = 0
        # Verlet-skin reuse of the bucket grid (Engine.skin > 0): binned positions, wrapping lattice
        # vectors and the "an atom left its skin/2 sphere" word (ani_b200_verlet_positions)
        self.ref_pos = torch.zeros(n, 4, **f32)
        self.ref_shift = torch.zeros(n, 4, **f32)
        self.moved = torch.zeros(1, **i32)
        # partial sums of the virial W_ab = sum_pairs (dE/dDelta)_a Delta_b (ani_b200_aev_backward)
        self.virial = torch.zeros(_lib.ANI_VIRIAL_SLOTS, 9, dtype=torch.float64, device=device)


class StepResult(tp.NamedTuple):
    energies: Tensor          # (C,) float64: NN energy + self energies of the owned atoms
    atomic_energies: Tensor   # (C, A) float32: NN atomic energies (ensemble mean), 0 for padding
    member_atomic: Tensor     # (M, C, A) float32 per-member NN atomic energies
    grad: tp.Optional[Tensor]  # (C, A, 3) float32 dE/dcoords (forces = -grad) or None
    virial: tp.Optional[Tensor] = None  # (3, 3) float64 sum_pairs (dE/dDelta)_a Delta_b (stress = virial / volume)


class Engine:
    """Fused ANI energy(+force) step on one GPU.  ``lo_frac/hi_frac`` select the slice of
    bucket-sorted atoms this engine owns (multi-GPU sharding, see parallel.py)."""

    def __init__(self, consts: AEVConstants, nets: PackedNetworks, sae: tp.Optional[tp.Sequence[float]] = None,
                 nbr_cap: int = 128, cuda_graph: bool = True):
        if nets.in_dim != consts.out_dim:
            raise ValueError("network input width != AEV length")
        if nets.num_species != consts.num_species:
            raise ValueError("network / AEV species mismatch")
        self.consts, self.nets = consts, nets
        self.device = nets.device
        self.params = consts.to_struct()
        # internal column order of the tiled AEV operand / dE/dAEV rows: must be the one the layer-1 weights were packed in
        if nets.col_pad and nets.radial_len != consts.num_species * len(consts.shf_r):
            raise ValueError("the networks were packed for another radial AEV length")
        self.params.ang_pad = nets.col_pad
        self.nbr_cap = nbr_cap
        # > 0: buckets are built for cutoff + skin, so that a grid can be reused while no atom has moved
        # more than skin/2 (run(..., reuse=True); calculator.HostCalculator drives it)
        self.skin = 0.0
        self.sae = None
        if sae is not None:
            self.sae = torch.tensor(list(sae), dtype=torch.float64, device=self.device)
        self._ws: tp.Dict[tp.Tuple[int, int], Workspace] = {}
        self.cuda_graph = cuda_graph
        self.graph_after = 3   # eager launches of a problem shape before its CUDA graph is captured
        self._graphs: tp.Dict[tp.Any, torch.cuda.CUDAGraph] = {}   # insertion order = LRU order
        self.max_graphs = 16
        self._graph_seen: tp.Dict[tp.Any, int] = {}
        self.variant = nets.variant
        self.lib = _lib.lib(self.variant)
        self.launches_per_step = 0
        # per-stage CUDA-event timing (bench.py's roofline leg); off by default
        self.profile = False
        # zero-fill of dE/dAEV and the energy reduction on a forked side stream (see _launch).  Off by
        # default: measured on B200 at 10k atoms it changes the step by < 1 us (0.3899 vs 0.3905 ms) --
        # inside the graph the two kernels cost little more than their dependency edges
        self.side_stream = os.environ.get("ANI_B200_SIDE_STREAM", "0") != "0"
        self.overlap_reduce = os.environ.get("ANI_B200_OVERLAP_REDUCE", "1") != "0"
        # The MLP of a step: ONE persistent data-flow launch (csrc/gemm_fused.cuh) or the six chained launches of
        # csrc/gemm_tc.cuh -- the same tile code either way.  Measured on B200 over 2 k - 50 k atoms
        # (profiles/r02_sweep.md): the two are equal except where the chained launches quantise badly -- every one of
        # the six launches runs (row tiles x members) units on 148 persistent CTAs, e.g. 4.2 units per CTA at 10 k
        # atoms = 84 % balance, six times -- which the single list of the data-flow launch avoids (10 k atoms: 0.219 vs
        # 0.235 ms); for short lists (< 3 waves) the chained launches win, a launch boundary being a cheaper hand-over
        # of a row tile than an L2 counter when the six-layer chain is exposed.  "auto" applies exactly that rule;
        # ANI_B200_MLP_FUSED=0 / 1 forces one of them.
        # A third schedule runs inside ani_b200_mlp_step wherever it fits (mlp_schedule): resident chains
        # (csrc/gemm_resident.cuh), each (row tile, member) chain on one SM with its activations and gradients in
        # shared memory, up to 8 chains per SM.  Measured on B200 (1000 W, profiles/r03_bench_*), step against the
        # previous choice: water 999 atoms 0.115 vs 0.138 ms, gdb256 0.230 vs 0.252 ms, water 9 999 atoms 0.323 vs
        # 0.346 ms; the protein-in-water box of 50 k atoms (21 chains per SM) keeps the data-flow launch.
        self.mlp_mode = os.environ.get("ANI_B200_MLP_FUSED", "auto")
        self._num_sms = torch.cuda.get_device_properties(self.device).multi_processor_count
        self._side_stream: tp.Optional[torch.cuda.Stream] = None
        self._ev: tp.List[torch.cuda.Event] = []
        self.stage_events: tp.Dict[str, tp.List[tp.Tuple[torch.cuda.Event, torch.cuda.Event]]] = {}

    def _timed(self, name: str, fn: tp.Callable[[], int]) -> None:
        """Run one C-ABI stage; with ``profile`` on, bracket it with events on the launch stream."""
        if not self.profile:
            check(fn(), name)
            return
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        check(fn(), name)
        b.record()
        self.stage_events.setdefault(name, []).append((a, b))

    def stage_times_ms(self) -> tp.Dict[str, float]:
        """Mean device time per call of every stage (synchronises)."""
        torch.cuda.synchronize(self.device)
        return {k: sum(a.elapsed_time(b) for a, b in v) / len(v) for k, v in self.stage_events.items() if v}

    # -- workspaces ------------------------------------------------------------------------
    def workspace(self, n_conf: int, n_per_conf: int) -> Workspace:
        key = (n_conf, n_per_conf)
        ws = self._ws.get(key)
        if ws is None:
            ws = Workspace(n_conf, n_per_conf, self.consts.num_species, self.nets.ldx, self.nets.ld,
                           self.nets.num_members, self.nbr_cap, self.device, variant=self.variant)
            self._ws[key] = ws
        return ws

    # -- one step --------------------------------------------------------------------------
    def step(self, species: Tensor, coords: Tensor, cell: tp.Optional[Tensor] = None, pbc: bool = False,
             want_grad: bool = True, shard: tp.Tuple[int, int] = (0, 1), want_virial: bool = False,
             check: bool = False) -> StepResult:
        """species (C, A) int (element indices, -1 padding), coords (C, A, 3) on this device.
        ``shard = (rank, world)``: only atoms whose bucket-sorted position falls into this
        rank's slice are evaluated; gradients/energies are partial sums to be all-reduced.

        The launch sequence of a given problem shape is captured into a CUDA graph on its fourth
        use and replayed afterwards (``cuda_graph=False`` at construction disables this)."""
        dev = self.device
        n_conf, n_per_conf = species.shape
        if coords.shape != (n_conf, n_per_conf, 3):
            raise ValueError("coords must have shape (C, A, 3)")
        if species.device != dev or coords.device != dev:
            raise ValueError(f"inputs must live on {dev} (the B200 engine has no CPU path)")
        if pbc and cell is None:
            raise ValueError("If pbc is not None, cell should be present")
        if pbc and n_conf != 1:
            raise NotImplementedError("periodic batches (C > 1 with one shared cell) are not supported yet")
        ws = self.workspace(n_conf, n_per_conf)
        # inputs -> persistent buffers (what the graph reads)
        ws.species_i32.copy_(species.reshape(-1))
        ws.coords.copy_(coords.reshape(-1, 3))
        if pbc:
            ws.cell.copy_(cell.reshape(-1))
        res = self.run(ws, bool(pbc), want_grad, shard, want_virial=want_virial)
        if check:   # one 4-byte D2H read: cell too small / neighbour overflow / operand range raise here
            self.check_status(ws)
        return res

    def run(self, ws: Workspace, pbc: bool, want_grad: bool = True, shard: tp.Tuple[int, int] = (0, 1),
            reuse: bool = False, want_virial: bool = False) -> StepResult:
        """One step on inputs that are ALREADY in the workspace buffers (``ws.species_i32``,
        ``ws.coords``, ``ws.cell``) -- the entry point of host-driven loops that copy straight into
        them (calculator.HostCalculator).  The results alias workspace buffers."""
        n, n_conf, n_per_conf = ws.n, ws.n_conf, ws.n_per_conf
        rank, world = shard
        lo = (n * rank) // world
        hi = (n * (rank + 1)) // world
        if want_virial and (not want_grad or reuse or n_conf != 1):
            raise ValueError("the virial comes out of the force pass of a single system with a freshly built grid")
        key = (n_conf, n_per_conf, bool(pbc), bool(want_grad), lo, hi, self.nets.active_key, bool(reuse), self.skin,
               bool(want_virial), self.mlp_mode)
        if reuse and not self.skin > 0:
            raise ValueError("reuse=True needs Engine.skin > 0 and a previous step that built the grid")
        with torch.cuda.device(self.device):   # the C-ABI launches on the CURRENT device's stream
            if not self.cuda_graph or self.profile:
                self._launch(ws, bool(pbc), want_grad, lo, hi, reuse, want_virial)
            else:
                graph = self._graphs.get(key)
                if graph is not None:
                    self._graphs[key] = self._graphs.pop(key)   # most recently used last
                    graph.replay()
                elif self._graph_seen.get(key, 0) < self.graph_after:
                    # the first few uses of a shape run eagerly (one-off shapes never pay for a capture)
                    if len(self._graph_seen) > 4 * self.max_graphs:
                        self._graph_seen.clear()
                    self._graph_seen[key] = self._graph_seen.get(key, 0) + 1
                    self._launch(ws, bool(pbc), want_grad, lo, hi, reuse, want_virial)
                else:
                    self.note_composition(ws)
                    graph = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(graph):
                        self._launch(ws, bool(pbc), want_grad, lo, hi, reuse, want_virial)
                    while len(self._graphs) >= self.max_graphs:   # evict the least recently used capture
                        self._graphs.pop(next(iter(self._graphs)))
                    self._graphs[key] = graph
                    graph.replay()
        # kernels launched by this library in one step (memsets excluded):
        # prepare 1 (+1 grid kernel for open single systems), AEV fwd 1, GEMM fwd 3,
        # (zero + GEMM bwd 3 + AEV bwd 1), reduce 1
        mlp = ((self.lib.ani_b200_mlp_step_windows(C.byref(self.nets.model), ws.rows_cap) + (1 if want_grad else 0))
               if self._use_dataflow_mlp(hi - lo, ws.rows_cap) else (3 + (4 if want_grad else 0)))
        self.launches_per_step = 1 + (0 if (pbc or n_conf > 1) else 1) + 1 + mlp + (1 if want_grad else 0) + 1
        grad = ws.grad.view(n_conf, n_per_conf, 3) if want_grad else None
        virial = ws.virial.sum(0).view(3, 3) if want_virial else None
        return StepResult(ws.energies, ws.atomic.view(n_conf, n_per_conf),
                          ws.member_atomic.view(-1, n_conf, n_per_conf), grad, virial)

    def _launch(self, ws: Workspace, pbc: bool, want_grad: bool, lo: int, hi: int, reuse: bool = False,
                want_virial: bool = False) -> None:
        """Enqueue the kernels of one step on the current stream (graph-capturable: no allocation,
        no synchronisation, only this library's launches and two memsets)."""
        L = self.lib
        n, n_conf, n_per_conf = ws.n, ws.n_conf, ws.n_per_conf
        st = torch.cuda.current_stream(self.device).cuda_stream
        cell_ptr = ptr(ws.cell) if pbc else None
        mode = 0 if n_conf == 1 else 1
        c = self.consts
        # bucket grid + species-grouped row layout + live AEV column blocks (+ zero-fill of the force
        # accumulator): one fused entry point, five launches -- or, with a Verlet skin and reuse=True,
        # one launch that only refreshes the positions inside the grid of an earlier step
        if reuse:
            self._timed("prepare_step", lambda: L.ani_b200_verlet_positions(
                1, ptr(ws.coords), ptr(ws.grid), ptr(ws.sorted_orig), n, self.skin, ptr(ws.spos), ptr(ws.ref_pos),
                ptr(ws.ref_shift), ptr(ws.moved), ws.grad_ptr if want_grad else None, 3 * n if want_grad else 0,
                ptr(ws.aev_blocks), self.nets.ldx, st))
        else:
            self._timed("prepare_step", lambda: L.ani_b200_prepare_step(
                ptr(ws.coords), ptr(ws.species_i32), n_conf, n_per_conf, cell_ptr, int(bool(pbc)), mode,
                c.rcr + self.skin, ws.max_bins, ptr(ws.grid), ptr(ws.bin_start), ptr(ws.sorted_orig),
                ptr(ws.orig_to_sorted), ptr(ws.spos), ptr(ws.sbin), ptr(ws.bucket_ranges),
                lo, hi, c.num_species, ws.rows_cap, ptr(ws.row_of), ptr(ws.row_atom), ptr(ws.tile_species),
                ptr(ws.layout_info), len(c.shf_r), len(c.shf_a) * len(c.shf_z), c.out_dim, self.nets.ldx,
                self.nets.col_pad, ptr(ws.aev_blocks), ws.grad_ptr if want_grad else None, 3 * n if want_grad else 0,
                ptr(ws.virial) if want_virial else None, ws.virial.numel() if want_virial else 0,
                ptr(ws.bucket_species), ptr(ws.scratch), ptr(ws.status), st))
            if self.skin > 0:
                check(L.ani_b200_verlet_positions(
                    0, ptr(ws.coords), ptr(ws.grid), ptr(ws.sorted_orig), n, self.skin, ptr(ws.spos),
                    ptr(ws.ref_pos), ptr(ws.ref_shift), ptr(ws.moved), None, 0, None, self.nets.ldx, st),
                    "verlet_positions")
        # Two small kernels leave the critical path on a side stream (forked and joined with events, so
        # the whole thing still captures into one CUDA graph): the zero-fill of dE/dAEV runs beside the
        # AEV forward / forward GEMMs, the energy reduction beside the backward GEMMs / AEV backward.
        main = torch.cuda.current_stream(self.device)
        side = main if (self.profile or not self.side_stream) else self._side()
        split = side is not main
        zero_first = want_grad and self.nets.num_members > 1
        if split and zero_first:
            self._ev[0].record(main)
            side.wait_event(self._ev[0])
            check(L.ani_b200_zero_live_blocks(C.byref(self.nets.model), ptr(ws.dx), ptr(ws.layout_info),
                                              ptr(ws.aev_blocks), side.cuda_stream), "zero_live_blocks")
            self._ev[1].record(side)
        self._timed("aev_forward", lambda: L.ani_b200_aev_forward(
            C.byref(self.params), ptr(ws.grid), ptr(ws.bin_start), ptr(ws.spos), ptr(ws.sbin),
            ptr(ws.bucket_ranges), ptr(ws.bucket_species) if not reuse else None,
            ws.aev_blocks.data_ptr() + 4 * (ws.n_blocks + 1), n, lo, hi,
            ptr(ws.row_of), ptr(ws.x), self.nets.ldx, 1, ptr(ws.nbr_cnt), ptr(ws.nbr_list), ws.nbr_cap,
            ptr(ws.status), st))

        def reduce_on(stream_handle):
            return L.ani_b200_reduce_energies(
                C.byref(self.nets.model), ptr(ws.e_member), ws.rows_cap, ptr(ws.row_of), ptr(ws.orig_to_sorted),
                ptr(ws.species_i32), n, lo, hi, n_conf, n_per_conf, ptr(self.sae), ptr(ws.atomic),
                ptr(ws.member_atomic), ws.energies_ptr, stream_handle)

        self.mlp_fused = self._use_dataflow_mlp(hi - lo, ws.rows_cap)
        if not split and self.mlp_fused:
            # the six GEMMs of the step as ONE persistent data-flow launch (csrc/gemm_fused.cuh)
            self._timed("mlp_forward_backward", lambda: L.ani_b200_mlp_step(
                C.byref(self.nets.model), ptr(ws.x), ptr(ws.dx), ws.rows_cap, ptr(ws.row_atom),
                ptr(ws.layout_info), ptr(ws.aev_blocks), ptr(ws.act1), ptr(ws.act2), ptr(ws.act3), ptr(ws.e_member),
                int(want_grad), ptr(ws.mlp_sync), ptr(ws.status), st))
        elif not split:
            self._timed("mlp_forward_backward", lambda: L.ani_b200_mlp_forward_backward(
                C.byref(self.nets.model), ptr(ws.x), ptr(ws.dx), ws.rows_cap, ptr(ws.row_atom),
                ptr(ws.layout_info), ptr(ws.aev_blocks), ptr(ws.act1), ptr(ws.act2), ptr(ws.act3), ptr(ws.e_member),
                int(want_grad), ptr(ws.status), st))
        else:
            check(L.ani_b200_mlp_forward(
                C.byref(self.nets.model), ptr(ws.x), ws.rows_cap, ptr(ws.row_atom), ptr(ws.layout_info),
                ptr(ws.aev_blocks), ptr(ws.act1), ptr(ws.act2), ptr(ws.act3), ptr(ws.e_member), int(want_grad),
                ptr(ws.status), st), "mlp_forward")
            self._ev[2].record(main)
            side.wait_event(self._ev[2])
            check(reduce_on(side.cuda_stream), "reduce_energies")
            self._ev[3].record(side)
            if want_grad:
                if zero_first:
                    main.wait_event(self._ev[1])
                check(L.ani_b200_mlp_backward(
                    C.byref(self.nets.model), ptr(ws.dx), ws.rows_cap, ptr(ws.row_atom), ptr(ws.layout_info),
                    ptr(ws.aev_blocks), ptr(ws.act1), ptr(ws.act2), ptr(ws.act3), int(zero_first), ptr(ws.status), st),
                    "mlp_backward")
        # the energy reduction only needs the MLP's forward outputs: beside the AEV backward (a forked branch of the
        # captured graph), not after it
        overlap = want_grad and not split and self.overlap_reduce and not self.profile
        if overlap:
            side2 = self._side()
            self._ev[2].record(main)
            side2.wait_event(self._ev[2])
            check(reduce_on(side2.cuda_stream), "reduce_energies")
            self._ev[3].record(side2)
        if want_grad:
            self._timed("aev_backward", lambda: L.ani_b200_aev_backward(
                C.byref(self.params), ptr(ws.grid), ptr(ws.spos), ptr(ws.sorted_orig),
                ws.aev_blocks.data_ptr() + 4 * (ws.n_blocks + 1), n, lo, hi,
                ptr(ws.row_of), ptr(ws.dx), self.nets.ldx, ptr(ws.nbr_cnt), ptr(ws.nbr_list), ws.nbr_cap,
                ws.grad_ptr, ptr(ws.status), ws.max_elements, ptr(ws.virial) if want_virial else None, st))
        if overlap or split:
            main.wait_event(self._ev[3])
        else:
            self._timed("reduce_energies", lambda: reduce_on(st))
        if ws.reducer is not None:
            # multi-GPU: sum the partial forces / energies of all ranks over NVLink peer memory (one launch,
            # part of the captured graph); without forces only the energies matter but the buffer is small
            def reduce_all() -> int:
                ws.reducer.launch(ws.grad, ws.energies)
                return 0
            self._timed("allreduce", reduce_all)

    def step_members(self, species: Tensor, coords: Tensor, cell: tp.Optional[Tensor] = None, pbc: bool = False
                     ) -> tp.Tuple[Tensor, Tensor]:
        """Energies (M_active, C) float64 and dE_m/dcoords (M_active, C, A, 3) float32 of every ACTIVE ensemble member
        in ONE pass (arch.py:403-436 differentiates every member by autograd; round 1 ran the engine once per member):
        one preparation, one AEV forward, one MLP launch whose layer-1 backward writes a per-member dE_m/dAEV slab
        (``ani_b200_mlp_step(want_backward=2)``), then the AEV backward once per member on its slab.  Eager (no
        graph): an analysis call, not the MD loop."""
        dev = self.device
        n_conf, n_per_conf = species.shape
        if pbc and n_conf != 1:
            raise NotImplementedError("periodic batches: call once per conformer")
        ws = self.workspace(n_conf, n_per_conf)
        n, L, c = ws.n, self.lib, self.consts
        nets = self.nets
        M, ldx = nets.num_members, nets.ldx
        active = list(nets.active)
        if getattr(ws, "dx_members", None) is None:
            ws.dx_members = torch.zeros(M, ws.rows_cap, ldx, dtype=torch.float32, device=dev)
        model = _lib.MLPModel.from_buffer_copy(nets.model)     # every active member with weight 1 (not 1 / M)
        for m in range(_lib.ANI_MAX_MEMBERS):
            model.member_scale[m] = 1.0 if m in active else 0.0
        grads = torch.zeros(len(active), n, 3, dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            st = torch.cuda.current_stream(dev).cuda_stream
            ws.species_i32.copy_(species.reshape(-1))
            ws.coords.copy_(coords.reshape(-1, 3))
            if pbc:
                ws.cell.copy_(cell.reshape(-1))
            check(L.ani_b200_prepare_step(
                ptr(ws.coords), ptr(ws.species_i32), n_conf, n_per_conf, ptr(ws.cell) if pbc else None, int(bool(pbc)),
                0 if n_conf == 1 else 1, c.rcr, ws.max_bins, ptr(ws.grid), ptr(ws.bin_start), ptr(ws.sorted_orig),
                ptr(ws.orig_to_sorted), ptr(ws.spos), ptr(ws.sbin), ptr(ws.bucket_ranges), 0, n, c.num_species,
                ws.rows_cap, ptr(ws.row_of), ptr(ws.row_atom), ptr(ws.tile_species), ptr(ws.layout_info),
                len(c.shf_r), len(c.shf_a) * len(c.shf_z), c.out_dim, ldx, self.nets.col_pad, ptr(ws.aev_blocks), None, 0,
                None, 0,
                ptr(ws.bucket_species), ptr(ws.scratch), ptr(ws.status), st), "prepare_step")
            mask_ptr = ws.aev_blocks.data_ptr() + 4 * (ws.n_blocks + 1)
            check(L.ani_b200_aev_forward(
                C.byref(self.params), ptr(ws.grid), ptr(ws.bin_start), ptr(ws.spos), ptr(ws.sbin),
                ptr(ws.bucket_ranges), ptr(ws.bucket_species), mask_ptr, n, 0, n, ptr(ws.row_of), ptr(ws.x), ldx, 1,
                ptr(ws.nbr_cnt),
                ptr(ws.nbr_list), ws.nbr_cap, ptr(ws.status), st), "aev_forward")
            check(L.ani_b200_mlp_step(
                C.byref(model), ptr(ws.x), ptr(ws.dx_members), ws.rows_cap, ptr(ws.row_atom), ptr(ws.layout_info),
                ptr(ws.aev_blocks), ptr(ws.act1), ptr(ws.act2), ptr(ws.act3), ptr(ws.e_member), 2, ptr(ws.mlp_sync),
                ptr(ws.status), st), "mlp_step")
            for k, m in enumerate(active):
                check(L.ani_b200_aev_backward(
                    C.byref(self.params), ptr(ws.grid), ptr(ws.spos), ptr(ws.sorted_orig), mask_ptr, n, 0, n,
                    ptr(ws.row_of), ws.dx_members[m].data_ptr(), ldx, ptr(ws.nbr_cnt), ptr(ws.nbr_list), ws.nbr_cap,
                    grads[k].data_ptr(), ptr(ws.status), 0, None, st), "aev_backward")
            check(L.ani_b200_reduce_energies(
                C.byref(model), ptr(ws.e_member), ws.rows_cap, ptr(ws.row_of), ptr(ws.orig_to_sorted),
                ptr(ws.species_i32), n, 0, n, n_conf, n_per_conf, None, ptr(ws.atomic), ptr(ws.member_atomic),
                ptr(ws.energies), st), "reduce_energies")
        e_m = ws.member_atomic.view(M, n_conf, n_per_conf)[active].double().sum(-1)          # (M_active, C)
        if self.sae is not None:
            sp = species.clamp(min=0)
            e_m = e_m + self.sae[sp].masked_fill(species < 0, 0.0).sum(-1).unsqueeze(0)
        return e_m, grads.view(len(active), n_conf, n_per_conf, 3)

    def mlp_schedule(self, owned: int, rows_cap: int) -> str:
        """How the MLP of a step over `owned` atoms (workspace of `rows_cap` rows) runs: "resident" (one launch of
        csrc/gemm_resident.cuh), "dataflow" (one launch of csrc/gemm_fused.cuh; "chains" with ANI_B200_MLP_CHAIN=1) or
        "chained" (six launches); see __init__.  ani_b200_mlp_step picks its kernel itself (ani_b200_mlp_step_kernel)."""
        if self.mlp_mode == "0":
            return "chained"
        kernel = self.lib.ani_b200_mlp_step_kernel(C.byref(self.nets.model), rows_cap)
        step = {0: "dataflow", 1: "chains", 2: "resident"}[kernel]
        if self.mlp_mode == "1" or step == "resident":
            return step
        units = (-(-owned // TILE) + 1) * self.nets.num_members     # per layer: row tiles x members (>= 1 column tile)
        waves = units / self._num_sms
        return step if waves >= 3.0 and waves / math.ceil(waves) < 0.9 else "chained"

    def _use_dataflow_mlp(self, owned: int, rows_cap: int) -> bool:
        """One launch of ani_b200_mlp_step (True) or six chained launches (False) for `owned` atoms."""
        return self.mlp_schedule(owned, rows_cap) != "chained"

    def note_composition(self, ws: Workspace) -> None:
        """Before a graph capture (the shape has already run eagerly): read the element mask of the last
        step once and let the AEV backward size its shared-memory gradient table for that many elements
        (more elements at replay time still give the right answer, from global memory)."""
        mask = int(ws.aev_blocks[ws.n_blocks + 1].item())
        ws.max_elements = bin(mask).count("1")

    def _side(self) -> "torch.cuda.Stream":
        if self._side_stream is None:
            self._side_stream = torch.cuda.Stream(self.device)
            self._ev = [torch.cuda.Event() for _ in range(4)]
        return self._side_stream

    # -- status ----------------------------------------------------------------------------
    def check_status(self, ws: tp.Optional[Workspace] = None) -> None:
        """Raise for device-side conditions (one D2H read; call when results are consumed)."""
        for w in ([ws] if ws is not None else list(self._ws.values())):
            code = int(w.status.item())
            if code == 0:
                continue
            w.status.zero_()
            if code & _lib.STATUS_CELL_TOO_SMALL:
                raise RuntimeError("Cell is too small to perform pbc calculations")  # neighbors.py:402-403
            if code & _lib.STATUS_NBR_OVERFLOW:
                raise RuntimeError(f"an atom has more than nbr_cap={w.nbr_cap} neighbours within Rcr; "
                                   "construct the engine with a larger nbr_cap (<= 256)")
            if code & _lib.STATUS_ANG_OVERFLOW:
                raise RuntimeError(f"an atom has more than {_lib.ANI_MAX_ANG} neighbours within Rca")
            if code & _lib.STATUS_PAIR_OVERFLOW:
                raise RuntimeError("half neighbour list capacity exceeded")
            if code & _lib.STATUS_INTERNAL:
                raise RuntimeError("a device-side barrier of libani_b200 timed out (internal error)")
            if code & _lib.STATUS_OPERAND_RANGE:
                raise _lib.OperandRangeError(
                    "an AEV, activation or gradient left the range of the half-precision GEMM operand pieces "
                    "(inf/NaN input, or |value| >= 1023 / |gradient| >= 16); the 3 x bfloat16 build of the library "
                    "(variant 'bf16x3') has no such limit -- models.ANI switches to it automatically")

    def grid_info(self, ws: Workspace) -> Grid:
        g = Grid()
        raw = ws.grid.cpu().numpy().tobytes()
        C.memmove(C.byref(g), raw, C.sizeof(Grid))
        return g
