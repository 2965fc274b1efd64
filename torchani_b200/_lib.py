"""ctypes binding of ``libani_b200.so`` (the C-ABI declared in ``include/ani_b200.h``).

There is exactly one compute path: the CUDA library.  If it is missing or does not load the
import fails loudly -- there is no CPU or PyTorch fallback.
"""
from __future__ import annotations

import ctypes as C
import os
import typing as tp

HERE = os.path.dirname(os.path.abspath(__file__))
# ANI_B200_LIB selects another build of the same library (e.g. the 3 x bf16 operand variant)
LIB_PATH = os.environ.get("ANI_B200_LIB") or os.path.join(HERE, "libani_b200.so")

ANI_MAX_SPECIES = 8
ANI_MAX_SHFR = 32
ANI_MAX_SHFA = 8
ANI_MAX_SHFZ = 8
ANI_MAX_MEMBERS = 16
ANI_TILE_ROWS = 128
ANI_MAX_ANG = 96
ANI_VIRIAL_SLOTS = 64

STATUS_NBR_OVERFLOW = 1
STATUS_ANG_OVERFLOW = 2
STATUS_CELL_TOO_SMALL = 4
STATUS_PAIR_OVERFLOW = 8
STATUS_OPERAND_RANGE = 16
STATUS_INTERNAL = 32


class AEVParams(C.Structure):
    _fields_ = [
        ("rcr", C.c_float), ("rca", C.c_float),
        ("eta_r", C.c_float), ("eta_a", C.c_float), ("zeta", C.c_float),
        ("n_shf_r", C.c_int32), ("n_shf_a", C.c_int32), ("n_shf_z", C.c_int32),
        ("num_species", C.c_int32), ("cutoff_kind", C.c_int32),
        ("shf_r", C.c_float * ANI_MAX_SHFR), ("shf_a", C.c_float * ANI_MAX_SHFA),
        ("cos_z", C.c_float * ANI_MAX_SHFZ), ("sin_z", C.c_float * ANI_MAX_SHFZ),
        ("ang_pad", C.c_int32),
    ]


class Grid(C.Structure):
    _fields_ = [
        ("cell", C.c_float * 9), ("inv", C.c_float * 9), ("origin", C.c_float * 3),
        ("dims", C.c_int32 * 3), ("pbc", C.c_int32), ("nbins", C.c_int32), ("mode", C.c_int32),
        ("n_per_conf", C.c_int32), ("n_real", C.c_int32),
    ]


class MLPSpecies(C.Structure):
    _fields_ = [("h1", C.c_int32), ("h2", C.c_int32), ("h3", C.c_int32), ("pad_", C.c_int32),
                ("w_scale", C.c_float * 4)] + [
        (k, C.c_void_p) for k in ("b1", "b2", "b3", "w4", "b4", "t_f1", "t_f2", "t_f3", "t_b3", "t_b2", "t_b1")
    ]


class MLPModel(C.Structure):
    _fields_ = [
        ("num_species", C.c_int32), ("num_members", C.c_int32), ("in_dim", C.c_int32), ("ldx", C.c_int32),
        ("h1_max", C.c_int32), ("h2_max", C.c_int32), ("h3_max", C.c_int32), ("pad_", C.c_int32),
        ("celu_alpha", C.c_float), ("member_scale", C.c_float * ANI_MAX_MEMBERS),
        ("sp", MLPSpecies * ANI_MAX_SPECIES),
        ("b1_compact", C.c_void_p),
    ]


_P = C.c_void_p
_I = C.c_int
_F = C.c_float

_PROTOTYPES = {
    "ani_b200_abi_version": (C.c_int, []),
    "ani_b200_operand_format": (C.c_int, [_P, _P, _P]),
    "ani_b200_error_string": (C.c_char_p, [_I]),
    "ani_b200_last_cuda_error": (C.c_char_p, []),
    "ani_b200_build_cells": (C.c_int, [_P, _P, _I, _I, _P, _I, _I, _F, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "ani_b200_species_layout": (C.c_int, [_P, _P, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P]),
    "ani_b200_aev_forward": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _P, _P, _I, _I, _P, _P, _I, _P, _P]),
    "ani_b200_aev_backward": (C.c_int, [_P, _P, _P, _P, _P, _I, _I, _I, _P, _P, _I, _P, _P, _I, _P, _P, _I, _P, _P]),
    "ani_b200_pairs_to_rows": (C.c_int, [_P, _P, _P, C.c_int64, _I, _I, _P, _P, _P, _P, _P, _P]),
    "ani_b200_full_nbrlist_to_rows": (C.c_int, [_P, _I, _P, _P, _P, _I, _F, _I, _P, _P, _P, _P, _P, _P]),
    "ani_b200_aev_forward_rows": (C.c_int, [_P, _P, _P, _P, _P, _P, _I, _P, _P, _I, _I, _I, _P, _P]),
    "ani_b200_aev_backward_rows": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _I, _P, _P, _I, _I, _P, _P, _P]),
    "ani_b200_prepare_step": (C.c_int, [_P, _P, _I, _I, _P, _I, _I, C.c_float, _I, _P, _P, _P, _P, _P, _P, _P,
                                        _I, _I, _I, _I, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _I, _P, _I, _P, _P, _P, _P]),
    "ani_b200_verlet_positions": (C.c_int, [_I, _P, _P, _P, _I, _F, _P, _P, _P, _P, _P, _I, _P, _I, _P]),
    "ani_b200_debug_gemm_trace": (C.c_int, [_P, _I]),
    "ani_b200_half_neighbor_count": (C.c_int, [_P, _P, _P, _P, _P, _I, _F, _P, _P]),
    "ani_b200_half_neighbor_fill": (C.c_int, [_P, _P, _P, _P, _P, _I, _F, _P, C.c_int64, _P, _P, _P, _P, _P, _P]),
    "ani_b200_mlp_forward_backward": (C.c_int, [_P, _P, _P, _I, _P, _P, _P, _P, _P, _P, _P, _I, _P, _P]),
    "ani_b200_mlp_step_windows": (C.c_int, [_P, _I]),
    "ani_b200_mlp_step_kernel": (C.c_int, [_P, _I]),
    "ani_b200_mlp_resident_plan": (C.c_int, [_P, _P]),
    "ani_b200_mlp_step": (C.c_int, [_P, _P, _P, _I, _P, _P, _P, _P, _P, _P, _P, _I, _P, _P, _P]),
    "ani_b200_mlp_forward": (C.c_int, [_P, _P, _I, _P, _P, _P, _P, _P, _P, _P, _I, _P, _P]),
    "ani_b200_zero_live_blocks": (C.c_int, [_P, _P, _P, _P, _P]),
    "ani_b200_mlp_backward": (C.c_int, [_P, _P, _I, _P, _P, _P, _P, _P, _P, _I, _P, _P]),
    "ani_b200_pack_b_operand": (C.c_int, [_P, _I, _I, _I, _I, _F, _I, C.c_longlong, _P, C.c_longlong, _P]),
    "ani_b200_comm_create": (C.c_int, [_I, _I, C.c_longlong, C.c_longlong, _P]),
    "ani_b200_comm_handle": (C.c_int, [_P, _P]),
    "ani_b200_comm_connect": (C.c_int, [_P, _P]),
    "ani_b200_comm_buffers": (C.c_int, [_P, _P, _P, _P]),
    "ani_b200_comm_allreduce": (C.c_int, [_P, _P, _P, _P]),
    "ani_b200_comm_destroy": (C.c_int, [_P]),
    "ani_b200_active_aev_blocks": (C.c_int, [_P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P]),
    "ani_b200_reduce_energies": (C.c_int, [_P, _P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P]),
}

EXPORTED_SYMBOLS = tuple(_PROTOTYPES)


class ANIB200Error(RuntimeError):
    pass


VARIANTS = ("", "bf16x3")   # "" = the default build (2 x fp16 operand pieces), "bf16x3" = 3 x bfloat16 pieces


def variant_path(variant: str = "") -> str:
    """Path of a build variant of the library (build.py: same sources, other operand format)."""
    if not variant:
        return LIB_PATH
    return os.path.join(os.path.dirname(LIB_PATH), f"libani_b200_{variant}.so")


def available(variant: str = "") -> bool:
    return os.path.exists(variant_path(variant))


def _load(path: str) -> C.CDLL:
    if not os.path.exists(path):
        raise ImportError(
            f"{path} is missing: build it with `python -m torchani_b200.build` "
            "(nvcc, sm_100a).  torchani_b200 has no CPU / PyTorch fallback."
        )
    lib = C.CDLL(path)   # RTLD_LOCAL: the variants export the same C symbols side by side
    for name, (res, args) in _PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.ani_b200_abi_version() != 4:
        raise ImportError(f"{path}: ABI version mismatch")
    return lib


_libs: tp.Dict[str, C.CDLL] = {}


def lib(variant: tp.Optional[str] = None) -> C.CDLL:
    """The C-ABI library; ``variant`` selects another operand-format build of the same sources (both can be
    loaded at once -- the automatic fallback of models.ANI uses that)."""
    v = variant or ""
    if v not in _libs:
        _libs[v] = _load(variant_path(v))
    return _libs[v]


class OperandFormat(tp.NamedTuple):
    parts: int           # 16-bit pieces per value: 2 = IEEE half, 3 = bfloat16
    value_scale: float   # power-of-two scale of AEV / activation operands
    grad_scale: float    # power-of-two scale of gradient operands


_fmts: tp.Dict[str, OperandFormat] = {}


def operand_format(variant: tp.Optional[str] = None) -> OperandFormat:
    """The tiled-operand format a library build was compiled for (ani_b200_operand_format)."""
    v = variant or ""
    if v not in _fmts:
        parts, vs, gs = C.c_int32(0), C.c_float(0), C.c_float(0)
        check(lib(v).ani_b200_operand_format(C.byref(parts), C.byref(vs), C.byref(gs)), "operand_format")
        _fmts[v] = OperandFormat(int(parts.value), float(vs.value), float(gs.value))
    return _fmts[v]


class OperandRangeError(RuntimeError):
    """A value left the range of the half-precision GEMM operand pieces (ANI_STATUS_OPERAND_RANGE)."""


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        l = lib()
        msg = l.ani_b200_error_string(rc).decode()
        if rc == -3:
            msg += " -- " + l.ani_b200_last_cuda_error().decode()
        raise ANIB200Error(f"{what}: {msg}" if what else msg)


def ptr(t) -> int:
    """Raw device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()
