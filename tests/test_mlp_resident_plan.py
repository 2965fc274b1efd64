"""Host side of the resident-chain MLP kernel (csrc/gemm_resident.cuh): its shared-memory plan for the ANI-1x and ANI-2x
networks and which kernel ani_b200_mlp_step picks.  No GPU needed: both are host functions of the library."""
import ctypes as C

from torchani_b200 import _lib, models, synthetic

KB = 1024
AVAIL = (227 - 12) * KB - 1024   # dynamic shared memory of the MLP kernels minus the 1 KB alignment slack


def model_of(dims, symbols):
    m = _lib.MLPModel()
    m.num_species = len(symbols)
    m.num_members = 8
    for s, sym in enumerate(symbols):
        h = [(v + 31) // 32 * 32 for v in dims[sym]]   # PackedNetworks pads every hidden width to a multiple of 32
        m.sp[s].h1, m.sp[s].h2, m.sp[s].h3 = h
    m.h1_max, m.h2_max, m.h3_max = (max(getattr(m.sp[s], f"h{i}") for s in range(len(symbols))) for i in (1, 2, 3))
    return m


def plan(lib, m):
    out = (C.c_int32 * 5)()
    assert lib.ani_b200_mlp_resident_plan(C.byref(m), out) == 0
    return dict(resident=out[0], ring=out[1], layer1_ring=out[2], avail=out[3], fits=bool(out[4]))


def test_resident_plan_fits_ani2x_and_ani1x_with_fp16_pieces():
    lib = _lib.lib()
    p2 = plan(lib, model_of(synthetic.DIMS_2X, models.SYMBOLS_2X))
    p1 = plan(lib, model_of(synthetic.DIMS_1X, models.SYMBOLS_1X))
    print("resident plan ANI-2x:", p2)
    print("resident plan ANI-1x:", p1)
    # widest hidden layer 256 (ANI-2x H) -> 8 K-blocks of 16 KB; ANI-1x 160 -> 5
    assert p2 == dict(resident=128 * KB, ring=2 * 32 * KB, layer1_ring=4 * 48 * KB, avail=AVAIL, fits=True)
    assert p1 == dict(resident=80 * KB, ring=4 * 32 * KB, layer1_ring=4 * 48 * KB, avail=AVAIL, fits=True)
    for p in (p1, p2):
        assert p["resident"] + p["ring"] <= p["avail"] and p["layer1_ring"] <= p["avail"]


def test_resident_plan_refuses_bf16_pieces():
    """3 x bf16 pieces: 24 KB per resident K-block and 48 KB per weight stage leave no two-stage ring."""
    lib = _lib.lib("bf16x3")
    for dims, symbols in ((synthetic.DIMS_2X, models.SYMBOLS_2X), (synthetic.DIMS_1X, models.SYMBOLS_1X)):
        m = model_of(dims, symbols)
        assert not plan(lib, m)["fits"]
        assert lib.ani_b200_mlp_step_kernel(C.byref(m), 128 * 80) == 0       # the data-flow launch


def test_step_kernel_selection(monkeypatch):
    lib = _lib.lib()
    m = model_of(synthetic.DIMS_2X, models.SYMBOLS_2X)
    monkeypatch.delenv("ANI_B200_MLP_CHAIN", raising=False)
    monkeypatch.delenv("ANI_B200_MLP_RESIDENT", raising=False)
    k = lambda model, rows_cap: lib.ani_b200_mlp_step_kernel(C.byref(model), rows_cap)   # noqa: E731
    short, long = 128 * 80, 128 * 400          # 640 chains of 8 members (10 k atoms), 3 200 (50 k atoms)
    assert k(m, short) == 2 and k(m, long) == 0                         # resident chains up to 8 per SM (148 SMs)
    assert lib.ani_b200_mlp_step_windows(C.byref(m), short) == 1
    monkeypatch.setenv("ANI_B200_MLP_RESIDENT", "0")
    assert k(m, short) == 0
    monkeypatch.setenv("ANI_B200_MLP_RESIDENT", "1")
    assert k(m, long) == 2
    monkeypatch.setenv("ANI_B200_MLP_CHAIN", "1")
    assert k(m, short) == 1                                             # the opt-in independent chains come first
    monkeypatch.delenv("ANI_B200_MLP_CHAIN")
    wide = model_of({**synthetic.DIMS_2X, "H": (288, 192, 160)}, models.SYMBOLS_2X)
    assert not plan(lib, wide)["fits"]                                  # a hidden layer wider than one accumulator
    assert k(wide, short) == 0
