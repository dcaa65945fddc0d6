"""The case table of the bit-exact conv tests (tests/test_conv_exact_gpu.py), checked on the host: which kernel each case
runs (po2_conv2d_kernel_kind / po2_conv2d_wgrad_kernel_kind answer without a device), which K3 branch it reaches
(a model of plan_umma, cross-checked against the library's packed-operand size), that its sums stay exact in fp32, and
that the entry points refuse an x / output gradient their kernel would read with 128-bit loads from a pointer that is
not 16-byte aligned (PO2_E_ALIGN, before any launch)."""
import ctypes

import pytest

from po2_quantization_b200 import _lib

PO2_E_ALIGN = -5
PO2_E_UNSUPPORTED = -10
SMS = 148                        # B200; the library assumes 148 where it cannot ask a device

# ---- forward cases -------------------------------------------------------------------------------------------------
# (name, B, C, H, W, K, k, stride, groups, compute, kind, branches); pad = k // 2.  kind: po2_conv2d_kernel_kind on a
# B200 (0 direct fp32, 1 depthwise, 2 register-fed tcgen05 K3, 3 TMA-fed K3T, 4 pointwise cluster GEMM).  branches:
# vec / scalar (depthwise); vec4 / scalar / hw1 (K3 producer); s2 (4-phase staging); flat (1x1 map as one row); cpad
# (Cpad > C); nchunk (> 1 channel chunk); ntiles (> 1 N tile); ntail (partial last N tile); mloop (CTAs loop over
# items); mode0 / mode4 / mode1 (K3T); split / single (cluster CTAs over C).  K3 numbers from plan_umma at 148 SMs.
FWD = [
    ("direct grouped 16->32 g4 @8", 2, 16, 8, 8, 32, 3, 1, 4, 0, 0, ()),                    # groups 4: no tensor-core kernel
    ("direct 5x5 8->8 @12", 2, 8, 12, 12, 8, 5, 1, 1, 0, 0, ()),                            # 5x5
    ("direct fp32 mode resnet 16->16 @32", 8, 16, 32, 32, 16, 3, 1, 1, 1, 0, ()),          # compute 1
    ("dw vec s1 32 @16", 4, 32, 16, 16, 32, 3, 1, 32, 0, 1, ("vec",)),                      # W % 4 == 0, Q % 4 == 0
    ("dw vec s2 24 @16", 4, 24, 16, 16, 24, 3, 2, 24, 0, 1, ("vec",)),                      # W == 2Q = 16
    ("dw scalar 7 @9x7", 3, 7, 9, 7, 7, 3, 1, 7, 0, 1, ("scalar",)),                         # odd W, C % 4 != 0
    ("dw scalar s2 5 @1x1", 2, 5, 1, 1, 5, 3, 2, 5, 0, 1, ("scalar",)),                      # 1x1 map, stride 2
    # K3, bf16 operands                                                          plan_umma: Cpad, NT x ntiles_n, nchunk, items / m_step
    ("k3 3x3 s1 16->16 @16", 4, 16, 16, 16, 16, 3, 1, 1, 0, 2, ("vec4",)),                   # 16, 16x1, 1, 10/10
    ("k3 3x3 s1 24->40 @14x9", 3, 24, 14, 9, 40, 3, 1, 1, 0, 2, ("scalar", "cpad", "ntiles", "ntail")),   # 32, 16x3, 1, 4/4
    ("k3 3x3 s2 16->32 @16", 4, 16, 16, 16, 32, 3, 2, 1, 0, 2, ("s2", "scalar", "ntiles")),  # 16, 16x2, 1, 3/3; 4 phases
    ("k3 1x1 s1 32->48 @6", 4, 32, 6, 6, 48, 1, 1, 1, 0, 2, ("flat", "vec4", "ntiles")),     # 32, 16x3, 1, 2/2; rows of 36
    ("k3 1x1 s2 32->64 @8", 4, 32, 8, 8, 64, 1, 2, 1, 0, 2, ("scalar", "ntiles")),           # 32, 16x4, 1, 1/1
    ("k3 3x3 20->17 @8 (Cpad, K 17)", 3, 20, 8, 8, 17, 3, 1, 1, 0, 2, ("vec4", "cpad", "ntiles", "ntail")),  # 32, 16x2, 1, 2/2
    ("k3 3x3 32->300 @8 (N tiles)", 2, 32, 8, 8, 300, 3, 1, 1, 0, 2, ("vec4", "ntiles", "ntail")),  # 32, 16x19, 1, 2/2
    ("k3 3x3 256->32 @8 (chunks)", 4, 256, 8, 8, 32, 3, 1, 1, 0, 2, ("vec4", "nchunk", "ntiles")),  # 256, 16x2, 3 (CC 96), 3/3
    ("k3 3x3 32->32 @1x1 (hw1)", 16, 32, 1, 1, 32, 3, 1, 1, 0, 2, ("hw1", "ntiles")),        # 32, 16x2, 1, 1/1
    ("k3 3x3 16->16 H=1", 4, 16, 1, 32, 16, 3, 1, 1, 0, 2, ("vec4",)),                       # 16, 16x1, 1, 3/3
    ("k3 3x3 16->16 W=1", 4, 16, 32, 1, 16, 3, 1, 1, 0, 2, ("scalar",)),                     # 16, 16x1, 1, 3/3
    ("k3 3x3 32->32 @16 B=1", 1, 32, 16, 16, 32, 3, 1, 1, 0, 2, ("vec4", "ntiles")),         # 32, 16x2, 1, 3/3
    ("k3 resnet 16->16 @32 B=128", 128, 16, 32, 32, 16, 3, 1, 1, 0, 2, ("vec4", "mloop")),   # 16, 16x1, 1, 1090/148
    # K3, tf32 operands: the shapes K3T declines
    ("k3 tf32 3x3 s2 16->32 @16", 4, 16, 16, 16, 32, 3, 2, 1, 2, 2, ("s2", "scalar", "nchunk", "ntiles")),  # 16, 16x2, 2, 3/3
    ("k3 tf32 3x3 12->16 @16 (C % 8)", 4, 12, 16, 16, 16, 3, 1, 1, 2, 2, ("vec4", "cpad")),  # 16, 16x1, 1, 10/10
    ("k3 tf32 3x3 16->16 @12", 4, 16, 12, 12, 16, 3, 1, 1, 2, 2, ("vec4",)),                 # 16, 16x1, 1, 6/6; W 12
    ("k3 tf32 3x3 16->24 @40", 2, 16, 40, 40, 24, 3, 1, 1, 2, 2, ("vec4", "ntiles", "ntail")),  # 16, 16x2, 1, 27/27; W 40
    ("k3 tf32 1x1 32->48 @6", 4, 32, 6, 6, 48, 1, 1, 1, 2, 2, ("flat", "vec4", "ntiles")),   # 32, 16x3, 1, 2/2; HW 36
    ("k3 tf32 3x3 16->16 W=1", 4, 16, 32, 1, 16, 3, 1, 1, 2, 2, ("scalar",)),                # 16, 16x1, 1, 3/3
    # K3T (plan_tma: mode 0 for 3x3 at 16 < W <= 32, mode 4 at W 4 / 8 / 16, mode 1 / 2 for 1x1 at HW % 32 == 0)
    ("k3t mode0 16->16 @32", 4, 16, 32, 32, 16, 3, 1, 1, 2, 3, ("mode0",)),
    ("k3t mode0 24->40 @20x24", 3, 24, 20, 24, 40, 3, 1, 1, 2, 3, ("mode0",)),
    ("k3t mode4 16->32 @16", 4, 16, 16, 16, 32, 3, 1, 1, 2, 3, ("mode4",)),                # W 16
    ("k3t mode4 32->32 @8", 8, 32, 8, 8, 32, 3, 1, 1, 2, 3, ("mode4",)),                   # W 8
    ("k3t mode4 64->64 @4", 16, 64, 4, 4, 64, 3, 1, 1, 2, 3, ("mode4",)),                  # W 4
    ("k3t 1x1 32->64 @8", 4, 32, 8, 8, 64, 1, 1, 1, 2, 3, ("mode1",)),                     # HW 64 = 2 runs
    ("k3t resnet 16->16 @32 B=128", 128, 16, 32, 32, 16, 3, 1, 1, 2, 3, ("mode0",)),
    # pointwise cluster GEMM (1x1 maps of <= 16 pixels); tiles 32 x 64, KS = min(ceil(148 / tiles), C / 32, 8)
    ("pw split 576->160 @1", 16, 576, 1, 1, 160, 1, 1, 1, 0, 4, ("split",)),               # 3 tiles: KS 8
    ("pw split 960->100 @2x2 tf32", 8, 960, 2, 2, 100, 1, 1, 1, 2, 4, ("split",)),          # 2 tiles: KS 8
    ("pw single 24->40 @4x4", 4, 24, 4, 4, 40, 1, 1, 1, 0, 4, ("single",)),                # C 24 < 64: KS 1
    ("pw single 30->70 @3x3 fp32", 5, 30, 3, 3, 70, 1, 1, 1, 1, 4, ("single",)),            # C % 4 != 0
]

# ---- data gradient: the forward kernel on the transposed, rotated weight (in = K channels, out = C) ------------------
# (name, B, C, H, W, K, k, compute, packed): packed -- the multi-descriptor quantizer can emit the operand (no padding)
DGRAD = [
    ("dg 3x3 16<-32 @16", 4, 16, 16, 16, 32, 3, 0, True),
    ("dg 3x3 20<-24 @8 (C, K % 16)", 3, 20, 8, 8, 24, 3, 0, False),
    ("dg 1x1 33<-17 @6x10", 2, 33, 6, 10, 17, 1, 0, False),
    ("dg 3x3 16<-16 @9x7 scalar", 3, 16, 9, 7, 16, 3, 0, True),
    ("dg tf32 3x3 32<-32 @16", 4, 32, 16, 16, 32, 3, 2, True),
    ("dg tf32 3x3 20<-12 @8", 3, 20, 8, 8, 12, 3, 2, False),
    ("dg tf32 1x1 48<-32 @8", 4, 48, 8, 8, 32, 1, 2, True),
    ("dg tf32 3x3 24<-40 @12", 2, 24, 12, 12, 40, 3, 2, False),
]

# ---- weight gradient ------------------------------------------------------------------------------------------------
# (name, B, C, H, W, K, k, compute, kind, branches); kind: po2_conv2d_wgrad_kernel_kind on a B200 (1 K5, 2 K5T,
# 3 pointwise GEMM).  K5: vec4 / scalar staging, copies3 (three shifted copies, Cpad <= 32), M128 (K > 64).
# K5T: merged (W == 32 or 1x1 with HW % 32 == 0) / runs (one box per 32-pixel run), rsplit (9 C > 512: filter rows
# over blockIdx.y), M128.
WGRAD = [
    ("k5 3x3 16->16 @16", 4, 16, 16, 16, 16, 3, 0, 1, ("vec4", "copies3")),
    ("k5 3x3 24->40 @14x9", 3, 24, 14, 9, 40, 3, 0, 1, ("scalar", "copies3")),
    ("k5 3x3 64->96 @8", 4, 64, 8, 8, 96, 3, 0, 1, ("vec4", "M128")),
    ("k5 1x1 100->72 @7x9", 3, 100, 7, 9, 72, 1, 0, 1, ("scalar", "M128")),
    ("k5 tf32 3x3 12->16 @8 (K5T declines C % 8)", 4, 12, 8, 8, 16, 3, 2, 1, ("vec4", "copies3")),
    ("k5t 3x3 8->8 @32", 3, 8, 32, 32, 8, 3, 2, 2, ("merged",)),
    ("k5t 3x3 16->24 @8", 6, 16, 8, 8, 24, 3, 2, 2, ("runs",)),
    ("k5t 3x3 64->128 @8", 8, 64, 8, 8, 128, 3, 2, 2, ("runs", "rsplit", "M128")),
    ("k5t 3x3 16->16 @16x32", 5, 16, 16, 32, 16, 3, 2, 2, ("merged",)),
    ("k5t 1x1 40->72 @6", 3, 40, 6, 6, 72, 1, 2, 2, ("runs", "M128")),
    ("k5t 1x1 32->128 @8", 4, 32, 8, 8, 128, 1, 2, 2, ("merged", "M128")),
    ("pw 64->384 @2", 16, 64, 2, 2, 384, 1, 2, 3, ()),
    ("pw 20->200 @3 bf16", 3, 20, 3, 3, 200, 1, 0, 3, ()),
]

# ---- stem / depthwise backward (CUDA-core kernels of csrc/po2_conv_bwd.cu) ------------------------------------------
STEM = [(5, 3, 32, 32, 16), (2, 3, 9, 7, 8)]                                 # (B, C, H, W, K), 3x3 pad 1
# (name, B, C, H, W, stride): dgrad and wgrad of a depthwise 3x3 pad-1 layer
DEPTHWISE = [("dw 32 @16", 4, 32, 16, 16, 1), ("dw 7 @9x7 (C % 4)", 3, 7, 9, 7, 1), ("dw 12 @1x1", 8, 12, 1, 1, 1),
             ("dw 6 @2x1", 5, 6, 2, 1, 1), ("dw 9 @1x2", 4, 9, 1, 2, 1), ("dw 16 @8 B=1", 1, 16, 8, 8, 1),
             ("dw 24 s2 @16", 4, 24, 16, 16, 2)]
# (name, B, C, H, W, K, k): dense stride-2 layers whose backward goes through po2_dilate2
STRIDE2 = [("s2 3x3 16->32 @16", 4, 16, 16, 16, 32, 3), ("s2 1x1 16->32 @16", 4, 16, 16, 16, 32, 1),
           ("s2 3x3 8->16 @12x8", 3, 8, 12, 8, 16, 3)]


def out_hw(H, W, k, stride):
    pad = k // 2
    return (H + 2 * pad - k) // stride + 1, (W + 2 * pad - k) // stride + 1


def fwd_exact(C, k, groups):
    """every partial sum of the forward is a multiple of the lattice step 2^-10 below 2^23 steps (one bit of margin
    for the tensor core's aligned adders): |x| <= 4, |w| <= 2^7 steps, k*k*C/groups terms"""
    return 4 * k * k * (C // groups) * 2 ** 7 < 2 ** 23


def dgrad_exact(K, k):
    return 4 * k * k * K * 2 ** 7 < 2 ** 23


def wgrad_exact(B, P, Q):
    return 16 * B * P * Q < 2 ** 23


def k3_plan(B, C, H, W, K, k, stride, compute, sms=SMS):
    """plan_umma (csrc/po2_conv.cu) for the forward geometry: the fields that pick K3's branches"""
    tf32 = compute == 2
    G = 4 if tf32 else 8
    KCH, eb = 2 * G, (4 if tf32 else 2)
    P, Q = out_hw(H, W, k, stride)
    k3 = k == 3
    if not k3 and stride == 1:                      # a 1x1 map becomes one row of H*W pixels
        W, H, Q, P = H * W, 1, P * Q, 1
    ntaps = k * k
    pitch, rows_img, top = Q + k3, P + k3, int(k3)
    Ltot = (B * rows_img + top) * pitch
    if not k3:
        nphase, hb, ha = 1, 0, 0
    elif stride == 1:
        nphase, hb, ha = 1, pitch + 1, pitch + 1
    else:
        nphase, hb, ha = 4, pitch + 1, 0
    strip = 128 + hb + ha
    Cpad = -(-C // KCH) * KCH
    Kp = -(-K // 16) * 16
    NT = min(Kp, 256)
    while NT > 16 and ntaps * Cpad * NT * eb > 112 * 1024:
        NT -= 16
    assert ntaps * Cpad * NT * eb <= 112 * 1024
    nitems_m = -(-Ltot // 128)
    while NT > 16 and nitems_m * -(-Kp // (NT - 16)) <= sms:
        NT -= 16
    ntiles_n = -(-Kp // NT)
    NT = -(-(-(-Kp // ntiles_n)) // 16) * 16
    CC = Cpad
    while CC > KCH and nphase * CC * strip * eb > 32 * 1024:
        CC -= KCH
    m_step = min(nitems_m, max(sms // ntiles_n, 1))
    return dict(Cpad=Cpad, NT=NT, ntiles_n=ntiles_n, nchunk=-(-Cpad // CC), nitems_m=nitems_m, m_step=m_step,
                nphase=nphase, flat=(not k3 and stride == 1), vec4=(stride == 1 and W % 4 == 0),
                hw1=(H * W == 1 and C % 4 == 0), pack_bytes=ntiles_n * ntaps * Cpad * NT * eb)


def k3_branches(plan, C, K):
    """the K3 branches a plan reaches (the names of the FWD table)"""
    b = {"vec4"} if plan["vec4"] else ({"hw1"} if plan["hw1"] else {"scalar"})
    if plan["nphase"] == 4:
        b.add("s2")
    if plan["flat"]:
        b.add("flat")
    if plan["Cpad"] > C:
        b.add("cpad")
    if plan["nchunk"] > 1:
        b.add("nchunk")
    if plan["ntiles_n"] > 1:
        b.add("ntiles")
    if plan["ntiles_n"] * plan["NT"] > K:
        b.add("ntail")
    if plan["m_step"] < plan["nitems_m"]:
        b.add("mloop")
    return b


@pytest.fixture(scope="module")
def lib():
    return _lib.load()


def _fwd_args(case):
    name, B, C, H, W, K, k, stride, groups, compute, kind, branches = case
    return (B, C, H, W, K, k, k, stride, k // 2, groups, compute)


@pytest.mark.parametrize("case", FWD, ids=lambda c: c[0])
def test_forward_case_runs_the_kernel_it_names(lib, case):
    name, B, C, H, W, K, k, stride, groups, compute, kind, branches = case
    assert fwd_exact(C, k, groups), name
    got = lib.po2_conv2d_kernel_kind(*_fwd_args(case))
    # K3T needs the driver's tensor-map encoder: without a device the query answers 2 for its shapes
    assert got == kind or (kind == 3 and got == 2), (name, got)
    if kind in (2, 3):
        plan = k3_plan(B, C, H, W, K, k, stride, compute)
        assert lib.po2_conv2d_pack_bytes(*_fwd_args(case)) == -(-plan["pack_bytes"] // 256) * 256, name
        if kind == 2:
            assert set(branches) == k3_branches(plan, C, K), (name, sorted(k3_branches(plan, C, K)))
    elif kind == 1:
        P, Q = out_hw(H, W, k, stride)
        vec = W % 4 == 0 and Q % 4 == 0 and (stride == 1 or W == 2 * Q)
        assert branches == (("vec",) if vec else ("scalar",)), name
    elif kind == 4:
        tiles = -(-(B * H * W) // 32) * -(-K // 64)
        ks = max(min(-(-SMS // tiles), C // 32, 8), 1)
        assert branches == (("split",) if ks > 1 else ("single",)), (name, ks)


@pytest.mark.parametrize("case", DGRAD, ids=lambda c: c[0])
def test_dgrad_case_runs_on_the_tensor_core_kernel(lib, case):
    name, B, C, H, W, K, k, compute, packed = case
    assert dgrad_exact(K, k), name
    # the data gradient is the forward conv of the output gradient (K channels) into C channels
    assert lib.po2_conv2d_kernel_kind(B, K, H, W, C, k, k, 1, k // 2, 1, compute) in (2, 3), name
    assert lib.po2_conv2d_dgrad_workspace(B, C, H, W, K, k, k, k // 2, compute) > 0, name
    assert (lib.po2_conv2d_dgrad_pack_bytes(B, C, H, W, K, k, k, k // 2, compute) > 0) == packed, name


def test_dgrad_workspace_is_zero_where_dgrad_refuses_the_shape(lib):
    """5x5 pad 2 and 3x3 pad 0 have no tensor-core data gradient: the workspace query agrees with po2_conv2d_dgrad."""
    ok, big = ctypes.c_void_p(0x1000), 1 << 30
    for B, C, H, W, K, k, pad in ((2, 8, 8, 8, 8, 5, 2), (2, 8, 8, 8, 8, 3, 0)):
        for compute in (0, 2):
            assert lib.po2_conv2d_dgrad_workspace(B, C, H, W, K, k, k, pad, compute) == 0
            assert lib.po2_conv2d_dgrad(ok, ok, ok, ok, B, C, H, W, K, k, k, 1, pad, 1, 0, 4, 1, compute, ok, big,
                                        None) == PO2_E_UNSUPPORTED


@pytest.mark.parametrize("case", WGRAD, ids=lambda c: c[0])
def test_wgrad_case_runs_the_kernel_it_names(lib, case):
    name, B, C, H, W, K, k, compute, kind, branches = case
    assert wgrad_exact(B, H, W), name
    got = lib.po2_conv2d_wgrad_kernel_kind(B, C, H, W, K, k, k, 1, k // 2, 1, compute)
    # K5T also needs the tensor-map encoder: without a device its shapes report K5
    assert got == kind or (kind == 2 and got == 1), (name, got)
    if kind == 1:
        plan = k3_plan(B, C, H, W, K, k, 1, 0)
        assert ("vec4" in branches) == plan["vec4"], name
        assert ("copies3" in branches) == (k == 3 and plan["Cpad"] <= 32), name
    if kind in (1, 2):
        assert ("M128" in branches) == (K > 64), name
    if kind == 2:
        HW = H * W
        assert ("merged" in branches) == ((W == 32) if k == 3 else HW % 32 == 0), name
        assert ("rsplit" in branches) == (k == 3 and 9 * C > 512), name


def test_backward_tables_stay_exact():
    for B, C, H, W, K in STEM:
        assert wgrad_exact(B, H, W) and fwd_exact(C, 3, 1)
    for name, B, C, H, W, stride in DEPTHWISE:
        assert wgrad_exact(B, H, W) and dgrad_exact(1, 3), name
    for name, B, C, H, W, K, k in STRIDE2:
        assert wgrad_exact(B, H, W) and dgrad_exact(K, k) and fwd_exact(C, k, 1), name


def test_misaligned_operands_are_refused_before_any_launch(lib):
    """A kind-2 geometry (stride 1, W % 4 == 0: 128-bit producer loads) with x / the output gradient at 0x1004: every
    entry point returns PO2_E_ALIGN with enough (fake) workspace, before it would launch anything."""
    ok, bad = ctypes.c_void_p(0x1000), ctypes.c_void_p(0x1004)
    big = 1 << 30
    geo = (4, 16, 16, 16, 16, 3, 3, 1, 1, 1)                      # B C H W K R S stride pad groups
    for compute in (0, 2):
        assert lib.po2_conv2d_kernel_kind(*geo, compute) in (2, 3)
        assert lib.po2_conv2d_fwd(bad, ok, ok, ok, *geo, 0, 4, 1, compute, ok, big, None) == PO2_E_ALIGN
        assert lib.po2_conv2d_fwd_ep(bad, ok, ok, ok, *geo, 0, 4, 1, compute, ok, big, ok, ok, None, 1, None) == PO2_E_ALIGN
        assert lib.po2_conv2d_fwd_packed(bad, ok, ok, ok, *geo, compute, None) == PO2_E_ALIGN
        assert lib.po2_conv2d_fwd_packed_ep(bad, ok, ok, ok, *geo, compute, ok, ok, ok, 2, None) == PO2_E_ALIGN
        assert lib.po2_qconv2d_fwd(bad, ok, ok, ok, ok, *geo, 4, 1, 0, 0, compute, ok, big, ok, None) == PO2_E_ALIGN
        dg = (4, 16, 16, 16, 16, 3, 3)                             # B C H W K R S
        assert lib.po2_conv2d_dgrad(bad, ok, ok, ok, *dg, 1, 1, 1, 0, 4, 1, compute, ok, big, None) == PO2_E_ALIGN
        assert lib.po2_conv2d_dgrad_packed(bad, ok, ok, ok, *dg, 1, compute, None) == PO2_E_ALIGN
        assert lib.po2_conv2d_wgrad_kernel_kind(*geo, compute) in (1, 2)
        for g_out, x in ((bad, ok), (ok, bad)):
            assert lib.po2_conv2d_wgrad(g_out, x, ok, *geo, compute, ok, big, None) == PO2_E_ALIGN
            assert lib.po2_conv2d_wgrad_z(g_out, x, ok, *geo, compute, ok, big, ok, None) == PO2_E_ALIGN
    # the hw1 producer (3x3 on a 1x1 map, C % 4 == 0) loads channel groups with 128-bit loads too
    assert lib.po2_conv2d_fwd(bad, ok, ok, ok, 16, 32, 1, 1, 32, 3, 3, 1, 1, 1, 0, 4, 1, 0, ok, big, None) == PO2_E_ALIGN
    # the small-pointwise GEMM reads the fp32 weight with 128-bit loads when C % 4 == 0
    assert lib.po2_conv2d_kernel_kind(4, 24, 4, 4, 40, 1, 1, 1, 0, 1, 0) == 4
    assert lib.po2_conv2d_fwd(ok, bad, ok, ok, 4, 24, 4, 4, 40, 1, 1, 1, 0, 1, 0, 4, 1, 0, ok, big, None) == PO2_E_ALIGN
