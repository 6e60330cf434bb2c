"""-m gpu: gcgcn_gemm on every kernel route, and gcgcn_colsum, against float64.

The C entry point is called directly so that operand strides, pointer offsets and the workspace size are under the
test's control; the kernel timer tells which route ran, and every case asserts the one it was built to reach.

Two input families per case:
  * exact integers: A, B in [-8, 8], small integer alpha, beta, C and bias, K small enough that every partial sum
    stays below 2^24.  Every route, whatever its summation order or K split, must then equal float64 bit for bit --
    a single dropped, duplicated or misplaced element shows, which a tolerance could hide.
  * normal operands, within 2e-6 * max|ref| * sqrt(K) (a bound that single-pass TF32 misses).
"""
import math

import pytest
import torch

from gcgcn_b200 import _lib
from gcgcn_b200.functional import _stream

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
WS_FULL = 24 << 20                  # the GEMM's workspace cap (api.cu GEMM_WS_BYTES)
BLOB = 2 * 8 * (128 * 16 + 16)      # one pre-split 128 x 32 operand blob, hi and lo parts (gemm_tc.cu TC_B_BLOB_BYTES)
PAD_AB = 1e30                       # fills A and B outside their windows: a read of it would wreck the result
PAD_C = -777.25                     # fills C outside its window: must come back bit-identical
MAIN = {(0, 0): "nn", (0, 1): "nt", (1, 0): "tn", (1, 1): "tt"}

# (ld padding, base offset in floats) of A, B and C: tight and aligned; odd leading dimensions with unaligned bases;
# leading dimensions that are multiples of 4 on unaligned bases; padded rows on aligned bases (vector paths, ldc > N)
LAYOUTS = [((0, 0), (0, 0), (0, 0)), ((1, 1), (3, 2), (4, 3)), ((4, 3), (0, 1), (1, 0)),
           ((3, 0), (4, 0), (4, 0)), ((4, 0), (4, 0), (3, 1))]


def sms():
    return torch.cuda.get_device_properties(DEV).multi_processor_count


def cdiv(a, b):
    return -(-a // b)


def tc_splits(M, N, K, ws_bytes):
    """K splits launch_gemm_tc chooses (gemm_tc.cu)."""
    tiles = cdiv(M, 128) * cdiv(N, 128)
    if tiles >= sms() or K < 4096 or not ws_bytes:
        return 1
    s = min(max(sms() // tiles, 1), cdiv(K, 512), min(ws_bytes, WS_FULL) // (M * N * 4))
    return 1 if s < 2 else cdiv(K, cdiv(cdiv(K, s), 32) * 32)


def simt_splits(M, N, K, ws_bytes):
    """K splits of the CUDA-core kernel (gemm.cu launch_gemm)."""
    tiles = cdiv(M, 64) * cdiv(N, 64)
    if tiles >= 2 * sms() or K < 2048 or not ws_bytes:
        return 1
    s = min(cdiv(2 * sms(), tiles), cdiv(K, 512), min(ws_bytes, WS_FULL) // (M * N * 4))
    return 1 if s < 2 else cdiv(K, cdiv(cdiv(K, s), 16) * 16)


def is_tc(M, N, K):
    return K >= 1 and M * N * K >= 2e6


def reduce_name(M, N, splits, C, bias):
    """The split-K reduce kernel launch_splitk_reduce picks (the workspace is 16-byte aligned here)."""
    vec = N % 4 == 0 and C.stride(0) % 4 == 0 and C.data_ptr() % 16 == 0 and (bias is None or bias.data_ptr() % 16 == 0)
    if vec and splits >= 16 and M * N // 4 <= 64 * 1024:
        return "splitk_reduce4_wide"
    return "splitk_reduce4" if vec else "splitk_reduce"


def expected_route(ta, tb, M, N, K, ws_bytes, C, bias):
    """Kernel names one gcgcn_gemm call should launch."""
    if M == 0 or N == 0:
        return set()
    if is_tc(M, N, K):
        splits = tc_splits(M, N, K, ws_bytes)
        kblocks = cdiv(K, 32)
        bpre = (splits == 1 and not ta and M >= 4096 and N * K * 4 <= (8 << 20)
                and cdiv(N, 128) * kblocks * BLOB <= min(ws_bytes or 0, WS_FULL))
        if bpre and kblocks <= 4:
            names = {"gemm_presplit_b", "gemm_tc_nn<A in TMEM>"}
        elif bpre:
            names = {"gemm_presplit_b", f"gemm_tc_{MAIN[ta, tb]}<presplit B>"}
        else:
            names = {"gemm_tc_tn<MN-major>" if (ta, tb) == (1, 0) else f"gemm_tc_{MAIN[ta, tb]}"}
    else:
        splits = simt_splits(M, N, K, ws_bytes)
        names = {f"gemm_{MAIN[ta, tb]}"}
    if splits > 1:
        names.add(reduce_name(M, N, splits, C, bias))
    return names


class Strided:
    """A rows x cols float32 matrix stored with leading dimension cols + pad at `off` floats into a device buffer
    filled with `fill` elsewhere."""

    def __init__(self, values, pad, off, fill):
        rows, cols = values.shape
        self.ld = cols + pad
        self.buf = torch.full((off + max(rows, 1) * self.ld + 8,), fill, dtype=torch.float32, device=DEV)
        self.view = self.buf[off:off + rows * self.ld].view(rows, self.ld)[:, :cols]
        self.view.copy_(values)
        self.mask = torch.zeros_like(self.buf, dtype=torch.bool)
        self.mask[off:off + rows * self.ld].view(rows, self.ld)[:, :cols] = True
        self.outside = self.buf[~self.mask].clone()

    def untouched(self):
        return torch.equal(self.buf[~self.mask], self.outside)


def gemm(ta, tb, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, bias=None, ws_bytes=WS_FULL):
    """One gcgcn_gemm call on raw pointers; returns the kernel names it launched.  ws_bytes = 0: no workspace."""
    ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=DEV) if ws_bytes else None
    st = _stream(DEV)
    torch.cuda.synchronize()
    _lib.timing_begin(st)
    _lib.call("gcgcn_gemm", ta, tb, M, N, K, float(alpha), A, lda, B, ldb, float(beta), C, ldc, bias,
              None if ws is None else ws.data_ptr(), ws_bytes, st)
    ran = set(_lib.timing_end(st)) - {"(between calls)"}
    torch.cuda.synchronize()
    return ran


def operands(ta, tb, M, N, K, family, seed, row_scale=None):
    """CPU float32 op-storage A, B, C, bias and (alpha, beta) of one family."""
    g = torch.Generator().manual_seed(seed)
    ashape, bshape = ((K, M) if ta else (M, K)), ((N, K) if tb else (K, N))
    if family == "int":
        a = torch.randint(-8, 9, ashape, generator=g).float()
        b = torch.randint(-8, 9, bshape, generator=g).float()
        c = torch.randint(-4, 5, (M, N), generator=g).float()
        bias = torch.randint(-4, 5, (N,), generator=g).float()
        return a, b, c, bias, 0.5, -2.0
    a = torch.randn(ashape, generator=g)
    b = torch.randn(bshape, generator=g)
    c = torch.randn(M, N, generator=g)
    bias = torch.randn(N, generator=g)
    if row_scale is not None:          # rows of op(A) scaled by powers of two
        a = a * (row_scale[None, :] if ta else row_scale[:, None])
        return a, b, c, None, 1.0, 0.0
    return a, b, c, bias, 0.5, 2.0


def reference(ta, tb, a, b, c, bias, alpha, beta):
    A = a.to(DEV, torch.float64)
    B = b.to(DEV, torch.float64)
    r = alpha * ((A.t() if ta else A) @ (B.t() if tb else B))
    if beta != 0.0:
        r = r + beta * c.to(DEV, torch.float64)
    if bias is not None:
        r = r + bias.to(DEV, torch.float64)
    return r


def check(out, ref, family, K, what):
    """Exact for integers, else within 2e-6 * max|ref| * sqrt(K); returns the error relative to max|ref|."""
    out = out.double()
    assert torch.isfinite(out).all(), f"{what}: non-finite output"
    err = float((out - ref).abs().max()) if ref.numel() else 0.0
    scale = max(1.0, float(ref.abs().max())) if ref.numel() else 1.0
    if family == "int":
        assert err == 0.0, f"{what}: integer product off by {err}"
    else:
        assert err <= 2e-6 * scale * math.sqrt(max(1, K)), f"{what}: max|diff| {err:.3e} (max|ref| {scale:.3e})"
    return err / scale


def run_case(ta, tb, M, N, K, family, layout=LAYOUTS[0], ws_bytes=WS_FULL, seed=0, c_fill=None, bias_off=0,
             expect=None):
    """Build strided operands, call gcgcn_gemm, check the result, the untouched C padding and the route.  Returns
    (output, names, relative error)."""
    a, b, c, bias, alpha, beta = operands(ta, tb, M, N, K, family, seed)
    (pa, oa), (pb, ob), (pc, oc) = layout
    A, B = Strided(a, pa, oa, PAD_AB), Strided(b, pb, ob, PAD_AB)
    C = Strided(c, pc, oc, PAD_C)
    if c_fill is not None:                # beta = 0 over garbage: C must not be read
        C.view.fill_(c_fill)
        beta = 0.0
    bias_buf = torch.zeros(N + 4, device=DEV)
    bias_dev = bias_buf[bias_off:bias_off + N]
    bias_dev.copy_(bias)
    ran = gemm(ta, tb, M, N, K, alpha, A.view.data_ptr(), A.ld, B.view.data_ptr(), B.ld, beta, C.view.data_ptr(), C.ld,
               bias_dev.data_ptr(), ws_bytes)
    what = f"ta={ta} tb={tb} M={M} N={N} K={K} {family} layout={layout} ws={ws_bytes}"
    want = expected_route(ta, tb, M, N, K, ws_bytes, C.view, bias_dev) if expect is None else expect
    assert ran == want, f"{what}: ran {sorted(ran)}, expected {sorted(want)}"
    assert C.untouched(), f"{what}: C changed outside its M x N window"
    ref = reference(ta, tb, a, b, c, bias, alpha, beta)
    rel = check(C.view, ref, family, K, what)
    return C.view.clone(), ran, rel


# route -> (M, N, K); every transpose combination of each shape is run.  With ta = 1 the pre-split and TMEM shapes
# take the plain tensor-core kernels (the weight operand is pre-split only for an untransposed A).
ROUTES = {
    "simt": (37, 51, 77),
    "simt_splitk": (16, 16, 5000),
    "tc": (300, 260, 200),
    "tc_presplit_b": (4100, 130, 200),
    "tc_tmem_k100": (4100, 300, 100),
    "tc_tmem_k128": (4097, 256, 128),
    "tc_splitk": (256, 200, 9000),
}
TRANS = [(0, 0), (0, 1), (1, 0), (1, 1)]


@pytest.mark.parametrize("layout", range(len(LAYOUTS)))
@pytest.mark.parametrize("ta,tb", TRANS)
@pytest.mark.parametrize("route", list(ROUTES))
def test_strided_operands_on_every_route(route, ta, tb, layout):
    """Operands and C as windows into larger buffers (ld = width + {0, 1, 3, 4}, bases 0..3 floats off 16 bytes)."""
    M, N, K = ROUTES[route]
    for family in ("int", "normal"):
        run_case(ta, tb, M, N, K, family, LAYOUTS[layout], seed=layout)


@pytest.mark.parametrize("ta,tb", TRANS)
@pytest.mark.parametrize("route", ["simt", "simt_splitk", "tc", "tc_presplit_b", "tc_splitk"])
def test_rows_scaled_across_exponents(route, ta, tb):
    """Rows of op(A) scaled by 2^-20 .. 2^20: the hi/lo operand split must hold each row to its own scale."""
    M, N, K = ROUTES[route]
    scale = 2.0 ** torch.linspace(-20, 20, M).round()
    a, b, c, _, _, _ = operands(ta, tb, M, N, K, "normal", 7, row_scale=scale)
    A, B, C = Strided(a, 0, 0, PAD_AB), Strided(b, 0, 0, PAD_AB), Strided(c, 0, 0, PAD_C)
    ran = gemm(ta, tb, M, N, K, 1.0, A.view.data_ptr(), A.ld, B.view.data_ptr(), B.ld, 0.0, C.view.data_ptr(), C.ld)
    assert ran == expected_route(ta, tb, M, N, K, WS_FULL, C.view, None)
    ref = reference(ta, tb, a, b, c, None, 1.0, 0.0)
    err = (C.view.double() - ref).abs().amax(1)
    bound = 2e-6 * ref.abs().amax(1) * math.sqrt(K)
    assert bool((err <= bound).all()), f"worst row: err/bound = {float((err / bound).max()):.3f}"


# split-K cases by reduce kernel: (ta, tb, M, N, K, C layout, bias offset)
SPLITK = {
    "simt_vec4": (0, 0, 16, 16, 5000, LAYOUTS[0][2], 0),
    "simt_wide": (1, 0, 12, 16, 10000, LAYOUTS[0][2], 0),
    "simt_scalar": (0, 1, 12, 13, 10000, LAYOUTS[0][2], 0),
    "tc_wide": (1, 0, 128, 128, 40000, LAYOUTS[0][2], 0),
    "tc_wide_nn": (0, 0, 128, 128, 40000, (4, 0), 0),
    "tc_vec4": (1, 0, 512, 512, 8192, LAYOUTS[0][2], 0),
    "tc_scalar_n130": (1, 0, 128, 130, 20000, LAYOUTS[0][2], 0),
    "tc_scalar_c_offset": (1, 0, 128, 128, 40000, (0, 1), 0),
    "tc_scalar_bias_offset": (0, 1, 128, 128, 40000, (0, 0), 1),
}
SPLITK_REDUCE = {"simt_vec4": "splitk_reduce4", "simt_wide": "splitk_reduce4_wide", "simt_scalar": "splitk_reduce",
                 "tc_wide": "splitk_reduce4_wide", "tc_wide_nn": "splitk_reduce4_wide", "tc_vec4": "splitk_reduce4",
                 "tc_scalar_n130": "splitk_reduce", "tc_scalar_c_offset": "splitk_reduce",
                 "tc_scalar_bias_offset": "splitk_reduce"}


@pytest.mark.parametrize("case", list(SPLITK))
def test_split_k_on_each_reduce_kernel(case):
    """alpha != 1, beta != 0 and a bias on every reduce kernel; two runs bitwise equal."""
    ta, tb, M, N, K, c_layout, bias_off = SPLITK[case]
    layout = ((0, 0), (0, 0), c_layout)
    for family in ("int", "normal"):
        r1, ran, _ = run_case(ta, tb, M, N, K, family, layout, seed=3, bias_off=bias_off)
        assert SPLITK_REDUCE[case] in ran, f"{case}: ran {sorted(ran)}"
        r2, _, _ = run_case(ta, tb, M, N, K, family, layout, seed=3, bias_off=bias_off)
        assert torch.equal(r1, r2), f"{case}: two runs differ"


@pytest.mark.parametrize("ta,tb", [(0, 0), (1, 0)])
@pytest.mark.parametrize("case", list(ROUTES) + ["tc_splitk_scalar"])
def test_beta_zero_does_not_read_c(case, ta, tb):
    """beta = 0 over a C full of NaN gives a finite, exact result on every route."""
    if case == "tc_splitk_scalar":
        M, N, K = 128, 130, 20000
    else:
        M, N, K = ROUTES[case]
    run_case(ta, tb, M, N, K, "int", LAYOUTS[1] if ta else LAYOUTS[0], c_fill=float("nan"))


@pytest.mark.parametrize("ta,tb", TRANS)
@pytest.mark.parametrize("M,N", [(37, 51), (300, 260), (4100, 130)])
def test_k_zero_gives_beta_c_plus_bias(M, N, ta, tb):
    g = torch.Generator().manual_seed(M + N)
    c = torch.randint(-4, 5, (M, N), generator=g).float()
    bias = torch.randint(-4, 5, (N,), generator=g).float().to(DEV)
    A = torch.full((4,), PAD_AB, device=DEV)
    for beta in (-2.0, 0.0):
        C = Strided(c, 3, 1, PAD_C)
        if beta == 0.0:
            C.view.fill_(float("nan"))
        ran = gemm(ta, tb, M, N, 0, 0.5, A.data_ptr(), 1, A.data_ptr(), 1, beta, C.view.data_ptr(), C.ld,
                   bias.data_ptr())
        assert ran == {f"gemm_{MAIN[ta, tb]}"}, ran
        assert C.untouched()
        want = (beta * c.to(DEV) if beta else torch.zeros(M, N, device=DEV)) + bias
        assert torch.equal(C.view, want)


@pytest.mark.parametrize("M,N,K", [(0, 51, 77), (37, 0, 77), (0, 0, 0), (0, 1024, 40000), (4100, 0, 128)])
def test_empty_output_leaves_c_untouched(M, N, K):
    A = torch.full((16,), PAD_AB, device=DEV)
    C = torch.full((64,), PAD_C, device=DEV)
    before = C.clone()
    for ta, tb in TRANS:
        ran = gemm(ta, tb, M, N, K, 1.0, A.data_ptr(), max(1, K), A.data_ptr(), max(1, N), 0.0, C.data_ptr(), max(1, N))
        assert ran == set()
    assert torch.equal(C, before)


# (ta, tb, M, N, K, full-workspace route, no-/short-workspace route, bytes of the short workspace)
LEVERS = {
    "presplit_b": (0, 1, 4100, 130, 200, {"gemm_presplit_b", "gemm_tc_nt<presplit B>"}, {"gemm_tc_nt"},
                   2 * 7 * BLOB - BLOB),
    "tmem": (0, 0, 4100, 300, 100, {"gemm_presplit_b", "gemm_tc_nn<A in TMEM>"}, {"gemm_tc_nn"}, 3 * 4 * BLOB - BLOB),
    "tc_splitk": (1, 0, 128, 128, 40000, {"gemm_tc_tn<MN-major>", "splitk_reduce4_wide"}, {"gemm_tc_tn<MN-major>"},
                  2 * 128 * 128 * 4 - 4),
    "simt_splitk": (0, 0, 16, 16, 5000, {"gemm_nn", "splitk_reduce4"}, {"gemm_nn"}, 2 * 16 * 16 * 4 - 4),
}


@pytest.mark.parametrize("lever", list(LEVERS))
def test_workspace_size_selects_the_route(lever):
    """No workspace, one blob (or one partial) short of what the faster route needs, and the full 24 MB: the route
    changes, the result does not leave the bound."""
    ta, tb, M, N, K, full, reduced, short = LEVERS[lever]
    for ws_bytes, want in ((WS_FULL, full), (short, reduced), (0, reduced)):
        for family in ("int", "normal"):
            run_case(ta, tb, M, N, K, family, ws_bytes=ws_bytes, seed=11, expect=want)


LONG_K = [(128, 128, 119808), (128, 256, 119808), (128, 1024, 119808), (128, 128, 140000)]


@pytest.mark.parametrize("ws_bytes", [WS_FULL, 0], ids=["ws", "no-ws"])
@pytest.mark.parametrize("M,N,K", LONG_K)
def test_long_k_weight_gradients(M, N, K, ws_bytes):
    """The weight-gradient shapes of the benchmark, [K, 128]^T [K, N] over every node row, with and without a
    workspace (without one the product is not split across CTAs)."""
    for family in ("int", "normal"):
        _, ran, rel = run_case(1, 0, M, N, K, family, ws_bytes=ws_bytes, seed=5)
        assert any(n.startswith("splitk_reduce") for n in ran) == bool(ws_bytes), ran
        print(f"long K {family}: [{K},{M}]^T[{K},{N}] ws={ws_bytes}: max|err|/max|ref| = {rel:.3e}")


def test_every_gemm_kernel_is_reached():
    """One case per route; together they launch every kernel name gcgcn_gemm can reach (the pre-split-A route needs
    a generated operand and is covered by the classifier tests)."""
    seen = set()
    for route, (M, N, K) in ROUTES.items():
        for ta, tb in TRANS:
            seen |= run_case(ta, tb, M, N, K, "int")[1]
    for case in SPLITK:
        ta, tb, M, N, K, c_layout, bias_off = SPLITK[case]
        seen |= run_case(ta, tb, M, N, K, "int", ((0, 0), (0, 0), c_layout), bias_off=bias_off)[1]
    everything = {f"gemm_{t}" for t in MAIN.values()} | {"gemm_tc_nn", "gemm_tc_nt", "gemm_tc_tt", "gemm_tc_tn<MN-major>",
                                                          "gemm_tc_nn<presplit B>", "gemm_tc_nt<presplit B>",
                                                          "gemm_tc_nn<A in TMEM>", "gemm_presplit_b", "splitk_reduce",
                                                          "splitk_reduce4", "splitk_reduce4_wide"}
    assert seen == everything, (sorted(everything - seen), sorted(seen - everything))


# ---------------------------------------------------------------------------------------------------- gcgcn_colsum
COLSUM_N = [1, 97, 127, 128, 129, 1024]
COLSUM_M = [0, 1, 63, 64, 65, 4097, 119808]


def colsum(X, ldx, M, N):
    out = torch.full((N,), float("nan"), device=DEV)
    ws = torch.empty(16 << 20, dtype=torch.uint8, device=DEV)
    st = _stream(DEV)
    torch.cuda.synchronize()
    _lib.timing_begin(st)
    _lib.call("gcgcn_colsum", X, M, N, ldx, out.data_ptr(), ws.data_ptr(), ws.numel(), st)
    ran = set(_lib.timing_end(st)) - {"(between calls)"}
    return out, ran


@pytest.mark.parametrize("layout", ["tight", "ldx+3", "ldx+4,offset1"])
@pytest.mark.parametrize("N", COLSUM_N)
@pytest.mark.parametrize("M", COLSUM_M)
def test_colsum_against_fp64(M, N, layout):
    """Column sums (every bias gradient): exact on integers, within ~1e-6 sqrt(M) of each column's scale on normal
    inputs, bitwise reproducible.  The one-float offset sends N = 128 to the generic path."""
    pad, off = {"tight": (0, 0), "ldx+3": (3, 0), "ldx+4,offset1": (4, 1)}[layout]
    ldx = N + pad
    buf = torch.empty(off + max(M, 1) * ldx, device=DEV)
    X = buf[off:off + M * ldx].view(M, ldx)[:, :N]
    g = torch.Generator(device=DEV).manual_seed(M * 31 + N)
    fast = N == 128 and ldx % 4 == 0 and off == 0 and M > 0
    for family in ("int", "normal"):
        if family == "int":
            buf.copy_(torch.randint(-8, 9, buf.shape, generator=g, device=DEV).float())
        else:
            buf.copy_(torch.randn(buf.shape, generator=g, device=DEV))
        out, ran = colsum(X.data_ptr(), ldx, M, N)
        assert ran == (set() if M == 0 else {"colsum128_partial" if fast else "colsum_partial", "reduce_partials"}), ran
        ref = X.double().sum(0)
        if family == "int":
            assert torch.equal(out.double(), ref), f"M={M} N={N}: {float((out.double() - ref).abs().max())}"
        else:
            col_scale = X.double().abs().amax(0) if M else torch.ones(N, device=DEV, dtype=torch.float64)
            err = (out.double() - ref).abs()
            assert bool((err <= 1e-6 * math.sqrt(max(M, 1)) * col_scale).all()), float((err / col_scale).max())
        again, _ = colsum(X.data_ptr(), ldx, M, N)
        assert torch.equal(out, again)
