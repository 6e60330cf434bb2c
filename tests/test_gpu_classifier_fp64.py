"""-m gpu: the relation classifier and the trainer's loss against float64 on every route, the bilinear form in both its
operand types.

The bilinear form runs on three tensor-core modes of gemm_tc.cu, in fp32 (3xTF32) or on bf16 operands: the row-dot
epilogue (forward), the row-accumulate epilogue (dh, dt) and the weight-gradient GEMM whose [pairs, R*128] operand its
producers generate from t and dout, walked in 4096-row ranges (one range: the epilogue applies beta; several: split-K
partials and an fp32 reduction) (dW').  BilinearFn makes the backward in host calls of up to FUSED_CHUNK_PAIRS pairs
that accumulate dW' through beta = 1.  The cases below put P on both sides of every one of those boundaries and of the
128-pair row tiles, and R from 1 to past the 148 SMs of a B200, call the C entry points with the strides, accumulation
and beta the header documents, and run the loss and the per-document bias on a ragged batch with a document of 65 536
pairs.

fp32 is checked against float64 (oracle/classifier_oracle.py), bf16 against float64 of the rounded operands
(tests/classifier_bf16_oracle.py): either way only the kernels' fp32 accumulation is left.  Every bound sits at least 4x
above the error measured on a B200 (noted beside it) and well below the 1e-4 that a 3xTF32 route which lost one of its
three products would still meet on some quantities (bf16: a wrong instruction descriptor, operand layout or rounding
shows up as errors of 1e-3 and more); the exception is an fp32 sum that one tensor-core accumulator carries over
thousands of rows (LONG_TOL).
"""
import pytest
import torch

from classifier_bf16_oracle import bilinear_bf16
from oracle import classifier_oracle as CO
from gcgcn_b200 import _lib
from gcgcn_b200 import classifier as C
from gcgcn_b200.batch import RaggedBatch

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
D = 128
ERR_INVALID_ARG, ERR_WORKSPACE = -1, -4
F32, BF16 = torch.float32, torch.bfloat16
DTYPES = [pytest.param(F32, id="f32"), pytest.param(BF16, id="bf16")]
ORACLE = {F32: CO.bilinear, BF16: bilinear_bf16}
# row-dot forward, row-accumulate dh and dt, the generated-operand weight gradient; then the operand converters
KERNELS = {F32: ("gemm_tc_rowdot<A in TMEM>", "gemm_tc_rowacc<A in TMEM>", "gemm_tc_tn<presplit A>",
                 "gemm_presplit_b", "gemm_presplit_a"),
           BF16: ("gemm_tc_rowdot<bf16>", "gemm_tc_rowacc<bf16>", "gemm_tc_wgrad<bf16>")}

# max |got - ref| / max |ref| against float64 (of the rounded operands for bf16); the worst value measured over ROUTES
# on a B200 (1000 W) beside each
TOL = {F32: {"out": 6e-6,        # 1.5e-6
             "dh": 7e-6,         # 1.7e-6
             "dt": 7e-6,         # 1.7e-6
             "dW": 8e-6,         # 2.2e-6 (P 128: 3.6x below)
             "dbias": 1.2e-6},   # 3.0e-7
       BF16: {"out": 1.2e-6,     # 2.5e-7
              "dh": 2.5e-6,      # 5.9e-7 (P 532481)
              "dt": 3e-6,        # 6.9e-7 (P 8193, R 150)
              "dW": 2.5e-5,      # 5.4e-6 (P 4096: one 4096-row accumulation); 2.8e-7 below 128 rows
              "dbias": 1.2e-6}}  # 3.0e-7
# One fp32 tensor-core accumulator fed by thousands of rows comes out small by about 2.5e-5 per 4096 rows (its fp32 adds
# truncate, DESIGN.md section 4a).  dW' takes one accumulator per min(P, 4096)-row range, so from a few hundred pairs on
# that drift outgrows TOL's margin.  Measured: dW' 2.7e-5 to 3.9e-5 at every P from 4095 to 532481 (3.1e-5 at 4095,
# 3.0e-5 at 532481).  Four times that would pass 1e-4, so these keep DESIGN.md section 2's 1e-4.
LONG_TOL = 1e-4


def tol(dtype, k, P):
    return LONG_TOL if dtype == F32 and k == "dW" and P >= 256 else TOL[dtype][k]


def stream():
    return torch.cuda.current_stream(DEV).cuda_stream


def rel_err(got, ref):
    got, ref = got.double(), ref.double()
    assert got.shape == ref.shape, (got.shape, ref.shape)
    return float((got - ref).abs().max()) / max(float(ref.abs().max()), 1e-30)


def bilinear_inputs(P, R, seed):
    """h, t as pair_dense leaves them (tanh), W and bias with nn.Bilinear's init, a random upstream gradient."""
    gen = torch.Generator(device=DEV).manual_seed(seed)
    h = torch.tanh(torch.randn(P, D, generator=gen, device=DEV))
    t = torch.tanh(torch.randn(P, D, generator=gen, device=DEV))
    W = (torch.rand(R, D, D, generator=gen, device=DEV) * 2 - 1) / D ** 0.5
    bias = (torch.rand(R, generator=gen, device=DEV) * 2 - 1) / D ** 0.5
    dout = torch.randn(P, R, generator=gen, device=DEV)
    return h, t, W, bias, dout


def run_bilinear(dtype, h, t, W, bias, dout):
    """BilinearFn forward and backward; returns (out, dh, dt, dW, dbias) and {kernel: launches}."""
    leaves = [x.clone().requires_grad_(True) for x in (h, t, W, bias)]
    torch.cuda.synchronize()
    _lib.timing_begin(stream())
    out = C.BilinearFn.apply(*leaves, dtype)
    out.backward(dout)
    ran = {k: v[0] for k, v in _lib.timing_end(stream()).items()}
    torch.cuda.synchronize()
    return (out.detach(),) + tuple(x.grad for x in leaves), ran


ROUTES = ([(P, 97) for P in (1, 127, 128, 129, 4095, 4096, 4097, 8191, 8192, 8193, 12289, 270336, 532481)]
          + [(P, R) for R in (1, 2, 33, 150) for P in (127, 8193)])


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("P,R", ROUTES)
def test_bilinear_against_float64(P, R, dtype):
    """128 / 129: one row tile / two; 4096 / 4097: one 4096-row range / two, the second of one row; 8193: three ranges,
    the last of one row; 12289: four ranges and a row; 270336: two host calls (262144 + 8192); 532481: three, the last
    of one pair.  R = 1: one relation tile; R = 150: more relation tiles than SMs.  Only the kernels of dtype run."""
    h, t, W, bias, dout = bilinear_inputs(P, R, seed=P * 1000 + R)
    got, ran = run_bilinear(dtype, h, t, W, bias, dout)
    rowdot, rowacc, wgrad = KERNELS[dtype][:3]
    calls = -(-P // C.FUSED_CHUNK_PAIRS)
    assert ran.get(rowdot) == 1 and ran.get(rowacc) == 2 * calls and ran.get(wgrad) == calls, ran
    assert not [k for k in ran if k.startswith("gemm") and k not in KERNELS[dtype]], ran
    ref = ORACLE[dtype](h, t, W, bias, dout)
    errs = {k: rel_err(g, r) for k, g, r in zip(TOL[dtype], got, ref)}
    print(f"{dtype} P {P} R {R}: " + ", ".join(f"{k} {e:.2e}" for k, e in errs.items()))
    for k, e in errs.items():
        assert e <= tol(dtype, k, P), f"P {P} R {R} {k}: {e:.3e} > {tol(dtype, k, P):.1e}"


@pytest.mark.parametrize("dtype", DTYPES)
def test_bilinear_is_deterministic(dtype):
    """Fixed-order reductions, no atomics: two runs are bitwise equal."""
    args = bilinear_inputs(12289, 97, seed=7)
    a, _ = run_bilinear(dtype, *args)
    b, _ = run_bilinear(dtype, *args)
    for k, x, y in zip(TOL[dtype], a, b):
        assert torch.equal(x, y), k


# ---- the C entry points, called the way classifier.py calls them ---------------------------------------------------
def lib():
    return _lib.load()


def p(x):
    return None if x is None else x.data_ptr()


def weights(W):
    return CO.wprime(W.double()).float().contiguous(), CO.wsecond(W.double()).float().contiguous()


@pytest.mark.parametrize("dtype", DTYPES)
def test_fwd_accumulates_into_a_strided_output_without_bias(dtype):
    """accumulate = 1 into a prefilled out of row stride ldo > R, bias null: out[:, :R] += the bilinear form, columns
    R.. untouched; a workspace of exactly gcgcn_bilinear_ws_bytes suffices."""
    P, R, ldo, code = 1000, 33, 40, C.DTYPES[dtype]
    h, t, W, _, _ = bilinear_inputs(P, R, seed=11)
    Wm, _ = weights(W)
    gen = torch.Generator(device=DEV).manual_seed(12)
    out = torch.full((P, ldo), -7.25, device=DEV)
    out[:, :R] = torch.randn(P, R, generator=gen, device=DEV)
    before = out.clone()
    ws = torch.empty(int(lib().gcgcn_bilinear_ws_bytes(P, R, code)), dtype=torch.uint8, device=DEV)
    _lib.call("gcgcn_bilinear_fwd", p(h), p(t), p(Wm), None, P, R, code, 1, p(out), ldo, p(ws), ws.numel(), stream())
    torch.cuda.synchronize()
    assert torch.equal(out[:, R:], before[:, R:])
    e = rel_err(out[:, :R], before[:, :R].double() + ORACLE[dtype](h, t, W))
    print(f"{dtype} fwd accumulate: {e:.2e}")
    assert e <= TOL[dtype]["out"]                                           # fp32 1.2e-6, bf16 1.8e-7


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("P", [100, 8193])
@pytest.mark.parametrize("beta", [0.0, 1.0])
def test_fused_bwd_beta(beta, P, dtype):
    """beta = 0 overwrites dWm (NaN before: never read), beta = 1 adds to it; dh and dt are written whole.  P = 100: one
    4096-row range (the epilogue applies beta); 8193: three (the split-K reduction does)."""
    R, code = 33, C.DTYPES[dtype]
    h, t, W, _, dout = bilinear_inputs(P, R, seed=21 + P)
    Wm, Wm2 = weights(W)
    gen = torch.Generator(device=DEV).manual_seed(22)
    prior = torch.randn(D, R * D, generator=gen, device=DEV) if beta else torch.full((D, R * D), float("nan"), device=DEV)
    dWm = prior.clone()
    dh = torch.full_like(h, float("nan"))
    dt = torch.full_like(t, float("nan"))
    ws = torch.empty(int(lib().gcgcn_bilinear_bwd_ws_bytes(P, R, code)), dtype=torch.uint8, device=DEV)
    _lib.call("gcgcn_bilinear_bwd", p(h), p(t), p(Wm), p(Wm2), p(dout), P, R, code, beta, p(dh), p(dt), p(dWm), p(ws),
              ws.numel(), stream())
    torch.cuda.synchronize()
    _, rdh, rdt, rdW, _ = ORACLE[dtype](h, t, W, None, dout)
    want = CO.wprime(rdW) + (prior.double() if beta else 0.0)
    errs = {"dh": rel_err(dh, rdh), "dt": rel_err(dt, rdt), "dW": rel_err(dWm, want)}
    print(f"{dtype} bwd P {P} beta {beta}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    for k, e in errs.items():                                               # fp32 P 8193: dh 1.4e-6, dt 1.3e-6, dW' 3.3e-5
        assert e <= tol(dtype, k, P), f"{k}: {e:.3e} > {tol(dtype, k, P):.1e}"


@pytest.mark.parametrize("dtype", DTYPES)
def test_zero_rows_launch_nothing(dtype):
    R, code = 97, C.DTYPES[dtype]
    h, t, W, bias, dout = bilinear_inputs(4, R, seed=31)
    Wm, Wm2 = weights(W)
    out = torch.full((4, R), 3.0, device=DEV)
    dh, dt, dWm = torch.full_like(h, 3.0), torch.full_like(t, 3.0), torch.full((D, R * D), 3.0, device=DEV)
    ws = torch.empty(4096, dtype=torch.uint8, device=DEV)
    before = _lib.launch_count()
    assert lib().gcgcn_bilinear_fwd(p(h), p(t), p(Wm), p(bias), 0, R, code, 0, p(out), R, p(ws), ws.numel(), stream()) == 0
    assert lib().gcgcn_bilinear_bwd(p(h), p(t), p(Wm), p(Wm2), p(dout), 0, R, code, 0.0, p(dh), p(dt), p(dWm), p(ws),
                                    ws.numel(), stream()) == 0
    assert _lib.launch_count() == before
    torch.cuda.synchronize()
    assert bool((out == 3).all() and (dh == 3).all() and (dt == 3).all() and (dWm == 3).all())
    # and through the autograd function: an empty forward and backward
    leaves = [x[:0].clone().requires_grad_(True) for x in (h, t)] + [W.clone().requires_grad_(True),
                                                                     bias.clone().requires_grad_(True)]
    z = C.BilinearFn.apply(*leaves, dtype)
    z.backward(torch.zeros_like(z))
    assert z.shape == (0, R) and not leaves[2].grad.any() and not leaves[3].grad.any()


def call_entry(which, code, ws_bytes, P=8192, R=97):
    """One call of gcgcn_bilinear_fwd or _bwd on zeroed outputs; returns (rc, launches, whether an output was written)."""
    h, t, W, bias, dout = bilinear_inputs(P, R, seed=51)
    Wm, Wm2 = weights(W)
    out = torch.zeros(P, R, device=DEV)
    dh, dt, dWm = torch.zeros_like(h), torch.zeros_like(t), torch.zeros(D, R * D, device=DEV)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=DEV)
    before = _lib.launch_count()
    if which == "fwd":
        rc = lib().gcgcn_bilinear_fwd(p(h), p(t), p(Wm), p(bias), P, R, code, 0, p(out), R, p(ws), ws_bytes, stream())
    else:
        rc = lib().gcgcn_bilinear_bwd(p(h), p(t), p(Wm), p(Wm2), p(dout), P, R, code, 0.0, p(dh), p(dt), p(dWm), p(ws),
                                      ws_bytes, stream())
    launches = _lib.launch_count() - before
    torch.cuda.synchronize()
    return rc, launches, bool(out.any() or dh.any() or dt.any() or dWm.any())


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("which", ["fwd", "bwd"])
def test_workspace_one_byte_short_is_refused_before_any_launch(which, dtype):
    P, R, code = 8192, 97, C.DTYPES[dtype]
    need = int(lib().gcgcn_bilinear_ws_bytes(P, R, code) if which == "fwd" else lib().gcgcn_bilinear_bwd_ws_bytes(P, R, code))
    rc, launches, written = call_entry(which, code, need - 1, P, R)
    assert rc == ERR_WORKSPACE, (rc, lib().gcgcn_last_error())
    assert launches == 0 and not written


@pytest.mark.parametrize("which", ["fwd", "bwd"])
def test_unknown_dtype_is_refused_before_any_launch(which):
    """Only GCGCN_F32 (0) and GCGCN_BF16 (1) name an operand type; a workspace ample for either does not matter."""
    P, R = 8192, 97
    need = max(int(f(P, R, code)) for f in (lib().gcgcn_bilinear_ws_bytes, lib().gcgcn_bilinear_bwd_ws_bytes)
               for code in C.DTYPES.values())
    for code in (2, -1):
        rc, launches, written = call_entry(which, code, need, P, R)
        assert rc == ERR_INVALID_ARG and b"dtype" in lib().gcgcn_last_error(), (rc, lib().gcgcn_last_error())
        assert launches == 0 and not written


# ---- the loss and the per-document bias on a ragged batch ----------------------------------------------------------
SIZES = [1, 2, 42, 3, 256]                     # 1 + 4 + 1764 + 9 + 65536 pairs


def doc_slices():
    lo = 0
    for n in SIZES:
        yield n, slice(lo, lo + n * n)
        lo += n * n


@pytest.mark.parametrize("R", [97, 1])
def test_pair_bce_against_float64(R):
    """Logits with |z| <= 8, where float64 and torch's clamped fp32 BCE agree: the fp32 sigmoid that torch's arithmetic
    takes the log of rounds 1 - p to about 6e-8 / (1 - p) of itself, 2e-4 of the BCE at z = 8; loss and dz per
    document."""
    bt = RaggedBatch(SIZES, DEV)
    gen = torch.Generator(device=DEV).manual_seed(60 + R)
    z = (torch.randn(bt.total_pairs, R, generator=gen, device=DEV) * 3).clamp(-8.0, 8.0)
    y = (torch.rand(bt.total_pairs, R, generator=gen, device=DEV) < 0.1).float()
    dloss = torch.randn(bt.num_docs, generator=gen, device=DEV)
    zg = z.clone().requires_grad_(True)
    loss = C.pair_bce_loss(zg, y, bt)
    (loss * dloss).sum().backward()
    torch.cuda.synchronize()
    rloss, rdz = CO.pair_bce(z, y, SIZES, dloss)
    assert loss[0] == 0 and not zg.grad[0].any()
    e_loss = float(((loss.detach().double() - rloss).abs() / rloss.abs().clamp_min(1e-30))[1:].max())
    e_dz = max(rel_err(zg.grad[s], rdz[s]) for n, s in doc_slices() if n > 1)
    print(f"pair_bce R {R}: loss {e_loss:.2e}, dz {e_dz:.2e}")
    assert e_loss <= 3e-6 and e_dz <= 1e-6                                  # R 97: 7.1e-7, 2.4e-7; R 1: 4.9e-7, 1.9e-7


def test_pair_bce_saturated_against_torch_fp32():
    """Saturated logits: torch's fp32 clamp of the logs at -100 decides the value, so the reference is torch's own BCE."""
    import torch.nn.functional as F
    R = 97
    bt = RaggedBatch(SIZES, DEV)
    gen = torch.Generator(device=DEV).manual_seed(70)
    z = torch.randn(bt.total_pairs, R, generator=gen, device=DEV) * 6
    sat = torch.tensor([40.0, -40.0, 120.0, -120.0, 17.0, -17.0], device=DEV)
    pick = torch.rand(bt.total_pairs, R, generator=gen, device=DEV) < 0.05
    z[pick] = sat[torch.randint(0, 6, (int(pick.sum()),), generator=gen, device=DEV)]
    y = (torch.rand(bt.total_pairs, R, generator=gen, device=DEV) < 0.1).float()
    dloss = torch.randn(bt.num_docs, generator=gen, device=DEV)
    zg = z.clone().requires_grad_(True)
    loss = C.pair_bce_loss(zg, y, bt)
    (loss * dloss).sum().backward()
    zt = z.clone().requires_grad_(True)
    want = []
    for n, s in doc_slices():
        per = F.binary_cross_entropy(torch.sigmoid(zt[s].view(n, n, R)), y[s].view(n, n, R), reduction="none").mean(-1)
        off = ~torch.eye(n, dtype=torch.bool, device=DEV)
        want.append(per[off].sum() / (n * n - n) if n > 1 else per.sum() * 0)
    want = torch.stack(want)
    (want * dloss).sum().backward()
    torch.cuda.synchronize()
    e_loss = float((loss.detach() - want.detach()).abs().max())
    e_dz = float((zg.grad - zt.grad).abs().max())
    print(f"pair_bce saturated: loss {e_loss:.2e}, dz {e_dz:.2e}")
    assert e_loss <= 4e-6 and e_dz <= 4e-9                                  # 9.5e-7, 9.3e-10 (absolute)


@pytest.mark.parametrize("R", [97, 1])
def test_doc_bias_against_float64(R):
    """Forward bit-exact against an fp32 add; backward (a sequential fp32 sum of up to 65 536 pairs) against float64."""
    bt = RaggedBatch(SIZES, DEV)
    gen = torch.Generator(device=DEV).manual_seed(80 + R)
    z = torch.randn(bt.total_pairs, R, generator=gen, device=DEV)
    v = torch.randn(bt.num_docs, R, generator=gen, device=DEV)
    dz = torch.randn(bt.total_pairs, R, generator=gen, device=DEV)
    vg = v.clone().requires_grad_(True)
    out = C.DocBiasFn.apply(z, vg, bt)
    out.backward(dz)
    torch.cuda.synchronize()
    counts = torch.tensor([n * n for n in SIZES], device=DEV)
    assert torch.equal(out.detach(), z + v.repeat_interleave(counts, dim=0))
    ref = CO.doc_bias_bwd(dz, SIZES)
    assert torch.equal(vg.grad[0], dz[0])                                   # one pair: the sum is the value
    # error per (document, relation) over the root sum of squares of its terms: a sum of random signs may be near zero
    scale = torch.stack([dz[s].double().pow(2).sum(0).sqrt() for _, s in doc_slices()])
    e = float(((vg.grad.double() - ref).abs() / scale).max())
    print(f"doc_bias_bwd R {R}: {e:.2e}")
    assert e <= 8e-5                                                        # R 97: 1.8e-5, R 1: 2.3e-6
