"""-m gpu: the relation classifier and the trainer's loss against the float64 oracle (oracle/classifier_oracle.py) on
every route.

The bilinear form runs on three tensor-core modes of gemm_tc.cu: the row-dot epilogue (forward), the row-accumulate
epilogue (dh, dt) and the weight-gradient GEMM whose [pairs, R*128] operand its producers generate from t and dout,
split-K over 4096-row ranges with an fp32 reduction (dW').  BilinearFn takes that fused backward from 8192 pairs on,
in host calls of up to 262144 pairs that accumulate dW' through beta = 1; below 8192 pairs it materialises h W' chunk
by chunk.  The cases below put P on both sides of every one of those boundaries and R from 1 to past the 148 SMs of a
B200, call the C entry points with the strides, accumulation and beta the header documents, and run the loss and the
per-document bias on a ragged batch with a document of 65 536 pairs.

Every bound sits at least 4x above the error measured on a B200 (noted beside it) and well below the 1e-4 that a
3xTF32 route which lost one of its three products would still meet on some quantities; the exception is a sum that one
tensor-core accumulator carries over thousands of rows (LONG_TOL).
"""
import pytest
import torch

from oracle import classifier_oracle as CO
from gcgcn_b200 import _lib
from gcgcn_b200 import classifier as C
from gcgcn_b200.batch import RaggedBatch

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
D = 128
ERR_UNSUPPORTED, ERR_WORKSPACE = -2, -4
FUSED_WGRAD = "gemm_tc_tn<presplit A>"           # the generated-operand weight-gradient GEMM, once per fused host call
ROWDOT = "gemm_tc_rowdot<A in TMEM>"

# max |got - ref| / max |ref| against float64; the worst value measured over ROUTES on a B200 (1000 W) beside each
TOL = {"out": 6e-6,        # 1.5e-6
       "dh": 2e-5,         # 4.4e-6 (P 127, R 150: chunked, 512-row split-K ranges); fused 1.7e-6
       "dt": 7e-6,         # 1.7e-6
       "dW": 8e-6,         # 1.8e-6 (P 127)
       "dbias": 1.2e-6}    # 2.9e-7
# One tensor-core accumulator fed by thousands of rows comes out small by about 2.5e-5 per 4096 rows (its fp32 adds
# truncate, DESIGN.md section 4a).  Measured: dW' of the fused backward (4096-row ranges) 2.7e-5 to 3.9e-5 at every P
# from 8192 to 532481 (3.0e-5 at 532481), and dh, dW' of the chunked backward at P = 8191 (accumulators of 6208 and
# 8191 rows) 5.5e-5 and 6.9e-5.  Four times that would pass 1e-4, so these keep DESIGN.md section 2's 1e-4.
LONG_TOL = 1e-4


def tol(k, P):
    long_sum = (k == "dW" and P >= 4096) or (k == "dh" and 4096 <= P < C.FUSED_MIN_PAIRS)
    return LONG_TOL if long_sum else TOL[k]


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


def run_bilinear(h, t, W, bias, dout):
    """BilinearFn forward and backward; returns (out, dh, dt, dW, dbias) and {kernel: launches}."""
    leaves = [x.clone().requires_grad_(True) for x in (h, t, W, bias)]
    torch.cuda.synchronize()
    _lib.timing_begin(stream())
    out = C.BilinearFn.apply(*leaves)
    out.backward(dout)
    ran = {k: v[0] for k, v in _lib.timing_end(stream()).items()}
    torch.cuda.synchronize()
    return (out.detach(),) + tuple(x.grad for x in leaves), ran


def fused_calls(P):
    """Host calls of the fused backward that BilinearFn makes for P pairs."""
    calls, rest = 0, P
    while rest >= C.FUSED_MIN_PAIRS:
        rest -= rest if rest <= C.FUSED_CHUNK_PAIRS + C.FUSED_MIN_PAIRS else C.FUSED_CHUNK_PAIRS
        calls += 1
    return calls


ROUTES = ([(P, 97) for P in (1, 127, 8191, 8192, 8193, 12289, 270336, 532481)]
          + [(P, R) for R in (1, 2, 33, 150) for P in (127, 8193)])


@pytest.mark.parametrize("P,R", ROUTES)
def test_bilinear_against_float64(P, R):
    """P = 1, 127, 8191: chunked backward; 8192: the fused minimum, two whole 4096-row ranges; 8193: three ranges, the
    last of one row; 12289: four ranges and a row; 270336: the largest single fused call; 532481: three calls of
    262144, 262144 and 8193 pairs.  R = 1: one relation tile; R = 150: more relation tiles than SMs."""
    h, t, W, bias, dout = bilinear_inputs(P, R, seed=P * 1000 + R)
    got, ran = run_bilinear(h, t, W, bias, dout)
    assert ran.get(ROWDOT) == 1, ran
    assert ran.get(FUSED_WGRAD, 0) == fused_calls(P), ran
    assert fused_calls(P) == {8192: 1, 8193: 1, 12289: 1, 270336: 1, 532481: 3}.get(P, 0)
    ref = CO.bilinear(h, t, W, bias, dout)
    errs = {k: rel_err(g, r) for k, g, r in zip(TOL, got, ref)}
    print(f"P {P} R {R}: " + ", ".join(f"{k} {e:.2e}" for k, e in errs.items()))
    for k, e in errs.items():
        assert e <= tol(k, P), f"P {P} R {R} {k}: {e:.3e} > {tol(k, P):.1e}"


def test_bilinear_is_deterministic():
    """Fixed-order reductions, no atomics: two runs are bitwise equal."""
    args = bilinear_inputs(12289, 97, seed=7)
    a, _ = run_bilinear(*args)
    b, _ = run_bilinear(*args)
    for k, x, y in zip(TOL, a, b):
        assert torch.equal(x, y), k


# ---- the C entry points, called the way classifier.py calls them ---------------------------------------------------
def lib():
    return _lib.load()


def p(x):
    return None if x is None else x.data_ptr()


def weights(W):
    return CO.wprime(W.double()).float().contiguous(), CO.wsecond(W.double()).float().contiguous()


def test_fwd_accumulates_into_a_strided_output_without_bias():
    """accumulate = 1 into a prefilled out of row stride ldo > R, bias null: out[:, :R] += h W t, columns R.. untouched;
    a workspace of exactly gcgcn_bilinear_ws_bytes suffices."""
    P, R, ldo = 1000, 33, 40
    h, t, W, _, _ = bilinear_inputs(P, R, seed=11)
    Wm, _ = weights(W)
    gen = torch.Generator(device=DEV).manual_seed(12)
    out = torch.full((P, ldo), -7.25, device=DEV)
    out[:, :R] = torch.randn(P, R, generator=gen, device=DEV)
    before = out.clone()
    ws = torch.empty(int(lib().gcgcn_bilinear_ws_bytes(P, R)), dtype=torch.uint8, device=DEV)
    _lib.call("gcgcn_bilinear_fwd", p(h), p(t), p(Wm), None, P, R, 1, p(out), ldo, p(ws), ws.numel(), stream())
    torch.cuda.synchronize()
    assert torch.equal(out[:, R:], before[:, R:])
    e = rel_err(out[:, :R], before[:, :R].double() + CO.bilinear(h, t, W))
    print(f"fwd accumulate: {e:.2e}")
    assert e <= TOL["out"]                                                  # 1.2e-6


@pytest.mark.parametrize("beta", [0.0, 1.0])
def test_fused_bwd_beta(beta):
    """beta = 0 overwrites dWm (NaN before: never read), beta = 1 adds to it; dh and dt are written whole."""
    P, R = 8193, 33
    h, t, W, _, dout = bilinear_inputs(P, R, seed=21)
    Wm, Wm2 = weights(W)
    gen = torch.Generator(device=DEV).manual_seed(22)
    prior = torch.randn(D, R * D, generator=gen, device=DEV) if beta else torch.full((D, R * D), float("nan"), device=DEV)
    dWm = prior.clone()
    dh = torch.full_like(h, float("nan"))
    dt = torch.full_like(t, float("nan"))
    ws = torch.empty(int(lib().gcgcn_bilinear_bwd_ws_bytes(P, R)), dtype=torch.uint8, device=DEV)
    _lib.call("gcgcn_bilinear_bwd", p(h), p(t), p(Wm), p(Wm2), p(dout), P, R, beta, p(dh), p(dt), p(dWm), p(ws),
              ws.numel(), stream())
    torch.cuda.synchronize()
    _, rdh, rdt, rdW, _ = CO.bilinear(h, t, W, None, dout)
    want = CO.wprime(rdW) + (prior.double() if beta else 0.0)
    errs = {"dh": rel_err(dh, rdh), "dt": rel_err(dt, rdt), "dW": rel_err(dWm, want)}
    print(f"bwd beta {beta}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    for k, e in errs.items():                                               # dh 1.4e-6, dt 1.3e-6, dW' 3.3e-5
        assert e <= tol(k, P), f"{k}: {e:.3e} > {tol(k, P):.1e}"


def test_chunked_kernels_with_strided_dout():
    """gcgcn_bilinear_reduce_fwd (accumulate, bias, ldo > R), gcgcn_bilinear_outer_bwd and gcgcn_bilinear_dt_bwd with
    dout of row stride ldd > R (NaN past column R: never read), R = 33 (one relation past a warp's 32)."""
    P, R, ldd, ldo = 300, 33, 37, 41
    h, t, W, bias, dout = bilinear_inputs(P, R, seed=31)
    Y = (h.double() @ CO.wprime(W.double())).float()                     # [P, R*128], the chunked route's h W'
    dpad = torch.full((P, ldd), float("nan"), device=DEV)
    dpad[:, :R] = dout
    gen = torch.Generator(device=DEV).manual_seed(32)
    out = torch.full((P, ldo), -7.25, device=DEV)
    out[:, :R] = torch.randn(P, R, generator=gen, device=DEV)
    before = out.clone()
    dY = torch.empty(P, R * D, device=DEV)
    dt = torch.full_like(t, float("nan"))
    _lib.call("gcgcn_bilinear_reduce_fwd", p(Y), p(t), p(bias), P, R, 1, p(out), ldo, stream())
    _lib.call("gcgcn_bilinear_outer_bwd", p(dpad), ldd, p(t), P, R, p(dY), stream())
    _lib.call("gcgcn_bilinear_dt_bwd", p(dpad), ldd, p(Y), P, R, p(dt), stream())
    torch.cuda.synchronize()
    Y3 = Y.double().view(P, R, D)
    assert torch.equal(out[:, R:], before[:, R:])
    e_out = rel_err(out[:, :R], before[:, :R].double() + torch.einsum("prb,pb->pr", Y3, t.double()) + bias.double())
    assert torch.equal(dY, (dout[:, :, None] * t[:, None, :]).reshape(P, R * D))        # one fp32 product each
    e_dt = rel_err(dt, torch.einsum("pr,prb->pb", dout.double(), Y3))
    print(f"reduce_fwd {e_out:.2e}, dt_bwd {e_dt:.2e}")
    assert e_out <= 5e-7 and e_dt <= 8e-7                                   # 1.0e-7, 1.9e-7


def test_bwd_below_the_fused_minimum_is_refused_before_any_launch():
    P, R = 8191, 97
    h, t, W, _, dout = bilinear_inputs(P, R, seed=41)
    Wm, Wm2 = weights(W)
    dh, dt, dWm = torch.zeros_like(h), torch.zeros_like(t), torch.zeros(D, R * D, device=DEV)
    ws = torch.empty(int(lib().gcgcn_bilinear_bwd_ws_bytes(P, R)), dtype=torch.uint8, device=DEV)
    before = _lib.launch_count()
    rc = lib().gcgcn_bilinear_bwd(p(h), p(t), p(Wm), p(Wm2), p(dout), P, R, 0.0, p(dh), p(dt), p(dWm), p(ws),
                                  ws.numel(), stream())
    assert rc == ERR_UNSUPPORTED, lib().gcgcn_last_error()
    assert _lib.launch_count() == before
    torch.cuda.synchronize()
    assert not dh.any() and not dt.any() and not dWm.any()


@pytest.mark.parametrize("which", ["fwd", "bwd"])
def test_workspace_one_byte_short_is_refused_before_any_launch(which):
    P, R = 8192, 97
    h, t, W, bias, dout = bilinear_inputs(P, R, seed=51)
    Wm, Wm2 = weights(W)
    out = torch.zeros(P, R, device=DEV)
    dh, dt, dWm = torch.zeros_like(h), torch.zeros_like(t), torch.zeros(D, R * D, device=DEV)
    need = int(lib().gcgcn_bilinear_ws_bytes(P, R) if which == "fwd" else lib().gcgcn_bilinear_bwd_ws_bytes(P, R))
    ws = torch.empty(need, dtype=torch.uint8, device=DEV)
    before = _lib.launch_count()
    if which == "fwd":
        rc = lib().gcgcn_bilinear_fwd(p(h), p(t), p(Wm), p(bias), P, R, 0, p(out), R, p(ws), need - 1, stream())
    else:
        rc = lib().gcgcn_bilinear_bwd(p(h), p(t), p(Wm), p(Wm2), p(dout), P, R, 0.0, p(dh), p(dt), p(dWm), p(ws),
                                      need - 1, stream())
    assert rc == ERR_WORKSPACE, (rc, lib().gcgcn_last_error())
    assert _lib.launch_count() == before
    torch.cuda.synchronize()
    assert not out.any() and not dh.any() and not dt.any() and not dWm.any()


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
