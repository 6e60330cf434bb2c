"""-m gpu: the bilinear form on bf16 operands (gcgcn_bilinear_bf16_fwd / _bwd, classifier.BilinearBf16Fn,
relation_logits(dtype=torch.bfloat16), GraphHead(classifier_dtype=torch.bfloat16)).

Against float64 of the rounded operands (tests/classifier_bf16_oracle.py) the only error left is the kernels' fp32
accumulation, so the bounds sit at the scale of the fp32 route's own float64 tests (test_gpu_classifier_fp64.py), each
at least 4x above the error measured on a B200 (noted beside it): a wrong instruction descriptor, operand layout or
rounding shows up as errors of 1e-3 and more.  Against the fp32 route the difference is the bf16 rounding itself, and
the bound is relative (max |difference| / max |fp32 value|).

P runs on both sides of every boundary of the kernels: 128-pair row tiles, 4096-row ranges of the weight gradient (one
range: the epilogue applies beta; several: split-K partials and the fp32 reduction), and the host calls of
FUSED_CHUNK_PAIRS pairs; R from one relation to more relation tiles than the B200's 148 SMs.
"""
import pytest
import torch

from classifier_bf16_oracle import bilinear_bf16
from oracle import classifier_oracle as CO
from gcgcn_b200 import _lib
from gcgcn_b200 import classifier as C
from gcgcn_b200 import synthetic as S
from gcgcn_b200.head import GraphHead, HeadBatch
from gcgcn_b200.sharding import FlatTrainer

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
D = 128
ERR_WORKSPACE = -4
ROWDOT, ROWACC, WGRAD = "gemm_tc_rowdot<bf16>", "gemm_tc_rowacc<bf16>", "gemm_tc_wgrad<bf16>"
FP32_ROUTE = ("gemm_tc_rowdot<A in TMEM>", "gemm_tc_rowacc<A in TMEM>", "gemm_tc_tn<presplit A>", "gemm_presplit_b",
              "gemm_presplit_a", "bilinear_reduce", "bilinear_outer", "bilinear_dt")

# max |got - ref| / max |ref| against float64 of the rounded operands; the worst value measured on a B200 beside each
TOL = {"out": 1.2e-6,       # 2.5e-7
       "dh": 2.5e-6,        # 5.9e-7 (P 532481)
       "dt": 3e-6,          # 6.9e-7 (P 8193, R 150)
       "dW": 2.5e-5,        # 5.4e-6 (P 4096: one 4096-row accumulation); 2.8e-7 below 128 rows
       "dbias": 1.2e-6}     # 3.0e-7
# relative bound against the fp32 route (the bf16 rounding of the operands)
VS_FP32 = 2e-2


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
    """BilinearBf16Fn forward and backward; returns (out, dh, dt, dW, dbias) and {kernel: launches}."""
    leaves = [x.clone().requires_grad_(True) for x in (h, t, W, bias)]
    torch.cuda.synchronize()
    _lib.timing_begin(stream())
    out = C.BilinearBf16Fn.apply(*leaves)
    out.backward(dout)
    ran = {k: v[0] for k, v in _lib.timing_end(stream()).items()}
    torch.cuda.synchronize()
    return (out.detach(),) + tuple(x.grad for x in leaves), ran


ROUTES = ([(P, 97) for P in (1, 127, 128, 129, 4095, 4096, 4097, 8191, 8192, 270336, 532481)]
          + [(P, R) for R in (1, 2, 33, 150) for P in (127, 8193)])


@pytest.mark.parametrize("P,R", ROUTES)
def test_bilinear_bf16_against_float64(P, R):
    """4096 / 4097: one range / two, the second of one row; 270336: two host calls (262144 + 8192); 532481: three, the
    last of one pair.  Only the bf16 kernels run."""
    h, t, W, bias, dout = bilinear_inputs(P, R, seed=P * 1000 + R)
    got, ran = run_bilinear(h, t, W, bias, dout)
    calls = -(-P // C.FUSED_CHUNK_PAIRS)
    assert ran.get(ROWDOT) == 1 and ran.get(ROWACC) == 2 * calls and ran.get(WGRAD) == calls, ran
    assert not [k for k in ran if k in FP32_ROUTE or (k.startswith("gemm") and "<bf16>" not in k)], ran
    ref = bilinear_bf16(h, t, W, bias, dout)
    errs = {k: rel_err(g, r) for k, g, r in zip(TOL, got, ref)}
    print(f"P {P} R {R}: " + ", ".join(f"{k} {e:.2e}" for k, e in errs.items()))
    for k, e in errs.items():
        assert e <= TOL[k], f"P {P} R {R} {k}: {e:.3e} > {TOL[k]:.1e}"


def test_bilinear_bf16_is_deterministic():
    """Fixed-order reductions, no atomics: two runs are bitwise equal."""
    args = bilinear_inputs(12289, 97, seed=7)
    a, _ = run_bilinear(*args)
    b, _ = run_bilinear(*args)
    for k, x, y in zip(TOL, a, b):
        assert torch.equal(x, y), k


# ---- the C entry points ---------------------------------------------------------------------------------------------
def lib():
    return _lib.load()


def p(x):
    return None if x is None else x.data_ptr()


def weights(W):
    return CO.wprime(W.double()).float().contiguous(), CO.wsecond(W.double()).float().contiguous()


def test_fwd_accumulates_into_a_strided_output_without_bias():
    """accumulate = 1 into a prefilled out of row stride ldo > R, bias null: out[:, :R] += the bilinear form, columns
    R.. untouched; a workspace of exactly gcgcn_bilinear_bf16_ws_bytes suffices."""
    P, R, ldo = 1000, 33, 40
    h, t, W, _, _ = bilinear_inputs(P, R, seed=11)
    Wm, _ = weights(W)
    gen = torch.Generator(device=DEV).manual_seed(12)
    out = torch.full((P, ldo), -7.25, device=DEV)
    out[:, :R] = torch.randn(P, R, generator=gen, device=DEV)
    before = out.clone()
    ws = torch.empty(int(lib().gcgcn_bilinear_bf16_ws_bytes(P, R)), dtype=torch.uint8, device=DEV)
    _lib.call("gcgcn_bilinear_bf16_fwd", p(h), p(t), p(Wm), None, P, R, 1, p(out), ldo, p(ws), ws.numel(), stream())
    torch.cuda.synchronize()
    assert torch.equal(out[:, R:], before[:, R:])
    e = rel_err(out[:, :R], before[:, :R].double() + bilinear_bf16(h, t, W))
    print(f"fwd accumulate: {e:.2e}")
    assert e <= TOL["out"]                                                  # 1.8e-7


@pytest.mark.parametrize("P", [100, 8193])
@pytest.mark.parametrize("beta", [0.0, 1.0])
def test_bwd_beta(P, beta):
    """beta = 0 overwrites dWm (NaN before: never read), beta = 1 adds to it; dh and dt are written whole.  P = 100: one
    4096-row range (the epilogue applies beta); 8193: three (the split-K reduction does)."""
    R = 33
    h, t, W, _, dout = bilinear_inputs(P, R, seed=21 + P)
    Wm, Wm2 = weights(W)
    gen = torch.Generator(device=DEV).manual_seed(22)
    prior = torch.randn(D, R * D, generator=gen, device=DEV) if beta else torch.full((D, R * D), float("nan"), device=DEV)
    dWm = prior.clone()
    dh = torch.full_like(h, float("nan"))
    dt = torch.full_like(t, float("nan"))
    ws = torch.empty(int(lib().gcgcn_bilinear_bf16_bwd_ws_bytes(P, R)), dtype=torch.uint8, device=DEV)
    _lib.call("gcgcn_bilinear_bf16_bwd", p(h), p(t), p(Wm), p(Wm2), p(dout), P, R, beta, p(dh), p(dt), p(dWm), p(ws),
              ws.numel(), stream())
    torch.cuda.synchronize()
    _, rdh, rdt, rdW, _ = bilinear_bf16(h, t, W, None, dout)
    want = CO.wprime(rdW) + (prior.double() if beta else 0.0)
    errs = {"dh": rel_err(dh, rdh), "dt": rel_err(dt, rdt), "dW": rel_err(dWm, want)}
    print(f"bwd P {P} beta {beta}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    for k, e in errs.items():
        assert e <= TOL[k], f"{k}: {e:.3e} > {TOL[k]:.1e}"


def test_zero_rows_launch_nothing():
    R = 97
    h, t, W, bias, dout = bilinear_inputs(4, R, seed=31)
    Wm, Wm2 = weights(W)
    out = torch.full((4, R), 3.0, device=DEV)
    dh, dt, dWm = torch.full_like(h, 3.0), torch.full_like(t, 3.0), torch.full((D, R * D), 3.0, device=DEV)
    ws = torch.empty(4096, dtype=torch.uint8, device=DEV)
    before = _lib.launch_count()
    assert lib().gcgcn_bilinear_bf16_fwd(p(h), p(t), p(Wm), p(bias), 0, R, 0, p(out), R, p(ws), ws.numel(), stream()) == 0
    assert lib().gcgcn_bilinear_bf16_bwd(p(h), p(t), p(Wm), p(Wm2), p(dout), 0, R, 0.0, p(dh), p(dt), p(dWm), p(ws),
                                         ws.numel(), stream()) == 0
    assert _lib.launch_count() == before
    torch.cuda.synchronize()
    assert bool((out == 3).all() and (dh == 3).all() and (dt == 3).all() and (dWm == 3).all())
    # and through the autograd function: an empty forward and backward
    leaves = [x[:0].clone().requires_grad_(True) for x in (h, t)] + [W.clone().requires_grad_(True),
                                                                     bias.clone().requires_grad_(True)]
    z = C.BilinearBf16Fn.apply(*leaves)
    z.backward(torch.zeros_like(z))
    assert z.shape == (0, R) and not leaves[2].grad.any() and not leaves[3].grad.any()


@pytest.mark.parametrize("which", ["fwd", "bwd"])
def test_workspace_one_byte_short_is_refused_before_any_launch(which):
    P, R = 8192, 97
    h, t, W, bias, dout = bilinear_inputs(P, R, seed=51)
    Wm, Wm2 = weights(W)
    out = torch.zeros(P, R, device=DEV)
    dh, dt, dWm = torch.zeros_like(h), torch.zeros_like(t), torch.zeros(D, R * D, device=DEV)
    need = int(lib().gcgcn_bilinear_bf16_ws_bytes(P, R) if which == "fwd" else lib().gcgcn_bilinear_bf16_bwd_ws_bytes(P, R))
    ws = torch.empty(need, dtype=torch.uint8, device=DEV)
    before = _lib.launch_count()
    if which == "fwd":
        rc = lib().gcgcn_bilinear_bf16_fwd(p(h), p(t), p(Wm), p(bias), P, R, 0, p(out), R, p(ws), need - 1, stream())
    else:
        rc = lib().gcgcn_bilinear_bf16_bwd(p(h), p(t), p(Wm), p(Wm2), p(dout), P, R, 0.0, p(dh), p(dt), p(dWm), p(ws),
                                           need - 1, stream())
    assert rc == ERR_WORKSPACE, (rc, lib().gcgcn_last_error())
    assert _lib.launch_count() == before
    torch.cuda.synchronize()
    assert not out.any() and not dh.any() and not dt.any() and not dWm.any()


# ---- against the fp32 route -----------------------------------------------------------------------------------------
def test_relation_logits_bf16_against_fp32():
    """relation_logits in both dtypes on the bench's 12-document batch x 16 (99 312 pairs): logits and the gradients of
    h, t and of every classifier parameter within VS_FP32 of the fp32 route.  The argmax agreement is reported, not
    gated: the bf16 rounding moves near-ties."""
    P, R = 99312, 97
    torch.manual_seed(3)
    bili, cls = torch.nn.Bilinear(D, D, R).to(DEV), torch.nn.Linear(2 * D, R).to(DEV)
    gen = torch.Generator(device=DEV).manual_seed(4)
    h = torch.tanh(torch.randn(P, D, generator=gen, device=DEV))
    t = torch.tanh(torch.randn(P, D, generator=gen, device=DEV))
    up = torch.randn(P, R, generator=gen, device=DEV)
    res = {}
    for dt in (torch.float32, torch.bfloat16):
        hh, tt = h.clone().requires_grad_(True), t.clone().requires_grad_(True)
        z = C.relation_logits(hh, tt, bili, cls, dtype=dt)
        params = [hh, tt] + list(bili.parameters()) + list(cls.parameters())
        res[dt] = [z.detach()] + list(torch.autograd.grad(z, params, up))
    names = ["logits", "dh", "dt", "dW", "dbias", "dcls.weight", "dcls.bias"]
    errs = {k: rel_err(b, a) for k, a, b in zip(names, res[torch.float32], res[torch.bfloat16])}
    agree = float((res[torch.float32][0].argmax(1) == res[torch.bfloat16][0].argmax(1)).float().mean())
    print("bf16 vs fp32: " + ", ".join(f"{k} {e:.2e}" for k, e in errs.items()) + f"; argmax agreement {agree:.4%}")
    # measured: logits 2.0e-3, dh 2.4e-3, dt 2.2e-3, dW 2.2e-3, the fp32 linear layer's gradients 0; argmax 99.72 %
    for k, e in errs.items():
        assert e <= VS_FP32, f"{k}: {e:.3e} > {VS_FP32}"


def head_inputs(seed=0):
    docs = S.make_batch()                                    # 12 ragged documents
    hb = HeadBatch([S.make_wire(d) for d in docs], DEV)
    gen = torch.Generator(device=DEV).manual_seed(seed)
    ctx = torch.tanh(torch.randn(hb.total_tokens, D, generator=gen, device=DEV))
    labels = (torch.rand(hb.batch.total_pairs, 97, generator=gen, device=DEV) < 0.02).float()
    return hb, ctx, labels


def run_head(head, hb, ctx, labels, **kw):
    c = ctx.clone().requires_grad_(True)
    head.zero_grad(set_to_none=True)
    torch.cuda.synchronize()
    _lib.timing_begin(stream())
    out = head(c, hb, labels=labels, **kw)
    out["loss"].sum().backward()
    ran = {k: v[0] for k, v in _lib.timing_end(stream()).items()}
    torch.cuda.synchronize()
    grads = {k: p.grad.detach().clone() for k, p in head.named_parameters() if p.grad is not None}
    return out["logits"].detach(), out["loss"].detach(), c.grad, grads, ran


def compare_heads(a, b, what):
    """rel_err of logits, loss, d context and every parameter gradient of run b against run a.  The biases and weights in
    front of a softmax over one element (attention_all etc. on short documents, the weighted-adjacency linears) have a
    gradient of exactly zero in exact arithmetic: both runs give rounding residue there, and only its size is checked."""
    (z32, l32, dc32, g32, _), (z16, l16, dc16, g16, _) = a, b
    assert sorted(g16) == sorted(g32)
    errs = {"logits": rel_err(z16, z32), "loss": rel_err(l16, l32), "dcontext": rel_err(dc16, dc32)}
    gmax = max(float(g.abs().max()) for g in g32.values())
    zero = [k for k in g32 if float(g32[k].abs().max()) <= 1e-5 * gmax]
    for k in zero:
        assert float(g16[k].abs().max()) <= 1e-4 * gmax, (k, float(g16[k].abs().max()), gmax)
    errs.update({k: rel_err(g16[k], g32[k]) for k in g32 if k not in zero})
    worst = sorted(errs.items(), key=lambda kv: -kv[1])[:6]
    print(f"{what} ({len(zero)} zero gradients), worst: " + ", ".join(f"{k} {e:.2e}" for k, e in worst))
    return errs


def test_graph_head_bf16_classifier_against_fp32():
    """GraphHead with the bf16 classifier on one ragged batch.  Against the fp32 classifier, both on bf16 edges: logits,
    the loss and the gradients of context and of every parameter within VS_FP32.  Against the all-fp32 head (bf16 edges
    as well): logits, loss, d context and the classifier's gradients within VS_FP32 -- two small, cancelling gradients
    of the edge-feature producer move by more than that with the bf16 edge storage alone (measured 6.1e-2 and 4.7e-2),
    which this comparison reports but does not gate.  The default call runs the fp32 kernels only; one FlatTrainer step
    on the bf16 head."""
    torch.manual_seed(0)
    head = GraphHead().to(DEV).eval()
    hb, ctx, labels = head_inputs()
    fp32 = run_head(head, hb, ctx, labels)
    ran32 = fp32[4]
    assert ran32.get("gemm_tc_rowdot<A in TMEM>") == 1 and not [k for k in ran32 if "bf16" in k], ran32
    edges16 = run_head(head, hb, ctx, labels, edge_dtype=torch.bfloat16)
    both16 = run_head(head, hb, ctx, labels, edge_dtype=torch.bfloat16, classifier_dtype=torch.bfloat16)
    ran16 = both16[4]
    assert ran16.get(ROWDOT) == 1 and ran16.get(WGRAD) == 1 and not [k for k in ran16 if k in FP32_ROUTE[:3]], ran16
    errs = compare_heads(edges16, both16, "bf16 classifier vs fp32 classifier, bf16 edges")
    for k, e in errs.items():
        assert e <= VS_FP32, f"{k}: {e:.3e} > {VS_FP32}"
    errs = compare_heads(fp32, both16, "all bf16 vs all fp32")
    for k, e in errs.items():
        if k in ("logits", "loss", "dcontext") or k.startswith(("bili_layer_01.", "classification_layer_01.")):
            assert e <= VS_FP32, f"{k}: {e:.3e} > {VS_FP32}"
    # parameters and gradients stay fp32: the flat trainer steps the bf16-classifier head unchanged
    tr = FlatTrainer(head, lr=1e-3)
    before = tr.flat_params.clone()
    tr.zero_grad()
    c = ctx.clone().requires_grad_(True)
    head(c, hb, labels=labels, edge_dtype=torch.bfloat16, classifier_dtype=torch.bfloat16)["loss"].sum().backward()
    tr.step()
    torch.cuda.synchronize()
    assert torch.isfinite(tr.flat_params).all() and not torch.equal(tr.flat_params, before)
    assert head.bili_layer_01.weight.dtype == torch.float32 and head.bili_layer_01.weight.grad.dtype == torch.float32


def test_graph_head_refuses_other_classifier_dtypes():
    head = GraphHead().to(DEV).eval()
    hb, ctx, _ = head_inputs()
    with pytest.raises(_lib.GcgcnError, match="classifier_dtype"):
        head(ctx, hb, classifier_dtype=torch.float16)
