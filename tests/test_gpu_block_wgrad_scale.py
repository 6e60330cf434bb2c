"""-m gpu: the graph blocks' parameter gradients at split-K scale, against the oracle in float64.

Every weight-gradient product of the blocks (WnX, We, Wout, Wq and the batched dense-connect dWinner) reduces over
all node rows of the batch, and the GEMM starts to split K across CTAs at 4096 rows.  The other block tests compare
parameter gradients on batches of at most ~1300 rows; these batches have more than 8192, so the split-K weight
gradients and their reduce kernels are what is checked.  The reference is the oracle run per document on float64
state and inputs, with the upstream gradients of gpu_common.run_blocks, summed in float64; a CPU test checks that
this reference agrees with the float32 oracle.
"""
import pytest
import torch

from gpu_common import DEV, device_blocks, run_blocks
from helpers import FP32_TOL, PREFIXES, VARIANTS, blocks_state, maxdiff, oracle_blocks, sub, upstream
from oracle import gcgcn_oracle as O
from gcgcn_b200 import _lib, synthetic as S
from gcgcn_b200.functional import _stream, block_supported

MIN_ROWS = 8192
MARGIN = 2e-6       # documents with a relu pre-activation this close to 0 have ill-conditioned gradients
ZERO_GRAD = 1e-12   # largest reference entry of a gradient that is exactly zero in exact arithmetic


def oracle_grads_fp64(doc, state, layers, heads, device):
    """Parameter gradients of one document from the oracle in float64 (state, inputs and upstream gradients cast to
    double), and the smallest |relu pre-activation| of its forward pass."""
    dev = torch.device(device)
    ps = {k: v.detach().to(dev, torch.float64).requires_grad_(True) for k, v in state.items()}
    x0, e0, e1 = (t.to(dev, torch.float64).requires_grad_(True) for t in (doc.x0, doc.e0, doc.e1))
    O.RELU_MARGIN_PROBE = []
    try:
        r = O.graph_blocks(x0, e0, e1, doc.adj.to(dev, torch.float64), sub(ps, PREFIXES[0]), sub(ps, PREFIXES[1]),
                           sub(ps, PREFIXES[2]), sub(ps, PREFIXES[3]), layers, heads, 1.0, None, False)
        margin = min(O.RELU_MARGIN_PROBE)
    finally:
        O.RELU_MARGIN_PROBE = None
    dy1, dy2 = upstream(doc.doc_id, r["y1"].shape, r["y2"].shape)
    ((r["y1"] * dy1.to(dev, torch.float64)).sum() + (r["y2"] * dy2.to(dev, torch.float64)).sum()).backward()
    return margin, {k: v.grad for k, v in ps.items()}


def add_into(total, grads):
    for k, v in grads.items():
        if v is not None:
            total[k] = total[k] + v if k in total else v.clone()


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_fp64_oracle_agrees_with_fp32_oracle(variant):
    """CPU: the float64 reference really runs in double and computes what the float32 oracle does."""
    layers, heads = VARIANTS[variant]
    _, state = blocks_state(layers, heads)
    checked = 0
    for i in (5, 8, 10, 11):
        d = S.make_doc(i)
        margin, g64 = oracle_grads_fp64(d, state, layers, heads, "cpu")
        if margin <= MARGIN:
            continue
        g32 = oracle_blocks(d, state, layers, heads)["dparams"]
        for k, v in g64.items():
            if v is None:
                assert g32[k] is None, k
                continue
            assert v.dtype == torch.float64 and g32[k].dtype == torch.float32, k
            assert maxdiff(v, g32[k]) <= FP32_TOL, f"d{k}: {maxdiff(v, g32[k]):.3e}"
        checked += 1
    assert checked >= 3


@pytest.mark.gpu
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_block_weight_gradients_at_split_k_scale(variant):
    layers, heads = VARIANTS[variant]
    gb, state = device_blocks(layers, heads)
    docs, ref, rows, i = [], {}, 0, 0
    while rows < MIN_ROWS:                 # well-conditioned DocRED-size documents, > 8192 node rows in all
        d = S.make_doc(i)
        i += 1
        margin, g = oracle_grads_fp64(d, state, layers, heads, DEV)
        if margin > MARGIN:
            docs.append(d)
            add_into(ref, g)
            rows += d.n
    big, big_id = None, 100000
    while big is None:                     # one 100-entity document: the whole batch leaves the block kernels
        d = S.make_doc(big_id, n=100, L=32)
        margin, g = oracle_grads_fp64(d, state, layers, heads, DEV)
        if margin > MARGIN:
            big, big_grads = d, g
        big_id += 1
    ref_big = dict(ref)
    add_into(ref_big, big_grads)

    for route, batch, want in (("block-kernels", docs, ref), ("row-tiled", docs + [big], ref_big)):
        st = _stream(DEV)
        torch.cuda.synchronize()
        _lib.timing_begin(st)
        res = run_blocks(gb, batch)
        ran = set(_lib.timing_end(st))
        bt = res["bt"]
        assert bt.total_nodes >= MIN_ROWS
        assert block_supported(bt, heads, layers, True) == (route == "block-kernels")
        assert any(n.startswith("splitk_reduce") for n in ran), sorted(ran)
        report, bad = [], []
        for k, v in res["dparams"].items():
            if v is None:                 # linears_k gets no gradient (the reference's unused key projection)
                assert k not in want, k
                continue
            r = want[k]
            scale = float(r.abs().max())
            err = float((v.double() - r).abs().max())
            # a gradient that vanishes exactly (the reference holds float64 round-off of 0, e.g. the bias of
            # linear_node_h, which the softmax over each row cancels) has no scale: it gets the absolute FP32_TOL
            bound = 1e-4 * scale if scale > ZERO_GRAD else FP32_TOL
            report.append(f"  d{k}: max|diff| {err:.3e}  max|ref| {scale:.3e}  bound {bound:.1e}")
            if not err <= bound:
                bad.append(report[-1])
        print(f"\n{variant} {route}: {len(batch)} documents, {bt.total_nodes} node rows\n" + "\n".join(report))
        assert not bad, f"{variant} {route}:\n" + "\n".join(bad)
