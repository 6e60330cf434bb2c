"""-m gpu: the individual entry points of the C ABI against the oracle / plain fp64 math."""
import numpy as np
import pytest
import torch

from helpers import FP32_TOL, BF16_TOL, assert_close, golden, maxdiff
from oracle import gcgcn_oracle as O
from gcgcn_b200 import _lib, functional as F, synthetic as S
from gcgcn_b200.batch import PairTables, PoolTable, RaggedBatch, node_relative_pos
from gcgcn_b200.modules import pair_gather, pool_nodes

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.mark.parametrize("ta,tb", [(0, 0), (0, 1), (1, 0), (1, 1)])
@pytest.mark.parametrize("M,N,K", [(243, 128, 128), (64, 64, 16), (1, 1, 1), (130, 1024, 129), (128, 1024, 5000),
                                   (64, 64, 40000), (37, 51, 77), (300, 8, 3),
                                   # tall A, weight-like B: the pre-split-B (bulk copy) variant, ragged edges included
                                   (4224, 1024, 128), (5000, 130, 129), (4100, 128, 1000),
                                   # short M, K = "every node row": the MN-major weight-gradient variant (with ta=1, tb=0)
                                   (128, 1024, 20000), (100, 260, 9001), (256, 128, 8200),
                                   # K <= 128 with several column tiles: row operand resident in tensor memory
                                   (4100, 300, 100), (8192, 1024, 64), (4097, 256, 128),
                                   # split K on the CUDA-core kernel (M*N*K < 2e6, K >= 2048), on the scalar reduce
                                   (16, 16, 5000), (12, 13, 10000), (128, 130, 20000)])
def test_gemm_against_fp64(ta, tb, M, N, K):
    g = torch.Generator().manual_seed(M * 7 + N * 3 + K)
    a = torch.randn((K, M) if ta else (M, K), generator=g)
    b = torch.randn((N, K) if tb else (K, N), generator=g)
    bias = torch.randn(N, generator=g)
    c0 = torch.randn(M, N, generator=g)
    ref = (a.double().t() if ta else a.double()) @ (b.double().t() if tb else b.double())
    ref = 0.5 * ref + 2.0 * c0.double() + bias.double()
    out = F.gemm(a.to(DEV), b.to(DEV), ta, tb, bias=bias.to(DEV), out=c0.clone().to(DEV), alpha=0.5, beta=2.0)
    scale = max(1.0, float(ref.abs().max()))
    assert maxdiff(out, ref) <= 2e-6 * scale * max(1, K) ** 0.5


@pytest.mark.parametrize("M,N,K", [(37, 51, 77), (300, 130, 200), (128, 128, 40000)])
def test_gemm_writes_a_row_strided_out_in_place(M, N, K):
    """out = a column slice of a wider buffer: written with its own row stride, the other columns left bit-identical;
    an out whose columns are not contiguous is refused."""
    g = torch.Generator().manual_seed(M + N + K)
    a, b = torch.randn(K, M, generator=g), torch.randn(K, N, generator=g)
    wide = torch.randn(M, N + 9, generator=g).to(DEV)
    before = wide.clone()
    out = F.gemm(a.to(DEV), b.to(DEV), True, False, out=wide[:, 5:5 + N])
    ref = a.double().t() @ b.double()
    assert maxdiff(wide[:, 5:5 + N], ref) <= 2e-6 * float(ref.abs().max()) * K ** 0.5
    assert out.data_ptr() == wide[:, 5:].data_ptr()
    assert torch.equal(wide[:, :5], before[:, :5]) and torch.equal(wide[:, 5 + N:], before[:, 5 + N:])
    with pytest.raises(_lib.GcgcnError, match="unit column stride"):
        F.gemm(a.to(DEV), b.to(DEV), True, False, out=torch.zeros(N, M, device=DEV).t())


def test_gemm_is_deterministic_with_split_k():
    g = torch.Generator().manual_seed(0)
    a, b = torch.randn(30000, 128, generator=g).to(DEV), torch.randn(30000, 256, generator=g).to(DEV)
    r1 = F.gemm(a, b, True, False)
    r2 = F.gemm(a, b, True, False)
    assert torch.equal(r1, r2)


@pytest.mark.parametrize("dtype,tol", [(torch.float32, 1e-6), (torch.bfloat16, BF16_TOL)])
def test_edge_mean_forward_backward(dtype, tol):
    docs = S.make_batch((0, 4, 11, 10))
    bt = RaggedBatch([d.n for d in docs], DEV)
    e = torch.cat([d.e0.reshape(-1, 128) for d in docs]).to(DEV, dtype).requires_grad_(True)
    ebar = F.EdgeMeanFn.apply(e, bt)
    g = torch.randn(ebar.shape, generator=torch.Generator().manual_seed(1)).to(DEV)
    (ebar * g).sum().backward()
    for d, eb, de, gg in zip(docs, bt.split_nodes(ebar), bt.split_pairs(e.grad), bt.split_nodes(g)):
        src = d.e0.to(dtype).float()
        assert_close(eb, src.mean(1), 1e-6, "ebar")
        assert_close(de.float(), (gg.cpu() / d.n).unsqueeze(1).expand(-1, d.n, -1), tol, "de")
    assert e.grad.dtype == dtype


def test_pooling_matches_oracle_and_golden():
    docs = S.make_batch()
    tab = PoolTable.from_spans([d.spans for d in docs], [d.L for d in docs], device=DEV)
    ctx = torch.cat([d.ctx for d in docs]).to(DEV).requires_grad_(True)
    x0 = pool_nodes(ctx, tab)
    gold = golden("pool_pairs.npz")
    assert_close(x0, gold["x0"], 2e-6, "x0 vs reference golden")
    g = torch.randn(x0.shape, generator=torch.Generator().manual_seed(2))
    (x0 * g.to(DEV)).sum().backward()
    row, tok = 0, 0
    for d in docs:
        c = d.ctx.clone().requires_grad_(True)
        ref = O.pool_nodes(O.build_node_pos(d.spans, d.L), c.unsqueeze(0))
        (ref * g[row:row + d.n]).sum().backward()
        assert_close(x0[row:row + d.n], ref, 2e-6, "x0 vs oracle")
        assert_close(ctx.grad[tok:tok + d.L], c.grad, 2e-6, "dctx")
        row, tok = row + d.n, tok + d.L


def test_pooling_bit_exact_when_each_entity_has_one_token():
    # a single-term sum has no rounding freedom: gather must reproduce the rows exactly
    L, n = 40, 7
    spans = [[[3 * e, 3 * e + 1]] for e in range(n)]
    tab = PoolTable.from_spans([spans], [L], device=DEV)
    ctx = torch.randn(L, 128, generator=torch.Generator().manual_seed(3))
    x0 = pool_nodes(ctx.to(DEV), tab)
    assert torch.equal(x0.cpu(), ctx[[3 * e for e in range(n)]])


def test_pair_gather_forward_is_bit_exact_and_backward_matches_autograd():
    docs = S.make_batch((2, 7, 11))
    bt = RaggedBatch([d.n for d in docs], DEV)
    gen = torch.Generator().manual_seed(5)
    dis = torch.randn(21, 20, generator=gen)
    feats = [torch.randn(d.n, 404, generator=gen) for d in docs]
    rps = [node_relative_pos(d.first_pos) for d in docs]
    tabs = PairTables(bt, rps, device=DEV)
    feat_dev = torch.cat(feats).to(DEV).requires_grad_(True)
    dis_dev = dis.clone().to(DEV).requires_grad_(True)
    ph, pt = pair_gather(feat_dev, dis_dev, tabs, bt)
    gh = torch.randn(ph.shape, generator=gen)
    gt = torch.randn(pt.shape, generator=gen)
    ((ph * gh.to(DEV)).sum() + (pt * gt.to(DEV)).sum()).backward()
    dis_ref = dis.clone().requires_grad_(True)
    total = 0
    for b, (d, f, rp) in enumerate(zip(docs, feats, rps)):
        lo, hi = int(bt.pair_ptr_host[b]), int(bt.pair_ptr_host[b + 1])
        f = f.clone().requires_grad_(True)
        rh, rt = O.pair_gather_classifier(f, torch.from_numpy(rp), dis_ref)
        assert torch.equal(ph[lo:hi].cpu(), rh.reshape(-1, 424))       # pure copy: bit-exact
        assert torch.equal(pt[lo:hi].cpu(), rt.reshape(-1, 424))
        total = total + (rh.reshape(-1, 424) * gh[lo:hi]).sum() + (rt.reshape(-1, 424) * gt[lo:hi]).sum()
        (rh.reshape(-1, 424) * gh[lo:hi]).sum().backward(retain_graph=True)
        (rt.reshape(-1, 424) * gt[lo:hi]).sum().backward()
        n0 = int(bt.node_ptr_host[b])
        assert_close(feat_dev.grad[n0:n0 + d.n], f.grad, 1e-4, "dfeat")
    assert_close(dis_dev.grad, dis_ref.grad, 2e-3, "ddis (sum over ~1e3 pairs per row)")


def test_pair_gather_inloop_form_and_golden_rows():
    gold = golden("pool_pairs.npz")
    docs = S.make_batch()
    bt = RaggedBatch([d.n for d in docs], DEV)
    x0 = torch.from_numpy(gold["x0"])
    ner, dis = torch.from_numpy(gold["ner_table"]), torch.from_numpy(gold["dis_table"])
    node_type = torch.cat([d.node_type for d in docs])
    feats = torch.cat([x0, x0, torch.tanh(x0), ner[node_type]], 1)
    rps = [node_relative_pos(d.first_pos) for d in docs]
    assert np.array_equal(np.concatenate([r.reshape(-1) for r in rps]), gold["rel_pos"])
    tabs = PairTables(bt, rps, device=DEV)
    ph, pt = pair_gather(feats.to(DEV), dis.to(DEV), tabs, bt)
    pick = torch.cat([int(bt.pair_ptr_host[b]) + torch.arange(0, d.n * d.n, 7) for b, d in enumerate(docs)])
    assert torch.equal(ph.cpu()[pick], torch.from_numpy(gold["pair_h_rows"]))
    assert torch.equal(pt.cpu()[pick], torch.from_numpy(gold["pair_t_rows"]))
    # in-loop form (G:321-322): no distance part, h[i,j] = x[j], t[i,j] = x[i]
    tabs2 = PairTables(bt, None, device=DEV)
    eh, et = pair_gather(x0.to(DEV), None, tabs2, bt)
    for b, d in enumerate(docs):
        lo = int(bt.pair_ptr_host[b])
        n0 = int(bt.node_ptr_host[b])
        qh, qt = O.pair_gather_inloop(x0[n0:n0 + d.n], 1)
        assert torch.equal(eh[lo:lo + d.n * d.n].cpu(), qh.reshape(-1, 128))
        assert torch.equal(et[lo:lo + d.n * d.n].cpu(), qt.reshape(-1, 128))


def test_empty_batch_is_a_no_op():
    bt = RaggedBatch([], DEV)
    e = torch.zeros(0, 128, device=DEV)
    assert F.EdgeMeanFn.apply(e, bt).shape == (0, 128)
