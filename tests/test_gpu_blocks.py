"""-m gpu: the batched hot path (GraphBlocks) against the oracle and the reference's golden
vectors: configs 1-4 of BASELINE.json at test size, plus size-independent properties on a
full-size shard."""
import numpy as np
import pytest
import torch

from helpers import BF16_TOL, FP32_TOL, VARIANTS, assert_close, golden, maxdiff, oracle_blocks
from gpu_common import DEV, cat_inputs, device_blocks, run_blocks
from gcgcn_b200 import _lib, synthetic as S
from gcgcn_b200.batch import RaggedBatch

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("fused", [True, False], ids=["block-kernels", "per-op"])
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_batched_blocks_match_oracle_and_reference_golden(variant, fused):
    layers, heads = VARIANTS[variant]
    gb, state = device_blocks(layers, heads)
    gb.fused = fused      # True: gcgcn_caggc_* / gcgcn_mha_stack_* (attention on chip); False: one entry point per op
    docs = S.make_batch()
    before = _lib.launch_count()
    res = run_blocks(gb, docs)
    assert _lib.launch_count() - before >= 20, "the CUDA path must be what ran"
    g = golden(f"graph_blocks_{variant}.npz")
    # reference golden (outputs and node gradients of every document)
    assert_close(res["y1"], g["y1"], FP32_TOL, "y1 vs reference")
    assert_close(res["y2"], g["y2"], FP32_TOL, "y2 vs reference")
    assert_close(res["dx0"], g["dx0"], FP32_TOL, "dx0 vs reference")
    bt = res["bt"]
    total = {}
    for b, d in enumerate(docs):
        r = oracle_blocks(d, state, layers, heads)
        assert_close(bt.split_nodes(res["y1"])[b], r["y1"], FP32_TOL, f"doc{b} y1")
        assert_close(bt.split_nodes(res["y2"])[b], r["y2"], FP32_TOL, f"doc{b} y2")
        assert_close(bt.split_pairs(res["a0"])[b], r["a0"], 1e-5, f"doc{b} a0")
        for h in range(heads):
            assert_close(bt.split_pairs(res["a1"][h])[b], r["a1"][h], 1e-5, f"doc{b} a1[{h}]")
        assert_close(bt.split_nodes(res["dx0"])[b], r["dx0"], FP32_TOL, f"doc{b} dx0")
        assert_close(bt.split_pairs(res["de0"])[b], r["de0"], FP32_TOL, f"doc{b} de0")
        assert_close(bt.split_pairs(res["de1"])[b], r["de1"], FP32_TOL, f"doc{b} de1")
        cs = g["de_checksums"][b]
        de0, de1 = bt.split_pairs(res["de0"])[b].double(), bt.split_pairs(res["de1"])[b].double()
        assert abs(float(de0.sum()) - cs[0]) <= 1e-2 and abs(float(de1.sum()) - cs[2]) <= 1e-2
        for k, v in r["dparams"].items():
            if v is not None:
                total[k] = total.get(k, 0) + v
    # parameter gradients summed over the batch: vs oracle (every element) and vs golden samples
    for k, v in res["dparams"].items():
        if "linears_k" in k:
            assert v is None                                           # quirk 3
            continue
        assert_close(v, total[k], 5 * FP32_TOL, "d" + k)              # sums of 12 documents
    off = 0
    for name, size in zip(g["grad_names"], g["grad_sample_sizes"]):
        assert_close(res["dparams"][str(name)].reshape(-1)[::37], g["grad_samples"][off:off + size],
                     5 * FP32_TOL, f"d{name} vs reference")
        off += size
    # append-before-update: the classifier sees cat[x0, x0, y1], never y2 (quirk 5)
    x0 = torch.cat([d.x0 for d in docs])
    assert torch.equal(res["node_feats"][:, :128].cpu(), x0) and torch.equal(res["node_feats"][:, 128:256].cpu(), x0)
    assert torch.equal(res["node_feats"][:, 256:], res["y1"])


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_train_mode_with_injected_keep_masks(variant):
    layers, heads = VARIANTS[variant]
    gb, state = device_blocks(layers, heads)
    g = golden(f"graph_blocks_{variant}.npz")
    gs = 128 // layers
    for i in (0, 5, 11):
        d = S.make_doc(i)
        keep = S.make_keep_masks(d.doc_id, d.n, layers, heads)
        gb.get_weighted_adj_matrix.inject_keep([keep["gat"]])
        gb.graphcnn[0].inject_keep(keep["cag"])
        gb.get_adj_matrix[0].inject_keep(keep["mha"])
        gb.graphcnn[1].inject_keep([m for hm in keep["mag"] for m in hm])
        gb.inject_keep([keep["out0"], keep["out1"]])
        res = run_blocks(gb, [d])
        r = oracle_blocks(d, state, layers, heads, keep=keep)
        for k in ("y1", "y2", "dx0", "de0", "de1"):
            assert_close(res[k].reshape(r[k].shape), r[k], FP32_TOL, f"train doc{i} {k}")
        assert_close(res["y1"], g[f"train{i}_y1"], FP32_TOL, "train y1 vs reference")
        assert_close(res["y2"], g[f"train{i}_y2"], FP32_TOL, "train y2 vs reference")
        assert_close(res["dx0"], g[f"train{i}_dx0"], FP32_TOL, "train dx0 vs reference")
        for k, v in res["dparams"].items():
            if v is not None:
                assert_close(v, r["dparams"][k], 2 * FP32_TOL, f"train d{k}")
    # and plain .train() really drops: outputs differ from eval, keep statistics are sane
    gb.train()
    d = S.make_doc(2)
    a = run_blocks(gb, [d], backward=False)
    gb.eval()
    b = run_blocks(gb, [d], backward=False)
    assert maxdiff(a["y1"], b["y1"]) > 1e-3
    zeros = float((a["y1"] == 0).float().mean())
    assert 0.1 < zeros < 0.3                                          # p = 0.2 (G:232)


@pytest.mark.parametrize("n,heads,layers", [(128, 4, 2), (128, 8, 2), (256, 4, 2), (256, 8, 2), (256, 4, 4),
                                            (65, 8, 2), (64, 4, 4)])
def test_entity_count_sweep(n, heads, layers):
    """config 4: fully connected graphs far beyond DocRED's 42 entities."""
    gb, state = device_blocks(layers, heads)
    d = S.make_doc(40 + n, n=n, L=64)
    res = run_blocks(gb, [d])
    r = oracle_blocks(d, state, layers, heads)
    for k in ("y1", "y2", "dx0", "de0", "de1"):
        assert_close(res[k].reshape(r[k].shape), r[k], FP32_TOL, f"n={n} {k}")
    for k, v in res["dparams"].items():
        if v is not None:
            assert_close(v, r["dparams"][k], 5 * FP32_TOL, f"n={n} d{k}")


@pytest.mark.parametrize("layers,heads", [(2, 4), (4, 8), (2, 8), (4, 4)])
def test_every_block_kernel_instantiation(layers, heads):
    """The fused route for all four (sub-layer width, head width) combinations x all four size classes."""
    gb, state = device_blocks(layers, heads)
    sizes = [64, 50, 48, 33, 32, 17, 16, 9, 1]
    docs = [S.make_doc(300 + i, n=n, L=32) for i, n in enumerate(sizes)]
    before = _lib.launch_count()
    res = run_blocks(gb, docs)
    assert _lib.launch_count() - before >= 20
    bt = res["bt"]
    total = {}
    for b, d in enumerate(docs):
        r = oracle_blocks(d, state, layers, heads)
        for k in ("y1", "y2", "dx0"):
            assert_close(bt.split_nodes(res[k])[b], r[k], FP32_TOL, f"L{layers} H{heads} n={d.n} {k}")
        for k in ("de0", "de1"):
            assert_close(bt.split_pairs(res[k])[b], r[k], FP32_TOL, f"L{layers} H{heads} n={d.n} {k}")
        for h in range(heads):
            assert_close(bt.split_pairs(res["a1"][h])[b], r["a1"][h], 1e-5, f"n={d.n} a1[{h}]")
        for k, v in r["dparams"].items():
            if v is not None:
                total[k] = total.get(k, 0) + v
    for k, v in res["dparams"].items():
        if v is not None:
            assert_close(v, total[k], 5 * FP32_TOL, f"L{layers} H{heads} d{k}")


def test_ragged_edge_cases():
    """n = 1, 2, 3 next to large documents, repeated sizes, documents in any order."""
    gb, state = device_blocks(2, 8)
    sizes = [1, 2, 3, 42, 1, 7, 33, 2, 64, 5]
    docs = [S.make_doc(200 + i, n=n, L=32) for i, n in enumerate(sizes)]
    res = run_blocks(gb, docs)
    bt = res["bt"]
    for b, d in enumerate(docs):
        r = oracle_blocks(d, state, 2, 8)
        for k in ("y1", "y2", "dx0"):
            assert_close(bt.split_nodes(res[k])[b], r[k], FP32_TOL, f"n={d.n} {k}")
        for k in ("de0", "de1"):
            assert_close(bt.split_pairs(res[k])[b], r[k], FP32_TOL, f"n={d.n} {k}")


def test_bf16_edge_storage():
    """config 3: BERT-variant graph head with the n^2 edge tensors stored in bf16, fp32 accumulation.
    The reference cannot execute in bf16 (SURVEY.md section 7), so the oracle is the fp32 reference:
    forward outputs are compared with the fp32 oracle on the *unrounded* inputs; gradients (whose
    scale is set by the arbitrary N(0,1) upstream gradient, |dx0| ~ 10) with the fp32 oracle on the
    identical, bf16-representable edge values.  Tolerance 2e-2 absolute in both cases."""
    import copy
    layers, heads = VARIANTS["bert"]
    gb, state = device_blocks(layers, heads)
    docs = S.make_batch()
    res = run_blocks(gb, docs, edge_dtype=torch.bfloat16)
    assert res["de0"].dtype == torch.bfloat16 and res["de1"].dtype == torch.bfloat16
    bt = res["bt"]
    for b, d in enumerate(docs):
        r = oracle_blocks(d, state, layers, heads, backward=False)
        for k in ("y1", "y2"):
            assert_close(bt.split_nodes(res[k])[b], r[k], BF16_TOL, f"bf16 doc{b} {k}")
        dq = copy.copy(d)
        dq.e0, dq.e1 = d.e0.bfloat16().float(), d.e1.bfloat16().float()
        r = oracle_blocks(dq, state, layers, heads)
        for k in ("y1", "y2", "dx0"):
            assert_close(bt.split_nodes(res[k])[b], r[k], FP32_TOL * 5, f"bf16-in doc{b} {k}")
        for k in ("de0", "de1"):
            assert_close(bt.split_pairs(res[k])[b].float(), r[k], BF16_TOL, f"bf16 doc{b} {k}")


def test_full_size_shard_properties():
    """A shard at bench scale (1200 documents, n cycling through the 12-value list): checks that do
    not need the oracle on every document -- batch invariance, permutation equivariance, run-to-run
    determinism -- plus the oracle on a sample of documents."""
    gb, state = device_blocks(2, 8)
    ids = list(range(1200))
    docs = [S.make_doc(i) for i in ids]
    res = run_blocks(gb, docs)
    bt = res["bt"]
    assert bt.total_nodes == 100 * 243 and bt.total_pairs == 100 * 6207
    # determinism
    res2 = run_blocks(gb, docs)
    for k in ("y1", "y2", "dx0", "de0", "de1"):
        assert torch.equal(res[k], res2[k]), k
    # batch invariance: a document's result does not depend on its neighbours
    sample = [0, 13, 599, 1187, 1199]
    y1s, y2s, dxs = bt.split_nodes(res["y1"]), bt.split_nodes(res["y2"]), bt.split_nodes(res["dx0"])
    de0s = bt.split_pairs(res["de0"])
    for i in sample:
        alone = run_blocks(gb, [docs[i]])
        # (not bit-identical: tiny products take the CUDA-core GEMM, large ones the tcgen05 3xTF32 GEMM)
        assert_close(alone["y1"], y1s[i], 2e-5, "batch invariance y1")
        assert_close(alone["y2"], y2s[i], 2e-5, "batch invariance y2")
        assert_close(alone["dx0"], dxs[i], 2e-5, "batch invariance dx0")
        r = oracle_blocks(docs[i], state, 2, 8)
        assert_close(y1s[i], r["y1"], FP32_TOL, "y1")
        assert_close(y2s[i], r["y2"], FP32_TOL, "y2")
        assert_close(dxs[i], r["dx0"], FP32_TOL, "dx0")
        assert_close(de0s[i], r["de0"], FP32_TOL, "de0")
    # permutation equivariance: relabelling the entities of a document permutes its outputs
    d = docs[3]
    perm = torch.randperm(d.n, generator=torch.Generator().manual_seed(0))
    import copy
    dp = copy.copy(d)
    dp.x0, dp.e0, dp.e1 = d.x0[perm], d.e0[perm][:, perm], d.e1[perm][:, perm]
    dp.adj = d.adj[perm][:, perm]
    a, b = run_blocks(gb, [d], backward=False), run_blocks(gb, [dp], backward=False)
    assert_close(a["y2"][perm.to(DEV)], b["y2"], 1e-5, "permutation equivariance")
    # weight gradients of the shard = sum of per-document gradients (linearity), checked on a slice.
    # relu'(x) jumps at 0: documents with a pre-activation within float rounding of 0 (about 1 in 40,
    # e.g. doc 14) have ill-conditioned gradients and are left out of this comparison.
    from helpers import relu_margin
    well = [dd for dd in docs[:40] if relu_margin(dd, state, 2, 8) > 2e-6][:24]
    assert len(well) == 24
    part = run_blocks(gb, well)
    tot = {}
    for dd in well:
        r = oracle_blocks(dd, state, 2, 8)
        for k, v in r["dparams"].items():
            if v is not None:
                tot[k] = tot.get(k, 0) + v
    for k, v in part["dparams"].items():
        if v is not None:
            assert_close(v, tot[k], 24 * FP32_TOL, f"summed d{k}")   # 24 documents x 1e-4


@pytest.mark.parametrize("layers,heads", [(2, 8), (4, 4)])
def test_large_and_small_documents_in_one_batch(layers, heads):
    """max n > 64 takes the whole batch off the block kernels onto the row-tiled stack kernels (gcn_stack_tiled.cu):
    documents smaller than a tile, tile-boundary sizes and non-multiples of 8 in the same launch."""
    gb, state = device_blocks(layers, heads)
    # document ids picked so that no relu pre-activation lies within 4e-6 of zero for either configuration
    # (helpers.relu_margin; DESIGN.md section 2: a pre-activation inside float rounding of 0 may flip one unit)
    picks = [(426, 130), (458, 66), (502, 40), (550, 7), (647, 96), (661, 97), (700, 1)]
    docs = [S.make_doc(i, n=n, L=32) for i, n in picks]
    res = run_blocks(gb, docs)
    bt = res["bt"]
    total = {}
    for b, d in enumerate(docs):
        r = oracle_blocks(d, state, layers, heads)
        for k in ("y1", "y2", "dx0"):
            assert_close(bt.split_nodes(res[k])[b], r[k], FP32_TOL, f"L{layers} H{heads} n={d.n} {k}")
        for k in ("de0", "de1"):
            assert_close(bt.split_pairs(res[k])[b], r[k], FP32_TOL, f"L{layers} H{heads} n={d.n} {k}")
        for k, v in r["dparams"].items():
            if v is not None:
                total[k] = total.get(k, 0) + v
    for k, v in res["dparams"].items():
        if v is not None:
            assert_close(v, total[k], 5 * FP32_TOL, f"L{layers} H{heads} d{k}")


def test_train_mode_keep_masks_on_a_large_document():
    """Injected dropout masks (all five sites) at n = 100: the keep-mask route of the row-tiled kernels."""
    layers, heads = 2, 8
    gb, state = device_blocks(layers, heads)
    d = S.make_doc(79, n=100, L=32)
    keep = S.make_keep_masks(d.doc_id, d.n, layers, heads)
    gb.get_weighted_adj_matrix.inject_keep([keep["gat"]])
    gb.graphcnn[0].inject_keep(keep["cag"])
    gb.get_adj_matrix[0].inject_keep(keep["mha"])
    gb.graphcnn[1].inject_keep([m for hm in keep["mag"] for m in hm])
    gb.inject_keep([keep["out0"], keep["out1"]])
    res = run_blocks(gb, [d])
    r = oracle_blocks(d, state, layers, heads, keep=keep)
    for k in ("y1", "y2", "dx0", "de0", "de1"):
        assert_close(res[k].reshape(r[k].shape), r[k], FP32_TOL, f"train n=100 {k}")
    for k, v in res["dparams"].items():
        if v is not None:
            assert_close(v, r["dparams"][k], 5 * FP32_TOL, f"train n=100 d{k}")
