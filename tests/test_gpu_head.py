"""-m gpu: the whole graph head (G:293-358: pooling, two hops of edge-feature producer + graph block, pair features,
Bilinear + Linear classifier) and the trainer's loss (C:355-364) on the GPU from the wire format, against goldens written
by the UNMODIFIED reference model's own forward/backward with the same weights (tests/golden/edge_head.npz,
make_golden_edge.py) -- SURVEY.md section 4's integration check with the real classifier: logits <= 1e-4, identical
relation argmax, loss, d loss / d context_output and every head parameter's gradient."""
import numpy as np
import pytest
import torch

from helpers import FP32_TOL, golden, head_labels, head_shapes, head_state
from gcgcn_b200 import synthetic as S
from gcgcn_b200.featurize import wire_from_record
from gcgcn_b200.head import GraphHead, HeadBatch

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
BIG_STRIDE = 997


def make_head(seed=0):
    m = GraphHead()
    m.load_state_dict(head_state(seed), strict=True)       # the reference's key names, nothing missing or extra
    return m.to(DEV).eval()


def rel(a, b):
    a, b = torch.as_tensor(a).double().cpu().reshape(-1), torch.as_tensor(b).double().cpu().reshape(-1)
    return float((a - b).abs().max()) / max(float(b.abs().max()), 1e-3)


def golden_doc(g, idx):
    seed, n, L, Sx, _ = g[f"d{idx}_meta"].tolist()
    item = S.make_record(seed, n=n, L=L, S=None if Sx < 0 else Sx)
    return seed, n, wire_from_record(item)


@pytest.mark.parametrize("idx", [0, 1, 2, 3])
def test_head_matches_the_reference_model(idx):
    g = golden("edge_head.npz")
    seed, n, w = golden_doc(g, idx)
    head = make_head()
    hb = HeadBatch([w], DEV)
    ctx = torch.from_numpy(g[f"d{idx}_ctx"]).to(DEV).requires_grad_(True)
    labels = head_labels(seed, n).view(-1, 97).to(DEV)
    out = head(ctx, hb, labels=labels)
    out["loss"].sum().backward()
    torch.cuda.synchronize()
    logits = out["logits"].detach().cpu().view(n, n, 97)
    ref = torch.from_numpy(g[f"d{idx}_logits"])
    assert float((logits - ref).abs().max()) <= FP32_TOL
    assert float((logits.argmax(-1) == ref.argmax(-1)).float().mean()) >= 0.999          # north_star: >= 99.9 %
    assert float((out["e0"].detach().cpu().view(n, n, 128) - torch.from_numpy(g[f"d{idx}_e0"])).abs().max()) <= FP32_TOL
    assert float((out["e1"].detach().cpu().view(n, n, 128) - torch.from_numpy(g[f"d{idx}_e1"])).abs().max()) <= FP32_TOL
    assert abs(float(out["loss"][0].detach()) - float(g[f"d{idx}_loss"].reshape(-1)[0])) <= 1e-5
    assert rel(ctx.grad, g[f"d{idx}_dctx"]) <= 2e-4, "dctx"
    checked = 0
    for k, p in head.named_parameters():
        key = f"d{idx}_g_{k}"
        if key not in g.files:
            # no gradient in the reference either: MAGGC is dead for the logits at graph_hop = 2 (G:338), linears_k unused
            assert p.grad is None or k == "ner_emb.weight", k
            continue
        a = p.grad.detach().cpu().numpy().reshape(-1)
        a = a if a.size <= 40000 else a[::BIG_STRIDE]
        assert rel(a, g[key]) <= 2e-4, k
        checked += 1
    assert checked == 37          # GAT 8, CAGGC 6, hop-0 producer 16, dense 2, bilinear 2, linear 2, dis_embed (hop 1 is dead, G:338)


def test_batched_head_equals_the_per_document_goldens():
    g = golden("edge_head.npz")
    docs = [golden_doc(g, i) for i in range(4)]
    head = make_head()
    hb = HeadBatch([w for _, _, w in docs], DEV)
    ctx = torch.cat([torch.from_numpy(g[f"d{i}_ctx"]) for i in range(4)]).to(DEV).requires_grad_(True)
    labels = torch.cat([head_labels(s, n).view(-1, 97) for s, n, _ in docs]).to(DEV)
    out = head(ctx, hb, labels=labels)
    out["loss"].sum().backward()
    torch.cuda.synchronize()
    lo = 0
    for i, (s, n, _) in enumerate(docs):
        ref = torch.from_numpy(g[f"d{i}_logits"]).view(-1, 97)
        assert float((out["logits"][lo:lo + n * n].detach().cpu() - ref).abs().max()) <= FP32_TOL
        assert abs(float(out["loss"][i].detach()) - float(g[f"d{i}_loss"].reshape(-1)[0])) <= 1e-5
        lo += n * n
    dctx = torch.cat([torch.from_numpy(g[f"d{i}_dctx"]) for i in range(4)])
    assert rel(ctx.grad, dctx) <= 2e-4
    # parameter gradients add up over the documents
    for k in ("bili_layer_01.bias", "dense_layer.bias", "linear_sentence_att.0.bias", "word_attention.0.attention_all.weight",
              "graphcnn.0.linear_layer.weight", "dis_embed.weight"):
        want = sum(g[f"d{i}_g_{k}"] for i in range(4))
        got = dict(head.named_parameters())[k].grad.detach().cpu().numpy().reshape(-1)
        assert rel(got, want) <= 2e-4, k


def test_loss_kernel_alone_matches_torch_bce():
    from gcgcn_b200.batch import RaggedBatch
    from gcgcn_b200.classifier import pair_bce_loss
    sizes = [5, 1, 7, 3]
    bt = RaggedBatch(sizes, DEV)
    gen = torch.Generator().manual_seed(3)
    z = (torch.randn(bt.total_pairs, 97, generator=gen) * 6).requires_grad_(True)
    z.data[0, :5] = torch.tensor([40.0, -40.0, 120.0, -120.0, 0.0])          # saturated sigmoids: the -100 clamp
    y = (torch.rand(bt.total_pairs, 97, generator=gen) < 0.1).float()
    zg = z.detach().to(DEV).requires_grad_(True)
    loss = pair_bce_loss(zg, y.to(DEV), bt)
    w = torch.tensor([1.0, 2.0, -0.5, 3.0])
    (loss * w.to(DEV)).sum().backward()
    want, lo = [], 0
    for n in sizes:
        zz, yy = z[lo:lo + n * n].view(n, n, 97), y[lo:lo + n * n].view(n, n, 97)
        per = torch.nn.functional.binary_cross_entropy(torch.sigmoid(zz), yy, reduction="none").mean(-1)
        off = ~torch.eye(n, dtype=torch.bool)
        want.append(per[off].sum() / max(n * n - n, 1) if n > 1 else per.sum() * 0)
        lo += n * n
    want = torch.stack(want)
    (want * w).sum().backward()
    assert float((loss.detach().cpu() - want.detach()).abs().max()) <= 1e-5
    assert float((zg.grad.cpu() - z.grad).abs().max()) <= 1e-6


@pytest.mark.parametrize("P", [1, 127, 1000, 8192 + 77, 20011])
def test_bilinear_classifier_against_torch(P):
    """G:356-358 on its own: Bilinear(128, 128, 97) + Linear(256, 97) over P pairs (P not a multiple of the 128-row tile,
    and more than one 4096-row range of the weight gradient) against torch's own modules on the CPU."""
    from gcgcn_b200 import classifier as C
    torch.manual_seed(P)
    bili, cls = torch.nn.Bilinear(128, 128, 97), torch.nn.Linear(256, 97)
    gen = torch.Generator().manual_seed(P + 1)
    h = torch.tanh(torch.randn(P, 128, generator=gen)).requires_grad_(True)
    t = torch.tanh(torch.randn(P, 128, generator=gen)).requires_grad_(True)
    up = torch.randn(P, 97, generator=gen)
    want = bili(h, t) + cls(torch.cat([h, t], -1))
    # gradients: float64 reference (the parameter gradients sum P terms; an fp32 CPU sum of 20 000 terms is itself
    # only good to ~1e-4 of its magnitude, which is what the comparison would then measure)
    import copy
    b64, c64 = copy.deepcopy(bili).double(), copy.deepcopy(cls).double()
    h64, t64 = h.detach().double().requires_grad_(True), t.detach().double().requires_grad_(True)
    ((b64(h64, t64) + c64(torch.cat([h64, t64], -1))) * up.double()).sum().backward()
    ref = {"h": h64.grad, "t": t64.grad, "W": b64.weight.grad, "b": b64.bias.grad, "Wc": c64.weight.grad, "bc": c64.bias.grad}
    bg, cg = copy.deepcopy(bili).to(DEV), copy.deepcopy(cls).to(DEV)
    for m in (bg, cg):
        m.zero_grad()
    hg, tg = h.detach().to(DEV).requires_grad_(True), t.detach().to(DEV).requires_grad_(True)
    got = C.relation_logits(hg, tg, bg, cg)
    (got * up.to(DEV)).sum().backward()
    torch.cuda.synchronize()
    assert float((got.detach().cpu() - want.detach()).abs().max()) <= FP32_TOL
    for k, g in (("h", hg.grad), ("t", tg.grad), ("W", bg.weight.grad), ("b", bg.bias.grad), ("Wc", cg.weight.grad),
                 ("bc", cg.bias.grad)):
        assert rel(g, ref[k]) <= 1e-4, k


@pytest.mark.parametrize("idx", [0, 1])
def test_bert_variant_head_matches_the_reference_model(idx):
    """models/GraphCNN_multihead_bert_gate_cls.py: L_s = 4, H = 4 and ``linear_cls`` on the encoder's first-token feature
    (B:346-347), against goldens from the unmodified reference model (its BERT encoder stubbed: ctx and cls_feat are the
    head's inputs)."""
    g = golden("edge_head_bert.npz")
    seed, n, w = golden_doc(g, idx)
    head = GraphHead(4, 4, cls_dim=768)
    head.load_state_dict(head_state(0, 4, 4, cls_dim=768), strict=True)
    head = head.to(DEV).eval()
    hb = HeadBatch([w], DEV)
    ctx = torch.from_numpy(g[f"d{idx}_ctx"]).to(DEV).requires_grad_(True)
    cls_feat = torch.from_numpy(g[f"d{idx}_cls_feat"]).view(1, -1).to(DEV)
    labels = head_labels(seed, n).view(-1, 97).to(DEV)
    out = head(ctx, hb, labels=labels, cls_feat=cls_feat)
    out["loss"].sum().backward()
    torch.cuda.synchronize()
    ref = torch.from_numpy(g[f"d{idx}_logits"])
    logits = out["logits"].detach().cpu().view(n, n, 97)
    assert float((logits - ref).abs().max()) <= FP32_TOL
    assert float((logits.argmax(-1) == ref.argmax(-1)).float().mean()) >= 0.999
    assert abs(float(out["loss"][0].detach()) - float(g[f"d{idx}_loss"].reshape(-1)[0])) <= 1e-5
    assert rel(ctx.grad, g[f"d{idx}_dctx"]) <= 2e-4
    checked = 0
    for k, p in head.named_parameters():
        key = f"d{idx}_g_{k}"
        if key in g.files:
            a = p.grad.detach().cpu().numpy().reshape(-1)
            assert rel(a if a.size <= 40000 else a[::BIG_STRIDE], g[key]) <= 2e-4, k
            checked += 1
    assert checked == 43          # GAT 8, CAGGC 4*2 + 2, hop-0 producer 16, dense 2, bilinear 2, linear 2, linear_cls 2, dis_embed
