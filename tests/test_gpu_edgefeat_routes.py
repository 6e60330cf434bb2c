"""-m gpu: the word-level attention of the edge-feature producer (csrc/edgefeat.cu) on both of its kernel routes,
against oracle/edge_oracle.py run in float64.

A batch whose longest active first sentence has at most WP_MAX_LEN = 96 tokens runs the per-document kernels
(the sentence in shared memory, three logits per lane, backward entries in chunks of 32); any other batch runs the
per-warp kernels.  Records from ``synthetic`` never have a first sentence past 40 tokens, so the records here are
built by hand: first sentences of 1 to 512 tokens (and one that max_length cuts short), mentions on the first and
last token and far enough apart to reach every distance bucket, 1 to 72 active slots per document, max_num
truncation and inactive later slots.  Every case that fits the per-document route runs twice: on the route the
batch selects, and on the per-warp route forced by withholding the per-document tables.

Tolerances as in test_gpu_edgefeat.py: 1e-4 absolute on context_sent_att, 1e-4 of the largest reference entry on
every gradient.
"""
import networkx as nx
import numpy as np
import pytest
import torch

from helpers import FP32_TOL, head_state, maxdiff
from oracle import featurize_oracle as FO
from test_gpu_edgefeat import DEV, gpu_edges, oracle_edges, producer
from gcgcn_b200 import _lib
from gcgcn_b200.batch import DIS_PLUS, RaggedBatch
from gcgcn_b200.edgefeat import EdgeTables
from gcgcn_b200.featurize import wire_from_record

pytestmark = pytest.mark.gpu

WP_MAX_LEN = 96                  # csrc/edgefeat.cu: longest first sentence of the per-document route
GRAD_TOL = 1e-4
DOC_KERNELS = {"word_pool_fwd<doc>", "word_pool_bwd<doc>"}
WARP_KERNELS = {"word_pool_fwd", "word_pool_bwd_logit", "word_pool_bwd_token"}


def make_case(first_len, starts, slots=None, doc_len=None, extra=1, S=3, trunc=False, seed=0):
    """A record with the schema of ``synthetic.make_record`` whose first sentence is [0, first_len).

    starts: the one-token mention of each entity that the first sentence holds (each also has a mention later on);
    slots:  how many ordered pairs of those entities share the first sentence, in a random slot among up to S - 1
            later sentences (default: every pair); the other pairs share later sentences only;
    extra:  entities mentioned in later sentences only;
    trunc:  one more pair lists the first sentence as its sixth sentence, which max_num = 5 cuts away.
    Every edge has at most S slots of which one is active, so no pair divides by 1e-10 (G:213)."""
    rng = np.random.RandomState(1000 + seed)
    doc_len = first_len + 40 if doc_len is None else doc_len
    bounds = [first_len]
    while bounds[-1] < doc_len:
        bounds.append(min(doc_len, bounds[-1] + int(rng.randint(8, 30))))
    later = list(zip(bounds[:-1], bounds[1:]))
    first = (0, first_len)

    def some_later():
        return later[rng.randint(len(later))]

    def mention(sent):
        a = int(rng.randint(sent[0], sent[1]))
        return a, min(sent[1], a + int(rng.randint(1, 3)))

    g = nx.DiGraph()
    k = len(starts)
    for e, p in enumerate(starts):
        g.add_node(e, exist_pos=[(int(p), int(p) + 1), mention(some_later())], type=[1 + e % 6])
    for e in range(k, k + extra):
        g.add_node(e, exist_pos=[mention(some_later())], type=[1 + e % 6])
    pairs = [(a, b) for a in range(k) for b in range(k) if a != b]
    slots = len(pairs) if slots is None else slots
    assert slots + trunc <= len(pairs)
    for i, pi in enumerate(rng.permutation(len(pairs))):
        a, b = pairs[pi]
        sents = [some_later() for _ in range(rng.randint(0, S))]
        if i < slots:
            sents.insert(rng.randint(len(sents) + 1), first)
        elif trunc and i == slots:
            sents = [some_later() for _ in range(5)] + [first]
        if sents:
            pos = [g.nodes[a]["exist_pos"][0] + g.nodes[b]["exist_pos"][0] if s == first else mention(s) + mention(s)
                   for s in sents]
            g.add_edge(a, b, sentences=sents, position=pos)
    for e in range(k, k + extra):
        s = some_later()
        g.add_edge(e, 0, sentences=[s], position=[mention(s) + mention(s)])
    g.graph["max_sentence_num"] = 6 if trunc else S
    return {"document": rng.randint(1, 1000, size=doc_len).tolist(), "graph": g}


def spread(first_len, k):
    """k mention starts from the first to the last token of the sentence."""
    return np.linspace(0, first_len - 1, k).round().astype(int).tolist()


def length_case(first_len, doc_len=None):
    starts = spread(first_len, 4) if first_len >= 4 else [0, first_len - 1]
    return make_case(first_len, starts, doc_len=doc_len, seed=first_len)


# (first sentence, document) tokens; (560, 600): max_length = 512 cuts the first sentence, and its mention at token
# 559 lies past the cut, so distances of 512+ (bucket 10) occur too
LENGTHS = [(1, None), (2, None), (31, None), (32, None), (33, None), (63, None), (64, None), (65, None), (95, None),
           (96, None), (97, None), (130, None), (257, None), (511, None), (512, None), (560, 600)]
# (first sentence, entities in it, active slots, max_num truncation): E = 2 x slots backward entries per document
ENTRIES = [(40, 2, 1, False), (70, 5, 16, False), (70, 5, 17, True), (90, 7, 32, False), (90, 7, 33, True),
           (96, 9, 72, False)]


def entries_case(first_len, k, slots, trunc):
    return make_case(first_len, spread(first_len, k), slots=slots, S=2, trunc=trunc, seed=100 + slots)


def active_rows(item):
    """Distance-table rows that the tokens of the active slots (sentence holds token 0, G:302) look up."""
    d = FO.from_list_to_tensor(item)
    sen = d["sen_matrix"]
    act = sen[:, :, :, 0:1] & sen
    return set(np.unique(d["pos_matrix_h"][act]).tolist()) | set(np.unique(d["pos_matrix_t"][act]).tolist())


def rel_err(a, b):
    """max |a - b| / max |b|, the rel_close rule of test_gpu_edgefeat.py."""
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    assert a.shape == b.shape, (a.shape, b.shape)
    return float((a - b).abs().max()) / max(float(b.abs().max()), 1e-2)


def check_batch(items, hop, seed, what):
    """Run the documents as one batch on the route it selects and, when that is the per-document route, on the
    per-warp route too; compare every document with its own float64 oracle run and the parameter gradients with
    their sum.  Returns the tables of the batch and {route: (max |e - e_ref|, worst relative gradient error)}."""
    wires = [wire_from_record(it) for it in items]
    state = head_state(seed)
    # most slots pass the relu of the sentence-level score (G:212) and so send gradient into the word attention
    state[f"sentence_attention.{hop}.attention_all.bias"] = torch.full((1,), 0.25)
    gen = torch.Generator().manual_seed(seed)
    ctxs = [torch.tanh(torch.randn(w.length, 128, generator=gen)) for w in wires]
    xs = [torch.tanh(torch.randn(w.n, 128, generator=gen)) for w in wires]
    ups = [torch.randn(w.n * w.n, 128, generator=gen) for w in wires]
    s64 = {k: v.double() for k, v in state.items()}
    refs = []
    for b, (it, w, c, x, u) in enumerate(zip(items, wires, ctxs, xs, ups)):
        dense = FO.from_list_to_tensor(it)
        refs.append(oracle_edges(hop, c.double(), x.double(), dense, s64, u.double().view(w.n, w.n, 128)))
        if dense["sen_matrix"][:, :, :, 0].any():
            assert float(refs[-1][1].abs().max()) > 0, f"{what}: no active slot of document {b} passes the relu"
    gsum = {k: sum(r[3][k] for r in refs) for k in refs[0][3]}
    assert len(gsum) == 17                                  # 16 parameters of the hop + dis_embed.weight
    ef = producer(state)
    bt = RaggedBatch([w.n for w in wires], DEV)
    result = {}
    tabs = EdgeTables(wires, bt, DEV)
    assert (tabs.pair_denom_host >= 1).all()
    routes = ["doc", "warp"] if tabs.max_active_len <= WP_MAX_LEN else ["warp"]
    for route in routes:
        tabs = EdgeTables(wires, bt, DEV)
        if route == "warp" and tabs.max_active_len <= WP_MAX_LEN:
            tabs.c_struct.adoc_tok0 = None                  # word_pool_doc_path() is false without the per-document tables
        st = torch.cuda.current_stream().cuda_stream
        _lib.timing_begin(st)
        e, dc, dx, gg = gpu_edges(ef, hop, torch.cat(ctxs), torch.cat(xs), state["dis_embed.weight"], tabs,
                                  torch.cat(ups))
        ran = set(_lib.timing_end(st))
        want, other = (DOC_KERNELS, WARP_KERNELS) if route == "doc" else (WARP_KERNELS, DOC_KERNELS)
        assert want <= ran and not other & ran, f"{what}: {route} route expected, ran {sorted(ran)}"
        fwd, grad = 0.0, 0.0
        p0 = t0 = n0 = 0
        for b, (w, r) in enumerate(zip(wires, refs)):
            eo, dco, dxo, _ = r
            fwd = max(fwd, maxdiff(e[p0:p0 + w.n * w.n].cpu().view(w.n, w.n, 128), eo))
            for name, a, ref in (("d context", dc[t0:t0 + w.length], dco), ("d node_feat", dx[n0:n0 + w.n], dxo)):
                err = rel_err(a, ref)
                assert err <= GRAD_TOL, f"{what} {route} doc {b} {name}: {err:.3e} > {GRAD_TOL:.0e}"
                grad = max(grad, err)
            p0, t0, n0 = p0 + w.n * w.n, t0 + w.length, n0 + w.n
        assert fwd <= FP32_TOL, f"{what} {route}: max|e - e_ref| = {fwd:.3e} > {FP32_TOL:.0e}"
        for k, v in gsum.items():
            err = rel_err(gg[k], v)
            assert err <= GRAD_TOL, f"{what} {route} {k}: {err:.3e} > {GRAD_TOL:.0e}"
            grad = max(grad, err)
        result[route] = (fwd, grad)
        print(f"{what} [{route}]: max|e - e_ref| {fwd:.2e}, worst gradient error {grad:.2e} of the largest entry")
    return tabs, result


@pytest.mark.parametrize("first_len,doc_len", LENGTHS)
def test_first_sentence_length(first_len, doc_len):
    item = length_case(first_len, doc_len)
    tabs, result = check_batch([item], first_len % 2, first_len, f"first sentence {first_len}")
    assert tabs.max_active_len == min(first_len, 512)
    assert list(result) == (["doc", "warp"] if first_len <= WP_MAX_LEN else ["warp"])


@pytest.mark.parametrize("first_len,k,slots,trunc", ENTRIES)
def test_entries_per_document(first_len, k, slots, trunc):
    item = entries_case(first_len, k, slots, trunc)
    tabs, result = check_batch([item], slots % 2, slots, f"E = {2 * slots}")
    assert tabs.num_slots == slots and tabs.max_active_len == first_len
    assert list(result) == ["doc", "warp"]


def test_cases_reach_every_distance_bucket():
    """The cases above look up every row dis_plus - 9 .. dis_plus + 9 of the distance table that a sentence of 512
    tokens can reach (the truncated one adds dis_plus - 10), the per-document route every row up to +-7."""
    doc_items = [length_case(f, d) for f, d in LENGTHS if f <= WP_MAX_LEN] + [entries_case(*c) for c in ENTRIES]
    warp_items = doc_items + [length_case(f, d) for f, d in LENGTHS if f > WP_MAX_LEN]
    doc_rows = set().union(*map(active_rows, doc_items))
    warp_rows = set().union(*map(active_rows, warp_items))
    assert set(range(DIS_PLUS - 7, DIS_PLUS + 8)) <= doc_rows, sorted(doc_rows)
    assert set(range(DIS_PLUS - 9, DIS_PLUS + 10)) <= warp_rows, sorted(warp_rows)
    assert DIS_PLUS - 10 in warp_rows


def test_mixed_batch_moves_to_the_per_warp_route():
    """Twenty short documents, four of them without an active slot, and one with a first sentence of 120 tokens: that
    document alone moves the whole batch to the per-warp kernels."""
    items = []
    for i in range(20):
        fl = 6 + (7 * i) % 35
        if i % 5 == 2:
            items.append(make_case(fl, [0, fl - 1], slots=0, seed=300 + i))
        else:
            items.append(make_case(fl, spread(fl, 2 + i % 3), seed=300 + i))
    items.insert(9, make_case(120, spread(120, 4), seed=399))
    tabs, result = check_batch(items, 1, 7, "mixed batch")
    assert tabs.max_active_len == 120 and tabs.num_active_docs == 17
    assert list(result) == ["warp"]


def test_large_batch_spreads_the_weight_reductions():
    """Enough active tokens and pairs that word_table_bwd_kernel (8 warps per SM) and sent_pool_bwd_kernel (32 warps
    per SM) take more than one item per warp, and their partial sums have about a thousand and five thousand parts."""
    lens = [70 + (13 * i) % 27 for i in range(60)]
    items = [make_case(fl, spread(fl, 10), S=2, extra=0, doc_len=fl + 24, seed=500 + i) for i, fl in enumerate(lens)]
    tabs, result = check_batch(items, 0, 11, "large batch")
    sms = torch.cuda.get_device_properties(DEV).multi_processor_count
    assert tabs.num_tokens >= 4096 and tabs.num_tokens > 8 * sms, tabs.num_tokens
    assert tabs.num_pairs >= 5000 and tabs.num_pairs > 32 * sms, tabs.num_pairs
    assert list(result) == ["doc", "warp"]
