"""Time the merge of sorted candidate rankings (csrc/rank.cu, gcgcn_rank_merge) and RelationEvaluator.merged
(gcgcn_b200/evaluate.py) with CUDA events, at two sizes of the BASELINE document mix: DocRED-dev size (1000 documents,
about 48 M candidates) and three 6144-document bench shards (18432 documents, about 880 M).

Per size and per R = 2, 4, 8 parts (documents dealt with shard_documents, every part an evaluator with global ids):
- `merge`: the ceil(log2 R) pairwise merge rounds alone, over the parts' sorted runs, into preallocated buffers;
- `merged`: RelationEvaluator.merged(parts) end to end, every part re-ranked (its sort included) and the merged
  buffers allocated as a user's call does;
- `sort_concat`: gcgcn_rank_sort over the concatenation of the parts' candidates (the single-device alternative:
  gather everything, then sort once), alternated with the two above in every repetition.
Bytes are computed from the shapes, two ways: `bytes_floor` is the merge's algorithmic floor, 16 bytes per candidate
per round (read key and payload of both runs, write them merged); `bytes_kernels` is what the merge kernels load and
store, counted from their code (the floor plus the partition's binary searches), not read from a hardware counter.
`merge_gbs` is bytes_kernels over the measured merge time.  Every working set is far larger than the 126 MB L2.

    python scripts/time_rank_merge.py --out profiles/r03_rank_merge.json
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from gcgcn_b200 import _lib, synthetic  # noqa: E402
from gcgcn_b200.batch import RaggedBatch, shard_documents  # noqa: E402
from gcgcn_b200.evaluate import SORT_TILE, RelationEvaluator  # noqa: E402
from gcgcn_b200.functional import _p, _stream  # noqa: E402

HBM_GBS = 6460.5        # the project's measured HBM figure on the B200 (SURVEY.md, MEASURED_PEAKS hbm_gbs)
R = 97


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def timed(fn, dev):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(torch.cuda.current_stream(dev))
    fn()
    b.record(torch.cuda.current_stream(dev))
    b.synchronize()
    return a.elapsed_time(b)


def make_parts(sizes, parts, dev, seed):
    """One evaluator with global ids per shard of `sizes`, fed random logits (scale 4: many saturated ties)."""
    evs = []
    for k, docs in enumerate(shard_documents(sizes, parts)):
        bt = RaggedBatch(sizes[docs], dev)
        gen = torch.Generator(device=dev).manual_seed(seed + k)
        z = torch.randn(bt.total_pairs, R, generator=gen, device=dev) * 4.0
        ev = RelationEvaluator(R, dev, doc_sizes=sizes)
        ev.add(z, None, bt, doc_index=docs)
        del z
        evs.append(ev)
    return evs


def merge_plan(counts):
    """The merge rounds of RelationEvaluator.merged: per round the (a, b) run pairs; an odd last run moves up."""
    rounds, runs = [], list(range(len(counts)))
    sizes = dict(enumerate(counts))
    nxt_id = len(counts)
    while len(runs) > 1:
        pairs, nxt = [], []
        for a, b in zip(runs[0::2], runs[1::2]):
            pairs.append((a, b, nxt_id))
            sizes[nxt_id] = sizes[a] + sizes[b]
            nxt.append(nxt_id)
            nxt_id += 1
        if len(runs) % 2:
            nxt.append(runs[-1])
        rounds.append(pairs)
        runs = nxt
    return rounds, sizes


def one_config(sizes, parts, reps, dev):
    evs = make_parts(sizes, parts, dev, 1000 * parts)
    for ev in evs:
        ev.rank()
    counts = [ev.count for ev in evs]
    N = sum(counts)
    lib = _lib.load()
    st = _stream(dev)
    rounds, run_sizes = merge_plan(counts)
    bufs = {i: ev.ranked for i, ev in enumerate(evs)}
    for pairs in rounds:
        for _, _, o in pairs:
            bufs[o] = (torch.empty(run_sizes[o], dtype=torch.int32, device=dev),
                       torch.empty(run_sizes[o], dtype=torch.int32, device=dev))
    mws = torch.empty(int(lib.gcgcn_rank_merge_ws_bytes(N)), dtype=torch.uint8, device=dev)

    def merge():
        for pairs in rounds:
            for a, b, o in pairs:
                (ka, pa), (kb, pb), (ko, po) = bufs[a], bufs[b], bufs[o]
                _lib.call("gcgcn_rank_merge", _p(ka), _p(pa), ka.numel(), _p(kb), _p(pb), kb.numel(), _p(ko), _p(po),
                          _p(mws), mws.numel(), st)

    def merged():
        for ev in evs:
            ev._ranked = None                   # re-rank every part: merged() as a user calls it on fresh parts
        return RelationEvaluator.merged(evs)

    score = torch.cat([ev.scores for ev in evs])
    payload = torch.cat([ev._chunks[0][1] for ev in evs])
    key_c, pay_c = torch.empty_like(payload), torch.empty_like(payload)
    sws = torch.empty(int(lib.gcgcn_rank_ws_bytes(N)), dtype=torch.uint8, device=dev)

    def sort_concat():
        _lib.call("gcgcn_rank_sort", _p(score), _p(payload), N, _p(key_c), _p(pay_c), _p(sws), sws.numel(), st)

    merge()
    m = merged()
    sort_concat()
    torch.cuda.synchronize()
    # the merged ranking holds the keys of the one sort (ties may order differently: the concatenation is not in
    # global id order), and the merge of the preallocated runs equals merged()
    keys_equal = bool(torch.equal(m.ranked[0], key_c))
    final = bufs[rounds[-1][-1][2]] if rounds else bufs[0]
    merge_equals_merged = bool(torch.equal(final[0], m.ranked[0]) and torch.equal(final[1], m.ranked[1]))
    del m
    t = {k: [] for k in ("merge", "merged", "sort_concat")}
    for _ in range(reps):
        t["merge"].append(timed(merge, dev))
        t["sort_concat"].append(timed(sort_concat, dev))
        t["merged"].append(timed(lambda: merged(), dev))
        torch.cuda.synchronize()
    med = {k: float(np.median(v)) for k, v in t.items()}
    spread = {k: [float(min(v)), float(max(v))] for k, v in t.items()}
    n_rounds = len(rounds)
    outs = [run_sizes[o] for pairs in rounds for _, _, o in pairs]
    floor = 16 * sum(outs)
    kernels = 0
    for n in outs:              # + per tile boundary a binary search reading two (key, payload) items per step, the
        tiles = math.ceil(n / SORT_TILE)                 # split written once and read twice
        kernels += 16 * n + (tiles + 1) * (16 * math.ceil(math.log2(n + 1)) + 8) + tiles * 16
    return {
        "parts": parts, "candidates": N, "part_candidates": counts, "rounds": n_rounds,
        "ms_median": med, "ms_min_max": spread, "reps": reps,
        "bytes_floor_merge": floor, "bytes_floor_per_candidate_per_round": 16,
        "bytes_kernels_merge": kernels,
        "merge_floor_ms_at_hbm_reference": floor / (HBM_GBS * 1e9) * 1e3,
        "merge_gbs": kernels / (med["merge"] * 1e-3) / 1e9,
        "merge_floor_over_time_fraction_of_hbm": floor / (med["merge"] * 1e-3) / 1e9 / HBM_GBS,
        "merge_vs_sort_concat": med["merge"] / med["sort_concat"],
        "merged_vs_sort_concat": med["merged"] / med["sort_concat"],
        "checks": {"merged_keys_equal_sort_of_concatenation": keys_equal,
                   "merge_rounds_equal_merged": merge_equals_merged},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parts", type=int, nargs="+", default=[2, 4, 8])
    ap.add_argument("--docs", type=int, nargs="+", default=[1000, 18432])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_rank_merge.py needs a CUDA device")
    dev = torch.device("cuda:0")
    out = {"gpu": gpu_info(), "hbm_gbs_reference": HBM_GBS,
           "timing": "CUDA events around each call; merge, sort_concat and merged alternate in every repetition; "
                     "one device: merged() ranks the parts one after another (under all_gather each rank ranks "
                     "its own part concurrently, and only the merge rounds run after the exchange)",
           "sizes": {}}
    for num_docs in args.docs:
        sizes = synthetic.shard_doc_sizes(num_docs)
        out["sizes"][f"{num_docs}_docs"] = {f"R{p}": one_config(sizes, p, args.reps, dev) for p in args.parts}
        torch.cuda.empty_cache()
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
