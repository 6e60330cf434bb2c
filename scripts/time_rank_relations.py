"""Time the per-relation evaluation (gcgcn_b200/evaluate.py: per_relation, result_at, predictions_at; csrc/rank.cu)
with CUDA events at two sizes of the BASELINE document mix: DocRED-dev size (1000 documents, about 48 M candidates)
and the 6144-document bench shard (about 293 M), R = 97.

Per size, on one evaluator that is already ranked (its sort is not timed):
- `partition`: gcgcn_rank_by_relation alone, into preallocated buffers;
- `curve_relations`: gcgcn_rank_curve_relations alone (no read-back);
- `per_relation`: per_relation() end to end with the partition redone every call (partition, curve, one read-back of
  the (R - 1) x 80-byte results);
- `result_at` and `predictions_at` at the evaluator's own per-relation best-F1 thresholds (selection, and for
  predictions_at the decode of the selected candidates);
- `result`: result() on the same ranked evaluator, for scale (one whole-set curve and its read-back).
The five user-facing calls alternate in every repetition.  Bytes are computed from the shapes, not read from a
hardware counter: `bytes_floor` is what each step must move (partition 20 B per candidate: 4 upsweep + 8 in + 8 out;
curve 8 B: the payload read by the count and the main pass; selection 8 B per candidate in + 8 B per selected out),
`bytes_kernels` what these kernels move (the selection reads key and payload in its count and in its scatter pass:
16 B per candidate + 8 B per selected).  Every working set is far larger than the 126 MB L2.

    python scripts/time_rank_relations.py --out profiles/r03_rank_relations.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from gcgcn_b200 import _lib, synthetic  # noqa: E402
from gcgcn_b200.batch import RaggedBatch  # noqa: E402
from gcgcn_b200.evaluate import RESULT_BYTES, RelationEvaluator  # noqa: E402
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


def one_size(num_docs, reps, dev):
    sizes = synthetic.shard_doc_sizes(num_docs)
    bt = RaggedBatch(sizes, dev)
    gen = torch.Generator(device=dev).manual_seed(num_docs)
    z = torch.randn(bt.total_pairs, R, generator=gen, device=dev) * 4.0
    labels = (torch.rand(bt.total_pairs, R, generator=gen, device=dev) < 0.02).float()
    intrain = (torch.rand(bt.total_pairs, R, generator=gen, device=dev) < 0.5) & (labels > 0.5)
    ev = RelationEvaluator(R, dev)
    ev.add(z, labels, bt, intrain=intrain)
    del z, labels, intrain
    count = ev.count
    ev.result()
    theta = ev.per_relation()["theta"]
    key, pay, _ = ev._ranked
    lib = _lib.load()
    ws = torch.empty(int(lib.gcgcn_rank_relations_ws_bytes(count, R)), dtype=torch.uint8, device=dev)
    rel_key, rel_pay = torch.empty_like(key), torch.empty_like(pay)
    res_buf = torch.empty((R - 1) * RESULT_BYTES, dtype=torch.uint8, device=dev)
    theta_d = torch.full((R - 1,), -1.0, dtype=torch.float64, device=dev)
    st = _stream(dev)

    def partition():
        _lib.call("gcgcn_rank_by_relation", _p(key), _p(pay), count, R, _p(rel_key), _p(rel_pay), _p(ws), ws.numel(),
                  st)

    def curve_relations():
        _lib.call("gcgcn_rank_curve_relations", _p(rel_key), _p(rel_pay), count, R, None, 1, _p(theta_d), _p(res_buf),
                  _p(ws), ws.numel(), st)

    def per_relation():
        ev._by_relation = None                  # the partition is redone, as on a freshly ranked evaluator
        ev.per_relation()

    calls = {"per_relation": per_relation, "result_at": lambda: ev.result_at(theta),
             "predictions_at": lambda: ev.predictions_at(theta), "result": lambda: ev.result()}
    for f in (partition, curve_relations, *calls.values()):     # warm-up: module loads, allocator
        f()
    torch.cuda.synchronize()
    selected = ev.result_at(theta)["count_selected"]
    t = {k: [] for k in ("partition", "curve_relations", *calls)}
    for _ in range(reps):
        t["partition"].append(timed(partition, dev))
        t["curve_relations"].append(timed(curve_relations, dev))
        for k, f in calls.items():
            t[k].append(timed(f, dev))
    med = {k: float(np.median(v)) for k, v in t.items()}
    spread = {k: [float(min(v)), float(max(v))] for k, v in t.items()}
    floor = {"partition": 20 * count, "curve_relations": 8 * count, "selection": 8 * count + 8 * selected}
    floor["per_relation"] = floor["partition"] + floor["curve_relations"]
    kernels = {"partition": 20 * count, "curve_relations": 8 * count, "selection": 16 * count + 8 * selected}
    ms = lambda b: b / (HBM_GBS * 1e9) * 1e3
    return {
        "documents": num_docs, "candidates": count, "candidates_per_relation": count // (R - 1),
        "selected_at_best_f1_thresholds": selected,
        "ms_median": med, "ms_min_max": spread, "reps": reps,
        "bytes_floor": floor, "bytes_kernels": kernels,
        "floor_ms_at_hbm_reference": {k: ms(b) for k, b in floor.items()},
        "kernel_gbs": {"partition": kernels["partition"] / (med["partition"] * 1e-3) / 1e9,
                       "curve_relations": kernels["curve_relations"] / (med["curve_relations"] * 1e-3) / 1e9,
                       "result_at": kernels["selection"] / (med["result_at"] * 1e-3) / 1e9},
        "per_relation_vs_floor": med["per_relation"] / ms(floor["per_relation"]),
        "result_at_vs_floor": med["result_at"] / ms(floor["selection"]),
        "per_relation_vs_result": med["per_relation"] / med["result"],
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--docs", type=int, nargs="+", default=[1000, 6144])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_rank_relations.py needs a CUDA device")
    dev = torch.device("cuda:0")
    out = {"gpu": gpu_info(), "hbm_gbs_reference": HBM_GBS,
           "timing": "CUDA events around each call on an already ranked evaluator; per_relation, result_at, "
                     "predictions_at and result alternate in every repetition; partition and curve_relations are the "
                     "kernels alone into preallocated buffers",
           "sizes": {f"{n}_docs": one_size(n, args.reps, dev) for n in args.docs}}
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
