"""Time the relation evaluation (gcgcn_b200/evaluate.py) with CUDA events at two sizes of the BASELINE document mix:
DocRED-dev size (1000 documents, about 48 M candidates) and the 6144-document bench shard (about 293 M).

Per size: add() (the candidate kernel), the sort alone, the curve alone (kernels, no read-back), result() on an
unsorted evaluator (sort + curve + the read-back of the result struct) and add() + result() together, alternating
every repetition with torch.sort(stable=True) on the same scores.  Bytes are computed from the shapes, two ways:
`bytes_floor` is the algorithmic floor (candidates read logits and labels once and write 8 bytes per candidate, a sort
moves 16 bytes per candidate in each of its 4 passes of 8-bit digits, the curve reads the 4-byte ranked payloads once);
`bytes_kernels` is what these kernels move (the reduce-then-scan sort reads the keys once more per pass for its
counts: 20 bytes per candidate per pass; the curve reads the payloads twice).  `floor_over_time_fraction_of_hbm` is
the floor over the measured time -- how far from the floor a step is, not the bandwidth the kernels reach; that is
`kernel_gbs`.  Every working set is far larger than the 126 MB L2.

    python scripts/time_rank_eval.py --out profiles/r03_rank_eval.json
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
    count = int((sizes * sizes - sizes).sum()) * (R - 1)

    ev = RelationEvaluator(R, dev)
    ev.add(z, labels, bt)
    ev.result()
    key, pay, ws = ev._ranked
    score, payload = ev._chunks[0]
    res_buf = torch.empty(RESULT_BYTES, dtype=torch.uint8, device=dev)
    st = _stream(dev)

    def sort():
        _lib.call("gcgcn_rank_sort", _p(score), _p(payload), count, _p(key), _p(pay), _p(ws), ws.numel(), st)

    def curve():
        _lib.call("gcgcn_rank_curve", _p(key), _p(pay), count, 0, 0, -1.0, _p(res_buf), _p(ws), ws.numel(), st)

    def add():
        e = RelationEvaluator(R, dev)
        e.add(z, labels, bt)
        return e

    def add_result():
        add().result()

    def result_only(e):
        return lambda: e.result()

    def torch_sort():
        torch.sort(score, descending=True, stable=True)

    for f in (sort, curve, add, add_result, torch_sort):       # warm-up: module loads, allocator, torch's algorithms
        f()
    torch.cuda.synchronize()
    t = {k: [] for k in ("add", "sort", "torch_sort", "curve", "result", "add_result")}
    for _ in range(reps):
        t["sort"].append(timed(sort, dev))
        t["torch_sort"].append(timed(torch_sort, dev))
        t["curve"].append(timed(curve, dev))
        t["add"].append(timed(add, dev))
        e = add()
        torch.cuda.synchronize()
        t["result"].append(timed(result_only(e), dev))
        del e
        t["add_result"].append(timed(add_result, dev))
        t["torch_sort"].append(timed(torch_sort, dev))
    med = {k: float(np.median(v)) for k, v in t.items()}
    spread = {k: [float(min(v)), float(max(v))] for k, v in t.items()}
    b_cand = 2 * 4 * bt.total_pairs * R + 8 * count
    b_sort = 4 * 16 * count
    b_curve = 4 * count
    k_sort, k_curve = 4 * 20 * count, 8 * count
    frac = lambda b, ms: b / (ms * 1e-3) / 1e9 / HBM_GBS
    gbs = lambda b, ms: b / (ms * 1e-3) / 1e9
    return {
        "documents": num_docs, "pairs": bt.total_pairs, "candidates": count,
        "ms_median": med, "ms_min_max": spread, "reps": reps,
        "bytes_floor": {"add": b_cand, "sort": b_sort, "curve": b_curve, "total": b_cand + b_sort + b_curve},
        "bytes_kernels": {"add": b_cand, "sort": k_sort, "curve": k_curve, "total": b_cand + k_sort + k_curve},
        "floor_ms": (b_cand + b_sort + b_curve) / (HBM_GBS * 1e9) * 1e3,
        "floor_over_time_fraction_of_hbm": {"add": frac(b_cand, med["add"]), "sort": frac(b_sort, med["sort"]),
                                            "curve": frac(b_curve, med["curve"]),
                                            "add_result": frac(b_cand + b_sort + b_curve, med["add_result"])},
        "kernel_gbs": {"add": gbs(b_cand, med["add"]), "sort": gbs(k_sort, med["sort"]),
                       "curve": gbs(k_curve, med["curve"])},
        "sort_vs_torch_sort": med["sort"] / med["torch_sort"],
        "add_result_vs_floor": med["add_result"] / ((b_cand + b_sort + b_curve) / (HBM_GBS * 1e9) * 1e3),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_rank_eval.py needs a CUDA device")
    dev = torch.device("cuda:0")
    out = {"gpu": gpu_info(), "hbm_gbs_reference": HBM_GBS,
           "timing": "CUDA events around each call; sort and curve alone reuse one evaluator's buffers, add and result "
                     "allocate like a user's call; torch.sort(stable=True) timed twice per repetition, interleaved",
           "sizes": {"docred_dev_1000_docs": one_size(1000, args.reps, dev),
                     "bench_shard_6144_docs": one_size(6144, args.reps, dev)}}
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
