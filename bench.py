#!/usr/bin/env python
"""bench.py -- document graphs/s of the fused CAGGC+MAGGC graph blocks (fwd+bwd) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

A "step" is one pass (forward + backward, all gradients) of the graph hot path over one shard of
synthetic DocRED-shaped document graphs that is resident in HBM: BASELINE.json configs[1]
(GCGCN_glove graph blocks, L_s=2, H=8, fp32) with the 12-document batch of SURVEY.md section 8d
(n = 42,35,...,5) tiled --tile times per GPU so that one step streams far more than the 126 MB L2.
With N > 1 every rank owns its own shard (documents are independent: weak scaling, no data-path
collective) and the ranks all-reduce the parameter-gradient bucket once per step (training use).

Prints ONE JSON line (rank 0).  `value` = documents of all ranks / max-over-ranks device time.
`e2e` = the same step driven from pinned HOST buffers: inputs copied host->device and results
device->host inside the timed region.  `roofline` describes the dominant kernel (per-kernel CUDA
events recorded by the library on the launching stream during the timed region) and the whole
path (`path_*`: SURVEY section 8d algorithmic bytes per document / step time).  `cpu_baseline` is
the oracle (CPU restatement of the reference, pinned bit-exact to it) timed on this box's cores.

`aux` holds the separately timed mention->entity pooling and classifier-side pair gathers (SURVEY 8d: own
bytes, own roofline fraction).

    python bench.py --train-docs 100000 [--micro K]     (torchrun for N > 1)
times BASELINE.json configs[4] instead: one pass of doc-sharded training over 100 000 synthetic documents
(forward+backward per micro-batch, ONE NCCL all-reduce of the flat gradient bucket, ONE fused Adam kernel per
optimiser step; strong scaling), see run_training_arm.

--impl reference times that same CPU oracle as its own arm (the reference is PyTorch code that
cannot travel to the GPU box; oracle/gcgcn_oracle.py issues the same ATen ops, see DESIGN.md).
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "document graphs/sec (fwd+bwd graph blocks)"
UNIT = "graphs/s"
VARIANTS = {"glove": (2, 8), "bert": (4, 4)}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps (or calls) of every GPU measurement of the run")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (y1, y2, a0, a1, dx0, de0, "
                         "de1 and every parameter gradient) as DIR/<name>.npy in float32: whole when an array has at "
                         "most 2^20 elements, else a fixed seeded sample of 2^20 of its elements (rank 0's shard)")
    ap.add_argument("--impl", default="gcgcn_b200", choices=["gcgcn_b200", "reference"])
    ap.add_argument("--variant", default="glove", choices=list(VARIANTS))
    ap.add_argument("--dtype", default="fp32", choices=["fp32", "bf16"], help="edge-tensor storage")
    ap.add_argument("--tile", type=int, default=512, help="12-document batches per GPU per step")
    ap.add_argument("--nodes", type=int, default=0, help="configs[3] entity-count sweep: every document has this many "
                                                         "entities (128 / 256 in the sweep); 0 = the DocRED-shaped batch")
    ap.add_argument("--docs", type=int, default=0, help="documents per GPU per step with --nodes (default: 6 GB per edge tensor)")
    ap.add_argument("--heads", type=int, default=0, help="override head_num (4 / 8 in the sweep)")
    ap.add_argument("--graph", action="store_true", help="time CUDA-graph replays of the captured pass instead of eager launches")
    ap.add_argument("--train", action="store_true", help="module.train(): dropout keep-masks drawn by torch every step "
                                                         "(the headline is the dropout-free pass, SURVEY 8d)")
    ap.add_argument("--train-docs", type=int, default=0, help="configs[4]: train over this many synthetic documents "
                    "(100000 in BASELINE.json), sharded by micro-batch over the ranks, one fused Adam step per "
                    "micro-batch per rank after one NCCL all-reduce of the flat gradient bucket; --steps is ignored "
                    "(the timed region is the whole pass over the documents)")
    ap.add_argument("--micro", type=int, default=6252, help="documents per micro-batch per rank with --train-docs")
    ap.add_argument("--no-overlap", action="store_true", help="keep the hop-1 edge pass on the main stream (GraphBlocks(overlap=False))")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-aux", action="store_true", help="skip the separate pooling / pair-gather timings")
    ap.add_argument("--no-sweep", action="store_true", help="skip the configs[2] / configs[3] points of the aux section")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "gcgcn_b200" or args.train_docs):
        ap.error("--dump-outputs applies to the graph-block step of the gcgcn_b200 arm")
    return args


def claim_stdout():
    """Send everything libraries print to stdout (NCCL's version banner, ...) to stderr and return an emit(text)
    that writes to the real stdout: the bench prints exactly ONE line there."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)

    def emit(text: str):
        sys.stdout.flush()
        os.write(real, (text + "\n").encode())
    return emit


# ------------------------------------------------------------------------------- CPU oracle arm
def cpu_oracle_rate(variant: str, seconds: float, max_passes: int = 1000, warmup: int = 1):
    """graphs/s of the CPU oracle, documents one at a time like the reference trainer (C:339),
    fwd+bwd, all host threads."""
    import torch
    from helpers import blocks_state, oracle_blocks
    from gcgcn_b200 import synthetic

    layers, heads = VARIANTS[variant]
    torch.set_num_threads(os.cpu_count() or 1)
    _, state = blocks_state(layers, heads)
    docs = synthetic.make_batch()
    for _ in range(warmup):
        for d in docs:
            oracle_blocks(d, state, layers, heads)
    times = []
    t_end = time.perf_counter() + seconds
    while len(times) < max_passes and (time.perf_counter() < t_end or len(times) < 2):
        t0 = time.perf_counter()
        for d in docs:
            oracle_blocks(d, state, layers, heads)
        times.append(time.perf_counter() - t0)
    med = statistics.median(times)
    return len(docs) / med, {"cores": torch.get_num_threads(), "host_cpus": os.cpu_count(), "passes": len(times),
                             "sample": f"{len(times)} passes over the 12-document batch (SURVEY 8d), "
                                       f"fwd+bwd, one document at a time, median pass {med * 1e3:.1f} ms"}


def cuda_oracle_rate(variant: str, dev, passes: int):
    """SURVEY 8d, config 2: the reference's own PyTorch path on the B200 itself -- the oracle's ATen ops (the same
    calls the reference modules make, pinned bit-exact to them) issued eagerly on `dev`, documents one at a time
    like the reference trainer (C:339), fwd+bwd, inputs resident on the device, CUDA_LAUNCH_BLOCKING unset.
    A reported baseline (about 1000 library launches per document), not a path of this package."""
    import torch
    from helpers import blocks_state, oracle_blocks
    from gcgcn_b200 import synthetic
    import copy

    layers, heads = VARIANTS[variant]
    _, state = blocks_state(layers, heads)
    state = {k: v.to(dev) for k, v in state.items()}
    docs = []
    for d in synthetic.make_batch():
        d = copy.copy(d)
        d.x0, d.e0, d.e1, d.adj = d.x0.to(dev), d.e0.to(dev), d.e1.to(dev), d.adj.to(dev)
        docs.append(d)

    def one_pass():
        for d in docs:
            oracle_blocks(d, state, layers, heads, device=dev)

    one_pass()
    torch.cuda.synchronize(dev)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(passes):
        one_pass()
    ev1.record()
    torch.cuda.synchronize(dev)
    sec = ev0.elapsed_time(ev1) * 1e-3 / passes
    return {"value": len(docs) / sec, "unit": UNIT, "kind": "port on cuda (eager ATen ops of the reference modules)",
            "sample": f"{passes} passes over the 12-document batch, fwd+bwd, one document at a time, "
                      f"{sec * 1e3:.1f} ms per pass (CUDA events)"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    layers, heads = VARIANTS[args.variant]
    import torch
    from helpers import blocks_state, oracle_blocks
    from gcgcn_b200 import synthetic
    torch.set_num_threads(os.cpu_count() or 1)
    _, state = blocks_state(layers, heads)
    docs = synthetic.make_batch()
    for _ in range(max(args.warmup, 1)):
        for d in docs:
            oracle_blocks(d, state, layers, heads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        for d in docs:
            oracle_blocks(d, state, layers, heads)
    dt = time.perf_counter() - t0
    value = args.steps * len(docs) / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"configs[1]: GCGCN_{args.variant} graph blocks fwd+bwd, the 12-document DocRED-shaped "
                               "batch (n=42..5, SURVEY 8d), 12 documents per step on the host cores -- a bounded "
                               "sample of the GPU arm's workload (the same batch x 512 per GPU per step)",
                   "variant": args.variant, "layer_num": layers, "head_num": heads, "docs_per_step": len(docs),
                   "step": "reference arm: one step = one pass over the 12-document batch, one document at a "
                           "time as the reference trainer does (C:339)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                         "sample": "12-document batch per step, fwd+bwd, one document at a time; "
                                   "oracle/gcgcn_oracle.py (same ATen ops as the reference, pinned bit-exact)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def workload_name(args):
    if getattr(args, "nodes", 0):
        return (f"configs[3]: entity-count sweep, fully connected graphs of {args.nodes} entities, "
                f"head_num {args.heads or VARIANTS[args.variant][1]}, graph blocks fwd+bwd")
    return (f"configs[1]: GCGCN_{args.variant} graph blocks fwd+bwd, 12-document DocRED-shaped batch "
            f"(n=42..5, SURVEY 8d) x {args.tile} = {12 * args.tile} documents per GPU per step")


# ------------------------------------------------------------------------------- clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "25"], stdout=self.tmp, stderr=subprocess.DEVNULL)
            atexit.register(self.proc.kill)     # no sampler outlives a run that fails before stop()
        except OSError:
            self.proc = None

    def count(self) -> int:
        try:
            with open(self.tmp.name) as f:
                return sum(1 for _ in f)
        except OSError:
            return 0

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        self.tmp.flush()
        self.tmp.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.tmp.read().splitlines():
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        self.tmp.close()
        os.unlink(self.tmp.name)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


# ------------------------------------------------------------------------------- roofline helpers
def read_peaks():
    """(HBM GB/s, TF32 tensor TFLOP/s, provenance).  MEASURED_PEAKS.json holds a copy bandwidth and a cuBLAS
    bf16 GEMM rate; the projection GEMMs run kind::tf32, whose dense rate is half the bf16 one, so the
    tensor denominator is bf16_tflops_sustained / 2 (the kernels are timed inside a long step)."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            pk = json.load(f)
        return (float(pk["hbm_gbs"]), float(pk.get("bf16_tflops_sustained", pk["bf16_tflops"])) / 2.0,
                "measured (MEASURED_PEAKS.json: hbm_gbs; bf16_tflops_sustained / 2 for kind::tf32)")
    return 6650.0, 1400.0 / 2.0, "fallback (B200_PROFILING.md: 6.65 TB/s; 1.4 PFLOP/s sustained bf16 / 2 for tf32)"


def kernel_bytes(name: str, bt, H: int, L: int, esz: int) -> float:
    """Algorithmic HBM bytes of all launches of one kernel name in one step: every operand once
    (SURVEY 8d for the edge streams; the [rows, H*128] intermediates of the block kernels likewise)."""
    n1, n2, d = bt.total_nodes, bt.total_pairs, 128
    node, slab = n1 * d * 4, n1 * H * d * 4           # one [rows,128] / [rows,H*128] fp32 array
    table = {
        "edge_row_fwd<score+mean>": n2 * d * esz + n2 * 4 + node,             # read e0; write A, ebar
        "edge_row_fwd<mean>": n2 * d * esz + node,                             # read e1; write ebar
        "edge_row_bwd<score+mean>": 2 * n2 * d * esz + n2 * 4 + node,          # read e0, dS, debar; write de0
        "edge_row_bwd<mean>": n2 * d * esz + node,                             # write de1
        # MAGGC block kernels (H heads): read Zx, E, x, q; write Z_(l>0), G, F, P
        "block_fwd<mha>": 2 * slab + 2 * node + slab * (L - 1) / L + 2 * slab + H * n2 * 4,
        "tile_fwd": 2 * slab + 2 * node + slab * (L - 1) / L + 2 * slab + H * n2 * 4,      # the same block on packed tiles
        # read P, Z, G, dF, q; write dZ, dE, dq
        "block_bwd<dq>": H * n2 * 4 + 3 * slab + node + 2 * slab + node,
        # CAGGC block kernels (one head): read A, Zx, E, x; write Z_(l>0), G, F  /  read A, Z, G, dF; write dZ, dE, dS
        "block_fwd<given>": n2 * 4 + 3 * node + node * (L - 1) / L + 2 * node,
        "block_bwd<dS>": n2 * 4 + 3 * node + 2 * node + n2 * 4,
    }
    return float(table.get(name, 0.0))


def kernel_roofline(name, launches, ms, flop, bt, H, L, esz, steps, hbm_peak, tensor_peak):
    """{bound, achieved, peak, unit, frac} of one kernel name over the timed region (or None)."""
    secs = ms * 1e-3
    if secs <= 0:
        return None
    if flop > 0:          # dense projections: 3 TF32 MMA passes per fp32-accurate product
        ach = 3.0 * flop / secs / 1e12
        return {"bound": "tensor", "achieved": ach, "peak": tensor_peak, "unit": "TFLOP/s", "frac": ach / tensor_peak,
                "fp32_equivalent_tflops": flop / secs / 1e12,
                "note": "executed TF32 flops = 3 x 2MNK (hi*hi + hi*lo + lo*hi split for fp32 parity)"}
    kb = kernel_bytes(name, bt, H, L, esz) * steps
    if kb > 0:
        ach = kb / secs / 1e9
        return {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                "bytes_per_launch": kb / max(launches, 1)}
    return None


# ------------------------------------------------------------------------------- pooling / pair gathers
def aux_rates(dev, hbm_peak, tensor_peak, iters, tiles=128):
    """SURVEY 8d: the mention->entity pooling (a1) and the classifier-side pair gathers (a8) are timed apart from
    the graph blocks, each against its own algorithmic bytes.  12-document batch x `tiles`, device-resident,
    CUDA events around `iters` back-to-back calls after 3 warm-up calls (outputs of the gathers are 2.7 GB per
    call at 128 tiles: larger than L2)."""
    import torch
    from gcgcn_b200 import synthetic
    from gcgcn_b200.batch import PairTables, PoolTable, RaggedBatch, node_relative_pos
    from gcgcn_b200.modules import pair_dense, pair_gather, pool_nodes

    docs = synthetic.make_batch() * tiles
    bt = RaggedBatch([d.n for d in docs], dev)
    tab = PoolTable.from_spans([d.spans for d in docs], [d.L for d in docs], device=dev)
    rp12 = [node_relative_pos(d.first_pos) for d in docs[:12]]
    tabs = PairTables(bt, rp12 * tiles, device=dev)
    gen = torch.Generator(device=dev).manual_seed(7)
    ctx = torch.randn(tab.total_tokens, 128, device=dev, generator=gen).requires_grad_(True)
    feat = torch.randn(bt.total_nodes, 404, device=dev, generator=gen).requires_grad_(True)
    dis = torch.randn(21, 20, device=dev, generator=gen).requires_grad_(True)
    dx0 = torch.randn(bt.total_nodes, 128, device=dev, generator=gen)
    dh = torch.randn(bt.total_pairs, 424, device=dev, generator=gen)
    dt = torch.randn(bt.total_pairs, 424, device=dev, generator=gen)

    def clock(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters * 1e-3

    keep = {}

    def pool_f():
        keep["x0"] = pool_nodes(ctx, tab)

    def pool_b():
        torch.autograd.grad(keep["x0"], ctx, dx0, retain_graph=True)

    def pair_f():
        keep["p"] = pair_gather(feat, dis, tabs, bt)

    def pair_b():
        torch.autograd.grad(keep["p"], [feat, dis], [dh, dt], retain_graph=True)

    # the same classifier input without the gathered intermediate: tanh(dense_layer(.)) folded in (SURVEY 8f row 2)
    dense = torch.nn.Linear(424, 128).to(dev)
    dh128, dt128 = dh[:, :128].contiguous(), dt[:, :128].contiguous()

    def dense_f():
        keep["d"] = pair_dense(feat, dense, dis, tabs, bt)

    def dense_b():
        torch.autograd.grad(keep["d"], [feat, dis], [dh128, dt128], retain_graph=True)

    nnz = int(tab.tok_idx_host.size)
    n1, n2 = bt.total_nodes, bt.total_pairs
    touched = int((tab.tok_ptr_host[1:] > tab.tok_ptr_host[:-1]).sum())
    work = {  # SURVEY 8d: B_pool = s*d*(nnz + n) + 8*nnz index bytes; pair gathers write 2*n^2*424*s (+ n*404*s + idx)
        "pool_fwd": (pool_f, 512 * (nnz + n1) + 8 * nnz),
        "pool_bwd": (pool_b, 512 * (nnz + tab.total_tokens) + 8 * nnz),
        "pair_gather_fwd": (pair_f, 2 * n2 * 424 * 4 + n1 * 404 * 4 + 4 * n2 * 4),
        "pair_gather_bwd": (pair_b, 2 * n2 * 424 * 4 + n1 * 404 * 4 + 2 * n2 * 4),
        # writes 2 n^2 128 s (+ node-level projection n 404 s in, n 128 s out); backward reads dout and out, writes dpre
        # and reads it back twice (segmented sums over node rows and over distance rows)
        "pair_dense_fwd": (dense_f, 2 * n2 * 128 * 4 + n1 * (404 + 128) * 4 + 4 * n2 * 4),
        "pair_dense_bwd": (dense_b, 2 * n2 * 128 * 4 * 5 + n1 * (404 + 128) * 4 + 2 * n2 * 4),
    }
    out = {"documents": len(docs), "entities": n1, "pairs": n2, "mention_tokens": nnz, "tokens": tab.total_tokens,
           "tokens_in_a_mention": touched}
    for name, (fn, nbytes) in work.items():
        sec = clock(fn)
        out[name] = {"us": sec * 1e6, "bytes": nbytes, "achieved": nbytes / sec / 1e9, "unit": "GB/s",
                     "frac": nbytes / sec / 1e9 / hbm_peak, "graphs_per_s": len(docs) / sec}
    del keep["p"], keep["d"], dh, dt, dh128, dt128
    torch.cuda.empty_cache()

    # ---- SURVEY 8f row 1: the edge-feature producer (word + sentence attention) on the same 1536 documents ----
    from gcgcn_b200.edgefeat import EdgeFeatures, EdgeTables
    wires = [synthetic.make_wire(d) for d in docs[:12]] * tiles
    etabs = EdgeTables(wires, bt, dev)
    torch.manual_seed(2)
    producer = EdgeFeatures().to(dev)
    x_nodes = torch.tanh(torch.randn(n1, 128, device=dev, generator=gen)).requires_grad_(True)
    de = torch.randn(n2, 128, device=dev, generator=gen)

    def edge_f():
        keep["e"] = producer(0, ctx, x_nodes, dis, etabs)

    def edge_b():
        torch.autograd.grad(keep["e"], [ctx, x_nodes, dis] + list(producer.word_attention[0].parameters()), de,
                            retain_graph=True, allow_unused=True)

    for name, fn, nbytes in (("edge_features_fwd", edge_f, n2 * 512 + etabs.num_tokens * 1024),
                             ("edge_features_bwd", edge_b, n2 * 512 + etabs.num_tokens * 1024)):
        sec = clock(fn)
        out[name] = {"us": sec * 1e6, "bytes": nbytes, "achieved": nbytes / sec / 1e9, "unit": "GB/s",
                     "frac": nbytes / sec / 1e9 / hbm_peak, "graphs_per_s": len(docs) / sec,
                     "active_slots": etabs.num_slots, "active_tokens": etabs.num_tokens,
                     "note": "algorithmic bytes: the [pairs, 128] edge tensor written (fwd) / its gradient read (bwd) once "
                             "+ the active context rows; the reference forms [n, n, S, L, 128] tensors here"}
    del keep["e"], de
    torch.cuda.empty_cache()

    # ---- SURVEY 8f row 2: Bilinear(128,128,97) + Linear(256,97) + the trainer's loss on 256 documents ----
    from gcgcn_b200.classifier import pair_bce_loss, relation_logits
    cdocs = 12 * 16
    cbt = RaggedBatch([d.n for d in docs[:cdocs]], dev)
    P = cbt.total_pairs
    torch.manual_seed(3)
    bili = torch.nn.Bilinear(128, 128, 97).to(dev)
    cls = torch.nn.Linear(256, 97).to(dev)
    fh = torch.tanh(torch.randn(P, 128, device=dev, generator=gen)).requires_grad_(True)
    ft = torch.tanh(torch.randn(P, 128, device=dev, generator=gen)).requires_grad_(True)
    labels = (torch.rand(P, 97, device=dev, generator=gen) < 0.02).float()

    def cls_f():
        keep["z"] = relation_logits(fh, ft, bili, cls)
        keep["loss"] = pair_bce_loss(keep["z"], labels, cbt)

    def cls_b():
        torch.autograd.grad(keep["loss"].sum(), [fh, ft] + list(bili.parameters()) + list(cls.parameters()), retain_graph=True)

    flop = 2.0 * P * (128 * 128 * 97 + 256 * 97)
    for name, fn, mult in (("classifier_fwd", cls_f, 1.0), ("classifier_bwd", cls_b, 3.0)):
        sec = clock(fn)
        out[name] = {"us": sec * 1e6, "pairs": P, "documents": cdocs, "fp32_equivalent_tflops": mult * flop / sec / 1e12,
                     "executed_tf32_tflops": 3.0 * mult * flop / sec / 1e12, "unit": "TFLOP/s",
                     "frac": 3.0 * mult * flop / sec / 1e12 / tensor_peak, "graphs_per_s": cdocs / sec,
                     "note": "forward: ONE tcgen05 pass, h resident in tensor memory per 128-pair tile, W' streamed as pre-split "
                             "blobs, every accumulator tile contracted with t in the epilogue (h W' never stored); backward: "
                             "two row-accumulate passes of the same kernel (dt, dh) + a weight-gradient GEMM whose "
                             "[pairs, 97*128] operand is generated in its producers from t and dout; flops counted: "
                             "2 P (128*128*97 + 256*97), x3 for forward+backward, x3 again for the executed TF32 passes"}
    del keep["z"], keep["loss"]
    torch.cuda.empty_cache()

    # ---- drop-in use (B = 1): the reference's own call sequence (G:330-341) with the drop-in modules, one document at
    # a time like the reference trainer (C:339), fwd+bwd, over the 12-document batch ----
    from gcgcn_b200.modules import GraphBlocks
    torch.manual_seed(0)
    gbm = GraphBlocks(2, 8).to(dev).eval()
    gat, mha, cag, mag = gbm.get_weighted_adj_matrix, gbm.get_adj_matrix[0], gbm.graphcnn[0], gbm.graphcnn[1]
    b1 = []
    for d in docs[:12]:
        b1.append((d.x0.to(dev).requires_grad_(True), d.e0.to(dev).requires_grad_(True), d.e1.to(dev).requires_grad_(True),
                   torch.eq(d.adj.to(dev), 0), torch.randn(d.n, 128, device=dev), torch.randn(d.n, 128, device=dev)))

    def dropin_pass():
        for x, e0_, e1_, mask, g1, g2 in b1:
            a0 = gat(x, e0_, mask)                                   # G:332
            y1 = cag(x, e0_, a0)                                     # G:333
            a1 = mha(y1, e1_)                                        # G:336
            y2 = mag(y1, e1_, a1)                                    # G:337
            torch.autograd.backward([y1, y2], [g1, g2])

    sec = clock(dropin_pass)
    out["dropin_b1"] = {"us_per_document": sec * 1e6 / 12, "graphs_per_s": 12 / sec,
                        "note": "per-document drop-in modules (GATAttention -> GraphConvolution -> MultiHeadAttention -> "
                                "MultiGraphConvolution forward + backward), B = 1 per call, 12 documents one at a time; "
                                "compare cpu_baseline.reference_eager_cuda (the reference's ATen ops on the same GPU)"}
    return out




# ------------------------------------------------------------------------------- configs[2] / configs[3] inside the default run
def graph_block_point(dev, layers, heads, sizes, edge_dtype, hbm_peak, steps, warmup=3):
    """One device-resident measurement of the graph blocks (fwd+bwd, eval mode) on a batch of `sizes` entity counts:
    graphs/s and the whole-path fraction of the HBM roofline (SURVEY 8d algorithmic bytes / step time)."""
    import torch
    from gcgcn_b200.batch import RaggedBatch
    from gcgcn_b200.modules import GraphBlocks
    torch.manual_seed(0)
    gbs = GraphBlocks(layers, heads).to(dev).eval()
    btx = RaggedBatch(sizes, dev)
    gen = torch.Generator(device=dev).manual_seed(7)
    x0 = torch.tanh(torch.randn(btx.total_nodes, 128, device=dev, generator=gen)).requires_grad_(True)
    e0 = torch.randn(btx.total_pairs, 128, device=dev, generator=gen).to(edge_dtype).requires_grad_(True)
    e1 = torch.randn(btx.total_pairs, 128, device=dev, generator=gen).to(edge_dtype).requires_grad_(True)
    dy1 = torch.randn(btx.total_nodes, 128, device=dev, generator=gen)
    dy2 = torch.randn(btx.total_nodes, 128, device=dev, generator=gen)
    ps = [p for n, p in gbs.named_parameters() if "linears_k" not in n]

    def one():
        x0.grad = e0.grad = e1.grad = None
        for p in ps:
            p.grad = None
        out = gbs(x0, e0, e1, btx, with_node_feats=False)
        torch.autograd.backward([out["y1"], out["y2"]], [dy1, dy2])

    for _ in range(warmup):
        one()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        one()
    ev1.record()
    torch.cuda.synchronize()
    sec = ev0.elapsed_time(ev1) * 1e-3 / steps
    esz = 4 if edge_dtype == torch.float32 else 2
    alg = btx.algorithmic_bytes(esz, backward=True)
    res = {"documents": btx.num_docs, "max_entities": btx.max_nodes, "layer_num": layers, "head_num": heads,
           "edge_storage": "fp32" if esz == 4 else "bf16", "ms_per_step": sec * 1e3, "graphs_per_s": btx.num_docs / sec,
           "path_bytes_per_step": alg, "path_achieved_gbs": alg / sec / 1e9, "path_frac": alg / sec / 1e9 / hbm_peak,
           "edge_bytes_per_tensor": btx.total_pairs * 128 * esz}
    del x0, e0, e1, dy1, dy2, gbs
    torch.cuda.empty_cache()
    return res


def sweep_and_variants(dev, hbm_peak, steps, edge_gb=4.0):
    """BASELINE.json configs[3] (entity-count sweep 42/128/256 x 4/8 heads, fully connected, n^2 edge tensors of
    `edge_gb` GB each so that every point streams far more than L2) and configs[2] (the BERT graph head L_s=4, H=4 with
    bf16 edge storage on the DocRED-shaped batch), measured inside the default run so that the driver's record carries
    them."""
    import numpy as np
    import torch
    from gcgcn_b200 import synthetic
    out = {"sweep": [], "note": f"device-resident inputs, CUDA events around {steps} steps after 3 warm-up steps; "
                                "path_frac = SURVEY 8d algorithmic bytes / step time / measured HBM peak"}
    for n in (42, 128, 256):
        for h in (4, 8):
            ndoc = max(1, int(edge_gb * 1e9 // (n * n * 512)))
            r = graph_block_point(dev, 2, h, np.full(ndoc, n, dtype=np.int64), torch.float32, hbm_peak, steps)
            r["workload"] = f"configs[3]: {ndoc} fully connected graphs of {n} entities, {h} heads"
            out["sweep"].append(r)
    r = graph_block_point(dev, 4, 4, synthetic.shard_doc_sizes(12 * 512), torch.bfloat16, hbm_peak, steps)
    r["workload"] = "configs[2]: GCGCN_Bert graph head (L_s=4, H=4), bf16 edge storage, fp32 accumulate, 6144 documents"
    out["config2_bert_bf16"] = r
    r = graph_block_point(dev, 4, 4, synthetic.shard_doc_sizes(12 * 512), torch.float32, hbm_peak, steps)
    r["workload"] = "GCGCN_Bert graph head shapes (L_s=4, H=4), fp32 edge storage, 6144 documents"
    out["bert_head_fp32"] = r
    return out


# ------------------------------------------------------------------------------- end-to-end arm
def run_e2e(args, dev, gb, bt, gb_params, timed, world, ndocs):
    """The e2e leg of run_gpu_arm (see the comment at its call site).  Two complete device-side input sets (context,
    upstream gradients and every index table) are alternated: while step i computes on one, step i+1's inputs are
    copied into the other on a copy stream.  One window = `count` steps and exactly `count` full host->device input
    copies, all inside the window; it closes after the last device->host read."""
    import numpy as np
    import torch
    from gcgcn_b200 import synthetic
    from gcgcn_b200.batch import PoolTable, RaggedBatch
    from gcgcn_b200.edgefeat import EdgeFeatures, EdgeTables
    from gcgcn_b200.modules import pool_nodes
    from gcgcn_b200.sharding import GradBucket

    docs12 = synthetic.make_batch()
    wires12 = [synthetic.make_wire(d) for d in docs12]
    reps = ndocs // 12
    wires = wires12 * reps
    torch.manual_seed(1)
    producer = EdgeFeatures().to(dev)
    producer.train(gb.training)
    dis_embed = torch.randn(21, 20, device=dev).requires_grad_(True)
    params = list(gb_params) + list(producer.parameters()) + [dis_embed]
    bucket = GradBucket(params)

    class Set:
        """one device-side input set + the pinned host buffers it is refilled from"""
        def __init__(self):
            self.bt = RaggedBatch(bt.sizes, dev)
            self.pool = PoolTable.from_spans([d.spans for d in docs12] * reps, [d.L for d in docs12] * reps, device=dev)
            self.edge = EdgeTables(wires, self.bt, dev)
            tok = self.pool.total_tokens
            self.ctx = torch.empty(tok, 128, device=dev)
            self.dy1 = torch.empty(bt.total_nodes, 128, device=dev)
            self.dy2 = torch.empty(bt.total_nodes, 128, device=dev)
            # entities pooled + the producer's active context rows fetched in one pass (one gather, one transpose)
            self.rows = PoolTable.concat(self.pool, self.edge.gather, dev)
            self.tables = [self.bt.node_ptr, self.bt.pair_ptr, self.bt.row_doc, self.bt.doc_order]
            self.tables += [getattr(self.rows, k) for k in ("ent_ptr", "tok_idx", "w", "tok_ptr", "ent_idx", "w_t")]
            self.tables += list(self.edge.dev.values()) + [self.edge.pair_idx, self.edge.pair_denom]

    sets = [Set(), Set()]
    gen = torch.Generator().manual_seed(4242 + int(os.environ.get("RANK", "0")))
    tok = sets[0].pool.total_tokens
    host = {"ctx": torch.tanh(torch.randn(tok, 128, generator=gen)).pin_memory(),
            "dy1": torch.randn(bt.total_nodes, 128, generator=gen).pin_memory(),
            "dy2": torch.randn(bt.total_nodes, 128, generator=gen).pin_memory()}
    host_tables = [t.detach().cpu().pin_memory() for t in sets[0].tables]
    host_out = {k: torch.empty(bt.total_nodes, 128).pin_memory() for k in ("y1", "y2")}
    host_grads = torch.empty(bucket.flat.numel()).pin_memory()
    h2d = sum(t.numel() * t.element_size() for t in host.values()) + sum(t.numel() * t.element_size() for t in host_tables)
    d2h = 2 * bt.total_nodes * 128 * 4 + host_grads.numel() * 4
    copy_stream = torch.cuda.Stream(dev)
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    freed = [torch.cuda.Event(), torch.cuda.Event()]
    window = {"i": 0, "count": 0}

    def stage(sidx):
        st = sets[sidx]
        with torch.cuda.stream(copy_stream), torch.no_grad():
            copy_stream.wait_event(freed[sidx])
            st.ctx.copy_(host["ctx"], non_blocking=True)
            st.dy1.copy_(host["dy1"], non_blocking=True)
            st.dy2.copy_(host["dy2"], non_blocking=True)
            for h, dv in zip(host_tables, st.tables):
                dv.copy_(h, non_blocking=True)
            ready[sidx].record(copy_stream)

    def e2e_step():
        i = window["i"]
        sidx = i % 2
        main = torch.cuda.current_stream(dev)
        if i == 0:
            stage(sidx)
        if i + 1 < window["count"]:
            stage(1 - sidx)                               # next step's inputs: overlaps this step's kernels
        main.wait_event(ready[sidx])
        st = sets[sidx]
        for p in params:
            p.grad = None
        ctx = st.ctx.detach().requires_grad_(True)
        rows = pool_nodes(ctx, st.rows)                                       # G:297-298 + the rows G:300 reads
        x0, act = rows[:bt.total_nodes], rows[bt.total_nodes:]
        e0 = producer(0, None, x0, dis_embed, st.edge, ctx_act=act)           # G:313-326, hop 0
        y1, _ = gb.hop0(x0, e0, st.bt)                                        # G:330-341
        e1 = producer(1, None, y1, dis_embed, st.edge, ctx_act=act)           # hop 1 consumes y1
        y2, _ = gb.hop1(y1, e1, st.bt)
        torch.autograd.backward([y1, y2], [st.dy1, st.dy2])
        bucket.pack()
        if world > 1:
            bucket.all_reduce()
        host_out["y1"].copy_(y1.detach(), non_blocking=True)
        host_out["y2"].copy_(y2.detach(), non_blocking=True)
        host_grads.copy_(bucket.flat, non_blocking=True)
        freed[sidx].record(main)
        window["i"] = i + 1

    def e2e_window(count):
        window.update(i=0, count=count)
        copy_stream.synchronize()
        ms_w, launches, _, _ = timed(e2e_step, count)
        copy_stream.synchronize()
        return ms_w, launches

    e2e_window(3)                                         # warm-up window (pinned pages touched, pools grown)
    steps = args.steps
    ms_e, launches = e2e_window(steps)
    # the same pipeline with the inputs already resident (no copies): what the copies cost on top of the kernels
    def dev_step():
        st = sets[0]
        for p in params:
            p.grad = None
        ctx = st.ctx.detach().requires_grad_(True)
        rows = pool_nodes(ctx, st.rows)
        x0, act = rows[:bt.total_nodes], rows[bt.total_nodes:]
        e0 = producer(0, None, x0, dis_embed, st.edge, ctx_act=act)
        y1, _ = gb.hop0(x0, e0, st.bt)
        e1 = producer(1, None, y1, dis_embed, st.edge, ctx_act=act)
        y2, _ = gb.hop1(y1, e1, st.bt)
        torch.autograd.backward([y1, y2], [st.dy1, st.dy2])
    for _ in range(3):
        dev_step()
    ms_d, _, _, _ = timed(dev_step, steps)
    for p in gb_params:
        p.grad = None
    return {"value": world * ndocs * steps / (ms_e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
            "d2h_bytes_per_step": d2h, "ms_per_step": ms_e / steps, "steps": steps,
            "h2d_gbs": h2d * steps / (ms_e * 1e-3) / 1e9, "gpu_launches_per_step": launches / steps,
            "device_resident_ms_per_step": ms_d / steps,
            "active_slots": sets[0].edge.num_slots, "active_tokens": sets[0].edge.num_tokens, "tokens": tok,
            "wire_bytes_per_doc": sum(w.nbytes for w in wires12) / 12.0,
            "note": "inputs from pinned host memory every step: context_output of all documents (fp32), the upstream "
                    "gradients dy1/dy2 and every index table (batch offsets, pooling CSR, active-slot tables of the "
                    "edge-feature producer); the edge tensors e0/e1 are produced on the device by the producer "
                    "(G:299-327) from context + node features and consumed by CAGGC/MAGGC there; y1, y2 and the "
                    "parameter-gradient bucket (graph blocks + producer) are read back; d loss/d context stays on the "
                    "device (its consumer, the encoder's backward, lives there).  Double-buffered: the copy of step "
                    "i+1 overlaps the kernels of step i; exactly one full input copy per timed step, none staged "
                    "before the window opens; the window closes after the last device->host read."}


# ------------------------------------------------------------------------------- --dump-outputs
DUMP_ELEMENTS = 1 << 20      # 4 MB of float32 per array: the seven step outputs + the parameter gradients stay < 64 MB


def dump_outputs(out_dir: str, arrays: dict):
    """Write every tensor as out_dir/<name>.npy in float32 (float64 stays float64): whole when it has at most
    DUMP_ELEMENTS elements, else its elements at DUMP_ELEMENTS sorted positions drawn by a generator of fixed seed
    (the same positions in every run with the same arguments), flattened."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_ELEMENTS:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_ELEMENTS, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        t = t.to(torch.float64 if t.dtype == torch.float64 else torch.float32)
        np.save(os.path.join(out_dir, f"{name}.npy"), t.cpu().numpy())


# ------------------------------------------------------------------------------- GPU arm
def run_gpu_arm(args):
    import torch
    import torch.distributed as dist
    from gcgcn_b200 import _lib, synthetic
    from gcgcn_b200.batch import RaggedBatch
    from gcgcn_b200.modules import GraphBlocks
    from gcgcn_b200.sharding import GradBucket

    emit = claim_stdout()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; gcgcn_b200 has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL_DEBUG is left as the environment sets it: claim_stdout() already keeps NCCL's banner off stdout
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()

    layers, heads = VARIANTS[args.variant]
    if args.heads:
        heads = args.heads
    edt = torch.float32 if args.dtype == "fp32" else torch.bfloat16
    esz = 4 if args.dtype == "fp32" else 2
    torch.manual_seed(0)
    gb = GraphBlocks(layers, heads, overlap=not args.no_overlap).to(dev).eval()
    if args.train:
        gb.train()
    if args.nodes:
        import numpy as np
        ndoc = args.docs or max(1, int(6e9 // (args.nodes * args.nodes * 128 * (4 if args.dtype == "fp32" else 2))))
        sizes = np.full(ndoc, args.nodes, dtype=np.int64)
    else:
        sizes = synthetic.shard_doc_sizes(12 * args.tile)
    bt = RaggedBatch(sizes, dev)
    ndocs = bt.num_docs

    # synthetic inputs of SURVEY 8d's distribution, generated on the device (seeded per rank)
    gen = torch.Generator(device=dev).manual_seed(1337 + rank)
    x0 = torch.tanh(torch.randn(bt.total_nodes, 128, device=dev, generator=gen)).requires_grad_(True)
    e0 = torch.randn(bt.total_pairs, 128, device=dev, generator=gen).to(edt).requires_grad_(True)
    e1 = torch.randn(bt.total_pairs, 128, device=dev, generator=gen).to(edt).requires_grad_(True)
    dy1 = torch.randn(bt.total_nodes, 128, device=dev, generator=gen)
    dy2 = torch.randn(bt.total_nodes, 128, device=dev, generator=gen)
    params = [p for n, p in gb.named_parameters() if "linears_k" not in n]
    bucket = GradBucket(params)
    overlapped = None
    if world > 1:
        # backward runs MAGGC -> CAGGC: the MAGGC / MultiHeadAttention gradients are final first, and their all-reduce
        # (1.8 of the 2.2 MB) rides a side stream under the CAGGC backward; the CAGGC / GAT bucket follows
        from gcgcn_b200.sharding import OverlappedBuckets
        named = [(n, p) for n, p in gb.named_parameters() if "linears_k" not in n]
        late = [p for n, p in named if n.startswith(("graphcnn.0", "get_weighted_adj_matrix"))]
        early = [p for n, p in named if not n.startswith(("graphcnn.0", "get_weighted_adj_matrix"))]
        overlapped = OverlappedBuckets([early, late])

    def run_step(inp):
        x0_, e0_, e1_, dy1_, dy2_ = inp
        x0_.grad = e0_.grad = e1_.grad = None
        for p in params:
            p.grad = None
        if overlapped is not None:
            overlapped.reset()
        out = gb(x0_, e0_, e1_, bt, with_node_feats=False)      # (the classifier's input; SURVEY 8d times the blocks)
        torch.autograd.backward([out["y1"], out["y2"]], [dy1_, dy2_])
        if overlapped is not None:
            overlapped.finish()
        return out

    def step():
        return run_step((x0, e0, e1, dy1, dy2))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, with_kernel_events=False):
        """(ms, launches, per-kernel table, what the last of the `steps` calls of fn returned)"""
        barrier()
        stream = torch.cuda.current_stream().cuda_stream
        launches0 = _lib.launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if with_kernel_events:
            _lib.timing_begin(stream)
        ev0.record()
        for _ in range(steps - 1):
            fn()
        last = fn()
        ev1.record()
        barrier()
        kern = _lib.timing_end(stream) if with_kernel_events else {}
        ms = ev0.elapsed_time(ev1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, _lib.launch_count() - launches0, kern, last

    # nvidia-smi needs ~1 s to start: the sampler runs from the warm-up steps to the end of the timed region
    sampler = ClockSampler(local) if rank == 0 else None
    for _ in range(max(args.warmup, 3)):
        step()
    # per-kernel breakdown: an eager pass with the library's per-launch events (not the headline)
    ms_eager, launches, kern, _ = timed(step, args.steps, with_kernel_events=True)
    graphed = None
    if args.graph:
        from gcgcn_b200.graphs import GraphedPass
        x0.grad = e0.grad = e1.grad = None
        for p in params:
            p.grad = None

        def fwd_bwd():
            out = gb(x0, e0, e1, bt)
            torch.autograd.backward([out["y1"], out["y2"]], [dy1, dy2])
            return out

        graphed = GraphedPass(fwd_bwd, dev)

        def step():                                   # noqa: F811  (the timed step from here on)
            out = graphed.replay()
            if world > 1:
                bucket.pack()
                bucket.all_reduce()
                bucket.unpack()
            return out

        for _ in range(max(args.warmup, 3)):
            step()
    if sampler is not None:          # keep the GPU under the same load until a few samples exist
        t_wait = time.perf_counter() + 3.0
        while sampler.count() < 3 and time.perf_counter() < t_wait:
            step()
        torch.cuda.synchronize()
    ms, _, _, last = timed(step, args.steps)
    clocks = sampler.stop() if sampler else {}
    if clocks:
        clocks["window"] = "warm-up steps + timed region (same kernels, back to back)"
    value = world * ndocs * args.steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        grads = {"dx0": x0.grad, "de0": e0.grad, "de1": e1.grad}
        grads.update((f"grad.{n}", p.grad) for n, p in gb.named_parameters() if p.grad is not None)
        dump_outputs(args.dump_outputs, {"y1": last["y1"], "y2": last["y2"], "a0": last["a0"], "a1": last["a1"],
                                         **grads})
    del last

    # ---- end to end from pinned host buffers: what the caller of the plugin holds on the host is the encoder output
    # (context_output) and the wire format of the documents; the edge tensors e0/e1 are produced ON the device by the
    # edge-feature producer (G:299-327; they never exist on the host in the model), so one e2e step is
    #   H2D(ctx, upstream gradients, index tables) -> pooling -> producer(hop 0) -> CAGGC -> producer(hop 1) -> MAGGC
    #   -> backward of all of it -> D2H(y1, y2, parameter gradients)
    e2e = None
    if not args.no_e2e and not args.nodes:
        e2e = run_e2e(args, dev, gb, bt, params, timed, world, ndocs)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    hbm_peak, tensor_peak, peak_src = read_peaks()
    step_s = ms * 1e-3 / args.steps
    alg = bt.algorithmic_bytes(esz, backward=True)
    path_gbs = alg / step_s / 1e9
    traffic_tab = {}
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            traffic_tab = json.load(f)
    total_k = sum(v[1] for v in kern.values()) or 1.0
    ranked = sorted(((k, v) for k, v in kern.items() if not k.startswith("(")), key=lambda kv: -kv[1][1])
    breakdown = []
    for k, v in ranked[:30]:
        row = {"kernel": k, "launches": v[0], "ms_per_step": v[1] / args.steps, "share": v[1] / total_k}
        rl = kernel_roofline(k, v[0], v[1], v[2], bt, heads, layers, esz, args.steps, hbm_peak, tensor_peak)
        if rl:
            row.update(bound=rl["bound"], achieved=rl["achieved"], unit=rl["unit"], frac=rl["frac"])
        breakdown.append(row)
    gaps = kern.get("(between calls)", (0, 0.0, 0.0))
    breakdown.append({"kernel": "(time between C-ABI calls: torch packing/autograd glue)", "launches": gaps[0],
                      "ms_per_step": gaps[1] / args.steps, "share": gaps[1] / total_k})
    top = None
    if ranked:
        name, (cnt, tot_ms, flop) = ranked[0]
        rl = kernel_roofline(name, cnt, tot_ms, flop, bt, heads, layers, esz, args.steps, hbm_peak, tensor_peak) or \
            {"bound": "hbm", "achieved": 0.0, "peak": hbm_peak, "unit": "GB/s", "frac": 0.0}
        tr = traffic_tab.get(name)
        traffic = None
        if tr and "dram_bytes_per_step" in tr:      # ncu dram__bytes_read+write of this kernel, same workload
            traffic = tr["dram_bytes_per_step"] * args.steps / max(cnt, 1)
        dom = dict(rl)
        dom.update({"kernel": name, "traffic": traffic, "traffic_source": tr.get("source") if tr else None,
                    "launches_per_step": cnt / args.steps, "us_per_launch": tot_ms * 1e3 / cnt,
                    "share_of_step": tot_ms / total_k,
                    "bytes_model": "every operand of the kernel once, incl. the [rows, H*128] intermediates it reads "
                                   "and writes (NOT SURVEY 8d algorithmic bytes: those are the edge streams' only)"})
        tot = traffic_tab.get("(whole step)")
        traffic_total = tot.get("dram_bytes_per_step") if tot else None
        # headline roofline = the whole hot path: SURVEY 8d algorithmic bytes of one step / step time against the
        # measured HBM peak; the dominant kernel's own (operand-byte) roofline and the per-kernel table explain it
        top = {"bound": "hbm", "achieved": path_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": path_gbs / hbm_peak,
               "traffic": traffic_total, "traffic_total": traffic_total,
               "traffic_source": tot.get("source") if tot else None,
               "scope": "whole step (one pass of the hot path over the shard = one 'launch'): SURVEY 8d algorithmic "
                        "bytes s*d*(5n^2+8n) per document / step time vs the measured HBM peak",
               "path_bytes_per_step": alg, "path_achieved": path_gbs, "path_frac": path_gbs / hbm_peak,
               "peak_source": peak_src,
               "timing": "step: CUDA events around the K timed steps; per-kernel: per-launch CUDA events recorded by "
                         "the library on the launching stream during an eager pass of the same K steps",
               "dominant_kernel": dom, "kernels": breakdown}

    aux = None
    if not args.no_aux and not args.nodes:
        for t in (x0, e0, e1):
            t.grad = None
        aux = aux_rates(dev, hbm_peak, tensor_peak, args.steps)
        if not args.no_sweep and world == 1:
            del x0, e0, e1, dy1, dy2
            torch.cuda.empty_cache()
            aux.update(sweep_and_variants(dev, hbm_peak, args.steps))
    cpu = None
    if not args.no_cpu_baseline:
        rate, info = cpu_oracle_rate(args.variant, args.cpu_seconds)
        cpu = {"value": rate, "unit": UNIT, "cores": info["cores"], "kind": "port", "sample": info["sample"],
               "host_cpus": info["host_cpus"], "reference_eager_cuda": cuda_oracle_rate(args.variant, dev, args.steps)}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32" if args.dtype == "fp32" else "bf16", "data": "synthetic",
        "config": {"workload": workload_name(args), "variant": args.variant, "layer_num": layers, "head_num": heads,
                   "edge_storage": args.dtype, "accumulate": "fp32", "docs_per_gpu": ndocs, "total_nodes": bt.total_nodes,
                   "total_pairs": bt.total_pairs, "parallelism": f"doc-sharded dp{world}",
                   "l2": f"inputs larger than L2: {2 * bt.total_pairs * 128 * esz / 1e9:.2f} GB of edge features "
                         "streamed per step",
                   "collective": "none" if world == 1 else
                                 f"NCCL all-reduce of the {bucket.nbytes} B of parameter gradients per step in two buckets "
                                 "(MAGGC first, issued from a gradient hook on a side stream under the CAGGC backward)",
                   "launch": "eager (one C-ABI call per op)" if graphed is None else
                             "CUDA-graph replay of the captured forward+backward pass (same kernels as eager)",
                   "eager_ms_per_step": ms_eager / args.steps,
                   "dropout": "train mode: keep-masks from torch.rand every step" if args.train else "none (eval)"},
        "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": top, "cpu_baseline": cpu,
        "aux": aux,
    }
    emit(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------- configs[4]: training
def run_training_arm(args):
    """Doc-sharded training pass over --train-docs synthetic documents (BASELINE.json configs[4], SURVEY 8d/8e).

    The documents (n cycling through the 12-value list) are cut into micro-batches of --micro documents; micro-batch
    j belongs to rank j mod N and stays resident in that rank's HBM (1 GPU, 100 000 documents: 53 GB of edge
    features).  One optimiser step = every rank runs forward+backward on its next micro-batch (gradients accumulate
    straight into the flat bucket), ONE NCCL all-reduce of the bucket, ONE fused Adam kernel on every rank (replicated
    parameters stay bit-identical).  Strong scaling: the total work is fixed, `value` = documents / max-over-ranks
    device time of the whole pass.  The loss is the bench's synthetic one (upstream gradients dy1, dy2 drawn once per
    micro-batch): the classifier and its BCE loss are outside the hot path (SURVEY 8f row 2)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from gcgcn_b200 import _lib, synthetic
    from gcgcn_b200.batch import RaggedBatch
    from gcgcn_b200.modules import GraphBlocks
    from gcgcn_b200.sharding import FlatTrainer

    emit = claim_stdout()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; gcgcn_b200 has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()
    layers, heads = VARIANTS[args.variant]
    torch.manual_seed(0)                         # identical initial parameters on every rank
    gb = GraphBlocks(layers, heads).to(dev)
    gb.train() if args.train else gb.eval()
    trainer = FlatTrainer(gb, lr=1e-3)           # optim.Adam(lr) as at config/Config.py:300

    total, k = args.train_docs, max(12, args.micro // 12 * 12)
    n_micro = (total + k - 1) // k
    steps = (n_micro + world - 1) // world
    sizes_all = synthetic.shard_doc_sizes(total)
    mine = [j for j in range(n_micro) if j % world == rank]
    bounds = [(j * k, min(total, (j + 1) * k)) for j in mine]
    batches = {}
    for a, b in bounds:                          # all full micro-batches share one RaggedBatch (k is a multiple of 12)
        if b - a not in batches:
            batches[b - a] = RaggedBatch(sizes_all[a:b], dev)
    nodes = sum(batches[b - a].total_nodes for a, b in bounds)
    pairs = sum(batches[b - a].total_pairs for a, b in bounds)
    gen = torch.Generator(device=dev).manual_seed(1337 + rank)
    x_all = torch.tanh(torch.randn(nodes, 128, device=dev, generator=gen))
    dy1_all = torch.randn(nodes, 128, device=dev, generator=gen)
    dy2_all = torch.randn(nodes, 128, device=dev, generator=gen)
    e0_all = torch.randn(pairs, 128, device=dev, generator=gen)
    e1_all = torch.randn(pairs, 128, device=dev, generator=gen)
    micro, no, po = [], 0, 0
    for a, b in bounds:
        bt = batches[b - a]
        ns, ps = slice(no, no + bt.total_nodes), slice(po, po + bt.total_pairs)
        micro.append((bt, x_all[ns], e0_all[ps], e1_all[ps], dy1_all[ns], dy2_all[ns]))
        no, po = ns.stop, ps.stop
    docs_in_step = [min(total, (s + 1) * world * k) - s * world * k for s in range(steps)]

    def opt_step(s):
        trainer.zero_grad()
        if s < len(micro):
            bt, x, e0, e1, dy1, dy2 = micro[s]
            leaves = [t.detach().requires_grad_(True) for t in (x, e0, e1)]      # dx0, de0, de1 are path outputs
            out = gb(leaves[0], leaves[1], leaves[2], bt)
            torch.autograd.backward([out["y1"], out["y2"]], [dy1, dy2])
        trainer.all_reduce()
        trainer.step(grad_scale=1.0 / docs_in_step[s])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local) if rank == 0 else None
    for _ in range(max(args.warmup, 3)):
        opt_step(0)
    if sampler is not None:
        t_wait = time.perf_counter() + 3.0
        while sampler.count() < 3 and time.perf_counter() < t_wait:
            opt_step(0)
    barrier()
    launches0 = _lib.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for s in range(steps):
        opt_step(s)
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    launches = _lib.launch_count() - launches0
    clocks = sampler.stop() if sampler else {}
    # replicated parameters must still agree bit for bit
    check = trainer.flat_params.double().sum().reshape(1)
    if world > 1:
        lo, hi = check.clone(), check.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        in_sync = bool((lo == hi).item())
        dist.destroy_process_group()
    else:
        in_sync = True
    if rank != 0:
        return
    hbm_peak, _, peak_src = read_peaks()
    alg = int((5 * (sizes_all.astype(np.int64) ** 2).sum() + 8 * sizes_all.sum()) * 128 * 4)
    path_gbs = alg / (ms * 1e-3) / 1e9 / world
    line = {
        "metric": METRIC, "value": total / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"configs[4]: doc-sharded training on {total} synthetic documents (n cycling through "
                               f"SURVEY 8d's 12 values), graph blocks fwd+bwd + gradient all-reduce + fused Adam",
                   "variant": args.variant, "layer_num": layers, "head_num": heads, "edge_storage": "fp32",
                   "micro_batch_docs_per_rank": k, "micro_batches": n_micro, "optimizer_steps": steps,
                   "parallelism": f"doc-sharded dp{world}", "documents_resident_in_hbm_per_rank": sum(b - a for a, b in bounds),
                   "l2": f"every micro-batch streams {2 * batches[min(k, total)].total_pairs * 512 / 1e9:.2f} GB of edge "
                         "features, each document is read once per pass",
                   "collective": "none" if world == 1 else f"one NCCL all-reduce of {trainer.nbytes} B per optimiser step",
                   "optimizer": "Adam(lr=1e-3), one fused kernel over the flat parameter buffer (gcgcn_adam_step)",
                   "parameters_in_sync_after_pass": in_sync,
                   "semantics": "optimizer step per micro-batch, not per document as in the reference (C:368) -- "
                                "inherent to data parallelism (SURVEY 8e)",
                   "dropout": "in-kernel (train mode)" if args.train else "none (eval-mode kernels)"},
        "clocks": clocks, "e2e": None, "gpu_launches": launches,
        "roofline": {"bound": "hbm", "achieved": path_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": path_gbs / hbm_peak,
                     "traffic": None, "kernel": "(whole path, per GPU)", "peak_source": peak_src,
                     "path_note": "SURVEY 8d algorithmic bytes of all documents / pass time / GPUs vs the measured HBM peak"},
        "cpu_baseline": None,
    }
    emit(json.dumps(line))


def main():
    args = parse()
    if args.impl == "reference":
        run_reference_arm(args)
    elif args.train_docs:
        run_training_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
