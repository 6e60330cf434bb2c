"""Classifier forward (+ backward with --bwd) on P pairs, for profiling the bilinear kernels.
    python scripts/run_classifier.py [pairs] [iters] [--bwd] [--dtype fp32|bf16]

--dtype both [--out PATH] times the bilinear form's two operand types against each other in one process, alternating
them: BilinearFn in fp32 (3xTF32) and on bf16 operands, alone and inside relation_logits, forward and forward +
backward, at 99 312 and 794 496 pairs (the bench's 12-document batch x 16 and x 128), then a GraphHead forward +
backward (loss included) on a 192-document synthetic batch in both classifier dtypes.  CUDA events around ITERS steps
after a warm-up, the median of REPS such windows; per-kernel device times from the library's timing hooks.  Writes one
JSON record (default profiles/r03_classifier_bf16.json) with the GPU's name and power limit read in the same run."""
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gcgcn_b200 import _lib                                   # noqa: E402
from gcgcn_b200.classifier import BilinearFn, relation_logits            # noqa: E402

DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16}


def opt(name, default):
    return sys.argv[sys.argv.index(name) + 1] if name in sys.argv else default


def events_ms(step, iters):
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(iters):
        step()
    ev1.record()
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1) / iters


def kernels(step, iters):
    st = torch.cuda.current_stream().cuda_stream
    torch.cuda.synchronize()
    _lib.timing_begin(st)
    for _ in range(iters):
        step()
    kern = _lib.timing_end(st)
    return {k: {"launches": v[0] / iters, "ms": v[1] / iters} for k, v in sorted(kern.items(), key=lambda kv: -kv[1][1])}


def single(P, iters, bwd, dtype):
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    bili, cls = torch.nn.Bilinear(128, 128, 97).to(dev), torch.nn.Linear(256, 97).to(dev)
    h = torch.tanh(torch.randn(P, 128, device=dev)).requires_grad_(bwd)
    t = torch.tanh(torch.randn(P, 128, device=dev)).requires_grad_(bwd)
    up = torch.randn(P, 97, device=dev)

    def step():
        z = relation_logits(h, t, bili, cls, dtype=dtype)
        if bwd:
            torch.autograd.grad(z, [h, t] + list(bili.parameters()) + list(cls.parameters()), up)

    for _ in range(2):
        step()
    torch.cuda.synchronize()
    ms = events_ms(step, iters)
    flop = 2.0 * P * (128 * 128 * 97 + 256 * 97) * (3 if bwd else 1)
    print(f"{P} pairs, {'fwd+bwd' if bwd else 'fwd'} ({dtype}): {ms:.3f} ms, {flop / ms / 1e9:.1f} TFLOP/s")
    for k, v in kernels(step, iters).items():
        print(f"  {k:40s} {v['launches']:6.1f} launches  {v['ms']:9.4f} ms")


def gpu_identity():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"not read ({e})"
    return name, q


def both(out_path, iters, reps):
    dev = torch.device("cuda:0")
    name, power = gpu_identity()
    rec = {"gpu": name, "power_limit, max_sm_clock": power, "torch": torch.__version__, "iters": iters, "reps": reps,
           "method": "CUDA events around ITERS steps after 3 warm-up steps, median of REPS windows, the fp32 and bf16 "
                     "windows alternating; per-kernel times from gcgcn_timing_begin/end in a separate pass",
           "bilinear": {}, "classifier": {}, "graph_head": {}}
    print(f"{name}, power limit / max SM clock: {power}")
    for P in (99312, 794496):
        torch.manual_seed(0)
        bili, cls = torch.nn.Bilinear(128, 128, 97).to(dev), torch.nn.Linear(256, 97).to(dev)
        h = torch.tanh(torch.randn(P, 128, device=dev)).requires_grad_(True)
        t = torch.tanh(torch.randn(P, 128, device=dev)).requires_grad_(True)
        up = torch.randn(P, 97, device=dev)
        leaves = [h, t, bili.weight, bili.bias]
        allp = [h, t] + list(bili.parameters()) + list(cls.parameters())
        steps = {}
        for key, dt in DTYPES.items():
            steps[("bilinear", "fwd", key)] = lambda dt=dt: BilinearFn.apply(*leaves, dt)
            steps[("bilinear", "fwd+bwd", key)] = lambda dt=dt: torch.autograd.grad(BilinearFn.apply(*leaves, dt), leaves, up)
            steps[("classifier", "fwd", key)] = lambda dt=dt: relation_logits(h, t, bili, cls, dtype=dt)
            steps[("classifier", "fwd+bwd", key)] = lambda dt=dt: torch.autograd.grad(
                relation_logits(h, t, bili, cls, dtype=dt), allp, up)
        for what in ("bilinear", "classifier"):
            for mode in ("fwd", "fwd+bwd"):
                for key in DTYPES:
                    for _ in range(3):
                        steps[(what, mode, key)]()
                torch.cuda.synchronize()
                times = {key: [] for key in DTYPES}
                for _ in range(reps):
                    for key in DTYPES:
                        with torch.no_grad() if mode == "fwd" else torch.enable_grad():
                            times[key].append(events_ms(steps[(what, mode, key)], iters))
                entry = {}
                for key in DTYPES:
                    med = statistics.median(times[key])
                    with torch.no_grad() if mode == "fwd" else torch.enable_grad():
                        kern = kernels(steps[(what, mode, key)], iters)
                    entry[key] = {"ms": med, "ms_all": times[key], "us_per_1k_pairs": 1e3 * med / (P / 1000),
                                  "kernels": kern}
                entry["speedup_bf16"] = entry["fp32"]["ms"] / entry["bf16"]["ms"]
                rec[what].setdefault(str(P), {})[mode] = entry
                print(f"{what:10s} {mode:7s} P {P:6d}: fp32 {entry['fp32']['ms']:8.3f} ms, bf16 {entry['bf16']['ms']:8.3f} ms,"
                      f" x{entry['speedup_bf16']:.2f}")
                for key in DTYPES:
                    for k, v in list(entry[key]["kernels"].items())[:6]:
                        print(f"    {key} {k:36s} {v['launches']:5.1f}  {v['ms']:8.4f} ms")
        del h, t, up, leaves, allp, steps
        torch.cuda.empty_cache()

    # GraphHead forward + backward (loss included) on 192 synthetic documents, fp32 edges, both classifier dtypes
    from gcgcn_b200 import synthetic
    from gcgcn_b200.head import GraphHead, HeadBatch
    wires = [synthetic.make_wire(d) for d in synthetic.make_batch()] * 16
    hb = HeadBatch(wires, dev)
    torch.manual_seed(1)
    head = GraphHead().to(dev).train()
    gen = torch.Generator(device=dev).manual_seed(2)
    ctx = torch.tanh(torch.randn(hb.total_tokens, 128, device=dev, generator=gen)).requires_grad_(True)
    labels = (torch.rand(hb.batch.total_pairs, 97, device=dev, generator=gen) < 0.02).float()
    hsteps = {key: (lambda dt=dt: head(ctx, hb, labels=labels, classifier_dtype=dt)["loss"].sum().backward())
              for key, dt in DTYPES.items()}
    for key in DTYPES:
        for _ in range(3):
            hsteps[key]()
    torch.cuda.synchronize()
    times = {key: [] for key in DTYPES}
    for _ in range(reps):
        for key in DTYPES:
            times[key].append(events_ms(hsteps[key], iters))
    rec["graph_head"] = {"documents": len(wires), "pairs": hb.batch.total_pairs, "entities": hb.batch.total_nodes,
                         "edge_dtype": "fp32", "mode": "train, forward + backward with the loss"}
    for key in DTYPES:
        rec["graph_head"][key] = {"ms": statistics.median(times[key]), "ms_all": times[key],
                                  "kernels": dict(list(kernels(hsteps[key], iters).items())[:12])}
    rec["graph_head"]["speedup_bf16"] = rec["graph_head"]["fp32"]["ms"] / rec["graph_head"]["bf16"]["ms"]
    print(f"GraphHead fwd+bwd, {len(wires)} documents, {hb.batch.total_pairs} pairs: fp32 {rec['graph_head']['fp32']['ms']:.3f} ms,"
          f" bf16 classifier {rec['graph_head']['bf16']['ms']:.3f} ms, x{rec['graph_head']['speedup_bf16']:.2f}")
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(rec, f, indent=1)
    print(f"wrote {out_path}")


if __name__ == "__main__":
    assert torch.cuda.is_available(), "run_classifier.py times the GPU kernels: it needs a CUDA device"
    args = [a for i, a in enumerate(sys.argv[1:], 1)
            if not a.startswith("--") and sys.argv[i - 1] not in ("--dtype", "--out", "--reps")]
    iters = int(args[1]) if len(args) > 1 else 5
    kind = opt("--dtype", "fp32")
    if kind == "both":
        both(opt("--out", os.path.join(ROOT, "profiles", "r03_classifier_bf16.json")), iters, int(opt("--reps", "5")))
    else:
        single(int(args[0]) if args else 99312, iters, "--bwd" in sys.argv, DTYPES[kind])
