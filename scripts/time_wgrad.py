"""Device time of the weight-gradient GEMMs C = A^T B (A [K, M], B [K, N], K = every node row of a step), which run on
the MN-major tensor-core route."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gcgcn_b200 import _lib, functional as F  # noqa: E402

dev = torch.device("cuda:0")
K = 119808
st = torch.cuda.current_stream().cuda_stream
for M, N in ((128, 128), (128, 256), (128, 1024), (64, 64)):
    a = torch.randn(K, M, device=dev)
    b = torch.randn(K, N, device=dev)
    ref = None
    for rep in range(6):
        if rep == 3:
            _lib.timing_begin(st)
        out = F.gemm(a, b, True, False)
    t = _lib.timing_end(st)
    ref = a.double().t() @ b.double()
    err = float((out - ref).abs().max()) / float(ref.abs().max())
    tot = sum(v[1] for v in t.values()) / 3
    mb = (a.numel() + b.numel()) * 4 / 1e6
    print(f"M={M} N={N} K={K}: {tot * 1e3:.1f} us per call  ({mb / tot / 1e3:.0f} GB/s of operand bytes)  rel err {err:.2e}  "
          + " ".join(f"{k}:{v[1] / 3 * 1e3:.1f}us" for k, v in t.items()))
