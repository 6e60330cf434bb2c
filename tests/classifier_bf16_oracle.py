"""Float64 reference of the relation classifier's bilinear form on bf16-rounded operands (gcgcn_bilinear_fwd / _bwd
with dtype GCGCN_BF16, classifier.BilinearFn with torch.bfloat16), restated from the definitions in include/gcgcn_b200.h:

  out[p, r]     = sum_b (sum_a bf16(h[p, a]) bf16(W[r, a, b])) t[p, b] + bias[r]
  dt[p, b]      = sum_r dout[p, r] sum_a bf16(h[p, a]) bf16(W[r, a, b])
  dh[p, a]      = sum_r dout[p, r] sum_b bf16(t[p, b]) bf16(W[r, a, b])
  dW[r, a, b]   = sum_p bf16(h[p, a]) bf16(fp32(dout[p, r] t[p, b]))
  dbias[r]      = sum_p dout[p, r]

bf16(x) rounds an fp32 value to the nearest bf16, ties to even.  Everything after the stated roundings is float64, so
the only difference left between the kernels and this reference is their fp32 accumulation.  The fp32 reference in
oracle/classifier_oracle.py is the same walk over the same chunks: on operands that are already bf16 values the two agree
bit for bit in out, dh and dt.
"""
from __future__ import annotations

import torch

from oracle import classifier_oracle as CO

D = CO.D


def bf16(x: torch.Tensor) -> torch.Tensor:
    """x rounded to fp32, then to the nearest bf16 (ties to even), as float64.  Bit arithmetic on the fp32 pattern,
    independent of torch's own cast (tests/test_classifier_bf16_oracle_cpu.py holds the two against each other);
    finite inputs only (values past the largest bf16 become infinities, as in the hardware rounding)."""
    bits = x.float().contiguous().view(torch.int32).to(torch.int64) & 0xFFFFFFFF
    bits = (bits + 0x7FFF + ((bits >> 16) & 1)) & 0xFFFF0000
    bits = torch.where(bits >= 2 ** 31, bits - 2 ** 32, bits)
    return bits.to(torch.int32).view(torch.float32).double()


def bilinear_bf16(h, t, W, bias=None, dout=None, chunk=CO.CHUNK_ROWS):
    """out [P, R]; with dout [P, R] also (dh, dt, dW [R, 128, 128], dbias [R]), all float64 after the roundings above.
    h, t, W, dout are taken as fp32 values (rounded to fp32 first if they are not)."""
    h32, t32, W32 = h.float(), t.float(), W.float()
    hb, tb, td = bf16(h32), bf16(t32), t32.double()
    P, R = h.shape[0], W.shape[0]
    Wb = bf16(W32)
    Wp, Wpp = CO.wprime(Wb), CO.wsecond(Wb)
    out = hb.new_empty(P, R)
    grads = dout is not None
    if grads:
        d32 = dout.float()
        dd = d32.double()
        dh, dt = torch.empty_like(hb), torch.empty_like(hb)
        dWp = hb.new_zeros(D, R * D)
    for p0 in range(0, P, chunk):
        sl = slice(p0, min(P, p0 + chunk))
        Y = (hb[sl] @ Wp).view(-1, R, D)
        out[sl] = torch.einsum("prb,pb->pr", Y, td[sl])
        if grads:
            dc = dd[sl]
            dt[sl] = torch.einsum("pr,prb->pb", dc, Y)
            del Y
            Z = (tb[sl] @ Wpp).view(-1, R, D)
            dh[sl] = torch.einsum("pr,pra->pa", dc, Z)
            del Z
            G = bf16(d32[sl][:, :, None] * t32[sl][:, None, :])           # the fp32 product, rounded once
            dWp += hb[sl].t() @ G.reshape(-1, R * D)
            del G
        else:
            del Y
    if bias is not None:
        out += bias.double()
    if not grads:
        return out
    dW = torch.stack([dWp[:, r * D:(r + 1) * D] for r in range(R)])
    return out, dh, dt, dW, dd.sum(0)
