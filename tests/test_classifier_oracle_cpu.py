"""The float64 classifier oracle (oracle/classifier_oracle.py) on the host, against torch's own float64 modules and
autograd: the bilinear form and its gradients (chunked and unchunked), the W' / W'' layouts, the per-document loss
and the per-document bias.  No GPU needed."""
import pytest
import torch
import torch.nn.functional as F

from oracle import classifier_oracle as CO


def close(a, b, tol=1e-12):
    a, b = a.double(), b.double()
    assert a.shape == b.shape, (a.shape, b.shape)
    err = float((a - b).abs().max()) / max(float(b.abs().max()), 1e-300)
    assert err <= tol, f"{err:.3e} > {tol:.0e}"


def test_weight_layouts():
    W = torch.randn(3, 128, 128, dtype=torch.float64)
    Wp, Wpp = CO.wprime(W), CO.wsecond(W)
    assert Wp.shape == Wpp.shape == (128, 3 * 128)
    for r, a, b in ((0, 0, 0), (1, 2, 3), (2, 127, 5), (2, 9, 127)):
        assert Wp[a, r * 128 + b] == W[r, a, b]
        assert Wpp[b, r * 128 + a] == W[r, a, b]


@pytest.mark.parametrize("P,R,chunk", [(1, 1, 16), (7, 3, 16), (37, 5, 8), (40, 2, 40)])
def test_bilinear_matches_torch_autograd(P, R, chunk):
    gen = torch.Generator().manual_seed(P * 10 + R)
    h = torch.randn(P, 128, generator=gen, dtype=torch.float64).requires_grad_(True)
    t = torch.randn(P, 128, generator=gen, dtype=torch.float64).requires_grad_(True)
    W = torch.randn(R, 128, 128, generator=gen, dtype=torch.float64).requires_grad_(True)
    bias = torch.randn(R, generator=gen, dtype=torch.float64).requires_grad_(True)
    dout = torch.randn(P, R, generator=gen, dtype=torch.float64)
    want = F.bilinear(h, t, W, bias)
    (want * dout).sum().backward()
    out, dh, dt, dW, db = CO.bilinear(h.detach(), t.detach(), W.detach(), bias.detach(), dout, chunk=chunk)
    close(out, want.detach())
    close(CO.bilinear(h.detach(), t.detach(), W.detach(), bias.detach(), chunk=chunk), want.detach())
    for got, ref in ((dh, h.grad), (dt, t.grad), (dW, W.grad), (db, bias.grad)):
        close(got, ref)


@pytest.mark.parametrize("R", [1, 4])
def test_pair_bce_matches_torch_autograd(R):
    sizes = [1, 2, 5, 3]
    total = sum(n * n for n in sizes)
    gen = torch.Generator().manual_seed(R)
    z = (torch.randn(total, R, generator=gen, dtype=torch.float64) * 4).clamp(-14.9, 14.9).requires_grad_(True)
    y = (torch.rand(total, R, generator=gen) < 0.3).double()
    dloss = torch.randn(len(sizes), generator=gen, dtype=torch.float64)
    want, lo = [], 0
    for n in sizes:
        per = F.binary_cross_entropy(torch.sigmoid(z[lo:lo + n * n].view(n, n, R)), y[lo:lo + n * n].view(n, n, R),
                                     reduction="none").mean(-1)
        off = ~torch.eye(n, dtype=torch.bool)
        want.append(per[off].sum() / (n * n - n) if n > 1 else per.sum() * 0)
        lo += n * n
    want = torch.stack(want)
    (want * dloss).sum().backward()
    loss, dz = CO.pair_bce(z.detach(), y, sizes, dloss)
    close(loss, want.detach(), 1e-10)
    close(CO.pair_bce(z.detach(), y, sizes), want.detach(), 1e-10)
    close(dz, z.grad, 1e-10)
    assert loss[0] == 0 and (dz[0] == 0).all()


def test_doc_bias_matches_torch_autograd():
    sizes = [1, 3, 2]
    total = sum(n * n for n in sizes)
    gen = torch.Generator().manual_seed(0)
    z = torch.randn(total, 4, generator=gen, dtype=torch.float64)
    v = torch.randn(len(sizes), 4, generator=gen, dtype=torch.float64).requires_grad_(True)
    dz = torch.randn(total, 4, generator=gen, dtype=torch.float64)
    doc = torch.repeat_interleave(torch.arange(len(sizes)), torch.tensor([n * n for n in sizes]))
    want = z + v[doc]
    (want * dz).sum().backward()
    close(CO.doc_bias_fwd(z, v.detach(), sizes), want.detach(), 0.0)
    close(CO.doc_bias_bwd(dz, sizes), v.grad)
