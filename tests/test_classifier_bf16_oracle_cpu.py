"""The float64 reference of the bf16 bilinear form (tests/classifier_bf16_oracle.py) on the host: its rounding against
torch's own fp32 -> bf16 cast, its agreement with the fp32 oracle where the roundings change nothing, and the dtype
check of relation_logits.  No GPU needed."""
import pytest
import torch

from classifier_bf16_oracle import bf16, bilinear_bf16
from oracle import classifier_oracle as CO
from gcgcn_b200 import _lib
from gcgcn_b200.classifier import relation_logits


def test_rounding_is_torch_bfloat16():
    """Random magnitudes over the whole fp32 range, subnormals, exact ties (low 16 bits 0x8000) with odd and even
    upper halves, values next to a tie, and the rounding past the largest bf16 into infinity."""
    gen = torch.Generator().manual_seed(5)
    rand = torch.randn(200000, generator=gen) * torch.exp2(torch.randint(-140, 120, (200000,), generator=gen).float())
    hi = torch.randint(0, 0x7F7F, (4096,), generator=gen, dtype=torch.int32) << 16      # finite upper halves
    ties = torch.cat([hi | 0x8000, hi | 0x7FFF, hi | 0x8001, hi | 0x18000, hi]).view(torch.float32)
    special = torch.tensor([0.0, -0.0, 1e-45, -1e-45, 1.1754942e-38, 3.3895314e38, 3.4028235e38, -3.4028235e38, 1.0,
                            1.00390625, 1.005859375, -1.001953125])
    x = torch.cat([rand, ties, -ties, special])
    got = bf16(x)
    want = x.to(torch.bfloat16).double()
    assert torch.equal(got, want)
    assert torch.equal(torch.signbit(got), torch.signbit(want))


@pytest.mark.parametrize("P,R,chunk", [(1, 1, 16), (37, 5, 8), (40, 3, 40)])
def test_equals_the_fp32_oracle_on_bf16_values(P, R, chunk):
    """h, t, W already bf16 values: out, dh, dt and dbias are bitwise those of the fp32 oracle.  dW is not: its
    operand dout * t is rounded to bf16 even so."""
    gen = torch.Generator().manual_seed(P * 10 + R)
    h = torch.tanh(torch.randn(P, 128, generator=gen)).bfloat16().float()
    t = torch.tanh(torch.randn(P, 128, generator=gen)).bfloat16().float()
    W = (torch.randn(R, 128, 128, generator=gen) / 11).bfloat16().float()
    bias = torch.randn(R, generator=gen)
    dout = torch.randn(P, R, generator=gen)
    got = bilinear_bf16(h, t, W, bias, dout, chunk=chunk)
    ref = CO.bilinear(h, t, W, bias, dout, chunk=chunk)
    for k, g, r in zip(("out", "dh", "dt", "dW", "dbias"), got, ref):
        if k != "dW":
            assert torch.equal(g, r), k
    G = bf16(dout[:, :, None] * t[:, None, :])                               # [P, R, 128]
    want_dW = torch.einsum("pa,prb->rab", h.double(), G)
    assert torch.allclose(got[3], want_dW, rtol=1e-12, atol=1e-12)
    assert not torch.equal(got[3], ref[3])                                  # the rounding of dout * t is visible
    assert torch.equal(bilinear_bf16(h, t, W, bias, chunk=chunk), ref[0])


def test_rounds_every_operand_but_t_in_the_forward():
    """The forward rounds h and W but contracts with t unrounded."""
    gen = torch.Generator().manual_seed(3)
    P, R = 9, 2
    h, t = torch.randn(P, 128, generator=gen), torch.randn(P, 128, generator=gen)
    W = torch.randn(R, 128, 128, generator=gen) / 11
    want = torch.einsum("pa,rab,pb->pr", bf16(h), bf16(W), t.double())
    assert torch.allclose(bilinear_bf16(h, t, W), want, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("dtype", [torch.float16, torch.float64, torch.int32])
def test_relation_logits_refuses_other_dtypes(dtype):
    h = t = torch.zeros(4, 128)
    with pytest.raises(_lib.GcgcnError, match="dtype"):
        relation_logits(h, t, torch.nn.Bilinear(128, 128, 97), torch.nn.Linear(256, 97), dtype=dtype)
