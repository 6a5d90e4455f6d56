"""FP8 inference, host side: the quantisation mirror on hand-checked values, and the conditions fp8.enable refuses."""
import pytest
import torch

from efficientvlm_b200 import fp8


def _vals(t):
    return t.float().tolist()


def test_e4m3_satfinite_rounds_to_nearest_even_and_saturates():
    x = torch.tensor([449.0, 464.0, 1e6, -1e6, 2.0 ** -10, 3 * 2.0 ** -10, 2.0 ** -9, 3 * 2.0 ** -11, -(2.0 ** -10)])
    # 449 lies between 448 (the largest finite value) and the next step, so it rounds to 448; 464 and beyond saturate instead of giving
    # NaN; 2^-10 is half of the smallest subnormal 2^-9 (a tie: to even, 0); 3 * 2^-10 = 1.5 * 2^-9 is a tie between 2^-9 (odd) and
    # 2^-8 (even); 2^-9 is exact; 0.75 * 2^-9 rounds up to 2^-9
    assert _vals(fp8.e4m3_satfinite(x)) == [448.0, 448.0, 448.0, -448.0, 0.0, 2.0 ** -8, 2.0 ** -9, 2.0 ** -9, -0.0]
    assert torch.isnan(torch.tensor([1e6]).to(torch.float8_e4m3fn).float()).all()   # why the mirror clamps first


def test_quant_rows_reference_hand_checked_rows():
    x = torch.tensor([[448.0, -224.0, 2.0 ** -10, 2.0 ** -9, 3.0],
                      [1.0, 0.5, -0.25, 0.0, 2.0 ** -12],
                      [0.0, 0.0, 0.0, 0.0, 0.0],
                      [-896.0, 449.0, 1.0, 2.0 ** -9, 0.0]])
    q, s = fp8.quant_rows_reference(x)
    assert q.dtype == torch.float8_e4m3fn and s.dtype == torch.float32 and s.shape == (4,)
    # amax 448: inv = 1, scale = 1
    assert _vals(q[0]) == [448.0, -224.0, 0.0, 2.0 ** -9, 3.0] and float(s[0]) == 1.0
    # amax 1: inv = 448, scale = 1/448 (rounded once); 2^-12 * 448 = 0.109375 = 7 * 2^-6 is exact in e4m3
    assert _vals(q[1]) == [448.0, 224.0, -112.0, 0.0, 0.109375]
    assert float(s[1]) == float(torch.tensor(1.0) / torch.tensor(448.0))
    # all-zero row: q = 0, scale = 0
    assert _vals(q[2]) == [0.0] * 5 and float(s[2]) == 0.0
    # amax 896: inv = 0.5, 449 * 0.5 = 224.5 rounds to 224 (e4m3 steps are 16 there); 2^-10 is a tie and rounds to 0
    assert _vals(q[3]) == [-448.0, 224.0, 0.5, 0.0, 0.0] and float(s[3]) == 2.0


def test_quant_rows_reference_bf16_input_and_dequantised_error():
    g = torch.Generator().manual_seed(0)
    x = (torch.randn(7, 2493, generator=g) * torch.logspace(-3, 3, 7)[:, None]).to(torch.bfloat16)
    x[3, 17] = 1e4                         # an outlier sets its row's scale
    q, s = fp8.quant_rows_reference(x)
    deq = q.float() * s[:, None]
    # e4m3 keeps 3 mantissa bits: relative error <= 2^-4 above the normal range, absolute <= 2^-10 * scale below it
    err = (deq - x.float()).abs()
    assert bool((err <= x.float().abs() * 2.0 ** -4 + s[:, None] * 2.0 ** -10).all())
    assert float(q.float().abs().amax()) == 448.0


class _Tiny(torch.nn.Module):
    def __init__(self):
        super().__init__()
        from efficientvlm_b200.eff_vit import CLIPEncoderLayer
        self.layer = CLIPEncoderLayer(128, "quick_gelu", 2, 0.0, 256)


def test_enable_refuses_gated_training_and_cpu_models():
    m = _Tiny().eval()
    with pytest.raises(ValueError, match="materialised"):
        fp8.enable(m)                      # gates not folded into the weights
    m.gates_folded = True
    m.train()
    with pytest.raises(ValueError, match="eval mode"):
        fp8.enable(m)
    m.eval()
    with pytest.raises(ValueError, match="CUDA"):
        fp8.enable(m)                      # CPU parameters: no CPU path
    assert not fp8.enabled(m)
    with pytest.raises(TypeError):
        fp8.enable(object())
