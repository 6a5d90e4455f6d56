"""FP8 inference for a physically pruned model (e4m3 tensor cores, sm_100a).

`enable(model)` switches the GEMMs that dominate inference to e4m3 x e4m3 products with fp32 accumulation: every projection of the
vision and text / fusion / decoder transformer layers, the LM head transform and the tied vocabulary decoder.  Weights are quantised
once, one fp32 scale per output channel; activations are quantised per token row right before each product (kernels.quant_rows_e4m3,
include/evlm.h).  The patch embedding, attention, LayerNorm, embeddings and the small heads (ITM, pooler, bbox) stay bf16 / fp32.

The FP8 model is a different model from the bf16 one: its outputs equal an fp32 emulation of the same quantised arithmetic, not the
bf16 outputs (tests/test_gpu_fp8.py; scripts/fp8_infer_bench.py measures the agreement with bf16).  It is inference only: a forward
that would need a backward raises.  There is no CPU path.
"""
import torch

from . import ops
from .eff_bert import BertLayer, BertLMPredictionHead, BertPredictionHeadTransform
from .eff_vit import CLIPEncoderLayer


def _weight_groups(m):
    """The (stacked) weights of module m that FP8 covers, one tuple per GEMM operand; None for a module it does not cover."""
    if isinstance(m, CLIPEncoderLayer):
        a, f = m.self_attn, m.mlp
        return [(a.q_proj.weight, a.k_proj.weight, a.v_proj.weight), (a.out_proj.weight,), (f.fc1.weight,), (f.fc2.weight,)]
    if isinstance(m, BertLayer):
        s, o = m.attention.self, m.attention.output
        groups = [(s.query.weight, s.key.weight, s.value.weight), (o.dense.weight,)]
        if m.has_cross_attention:
            xs, xo = m.crossattention.self, m.crossattention.output
            groups += [(xs.query.weight,), (xs.key.weight, xs.value.weight), (xo.dense.weight,)]
        return groups + [(m.intermediate.dense.weight,), (m.output.dense.weight,)]
    if isinstance(m, BertPredictionHeadTransform):
        return [(m.dense.weight,)]
    if isinstance(m, BertLMPredictionHead):
        return [(m.decoder.weight,)]
    return None


def enable(model):
    """Run the covered products of `model` in FP8 from now on.  `model` must have been pruned by prune.materialize (its gates live in
    the weights), be in eval mode and live on a CUDA device.  Returns the model."""
    if not isinstance(model, torch.nn.Module):
        raise TypeError("fp8.enable expects an nn.Module, got %s" % type(model).__name__)
    if not getattr(model, "gates_folded", False):
        raise ValueError("fp8.enable needs a materialised model (prune.materialize): FP8 covers the gate-free inference path only")
    if model.training:
        raise ValueError("fp8.enable needs a model in eval mode: FP8 is inference only (call model.eval() first)")
    params = list(model.parameters())
    if not params or not all(p.is_cuda for p in params):
        raise ValueError("fp8.enable needs the model on a CUDA device: the FP8 kernels have no CPU path")
    covered = [(m, g) for m in model.modules() for g in [_weight_groups(m)] if g is not None]
    if not covered:
        raise ValueError("fp8.enable: the model has no layer FP8 covers")
    for m, groups in covered:
        for ws in groups:
            ops.weight_e4m3(*ws)          # quantised now, not inside a forward that a CUDA graph may be capturing
        m.evlm_fp8 = True
    return model


def e4m3_satfinite(v):
    """fp32 -> e4m3 with round-to-nearest-even and saturation to +-448 (cvt.rn.satfinite.e4m3); torch's own cast gives NaN above 464."""
    return torch.clamp(v, -448.0, 448.0).to(torch.float8_e4m3fn)


def quant_rows_reference(x):
    """Host mirror of kernels.quant_rows_e4m3, bit for bit: (q e4m3 [R, K], scale fp32 [R]) of the rows of x (any device)."""
    x = x.float()
    amax = x.abs().amax(dim=1, keepdim=True)
    nz = amax > 0
    inv = torch.where(nz, torch.full_like(amax, 448.0) / torch.where(nz, amax, torch.ones_like(amax)), torch.zeros_like(amax))
    scale = torch.where(nz, amax / 448.0, torch.zeros_like(amax))
    return e4m3_satfinite(x * inv), scale.squeeze(1)


def enabled(model):
    """True when fp8.enable has switched `model`."""
    return any(getattr(m, "evlm_fp8", False) for m in model.modules())
