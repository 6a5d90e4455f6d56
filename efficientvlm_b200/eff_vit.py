"""L0-gated CLIP ViT-B/16 image encoder — drop-in for the reference's `efficient_models/eff_vit.py` and its
unmasked twin `models/clip_vit.py` (same classes, constructor arguments, forward signatures, return tuples and
state_dict keys; gates default to None).  The modules only own parameters and routing; all arithmetic runs in the
sm_100a kernels behind `efficientvlm_b200.ops` (no PyTorch fallback).

Reference: /root/reference/efficient_models/eff_vit.py:82-474, /root/reference/models/clip_vit.py:357-393.
"""
from typing import Optional

import torch
from torch import nn

from . import ops


def find_pruneable_heads_and_indices(heads, n_heads, head_size, already_pruned_heads):
    """transformers==4.12.5 modeling_utils helper (removed in 5.x); call sites eff_vit.py:108-110, eff_bert.py:394-396."""
    mask = torch.ones(n_heads, head_size)
    heads = set(heads) - already_pruned_heads
    for head in heads:
        head = head - sum(1 if h < head else 0 for h in already_pruned_heads)
        mask[head] = 0
    mask = mask.view(-1).contiguous().eq(1)
    index = torch.arange(len(mask))[mask].long()
    return heads, index


def prune_linear_layer(layer: nn.Linear, index: torch.LongTensor, dim: int = 0) -> nn.Linear:
    """transformers prune_linear_layer semantics: keep only `index` rows (dim 0) / columns (dim 1)."""
    index = index.to(layer.weight.device)
    W = layer.weight.index_select(dim, index).clone().detach()
    b = None
    if layer.bias is not None:
        b = layer.bias.clone().detach() if dim == 1 else layer.bias[index].clone().detach()
    new_size = list(layer.weight.size())
    new_size[dim] = len(index)
    new_layer = nn.Linear(new_size[1], new_size[0], bias=layer.bias is not None).to(layer.weight.device)
    new_layer.weight.requires_grad = False
    new_layer.weight.copy_(W.contiguous())
    new_layer.weight.requires_grad = True
    if b is not None:
        new_layer.bias.requires_grad = False
        new_layer.bias.copy_(b.contiguous())
        new_layer.bias.requires_grad = True
    return new_layer


class CLIPAttention(nn.Module):
    """Parameter container for the multi-head attention block (eff_vit.py:82-121)."""

    def __init__(self, hidden_size, num_attention_heads, attention_dropout):
        super().__init__()
        self.embed_dim = hidden_size
        self.num_heads = num_attention_heads
        self.head_dim = self.embed_dim // self.num_heads
        assert self.head_dim * self.num_heads == self.embed_dim, (
            f"embed_dim must be divisible by num_heads (got `embed_dim`: {self.embed_dim} and `num_heads`: {self.num_heads}).")
        self.scale = self.head_dim ** -0.5
        self.dropout = attention_dropout
        self.k_proj = nn.Linear(hidden_size, self.embed_dim)
        self.v_proj = nn.Linear(hidden_size, self.embed_dim)
        self.q_proj = nn.Linear(hidden_size, self.embed_dim)
        self.out_proj = nn.Linear(hidden_size, self.embed_dim)
        self.pruned_heads = set()

    def prune_heads(self, heads):
        if len(heads) == 0:
            return
        heads, index = find_pruneable_heads_and_indices(heads, self.num_heads, self.head_dim, self.pruned_heads)
        self.q_proj = prune_linear_layer(self.q_proj, index)
        self.k_proj = prune_linear_layer(self.k_proj, index)
        self.v_proj = prune_linear_layer(self.v_proj, index)
        self.out_proj = prune_linear_layer(self.out_proj, index, dim=1)
        self.num_heads = self.num_heads - len(heads)
        self.embed_dim = self.head_dim * self.num_heads
        self.pruned_heads = self.pruned_heads.union(heads)
        ops.invalidate_weight_cache()


class CLIPMLP(nn.Module):
    def __init__(self, hidden_act, hidden_size, intermediate_size):
        super().__init__()
        if hidden_act != "quick_gelu":
            raise ValueError("the B200 ViT path implements CLIP's quick_gelu only (got %r)" % hidden_act)
        self.hidden_act = hidden_act
        self.fc1 = nn.Linear(hidden_size, intermediate_size)
        self.fc2 = nn.Linear(intermediate_size, hidden_size)


class CLIPEncoderLayer(nn.Module):
    evlm_fp8 = False      # set by fp8.enable: the four projections run in e4m3 (inference only)

    def __init__(self, hidden_size, hidden_act, num_attention_heads, attention_dropout, intermediate_size):
        super().__init__()
        self.self_attn = CLIPAttention(hidden_size, num_attention_heads, attention_dropout)
        self.layer_norm1 = nn.LayerNorm(hidden_size)
        self.mlp = CLIPMLP(hidden_act, hidden_size, intermediate_size)
        self.layer_norm2 = nn.LayerNorm(hidden_size)

    def _params(self):
        a, m = self.self_attn, self.mlp
        return (self.layer_norm1.weight, self.layer_norm1.bias, a.q_proj.weight, a.q_proj.bias, a.k_proj.weight, a.k_proj.bias,
                a.v_proj.weight, a.v_proj.bias, a.out_proj.weight, a.out_proj.bias, self.layer_norm2.weight, self.layer_norm2.bias,
                m.fc1.weight, m.fc1.bias, m.fc2.weight, m.fc2.bias)

    def forward(self, hidden_states, attention_mask=None, output_attentions: Optional[bool] = False, head_z=None, head_layer_z=None,
                mlp_z=None):
        """attention_mask: additive [B,1,N,N] (eff_vit.py:163-169) whose rows are identical (it is built from a per-key
        image mask, :334-341) or an additive key mask [B,N]."""
        B, N, _ = hidden_states.shape
        key_mask = None
        if attention_mask is not None:
            if attention_mask.dim() == 4:
                if attention_mask.size() != (B, 1, N, N):
                    raise ValueError(f"Attention mask should be of size {(B, 1, N, N)}, but is {attention_mask.size()}")
                key_mask = attention_mask[:, 0, 0, :]
            else:
                key_mask = attention_mask
            key_mask = key_mask.to(torch.float32).contiguous()
        a = self.self_attn
        cfg = ops.LayerCfg(a.num_heads, self.layer_norm1.eps, want_probs=bool(output_attentions), training=self.training,
                           attn_dropout=a.dropout, fp8=self.evlm_fp8)
        out, probs = ops.vit_layer(hidden_states, key_mask, head_z, head_layer_z, mlp_z, cfg, self._params())
        outputs = (out,)
        if output_attentions:
            outputs += (probs,)
        return outputs


class CLIPEncoder(nn.Module):
    def __init__(self, hidden_size, hidden_act, num_attention_heads, attention_dropout, intermediate_size, num_hidden_layers,
                 local_attn_depth):
        super().__init__()
        self.depth = num_hidden_layers
        self.local_attn_depth = local_attn_depth
        # extension: a distillation TEACHER only has every k-th attention map read (GeneralDistill.py:91-104 picks teacher
        # layers i*k + k-1); `attention_stride = k` skips materialising the others (their tuple entries are None)
        self.attention_stride = None
        self.layers = nn.ModuleList([CLIPEncoderLayer(hidden_size, hidden_act, num_attention_heads, attention_dropout, intermediate_size)
                                     for _ in range(num_hidden_layers)])

    def forward(self, inputs_embeds, idx_to_group_img=None, image_atts=None, output_attentions=None, output_hidden_states=None,
                head_z=None, head_layer_z=None, mlp_z=None):
        do_gather = idx_to_group_img is not None
        key_mask_blk = None
        if do_gather and (image_atts is not None):                                  # eff_vit.py:334-341
            full_atts = torch.ones(inputs_embeds.shape[:2], dtype=inputs_embeds.dtype, device=inputs_embeds.device)
            blk = torch.cat([image_atts.to(inputs_embeds.dtype), full_atts], dim=0)
            key_mask_blk = (1.0 - blk) * -10000.0                                   # [bs + B, N] additive key mask
        encoder_states = () if output_hidden_states else None
        all_attentions = () if output_attentions else None
        hidden_states = inputs_embeds
        mid_hooks = getattr(self, "_evlm_grad_mid", None)
        for idx, layer in enumerate(self.layers):
            if mid_hooks and idx == mid_hooks[0] and torch.is_grad_enabled() and hidden_states.requires_grad:
                # the input of layer `idx`: once autograd has its gradient, the parameter gradients of layers idx .. depth-1 are final
                # (FlatAdamW.enable_overlap: their exchange starts here, under the backward of the earlier layers)
                callbacks = list(mid_hooks[1])
                hidden_states.register_hook(lambda grad: [cb() for cb in callbacks] and None)
            if output_hidden_states:
                encoder_states = encoder_states + (hidden_states,)
            hz = head_z[idx] if head_z is not None else None
            hlz = head_layer_z[idx] if head_layer_z is not None else None
            mz = mlp_z[idx] if mlp_z is not None else None
            want_att = output_attentions
            if output_attentions and self.attention_stride and (idx % self.attention_stride) != self.attention_stride - 1:
                want_att = None
            if (self.local_attn_depth > 0) and (idx >= self.depth - self.local_attn_depth):
                if do_gather:
                    do_gather = False
                    hs_bs = torch.gather(hidden_states, dim=0, index=idx_to_group_img.view(-1, 1, 1).expand(
                        -1, hidden_states.shape[1], hidden_states.shape[2]))
                    hidden_states = torch.cat([hs_bs, hidden_states], dim=0)
                layer_outputs = layer(hidden_states, attention_mask=key_mask_blk, output_attentions=want_att, head_z=hz,
                                      head_layer_z=hlz, mlp_z=mz)
            else:
                layer_outputs = layer(hidden_states, attention_mask=None, output_attentions=want_att, head_z=hz,
                                      head_layer_z=hlz, mlp_z=mz)
            hidden_states = layer_outputs[0]
            if output_attentions:
                all_attentions = all_attentions + (layer_outputs[1] if want_att else None,)
        if output_hidden_states:
            encoder_states = encoder_states + (hidden_states,)
        return (hidden_states, encoder_states, all_attentions)


class CLIPVisionTransformer(nn.Module):
    def __init__(self, image_size, patch_size, hidden_size, hidden_act, num_attention_heads, attention_dropout, intermediate_size,
                 num_hidden_layers, local_attn_depth=0):
        super().__init__()
        self.image_size = image_size
        self.patch_size = patch_size
        self.num_patch_embed = (self.image_size // self.patch_size) ** 2
        self.patch_embed = nn.Conv2d(in_channels=3, out_channels=hidden_size, kernel_size=self.patch_size, stride=self.patch_size,
                                     bias=False)
        self.class_embedding = nn.Parameter(torch.randn(hidden_size))
        self.num_pos_embed = self.num_patch_embed + 1
        self.pos_embed = nn.Embedding(self.num_pos_embed, hidden_size)
        self.register_buffer("position_ids", torch.arange(self.num_pos_embed).expand((1, -1)))
        self.pre_layrnorm = nn.LayerNorm(hidden_size)  # [sic] reference spelling, part of the checkpoint format
        self.encoder = CLIPEncoder(hidden_size, hidden_act, num_attention_heads, attention_dropout, intermediate_size,
                                   num_hidden_layers, local_attn_depth=local_attn_depth)
        self.post_layernorm = nn.LayerNorm(hidden_size)

    def prune_heads(self, heads_to_prune):
        for layer, heads in heads_to_prune.items():
            self.encoder.layers[layer].self_attn.prune_heads(heads)

    def forward(self, x, idx_to_group_img=None, image_atts=None, output_attentions=None, output_hidden_states=None, head_z=None,
                head_layer_z=None, mlp_z=None):
        hidden_states = ops.vit_embed(x, self.patch_embed.weight, self.class_embedding, self.pos_embed.weight, self.pre_layrnorm.weight,
                                      self.pre_layrnorm.bias, self.pre_layrnorm.eps)
        encoder_outputs = self.encoder(inputs_embeds=hidden_states, idx_to_group_img=idx_to_group_img, image_atts=image_atts,
                                       output_attentions=output_attentions, output_hidden_states=output_hidden_states, head_z=head_z,
                                       head_layer_z=head_layer_z, mlp_z=mlp_z)
        outputs = ops.layer_norm(encoder_outputs[0], self.post_layernorm.weight, self.post_layernorm.bias, self.post_layernorm.eps)
        if getattr(self, "_evlm_grad_ready", None) and torch.is_grad_enabled() and outputs.requires_grad:
            # The image tokens are the first thing the forward produced, so their gradient is the last thing the rest of the model
            # contributes to: when autograd reaches it, every gradient outside the vision tower is final.  FlatAdamW.enable_overlap()
            # uses the moment to start the all-reduce of those gradients on a side stream while the vision tower's backward runs.
            callbacks = list(self._evlm_grad_ready)
            outputs.register_hook(lambda grad: [cb() for cb in callbacks] and None)
        if idx_to_group_img is not None:
            bs = len(idx_to_group_img)
            outputs, outputs_fullatts = torch.split(outputs, [bs, outputs.size(0) - bs])
            return (outputs, encoder_outputs[1], encoder_outputs[2], outputs_fullatts)
        return (outputs, encoder_outputs[1], encoder_outputs[2])
