"""L0-gated BERT text / cross-modal fusion encoder and its MLM / causal-LM heads — drop-in for the reference's
`efficient_models/eff_bert.py` and the unmasked twin `models/xbert.py` (same class names, forward signatures, return
structures and state_dict keys; gates default to None).  Modules own parameters and routing only; arithmetic runs in the
sm_100a kernels behind `efficientvlm_b200.ops`.

Reference: /root/reference/efficient_models/eff_bert.py:168-1714 (BertEmbeddings .. BertForMaskedLM).
"""
import json
import math
import os

import torch
import torch.nn.functional as F
from torch import nn

from . import kernels as K
from . import ops
from ._lib import ACT_GELU_ERF
from .eff_vit import find_pruneable_heads_and_indices, prune_linear_layer
GREEDY_SELECT_FUSED = os.environ.get("EVLM_NO_GREEDY_FUSED") is None      # profiling knob: the framework's 17 small launches per token
BEAM_SEARCH_ON_DEVICE = os.environ.get("EVLM_NO_DEVICE_BEAMS") is None    # beam search on CUDA tensors: device loop (off: the host loop)

from .outputs import (BaseModelOutputWithPastAndCrossAttentions, BaseModelOutputWithPoolingAndCrossAttentions,
                      CausalLMOutputWithCrossAttentions, MaskedLMOutput)


class BertConfig:
    """Lightweight equivalent of transformers.BertConfig (bert-base-uncased defaults); a transformers BertConfig works too."""

    def __init__(self, vocab_size=30522, hidden_size=768, num_hidden_layers=12, num_attention_heads=12, intermediate_size=3072,
                 hidden_act="gelu", hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1, max_position_embeddings=512,
                 type_vocab_size=2, initializer_range=0.02, layer_norm_eps=1e-12, pad_token_id=0, position_embedding_type="absolute",
                 **kwargs):
        self.vocab_size = vocab_size
        self.hidden_size = hidden_size
        self.num_hidden_layers = num_hidden_layers
        self.num_attention_heads = num_attention_heads
        self.intermediate_size = intermediate_size
        self.hidden_act = hidden_act
        self.hidden_dropout_prob = hidden_dropout_prob
        self.attention_probs_dropout_prob = attention_probs_dropout_prob
        self.max_position_embeddings = max_position_embeddings
        self.type_vocab_size = type_vocab_size
        self.initializer_range = initializer_range
        self.layer_norm_eps = layer_norm_eps
        self.pad_token_id = pad_token_id
        self.position_embedding_type = position_embedding_type
        self.chunk_size_feed_forward = 0
        self.output_attentions = False
        self.output_hidden_states = False
        self.use_return_dict = True
        self.use_cache = True
        self.is_encoder_decoder = False
        for k, v in kwargs.items():
            setattr(self, k, v)

    @classmethod
    def from_json_file(cls, path):
        with open(path) as f:
            return cls(**json.load(f))

    def to_dict(self):
        return dict(self.__dict__)


class BertEmbeddings(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.word_embeddings = nn.Embedding(config.vocab_size, config.hidden_size, padding_idx=config.pad_token_id)
        self.position_embeddings = nn.Embedding(config.max_position_embeddings, config.hidden_size)
        self.token_type_embeddings = nn.Embedding(config.type_vocab_size, config.hidden_size)
        self.LayerNorm = nn.LayerNorm(config.hidden_size, eps=config.layer_norm_eps)
        self.dropout = nn.Dropout(config.hidden_dropout_prob)
        self.register_buffer("position_ids", torch.arange(config.max_position_embeddings).expand((1, -1)))
        self.position_embedding_type = getattr(config, "position_embedding_type", "absolute")
        if self.position_embedding_type != "absolute":
            raise NotImplementedError("only absolute position embeddings are on the hot path (bert-base-uncased)")
        self.config = config

    def forward(self, input_ids=None, token_type_ids=None, position_ids=None, inputs_embeds=None, past_key_values_length=0):
        if inputs_embeds is not None:
            raise NotImplementedError("inputs_embeds is not used by any EfficientVLM driver; pass input_ids or encoder_embeds")
        p = self.dropout.p if self.training else 0.0
        return ops.bert_embed(input_ids, token_type_ids, position_ids, self.word_embeddings.weight, self.token_type_embeddings.weight,
                              self.position_embeddings.weight, self.LayerNorm.weight, self.LayerNorm.bias, self.LayerNorm.eps, p,
                              past_key_values_length, padding_idx=self.word_embeddings.padding_idx)


class BertSelfAttention(nn.Module):
    """Parameter container (query / key / value) — eff_bert.py:218-264."""

    def __init__(self, config, is_cross_attention):
        super().__init__()
        self.config = config
        if config.hidden_size % config.num_attention_heads != 0 and not hasattr(config, "embedding_size"):
            raise ValueError("The hidden size (%d) is not a multiple of the number of attention heads (%d)"
                             % (config.hidden_size, config.num_attention_heads))
        self.fp16 = getattr(config, "fp16", False)
        self.num_attention_heads = config.num_attention_heads
        self.attention_head_size = int(config.hidden_size / config.num_attention_heads)
        self.all_head_size = self.num_attention_heads * self.attention_head_size
        self.query = nn.Linear(config.hidden_size, self.all_head_size)
        kv_in = config.encoder_width if is_cross_attention else config.hidden_size
        self.key = nn.Linear(kv_in, self.all_head_size)
        self.value = nn.Linear(kv_in, self.all_head_size)
        self.dropout = nn.Dropout(config.attention_probs_dropout_prob)
        self.save_attention = False


class BertSelfOutput(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.dense = nn.Linear(config.hidden_size, config.hidden_size)
        self.LayerNorm = nn.LayerNorm(config.hidden_size, eps=config.layer_norm_eps)
        self.dropout = nn.Dropout(config.hidden_dropout_prob)


class BertAttention(nn.Module):
    def __init__(self, config, is_cross_attention=False):
        super().__init__()
        self.self = BertSelfAttention(config, is_cross_attention)
        self.output = BertSelfOutput(config)
        self.pruned_heads = set()

    def prune_heads(self, heads):
        if len(heads) == 0:
            return
        heads, index = find_pruneable_heads_and_indices(heads, self.self.num_attention_heads, self.self.attention_head_size,
                                                        self.pruned_heads)
        self.self.query = prune_linear_layer(self.self.query, index)
        self.self.key = prune_linear_layer(self.self.key, index)
        self.self.value = prune_linear_layer(self.self.value, index)
        self.output.dense = prune_linear_layer(self.output.dense, index, dim=1)
        self.self.num_attention_heads = self.self.num_attention_heads - len(heads)
        self.self.all_head_size = self.self.attention_head_size * self.self.num_attention_heads
        self.pruned_heads = self.pruned_heads.union(heads)
        ops.invalidate_weight_cache()

    def _params(self):
        s, o = self.self, self.output
        return (s.query.weight, s.query.bias, s.key.weight, s.key.bias, s.value.weight, s.value.bias, o.dense.weight, o.dense.bias,
                o.LayerNorm.weight, o.LayerNorm.bias)


class BertIntermediate(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.dense = nn.Linear(config.hidden_size, config.intermediate_size)
        if config.hidden_act != "gelu":
            raise ValueError("the B200 BERT path implements erf-GELU only (got %r)" % (config.hidden_act,))


class BertOutput(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.dense = nn.Linear(config.intermediate_size, config.hidden_size)
        self.LayerNorm = nn.LayerNorm(config.hidden_size, eps=config.layer_norm_eps)
        self.dropout = nn.Dropout(config.hidden_dropout_prob)


def _key_mask_from_ext(mask):
    """additive [B,1,1,Lk] / [B,Lk] -> contiguous fp32 [B,Lk]."""
    if mask is None:
        return None
    if mask.dim() == 4:
        if mask.shape[1] != 1 or mask.shape[2] != 1:
            raise NotImplementedError("per-query additive masks are expressed through is_decoder (causal) on this path")
        mask = mask[:, 0, 0, :]
    return mask.to(torch.float32).contiguous()


class BertLayer(nn.Module):
    evlm_fp8 = False      # set by fp8.enable: every projection of the layer runs in e4m3 (inference only)

    def __init__(self, config, layer_num):
        super().__init__()
        self.config = config
        self.chunk_size_feed_forward = getattr(config, "chunk_size_feed_forward", 0)
        self.seq_len_dim = 1
        self.attention = BertAttention(config)
        self.has_cross_attention = (layer_num >= config.fusion_layer)
        if self.has_cross_attention:
            self.layer_num = layer_num
            self.crossattention = BertAttention(config, is_cross_attention=True)
        self.intermediate = BertIntermediate(config)
        self.output = BertOutput(config)

    def forward(self, hidden_states, attention_mask=None, head_mask=None, encoder_hidden_states=None, encoder_attention_mask=None,
                past_key_value=None, output_attentions=False, head_z=None, head_layer_z=None, mlp_z=None, causal=False,
                encoder_batch_index=None):
        """attention_mask / encoder_attention_mask: additive key masks ([B,1,1,Lk] or [B,Lk]); `causal` replaces the
        reference's materialised [B,1,L,L] decoder mask (eff_bert.py:976-996).  encoder_batch_index (int32 [B], extension):
        text row b cross-attends to encoder_hidden_states[encoder_batch_index[b]] (== feeding index_select(0, index), with the
        K/V projection computed once per distinct encoder item)."""
        if head_mask is not None:
            raise NotImplementedError("head_mask is always None in EfficientVLM (get_head_mask(None, n))")
        cross_head_z = None
        if self.has_cross_attention and head_z is not None:
            assert isinstance(head_z, tuple)
            head_z, cross_head_z = head_z                                                       # eff_bert.py:494-496
        enc, enc_mask = None, None
        if self.has_cross_attention:
            assert encoder_hidden_states is not None, "encoder_hidden_states must be given for cross-attention layers"
            if type(encoder_hidden_states) == list:                                             # NLVR, eff_bert.py:518-529
                j = (self.layer_num - self.config.fusion_layer) % len(encoder_hidden_states)
                enc, enc_mask = encoder_hidden_states[j], encoder_attention_mask[j]
            else:
                enc, enc_mask = encoder_hidden_states, encoder_attention_mask
        sa = self.attention.self
        cfg = ops.LayerCfg(sa.num_attention_heads, self.output.LayerNorm.eps, want_probs=bool(output_attentions), training=self.training,
                           attn_dropout=sa.dropout.p, hidden_dropout=self.output.dropout.p, causal=causal,
                           has_cross=self.has_cross_attention,
                           cross_heads=self.crossattention.self.num_attention_heads if self.has_cross_attention else 0, fp8=self.evlm_fp8)
        params = self.attention._params()
        if self.has_cross_attention:
            params = params + self.crossattention._params()
        params = params + (self.intermediate.dense.weight, self.intermediate.dense.bias, self.output.dense.weight, self.output.dense.bias,
                           self.output.LayerNorm.weight, self.output.LayerNorm.bias)
        self.mlp_z = mlp_z                                                                      # eff_bert.py:543
        past = past_key_value[:2] if past_key_value is not None else None
        out, probs, probs_x, present = ops.bert_layer(hidden_states, _key_mask_from_ext(attention_mask), enc, _key_mask_from_ext(enc_mask),
                                                      head_z, cross_head_z, mlp_z, past, cfg, params,
                                                      enc_index=encoder_batch_index if self.has_cross_attention else None)
        outputs = (out,)
        if output_attentions:
            outputs = outputs + (probs,)
            if self.has_cross_attention:
                outputs = outputs + (probs_x,)
        return outputs + (present,)


def layer_gate_rows(i, fusion_layer):
    """(self-attention head row, cross-attention head row or None, FFN row) of the gate tensors that BertEncoder.forward hands layer i.
    Quirk Q1 (eff_bert.py:612-620): head gates of fusion layers come in (self, cross) pairs, and in multi_modal mode with concatenated
    gates the fusion layers re-use the *text* slots.  prune.py folds a captioning decoder's gates through the same table."""
    if i >= fusion_layer:
        first = (i - fusion_layer) * 2
        return first, first + 1, i - fusion_layer
    return i, None, i


class BertEncoder(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.config = config
        self.layer = nn.ModuleList([BertLayer(config, i) for i in range(config.num_hidden_layers)])
        self.fusion_layer = self.config.fusion_layer
        # extension (see eff_vit.CLIPEncoder.attention_stride): a distillation teacher materialises only every k-th attention map,
        # counted inside the text part and inside the fusion part; the other tuple entries are None
        self.attention_stride = None

    def forward(self, hidden_states, attention_mask=None, head_mask=None, encoder_hidden_states=None, encoder_attention_mask=None,
                past_key_values=None, use_cache=None, output_attentions=False, output_hidden_states=False, return_dict=True,
                mode="multi_modal", head_z=None, head_layer_z=None, mlp_z=None, causal=False, encoder_batch_index=None):
        all_hidden_states = () if output_hidden_states else None
        all_self_attentions = () if output_attentions else None
        all_cross_attentions = () if output_attentions else None
        next_decoder_cache = () if use_cache else None
        if mode == "text":
            start_layer, output_layer = 0, self.fusion_layer
        elif mode == "fusion":
            start_layer, output_layer = self.fusion_layer, self.config.num_hidden_layers
        elif mode == "multi_modal":
            start_layer, output_layer = 0, self.config.num_hidden_layers
        else:
            raise ValueError(f"mode {mode} is not supported")
        for i in range(start_layer, output_layer):
            layer_module = self.layer[i]
            if output_hidden_states:
                all_hidden_states = all_hidden_states + (hidden_states,)
            if head_z is not None:
                self_row, cross_row, mlp_row = layer_gate_rows(i, self.fusion_layer)
                cur_head_z = head_z[self_row] if cross_row is None else (head_z[self_row], head_z[cross_row])
                cur_mlp_z = mlp_z[mlp_row]
            else:
                cur_mlp_z, cur_head_z = None, None
            past_key_value = past_key_values[i] if past_key_values is not None else None
            want_att = output_attentions
            if output_attentions and self.attention_stride:
                local = i if i < self.fusion_layer else i - self.fusion_layer
                if (local % self.attention_stride) != self.attention_stride - 1:
                    want_att = False
            layer_outputs = layer_module(hidden_states, attention_mask, None, encoder_hidden_states, encoder_attention_mask,
                                         past_key_value, want_att, head_z=cur_head_z if head_z is not None else None,
                                         mlp_z=cur_mlp_z if mlp_z is not None else None, causal=causal,
                                         encoder_batch_index=encoder_batch_index)
            hidden_states = layer_outputs[0]
            if use_cache:
                next_decoder_cache += (layer_outputs[-1],)
            if output_attentions and want_att:
                all_self_attentions = all_self_attentions + (layer_outputs[1],)
                if len(layer_outputs) > 3:
                    all_cross_attentions = all_cross_attentions + (layer_outputs[2],)
            elif output_attentions:
                all_self_attentions = all_self_attentions + (None,)
                if layer_module.has_cross_attention and mode != "text":
                    all_cross_attentions = all_cross_attentions + (None,)
        if output_hidden_states:
            all_hidden_states = all_hidden_states + (hidden_states,)
        if not return_dict:
            return tuple(v for v in [hidden_states, next_decoder_cache, all_hidden_states, all_self_attentions, all_cross_attentions]
                         if v is not None)
        return BaseModelOutputWithPastAndCrossAttentions(last_hidden_state=hidden_states, past_key_values=next_decoder_cache,
                                                         hidden_states=all_hidden_states, attentions=all_self_attentions,
                                                         cross_attentions=all_cross_attentions)


class BertPooler(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.dense = nn.Linear(config.hidden_size, config.hidden_size)
        self.activation = nn.Tanh()

    def forward(self, hidden_states):
        return self.activation(ops.linear(hidden_states[:, 0], self.dense.weight, self.dense.bias))


class BertPredictionHeadTransform(nn.Module):
    evlm_fp8 = False      # set by fp8.enable

    def __init__(self, config):
        super().__init__()
        self.dense = nn.Linear(config.hidden_size, config.hidden_size)
        self.LayerNorm = nn.LayerNorm(config.hidden_size, eps=config.layer_norm_eps)

    def forward(self, hidden_states):
        h = (ops.linear_fp8 if self.evlm_fp8 else ops.linear)(hidden_states, self.dense.weight, self.dense.bias, act=ACT_GELU_ERF)
        return ops.layer_norm(h, self.LayerNorm.weight, self.LayerNorm.bias, self.LayerNorm.eps)


class BertLMPredictionHead(nn.Module):
    evlm_fp8 = False      # set by fp8.enable: the (tied) vocabulary product runs in e4m3

    def __init__(self, config):
        super().__init__()
        self.transform = BertPredictionHeadTransform(config)
        self.decoder = nn.Linear(config.hidden_size, config.vocab_size, bias=False)
        self.bias = nn.Parameter(torch.zeros(config.vocab_size))
        self.decoder.bias = self.bias  # same Parameter under two state_dict names (eff_bert.py:738-741)

    def forward(self, hidden_states):
        return (ops.linear_fp8 if self.evlm_fp8 else ops.linear)(self.transform(hidden_states), self.decoder.weight, self.bias)


class BertOnlyMLMHead(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.predictions = BertLMPredictionHead(config)

    def forward(self, sequence_output):
        return self.predictions(sequence_output)


class BertPreTrainedModel(nn.Module):
    """The slice of transformers.PreTrainedModel the reference relies on: config, weight init, weight tying."""
    config_class = BertConfig
    base_model_prefix = "bert"

    def __init__(self, config):
        super().__init__()
        self.config = config

    @property
    def dtype(self):
        return next(self.parameters()).dtype

    @property
    def device(self):
        return next(self.parameters()).device

    def _init_weights(self, module):                                                    # eff_bert.py:792-802
        if isinstance(module, (nn.Linear, nn.Embedding)):
            module.weight.data.normal_(mean=0.0, std=self.config.initializer_range)
        elif isinstance(module, nn.LayerNorm):
            module.bias.data.zero_()
            module.weight.data.fill_(1.0)
        if isinstance(module, nn.Linear) and module.bias is not None:
            module.bias.data.zero_()

    def init_weights(self):
        self.apply(self._init_weights)
        self.tie_weights()

    def get_output_embeddings(self):
        return None

    def get_input_embeddings(self):
        return None

    def tie_weights(self):
        out, inp = self.get_output_embeddings(), self.get_input_embeddings()
        if out is not None and inp is not None:
            out.weight = inp.weight

    def get_head_mask(self, head_mask, num_hidden_layers, *a, **k):
        if head_mask is not None:
            raise NotImplementedError("head_mask is never used by EfficientVLM")
        return [None] * num_hidden_layers


class BertModel(BertPreTrainedModel):
    def __init__(self, config, add_pooling_layer=True):
        super().__init__(config)
        self.embeddings = BertEmbeddings(config)
        self.encoder = BertEncoder(config)
        self.pooler = BertPooler(config) if add_pooling_layer else None
        self.init_weights()

    def get_input_embeddings(self):
        return self.embeddings.word_embeddings

    def set_input_embeddings(self, value):
        self.embeddings.word_embeddings = value

    def prune_heads(self, heads_to_prune, is_cross=None):                               # eff_bert.py:925-949
        if is_cross == "cross":
            for layer, heads in heads_to_prune.items():
                q, r = layer // 2, layer % 2
                blk = self.encoder.layer[3 + q]
                (blk.attention if r == 0 else blk.crossattention).prune_heads(heads)
        elif is_cross == "decoder":
            for layer, heads in heads_to_prune.items():
                q, r = layer // 2, layer % 2
                blk = self.encoder.layer[q]
                (blk.attention if r == 0 else blk.crossattention).prune_heads(heads)
        else:
            for layer, heads in heads_to_prune.items():
                self.encoder.layer[layer].attention.prune_heads(heads)

    def get_extended_attention_mask(self, attention_mask, input_shape, device, is_decoder):
        """Additive key mask [B,1,1,Lk] = (1 - m) * -10000 (eff_bert.py:1011-1012).  The causal part of the decoder mask
        (:976-996) is NOT materialised: the attention kernel applies `j > i + past -> -10000` itself."""
        if attention_mask.dim() == 3:
            raise NotImplementedError("3-D attention masks are not used by EfficientVLM")
        if attention_mask.dim() != 2:
            raise ValueError("Wrong shape for input_ids (shape {}) or attention_mask (shape {})".format(input_shape, attention_mask.shape))
        ext = attention_mask[:, None, None, :].to(dtype=torch.float32)
        return (1.0 - ext) * -10000.0

    def invert_attention_mask(self, encoder_attention_mask):
        """transformers ModuleUtilsMixin.invert_attention_mask (call site eff_bert.py:1106-1111); additive constant -10000:
        identical to -1e9 / finfo.min after softmax unless a whole row is masked."""
        m = encoder_attention_mask
        ext = m[:, None, None, :] if m.dim() == 2 else m[:, None, :, :]
        return (1.0 - ext.to(torch.float32)) * -10000.0

    def forward(self, input_ids=None, attention_mask=None, token_type_ids=None, position_ids=None, head_mask=None, inputs_embeds=None,
                encoder_embeds=None, encoder_hidden_states=None, encoder_attention_mask=None, past_key_values=None, use_cache=None,
                output_attentions=None, output_hidden_states=None, return_dict=None, is_decoder=False, mode="multi_modal", head_z=None,
                head_layer_z=None, mlp_z=None, encoder_batch_index=None):
        output_attentions = output_attentions if output_attentions is not None else self.config.output_attentions
        output_hidden_states = output_hidden_states if output_hidden_states is not None else self.config.output_hidden_states
        return_dict = return_dict if return_dict is not None else self.config.use_return_dict
        if is_decoder:
            use_cache = use_cache if use_cache is not None else self.config.use_cache
        else:
            use_cache = False
        if input_ids is not None and inputs_embeds is not None:
            raise ValueError("You cannot specify both input_ids and inputs_embeds at the same time")
        elif input_ids is not None:
            input_shape = input_ids.size()
            device = input_ids.device
        elif inputs_embeds is not None:
            input_shape = inputs_embeds.size()[:-1]
            device = inputs_embeds.device
        elif encoder_embeds is not None:
            input_shape = encoder_embeds.size()[:-1]
            device = encoder_embeds.device
        else:
            raise ValueError("You have to specify either input_ids or inputs_embeds or encoder_embeds")
        batch_size, seq_length = input_shape
        past_key_values_length = past_key_values[0][0].shape[2] if past_key_values is not None else 0
        if attention_mask is None:
            attention_mask = torch.ones((batch_size, seq_length + past_key_values_length), device=device)
        extended_attention_mask = self.get_extended_attention_mask(attention_mask, input_shape, device, is_decoder)
        if encoder_hidden_states is not None:
            if type(encoder_hidden_states) == list:
                encoder_batch_size, encoder_sequence_length, _ = encoder_hidden_states[0].size()
            else:
                encoder_batch_size, encoder_sequence_length, _ = encoder_hidden_states.size()
            if type(encoder_attention_mask) == list:
                encoder_extended_attention_mask = [self.invert_attention_mask(mask) for mask in encoder_attention_mask]
            elif encoder_attention_mask is None:
                encoder_extended_attention_mask = None   # all-ones mask == no mask
            else:
                encoder_extended_attention_mask = self.invert_attention_mask(encoder_attention_mask)
        else:
            encoder_extended_attention_mask = None
        self.get_head_mask(head_mask, self.config.num_hidden_layers)
        if encoder_embeds is None:
            embedding_output = self.embeddings(input_ids=input_ids, position_ids=position_ids, token_type_ids=token_type_ids,
                                               inputs_embeds=inputs_embeds, past_key_values_length=past_key_values_length)
        else:
            embedding_output = encoder_embeds
        encoder_outputs = self.encoder(embedding_output, attention_mask=extended_attention_mask, head_mask=None,
                                       encoder_hidden_states=encoder_hidden_states, encoder_attention_mask=encoder_extended_attention_mask,
                                       past_key_values=past_key_values, use_cache=use_cache, output_attentions=output_attentions,
                                       output_hidden_states=output_hidden_states, return_dict=return_dict, mode=mode, head_z=head_z,
                                       head_layer_z=head_layer_z, mlp_z=mlp_z, causal=bool(is_decoder),
                                       encoder_batch_index=encoder_batch_index)
        sequence_output = encoder_outputs[0]
        pooled_output = self.pooler(sequence_output) if self.pooler is not None else None
        if not return_dict:
            return (sequence_output, pooled_output) + tuple(encoder_outputs[1:])
        return BaseModelOutputWithPoolingAndCrossAttentions(last_hidden_state=sequence_output, pooler_output=pooled_output,
                                                            past_key_values=encoder_outputs.past_key_values,
                                                            hidden_states=encoder_outputs.hidden_states,
                                                            attentions=encoder_outputs.attentions,
                                                            cross_attentions=encoder_outputs.cross_attentions)


class LabelSmoothSoftmaxCEV1(nn.Module):
    """eff_bert.py:1263-1302 on the row-softmax CE kernel."""

    def __init__(self, lb_smooth=0.1, reduction="mean", ignore_index=-100):
        super().__init__()
        self.lb_smooth = lb_smooth
        self.reduction = reduction
        self.lb_ignore = ignore_index

    def forward(self, logits, label):
        rows = ops.xent_rows(logits.float(), label, self.lb_ignore, self.lb_smooth)
        if self.reduction == "mean":
            return ops.sum_scaled(rows) / label.ne(self.lb_ignore).sum()
        if self.reduction == "sum":
            return ops.sum_scaled(rows)
        return rows


def cross_entropy(logits, labels, reduction="mean", ignore_index=-100):
    """nn.CrossEntropyLoss semantics (mean over non-ignored rows) on the row-softmax CE kernel."""
    rows = ops.xent_rows(logits, labels, ignore_index, 0.0)
    if reduction == "mean":
        return ops.sum_scaled(rows) / labels.ne(ignore_index).sum()
    if reduction == "sum":
        return ops.sum_scaled(rows)
    return rows


class BertLMHeadModel(BertPreTrainedModel):
    def __init__(self, config, label_smoothing=0.0):
        super().__init__(config)
        self.bert = BertModel(config, add_pooling_layer=False)
        self.cls = BertOnlyMLMHead(config)
        self.label_smoothing = label_smoothing
        self.init_weights()

    def get_output_embeddings(self):
        return self.cls.predictions.decoder

    def set_output_embeddings(self, new_embeddings):
        self.cls.predictions.decoder = new_embeddings

    def get_input_embeddings(self):
        return self.bert.embeddings.word_embeddings

    def forward(self, input_ids=None, attention_mask=None, token_type_ids=None, position_ids=None, head_mask=None, inputs_embeds=None,
                encoder_hidden_states=None, encoder_attention_mask=None, labels=None, past_key_values=None, use_cache=None,
                output_attentions=None, output_hidden_states=None, return_dict=None, is_decoder=True, reduction="mean",
                mode="multi_modal", return_logits=False, head_z=None, mlp_z=None, encoder_batch_index=None):
        """eff_bert.py:1332-1443.  encoder_batch_index (extension, see BertLayer.forward): decoder row r cross-attends to
        encoder_hidden_states[encoder_batch_index[r]]."""
        return_dict = return_dict if return_dict is not None else self.config.use_return_dict
        if labels is not None:
            use_cache = False
        outputs = self.bert(input_ids, attention_mask=attention_mask, token_type_ids=token_type_ids, position_ids=position_ids,
                            head_mask=head_mask, inputs_embeds=inputs_embeds, encoder_hidden_states=encoder_hidden_states,
                            encoder_attention_mask=encoder_attention_mask, past_key_values=past_key_values, use_cache=use_cache,
                            output_attentions=output_attentions, output_hidden_states=output_hidden_states, return_dict=return_dict,
                            is_decoder=is_decoder, mode=mode, head_z=head_z, mlp_z=mlp_z, encoder_batch_index=encoder_batch_index)
        sequence_output = outputs[0]
        prediction_scores = self.cls(sequence_output)
        if return_logits:
            return prediction_scores[:, :-1, :].contiguous()
        lm_loss = None
        if labels is not None:
            # next-token prediction (eff_bert.py:1419-1430): instead of slicing the logits, shift the labels left and ignore the
            # last position — identical loss, no [B, L-1, V] copy.
            B, L, V = prediction_scores.shape
            shifted = torch.full_like(labels, -100)
            shifted[:, :-1] = labels[:, 1:]
            flat_logits, flat_labels = prediction_scores.view(-1, V), shifted.reshape(-1)
            if self.label_smoothing > 0:
                lm_loss = LabelSmoothSoftmaxCEV1(lb_smooth=self.label_smoothing, reduction=reduction)(flat_logits, flat_labels)
            else:
                lm_loss = cross_entropy(flat_logits, flat_labels, reduction=reduction)
            if reduction == "none":
                lm_loss = lm_loss.view(B, L)[:, :-1].sum(1)
        if not return_dict:
            output = (prediction_scores,) + tuple(outputs[2:])
            return ((lm_loss,) + output) if lm_loss is not None else output
        return CausalLMOutputWithCrossAttentions(loss=lm_loss, logits=prediction_scores, past_key_values=outputs.past_key_values,
                                                 hidden_states=outputs.hidden_states, attentions=outputs.attentions,
                                                 cross_attentions=outputs.cross_attentions)

    def prepare_inputs_for_generation(self, input_ids, past=None, attention_mask=None, **model_kwargs):
        input_shape = input_ids.shape
        if attention_mask is None:
            attention_mask = input_ids.new_ones(input_shape)
        if past is not None:
            input_ids = input_ids[:, -1:]
        return {"input_ids": input_ids, "attention_mask": attention_mask, "past_key_values": past,
                "encoder_hidden_states": model_kwargs.get("encoder_hidden_states", None),
                "encoder_attention_mask": model_kwargs.get("encoder_attention_mask", None), "is_decoder": True,
                "head_z": model_kwargs.get("head_z", None), "mlp_z": model_kwargs.get("mlp_z", None)}

    def _reorder_cache(self, past, beam_idx):
        return tuple(tuple(s.index_select(0, beam_idx) for s in layer_past) for layer_past in past)

    @torch.no_grad()
    def _generate_no_beam_search(self, input_ids, cur_len, max_length, do_sample, temperature, top_k, top_p, repetition_penalty,
                                 pad_token_id, eos_token_ids, batch_size, sync_free=False, **model_kwargs):
        """Greedy / sampling decode loop with KV cache (eff_bert.py:1472-1563).
        sync_free=True (extension): always run to max_length instead of asking the host after every token whether all sentences
        have ended.  The result is identical (finished sentences only receive padding, their log-probabilities stop accumulating,
        and the final end-of-sequence fill is a no-op for them), and the loop contains no device->host read, so a caller can capture
        the whole decode in one CUDA graph."""
        unfinished_sents = []
        cur_unfinished = input_ids.new(batch_size).fill_(1)
        logprobs = []
        past = None
        while cur_len < max_length:
            model_inputs = self.prepare_inputs_for_generation(input_ids, past=past, **model_kwargs)
            outputs = self(**model_inputs, return_dict=True, use_cache=True)
            past = outputs.past_key_values
            next_token_logits = outputs.logits[:, -1, :]
            if repetition_penalty != 1.0:
                for i in range(batch_size):
                    for previous_token in set(input_ids[i].tolist()):
                        if next_token_logits[i, previous_token] < 0:
                            next_token_logits[i, previous_token] *= repetition_penalty
                        else:
                            next_token_logits[i, previous_token] /= repetition_penalty
            fused = (not do_sample and next_token_logits.is_cuda and next_token_logits.dtype == torch.float32
                     and cur_unfinished.dtype == torch.int64 and len(eos_token_ids) <= 4 and GREEDY_SELECT_FUSED)
            if fused:
                # argmax, its log-softmax score, the padded token and the end-of-sequence bookkeeping below in ONE launch
                next_token, _scores, tokens_to_add, next_unfinished = K.greedy_select(next_token_logits, cur_unfinished, pad_token_id,
                                                                                      eos_token_ids)
            elif do_sample:
                if temperature != 1.0:
                    next_token_logits = next_token_logits / temperature
                next_token_logits = top_k_top_p_filtering(next_token_logits, top_k=top_k, top_p=top_p)
                next_token = torch.multinomial(F.softmax(next_token_logits, dim=-1), num_samples=1).squeeze(1)
            else:
                next_token = torch.argmax(next_token_logits, dim=-1)
            if not fused:
                _scores = F.log_softmax(next_token_logits, dim=-1)
                _scores = torch.gather(_scores, -1, next_token.unsqueeze(-1))
                tokens_to_add = next_token * cur_unfinished + pad_token_id * (1 - cur_unfinished)
            logprobs.append(_scores)
            unfinished_sents.append(cur_unfinished)
            input_ids = torch.cat([input_ids, tokens_to_add.unsqueeze(-1)], dim=-1)
            if model_kwargs.get("attention_mask", None) is not None:
                am = model_kwargs["attention_mask"]
                model_kwargs["attention_mask"] = torch.cat([am, am.new_ones((am.shape[0], 1))], dim=-1)
            cur_len = cur_len + 1
            if fused:
                cur_unfinished = next_unfinished
            else:
                for eos_token_id in eos_token_ids:
                    cur_unfinished = cur_unfinished.mul(tokens_to_add.ne(eos_token_id).long())
            if not sync_free and cur_unfinished.max() == 0:
                break
        if cur_len == max_length:
            input_ids[:, -1].masked_fill_(cur_unfinished.to(dtype=torch.bool), eos_token_ids[0])
        logprobs = torch.cat(logprobs, dim=1)
        unfinished_sents = torch.stack(unfinished_sents, dim=1).float()
        sum_logprobs = (logprobs * unfinished_sents).sum(dim=1)
        logprobs = sum_logprobs / unfinished_sents.sum(dim=1)
        pad_len = max_length - input_ids.shape[1]
        if pad_len > 0:
            padding_ids = input_ids.new(batch_size, pad_len).fill_(pad_token_id)
            input_ids = torch.cat([input_ids, padding_ids], dim=1)
        return input_ids, logprobs

    @torch.no_grad()
    def _beam_search(self, input_ids, num_beams, max_length, min_length, repetition_penalty, pad_token_id, eos_token_id,
                     length_penalty=1.0, early_stopping=False, **model_kwargs):
        """Beam search as the reference's captioning evaluation runs it (model_generation.py:474-483 -> transformers 4.12.5
        `GenerationMixin.generate` / `beam_search` with `BeamSearchScorer`; third-party code that is not under /root/reference: its
        published algorithm is restated here and in oracle/beam_search_oracle.py, parity unpinned).  Like there, `input_ids` holds one
        prompt per item and is expanded `num_beams` times here, while encoder states in `model_kwargs` arrive already expanded
        (model_generation.py:421-423).  Device side per step: one decoder forward with KV cache, log-softmax, the min-length /
        repetition-penalty processors, top 2 * num_beams over (beam, token), cache re-ordering; the hypothesis bookkeeping is the
        scorer's host loop over those 2 * num_beams candidates per item (one device -> host read per step)."""
        batch = input_ids.shape[0]
        dev = input_ids.device
        input_ids = input_ids.repeat_interleave(num_beams, dim=0)                     # _expand_inputs_for_generation
        if model_kwargs.get("attention_mask", None) is not None:
            model_kwargs["attention_mask"] = model_kwargs["attention_mask"].repeat_interleave(num_beams, dim=0)
        enc = model_kwargs.get("encoder_hidden_states", None)
        if enc is not None and not isinstance(enc, list) and enc.shape[0] != batch * num_beams:
            raise ValueError("encoder_hidden_states must hold batch * num_beams items (the caller expands them: model_generation.py:421-423)")
        hyps = [{"beams": [], "worst": 1e9} for _ in range(batch)]
        done = [False] * batch
        beam_scores = torch.zeros(batch, num_beams, dtype=torch.float32, device=dev)
        beam_scores[:, 1:] = -1e9
        beam_scores = beam_scores.view(-1)
        past = None
        while True:
            cur_len = input_ids.shape[1]
            outputs = self(**self.prepare_inputs_for_generation(input_ids, past=past, **model_kwargs), return_dict=True, use_cache=True)
            past = outputs.past_key_values
            scores = F.log_softmax(outputs.logits[:, -1, :].float(), dim=-1)
            if repetition_penalty != 1.0:                                             # RepetitionPenaltyLogitsProcessor
                seen = torch.gather(scores, 1, input_ids)
                scores.scatter_(1, input_ids, torch.where(seen < 0, seen * repetition_penalty, seen / repetition_penalty))
            if cur_len < min_length:                                                  # MinLengthLogitsProcessor
                scores[:, eos_token_id] = -float("inf")
            vocab = scores.shape[-1]
            scores = (scores + beam_scores[:, None]).view(batch, num_beams * vocab)
            top_scores, top_flat = torch.topk(scores, 2 * num_beams, dim=1, largest=True, sorted=True)
            h_scores, h_flat = top_scores.tolist(), top_flat.tolist()                # the step's one device -> host read
            new_scores, new_tokens, new_index = [], [], []
            for b in range(batch):                                                    # BeamSearchScorer.process
                if done[b]:
                    new_scores += [0.0] * num_beams
                    new_tokens += [pad_token_id] * num_beams
                    new_index += [0] * num_beams
                    continue
                kept = 0
                for rank, (sc, flat) in enumerate(zip(h_scores[b], h_flat[b])):
                    tok, bb = flat % vocab, b * num_beams + flat // vocab
                    if tok == eos_token_id:
                        if rank >= num_beams:
                            continue
                        _beam_hyp_add(hyps[b], input_ids[bb].clone(), sc, num_beams, length_penalty)
                    else:
                        new_scores.append(sc)
                        new_tokens.append(tok)
                        new_index.append(bb)
                        kept += 1
                    if kept == num_beams:
                        break
                if kept < num_beams:
                    raise ValueError("fewer than num_beams live candidates in the top 2 * num_beams (needs a vocabulary > 2 * num_beams)")
                if not done[b] and len(hyps[b]["beams"]) >= num_beams:               # BeamHypotheses.is_done
                    done[b] = early_stopping or hyps[b]["worst"] >= max(h_scores[b]) / cur_len ** length_penalty
            beam_scores = torch.tensor(new_scores, dtype=torch.float32, device=dev)
            beam_idx = torch.tensor(new_index, dtype=torch.long, device=dev)
            input_ids = torch.cat([input_ids.index_select(0, beam_idx), torch.tensor(new_tokens, dtype=input_ids.dtype, device=dev)[:, None]], dim=-1)
            if model_kwargs.get("attention_mask", None) is not None:
                am = model_kwargs["attention_mask"]
                model_kwargs["attention_mask"] = torch.cat([am, am.new_ones((am.shape[0], 1))], dim=-1)
            past = self._reorder_cache(past, beam_idx)
            if all(done) or input_ids.shape[1] >= max_length:
                break
        final_scores = beam_scores.tolist()
        for b in range(batch):                                                        # BeamSearchScorer.finalize
            if not done[b]:
                for k in range(num_beams):
                    _beam_hyp_add(hyps[b], input_ids[b * num_beams + k], final_scores[b * num_beams + k], num_beams, length_penalty)
        best = [sorted(h["beams"], key=lambda t: t[0])[-1][1] for h in hyps]
        lengths = [int(t.shape[-1]) for t in best]
        out_len = min(max(lengths) + 1, max_length)
        decoded = input_ids.new_full((batch, out_len), pad_token_id)
        for i, t in enumerate(best):
            decoded[i, :lengths[i]] = t[:out_len]
            if lengths[i] < max_length:
                decoded[i, lengths[i]] = eos_token_id
        return decoded

    @torch.no_grad()
    def _beam_search_device(self, input_ids, num_beams, max_length, min_length, repetition_penalty, pad_token_id, eos_token_id,
                            length_penalty=1.0, early_stopping=False, sync_free=False, **model_kwargs):
        """`_beam_search` with the scorer on the device: every decode position is one decoder forward, one `evlm_beam_step` (log-softmax,
        processors, top 2 * num_beams, BeamSearchScorer.process / BeamHypotheses bookkeeping) and one in-place `evlm_kv_beam_reorder` of
        the self-attention caches; `evlm_beam_finalize` picks the results.  All state lives in device tensors and the loop runs exactly
        max_length - prompt length steps with no device -> host read and no host -> device copy (finished items are frozen, so running
        past the point where every item is done changes nothing).  sync_free=False returns the host loop's tensor (trimmed to the
        output length with one read per call); sync_free=True returns [batch, max_length], pad after the output length, with no read at
        all, so a caller can capture the whole call in one CUDA graph."""
        batch, prompt_len = input_ids.shape
        rows = batch * num_beams
        dev = input_ids.device
        enc = model_kwargs.get("encoder_hidden_states", None)
        if enc is not None and not isinstance(enc, list) and enc.shape[0] != rows:
            raise ValueError("encoder_hidden_states must hold batch * num_beams items (the caller expands them: model_generation.py:421-423)")
        am = model_kwargs.pop("attention_mask", None)
        if am is None:
            mask = input_ids.new_ones((rows, max_length))     # the host loop's per-step `new_ones`, allocated once and sliced
        else:
            mask = am.new_ones((rows, max_length))
            mask[:, :prompt_len] = am.repeat_interleave(num_beams, dim=0)
        i32 = torch.int32
        tokens = torch.full((rows, max_length), pad_token_id, dtype=torch.int64, device=dev)
        tokens[:, :prompt_len] = input_ids.repeat_interleave(num_beams, dim=0)
        beam_scores = torch.zeros(batch, num_beams, dtype=torch.float32, device=dev)
        beam_scores[:, 1:] = -1e9
        beam_scores = beam_scores.view(-1)
        beam_src = torch.zeros(rows, dtype=i32, device=dev)
        done = torch.zeros(batch, dtype=i32, device=dev)
        hyp_tokens = torch.zeros(batch, num_beams, max_length, dtype=torch.int64, device=dev)
        hyp_len = torch.zeros(batch, num_beams, dtype=i32, device=dev)
        hyp_score = torch.zeros(batch, num_beams, dtype=torch.float64, device=dev)
        hyp_count = torch.zeros(batch, dtype=i32, device=dev)
        hyp_worst = torch.full((batch,), 1e9, dtype=torch.float64, device=dev)
        item_base = None
        past = None
        for cur_len in range(prompt_len, max_length):
            model_inputs = self.prepare_inputs_for_generation(tokens[:, :cur_len], past=past, attention_mask=mask[:, :cur_len], **model_kwargs)
            outputs = self(**model_inputs, return_dict=True, use_cache=True)
            past = outputs.past_key_values
            K.beam_step(outputs.logits[:, -1, :].float(), num_beams, cur_len, min_length, repetition_penalty, length_penalty, early_stopping,
                        eos_token_id, pad_token_id, tokens, beam_scores, beam_src, done, hyp_tokens, hyp_len, hyp_score, hyp_count, hyp_worst)
            if cur_len + 1 < max_length and not ops.kv_beam_reorder(past, beam_src, num_beams):
                if item_base is None:
                    item_base = torch.arange(rows, device=dev) // num_beams * num_beams
                past = self._reorder_cache(past, item_base + beam_src)
        out, lengths = K.beam_finalize(num_beams, max_length, max_length, length_penalty, eos_token_id, pad_token_id, tokens, beam_scores, done,
                                       hyp_tokens, hyp_len, hyp_score, hyp_count, hyp_worst)
        if sync_free:
            return out
        return out[:, :min(int(lengths.max()) + 1, max_length)].contiguous()      # the call's one device -> host read

    @torch.no_grad()
    def generate(self, input_ids, max_length=20, min_length=0, num_beams=1, do_sample=False, temperature=1.0, top_k=0, top_p=1.0,
                 repetition_penalty=1.0, pad_token_id=0, eos_token_id=None, sync_free=False, **model_kwargs):
        """Greedy / sampling generation (num_beams == 1) through the in-repo loop; num_beams > 1: beam search, the algorithm the
        reference's captioning evaluation gets from transformers 4.12.5's GenerationMixin (model_generation.py:474-483).  On CUDA tensors
        (2 <= num_beams <= 8, a vocabulary above 2 * num_beams, at least one step to decode) it runs `_beam_search_device`, else the host
        loop `_beam_search`.  sync_free=True (extension) runs every loop to max_length without host checks (same ids); beam search then
        returns [batch, max_length] with pad after the output length."""
        if num_beams != 1:
            if do_sample:
                raise NotImplementedError("beam sampling (num_beams > 1 with do_sample) is not used by the reference and not provided")
            if not isinstance(eos_token_id, int):
                raise ValueError("beam search takes one end-of-sequence id (the reference passes tokenizer.sep_token_id)")
            if (BEAM_SEARCH_ON_DEVICE and input_ids.is_cuda and 2 <= num_beams <= 8 and self.config.vocab_size > 2 * num_beams
                    and input_ids.shape[1] < max_length):
                return self._beam_search_device(input_ids, num_beams, max_length, min_length, repetition_penalty, pad_token_id, eos_token_id,
                                                sync_free=sync_free, **model_kwargs)
            ids = self._beam_search(input_ids, num_beams, max_length, min_length, repetition_penalty, pad_token_id, eos_token_id,
                                    **model_kwargs)
            if sync_free and ids.shape[1] < max_length:
                ids = torch.cat([ids, ids.new_full((ids.shape[0], max_length - ids.shape[1]), pad_token_id)], dim=1)
            return ids
        eos = [eos_token_id] if isinstance(eos_token_id, int) else list(eos_token_id or [])
        ids, _ = self._generate_no_beam_search(input_ids, input_ids.shape[1], max_length, do_sample, temperature, top_k, top_p,
                                               repetition_penalty, pad_token_id, eos, input_ids.shape[0], sync_free=sync_free, **model_kwargs)
        return ids


def _beam_hyp_add(hyp, tokens, sum_logprobs, num_beams, length_penalty):
    """BeamHypotheses.add (transformers 4.12.5 generation_beam_search.py): hyp = {"beams": [(score, tokens)], "worst": float}."""
    score = sum_logprobs / (tokens.shape[-1] ** length_penalty)
    if len(hyp["beams"]) < num_beams or score > hyp["worst"]:
        hyp["beams"].append((score, tokens))
        if len(hyp["beams"]) > num_beams:
            order = sorted((sc, i) for i, (sc, _) in enumerate(hyp["beams"]))
            del hyp["beams"][order[0][1]]
            hyp["worst"] = order[1][0]
        else:
            hyp["worst"] = min(score, hyp["worst"])


def top_k_top_p_filtering(logits, top_k=0, top_p=1.0, filter_value=-float("Inf"), min_tokens_to_keep=1):
    """eff_bert.py:1566-1598 (sampling utility; host-side selection logic on tiny [B, V] tensors)."""
    if top_k > 0:
        top_k = min(max(top_k, min_tokens_to_keep), logits.size(-1))
        indices_to_remove = logits < torch.topk(logits, top_k)[0][..., -1, None]
        logits[indices_to_remove] = filter_value
    if top_p < 1.0:
        sorted_logits, sorted_indices = torch.sort(logits, descending=True)
        cumulative_probs = torch.cumsum(F.softmax(sorted_logits, dim=-1), dim=-1)
        sorted_indices_to_remove = cumulative_probs > top_p
        if min_tokens_to_keep > 1:
            sorted_indices_to_remove[..., :min_tokens_to_keep] = 0
        sorted_indices_to_remove[..., 1:] = sorted_indices_to_remove[..., :-1].clone()
        sorted_indices_to_remove[..., 0] = 0
        indices_to_remove = sorted_indices_to_remove.scatter(1, sorted_indices, sorted_indices_to_remove)
        logits[indices_to_remove] = filter_value
    return logits


class BertForMaskedLM(BertPreTrainedModel):
    def __init__(self, config):
        super().__init__(config)
        self.bert = BertModel(config, add_pooling_layer=False)
        self.cls = BertOnlyMLMHead(config)
        self.init_weights()

    def get_output_embeddings(self):
        return self.cls.predictions.decoder

    def set_output_embeddings(self, new_embeddings):
        self.cls.predictions.decoder = new_embeddings

    def get_input_embeddings(self):
        return self.bert.embeddings.word_embeddings

    def gather_seq_out_by_pos(self, seq, pos):
        return torch.gather(seq, 1, pos.unsqueeze(2).expand(-1, -1, seq.size(-1)))

    def forward(self, input_ids=None, attention_mask=None, token_type_ids=None, position_ids=None, head_mask=None, inputs_embeds=None,
                encoder_embeds=None, encoder_hidden_states=None, encoder_attention_mask=None, labels=None, output_attentions=None,
                output_hidden_states=None, return_dict=None, is_decoder=False, mode="multi_modal", return_logits=False, masked_pos=None,
                head_z=None, head_layer_z=None, mlp_z=None):
        return_dict = return_dict if return_dict is not None else self.config.use_return_dict
        outputs = self.bert(input_ids, attention_mask=attention_mask, token_type_ids=token_type_ids, position_ids=position_ids,
                            head_mask=head_mask, inputs_embeds=inputs_embeds, encoder_embeds=encoder_embeds,
                            encoder_hidden_states=encoder_hidden_states, encoder_attention_mask=encoder_attention_mask,
                            output_attentions=output_attentions, output_hidden_states=output_hidden_states, return_dict=return_dict,
                            is_decoder=is_decoder, mode=mode, head_z=head_z, head_layer_z=head_layer_z, mlp_z=mlp_z)
        sequence_output = outputs[0]
        if masked_pos is not None:
            sequence_output = self.gather_seq_out_by_pos(sequence_output, masked_pos)
        prediction_scores = self.cls(sequence_output)
        if return_logits:
            return prediction_scores
        masked_lm_loss = None
        if labels is not None:
            masked_lm_loss = cross_entropy(prediction_scores.view(-1, self.config.vocab_size), labels.reshape(-1))
        if not return_dict:
            output = (prediction_scores,) + tuple(outputs[2:])
            return ((masked_lm_loss,) + output) if masked_lm_loss is not None else output
        return MaskedLMOutput(loss=masked_lm_loss, logits=prediction_scores, hidden_states=outputs.hidden_states,
                              attentions=outputs.attentions, cross_attentions=outputs.cross_attentions)
