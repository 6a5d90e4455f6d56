"""Mask materialisation: turn deterministic L0 gates into physically smaller weights (ragged head counts / FFN widths per layer).

Drop-in for `update_params` + `prune_model_with_z` of the reference's `utils/xvlm_utils.py:37-245` (retrieval / NLVR / grounding
models), `utils/vqa_utils.py:37-293` and `utils/caption_utils.py` (models with a `text_decoder`): same two-step recipe —
  1. `update_params`: fold the gate VALUES into the weights the gate multiplies (value projection rows + bias for head gates,
     FFN down-projection columns for intermediate gates), so that non-binary gates keep their scale;
  2. `prune_model_with_z`: `prune_heads` every head whose gate is exactly 0 and slice away the FFN columns whose gate is 0.
The layer counts come from the gate tensors instead of the literals 6 / 3 / 3 / 3 of the reference files.

The pruned modules run on the same kernels: the GEMMs take any N / K (the bf16 operands keep 16-byte row pitches, and the small-M
weight-stream kernel of the decode steps masks a partial last 8-element group of K), attention takes `num_heads` from the module.
Like the reference, a layer whose heads or FFN columns are ALL pruned is not representable by the forward code (the reference sets
the Linear to None and then fails in forward); this module refuses to produce such a layer.

Captioning models (`text_encoder is None`, the XVLML0Module gates drive `text_decoder`): the decoder's gates are folded exactly as the
gated decoder applies them on the one decode path where the reference gates it, beam search (captioning.XVLMForCaptioning.generate):
head_z = cat(text_head_z, cross_head_z) and mlp_z = cat(text_intermediate_z, cross_intermediate_z), indexed per layer by
`eff_bert.layer_gate_rows` (quirk Q1: with fusion layer F, layer i >= F takes self row 2(i - F), cross row 2(i - F) + 1 and FFN row
i - F, so the trailing cross_* rows are never read).  The reference's utils/caption_utils.py is not available, so parity with its
captioning recipe is unpinned; the target is the gated model's own decode (tests/test_caption_materialize.py).

NLVR2 models (`nlvr.XVLMForNLVR`): the text encoder runs in multi_modal mode with the same concatenated gates (nlvr.py `_gates`), so
its text + 2 x cross layers take their rows through the same table (`concat_gate_rows`).  The reference's xvlm_utils.py folds the
*intended* mapping for NLVR (text_head_z[i] / cross_head_z[2i]), not what its own gated forward applies; as for captioning, the target
here is the gated model's own forward (tests/test_pruned_retrieval_nlvr.py).  The two per-image copies of a fusion layer share one
cross-attention key / value parameter (`XVLMForNLVR.share_cross_attention`) but read different cross-head gate rows, so materialising
first gives every copy its own key / value Linear: each copy then folds and prunes its own heads.  A materialised model is
inference-only, so nothing needs the tie afterwards.
"""
import torch

from . import ops
from .eff_bert import layer_gate_rows
from .eff_vit import prune_linear_layer
from .nlvr import XVLMForNLVR

DIMS_PER_HEAD = 64


def _bert_of(model, attr):
    m = getattr(model, attr, None)
    if m is None:
        return None
    return m.bert if hasattr(m, "bert") else m


def _rows(z):
    """[layers, ...] gate tensor -> list of flat per-layer CPU vectors."""
    return [z[i].detach().cpu().reshape(-1).clone() for i in range(z.shape[0])]


def _scale_value(att_self, head_z):
    hz = torch.repeat_interleave(head_z, DIMS_PER_HEAD).to(att_self.value.weight.device)
    att_self.value.weight.data = att_self.value.weight.data.mul(hz[:, None])
    att_self.value.bias.data = att_self.value.bias.data.mul(hz)


def concat_gate_rows(zs, bert):
    """Per layer of `bert`: (self head gate row, cross head gate row or None, FFN gate row), the rows its gated multi_modal forward
    applies to that layer with head_z = cat(text_head_z, cross_head_z) and mlp_z = cat(text_intermediate_z, cross_intermediate_z): the
    decoder of a captioning model, the text encoder of an NLVR model (see the module docstring)."""
    heads = _rows(torch.cat((zs["text_head_z"], zs["cross_head_z"]), dim=0))
    mlps = _rows(torch.cat((zs["text_intermediate_z"], zs["cross_intermediate_z"]), dim=0))
    out = []
    for i in range(len(bert.encoder.layer)):
        s, c, m = layer_gate_rows(i, bert.encoder.fusion_layer)
        out.append((heads[s], None if c is None else heads[c], mlps[m]))
    return out


caption_decoder_gates = concat_gate_rows        # the name the captioning code and tests know it by


def _concat_plan(gates, what):
    """Per layer: (self heads to prune, cross heads to prune or None, FFN columns to keep); refuses a layer left empty."""
    return [(_zero_heads(s, what + " self", i), None if c is None else _zero_heads(c, what + " cross", i), _kept_columns(m, what, i))
            for i, (s, c, m) in enumerate(gates)]


def _concat_bert(model, zs):
    """(BERT whose gates are the concatenated rows of `concat_gate_rows`, its name in errors), or (None, None) for the other models."""
    if "text_head_z" not in zs:
        return None, None
    if _bert_of(model, "text_encoder") is None and _bert_of(model, "text_decoder") is not None:
        return _bert_of(model, "text_decoder"), "decoder"
    if isinstance(model, XVLMForNLVR):
        return _bert_of(model, "text_encoder"), "encoder"
    return None, None


def _untie_cross_kv(bert):
    """Every cross-attention layer gets its own copy of its key / value Linear (undoes XVLMForNLVR.share_cross_attention)."""
    for blk in bert.encoder.layer:
        if blk.has_cross_attention:
            s = blk.crossattention.self
            for name in ("key", "value"):
                lin = getattr(s, name)
                own = torch.nn.Linear(lin.in_features, lin.out_features, device=lin.weight.device, dtype=lin.weight.dtype)
                own.weight.copy_(lin.weight)
                own.bias.copy_(lin.bias)
                setattr(s, name, own)


@torch.no_grad()
def update_params(model, zs):
    """vqa_utils.py:37-104 / xvlm_utils.py:37-85: gate values folded into value projections and FFN down-projections."""
    vision = model.vision_encoder
    text = _bert_of(model, "text_encoder")
    decoder = _bert_of(model, "text_decoder")
    bert, what = _concat_bert(model, zs)
    if bert is not None:
        gates = concat_gate_rows(zs, bert)
        _concat_plan(gates, what)             # a layer that would be left empty is refused before any weight changes
        if "vision_head_z" in zs:
            _heads_to_prune(zs["vision_head_z"], "vision")
        if "vision_intermediate_z" in zs:
            _kept_dims(zs["vision_intermediate_z"], "vision")
        if what == "encoder":
            _untie_cross_kv(bert)
        for blk, (self_z, cross_z, mlp_z) in zip(bert.encoder.layer, gates):
            _scale_value(blk.attention.self, self_z)
            if cross_z is not None:
                _scale_value(blk.crossattention.self, cross_z)
            d = blk.output.dense
            d.weight.data = d.weight.data.mul(mlp_z.to(d.weight.device))
        zs = {k: v for k, v in zs.items() if k.startswith("vision_")}
    n_text = zs["text_head_z"].shape[0] if "text_head_z" in zs else (zs["text_intermediate_z"].shape[0] if "text_intermediate_z" in zs else 0)
    if "vision_intermediate_z" in zs:
        for layer, z in enumerate(_rows(zs["vision_intermediate_z"])):
            fc2 = vision.encoder.layers[layer].mlp.fc2
            fc2.weight.data = fc2.weight.data.mul(z.to(fc2.weight.device))
    if "vision_head_z" in zs:
        for layer, z in enumerate(_rows(zs["vision_head_z"])):
            att = vision.encoder.layers[layer].self_attn
            hz = torch.repeat_interleave(z, DIMS_PER_HEAD).to(att.v_proj.weight.device)
            att.v_proj.weight.data = att.v_proj.weight.data.mul(hz[:, None])
            att.v_proj.bias.data = att.v_proj.bias.data.mul(hz)
    if "text_intermediate_z" in zs:
        for layer, z in enumerate(_rows(zs["text_intermediate_z"])):
            d = text.encoder.layer[layer].output.dense
            d.weight.data = d.weight.data.mul(z.to(d.weight.device))
    if "text_head_z" in zs:
        for layer, z in enumerate(_rows(zs["text_head_z"])):
            _scale_value(text.encoder.layer[layer].attention.self, z)
    if "cross_intermediate_z" in zs:
        for layer, z in enumerate(_rows(zs["cross_intermediate_z"])):
            d = text.encoder.layer[n_text + layer].output.dense
            d.weight.data = d.weight.data.mul(z.to(d.weight.device))
    if "cross_head_z" in zs:
        rows = _rows(zs["cross_head_z"])
        for layer in range(len(rows) // 2):
            blk = text.encoder.layer[n_text + layer]
            _scale_value(blk.attention.self, rows[2 * layer])
            _scale_value(blk.crossattention.self, rows[2 * layer + 1])
    if decoder is not None and "decoder_intermediate_z" in zs:
        for layer, z in enumerate(_rows(zs["decoder_intermediate_z"])):
            d = decoder.encoder.layer[layer].output.dense
            d.weight.data = d.weight.data.mul(z.to(d.weight.device))
    if decoder is not None and "decoder_head_z" in zs:
        rows = _rows(zs["decoder_head_z"])
        for layer in range(len(rows) // 2):
            blk = decoder.encoder.layer[layer]
            _scale_value(blk.attention.self, rows[2 * layer])
            _scale_value(blk.crossattention.self, rows[2 * layer + 1])
    ops.invalidate_weight_cache()


def _zero_heads(row, what, layer):
    idx = torch.where(row == 0)[0].tolist()
    if len(idx) == row.numel():
        raise NotImplementedError("%s layer %d: every head is pruned; the forward code (reference and B200) cannot run a layer "
                                  "without heads" % (what, layer))
    return idx


def _kept_columns(row, what, layer):
    keep = row.nonzero().reshape(-1).tolist()
    if not keep:
        raise NotImplementedError("%s layer %d: every FFN column is pruned; the forward code cannot run a layer without an FFN" % (what, layer))
    return keep


def _heads_to_prune(z, what):
    return {layer: _zero_heads(row, what, layer) for layer, row in enumerate(_rows(z))}


def _kept_dims(z, what):
    return {layer: _kept_columns(row, what, layer) for layer, row in enumerate(_rows(z))}


def prune_intermediate_layers(bert, keep_dims, device=None):
    """vqa_utils.py:295-303."""
    for layer, keep in keep_dims.items():
        blk = bert.encoder.layer[layer]
        index = torch.LongTensor(keep).to(blk.intermediate.dense.weight.device)
        blk.intermediate.dense = prune_linear_layer(blk.intermediate.dense, index=index, dim=0)
        blk.output.dense = prune_linear_layer(blk.output.dense, index=index, dim=1)


def prune_vision_intermediate_layers(vision_encoder, keep_dims, device=None):
    """vqa_utils.py:305-313."""
    for layer, keep in keep_dims.items():
        mlp = vision_encoder.encoder.layers[layer].mlp
        index = torch.LongTensor(keep).to(mlp.fc1.weight.device)
        mlp.fc1 = prune_linear_layer(mlp.fc1, index=index, dim=0)
        mlp.fc2 = prune_linear_layer(mlp.fc2, index=index, dim=1)


@torch.no_grad()
def prune_model_with_z(zs, model):
    """vqa_utils.py:107-293 / xvlm_utils.py:88-245: physical head and FFN-column pruning from exact zeros in the gates."""
    if zs is None:
        return None, None
    vision = model.vision_encoder
    text = _bert_of(model, "text_encoder")
    decoder = _bert_of(model, "text_decoder")
    bert, what = _concat_bert(model, zs)
    if bert is not None:
        plan = _concat_plan(concat_gate_rows(zs, bert), what)
        for blk, (self_heads, cross_heads, _) in zip(bert.encoder.layer, plan):
            blk.attention.prune_heads(self_heads)
            if cross_heads is not None:
                blk.crossattention.prune_heads(cross_heads)
        prune_intermediate_layers(bert, {i: keep for i, (_, _, keep) in enumerate(plan)})
        zs = {k: v for k, v in zs.items() if k.startswith("vision_")}
    if "vision_head_z" in zs:
        vision.prune_heads(_heads_to_prune(zs["vision_head_z"], "vision"))
    if "text_head_z" in zs:
        text.prune_heads(_heads_to_prune(zs["text_head_z"], "text"))
    if "cross_head_z" in zs:
        text.prune_heads(_heads_to_prune(zs["cross_head_z"], "cross"), is_cross="cross")
    if decoder is not None and "decoder_head_z" in zs:
        decoder.prune_heads(_heads_to_prune(zs["decoder_head_z"], "decoder"), is_cross="decoder")
    if "vision_intermediate_z" in zs:
        prune_vision_intermediate_layers(vision, _kept_dims(zs["vision_intermediate_z"], "vision"))
    if "text_intermediate_z" in zs and "cross_intermediate_z" in zs:
        both = torch.cat((zs["text_intermediate_z"], zs["cross_intermediate_z"]), dim=0)
        prune_intermediate_layers(text, _kept_dims(both, "text/cross"))
    if decoder is not None and "decoder_intermediate_z" in zs:
        prune_intermediate_layers(decoder, _kept_dims(zs["decoder_intermediate_z"], "decoder"))
    ops.invalidate_weight_cache()
    return None, None


def materialize(model, zs=None):
    """update_params + prune_model_with_z with the model's own deterministic masks (l0_module.forward(training=False)) by
    default.  Returns the per-module sizes `l0_module.calculate_model_size` reports.  The pruned model is then run WITHOUT gates
    (the reference's `fake_forward`, model_generation.py:214-230): see `efficientvlm_b200.vqa.XVLMForVQA.forward(..., use_gates=False)`.
    Sets `model.gates_folded`: a captioning model's `generate`, an NLVR model's `forward(train=False)` and a retrieval model's
    `retrieval_eval.evaluation` then run without gates, and the training forwards refuse to run.  A layer that would be left without
    heads or FFN columns raises NotImplementedError; for captioning and NLVR models that happens before any weight changes."""
    if zs is None:
        with torch.no_grad():
            zs = model.l0_module.forward(training=False)
    update_params(model, zs)
    prune_model_with_z(zs, model)
    model.gates_folded = True
    return model.l0_module.calculate_model_size(zs) if hasattr(model, "l0_module") else None
