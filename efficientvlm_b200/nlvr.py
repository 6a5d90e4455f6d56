"""NLVR2 task models on the B200 hot path — drop-in for `efficient_models/model_nlvr.py::EffXVLMForNLVR` (L0-gated student) and
`models/model_nlvr.py::XVLMForNLVR` (un-gated teacher), plus the loss assembly of the `Eff_NLVR.py` pruning step.

The text encoder has `text + 2 x cross` layers (one copy of every fusion layer per image); the key / value projections of the two
copies are tied (`share_cross_attention`, model_nlvr.py:247-262) and every fusion layer cross-attends to ONE of the two images
(`encoder_hidden_states` is a list, eff_bert.py:518-529).  All of that is host-side routing over the same layer kernels.
"""
import torch
from torch import nn

from . import checkpoint, ops
from .distill import _kd_pairs, get_cor_teacher, soft_cross_entropy
from .eff_bert import BertConfig, cross_entropy
from .l0_module import NLVRL0Module
from .xvlm import XVLMBase, build_mlp, load_pretrained


def _nlvr_text_config(config):
    """model_nlvr.py:127-135: 6 (or 12) nominal layers -> text + 2 * cross encoder layers."""
    import os
    path = os.path.join(config["text_encoder"], "config.json") if config.get("text_encoder") else None
    config_text = BertConfig.from_json_file(path) if path and os.path.exists(path) else BertConfig()
    config_text.num_hidden_layers = config["text_num_hidden_layers"] if "text_num_hidden_layers" in config else 12
    assert config_text.num_hidden_layers in [6, 12], "param initialization not implemented"
    config_text.fusion_layer = config_text.num_hidden_layers // 2
    num_text_layers = config_text.fusion_layer
    num_cross_layers = config_text.num_hidden_layers - config_text.fusion_layer
    config_text.num_hidden_layers = num_text_layers + 2 * num_cross_layers
    return config_text, num_text_layers, num_cross_layers


class XVLMForNLVR(XVLMBase):
    """models/model_nlvr.py:126-245 — un-gated NLVR2 model (the distillation teacher of Eff_NLVR.py)."""
    gated = False
    gates_folded = False        # set by prune.materialize: the deterministic gates live in the (physically pruned) weights

    def __init__(self, config):
        config_text, num_text_layers, num_cross_layers = _nlvr_text_config(config)
        super().__init__(config, load_vision_params=False, load_text_params=False, use_contrastive_loss=False, use_matching_loss=False,
                         use_mlm_loss=False, use_bbox_loss=False, config_text=config_text)
        self.num_text_layers = num_text_layers  # overwrite
        self.num_cross_layers = num_cross_layers
        self.share_cross_attention(self.text_encoder.encoder)
        self.cls_head = build_mlp(input_dim=self.text_width, output_dim=2)
        if self.gated:
            self.l0_module = NLVRL0Module(config, target_sparsity=config["sparsity"])
        self.init_params = ["cls_head." + n for n, _ in self.cls_head.named_parameters()]

    def share_cross_attention(self, model):
        """model_nlvr.py:247-262: the key / value projections of the two per-image copies of a fusion layer are ONE parameter."""
        for i in range(self.num_cross_layers):
            layer_num = self.num_text_layers + i * 2
            modules_0 = model.layer[layer_num].crossattention.self._modules
            modules_1 = model.layer[layer_num + 1].crossattention.self._modules
            for name in modules_0.keys():
                if "key" in name or "value" in name:
                    module_0, module_1 = modules_0[name], modules_1[name]
                    if hasattr(module_0, "weight"):
                        module_0.weight = module_1.weight
                        if hasattr(module_0, "bias"):
                            module_0.bias = module_1.bias
        ops.invalidate_weight_cache()

    def load_pretrained(self, ckpt_rpath, config, load_nlvr_pretrain=False, is_eval=False):
        """model_nlvr.py:150-185: every pre-trained fusion layer initialises both of its per-image copies."""
        state_dict = load_pretrained(ckpt_rpath, config, is_eval=True) if is_eval else load_pretrained(ckpt_rpath, config, load_text=False)
        if not is_eval and not load_nlvr_pretrain:
            checkpoint.remap_keys(state_dict, checkpoint.nlvr_two_image_rule(self.num_text_layers))
        checkpoint.load_into(self, state_dict, ckpt_rpath)

    def _gates(self, train):
        if not self.gated or self.gates_folded:
            return dict(vision_head=None, vision_mlp=None, enc_head=None, enc_mlp=None)
        if train:
            zs = self.l0_module.forward(training=True)
        else:
            with torch.no_grad():
                zs = self.l0_module.forward(training=False)
        return dict(vision_head=zs["vision_head_z"], vision_mlp=zs["vision_intermediate_z"],
                    enc_head=torch.cat((zs["text_head_z"], zs["cross_head_z"]), dim=0),
                    enc_mlp=torch.cat((zs["text_intermediate_z"], zs["cross_intermediate_z"]), dim=0))

    def forward(self, image, text_ids, text_atts, targets, train=True, output_attentions=None, output_hidden_states=None):
        """image: [2B, 3, R, R] = the B first images followed by the B second images (model_nlvr.py:206-207).
        On a materialised model (prune.materialize) only the gate-free prediction `train=False` without KD outputs runs."""
        if self.gates_folded and (train or output_attentions):
            raise RuntimeError("this NLVR model was materialised (prune.materialize): its gates are folded into pruned weights, so the "
                               "training and distillation forwards, which apply full-width gates, cannot run on it; use train=False")
        z = self._gates(train)
        n = targets.size(0)
        kd = bool(output_attentions)
        ve = self.get_vision_embeds(image, output_attentions=output_attentions if kd else None,
                                    output_hidden_states=output_hidden_states if kd else None, head_z=z["vision_head"], mlp_z=z["vision_mlp"],
                                    _return_kd=kd)
        image_embeds, image_atts = ve[0], ve[1]
        image0_embeds, image1_embeds = torch.split(image_embeds, n)
        atts = [image_atts[:image0_embeds.size(0)], image_atts[image0_embeds.size(0):]]
        if not kd:
            output_cls = self.get_cross_embeds([image0_embeds, image1_embeds], atts, text_ids=text_ids, text_atts=text_atts,
                                               head_z=z["enc_head"], mlp_z=z["enc_mlp"])[:, 0, :]
            prediction = self.cls_head(output_cls)
            return cross_entropy(prediction, targets) if train else prediction
        image_hidden_states, image_attentions = ve[2], ve[3]
        outputs = self.get_cross_embeds([image0_embeds, image1_embeds], atts, text_ids=text_ids, text_atts=text_atts,
                                        output_attentions=output_attentions, output_hidden_states=output_hidden_states,
                                        head_z=z["enc_head"], mlp_z=z["enc_mlp"])
        prediction = self.cls_head(outputs[0][:, 0, :])
        loss = cross_entropy(prediction, targets) if train else None
        text_hidden_states, text_attentions, cross_attentions = outputs[1:]
        return {"loss": loss,
                "hidden_dict": {"image_hidden_states": image_hidden_states, "text_hidden_states": text_hidden_states},
                "attention_dict": {"image_attentions": image_attentions, "text_attentions": text_attentions},
                "cross_attention_dict": {"cross_attentions": cross_attentions},
                "logits_dict": {"cls_head_logits": prediction}}


class EffXVLMForNLVR(XVLMForNLVR):
    """efficient_models/model_nlvr.py:126-262 — L0-gated NLVR2 student (`l0_module` = NLVRL0Module)."""
    gated = True


# ----------------------------------------------------------------------------------------------------------------------
# Eff_NLVR.py:100-157 — KD terms and the loss mix of one pruning step
# ----------------------------------------------------------------------------------------------------------------------
def nlvr_kd_losses(student_outputs, teacher_outputs, temperature=1.0):
    sh, th = student_outputs["hidden_dict"], teacher_outputs["hidden_dict"]
    sa, ta = student_outputs["attention_dict"], teacher_outputs["attention_dict"]
    sc, tc = student_outputs["cross_attention_dict"], teacher_outputs["cross_attention_dict"]
    s_text_h = list(sh["text_hidden_states"])
    t_text_h = get_cor_teacher(th["text_hidden_states"], s_text_h)
    s_text_a = list(sa["text_attentions"])
    t_text_a = get_cor_teacher(ta["text_attentions"], s_text_a, is_attn=True)
    s_cross_a = list(sc["cross_attentions"])
    t_cross_a = get_cor_teacher(tc["cross_attentions"], s_cross_a, is_attn=True)
    s_img_h, s_img_a = list(sh["image_hidden_states"]), list(sa["image_attentions"])
    groups = [  # the slices 4 / 3 are literal in Eff_NLVR.py:116-123
        ("text_hidden", s_text_h[:4], t_text_h[:4], False, False),
        ("text_attention", s_text_a[:3], t_text_a[:3], True, False),
        ("cross_hidden", s_text_h[4:], t_text_h[4:], False, False),
        ("cross_self_attention", s_text_a[3:], t_text_a[3:], True, False),
        ("cross_attention", s_cross_a, t_cross_a, True, False),
        ("image_hidden", s_img_h, get_cor_teacher(th["image_hidden_states"], s_img_h), False, True),
        ("image_attention", s_img_a, get_cor_teacher(ta["image_attentions"], s_img_a, is_attn=True), True, False),
    ]
    S, T, W, spans = [], [], [], {}
    for name, s_list, t_list, is_attn, is_img in groups:
        s, t, w = _kd_pairs(s_list, t_list, is_attn, is_img)
        spans[name] = (len(S), len(S) + len(s))
        S += s
        T += t
        W += w
    per_pair = ops.mse_pairs(S, T, W)
    out = {name: per_pair[a:b].sum() for name, (a, b) in spans.items()}
    out["logits"] = soft_cross_entropy(student_outputs["logits_dict"]["cls_head_logits"] / temperature,
                                       teacher_outputs["logits_dict"]["cls_head_logits"] / temperature)
    return out


def nlvr_loss(student_outputs, teacher_outputs, l0_module=None, global_step=0, temperature=1.0):
    """`loss` of Eff_NLVR.py:141-155: 0.8 * task + 0.2 * (logit KL + text KD + 0.33 * (image KD + cross KD)) (+ Lagrangian)."""
    kd = nlvr_kd_losses(student_outputs, teacher_outputs, temperature)
    loss_small = student_outputs["loss"]
    loss_text_kd = kd["text_attention"] + kd["text_hidden"]
    loss_img_kd = kd["image_attention"] + kd["image_hidden"] * 0.1
    loss_cross_kd = (kd["cross_hidden"] + kd["cross_self_attention"] + kd["cross_attention"]) * 0.5
    loss_kd = kd["logits"] + loss_text_kd + (loss_img_kd + loss_cross_kd) * 0.33
    loss = 0.8 * loss_small + 0.2 * loss_kd
    parts = dict(loss_small=loss_small, loss_kd=loss_kd, loss_text_kd=loss_text_kd, loss_img_kd=loss_img_kd, loss_cross_kd=loss_cross_kd,
                 loss_logits_kd=kd["logits"], **{"kd_" + n: v for n, v in kd.items()})
    if l0_module is not None:
        lagrangian_loss, expected_sparsity, target_sparsity = l0_module.lagrangian_regularization(global_step)
        loss = loss + lagrangian_loss
        parts.update(loss_lagrangian=lagrangian_loss, expected_sparsity=expected_sparsity, target_sparsity=target_sparsity)
    return loss, parts
