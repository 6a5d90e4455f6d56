"""Teacher -> student distillation losses and the task models the benchmark drives.

* `get_cor_teacher`, `get_kd_loss`, `soft_cross_entropy` keep the signatures of the helpers copy-pasted into every
  reference driver (GeneralDistill.py:60-104, Eff_VQA.py:28-71, Eff_Retrieval.py:30-73, ...), but each `get_kd_loss` call is
  ONE multi-pair MSE launch and `gd_kd_losses` batches ALL ~50 (student, teacher) pairs of a GD step into a single launch.
* `XVLM` mirrors models/model_pretrain.py (teacher and student of general distillation);
  `EffXVLMforRetrieval` mirrors efficient_models/model_retrieval.py (L0-gated ITR model, BASELINE configs 1 and 4).
* `gd_loss` / `gd_step` restate the loss mix and step of GeneralDistill.py:286-387.
"""
import torch

from . import checkpoint, ops
from .l0_module import XVLML0Module
from .eff_bert import cross_entropy
from .xvlm import XVLMBase, load_pretrained


# ----------------------------------------------------------------------------------------------------------------------
# KD helpers (GeneralDistill.py:60-104)
# ----------------------------------------------------------------------------------------------------------------------
def get_cor_teacher(teacher_reps, student_reps, is_attn=False):
    teacher_reps = [None if t is None else t.detach() for t in teacher_reps]     # None: map skipped by attention_stride
    tn, sn = len(teacher_reps), len(student_reps)
    if is_attn:
        assert tn % sn == 0
        k = int(tn / sn)
        return [teacher_reps[i * k + k - 1] for i in range(sn)]
    assert (tn - 1) % (sn - 1) == 0
    k = int((tn - 1) / (sn - 1))
    return [teacher_reps[i * k] for i in range(sn)]


def _kd_pairs(student_reps, teacher_reps, is_attn=False, is_img=False):
    """(students, teachers, scales) of one get_kd_loss call: attention MSE is multiplied by the key length (:69), the
    image-hidden variant drops list index 6 (:70-78); `where(att <= -1e2, 0, att)` is a no-op on probabilities (quirk Q8)."""
    S, T, W = [], [], []
    for layer, (s, t) in enumerate(zip(student_reps, teacher_reps)):
        if is_img and not is_attn and layer == 6:
            continue
        S.append(s)
        T.append(t)
        W.append(float(s.shape[-1]) if is_attn else 1.0)
    return S, T, W


def get_kd_loss(student_reps=None, teacher_reps=None, is_attn=False, loss=None, device="cuda", is_img=False):
    S, T, W = _kd_pairs(student_reps, teacher_reps, is_attn, is_img)
    if not S:
        return 0
    return ops.sum_scaled(ops.mse_pairs(S, T, W))


def soft_cross_entropy(predicts, targets):
    """KLDivLoss(batchmean)(log_softmax(predicts), softmax(targets))  (GeneralDistill.py:84-89)."""
    V = predicts.shape[-1]
    p2, t2 = predicts.reshape(-1, V), targets.reshape(-1, V)
    return ops.sum_scaled(ops.kl_rows(p2, t2, 1.0), 1.0 / p2.shape[0])


def set_teacher_attention_stride(teacher, student):
    """The KD losses read only teacher attention maps i*k + k-1 (get_cor_teacher, k = teacher layers / student layers): tell the
    teacher's encoders to materialise just those.  A no-op (stride None) when the layer counts do not divide evenly."""
    def stride(tn, sn):
        return tn // sn if sn > 0 and tn % sn == 0 and tn // sn > 1 else None
    tv, sv = teacher.vision_encoder.encoder, student.vision_encoder.encoder
    tv.attention_stride = stride(len(tv.layers), len(sv.layers))
    tb, sb = teacher._bert().encoder, student._bert().encoder
    k_text = stride(tb.fusion_layer, sb.fusion_layer)
    k_fuse = stride(len(tb.layer) - tb.fusion_layer, len(sb.layer) - sb.fusion_layer)
    tb.attention_stride = k_text if (k_text == k_fuse and k_text and tb.fusion_layer % k_text == 0) else None


def gd_kd_losses(student_outputs, teacher_outputs, temperature=1.0):
    """All KD terms of a general-distillation step (GeneralDistill.py:300-366) with ONE MSE launch. Returns a dict of scalars."""
    sh, th = student_outputs["hidden_dict"], teacher_outputs["hidden_dict"]
    sa, ta = student_outputs["attention_dict"], teacher_outputs["attention_dict"]
    groups = [  # (name, student list, teacher list, is_attn, is_img)
        ("text_hidden", sh["text_hidden_states"], th["text_hidden_states"], False, False),
        ("text_attn", sa["text_attentions"], ta["text_attentions"], True, False),
        ("image_hidden", sh["image_hidden_states"], th["image_hidden_states"], False, True),
        ("image_attn", sa["image_attentions"], ta["image_attentions"], True, False),
        ("itm_pos_hidden", sh["itm_pos_hidden_states"], th["itm_pos_hidden_states"], False, False),
        ("itm_pos_attn", sa["itm_pos_attentions"], ta["itm_pos_attentions"], True, False),
        ("itm_neg_hidden", sh["itm_neg_hidden_states"], th["itm_neg_hidden_states"], False, False),
        ("itm_neg_attn", sa["itm_neg_attentions"], ta["itm_neg_attentions"], True, False),
    ]
    if "mlm_hidden_states" in sh:
        groups += [("mlm_hidden", sh["mlm_hidden_states"], th["mlm_hidden_states"], False, False),
                   ("mlm_attn", sa["mlm_attentions"], ta["mlm_attentions"], True, False)]
    S, T, W, spans = [], [], [], {}
    for name, s_list, t_list, is_attn, is_img in groups:
        t_cor = get_cor_teacher(t_list, s_list, is_attn=is_attn)
        s, t, w = _kd_pairs(s_list, t_cor, is_attn, is_img)
        spans[name] = (len(S), len(S) + len(s))
        S += s
        T += t
        W += w
    per_pair = ops.mse_pairs(S, T, W)
    out = {name: per_pair[a:b].sum() for name, (a, b) in spans.items()}
    sl, tl = student_outputs["logits_dict"], teacher_outputs["logits_dict"]
    out["itm_logits"] = soft_cross_entropy(sl["itm_head_logits"] / temperature, tl["itm_head_logits"] / temperature)
    if "mlm_logits" in sl:
        V = sl["mlm_logits"].shape[-1]
        s2, t2 = sl["mlm_logits"].reshape(-1, V), tl["mlm_logits"].reshape(-1, V)
        out["mlm_logits"] = ops.sum_scaled(ops.kl_rows(s2, t2, 1.0 / temperature), 1.0 / s2.shape[0])
    return out


def gd_loss(student_outputs, teacher_outputs, temperature=1.0):
    """loss_in_total of GeneralDistill.py:369-376 plus the logged components."""
    kd = gd_kd_losses(student_outputs, teacher_outputs, temperature)
    loss = student_outputs["loss"]
    loss_small = loss["loss_itc"] + loss["loss_itm"] + loss["loss_mlm"]
    loss_text_kd = kd["text_attn"] + kd["text_hidden"]
    loss_img_kd = kd["image_attn"] + 0.1 * kd["image_hidden"]
    loss_cross_kd = (kd["itm_neg_attn"] + kd["itm_neg_hidden"] + kd["itm_pos_attn"] + kd["itm_pos_hidden"] + kd["mlm_attn"]
                     + kd["mlm_hidden"])
    loss_kd = kd["itm_logits"] + kd["mlm_logits"] + loss_text_kd + loss_img_kd + loss_cross_kd
    total = loss_small * 0.6 + loss_kd * 0.4
    return total, dict(loss_small=loss_small, loss_kd=loss_kd, loss_text_kd=loss_text_kd, loss_img_kd=loss_img_kd,
                       loss_cross_kd=loss_cross_kd, loss_itm_kd=kd["itm_logits"], loss_mlm_kd=kd["mlm_logits"], **loss)


def _cut(t, a, b):
    return None if t is None else t[a:b]


# ----------------------------------------------------------------------------------------------------------------------
# task models
# ----------------------------------------------------------------------------------------------------------------------
class XVLMBaseUngated(XVLMBase):
    """models/xvlm.py flavour of XVLMBase: get_vision_embeds always returns the KD 4-tuple (models/xvlm.py:331-338)."""

    def get_vision_embeds(self, image, image_atts=None, idx_to_group_img=None, output_attentions=None, output_hidden_states=None):
        return super().get_vision_embeds(image, image_atts=image_atts, idx_to_group_img=idx_to_group_img,
                                         output_attentions=output_attentions, output_hidden_states=output_hidden_states, _return_kd=True)


class XVLM(XVLMBaseUngated):
    """models/model_pretrain.py:5-82 — the general-distillation teacher AND student (checkpoints optional here)."""

    def __init__(self, config, load_vision_params=False, load_text_params=False):
        super().__init__(config, load_vision_params=load_vision_params, load_text_params=load_text_params, use_contrastive_loss=True,
                         use_matching_loss=True, use_mlm_loss=True, use_bbox_loss=True, config_text=None)

    def forward(self, image, text_ids, text_atts, text_ids_masked=None, masked_pos=None, masked_ids=None, image_atts=None,
                idx_to_group_img=None, target_bbox=None, is_image=None, ret_bbox_loss=False, output_attentions=None,
                output_hidden_states=None):
        assert output_attentions == output_hidden_states
        if ret_bbox_loss:
            image_embeds, image_atts, image_embeds_fullatts, image_hidden_states, image_attentions = self.get_vision_embeds(
                image, image_atts=image_atts, idx_to_group_img=idx_to_group_img, output_attentions=output_attentions,
                output_hidden_states=output_hidden_states)
        else:
            image_embeds, image_atts, image_hidden_states, image_attentions = self.get_vision_embeds(
                image, output_attentions=output_attentions, output_hidden_states=output_hidden_states)
        if self.batch_passes and output_attentions and not ret_bbox_loss and text_ids_masked is not None:
            return self._forward_batched_passes(image_embeds, image_atts, image_hidden_states, image_attentions, text_ids, text_atts,
                                                text_ids_masked, masked_pos, masked_ids)
        text_embeds, text_hidden_states, text_attentions = self.get_text_embeds(text_ids, text_atts, output_attentions=output_attentions,
                                                                                output_hidden_states=output_hidden_states)
        hidden_dict = {"image_hidden_states": image_hidden_states, "text_hidden_states": text_hidden_states}
        attention_dict = {"image_attentions": image_attentions, "text_attentions": text_attentions}
        cross_attention_dict, logits_dict = {}, {}
        with torch.no_grad():
            self.temp.clamp_(0.001, 0.5)
        image_feat, text_feat = self.get_features(image_embeds, text_embeds)
        loss_itc = self.get_contrastive_loss(image_feat, text_feat)
        itm = self.get_matching_loss(image_embeds, image_atts, image_feat, text_embeds, text_atts, text_feat,
                                     output_attentions=output_attentions, output_hidden_states=output_hidden_states)
        loss_itm = itm["loss"]
        hidden_dict["itm_pos_hidden_states"] = itm["pos_hidden_states"]
        hidden_dict["itm_neg_hidden_states"] = itm["neg_hidden_states"]
        attention_dict["itm_pos_attentions"] = itm["pos_attentions"]
        attention_dict["itm_neg_attentions"] = itm["neg_attentions"]
        cross_attention_dict["itm_pos_cross_attentions"] = itm["pos_cross_attentions"]
        cross_attention_dict["itm_neg_cross_attentions"] = itm["neg_cross_attentions"]
        logits_dict["itm_head_logits"] = itm["logits"]
        mlm = self.get_mlm_loss(text_ids_masked, text_atts, image_embeds, image_atts, masked_pos, masked_ids,
                                output_attentions=output_attentions, output_hidden_states=output_hidden_states)
        loss_mlm = mlm[0]
        hidden_dict["mlm_hidden_states"] = mlm[2]
        attention_dict["mlm_attentions"] = mlm[3]
        logits_dict["mlm_logits"] = mlm[1]
        cross_attention_dict["mlm_cross_attentions"] = mlm[4]
        loss = {"loss_itc": loss_itc, "loss_itm": loss_itm, "loss_mlm": loss_mlm}
        if ret_bbox_loss:
            bbox_output = self.predict_bbox(image_embeds_fullatts, text_embeds, text_atts, output_attentions=output_attentions,
                                            output_hidden_states=output_hidden_states)
            loss_bbox, loss_giou = self.get_bbox_loss(bbox_output[0], target_bbox, is_image=is_image)
            loss["loss_bbox"], loss["loss_giou"] = loss_bbox, loss_giou
            if output_attentions is not None:
                hidden_dict["bbox_hidden_states"], attention_dict["bbox_attentions"], cross_attention_dict["bbox_cross_attentions"] = \
                    bbox_output[1:]
        return {"loss": loss, "hidden_dict": hidden_dict, "attention_dict": attention_dict, "cross_attention_dict": cross_attention_dict,
                "logits_dict": logits_dict}


    # The reference issues four encoder passes per GD step over the SAME weights: text(text_ids), fusion(ITM: B positives + 2B
    # negatives) and the 12-layer multi-modal MLM pass over text_ids_masked (models/model_pretrain.py:33-60).  Every encoder is
    # per-sample, so the passes that share weights are run as ONE batch here and split afterwards:
    #   text mode   on cat([text_ids, text_ids_masked])                    (2B rows)   -> ITC/ITM text states | MLM text states
    #   fusion mode on cat([ITM positives, ITM negatives, MLM rows])       (4B rows)   -> ITM logits | MLM sequence output
    # (multi_modal mode == text mode followed by fusion mode, eff_bert.py:564-640).  Half the launches of those layers and GEMM
    # tiles that fill the machine; the returned dicts are laid out exactly as the unbatched forward lays them out.
    batch_passes = True
    pack_cross_attention = True     # same-image rows of the fusion batch share one 128-row attention tile (evlm_attn_args.pack_items)

    def _forward_batched_passes(self, image_embeds, image_atts, image_hidden_states, image_attentions, text_ids, text_atts,
                                text_ids_masked, masked_pos, masked_ids):
        bs = text_ids.size(0)
        ids2 = torch.cat([text_ids, text_ids_masked], dim=0)
        atts2 = torch.cat([text_atts, text_atts], dim=0)
        emb2, hid2, att2 = self.get_text_embeds(ids2, atts2, output_attentions=True, output_hidden_states=True)
        b2 = (0, bs, 2 * bs)
        text_embeds, mlm_text = ops.split_rows(emb2, b2)
        hs = [ops.split_rows(t, b2) for t in hid2]
        ats = [ops.split_rows(t, b2) for t in att2]
        text_hidden_states, mlm_text_hidden = tuple(p[0] for p in hs), tuple(p[1] for p in hs)
        text_attentions, mlm_text_att = tuple(p[0] for p in ats), tuple(p[1] for p in ats)
        with torch.no_grad():
            self.temp.clamp_(0.001, 0.5)
        image_feat, text_feat = self.get_features(image_embeds, text_embeds)
        loss_itc = self.get_contrastive_loss(image_feat, text_feat)
        # ---- fusion pass: rows = [ITM positives B | (neg image, text) B | (image, neg text) B | MLM B]
        neg_img, neg_txt = self.sample_itm_negatives(image_feat, text_feat, None)
        # all four row groups attend to the SAME B images (group 1 through the sampled permutation): the image tokens are passed
        # once with a row -> image index, so every fusion layer projects K/V once per image instead of once per row
        ar = torch.arange(bs, device=image_embeds.device, dtype=torch.int32)
        img_index = torch.cat([ar, neg_img.to(torch.int32), ar, ar])
        iat4 = torch.cat([image_atts, image_atts.index_select(0, neg_img), image_atts, image_atts], dim=0)
        img_pack = None
        if self.pack_cross_attention and 3 * text_ids.size(1) <= 128 and text_ids.size(1) % 8 == 0:
            # rows b, 2B+b, 3B+b attend to the same image b: they share one attention tile; the neg-image rows stay single
            minus = torch.full((bs,), -1, device=ar.device, dtype=torch.int32)
            img_pack = torch.cat([torch.stack([ar, 2 * bs + ar, 3 * bs + ar], dim=1), torch.stack([bs + ar, minus, minus], dim=1)], dim=0).contiguous()
        txt4 = torch.cat([text_embeds, text_embeds, text_embeds.index_select(0, neg_txt), mlm_text], dim=0)
        tat4 = torch.cat([text_atts, text_atts, text_atts.index_select(0, neg_txt), text_atts], dim=0)
        last4, hid4, att4, catt4 = self.get_cross_embeds(image_embeds, iat4, text_embeds=txt4, text_atts=tat4, output_attentions=True,
                                                         output_hidden_states=True,
                                                         image_index=img_index if img_pack is None else (img_index, img_pack))
        n3 = 3 * bs
        b4 = (0, bs, n3, 4 * bs)
        last_itm, last_mlm = ops.split_rows(last4, (0, n3, 4 * bs))
        # ITM head (xvlm.py:465-489)
        itm_logits = self.itm_head(last_itm[:, 0, :])
        itm_labels = torch.zeros(n3, dtype=torch.long, device=image_embeds.device)
        itm_labels[:bs] = 1
        loss_itm = cross_entropy(itm_logits, itm_labels)
        # MLM head (eff_bert.py:1690-1714)
        mlm_enc = self.text_encoder
        seq = mlm_enc.gather_seq_out_by_pos(last_mlm, masked_pos)
        mlm_logits = mlm_enc.cls(seq)
        loss_mlm = cross_entropy(mlm_logits.view(-1, mlm_enc.config.vocab_size), masked_ids.reshape(-1))
        h4 = [ops.split_rows(t, b4) for t in hid4]
        a4 = [ops.split_rows(t, b4) for t in att4]
        c4 = [ops.split_rows(t, b4) for t in catt4]
        hidden_dict = {"image_hidden_states": image_hidden_states, "text_hidden_states": text_hidden_states,
                       "itm_pos_hidden_states": tuple(p[0] for p in h4), "itm_neg_hidden_states": tuple(p[1] for p in h4),
                       "mlm_hidden_states": mlm_text_hidden + tuple(p[2] for p in h4[1:])}
        attention_dict = {"image_attentions": image_attentions, "text_attentions": text_attentions,
                          "itm_pos_attentions": tuple(p[0] for p in a4), "itm_neg_attentions": tuple(p[1] for p in a4),
                          "mlm_attentions": mlm_text_att + tuple(p[2] for p in a4)}
        cross_attention_dict = {"itm_pos_cross_attentions": tuple(p[0] for p in c4),
                                "itm_neg_cross_attentions": tuple(p[1] for p in c4),
                                "mlm_cross_attentions": tuple(p[2] for p in c4)}
        logits_dict = {"itm_head_logits": itm_logits, "mlm_logits": mlm_logits}
        return {"loss": {"loss_itc": loss_itc, "loss_itm": loss_itm, "loss_mlm": loss_mlm}, "hidden_dict": hidden_dict,
                "attention_dict": attention_dict, "cross_attention_dict": cross_attention_dict, "logits_dict": logits_dict}


class EffXVLMforRetrieval(XVLMBase):
    """efficient_models/model_retrieval.py:7-92 — L0-gated ITR model."""
    gates_folded = False        # set by prune.materialize: retrieval_eval.evaluation then runs without gates, forward refuses

    def __init__(self, config):
        super().__init__(config, load_vision_params=False, load_text_params=False, use_contrastive_loss=True, use_matching_loss=True,
                         use_mlm_loss=False, use_bbox_loss=False)
        self.num_attention_heads = self.text_encoder.config.num_attention_heads
        self.l0_module = XVLML0Module(config, target_sparsity=config["sparsity"])
        self.init_params = []

    def load_pretrained(self, ckpt_rpath, config, is_eval=False):
        checkpoint.load_into(self, load_pretrained(ckpt_rpath, config, is_eval=is_eval, load_text=True), ckpt_rpath)

    def forward(self, image, text_ids, text_atts, idx=None, output_attentions=None, output_hidden_states=None):
        if self.gates_folded:
            raise RuntimeError("this retrieval model was materialised (prune.materialize): its gates are folded into pruned weights, so "
                               "the training forward, which applies full-width gates, cannot run on it; use retrieval_eval.evaluation")
        kd = bool(output_attentions)
        zs = self.l0_module.forward(training=kd)                                # model_retrieval.py:26-27,78-79
        oa, oh = (output_attentions, output_hidden_states) if kd else (None, None)
        ve = self.get_vision_embeds(image, output_attentions=oa, output_hidden_states=oh, head_z=zs["vision_head_z"],
                                    mlp_z=zs["vision_intermediate_z"])
        te = self.get_text_embeds(text_ids, text_atts, output_attentions=oa, output_hidden_states=oh, head_z=zs["text_head_z"],
                                  mlp_z=zs["text_intermediate_z"])
        if kd:
            image_embeds, image_atts, image_hidden_states, image_attentions = ve
            text_embeds, text_hidden_states, text_attentions = te
        else:
            image_embeds, image_atts = ve
            text_embeds = te
        image_feat, text_feat = self.get_features(image_embeds, text_embeds)
        loss_itc = self.get_contrastive_loss(image_feat, text_feat, idx=idx)
        itm = self.get_matching_loss(image_embeds, image_atts, image_feat, text_embeds, text_atts, text_feat, idx=idx,
                                     output_attentions=oa, output_hidden_states=oh, head_z=zs["cross_head_z"],
                                     mlp_z=zs["cross_intermediate_z"])
        if not kd:
            return loss_itc, itm
        hidden_dict = {"image_hidden_states": image_hidden_states, "text_hidden_states": text_hidden_states,
                       "itm_pos_hidden_states": itm["pos_hidden_states"], "itm_neg_hidden_states": itm["neg_hidden_states"]}
        attention_dict = {"image_attentions": image_attentions, "text_attentions": text_attentions,
                          "itm_pos_attentions": itm["pos_attentions"], "itm_neg_attentions": itm["neg_attentions"]}
        cross_attention_dict = {"itm_pos_cross_attentions": itm["pos_cross_attentions"],
                                "itm_neg_cross_attentions": itm["neg_cross_attentions"]}
        return {"loss": {"loss_itc": loss_itc, "loss_itm": itm["loss"]}, "hidden_dict": hidden_dict, "attention_dict": attention_dict,
                "cross_attention_dict": cross_attention_dict, "logits_dict": {"itm_head_logits": itm["logits"]}}


class XVLMforRetrieval(XVLMBaseUngated):
    """models/model_retrieval.py:5-63 — un-gated ITR model: the distillation teacher of Eff_Retrieval.py (KD outputs without the
    ITC loss; it samples its own ITM negatives, like the reference)."""

    def __init__(self, config):
        super().__init__(config, load_vision_params=False, load_text_params=False, use_contrastive_loss=True, use_matching_loss=True,
                         use_mlm_loss=False, use_bbox_loss=False)
        self.num_attention_heads = self.text_encoder.config.num_attention_heads
        self.init_params = []

    def forward(self, image, text_ids, text_atts, idx=None, output_attentions=None, output_hidden_states=None):
        if not output_attentions:
            image_embeds, image_atts = self.get_vision_embeds(image)[:2]
            text_embeds = self.get_text_embeds(text_ids, text_atts)
            image_feat, text_feat = self.get_features(image_embeds, text_embeds)
            loss_itc = self.get_contrastive_loss(image_feat, text_feat, idx=idx)
            loss_itm = self.get_matching_loss(image_embeds, image_atts, image_feat, text_embeds, text_atts, text_feat, idx=idx)
            return loss_itc, loss_itm
        image_embeds, image_atts, image_hidden_states, image_attentions = self.get_vision_embeds(
            image, output_attentions=output_attentions, output_hidden_states=output_hidden_states)
        text_embeds, text_hidden_states, text_attentions = self.get_text_embeds(text_ids, text_atts, output_attentions=output_attentions,
                                                                                output_hidden_states=output_hidden_states)
        image_feat, text_feat = self.get_features(image_embeds, text_embeds)
        itm = self.get_matching_loss(image_embeds, image_atts, image_feat, text_embeds, text_atts, text_feat, idx=idx,
                                     output_attentions=output_attentions, output_hidden_states=output_hidden_states)
        hidden_dict = {"image_hidden_states": image_hidden_states, "text_hidden_states": text_hidden_states,
                       "itm_pos_hidden_states": itm["pos_hidden_states"], "itm_neg_hidden_states": itm["neg_hidden_states"]}
        attention_dict = {"image_attentions": image_attentions, "text_attentions": text_attentions,
                          "itm_pos_attentions": itm["pos_attentions"], "itm_neg_attentions": itm["neg_attentions"]}
        cross_attention_dict = {"itm_pos_cross_attentions": itm["pos_cross_attentions"],
                                "itm_neg_cross_attentions": itm["neg_cross_attentions"]}
        return {"hidden_dict": hidden_dict, "attention_dict": attention_dict, "cross_attention_dict": cross_attention_dict,
                "logits_dict": {"itm_head_logits": itm["logits"]}}


def itr_kd_losses(student_outputs, teacher_outputs, temperature=1.0):
    """All KD terms of an ITR pruning step (Eff_Retrieval.py:100-163) with ONE multi-pair MSE launch."""
    sh, th = student_outputs["hidden_dict"], teacher_outputs["hidden_dict"]
    sa, ta = student_outputs["attention_dict"], teacher_outputs["attention_dict"]
    sc, tc = student_outputs["cross_attention_dict"], teacher_outputs["cross_attention_dict"]
    groups = [  # (name, student list, teacher list, is_attn, is_img)
        ("text_hidden", sh["text_hidden_states"], th["text_hidden_states"], False, False),
        ("text_attention", sa["text_attentions"], ta["text_attentions"], True, False),
        ("image_hidden", sh["image_hidden_states"], th["image_hidden_states"], False, True),
        ("image_attention", sa["image_attentions"], ta["image_attentions"], True, False),
        ("itm_pos_hidden", sh["itm_pos_hidden_states"], th["itm_pos_hidden_states"], False, False),
        ("itm_pos_attn", sa["itm_pos_attentions"], ta["itm_pos_attentions"], True, False),
        ("itm_pos_cross", sc["itm_pos_cross_attentions"], tc["itm_pos_cross_attentions"], True, False),
        ("itm_neg_hidden", sh["itm_neg_hidden_states"], th["itm_neg_hidden_states"], False, False),
        ("itm_neg_attn", sa["itm_neg_attentions"], ta["itm_neg_attentions"], True, False),
        ("itm_neg_cross", sc["itm_neg_cross_attentions"], tc["itm_neg_cross_attentions"], True, False),
    ]
    S, T, W, spans = [], [], [], {}
    for name, s_list, t_list, is_attn, is_img in groups:
        s_list = list(s_list)
        t_cor = get_cor_teacher(t_list, s_list, is_attn=is_attn)
        s, t, w = _kd_pairs(s_list, t_cor, is_attn, is_img)
        spans[name] = (len(S), len(S) + len(s))
        S += s
        T += t
        W += w
    per_pair = ops.mse_pairs(S, T, W)
    out = {name: per_pair[a:b].sum() for name, (a, b) in spans.items()}
    out["itm_logits"] = soft_cross_entropy(student_outputs["logits_dict"]["itm_head_logits"] / temperature,
                                           teacher_outputs["logits_dict"]["itm_head_logits"] / temperature)
    return out


def itr_loss(student_outputs, teacher_outputs, l0_module=None, global_step=0, temperature=1.0):
    """`loss` of Eff_Retrieval.py:165-178: ((itm-logit KL + 0.33 * (text + image + cross KD)) + itc + itm) * 0.5 (+ Lagrangian)."""
    kd = itr_kd_losses(student_outputs, teacher_outputs, temperature)
    loss_itc, loss_itm = student_outputs["loss"]["loss_itc"], student_outputs["loss"]["loss_itm"]
    loss_text_kd = kd["text_hidden"] + kd["text_attention"]
    loss_img_kd = 0.2 * kd["image_hidden"] + kd["image_attention"]
    loss_cross_kd = (kd["itm_neg_hidden"] + kd["itm_pos_hidden"] + kd["itm_pos_attn"] + kd["itm_pos_cross"] + kd["itm_neg_attn"]
                     + kd["itm_neg_cross"]) * 0.5
    loss_kd = kd["itm_logits"] + (loss_text_kd + loss_img_kd + loss_cross_kd) * 0.33
    loss_small = loss_itc + loss_itm
    loss = (loss_kd + loss_small) * 0.5
    parts = dict(loss_itc=loss_itc, loss_itm=loss_itm, loss_text_kd=loss_text_kd, loss_img_kd=loss_img_kd, loss_cross_kd=loss_cross_kd,
                 loss_itm_logits_kd=kd["itm_logits"], loss_kd=loss_kd, **{"kd_" + n: v for n, v in kd.items()})
    if l0_module is not None:
        lagrangian_loss, expected_sparsity, target_sparsity = l0_module.lagrangian_regularization(global_step)
        loss = loss + lagrangian_loss
        parts.update(lagrangian_loss=lagrangian_loss, expected_sparsity=expected_sparsity, target_sparsity=target_sparsity)
    return loss, parts
