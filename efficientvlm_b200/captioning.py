"""Image-captioning task models on the B200 hot path — drop-in for `efficient_models/model_generation.py::EffXVLMForCaptioning`
(L0-gated student) and `models/model_generation.py::XVLMForCaptioning` (un-gated teacher), plus the loss assembly of the
`Eff_Captioning.py` pruning step.

The reference classes own a tokenizer (`dataset.build_tokenizer(config['text_encoder'])` = BertTokenizer of bert-base-uncased).
Here it is injectable (`tokenizer=`): any object with the BertTokenizer surface the model uses (`cls_token`, `sep_token`,
`pad_token_id`, `sep_token_id`, `add_special_tokens`, `__call__`, `decode`); by default it is loaded with transformers from
`config['text_encoder']` and the constructor fails loudly when the files are not there.  `forward` also accepts an already
tokenised caption batch (an object with `.input_ids` / `.attention_mask`).

Reference behaviours kept on purpose: the student's task-loss-only branch runs the vision tower WITHOUT gates
(model_generation.py:365-366), greedy / sampling decoding runs the decoder WITHOUT gates (the kwargs are commented out at
:444-445, 457-458), beam search is delegated to transformers' GenerationMixin (un-vendored: not reproduced, SURVEY §8c).
"""
import torch

from . import checkpoint, ops
from .distill import _kd_pairs, get_cor_teacher
from .eff_bert import BertLMHeadModel
from .l0_module import XVLML0Module
from .xvlm import XVLMBase, load_pretrained


def _default_tokenizer(path):
    try:
        from transformers import BertTokenizer
        return BertTokenizer.from_pretrained(path)
    except Exception as e:  # pragma: no cover - depends on local files
        raise RuntimeError("EffXVLMForCaptioning needs the tokenizer files of %r (or pass tokenizer=...): %s" % (path, e))


class XVLMForCaptioning(XVLMBase):
    """models/model_generation.py:61-218 — un-gated captioning model (the distillation teacher of Eff_Captioning.py)."""
    gated = False
    gates_folded = False        # set by prune.materialize: the deterministic gates live in the (physically pruned) weights

    def __init__(self, config, tokenizer=None):
        super().__init__(config, load_vision_params=False, load_text_params=False, use_contrastive_loss=False, use_matching_loss=False,
                         use_mlm_loss=False, use_bbox_loss=False, config_text=None)
        self.tokenizer = tokenizer if tokenizer is not None else _default_tokenizer(config["text_encoder"])
        self.tokenizer.add_special_tokens({"bos_token": self.tokenizer.cls_token, "eos_token": self.tokenizer.sep_token})
        self.prompt = config["prompt"]
        self.prompt_length = len(self.tokenizer(self.prompt).input_ids) - 1
        self.max_tokens = config["max_tokens"]
        config_enc = self.text_encoder.config
        self.text_encoder = None
        self.text_decoder = BertLMHeadModel(config=config_enc, label_smoothing=config["label_smoothing"])
        if self.gated:
            self.l0_module = XVLML0Module(config, target_sparsity=config["sparsity"])

    def load_pretrained(self, ckpt_rpath, config, load_capt_pretrain=False, is_eval=False):
        """model_generation.py:322-343: the pre-trained text encoder becomes the caption decoder."""
        state_dict = load_pretrained(ckpt_rpath, config, is_eval=True) if is_eval else load_pretrained(ckpt_rpath, config, load_text=False)
        if not is_eval and not load_capt_pretrain:
            checkpoint.remap_keys(state_dict, checkpoint.caption_decoder_rule())
        checkpoint.load_into(self, state_dict, ckpt_rpath)

    def _tokenise(self, caption, device):
        if hasattr(caption, "input_ids"):
            return caption
        return self.tokenizer(caption, padding="longest", truncation=True, max_length=self.max_tokens, return_tensors="pt").to(device)

    def _zs(self, training):
        if not self.gated or self.gates_folded:
            return None
        if training:
            return self.l0_module.forward(training=True)
        with torch.no_grad():
            return self.l0_module.forward(training=False)

    def forward(self, image, caption, output_attentions=None, output_hidden_states=None):
        if self.gates_folded:
            raise RuntimeError("this captioning model was materialised (prune.materialize): its gates are folded into pruned weights, so the "
                               "training forward, which applies freshly sampled full-width gates, cannot run on it; use generate()")
        zs = self._zs(True)                                                    # model_generation.py:350 (sampled even when unused)
        dec_head = dec_mlp = vis_head = vis_mlp = None
        if zs is not None:
            vis_head, vis_mlp = zs["vision_head_z"], zs["vision_intermediate_z"]
            dec_head = torch.cat((zs["text_head_z"], zs["cross_head_z"]), dim=0)
            dec_mlp = torch.cat((zs["text_intermediate_z"], zs["cross_intermediate_z"]), dim=0)
        if output_attentions:
            image_embeds, image_hidden_states, image_attentions = self.vision_encoder(
                image, output_attentions=output_attentions, output_hidden_states=output_hidden_states, head_z=vis_head, mlp_z=vis_mlp)
        else:
            image_embeds = self.vision_encoder(image)[0]                       # un-gated on this branch, like the reference (:365-366)
        text = self._tokenise(caption, image.device)
        decoder_targets = text.input_ids.masked_fill(text.input_ids == self.tokenizer.pad_token_id, -100)
        decoder_targets[:, :self.prompt_length] = -100
        outputs = self.text_decoder(text.input_ids, attention_mask=text.attention_mask, encoder_hidden_states=image_embeds,
                                    encoder_attention_mask=None, labels=decoder_targets, return_dict=True,
                                    output_attentions=output_attentions, output_hidden_states=output_hidden_states, head_z=dec_head,
                                    mlp_z=dec_mlp)
        if not output_attentions:
            return outputs.loss
        return {"loss": outputs.loss,
                "hidden_dict": {"image_hidden_states": image_hidden_states, "decoder_hidden_states": outputs.hidden_states},
                "attention_dict": {"image_attentions": image_attentions, "decoder_attentions": outputs.attentions},
                "cross_attention_dict": {"decoder_cross_attentions": outputs.cross_attentions},
                "logits_dict": {"logits": outputs.logits}}

    @torch.no_grad()
    def generate(self, image, sample=False, num_beams=1, max_length=30, min_length=10, top_p=0.9, repetition_penalty=1.0,
                 num_return_sequences=1, greedy=False, return_ids=False, sync_free=False):
        """model_generation.py:407-484.  greedy / sample: the reference's own decode loop (`_generate_no_beam_search`); otherwise beam
        search (`BertLMHeadModel.generate`: transformers 4.12.5's algorithm restated, parity unpinned; on CUDA the scorer runs on the device).
        return_ids=True (extension) also returns the generated token ids; sync_free=True (extension) decodes to max_length without
        host checks or reads (same result, graph-capturable; beam-search ids are then [batch, max_length], pad-filled; see eff_bert).
        After prune.materialize the model decodes WITHOUT gates, on the vision tower and on the decoder, in every mode: the decoder's
        beam-search gates are folded into its weights, and greedy / sampling then run that folded decoder."""
        zs = self._zs(False)
        vis_head = vis_mlp = None
        if zs is not None:
            vis_head, vis_mlp = zs["vision_head_z"], zs["vision_intermediate_z"]
        prompt = [self.prompt] * image.size(0)
        image_embeds = self.vision_encoder(image, head_z=vis_head, mlp_z=vis_mlp)[0]
        if num_beams > 1:
            assert (sample is False) and (num_return_sequences == 1)
            image_embeds = image_embeds.repeat_interleave(num_beams, dim=0)
        if num_return_sequences > 1:
            assert (sample is True) and (num_beams == 1)
            image_embeds = image_embeds.repeat_interleave(num_return_sequences, dim=0)
            prompt = [self.prompt] * image_embeds.size(0)
        model_kwargs = {"encoder_hidden_states": image_embeds, "encoder_attention_mask": None}
        # the prompt never changes: its ids are tokenised and copied to the device once per (batch rows, device) — no per-call
        # host->device copy (which a CUDA-graph capture of the decode could not contain)
        key = (len(prompt), str(image.device))
        cache = self.__dict__.setdefault("_prompt_ids", {})
        if key not in cache:
            cache[key] = self.tokenizer(prompt, return_tensors="pt").input_ids.to(image.device)[:, :-1].contiguous()
        input_ids = cache[key].clone()

        def _get_captions(caption_ids):
            return [self.tokenizer.decode(output, skip_special_tokens=True)[len(self.prompt):] for output in caption_ids]

        if not (greedy or sample):
            # model_generation.py:471-483: beam search (`Eff_Captioning.py:201-202` evaluates with num_beams 3, max_length 20, min_length 5).
            # This is the one decode path on which the reference hands the decoder its gates (the greedy / sampling calls have them
            # commented out, :449-450,460-461).
            kw = {}
            if zs is not None:
                kw = dict(head_z=torch.cat((zs["text_head_z"], zs["cross_head_z"]), dim=0),
                          mlp_z=torch.cat((zs["text_intermediate_z"], zs["cross_intermediate_z"]), dim=0))
            outputs = self.text_decoder.generate(input_ids=input_ids, max_length=max_length, min_length=min_length, num_beams=num_beams,
                                                 eos_token_id=self.tokenizer.sep_token_id, pad_token_id=self.tokenizer.pad_token_id,
                                                 repetition_penalty=repetition_penalty, sync_free=sync_free, **kw, **model_kwargs)
            captions = _get_captions(outputs)
            return (captions, outputs) if return_ids else captions
        if greedy:
            assert (num_beams == 1) and (num_return_sequences == 1)
        outputs, logprobs = self.text_decoder._generate_no_beam_search(
            input_ids=input_ids, cur_len=input_ids.shape[1], max_length=max_length, do_sample=bool(sample) and not greedy, temperature=1,
            top_k=0, top_p=1, repetition_penalty=repetition_penalty, pad_token_id=self.tokenizer.pad_token_id,
            eos_token_ids=[self.tokenizer.sep_token_id], batch_size=image_embeds.size(0), sync_free=sync_free, **model_kwargs)
        captions = _get_captions(outputs)
        if greedy:
            return (captions, outputs) if return_ids else captions
        return (captions, logprobs, outputs) if return_ids else (captions, logprobs)


class EffXVLMForCaptioning(XVLMForCaptioning):
    """efficient_models/model_generation.py:303-484 — L0-gated captioning student (`l0_module` = XVLML0Module)."""
    gated = True


# ----------------------------------------------------------------------------------------------------------------------
# Eff_Captioning.py:96-148 — KD terms and the loss mix of one pruning step
# ----------------------------------------------------------------------------------------------------------------------
def caption_kd_losses(student_outputs, teacher_outputs, temperature=1.0):
    sh, th = student_outputs["hidden_dict"], teacher_outputs["hidden_dict"]
    sa, ta = student_outputs["attention_dict"], teacher_outputs["attention_dict"]
    sc, tc = student_outputs["cross_attention_dict"], teacher_outputs["cross_attention_dict"]
    groups = [
        ("image_hidden", sh["image_hidden_states"], th["image_hidden_states"], False, True),
        ("image_attention", sa["image_attentions"], ta["image_attentions"], True, False),
        ("decoder_hidden", sh["decoder_hidden_states"], th["decoder_hidden_states"], False, True),     # is_img=True in the driver (:130)
        ("decoder_attention", sa["decoder_attentions"], ta["decoder_attentions"], True, False),
        ("decoder_cross", sc["decoder_cross_attentions"], tc["decoder_cross_attentions"], True, False),
    ]
    S, T, W, spans = [], [], [], {}
    for name, s_list, t_list, is_attn, is_img in groups:
        s_list = list(s_list)
        s, t, w = _kd_pairs(s_list, get_cor_teacher(t_list, s_list, is_attn=is_attn), is_attn, is_img)
        spans[name] = (len(S), len(S) + len(s))
        S += s
        T += t
        W += w
    per_pair = ops.mse_pairs(S, T, W)
    out = {name: per_pair[a:b].sum() for name, (a, b) in spans.items()}
    sl, tl = student_outputs["logits_dict"]["logits"], teacher_outputs["logits_dict"]["logits"]
    V = sl.shape[-1]
    s2, t2 = sl.reshape(-1, V), tl.reshape(-1, V)
    out["logits"] = ops.sum_scaled(ops.kl_rows(s2, t2, 1.0 / temperature), 1.0 / s2.shape[0])
    return out


def caption_loss(student_outputs, teacher_outputs, l0_module=None, global_step=0, temperature=1.0):
    """`loss` of Eff_Captioning.py:138-148: 0.3 * (logit KL + image KD + decoder KD) + 0.7 * task (+ Lagrangian)."""
    kd = caption_kd_losses(student_outputs, teacher_outputs, temperature)
    loss_small = student_outputs["loss"]
    loss_img_kd = kd["image_attention"] + kd["image_hidden"] * 0.1
    loss_decoder_kd = kd["decoder_attention"] + kd["decoder_hidden"] + kd["decoder_cross"]
    loss_kd = kd["logits"] + loss_img_kd + loss_decoder_kd
    loss = loss_kd * 0.3 + loss_small * 0.7
    parts = dict(loss_small=loss_small, loss_kd=loss_kd, loss_img_kd=loss_img_kd, loss_decoder_kd=loss_decoder_kd, loss_logits_kd=kd["logits"],
                 **{"kd_" + n: v for n, v in kd.items()})
    if l0_module is not None:
        lagrangian_loss, expected_sparsity, target_sparsity = l0_module.lagrangian_regularization(global_step)
        loss = loss + lagrangian_loss
        parts.update(loss_lagrangian=lagrangian_loss, expected_sparsity=expected_sparsity, target_sparsity=target_sparsity)
    return loss, parts
