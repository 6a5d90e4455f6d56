#!/usr/bin/env python
"""bench.py — general-distillation (gd_4m_small) training step throughput, the metric BASELINE.json names.

    python bench.py --gpus 1 --steps 10 --warmup 3                 # ours: CUDA hot path, one process per GPU
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference --steps 2 --warmup 1          # reference arm: the CPU oracle port on the host cores
    python bench.py ... --dump-outputs DIR                         # also write the last timed step's outputs to DIR/*.npy

One step = student (CLIP-ViT-6 + BERT-3/3, train mode incl. dropout) forward with KD outputs, teacher (ViT-12 + BERT-6/6)
forward under no_grad, ITC / ITM / MLM losses, all KD losses (hidden + attention MSE with layer mapping, logit KL), backward,
data-parallel gradient mean-allreduce, global-norm clip 1.0, AdamW — on a batch of 128 image-text pairs per GPU at 224 px,
40 tokens, 8 masked positions (SURVEY §8d C2).  Synthetic data, random-init weights of the named architectures.

Prints ONE JSON line (rank 0).  `value` = pairs/s with inputs resident in HBM; `e2e` = the same step driven from pinned HOST
buffers (H2D copies and the loss read-back inside the timed region).
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

FLOP_PER_PAIR = 176.1e9  # SURVEY §8(d) C2: (3 x 4525 + 8970) GFLOP per 128-pair GPU batch
FLOP_PER_VQA_STEP_SAMPLE = 506.0e9     # SURVEY §8(d) C3: 8101 GFLOP per 16-sample pruning step at 480 px
FLOP_PER_VQA_INFER_SAMPLE = 165.0e9    # SURVEY §8(d) C5: 3967 GFLOP per 24-sample batch, dense (un-pruned) count
FLOP_PER_CAPTION = 57.0e9              # C5 captioning: ViT-6 forward at 384 px (55.8 GFLOP) + 16 single-token decoder steps (~1 GFLOP)
# region batch (48 images, 128 rows, local_attn_depth 2 of 6 / 4 of 12), from the C2 count: the ViT's non-local layers see 48 rows and its
# local layers 176, i.e. 544 / 768 of the GD step's ViT row-layers (student 2234 -> 1582, teacher 4468 -> 3165 GFLOP); the text / fusion
# passes are the GD step's (2291 / 4502) plus one more fusion pass for the bbox head (432 / 864): (3 x 4305 + 8531) GFLOP per 128 rows
FLOP_PER_REGION_ROW = 167.5e9
# NLVR2 step (Eff_NLVR.py; two 384 px images per text): ViT over 2 images per sample (2 x 55.8 GFLOP student, 2 x 111.6 teacher),
# 3 text + 6 fusion layers (student; 6 + 12 teacher) over 40 tokens, every fusion layer projecting K | V of one image's 577 tokens
# (1.7 + 12.3 GFLOP student, twice that teacher): 3 x 125.6 (student forward + backward) + 251.2 (teacher forward) GFLOP per sample
FLOP_PER_NLVR_SAMPLE = 628.0e9
FLOP_PER_ITR_PAIR = 381.4e9            # SURVEY §8(d) C4: 3 x 76.4 (student fwd + bwd) + 152.2 (teacher fwd) GFLOP per pair at 384 px

WORKLOADS = {
    # name: (metric, unit, default batch/GPU, image res, algorithmic FLOP per unit)
    "gd": ("GD train image-text pairs/s", "pairs/s", 128, 224, FLOP_PER_PAIR),
    "vqa_step": ("VQA-480 pruning step samples/s", "samples/s", 16, 480, FLOP_PER_VQA_STEP_SAMPLE),
    "vqa_infer": ("pruned VQA inference samples/s", "samples/s", 24, 480, FLOP_PER_VQA_INFER_SAMPLE),
    "itr_step": ("ITR-COCO pruning step pairs/s", "pairs/s", 128, 384, FLOP_PER_ITR_PAIR),
    "caption_infer": ("pruned COCO caption generation captions/s", "captions/s", 32, 384, FLOP_PER_CAPTION),
    # the region-batch half of a GD iteration (GeneralDistill.py:158-260, config `regions`): 128 region/caption rows over 48 images
    "gd_region": ("GD train region-text rows/s", "rows/s", 128, 224, FLOP_PER_REGION_ROW),
    # the fourth pruning driver (Eff_NLVR.py, configs/x-vlm-small-ft/NLVR.yaml: batch 10 per GPU, 384 px, two images per text)
    "nlvr_step": ("NLVR2 pruning step samples/s", "samples/s", 10, 384, FLOP_PER_NLVR_SAMPLE),
}


def make_cfg(kind, image_res):
    return dict(image_res=image_res, patch_size=16, use_clip_vit=True, use_swin=False,
                vision_config="config_clipvit_small.json" if kind == "student" else "config_clipvitB.json", text_encoder=None,
                text_num_hidden_layers=6 if kind == "student" else 12, embed_dim=256, temp=0.07)


def make_batch(B, image_res, seed, L=40, n_mask=8, vocab=30522):
    g = torch.Generator().manual_seed(seed)
    image = torch.randn(B, 3, image_res, image_res, generator=g)
    text_ids = torch.randint(1000, vocab, (B, L), generator=g)
    text_ids[:, 0] = 101
    text_atts = torch.ones(B, L, dtype=torch.long)
    masked_pos = torch.stack([torch.randperm(L - 1, generator=g)[:n_mask].sort().values + 1 for _ in range(B)])
    masked_ids = torch.gather(text_ids, 1, masked_pos)
    text_ids_masked = text_ids.clone().scatter_(1, masked_pos, 103)
    return [image, text_ids, text_atts, text_ids_masked, masked_pos, masked_ids]


def make_region_batch(R, n_img, image_res, seed, L=40, n_mask=8, vocab=30522, max_regions=5, patch=16):
    """A synthetic batch shaped like dataset/pretrain_dataset.py:478-526's collate: `n_img` images, each with one whole-image caption row
    (is_image = 1, full patch mask, box (0.5, 0.5, 1, 1)) and `max_regions - 1` region rows (patch mask = the box's patches + [CLS],
    :461-476), of which R rows are kept in random order."""
    g = torch.Generator().manual_seed(seed)
    image, text_ids, text_atts, text_ids_masked, masked_pos, masked_ids = make_batch(R, image_res, seed, L, n_mask, vocab)
    image = torch.randn(n_img, 3, image_res, image_res, generator=g)
    npatch = image_res // patch
    rows = [(i, j) for i in range(n_img) for j in range(max_regions)]
    keep = torch.randperm(len(rows), generator=g)[:R].tolist()
    if len(keep) < R:
        keep = (keep * (R // len(keep) + 1))[:R]
    idx, atts, boxes, is_image = [], [], [], []
    for k in keep:
        i, j = rows[k]
        idx.append(i)
        if j == 0:
            atts.append(torch.ones(1 + npatch * npatch, dtype=torch.long))
            boxes.append(torch.tensor([0.5, 0.5, 1.0, 1.0]))
            is_image.append(1)
            continue
        w, h = (torch.rand(2, generator=g) * 0.5 + 0.15).tolist()
        x, y = (torch.rand(1, generator=g).item() * (1 - w), torch.rand(1, generator=g).item() * (1 - h))
        x0 = min(math.floor(x * npatch), npatch - 1)
        x1 = max(x0 + 1, min(math.ceil((x + w) * npatch), npatch))
        y0 = min(math.floor(y * npatch), npatch - 1)
        y1 = max(y0 + 1, min(math.ceil((y + h) * npatch), npatch))
        m = torch.zeros(npatch, npatch, dtype=torch.long)
        m[y0:y1, x0:x1] = 1
        atts.append(torch.cat([torch.ones(1, dtype=torch.long), m.flatten()]))
        boxes.append(torch.tensor([x + w / 2, y + h / 2, w, h]))
        is_image.append(0)
    return [image, text_ids, text_atts, text_ids_masked, masked_pos, masked_ids, torch.tensor(idx), torch.stack(atts), torch.stack(boxes),
            torch.tensor(is_image, dtype=torch.long)]


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled every 200 ms DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([s.strip() for s in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(s) > 2 + i and s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.samples[0][1]) if self.samples[0][1] else None,
                "reasons": reasons, "samples": len(self.samples)}


class Tok:
    """The two fields of a tokenizer output the VQA models read."""

    def __init__(self, input_ids, attention_mask):
        self.input_ids, self.attention_mask = input_ids, attention_mask


def vqa_cfg(kind, image_res, sparsity=0.35):
    return dict(image_res=image_res, patch_size=16, use_clip_vit=True, use_swin=False,
                vision_config="config_clipvit_small.json" if kind == "student" else "config_clipvitB.json", text_encoder=None,
                text_num_hidden_layers=6 if kind == "student" else 12, num_dec_layers=3 if kind == "student" else 6, pad_token_id=0,
                sparsity=sparsity)


def make_vqa_batch(B, image_res, seed, Lq=16, La=4, k=2, vocab=30522):
    """SURVEY §8(d) C3: image [B,3,480,480], question ids [B,16], k=2 answers per question of 4 tokens ([CLS] a b [SEP]), weights 0.5."""
    g = torch.Generator().manual_seed(seed)
    image = torch.randn(B, 3, image_res, image_res, generator=g)
    q_ids = torch.randint(1000, vocab, (B, Lq), generator=g)
    q_ids[:, 0] = 101
    q_atts = torch.ones(B, Lq, dtype=torch.long)
    a_ids = torch.randint(1000, vocab, (B * k, La), generator=g)
    a_ids[:, 0], a_ids[:, -1] = 101, 102
    a_atts = torch.ones(B * k, La, dtype=torch.long)
    weights = torch.full((B * k,), 1.0 / k)
    rows = torch.arange(B, dtype=torch.int32).repeat_interleave(k)
    return [image, q_ids, q_atts, a_ids, a_atts, weights, rows]


def make_answer_list(n=3129, La=4, seed=7, vocab=30522):
    """VQA answer list stand-in: 3129 candidates x 4 tokens with distinct first answer tokens (the real list is mostly distinct)."""
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(1000, vocab, (n, La), generator=g)
    ids[:, 0], ids[:, -1] = 101, 102
    ids[:, 1] = torch.randperm(vocab - 1000, generator=g)[:n] + 1000
    return ids, torch.ones(n, La, dtype=torch.long)


def l0_noise(n, generator=None):
    """xvlm_l0_module.py:180-182: U(1e-6, 1 - 1e-6) drawn on the CPU generator (quirk Q5), one flat buffer for all gate types."""
    return torch.empty(n).uniform_(1e-6, 1 - 1e-6, generator=generator)


def cpu_vqa_arm(workload, steps, warmup, sample_batch, image_res, threads):
    """CPU oracle port of the VQA workloads (oracle/vqa_oracle.py, fp32) on a bounded sample of the same workload."""
    from efficientvlm_b200.vqa import EffXVLMForVQA, XVLMForVQA
    from oracle import vqa_oracle as V
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    student = EffXVLMForVQA(vqa_cfg("student", image_res))
    ssd = dict(student.state_dict())
    for k, v in student.named_parameters():
        ssd[k] = v
    ssd["text_decoder.cls.predictions.decoder.weight"] = ssd["text_decoder.bert.embeddings.word_embeddings.weight"]
    s_cfg = dict(vit_layers=6, vit_heads=12, text_layers=6, text_heads=12, dec_layers=3)
    layout, _ = V.l0_layout(768, 3072, 12, 6, 6)
    logas = {t: ssd["l0_module." + t.replace("_intermediate", "_int") + "_loga"] for t in layout}
    times = []
    if workload == "vqa_step":
        teacher = XVLMForVQA(vqa_cfg("teacher", image_res))
        tsd = dict(teacher.state_dict())
        tsd["text_decoder.cls.predictions.decoder.weight"] = tsd["text_decoder.bert.embeddings.word_embeddings.weight"]
        t_cfg = dict(vit_layers=12, vit_heads=12, text_layers=12, text_heads=12, dec_layers=6)
        image, q_ids, q_atts, a_ids, a_atts, weights, _ = make_vqa_batch(sample_batch, image_res, 1)
        batch = (image, q_ids, q_atts, a_ids, a_atts, [2] * sample_batch, weights)
        params = [p for p in student.parameters() if p.requires_grad]
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            zs = V.sample_gates(layout, logas, {t: l0_noise(logas[t].numel()).view(logas[t].shape) for t in layout})
            total, _, _ = V.vqa_step(ssd, tsd, s_cfg, t_cfg, batch, zs)
            grads = torch.autograd.grad(total, params, allow_unused=True)
            del grads
            if it >= warmup:
                times.append(time.perf_counter() - t0)
    else:
        image, q_ids, q_atts = make_vqa_batch(sample_batch, image_res, 1)[:3]
        l_ids, l_atts = make_answer_list()
        with torch.no_grad():
            ze = V.deterministic_gates(layout, {t: v.detach() for t, v in logas.items()})
            sd = {k: v.detach() for k, v in ssd.items()}
            for it in range(warmup + steps):
                t0 = time.perf_counter()
                V.eval_forward(sd, s_cfg, image, q_ids, q_atts, l_ids, l_atts, 128, ze)
                if it >= warmup:
                    times.append(time.perf_counter() - t0)
    med = sorted(times)[len(times) // 2]
    return sample_batch / med, med


def build_vqa_step(args, dev, rank, world):
    """BASELINE config 3: one modal-adaptive pruning step of Eff_VQA.py:99-199 — L0-gated student (ViT-6 + BERT 3/3 + decoder 3)
    forward with KD outputs, un-gated teacher (ViT-12 + BERT 6/6 + decoder 6) forward, task loss + eleven KD terms + Lagrangian,
    backward, the three AdamW steps (weights, log-alphas, lambdas: ascent), log-alpha clamp."""
    from efficientvlm_b200.optim import LinearWarmupDecay, create_L0_optimizer, create_optimizer
    from efficientvlm_b200.vqa import EffXVLMForVQA, XVLMForVQA, set_vqa_teacher_attention_stride, vqa_loss
    torch.manual_seed(42)
    student = EffXVLMForVQA(vqa_cfg("student", args.image_res)).to(dev).train()
    teacher = XVLMForVQA(vqa_cfg("teacher", args.image_res)).to(dev).eval()
    for p in teacher.parameters():
        p.requires_grad_(False)
    set_vqa_teacher_attention_stride(teacher, student)
    l0 = student.l0_module
    l0.set_lagrangian_warmup_steps(1000)

    class WeightsOnly:      # FlatAdamW owns every parameter exactly once: the gate parameters belong to the two L0 optimizers
        init_params = student.init_params

        @staticmethod
        def named_parameters():
            return [(n, p) for n, p in student.named_parameters() if not n.startswith("l0_module.")]
    opt = create_optimizer(dict(lr=5e-5, weight_decay=0.01, lr_mult=2), WeightsOnly)
    l0_opt, lag_opt = create_L0_optimizer(dict(reg_learning_rate=0.01), l0)
    opts = [opt, l0_opt, lag_opt]
    for o in opts:
        o.broadcast_parameters(0)
    sched = LinearWarmupDecay(opt, 100000, 0.1)
    n_noise = sum(la.numel() for la in l0.z_logas.values())
    gen = torch.Generator().manual_seed(42 + rank)      # per-rank gate noise (Eff_VQA.py:269 seeds every rank differently)
    host = [t.pin_memory() for t in make_vqa_batch(args.batch, args.image_res, 42 + rank)] + [l0_noise(n_noise, gen).pin_memory()]
    step_t = torch.zeros((), dtype=torch.float32, device=dev)

    def refresh_host():     # new gate noise for the next step, drawn on the host like the reference; part of the e2e H2D traffic
        host[-1].copy_(l0_noise(n_noise, gen))

    def device_step(image, q_ids, q_atts, a_ids, a_atts, weights, rows, noise):
        cursor = [0]

        def get_eps(size):
            n = size.numel()
            v = noise[cursor[0]:cursor[0] + n].view(size.shape)
            cursor[0] += n
            return v
        l0.get_eps = get_eps
        q, a = Tok(q_ids, q_atts), Tok(a_ids, a_atts)
        so = student(image, q, a, train=True, weights=weights, answer_rows=rows, output_attentions=True, output_hidden_states=True)
        with torch.no_grad():
            to = teacher(image, q, a, train=True, weights=weights, answer_rows=rows, output_attentions=True, output_hidden_states=True)
        loss, _ = vqa_loss(so, to, l0, step_t, 1.0)
        loss.backward()
        for o in opts:
            o.step()
        for o in opts:
            o.zero_grad()
        l0.constrain_parameters()
        step_t.add_(1.0)
        return loss

    def host_fn():
        sched.step()
        refresh_host()
    return dict(student=student, device_step=device_step, host=host, optimizers=opts, host_fn=host_fn, units=args.batch,
                schedule="student + teacher forward with KD outputs (teacher materialises only the attention maps the KD terms read), "
                         "k=2 answers per question through the decoder's row -> question cross-attention index, gate noise drawn on "
                         "the host every step and copied in with the batch")


def itr_cfg(kind, image_res, sparsity=0.25):
    return dict(image_res=image_res, patch_size=16, use_clip_vit=True, use_swin=False,
                vision_config="config_clipvit_small.json" if kind == "student" else "config_clipvitB.json", text_encoder=None,
                text_num_hidden_layers=6 if kind == "student" else 12, embed_dim=256, temp=0.07, sparsity=sparsity)


def make_itr_batch(B, image_res, seed, rank=0, L=40, vocab=30522):
    """SURVEY §8(d) C4: image [B,3,384,384], 40-token captions, idx = arange over the GLOBAL batch (this rank's slice)."""
    g = torch.Generator().manual_seed(seed)
    image = torch.randn(B, 3, image_res, image_res, generator=g)
    text_ids = torch.randint(1000, vocab, (B, L), generator=g)
    text_ids[:, 0] = 101
    text_atts = torch.ones(B, L, dtype=torch.long)
    idx = torch.arange(rank * B, (rank + 1) * B)
    return [image, text_ids, text_atts, idx]


def cpu_itr_arm(steps, warmup, sample_batch, image_res, threads):
    """CPU oracle port of the ITR pruning step (oracle/itr_oracle.py, fp32) on a bounded sample."""
    from efficientvlm_b200.distill import EffXVLMforRetrieval, XVLMforRetrieval
    from oracle import itr_oracle as R
    from oracle import xvlm_oracle as O
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    student, teacher = EffXVLMforRetrieval(itr_cfg("student", image_res)), XVLMforRetrieval(itr_cfg("teacher", image_res))
    ssd = dict(student.state_dict())
    for k, v in student.named_parameters():
        ssd[k] = v
    tsd = dict(teacher.state_dict())
    s_cfg = dict(vit_layers=6, vit_heads=12, text_layers=6, text_heads=12)
    t_cfg = dict(vit_layers=12, vit_heads=12, text_layers=12, text_heads=12)
    l0 = student.l0_module
    batch = tuple(make_itr_batch(sample_batch, image_res, 1))
    params = [p for p in student.parameters() if p.requires_grad]
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        zs = {t + "_z": O.l0_sample_z(l0.z_logas[t], l0_noise(l0.z_logas[t].numel()).view(l0.z_logas[t].shape)).reshape(l0.shapes[t]) for t in l0.types}
        total, _, _ = R.itr_step(ssd, tsd, s_cfg, t_cfg, batch, zs)
        grads = torch.autograd.grad(total, params, allow_unused=True)
        del grads
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    med = sorted(times)[len(times) // 2]
    return sample_batch / med, med


def cpu_caption_arm(steps, warmup, sample_batch, image_res, threads):
    """CPU oracle port of greedy captioning (oracle/xvlm_oracle.py: ViT + causal decoder with KV cache, fp32) on a bounded sample."""
    from efficientvlm_b200.captioning import EffXVLMForCaptioning
    from oracle import vqa_oracle as V
    from oracle import xvlm_oracle as O
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    cfg = dict(itr_cfg("student", image_res), prompt="a picture of ", max_tokens=40, label_smoothing=0.1)
    model = EffXVLMForCaptioning(cfg, tokenizer=PromptTokenizer())
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    sd["text_decoder.cls.predictions.decoder.weight"] = sd["text_decoder.bert.embeddings.word_embeddings.weight"]
    layout, _ = V.l0_layout(768, 3072, 12, 6, 6)
    logas = {t: sd["l0_module." + t.replace("_intermediate", "_int") + "_loga"] for t in layout if not t.startswith("decoder")}
    ze = V.deterministic_gates({t: layout[t] for t in logas}, logas)
    image = torch.randn(sample_batch, 3, image_res, image_res, generator=torch.Generator().manual_seed(1))
    times = []
    with torch.no_grad():
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            img, _, _ = O.vit_forward(sd, "vision_encoder", image, 12, 6, head_z=ze["vision_head_z"], mlp_z=ze["vision_intermediate_z"])
            ids = torch.tensor([PromptTokenizer.PROMPT[:-1]] * sample_batch)
            past = None
            for _ in range(20 - ids.shape[1]):
                step_ids = ids if past is None else ids[:, -1:]
                _, logits, o = O.lm_head_forward(sd, "text_decoder", 12, 6, 3, step_ids, torch.ones(sample_batch, ids.shape[1], dtype=torch.long), img,
                                                 torch.ones(img.shape[:2]), past_key_values=past)
                past = o["cache"]
                ids = torch.cat([ids, logits[:, -1].argmax(-1, keepdim=True)], 1)
            if it >= warmup:
                times.append(time.perf_counter() - t0)
    med = sorted(times)[len(times) // 2]
    return sample_batch / med, med


def build_itr_step(args, dev, rank, world):
    """BASELINE config 4: one ITR-COCO pruning step of Eff_Retrieval.py:96-197 — L0-gated student and un-gated teacher forward with
    KD outputs, ITC over the all_gather'ed image/text features of every rank, ITM with hard negatives, ten KD MSE terms + ITM-logit
    KL + Lagrangian, backward, gradient mean-allreduce, the three AdamW steps, log-alpha clamp."""
    from efficientvlm_b200 import ops
    from efficientvlm_b200.distill import EffXVLMforRetrieval, XVLMforRetrieval, itr_loss, set_teacher_attention_stride
    from efficientvlm_b200.optim import LinearWarmupDecay, create_L0_optimizer, create_optimizer
    torch.manual_seed(42)
    student = EffXVLMforRetrieval(itr_cfg("student", args.image_res)).to(dev).train()
    teacher = XVLMforRetrieval(itr_cfg("teacher", args.image_res)).to(dev).eval()
    for p in teacher.parameters():
        p.requires_grad_(False)
    set_teacher_attention_stride(teacher, student)
    l0 = student.l0_module
    l0.set_lagrangian_warmup_steps(1000)

    class WeightsOnly:      # FlatAdamW owns every parameter exactly once: the gate parameters belong to the two L0 optimizers
        init_params = student.init_params

        @staticmethod
        def named_parameters():
            return [(n, p) for n, p in student.named_parameters() if not n.startswith("l0_module.")]
    opt = create_optimizer(dict(lr=3e-5, weight_decay=0.01, lr_mult=2), WeightsOnly)
    l0_opt, lag_opt = create_L0_optimizer(dict(reg_learning_rate=0.01), l0)
    opts = [opt, l0_opt, lag_opt]
    for o in opts:
        o.broadcast_parameters(0)
    sched = LinearWarmupDecay(opt, 100000, 0.1)
    ops.manual_seed(42 + rank)
    torch.manual_seed(42 + rank)
    n_noise = sum(la.numel() for la in l0.z_logas.values())
    gen = torch.Generator().manual_seed(42 + rank)
    host = [t.pin_memory() for t in make_itr_batch(args.batch, args.image_res, 42 + rank, rank)] + [l0_noise(n_noise, gen).pin_memory()]
    step_t = torch.zeros((), dtype=torch.float32, device=dev)

    def device_step(image, text_ids, text_atts, idx, noise):
        cursor = [0]

        def get_eps(size):
            n = size.numel()
            v = noise[cursor[0]:cursor[0] + n].view(size.shape)
            cursor[0] += n
            return v
        l0.get_eps = get_eps
        so = student(image, text_ids, text_atts, idx=idx, output_attentions=True, output_hidden_states=True)
        with torch.no_grad():
            to = teacher(image, text_ids, text_atts, idx=idx, output_attentions=True, output_hidden_states=True)
        loss, _ = itr_loss(so, to, l0, step_t, 1.0)
        loss.backward()
        for o in opts:
            o.step()
        for o in opts:
            o.zero_grad()
        l0.constrain_parameters()
        step_t.add_(1.0)
        return loss

    def host_fn():
        sched.step()
        host[-1].copy_(l0_noise(n_noise, gen))
    return dict(student=student, device_step=device_step, host=host, optimizers=opts, host_fn=host_fn, units=args.batch,
                schedule="student + teacher forward with KD outputs (teacher materialises only the attention maps the KD terms read), ITC on "
                         "the packed all_gather of image/text features, ITM positives + negatives in one 3B fusion pass, gate noise drawn "
                         "on the host every step and copied in with the batch")


def make_nlvr_batch(B, image_res, seed, L=40, vocab=30522):
    """Eff_NLVR.py:90-97: image0 / image1 concatenated along the batch ([2B, 3, R, R]), one 40-token sentence per pair, a binary target."""
    g = torch.Generator().manual_seed(seed)
    image = torch.randn(2 * B, 3, image_res, image_res, generator=g)
    text_ids = torch.randint(1000, vocab, (B, L), generator=g)
    text_ids[:, 0] = 101
    return [image, text_ids, torch.ones(B, L, dtype=torch.long), torch.randint(0, 2, (B,), generator=g)]


def cpu_nlvr_arm(steps, warmup, sample_batch, image_res, threads):
    """CPU oracle port of the NLVR2 pruning step (oracle/nlvr_oracle.py, fp32) on a bounded sample."""
    from efficientvlm_b200.nlvr import EffXVLMForNLVR, XVLMForNLVR
    from oracle import nlvr_oracle as N
    from oracle import xvlm_oracle as O
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    student, teacher = EffXVLMForNLVR(itr_cfg("student", image_res)), XVLMForNLVR(itr_cfg("teacher", image_res))
    ssd = dict(student.state_dict())
    for k, v in student.named_parameters():
        ssd[k] = v
    tsd = dict(teacher.state_dict())
    for m, sd in ((student, ssd), (teacher, tsd)):          # tied cross-attention K / V: the shared tensor under both layer names
        for i in range(m.num_cross_layers):
            a, b = m.num_text_layers + 2 * i, m.num_text_layers + 2 * i + 1
            for kv in ("key", "value"):
                for wb in ("weight", "bias"):
                    sd["text_encoder.encoder.layer.%d.crossattention.self.%s.%s" % (a, kv, wb)] = \
                        sd["text_encoder.encoder.layer.%d.crossattention.self.%s.%s" % (b, kv, wb)]
    s_cfg = dict(vit_layers=6, vit_heads=12, text_layers=6, text_heads=12)
    t_cfg = dict(vit_layers=12, vit_heads=12, text_layers=12, text_heads=12)
    l0 = student.l0_module
    batch = tuple(make_nlvr_batch(sample_batch, image_res, 1))
    params = [p for p in student.parameters() if p.requires_grad]
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        zs = {t + "_z": O.l0_sample_z(l0.z_logas[t], l0_noise(l0.z_logas[t].numel()).view(l0.z_logas[t].shape)).reshape(l0.shapes[t]) for t in l0.types}
        so = N.nlvr_forward(ssd, s_cfg, *batch, zs=zs)
        with torch.no_grad():
            to = N.nlvr_forward(tsd, t_cfg, *batch)
        total, _ = N.nlvr_total_loss(so, to)
        grads = torch.autograd.grad(total, params, allow_unused=True)
        del grads
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    med = sorted(times)[len(times) // 2]
    return sample_batch / med, med


def build_nlvr_step(args, dev, rank, world):
    """The fourth pruning driver: one NLVR2 step of Eff_NLVR.py:73-190 — both images of a pair through the ViT as one 2B batch, the
    9-layer (student) / 18-layer (teacher) encoder whose fusion layers alternate between the two images with tied K / V projections,
    eight KD terms + the task loss + Lagrangian, backward, gradient mean-allreduce, the three AdamW steps, log-alpha clamp."""
    from efficientvlm_b200 import ops
    from efficientvlm_b200.nlvr import EffXVLMForNLVR, XVLMForNLVR, nlvr_loss
    from efficientvlm_b200.optim import LinearWarmupDecay, create_L0_optimizer, create_optimizer
    torch.manual_seed(42)
    student = EffXVLMForNLVR(itr_cfg("student", args.image_res)).to(dev).train()
    teacher = XVLMForNLVR(itr_cfg("teacher", args.image_res)).to(dev).eval()
    for p in teacher.parameters():
        p.requires_grad_(False)
    l0 = student.l0_module
    l0.set_lagrangian_warmup_steps(1000)

    class WeightsOnly:
        init_params = student.init_params

        @staticmethod
        def named_parameters():
            return [(n, p) for n, p in student.named_parameters() if not n.startswith("l0_module.")]
    opt = create_optimizer(dict(lr=3e-5, weight_decay=0.01, lr_mult=2), WeightsOnly)
    l0_opt, lag_opt = create_L0_optimizer(dict(reg_learning_rate=0.1), l0)
    opts = [opt, l0_opt, lag_opt]
    for o in opts:
        o.broadcast_parameters(0)
    sched = LinearWarmupDecay(opt, 100000, 0.1)
    ops.manual_seed(42 + rank)
    torch.manual_seed(42 + rank)
    n_noise = sum(la.numel() for la in l0.z_logas.values())
    gen = torch.Generator().manual_seed(42 + rank)
    host = [t.pin_memory() for t in make_nlvr_batch(args.batch, args.image_res, 42 + rank)] + [l0_noise(n_noise, gen).pin_memory()]
    step_t = torch.zeros((), dtype=torch.float32, device=dev)

    def device_step(image, text_ids, text_atts, targets, noise):
        cursor = [0]

        def get_eps(size):
            n = size.numel()
            v = noise[cursor[0]:cursor[0] + n].view(size.shape)
            cursor[0] += n
            return v
        l0.get_eps = get_eps
        kw = dict(targets=targets, train=True, output_attentions=True, output_hidden_states=True)
        so = student(image, text_ids, text_atts, **kw)
        with torch.no_grad():
            to = teacher(image, text_ids, text_atts, **kw)
        loss, _ = nlvr_loss(so, to, l0, step_t, 1.0)
        loss.backward()
        for o in opts:
            o.step()
        for o in opts:
            o.zero_grad()
        l0.constrain_parameters()
        step_t.add_(1.0)
        return loss

    def host_fn():
        sched.step()
        host[-1].copy_(l0_noise(n_noise, gen))
    return dict(student=student, device_step=device_step, host=host, optimizers=opts, host_fn=host_fn, units=args.batch,
                schedule="student + teacher forward with KD outputs, both images of every pair in one 2B ViT batch, fusion layers alternating "
                         "between the two images with tied K / V projections, gate noise drawn on the host every step and copied in with the batch")


class PromptTokenizer:
    """The BertTokenizer surface EffXVLMForCaptioning uses, for the fixed prompt only (bert-base-uncased ids of "a picture of");
    generated ids are not turned back into words — with random-init weights there is nothing to read."""
    cls_token, sep_token = "[CLS]", "[SEP]"
    pad_token_id, cls_token_id, sep_token_id = 0, 101, 102
    PROMPT = [101, 1037, 3861, 1997, 102]

    def add_special_tokens(self, mapping):
        pass

    def __call__(self, text, return_tensors=None, **kw):
        n = 1 if isinstance(text, str) else len(text)
        if return_tensors == "pt":
            return Tok(torch.tensor([self.PROMPT] * n), torch.ones(n, len(self.PROMPT), dtype=torch.long))
        return Tok(list(self.PROMPT), [1] * len(self.PROMPT))

    def decode(self, ids, skip_special_tokens=True):
        return ""


def build_caption_infer(args, dev, rank, world):
    """BASELINE config 5, captioning half: EffXVLMForCaptioning.generate(greedy=True) — deterministic masks on the vision tower,
    greedy decode with KV cache from the prompt "a picture of" to max_length 20 (Captioning.yaml), batch 32 at 384 px."""
    from efficientvlm_b200.captioning import EffXVLMForCaptioning
    torch.manual_seed(42)
    cfg = dict(itr_cfg("student", args.image_res, sparsity=args.sparsity), prompt="a picture of ", max_tokens=40, label_smoothing=0.1)
    model = EffXVLMForCaptioning(cfg, tokenizer=PromptTokenizer()).to(dev).eval()
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():
        for la in model.l0_module.z_logas.values():
            la.copy_((torch.randn(la.shape, generator=g) * 3.0 + args.loga_shift).to(dev))
    image = torch.randn(args.batch, 3, args.image_res, args.image_res, generator=torch.Generator().manual_seed(42 + rank))
    host = [image.pin_memory()]
    outputs = {}        # what generate() hands its caller in the latest step (under a captured graph: the graph's output buffers)

    if args.beams > 1:
        # the decode the reference's evaluation runs (Eff_Captioning.py:201-202, Captioning.yaml: num_beams 3, max_length 20, min_length 5):
        # the beam scorer reads 2 * num_beams candidates per item back to the host every step, so this is an eager, host-driven loop
        def beam_step(image):
            _, ids = model.generate(image, sample=False, num_beams=args.beams, max_length=20, min_length=5, return_ids=True)
            outputs["caption_ids"] = ids
            return ids.sum().float()
        return dict(device_step=beam_step, host=host, optimizers=[], host_fn=None, units=args.batch, eager_only=True, outputs=outputs,
                    schedule="beam search (num_beams %d, max_length 20, min_length 5: transformers 4.12.5's algorithm restated, "
                             "BertLMHeadModel._beam_search): one decoder pass over batch x beams rows per token with a re-ordered KV cache, "
                             "one device -> host read per token for the hypothesis bookkeeping (not graph-capturable)" % args.beams)

    def device_step(image):
        _, ids = model.generate(image, greedy=True, max_length=20, return_ids=True, sync_free=not args.eager)
        outputs["caption_ids"] = ids
        return ids.sum().float()
    return dict(device_step=device_step, host=host, optimizers=[], host_fn=None, units=args.batch, outputs=outputs,
                schedule="greedy decode loop of eff_bert.py:1472-1563 (one decoder pass per token, KV cache) run to max_length without the "
                         "per-token end-of-sequence check on the host (same ids; --eager keeps the check), so ViT + all decode steps are ONE "
                         "captured graph; the cross-attention K|V projections of the image tokens are computed once per caption batch")


def build_vqa_infer(args, dev, rank, world):
    """BASELINE config 5: EffXVLMForVQA.forward(train=False) = deterministic L0 masks, ViT + question encoder, rank_answer over the
    3129-entry answer list with k_test = 128 (decoder over batch x 128 candidates)."""
    from efficientvlm_b200.vqa import EffXVLMForVQA
    torch.manual_seed(42)
    model = EffXVLMForVQA(vqa_cfg("student", args.image_res, sparsity=args.sparsity)).to(dev).eval()
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():       # spread the log-alphas so that the deterministic masks remove ~sparsity of every gate type
        for la in model.l0_module.z_logas.values():
            la.copy_((torch.randn(la.shape, generator=g) * 3.0 + args.loga_shift).to(dev))
    l_ids, l_atts = (t.to(dev) for t in make_answer_list())
    image, q_ids, q_atts = make_vqa_batch(args.batch, args.image_res, 42 + rank)[:3]
    host = [image.pin_memory(), q_ids.pin_memory(), q_atts.pin_memory()]
    with torch.no_grad():
        zs = model.l0_module(training=False)
        kept = {k: float((v > 0).float().mean()) for k, v in zs.items()}
    kept_txt = ", ".join("%s %.2f" % (k[:-2], v) for k, v in kept.items())
    if args.materialize:
        # utils/vqa_utils.py recipe: fold the gates into the weights, prune the zeroed heads / FFN columns physically, run without gates
        from efficientvlm_b200 import prune
        n_before = sum(p.numel() for n, p in model.named_parameters() if not n.startswith("l0_module."))
        prune.materialize(model, zs)
        n_after = sum(p.numel() for n, p in model.named_parameters() if not n.startswith("l0_module."))
    outputs = {}        # the ranked answers of the latest step (under a captured graph: the graph's output buffers)

    def device_step(image, q_ids, q_atts):
        with torch.no_grad():
            if args.materialize:
                ids, probs, _ = model.fake_forward(image, Tok(q_ids, q_atts), Tok(l_ids, l_atts), k=128)
            else:
                ids, probs = model(image, Tok(q_ids, q_atts), Tok(l_ids, l_atts), train=False, k=128)
        outputs.update(answer_ids=ids, answer_probs=probs)
        return ids[:, 0].sum().float() + probs[:, 0].sum()     # one scalar that depends on every question's answer

    if args.materialize:
        schedule = "masks MATERIALISED (prune.materialize = update_params + prune_model_with_z of utils/vqa_utils.py): %.1f M -> %.1f M " \
                   "parameters, ragged head counts / FFN widths per layer, gate-free fake_forward (kept fraction per gate type: %s)" % (
                       n_before / 1e6, n_after / 1e6, kept_txt)
    else:
        schedule = "masked-dense: deterministic gates applied in the GEMM / attention epilogues (kept fraction per gate type: %s)" % kept_txt
    return dict(device_step=device_step, host=host, optimizers=[], host_fn=None, units=args.batch, outputs=outputs,
                schedule=schedule + "; candidates read their question through the cross-attention row index (no 128x tiling)")


def cpu_oracle_arm(steps, warmup, sample_batch, image_res, threads):
    """The reference's algorithm on the host cores (oracle port, fp32): bounded sample of the same workload."""
    from efficientvlm_b200.distill import XVLM
    from oracle import gd_oracle
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    student, teacher = XVLM(make_cfg("student", image_res)), XVLM(make_cfg("teacher", image_res))
    ssd = {k: v for k, v in student.state_dict().items()}
    tsd = {k: v for k, v in teacher.state_dict().items()}
    params = [p for p in student.parameters()]
    for k, v in student.named_parameters():
        ssd[k] = v
    ssd["text_encoder.cls.predictions.decoder.weight"] = ssd["text_encoder.bert.embeddings.word_embeddings.weight"]
    tsd["text_encoder.cls.predictions.decoder.weight"] = tsd["text_encoder.bert.embeddings.word_embeddings.weight"]
    s_cfg = dict(vit_layers=6, vit_heads=12, text_layers=6, text_heads=12)
    t_cfg = dict(vit_layers=12, vit_heads=12, text_layers=12, text_heads=12)
    batch = make_batch(sample_batch, image_res, 1)
    B = sample_batch
    negs = (torch.roll(torch.arange(B), 1), torch.roll(torch.arange(B), -1))
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        total, _, _ = gd_oracle.gd_step(ssd, tsd, s_cfg, t_cfg, batch, negs, negs)
        grads = torch.autograd.grad(total, [p for p in params if p.requires_grad], allow_unused=True)
        del grads
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    med = sorted(times)[len(times) // 2]
    return sample_batch / med, med


def cpu_region_arm(steps, warmup, sample_rows, image_res, threads):
    """The region-batch GD step on the host cores: oracle/gd_oracle.py's `region` branch (pinned by tests/test_oracle_golden.py::
    test_gd_region_oracle), `sample_rows` rows over 3/8 as many images (the 128 : 48 ratio of the full batch)."""
    from efficientvlm_b200.distill import XVLM
    from oracle import gd_oracle
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    student, teacher = XVLM(make_cfg("student", image_res)), XVLM(make_cfg("teacher", image_res))
    ssd, tsd = dict(student.state_dict()), dict(teacher.state_dict())
    params = [p for p in student.parameters()]
    for k, v in student.named_parameters():
        ssd[k] = v
    ssd["text_encoder.cls.predictions.decoder.weight"] = ssd["text_encoder.bert.embeddings.word_embeddings.weight"]
    tsd["text_encoder.cls.predictions.decoder.weight"] = tsd["text_encoder.bert.embeddings.word_embeddings.weight"]
    s_cfg = dict(vit_layers=6, vit_heads=12, text_layers=6, text_heads=12, local_attn_depth=2)
    t_cfg = dict(vit_layers=12, vit_heads=12, text_layers=12, text_heads=12, local_attn_depth=4)
    R = sample_rows
    b = make_region_batch(R, max(1, R * 3 // 8), image_res, 1)
    region = dict(idx_to_group_img=b[6], image_atts=b[7], target_bbox=b[8], is_image=b[9])
    negs = (torch.roll(torch.arange(R), 1), torch.roll(torch.arange(R), -1))
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        total, _, _ = gd_oracle.gd_step(ssd, tsd, s_cfg, t_cfg, b[:6], negs, negs, region=region)
        grads = torch.autograd.grad(total, [p for p in params if p.requires_grad], allow_unused=True)
        del grads
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    med = sorted(times)[len(times) // 2]
    return R / med, med


def torch_eager_gpu_arm(steps, warmup, batch_size, image_res, dev, autocast):
    """SURVEY 8(d)'s second comparator, opt-in (`--torch-gpu-baseline`): the SAME oracle port as the CPU arm run as eager PyTorch on this
    GPU — fp32, or bf16 autocast — at the full per-GPU batch, forward + backward of one GD step (no optimizer), device-timed with a
    synchronize on both sides.  A reported baseline only; nothing of the product runs in it."""
    from efficientvlm_b200.distill import XVLM
    from oracle import gd_oracle
    dev = torch.device(dev)
    torch.manual_seed(0)
    student, teacher = XVLM(make_cfg("student", image_res)).to(dev), XVLM(make_cfg("teacher", image_res)).to(dev)
    ssd = {k: v for k, v in student.state_dict().items()}
    tsd = {k: v for k, v in teacher.state_dict().items()}
    params = [p for p in student.parameters() if p.requires_grad]
    for k, v in student.named_parameters():
        ssd[k] = v
    ssd["text_encoder.cls.predictions.decoder.weight"] = ssd["text_encoder.bert.embeddings.word_embeddings.weight"]
    tsd["text_encoder.cls.predictions.decoder.weight"] = tsd["text_encoder.bert.embeddings.word_embeddings.weight"]
    s_cfg = dict(vit_layers=6, vit_heads=12, text_layers=6, text_heads=12)
    t_cfg = dict(vit_layers=12, vit_heads=12, text_layers=12, text_heads=12)
    batch = [t.to(dev) for t in make_batch(batch_size, image_res, 1)]
    negs = (torch.roll(torch.arange(batch_size), 1).to(dev), torch.roll(torch.arange(batch_size), -1).to(dev))

    def sync():
        if dev.type == "cuda":
            torch.cuda.synchronize(dev)
    times = []
    for it in range(warmup + steps):
        sync()
        t0 = time.perf_counter()
        with torch.autocast(dev.type, dtype=torch.bfloat16, enabled=autocast):
            total, _, _ = gd_oracle.gd_step(ssd, tsd, s_cfg, t_cfg, batch, negs, negs)
        grads = torch.autograd.grad(total, params, allow_unused=True)
        del grads, total
        sync()
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    med = sorted(times)[len(times) // 2]
    return {"value": batch_size / med, "unit": "pairs/s", "ms_per_step": med * 1e3, "batch": batch_size,
            "what": "oracle port as eager PyTorch on this GPU, %s, forward + backward of one GD step (no optimizer step), median of %d" % (
                "bf16 autocast" if autocast else "fp32", len(times))}


def build_gd(args, dev, rank, world):
    """BASELINE config 2 (the headline): one general-distillation step, see the module docstring."""
    from efficientvlm_b200 import ops
    from efficientvlm_b200.distill import XVLM, gd_loss, set_teacher_attention_stride
    from efficientvlm_b200.optim import LinearWarmupDecay, create_optimizer
    torch.manual_seed(42)   # identical initial weights on every rank (the reference broadcasts from rank 0)
    student = XVLM(make_cfg("student", args.image_res)).to(dev).train()
    teacher = XVLM(make_cfg("teacher", args.image_res)).to(dev).eval()
    for p in teacher.parameters():
        p.requires_grad_(False)
    set_teacher_attention_stride(teacher, student)     # the KD losses read every 2nd teacher attention map only
    opt = create_optimizer(dict(lr=1e-4, weight_decay=0.01, lr_mult=2), student, clip_grad_norm=1.0)
    opt.broadcast_parameters(0)
    sched = LinearWarmupDecay(opt, 100000, 2)
    ops.manual_seed(42 + rank)
    torch.manual_seed(42 + rank)
    host = [t.pin_memory() for t in make_batch(args.batch, args.image_res, 42 + rank)]

    def device_step(*batch):
        so = student(*batch, output_attentions=True, output_hidden_states=True)
        with torch.no_grad():
            to = teacher(*batch, output_attentions=True, output_hidden_states=True)
        total, _ = gd_loss(so, to, 1.0)
        total.backward()
        opt.step()
        opt.zero_grad()
        return total
    return dict(student=student, device_step=device_step, host=host, optimizers=[opt], host_fn=sched.step, units=args.batch,
                schedule="text passes batched 2B, fusion passes batched 4B with shared image K/V, teacher materialises only the "
                         "attention maps the KD losses read (every 2nd layer); same losses and gradients as the pass-by-pass schedule "
                         "(tests/test_gpu_models.py)")


def build_gd_region(args, dev, rank, world):
    """The region-batch half of a GD iteration (GeneralDistill.py:158-260; config `regions`: batch_size 128 rows, max_images 48,
    max_regions 5): its own zero_grad / backward / clip / step, `ret_bbox_loss=True`.  The last `local_attn_depth` ViT layers run on
    [rows + images] sequences under a per-row patch mask (eff_vit.py:334-367), a fourth fusion pass feeds the bbox head."""
    from efficientvlm_b200 import ops
    from efficientvlm_b200.distill import XVLM, gd_loss
    from efficientvlm_b200.optim import LinearWarmupDecay, create_optimizer
    torch.manual_seed(42)
    student = XVLM(make_cfg("student", args.image_res)).to(dev).train()
    teacher = XVLM(make_cfg("teacher", args.image_res)).to(dev).eval()
    for p in teacher.parameters():
        p.requires_grad_(False)
    opt = create_optimizer(dict(lr=1e-4, weight_decay=0.01, lr_mult=2), student, clip_grad_norm=1.0)
    opt.broadcast_parameters(0)
    sched = LinearWarmupDecay(opt, 100000, 2)
    ops.manual_seed(42 + rank)
    torch.manual_seed(42 + rank)
    n_img = max(1, args.batch * 3 // 8)
    host = [t.pin_memory() for t in make_region_batch(args.batch, n_img, args.image_res, 42 + rank)]

    def device_step(image, text_ids, text_atts, text_ids_masked, masked_pos, masked_ids, idx_to_group_img, image_atts, target_bbox, is_image):
        kw = dict(text_ids_masked=text_ids_masked, masked_pos=masked_pos, masked_ids=masked_ids, image_atts=image_atts,
                  idx_to_group_img=idx_to_group_img, target_bbox=target_bbox, is_image=is_image, ret_bbox_loss=True,
                  output_attentions=True, output_hidden_states=True)
        so = student(image, text_ids, text_atts, **kw)
        with torch.no_grad():
            to = teacher(image, text_ids, text_atts, **kw)
        _, parts = gd_loss(so, to, 1.0)
        loss_small = parts["loss_small"] + so["loss"]["loss_bbox"] + so["loss"]["loss_giou"]          # GeneralDistill.py:257
        total = 0.6 * loss_small + 0.4 * parts["loss_kd"]                                              # :259
        total.backward()
        opt.step()
        opt.zero_grad()
        return total
    return dict(student=student, device_step=device_step, host=host, optimizers=[opt], host_fn=sched.step, units=args.batch,
                schedule="pass-by-pass (the reference's order): ViT with the row gather before the local layers, text, ITM positive / "
                         "negative fusion, MLM fusion, bbox fusion over the un-masked image tokens; %d images per %d rows" % (n_img, args.batch))


def workload_text(args):
    if args.workload == "nlvr_step":
        return "NLVR2 pruning step (Eff_NLVR.py): L0 gates + Lagrangian, KD from the X-VLM-base NLVR teacher, two %dpx images per " \
               "40-token sentence, batch %d/GPU" % (args.image_res, args.batch)
    if args.workload == "gd_region":
        return "gd_4m_small GD step on a REGION batch (`regions`: 128 rows over 48 images, max_regions 5): teacher -> small student KD + " \
               "ITC/ITM/MLM + bbox L1/GIoU, local ViT layers on [rows + images] under per-row patch masks, %dpx, %d rows/GPU" % (
                   args.image_res, args.batch)
    if args.workload == "gd":
        return "gd_4m_small GD step: CLIP-ViT-B/16 X-VLM-base teacher -> small student, KD KL + hidden/attn MSE, %dpx, batch %d/GPU, " \
               "40 tokens, 8 masked" % (args.image_res, args.batch)
    if args.workload == "vqa_step":
        return "vqa_480 modal-adaptive pruning step: L0 hard-concrete gates + Lagrangian, KD from the X-VLM-base VQA teacher, %dpx, " \
               "batch %d/GPU, 16-token questions, 2 answers x 4 tokens" % (args.image_res, args.batch)
    if args.workload == "itr_step":
        return "ITR-COCO retrieval pruning step: L0 gates + Lagrangian, KD from the X-VLM-base teacher, ITC all_gather across ranks, " \
               "%dpx, batch %d/GPU (global batch 1024 at 8 GPUs), 40-token captions" % (args.image_res, args.batch)
    if args.workload == "caption_infer":
        return "pruned COCO captioning inference: deterministic L0 masks, greedy decode from the prompt to max_length 20, %dpx, batch %d/GPU" % (
            args.image_res, args.batch)
    return "pruned VQA inference: deterministic L0 masks, rank_answer over 3129 answers with k_test 128, %dpx, batch %d/GPU" % (
        args.image_res, args.batch)


DUMP_MAX_BYTES = 64 << 20
DUMP_ARENA_SAMPLE = 1 << 20     # parameter values kept per flat arena: 4 MB each, at most 12 arenas (three optimizers of four groups)


def dump_outputs(out_dir, wl, last):
    """Write what the timed path computed in its last step as `out_dir/<name>.npy` (floating data as float32, integers as float64), so
    that two builds run with the same arguments (hence the same seeded inputs) can be compared output for output.  Inference workloads:
    the arrays the model call returns.  Training steps: the loss the step returns and the parameters it updated, per flat arena of each
    optimizer — whole up to DUMP_ARENA_SAMPLE values, else that many at indices drawn from a fixed seed (the same every run)."""
    import numpy as np
    arrays = dict(wl.get("outputs") or {"loss": last})
    for i, opt in enumerate(wl["optimizers"]):
        for j, g in enumerate(opt.param_groups):
            p = g["p"]
            if p.numel() > DUMP_ARENA_SAMPLE:
                idx = torch.randint(p.numel(), (DUMP_ARENA_SAMPLE,), generator=torch.Generator().manual_seed(1000 * i + j)).sort().values
                p = p[idx.to(p.device)]
            arrays["params_opt%d_group%d" % (i, j)] = p
    arrays = {k: v.detach().cpu() for k, v in arrays.items()}
    arrays = {k: v.double() if (v.dtype == torch.float64 or not v.is_floating_point()) else v.float() for k, v in arrays.items()}
    nbytes = sum(v.numel() * v.element_size() for v in arrays.values())
    assert nbytes <= DUMP_MAX_BYTES, "--dump-outputs: %d bytes exceed the %d-byte limit" % (nbytes, DUMP_MAX_BYTES)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v.numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="gd", choices=sorted(WORKLOADS),
                    help="gd = BASELINE config 2 (headline, default); gd_region = the same iteration's region batch; vqa_step = config 3; itr_step = config 4; vqa_infer / "
                         "caption_infer = config 5")
    ap.add_argument("--batch", type=int, default=None, help="units per GPU (gd_4m_small: 128 pairs; vqa_480: 16; VQA test: 24)")
    ap.add_argument("--image-res", type=int, default=None)
    ap.add_argument("--cpu-sample-batch", type=int, default=None)
    ap.add_argument("--sparsity", type=float, default=0.35, help="vqa_infer: target sparsity recorded in the config (VQA_480.yaml:30)")
    ap.add_argument("--loga-shift", type=float, default=1.5, help="vqa_infer: mean of the synthetic log-alphas (sets the kept fraction)")
    ap.add_argument("--materialize", action="store_true", help="vqa_infer: physically prune the masked heads / FFN columns first (BASELINE config 5 "
                    "as worded: 'masks materialized') and run the gate-free forward")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-overlap", action="store_true", help="N > 1: one blocking gradient all-reduce per arena after the backward (round 1) "
                    "instead of starting the non-vision part under the vision tower's backward")
    ap.add_argument("--no-zero-skip", action="store_true", help="pruning workloads: run the dense gated FFN path (gates multiplied in the "
                    "epilogue, zeros still cost FLOPs) instead of the kept-column path")
    ap.add_argument("--gate-loga", type=float, default=None, help="vqa_step / itr_step: set every log-alpha to this value before the run "
                    "(sets the share of gates the hard-concrete sampler clamps to exactly 0: 0.0 -> ~17 %%, -1.0 -> ~35 %%, -2.2 -> ~60 %%)")
    ap.add_argument("--torch-gpu-baseline", action="store_true", help="(default at N=1 for gd since round 2; kept for old command lines)")
    ap.add_argument("--no-torch-gpu-baseline", action="store_true", help="gd, N=1: skip timing the oracle port as eager PyTorch on this GPU "
                    "(fp32 and bf16 autocast, reported as `torch_eager_gpu`: SURVEY 8d's same-box comparator; ~20 s)")
    ap.add_argument("--no-secondary", action="store_true", help="gd, N=1: skip the `secondary` entries (the second half of BASELINE.json's "
                    "metric: pruned VQA inference samples/s, masked and materialised, each from its own `bench.py --workload vqa_infer` run)")
    ap.add_argument("--beams", type=int, default=1, help="caption_infer: beam search with this many beams (the reference's evaluation "
                                                         "uses 3) instead of the greedy loop")
    ap.add_argument("--eager", action="store_true", help="issue every launch from Python each step instead of replaying the captured step graph")
    ap.add_argument("--profile-step", action="store_true", help="warm up, then run ONE step between cudaProfilerStart/Stop and exit")
    ap.add_argument("--gemm-breakdown", action="store_true", help="print the per-shape GEMM time table to stderr")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="after the timed steps, write what the last timed step computed "
                    "(model outputs, or the loss and a fixed sample of the updated parameters) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.profile_step):
        ap.error("--dump-outputs records the timed steps of --impl ours")
    metric, unit, def_batch, def_res, flop_per_unit = WORKLOADS[args.workload]
    args.batch = args.batch or def_batch
    args.image_res = args.image_res or def_res
    if args.cpu_sample_batch is None:
        args.cpu_sample_batch = {"gd": 32, "vqa_step": 2, "vqa_infer": 2, "itr_step": 4, "caption_infer": 2, "gd_region": 32, "nlvr_step": 2}[args.workload]
    # a hung collective must not hold the GPU box: dump every thread's stack and exit after EVLM_BENCH_WATCHDOG seconds
    import faulthandler
    faulthandler.dump_traceback_later(int(os.environ.get("EVLM_BENCH_WATCHDOG", "900")), exit=True)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    workload = workload_text(args)

    def cpu_arm(k, w):
        threads = os.cpu_count() or 1
        if args.workload == "gd":
            v, med = cpu_oracle_arm(k, w, args.cpu_sample_batch, args.image_res, threads)
        elif args.workload == "gd_region":
            v, med = cpu_region_arm(k, w, args.cpu_sample_batch, args.image_res, threads)
        elif args.workload == "itr_step":
            v, med = cpu_itr_arm(k, w, args.cpu_sample_batch, args.image_res, threads)
        elif args.workload == "nlvr_step":
            v, med = cpu_nlvr_arm(k, w, args.cpu_sample_batch, args.image_res, threads)
        elif args.workload == "caption_infer":
            v, med = cpu_caption_arm(k, w, args.cpu_sample_batch, args.image_res, threads)
        else:
            v, med = cpu_vqa_arm(args.workload, k, w, args.cpu_sample_batch, args.image_res, threads)
        return v, med, threads

    if args.impl == "reference":
        if rank != 0:
            return
        w = max(1, min(args.warmup, 1))
        k = args.steps
        v, med, threads = cpu_arm(k, w)
        sample = "oracle port (CPU fp32, torch autograd), %d-unit sample of the same workload, %d timed steps" % (args.cpu_sample_batch, k)
        print(json.dumps({"impl": "reference", "metric": metric, "value": v, "unit": unit, "n_gpus": args.gpus, "steps": k,
                          "warmup": w, "ms_per_step": med * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": "f32", "data": "synthetic", "config": {"workload": workload, "sample_batch": args.cpu_sample_batch},
                          "cpu_baseline": {"value": v, "unit": unit, "cores": threads, "kind": "port", "sample": sample},
                          "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    assert torch.cuda.is_available(), "bench.py (impl=ours) needs a CUDA device: the product has no CPU path"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=dev)
    from efficientvlm_b200 import kernels as K

    wl = {"gd": build_gd, "gd_region": build_gd_region, "nlvr_step": build_nlvr_step, "vqa_step": build_vqa_step, "vqa_infer": build_vqa_infer, "itr_step": build_itr_step,
          "caption_infer": build_caption_infer}[args.workload](args, dev, rank, world)
    from efficientvlm_b200 import ops as _ops
    _ops.ZERO_SKIP = not args.no_zero_skip
    if args.gate_loga is not None and wl["optimizers"] and args.workload in ("vqa_step", "itr_step", "nlvr_step"):
        for o in wl["optimizers"][1:2]:                # the gate optimizer's arena holds the log-alphas
            for g_ in o.param_groups:
                g_["p"].fill_(args.gate_loga)
    if world > 1 and wl["optimizers"] and not args.no_overlap and "student" in wl:
        wl["optimizers"][0].enable_overlap(wl["student"], "vision_encoder.")
    if wl.get("eager_only"):
        args.eager = True
    device_step, host, host_fn = wl["device_step"], wl["host"], wl["host_fn"]
    resident = [t.to(dev) for t in host]
    h2d_bytes = sum(t.numel() * t.element_size() for t in host)

    def eager_step(batch):
        total = device_step(*batch)
        if host_fn is not None:
            host_fn()
        return total

    if args.eager or args.profile_step:
        step = eager_step
    else:
        # the whole step (forward(s), losses, backward, allreduce, clip, AdamW) as ONE CUDA graph; see graph.py
        from efficientvlm_b200.graph import GraphedTrainStep
        graphed = GraphedTrainStep(device_step, resident, optimizers=wl["optimizers"], warmup=2, host_fn=None)

        def step(batch):
            out = graphed(*batch)
            if host_fn is not None:
                host_fn()
            return out

        # End-to-end loop: a prefetching input pipeline, as any training loop has.  Batch i+1 travels pinned host -> staging buffers
        # on a copy stream while step i computes; step i+1 starts with a device-to-device copy of the staging buffers into the graph's
        # static inputs.  Every step's H2D copy and loss read-back still happen inside the timed region.
        copy_stream = torch.cuda.Stream(device=dev)
        staging = [torch.empty_like(t) for t in resident]

        def prefetch():
            with torch.cuda.stream(copy_stream):
                for dst, src in zip(staging, host):
                    dst.copy_(src, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(copy_stream)
            return ev

        def e2e_loop(n):
            last = None
            ready = prefetch()
            for i in range(n):
                main = torch.cuda.current_stream(dev)
                main.wait_event(ready)
                for dst, src in zip(graphed.static_inputs, staging):
                    dst.copy_(src, non_blocking=True)
                copied = torch.cuda.Event()
                copied.record(main)
                out = graphed(*graphed.static_inputs)            # inputs already in place: replay only
                if i + 1 < n:
                    copy_stream.wait_event(copied)              # staging is free once the D2D copies have run
                    ready = prefetch()
                last = out.item()                               # D2H read of this step's loss
                ready.synchronize()                             # the in-flight H2D has read the pinned buffers ...
                if host_fn is not None:
                    host_fn()                                   # ... before the host refreshes them (scheduler, next gate noise)
            return last

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    host_ms = [0.0]

    def timed(n, from_host):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        last = None
        h0 = time.perf_counter()
        if from_host and not (args.eager or args.profile_step):
            last = e2e_loop(n)
        for _ in range(0 if (from_host and not (args.eager or args.profile_step)) else n):
            if from_host:
                batch = [t.to(dev, non_blocking=True) for t in host]
                last = step(batch).item()         # H2D of the batch (pinned -> device) + D2H read of the step's result
            else:
                last = step(resident)
        e1.record()
        host_ms[0] = (time.perf_counter() - h0) * 1e3 / n     # host time to ENQUEUE a step (diagnostic: launch-bound if ~ ms_per_step)
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            ms = t.item()
        return ms, last

    for _ in range(max(args.warmup, 3)):
        step(resident)
    if args.profile_step:
        # `ncu --profile-from-start off ... bench.py --profile-step`: exactly one steady-state step inside the profiler range
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStart()
        step(resident)
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStop()
        return
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    K.reset_launch_count()
    ms, last = timed(args.steps, False)
    launches = K.launch_count()          # launches issued from the host ...
    if not (args.eager or args.profile_step):
        launches += graphed.captured_launches * args.steps      # ... plus the libevlm kernel nodes each replay executes
    host_enqueue_ms = host_ms[0]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, wl, last)      # before the end-to-end window's steps overwrite the outputs and parameters
    ms_e2e, last_e2e = timed(args.steps, True)
    if sampler:
        sampler.stop_flag = True
    loss_val = float(last) if not torch.is_tensor(last) else float(last.item())

    # per-launch CUDA-event timing of the dominant kernel (tcgen05 GEMM) over one further step
    K.GEMM_PROFILE = []
    eager_step(resident)
    torch.cuda.synchronize()
    prof, K.GEMM_PROFILE = K.GEMM_PROFILE, None
    # same for the HBM-bound kernel families (LayerNorm, casts, KD MSE, row-softmax losses, AdamW): algorithmic bytes / CUDA-event time
    K.HBM_PROFILE = []
    eager_step(resident)
    torch.cuda.synchronize()
    hprof, K.HBM_PROFILE = K.HBM_PROFILE, None
    hbm_table = {}
    for name, a, b, nbytes in hprof:
        t = hbm_table.setdefault(name, [0, 0.0, 0])
        t[0] += 1
        t[1] += a.elapsed_time(b)
        t[2] += nbytes
    # M <= 32 forward products run on the weight-stream kernel (csrc/gemm_skinny.cu: HBM / launch-latency bound, a few microseconds each —
    # an event pair around such a launch mostly times the launch itself): they are not part of the tensor-core roofline line
    small_m = [r for r in prof if r[3][0] <= 32 and r[3][3] == 0 and r[3][4] == 0 and len(r) <= 4]
    small_m_ms = sum(r[0].elapsed_time(r[1]) for r in small_m)
    small_m_bytes = sum(2.0 * (r[3][1] * r[3][2] + r[3][0] * r[3][2] + r[3][0] * r[3][1]) for r in small_m)
    prof = [r for r in prof if not (r[3][0] <= 32 and r[3][3] == 0 and r[3][4] == 0 and len(r) <= 4)]
    gemm_ms = sum(r[0].elapsed_time(r[1]) for r in prof)
    gemm_flops_dense = sum(r[2] for r in prof)
    # zero-skip launches: executed FLOPs from the device-side kept counts of that step (read back here, outside every timed region)
    gemm_flops, skip_launches = 0.0, 0
    for r in prof:
        f = r[2]
        if len(r) > 4:
            skip_launches += 1
            for dim, t in r[4]:
                f *= min(dim, max(int(t.item()), 0)) / float(dim)
        gemm_flops += f
    prof = [r[:4] for r in prof]
    if args.gemm_breakdown and rank == 0:
        table = {}
        for a, b, f, shape in prof:
            t = table.setdefault(shape, [0, 0.0, 0.0])
            t[0] += 1
            t[1] += a.elapsed_time(b)
            t[2] += f
        print("GEMM breakdown (M, N, K, a_mn, b_mn): count, total ms, TFLOP/s", file=sys.stderr)
        for shape, (cnt, tms, fl) in sorted(table.items(), key=lambda kv: -kv[1][1]):
            print("  %-34s %4d %8.3f ms %8.1f" % (shape, cnt, tms, fl / (tms * 1e-3) / 1e12 if tms > 0 else 0), file=sys.stderr)
    # data-parallel exchange on its own (diagnostic): the gradient mean-allreduce of every arena, timed with CUDA events
    comm = None
    if world > 1 and wl["optimizers"]:
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for o in wl["optimizers"]:
            o.allreduce_gradients()
        barrier()
        c0.record()
        for _ in range(3):
            for o in wl["optimizers"]:
                o.allreduce_gradients()
        c1.record()
        barrier()
        nbytes = sum(g["g"].numel() * 4 for o in wl["optimizers"] for g in o.param_groups)
        t = torch.tensor([c0.elapsed_time(c1) / 3], device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        comm = {"grad_allreduce_ms": t.item(), "grad_bytes": nbytes, "algbw_gbps": nbytes / (t.item() * 1e-3) / 1e9,
                "note": "time of ALL arenas exchanged back to back, on their own (diagnostic).  In the step everything but the lower half of the "
                        "vision tower (%d of %d MB) is exchanged on a side stream under the vision tower's backward, in two stages "
                        "(FlatAdamW.enable_overlap); only the rest is exposed" % (sum((g_["size"] - g_.get("split2", g_.get("split", g_["size"]))) * 4 for g_ in wl["optimizers"][0].param_groups) >> 20,
                                               sum(g_["size"] * 4 for g_ in wl["optimizers"][0].param_groups) >> 20) if not args.no_overlap else
                "one NCCL all_reduce(AVG) per flat arena, after the backward (inside the captured step graph)"}
    barrier()
    if rank != 0:
        # Captured graphs keep NCCL work alive; tearing the process group down rank by rank can block on a peer that has
        # already left, so every rank leaves through a hard exit once the measurements are done.
        sys.stdout.flush()
        os._exit(0)
    peaks = {}
    for cand in (os.path.join(ROOT, "MEASURED_PEAKS.json"),):
        if os.path.exists(cand):
            peaks = json.load(open(cand))
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_burst = peaks.get("bf16_tflops", 1640.0)
    peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)" if peaks else "fallback (B200_PROFILING.md sustained ~1.4 PFLOP/s)"
    achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    units = wl["units"] * world * args.steps
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "gemm_traffic.json")     # per-launch DRAM bytes of the dominant GEMM from `ncu --set full`
    if args.workload == "gd" and os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    out = {
        "metric": metric, "value": units / (ms * 1e-3), "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": workload, "global_batch": args.batch * world, "parallelism": "dp%d" % world,
                   "launch_mode": "eager (Python issues every launch)" if (args.eager or args.profile_step) else
                   "one captured CUDA graph per step (efficientvlm_b200.graph.GraphedTrainStep), replayed",
                   "schedule": wl["schedule"],
                   "l2": "per-step working set (activations + attention maps, several GB) far exceeds the 126 MB L2; no explicit flush",
                   "final_loss" if args.workload != "vqa_infer" else "answer_checksum": loss_val,
                   "zero_skip": {"enabled": bool(_ops.ZERO_SKIP), "gemm_launches_on_kept_columns": skip_launches,
                                 "gemm_gflop_dense_gated": gemm_flops_dense / 1e9, "gemm_gflop_executed": gemm_flops / 1e9,
                                 "ffn_layer_calls": dict(_ops.SKIP_STATS), "gate_loga": args.gate_loga}},
        "e2e": {"value": units / (ms_e2e * 1e-3), "unit": unit, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                "pipeline": "every step: pinned host -> device copy of ITS batch (prefetched on a copy stream during the previous step, "
                            "as an input pipeline does), device-to-device copy into the step graph's static inputs, graph replay, "
                            ".item() read-back of the loss" if not (args.eager or args.profile_step) else "serial H2D, step, .item()"},
        "gpu_launches": int(launches), "host_enqueue_ms_per_step": host_enqueue_ms,
        "model_flops_utilization": {"flop_per_unit": flop_per_unit, "achieved_tflops_per_gpu": flop_per_unit * units / world / (ms * 1e-3) / 1e12,
                                    "frac_of_sustained_peak": flop_per_unit * units / world / (ms * 1e-3) / 1e12 / peak_tf,
                                    "frac_of_burst_peak": flop_per_unit * units / world / (ms * 1e-3) / 1e12 / peak_burst},
        "roofline": {"bound": "tensor", "kernel": "gemm_tcgen05_kernel (all QKV/O/FFN/vocab GEMMs of the step)", "achieved": achieved,
                     "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf, "frac_of_burst_peak": achieved / peak_burst, "peak_burst": peak_burst,
                     "traffic": traffic, "peak_source": peak_src,
                     "launches_per_step": len(prof), "gemm_ms_per_step": gemm_ms, "share_of_step": gemm_ms / (ms / args.steps),
                     "small_m_weight_stream_launches": {"launches": len(small_m), "eager_event_ms": round(small_m_ms, 3),
                                                        "gbytes": round(small_m_bytes / 1e9, 3),
                                                        "note": "M <= 32 products on gemm_skinny_kernel, excluded from this line; the event "
                                                                "time of a ~5 us eager launch is mostly launch latency"} if small_m else None},
        "clocks": sampler.summary() if sampler else None,
    }
    if comm is not None:
        out["comm"] = comm
    hbm_peak = peaks.get("hbm_gbs", 6500.0)
    out["hbm_kernels"] = {"peak_gbs": hbm_peak, "peak_source": "measured copy bandwidth (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback",
                          "note": "algorithmic bytes (operands read once, results written once) / CUDA-event time per launch, one eager step",
                          "kernels": [{"kernel": name, "launches": cnt, "ms": round(tms, 3), "gbytes": round(nb / 1e9, 3),
                                       "achieved_gbs": round(nb / 1e9 / (tms * 1e-3), 1) if tms > 0 else None,
                                       "frac": round(nb / 1e9 / (tms * 1e-3) / hbm_peak, 3) if tms > 0 else None}
                                      for name, (cnt, tms, nb) in sorted(hbm_table.items(), key=lambda kv: -kv[1][1])]}
    if world == 1 and not args.no_cpu_baseline:
        v, med, threads = cpu_arm(2, 1)
        out["cpu_baseline"] = {"value": v, "unit": unit, "cores": threads, "kind": "port",
                               "sample": "oracle port (CPU fp32), %d-unit sample of the same workload, median of 2 after 1 warm-up (%.1f s/step)" % (
                                   args.cpu_sample_batch, med)}
    if world == 1 and not args.no_torch_gpu_baseline and args.workload == "gd":
        torch.cuda.empty_cache()                       # (the step graph's private pool stays: ~20 GB of the 180 GB)
        out["torch_eager_gpu"] = {"fp32": torch_eager_gpu_arm(3, 2, args.batch, args.image_res, dev, False),
                                  "bf16_autocast": torch_eager_gpu_arm(3, 2, args.batch, args.image_res, dev, True)}
        bf = out["torch_eager_gpu"]["bf16_autocast"]["value"]
        out["torch_eager_gpu"]["ours_over_bf16_autocast"] = out["value"] / bf if bf else None
        out["torch_eager_gpu"]["note"] = ("the comparator runs forward + backward only (no gradient clip / AdamW), ours the whole step: "
                                          "the ratio is a lower bound")
    if world == 1 and args.workload == "gd" and not args.no_secondary:
        # BASELINE.json's metric has a second half ("pruned VQA samples/s"): one child run per flavour, its own graph / roofline / CPU arm
        import subprocess
        out["secondary"] = {}
        torch.cuda.empty_cache()                       # the child runs beside this process's ~25 GB: plenty of room in 180 GB
        for name, extra in (("vqa_infer", []), ("vqa_infer_materialized", ["--materialize"])):
            cmd = [sys.executable, os.path.abspath(__file__), "--workload", "vqa_infer", "--steps", str(args.steps), "--warmup", str(args.warmup),
                   "--no-secondary"] + extra + (["--no-cpu-baseline"] if (args.no_cpu_baseline or extra) else [])
            try:
                r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
                line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
                d = json.loads(line)
                out["secondary"][name] = {k: d.get(k) for k in ("metric", "value", "unit", "ms_per_step", "e2e", "gpu_launches", "roofline",
                                                                 "cpu_baseline", "clocks", "config", "model_flops_utilization")}
            except Exception as e:     # the headline line must not be lost to a failing side run
                out["secondary"][name] = {"error": repr(e)[:300]}
    print(json.dumps(out))
    sys.stdout.flush()
    if world > 1:
        os._exit(0)


if __name__ == "__main__":
    main()
