"""Drop-in boundary test (CPU; needs a checkout of swaggy-TN/EfficientVLM named by $EVLM_REFERENCE_ROOT, skipped without one):
the reference's OWN, unmodified task-model files (`efficient_models/model_{retrieval,generation,nlvr}.py`, `models/model_pretrain.py`)
and the ITR driver's own `evaluation` / `itm_eval` functions (`Eff_Retrieval.py:216-378`) are imported on top of our
`efficient_models.xvlm` / `models` packages (efficientvlm_b200/compat first on sys.path) and must reproduce the reference-generated
goldens.  Arithmetic comes from the test-only torch op backend (tests/ref_ops.py)."""
import os
import subprocess
import sys

import pytest

REF = os.environ.get("EVLM_REFERENCE_ROOT", "")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.skipif(not (REF and os.path.isdir(os.path.join(REF, "efficient_models"))),
                                reason="EVLM_REFERENCE_ROOT does not name a checkout of the reference code")

SCRIPT = r'''
import os, sys, types
ROOT, REF = sys.argv[1], sys.argv[2]
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "efficientvlm_b200", "compat"))   # our drop-in packages win ...
sys.path.append(REF)                                                    # ... the reference supplies everything else
import torch
from tests import ref_ops
from tests.helpers import load_golden, sd_from_spec, rel_err
import efficientvlm_b200.ops as ops, efficientvlm_b200.kernels as K

class MP:
    def setattr(self, obj, name, val): setattr(obj, name, val)
ref_ops.install(MP())
# the reference's task model, unmodified, on top of OUR XVLMBase / L0 module
import efficient_models.model_retrieval as mr
assert mr.__file__.startswith(REF), mr.__file__
import efficient_models.xvlm as ex
assert "efficientvlm_b200" in ex.__file__, ex.__file__
import efficientvlm_b200.eff_bert as eb
g = load_golden("retrieval_tiny")
cfg = dict(g["cfg"]); cfg["vision_config"] = dict(g["vis"]); cfg["text_encoder"] = None
orig = eb.BertConfig.__init__
def patched(self, **kw):
    m = dict(g["bert"]); m.update(kw); orig(self, **m)
eb.BertConfig.__init__ = patched
model = mr.EffXVLMforRetrieval(cfg).eval()
eb.BertConfig.__init__ = orig
sd = sd_from_spec(g["sd_spec"])
names = {"vision_head": "vision_head_loga", "text_head": "text_head_loga", "cross_head": "cross_head_loga",
         "vision_intermediate": "vision_int_loga", "text_intermediate": "text_int_loga", "cross_intermediate": "cross_int_loga"}
for k, v in g["l0_logas"].items():
    sd["l0_module." + names[k]] = v
model.load_state_dict(sd, strict=True)
from oracle import xvlm_oracle as O
def sampler(image_feat, text_feat, idx=None):
    w_i2t, w_t2i = O.itm_negative_weights(image_feat.detach(), text_feat.detach(), model.temp.detach(), idx)
    return w_t2i.argmax(1), w_i2t.argmax(1)
model.sample_itm_negatives = sampler
loss_itc, loss_itm = model(g["image"], g["text_ids"], g["text_atts"], idx=g["idx"])
e1, e2 = rel_err(loss_itc, g["loss_itc"]), rel_err(loss_itm, g["loss_itm"])
print("retrieval via reference task model: itc err %.2e itm err %.2e" % (e1, e2))
assert e1 < 2e-5 and e2 < 1e-4
# models/model_pretrain.py (GD teacher / student) imports `from models import XVLMBase`
import models
assert "efficientvlm_b200" in models.xvlm.__file__
import models.model_pretrain as mp
assert mp.__file__.startswith(REF)
assert issubclass(mp.XVLM, models.XVLMBase)
print("OK")
'''


def test_reference_task_models_run_on_our_core():
    r = subprocess.run([sys.executable, "-c", SCRIPT, ROOT, REF], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert "OK" in r.stdout


# ----------------------------------------------------------------------------------------------------------------------
# the other task-model files and the ITR driver's evaluation, same recipe
# ----------------------------------------------------------------------------------------------------------------------
PREAMBLE = r'''
import ast, datetime, os, sys, time, types
ROOT, REF = sys.argv[1], sys.argv[2]
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "efficientvlm_b200", "compat"))   # our drop-in packages win ...
sys.path.append(REF)                                                    # ... the reference supplies everything else
import numpy as np
import torch
from tests import ref_ops
from tests.helpers import L0_PARAM, Tokens, arm_eps, itr_eval_setup, load_golden, rel_err, sd_from_spec
from oracle.fake_tokenizer import FakeTokenizer
from oracle.ref_shim import make_config_dir          # writes a vision json + text_encoder/config.json; patches nothing

class MP:
    def setattr(self, obj, name, val): setattr(obj, name, val)
ref_ops.install(MP())

def l0_into(sd, g):
    for k, v in g["l0_logas"].items():
        sd["l0_module." + L0_PARAM[k]] = v
    sd["l0_module.lambda_1"] = torch.tensor(g["lambda_1"]); sd["l0_module.lambda_2"] = torch.tensor(g["lambda_2"])

def stub_dataset(tokenizer):
    # `efficient_models/model_generation.py:7` imports dataset.build_tokenizer; the real package drags in skimage / pycocotools
    ds = types.ModuleType("dataset"); ds.build_tokenizer = lambda *a, **k: tokenizer; sys.modules["dataset"] = ds

def ours(module):
    assert "efficientvlm_b200" in module.__file__, module.__file__

def theirs(module):
    assert module.__file__.startswith(REF), module.__file__
'''

CASES = {
    "vqa": r'''
stub_dataset(None)
import efficient_models.model_generation as mg, efficient_models.xvlm as ex, efficient_models.generation_l0_module as gl
theirs(mg); ours(ex); ours(gl)
g = load_golden("vqa_tiny")
vj, td = make_config_dir(dict(g["vis"]), dict(g["bert"]))
model = mg.EffXVLMForVQA(dict(g["scfg"], vision_config=vj, text_encoder=td)).eval()
sd = sd_from_spec(g["s_sd_spec"])
sd["text_decoder.cls.predictions.decoder.weight"] = sd["text_decoder.bert.embeddings.word_embeddings.weight"]
l0_into(sd, g)
model.load_state_dict(sd, strict=True)
q, a, al = Tokens(g["q_ids"], g["q_atts"]), Tokens(g["a_ids"], g["a_atts"]), Tokens(g["l_ids"], g["l_atts"])
arm_eps(model.l0_module, g["eps"])
so = model(g["image"], q, a, train=True, k=g["k"], weights=g["weights"], output_attentions=True, output_hidden_states=True)
e = [rel_err(so["loss"], g["s_loss"]), rel_err(so["logits_dict"]["logits"], g["s_logits"])]
ids, probs = model(g["image"], q, al, train=False, k=g["k_test"])       # the reference's own rank_answer loop on our decoder
e.append(rel_err(probs, g["topk_probs"]))
print("vqa errs", e)
assert max(e) < 1e-4 and torch.equal(ids, g["topk_ids"])
''',
    "nlvr": r'''
import efficient_models.model_nlvr as mn, efficient_models.nlvr_l0_module as nl
theirs(mn); ours(nl)
g = load_golden("nlvr_kd_tiny")
vj, td = make_config_dir(dict(g["vis"]), dict(g["bert"]))
m = mn.EffXVLMForNLVR(dict(g["scfg"], vision_config=vj, text_encoder=td)).eval()     # incl. the reference's share_cross_attention
sd = sd_from_spec(g["s_sd_spec"])
for i in range(m.num_cross_layers):
    a, b = m.num_text_layers + 2 * i, m.num_text_layers + 2 * i + 1
    for kv in ("key", "value"):
        for wb in ("weight", "bias"):
            sd["text_encoder.encoder.layer.%d.crossattention.self.%s.%s" % (a, kv, wb)] = sd["text_encoder.encoder.layer.%d.crossattention.self.%s.%s" % (b, kv, wb)]
l0_into(sd, g)
m.load_state_dict(sd, strict=True)
arm_eps(m.l0_module, g["eps"])
so = m(g["image"], g["text_ids"], g["text_atts"], targets=g["targets"], train=True, output_attentions=True, output_hidden_states=True)
e = [rel_err(so["logits_dict"]["cls_head_logits"], g["s_logits"]), rel_err(so["cross_attention_dict"]["cross_attentions"][-1], g["s_cross_last"])]
with torch.no_grad():
    pred = m(g["image"], g["text_ids"], g["text_atts"], targets=g["targets"], train=False)
e.append(rel_err(pred, g["pred_eval"]))
print("nlvr errs", e)
assert max(e) < 1e-4
''',
    "caption": r'''
g = load_golden("caption_kd_tiny")
stub_dataset(FakeTokenizer(g["bert"]["vocab_size"]))
import efficient_models.model_generation as mg
theirs(mg)
vj, td = make_config_dir(dict(g["vis"]), dict(g["bert"]))
base = os.path.dirname(td)      # the reference insists on config['text_encoder'] == 'data/bert-base-uncased' (a relative path)
os.makedirs(os.path.join(base, "data"), exist_ok=True)
os.symlink(td, os.path.join(base, "data", "bert-base-uncased"))
cwd = os.getcwd(); os.chdir(base)
m = mg.EffXVLMForCaptioning(dict(g["scfg"], vision_config=vj, text_encoder="data/bert-base-uncased")).eval()
os.chdir(cwd)
sd = sd_from_spec(g["s_sd_spec"])
sd["text_decoder.cls.predictions.decoder.weight"] = sd["text_decoder.bert.embeddings.word_embeddings.weight"]
l0_into(sd, g)
m.load_state_dict(sd, strict=True)
arm_eps(m.l0_module, g["eps"])
so = m(g["image"], g["captions"], output_attentions=True, output_hidden_states=True)
e = rel_err(so["logits_dict"]["logits"], g["s_logits"])
caps = m.generate(g["image"], greedy=True, max_length=10)      # the reference's generate() driving OUR decoder's greedy loop + KV cache
print("caption err", e, caps)
assert e < 1e-4 and caps == g["greedy_captions"]
# ... and its beam-search branch (model_generation.py:471-483, what Eff_Captioning.py:201-202 evaluates with): the reference hands
# text_decoder.generate() the gates and the pre-expanded image tokens; our decoder's generate() runs the restated HF algorithm
from efficientvlm_b200.captioning import EffXVLMForCaptioning as Ours
beams = m.generate(g["image"], sample=False, num_beams=3, max_length=12, min_length=5)
ours_m = Ours(dict(g["scfg"], vision_config=dict(g["vis"]), text_encoder=td), tokenizer=m.tokenizer).eval()   # (same id <-> word table)
ours_m.load_state_dict(sd, strict=True)
want = ours_m.generate(g["image"], sample=False, num_beams=3, max_length=12, min_length=5)
print("beam captions", beams, want)
assert beams == want and len(beams) == g["image"].shape[0]
''',
    "gd": r'''
# the HEADLINE path as GeneralDistill.py runs it: the reference's own models/model_pretrain.py::XVLM (incl. its "pretrained" tower
# loading through OUR build_vision_encoder / build_text_encoder, fed stand-in checkpoint files) as student and teacher, and the
# reference's own train-loop statements GeneralDistill.py:300-376 (lifted with `ast`) on the outputs of our kernels' host path
import contextlib, io
from tests.helpers import argmax_negatives
from oracle.make_golden_gd import config_dirs, reference_loss_code
import models, models.model_pretrain as mp
theirs(mp); ours(models.xvlm)
g = load_golden("gd_kd_tiny")
ms = []
for cfg, vis, key in ((g["scfg"], g["vis"], "s_sd_spec"), (g["tcfg"], g["tvis"], "t_sd_spec")):
    vj, td = config_dirs(dict(vis))
    with contextlib.redirect_stdout(io.StringIO()):          # the loaders list every missing key of the stand-in checkpoints
        m = mp.XVLM(dict(cfg, vision_config=vj, text_encoder=td)).eval()
    sd = sd_from_spec(g[key])
    sd["text_encoder.cls.predictions.decoder.weight"] = sd["text_encoder.bert.embeddings.word_embeddings.weight"]
    m.load_state_dict(sd, strict=True)
    m.sample_itm_negatives = argmax_negatives(m)
    ms.append(m)
student, teacher = ms
b = g["batch"]
kw = dict(text_ids_masked=b["text_ids_masked"], masked_pos=b["masked_pos"], masked_ids=b["masked_ids"], output_attentions=True,
          output_hidden_states=True)
student_outputs = student(b["image"], b["text_ids"], b["text_atts"], **kw)
with torch.no_grad():
    teacher_outputs = teacher(b["image"], b["text_ids"], b["text_atts"], **kw)
with contextlib.redirect_stdout(io.StringIO()):
    ns, code = reference_loss_code()
ns.update(student_outputs=student_outputs, teacher_outputs=teacher_outputs, device="cpu", args=types.SimpleNamespace(temperature=1.0))
exec(code, ns)
e = {k: rel_err(ns[k], v) for k, v in g["parts"].items()}
e["total"] = rel_err(ns["loss_in_total"], g["total"])
sp = dict(student.named_parameters())
grads = torch.autograd.grad(ns["loss_in_total"], [sp[n] for n in g["grad_names"]])
e["grads"] = max(rel_err(x, y) for x, y in zip(grads, g["grads"]))
print("gd errs", {k: float("%.2e" % v) for k, v in e.items()})
assert max(e.values()) < 2e-4
# ... and the region-batch half of the iteration (GeneralDistill.py:158-260, ret_bbox_loss=True) the same way
g = load_golden("gd_region_tiny")
ms = []
for cfg, vis, key in ((g["scfg"], g["vis"], "s_sd_spec"), (g["tcfg"], g["tvis"], "t_sd_spec")):
    vj, td = config_dirs(dict(vis))
    with contextlib.redirect_stdout(io.StringIO()):
        m = mp.XVLM(dict(cfg, vision_config=vj, text_encoder=td)).eval()
    sd = sd_from_spec(g[key])
    sd["text_encoder.cls.predictions.decoder.weight"] = sd["text_encoder.bert.embeddings.word_embeddings.weight"]
    m.load_state_dict(sd, strict=True)
    m.sample_itm_negatives = argmax_negatives(m)
    ms.append(m)
student, teacher = ms
b = g["batch"]
kw = dict(text_ids_masked=b["text_ids_masked"], masked_pos=b["masked_pos"], masked_ids=b["masked_ids"], image_atts=b["image_atts"],
          idx_to_group_img=b["idx_to_group_img"], target_bbox=b["target_bbox"], is_image=b["is_image"], ret_bbox_loss=True,
          output_attentions=True, output_hidden_states=True)
student_outputs = student(b["image"], b["text_ids"], b["text_atts"], **kw)
with torch.no_grad():
    teacher_outputs = teacher(b["image"], b["text_ids"], b["text_atts"], **kw)
with contextlib.redirect_stdout(io.StringIO()):
    ns, code = reference_loss_code(region=True)
ns.update(student_outputs=student_outputs, teacher_outputs=teacher_outputs, device="cpu", args=types.SimpleNamespace(temperature=1.0))
exec(code, ns)
e = {k: rel_err(ns[k], v) for k, v in g["parts"].items()}
e["total"] = rel_err(ns["loss_in_total"], g["total"])
e.update({k: rel_err(student_outputs["loss"][k], v) for k, v in g["loss"].items()})
sp = dict(student.named_parameters())
grads = torch.autograd.grad(ns["loss_in_total"], [sp[n] for n in g["grad_names"]])
e["grads"] = max(rel_err(x, y) for x, y in zip(grads, g["grads"]))
print("gd region errs", {k: float("%.2e" % v) for k, v in e.items()})
assert max(e.values()) < 2e-4
''',
    "gd_train_loop": r'''
# GeneralDistill.py::train(), the UNMODIFIED function, for 4 iterations (image batches and — where its own `random.random() <
# iter_perc` draw says so — region batches) on synthetic loaders: reference model files on our core, compat `create_optimizer` /
# `create_scheduler` / `ApexDDPAccelerator`, the reference's own `utils.MetricLogger`.  Then the same 4 iterations written directly
# against the product API (efficientvlm_b200.distill.XVLM + gd_loss + FlatAdamW + LinearWarmupDecay): logged losses and every
# student parameter after the last step must agree.
import contextlib, copy, io, random
from tests.helpers import argmax_negatives
from oracle.make_golden_gd import config_dirs
ref_ops.install_optimizer(MP())
ry = types.ModuleType("ruamel"); ry.yaml = types.ModuleType("ruamel.yaml"); sys.modules["ruamel"] = ry; sys.modules["ruamel.yaml"] = ry.yaml
ds = types.ModuleType("dataset"); ds.create_dataset = lambda *a, **k: None; sys.modules["dataset"] = ds
import typing, torch.utils.data.dataloader as _dl
if not hasattr(_dl, "T"): _dl.T = typing.TypeVar("T")        # GeneralDistill.py:24 imports a name torch 1.x exported (unused by the file)
import models, models.model_pretrain as mp, utils
import GeneralDistill as GD
theirs(GD); theirs(mp); theirs(utils); ours(models.xvlm)
import optim as c_optim, scheduler as c_sched, accelerators.apex_ddp_accelerator as c_acc
ours(c_optim); ours(c_sched); ours(c_acc)
assert GD.create_optimizer is c_optim.create_optimizer and GD.ApexDDPAccelerator is c_acc.ApexDDPAccelerator
g = load_golden("gd_region_tiny")
gi = load_golden("gd_kd_tiny")

def build(cls_of):
    ms = []
    for cfg, vis, key in ((g["scfg"], g["vis"], "s_sd_spec"), (g["tcfg"], g["tvis"], "t_sd_spec")):
        vj, td = config_dirs(dict(vis))
        with contextlib.redirect_stdout(io.StringIO()):
            m = cls_of(dict(cfg, vision_config=vj, text_encoder=td))
        sd = sd_from_spec(g[key])
        sd["text_encoder.cls.predictions.decoder.weight"] = sd["text_encoder.bert.embeddings.word_embeddings.weight"]
        m.load_state_dict(sd, strict=True)
        m.sample_itm_negatives = argmax_negatives(m)
        ms.append(m)
    return ms

bi, br = gi["batch"], g["batch"]
def image_batch(k):          # GeneralDistill.py:285-286's tuple
    gen = torch.Generator().manual_seed(100 + k)
    return [bi["image"] + 0.05 * torch.randn(bi["image"].shape, generator=gen), bi["text_ids"], bi["text_atts"], bi["text_ids_masked"],
            bi["masked_pos"], bi["masked_ids"]]
def region_batch():          # :166-170's tuple (dataset/pretrain_dataset.py:478-526's collate order)
    return [br["image"], br["idx_to_group_img"], br["text_ids"], br["text_atts"], br["text_ids_masked"], br["masked_pos"], br["masked_ids"],
            br["image_atts"], br["target_bbox"], br["is_image"]]
N_IT = 4
general_loader = [image_batch(k) for k in range(N_IT)]
region_loader = [region_batch()]
opt_cfg = dict(opt="adamW", lr=1e-3, weight_decay=0.01, lr_mult=2)
sch_cfg = dict(sched="linear", lr=1e-3, epochs=1, num_warmup_steps=2, num_training_steps=8)
config = dict(regions=dict(iter_perc=0.5), calc_image_bbox_loss=False, output_attentions=True, output_hidden_states=True,
              train_dataset_size=N_IT * bi["image"].shape[0], batch_size=bi["image"].shape[0], ckpt_frequent_step=3,
              accelerator=dict(SYNCBN=False, FP16_OPT_LEVEL="O1", FP16_LOSS_SCALE="dynamic", RNG_SEED=42, GRAD_ACCUMULATE_STEPS=1,
                               CLIP_GRAD_NORM=1.0))

class Saver:                 # utils/checkpointer.py's interface; keeps what train() hands over instead of writing to HDFS
    def __init__(self): self.saved = []
    def save_checkpoint(self, model_state, epoch, step, training_states=None):
        self.saved.append((epoch, step, sorted(model_state), training_states is not None))

# ---- (1) the reference driver -------------------------------------------------------------------------------------------
student, teacher = build(mp.XVLM)
optimizer = GD.create_optimizer(utils.AttrDict(opt_cfg), student)
scheduler = GD.create_scheduler(utils.AttrDict(sch_cfg), optimizer)
accelerator = GD.ApexDDPAccelerator(utils.AttrDict(config["accelerator"]), logger=None)
GD.args = types.SimpleNamespace(temperature=1.0)
saver = Saver()
random.seed(7); torch.manual_seed(7)
import efficientvlm_b200.ops as ops
ops.manual_seed(7)
cwd = os.getcwd(); import tempfile; os.chdir(tempfile.mkdtemp())          # train() appends to ./log.txt
buf = io.StringIO()
with contextlib.redirect_stdout(buf):
    stats = GD.train(teacher, student, general_loader, region_loader, optimizer, (0, 1), torch.device("cpu"), scheduler, config,
                     accelerator, saver)
os.chdir(cwd)
stats = {k: float(v) for k, v in stats.items()}
print("reference train():", {k: stats[k] for k in ("loss_kd", "loss_small", "region_loss_kd", "region_loss_small", "region_loss_giou", "lr")})
assert saver.saved and saver.saved[0][2] == ["config", "epoch", "lr_scheduler", "model", "optimizer"] and saver.saved[0][3]
assert scheduler.last_epoch == N_IT

# ---- (2) the same iterations on the product API ------------------------------------------------------------------------------
from efficientvlm_b200 import distill as D, optim as O2
s2, t2 = build(D.XVLM)
# (`init_params` — the lr x lr_mult group — lists whatever a model's tower loaders did not find in their checkpoint files
# (models/xvlm.py:296-315); the reference class was built over stand-in checkpoints here, so carry its list over)
s2.init_params = list(student.init_params)
opt2 = O2.create_optimizer(dict(opt_cfg), s2, clip_grad_norm=1.0)
sch2 = O2.LinearWarmupDecay(opt2, 8, 2)
random.seed(7); torch.manual_seed(7); ops.manual_seed(7)
t2.eval(); s2.train()
log = {k: [] for k in ("loss_kd", "loss_small", "region_loss_kd", "region_loss_small")}
n_region = 0
for k in range(N_IT):
    if random.random() < 0.5:                                              # GeneralDistill.py:158
        n_region += 1
        image, idx, text_ids, text_atts, tm, mpos, mids, iatts, tbox, is_img = region_batch()
        kw = dict(text_ids_masked=tm, masked_pos=mpos, masked_ids=mids, image_atts=iatts, idx_to_group_img=idx, target_bbox=tbox,
                  is_image=is_img, ret_bbox_loss=True, output_attentions=True, output_hidden_states=True)
        opt2.zero_grad()
        so = s2(image, text_ids, text_atts, **kw)
        with torch.no_grad():
            to = t2(image, text_ids, text_atts, **kw)
        _, parts = D.gd_loss(so, to, 1.0)
        small = parts["loss_small"] + so["loss"]["loss_bbox"] + so["loss"]["loss_giou"]
        (0.6 * small + 0.4 * parts["loss_kd"]).backward()
        opt2.step()
        log["region_loss_kd"].append(float(parts["loss_kd"])); log["region_loss_small"].append(float(small))
    image, text_ids, text_atts, tm, mpos, mids = image_batch(k)
    opt2.zero_grad()
    kw = dict(text_ids_masked=tm, masked_pos=mpos, masked_ids=mids, output_attentions=True, output_hidden_states=True)
    so = s2(image, text_ids, text_atts, **kw)
    with torch.no_grad():
        to = t2(image, text_ids, text_atts, **kw)
    total, parts = D.gd_loss(so, to, 1.0)
    total.backward()
    opt2.step(); sch2.step()
    log["loss_kd"].append(float(parts["loss_kd"])); log["loss_small"].append(float(parts["loss_small"]))
assert 0 < n_region < N_IT, n_region                                      # both branches of the loop ran
for k, v in log.items():
    mean = sum(v) / len(v)
    assert abs(mean - stats[k]) <= 2e-4 * max(1.0, abs(mean)), (k, mean, stats[k])     # the logger prints 5 decimals
p1, p2 = dict(student.named_parameters()), dict(s2.named_parameters())
assert set(p1) == set(p2)
# (key biases have an identically-zero true gradient — softmax is shift invariant — so Adam's m / sqrt(v) turns their rounding
# noise into O(lr) steps that depend on summation order: the one place the batched-pass schedule may differ from the pass-by-pass one)
worst = max((rel_err(p1[n], p2[n]), n) for n in p1 if not n.endswith(("key.bias", "k_proj.bias")))
print("parameters after %d iterations (%d with a region step): worst rel err %.2e (%s)" % (N_IT, n_region, worst[0], worst[1]))
assert worst[0] < 1e-5, worst
''',
    "teachers": r'''
# the un-gated teachers of the pruning steps: models/model_{generation,retrieval}.py, unmodified, on our `models` package
g = load_golden("caption_kd_tiny")
stub_dataset(FakeTokenizer(g["bert"]["vocab_size"]))
import models, models.model_generation as tg, models.model_retrieval as tr
theirs(tg); theirs(tr); ours(models.xvlm); ours(models.xbert)
from tests.helpers import argmax_negatives
# VQA teacher (Eff_VQA.py:62-63): task loss, logits, rank_answer ids
g = load_golden("vqa_tiny")
vj, td = make_config_dir(dict(g["tvis"]), dict(g["bert"]))
t = tg.XVLMForVQA(dict(g["tcfg"], vision_config=vj, text_encoder=td)).eval()
sd = sd_from_spec(g["t_sd_spec"])
sd["text_decoder.cls.predictions.decoder.weight"] = sd["text_decoder.bert.embeddings.word_embeddings.weight"]
t.load_state_dict(sd, strict=True)
q, a, al = Tokens(g["q_ids"], g["q_atts"]), Tokens(g["a_ids"], g["a_atts"]), Tokens(g["l_ids"], g["l_atts"])
with torch.no_grad():
    to = t(g["image"], q, a, train=True, k=g["k"], weights=g["weights"], output_attentions=True, output_hidden_states=True)
    ids, probs = t(g["image"], q, al, train=False, k=g["k_test"])
e = [rel_err(to["loss"], g["t_loss"]), rel_err(to["logits_dict"]["logits"], g["t_logits"]), rel_err(probs, g["t_topk_probs"])]
assert torch.equal(ids, g["t_topk_ids"])
# ITR teacher (Eff_Retrieval.py:104-106)
g = load_golden("itr_kd_tiny")
vj, td = make_config_dir(dict(g["tvis"]), dict(g["bert"]))
t = tr.XVLM(dict(g["tcfg"], vision_config=vj, text_encoder=td)).eval()
t.load_state_dict(sd_from_spec(g["t_sd_spec"]), strict=True)
t.sample_itm_negatives = argmax_negatives(t)
with torch.no_grad():
    to = t(g["image"], g["text_ids"], g["text_atts"], idx=g["idx"], output_attentions=True, output_hidden_states=True)
e += [rel_err(to["logits_dict"]["itm_head_logits"], g["t_itm_logits"]), rel_err(to["cross_attention_dict"]["itm_neg_cross_attentions"][-1], g["t_neg_cross_last"])]
# captioning teacher (Eff_Captioning.py)
g = load_golden("caption_kd_tiny")
vj, td = make_config_dir(dict(g["tvis"]), dict(g["bert"]))
base = os.path.dirname(td)
os.makedirs(os.path.join(base, "data"), exist_ok=True)
os.symlink(td, os.path.join(base, "data", "bert-base-uncased"))
cwd = os.getcwd(); os.chdir(base)
t = tg.XVLMForCaptioning(dict(g["tcfg"], vision_config=vj, text_encoder="data/bert-base-uncased")).eval()
os.chdir(cwd)
sd = sd_from_spec(g["t_sd_spec"])
sd["text_decoder.cls.predictions.decoder.weight"] = sd["text_decoder.bert.embeddings.word_embeddings.weight"]
t.load_state_dict(sd, strict=True)
with torch.no_grad():
    to = t(g["image"], g["captions"], output_attentions=True, output_hidden_states=True)
e.append(rel_err(to["logits_dict"]["logits"], g["t_logits"]))
print("teacher errs", e)
assert max(e) < 1e-4
''',
    "prune_utils": r'''
# the reference's own mask-materialisation utilities (utils/vqa_utils.py: update_params, prune_model_with_z — they mutate nn.Linear
# modules in place and call prune_heads, SURVEY 8b "Ownership" iv) operating on OUR model
import contextlib, io
import transformers.modeling_utils as mu, transformers.pytorch_utils as pu, transformers.file_utils as fu
mu.prune_linear_layer = pu.prune_linear_layer      # environment only: two names utils/vqa_utils.py imports moved / vanished
fu.TF_RETURN_INTRODUCTION = ""                      # between transformers 4.12.5 (the reference's pin) and the installed 5.x
import utils.vqa_utils as vu
theirs(vu)
from tests.helpers import build_with_tiny_bert
from efficientvlm_b200.vqa import EffXVLMForVQA
g, v = load_golden("vqa_pruned_tiny"), load_golden("vqa_tiny")
m = build_with_tiny_bert(EffXVLMForVQA, dict(v["scfg"], vision_config=dict(g["vis"]), text_encoder=None), v["bert"])
sd = sd_from_spec(g["sd_spec"])
sd["text_decoder.cls.predictions.decoder.weight"] = sd["text_decoder.bert.embeddings.word_embeddings.weight"]
m.load_state_dict(sd, strict=True)
m.eval()
with contextlib.redirect_stdout(io.StringIO()):      # the utilities print every pruned shape
    vu.update_params(m, g["zs"])
    vu.prune_model_with_z(g["zs"], m)
assert {k: tuple(t.shape) for k, t in m.state_dict().items()} == g["pruned_shapes"]
e = [rel_err(m.state_dict()[k], t) for k, t in g["probe"].items()]
ids, probs, _ = m.fake_forward(v["image"], Tokens(v["q_ids"], v["q_atts"]), Tokens(v["l_ids"], v["l_atts"]), k=v["k_test"])
e.append(rel_err(probs, g["topk_probs"]))
print("prune utils errs", max(e))
assert max(e) < 1e-4 and torch.equal(ids, g["topk_ids"])
''',
    "load_pretrained": r'''
# task-level checkpoint surgery: the reference classes' own load_pretrained methods (decoder initialised from the fusion layers, fusion
# layers duplicated for the two NLVR images, text_encoder -> text_decoder for captioning, bert. prefix removal for retrieval) against
# OUR classes' methods on the same synthetic pre-training checkpoint: identical resulting state_dicts
import contextlib, io
from tests.helpers import build_with_tiny_bert
from efficientvlm_b200.distill import XVLM as PretrainXVLM, EffXVLMforRetrieval
from efficientvlm_b200.vqa import EffXVLMForVQA
from efficientvlm_b200.nlvr import EffXVLMForNLVR
from efficientvlm_b200.captioning import EffXVLMForCaptioning
from oracle.det_init import det_state_dict
stub_dataset(FakeTokenizer(211))
import efficient_models.model_generation as mg, efficient_models.model_nlvr as mn, efficient_models.model_retrieval as mr
theirs(mg); theirs(mn); theirs(mr)

def pretrain_checkpoint(g, path, text_layers, image_res=64):
    """what GeneralDistill.py saves: a models/model_pretrain.py::XVLM state_dict under 'model' (here with a 64 px position grid)"""
    cfg = dict(image_res=image_res, patch_size=16, use_clip_vit=True, vision_config=dict(g["vis"]), text_encoder=None,
               text_num_hidden_layers=text_layers, embed_dim=64, temp=0.07)
    m = build_with_tiny_bert(PretrainXVLM, cfg, g["bert"])
    sd = det_state_dict(m.state_dict())
    torch.save({"model": sd}, path)

def filled(model, value):
    with torch.no_grad():
        for t in model.state_dict().values():
            if t.is_floating_point():
                t.fill_(value)
    return model

def compare(ref_model, our_model, ckpt, cfg, **kw):
    with contextlib.redirect_stdout(io.StringIO()):
        filled(ref_model, 7.0).load_pretrained(ckpt, dict(cfg), **kw)
        filled(our_model, 7.0).load_pretrained(ckpt, dict(cfg), **kw)
    a, b = ref_model.state_dict(), our_model.state_dict()
    assert list(a.keys()) == list(b.keys())
    loaded = 0
    for k in a:
        assert torch.equal(a[k], b[k]), k
        loaded += int(a[k].is_floating_point() and not bool((a[k] == 7.0).all()))
    return loaded, len(a)

tmp = os.path.dirname(make_config_dir({}, {})[0])
report = {}
# VQA student: decoder <- fusion layers
g = load_golden("vqa_tiny")
ckpt = os.path.join(tmp, "pre_vqa.th"); pretrain_checkpoint(g, ckpt, 6)
vj, td = make_config_dir(dict(g["vis"]), dict(g["bert"]))
cfg = dict(g["scfg"], vision_config=vj, text_encoder=td)
report["vqa"] = compare(mg.EffXVLMForVQA(cfg), build_with_tiny_bert(EffXVLMForVQA, dict(g["scfg"], vision_config=dict(g["vis"]), text_encoder=None), g["bert"]), ckpt, cfg)
ckpt32 = os.path.join(tmp, "pre_vqa32.th"); pretrain_checkpoint(g, ckpt32, 6, image_res=32)      # is_eval: loaded as is, no surgery
report["vqa_eval_domain"] = compare(mg.EffXVLMForVQA(cfg), build_with_tiny_bert(EffXVLMForVQA, dict(g["scfg"], vision_config=dict(g["vis"]), text_encoder=None), g["bert"]), ckpt32, cfg, is_eval=True)
# NLVR student: every fusion layer initialises both per-image copies
g = load_golden("nlvr_kd_tiny")
ckpt = os.path.join(tmp, "pre_nlvr.th"); pretrain_checkpoint(g, ckpt, 6)
vj, td = make_config_dir(dict(g["vis"]), dict(g["bert"]))
cfg = dict(g["scfg"], vision_config=vj, text_encoder=td)
ours_cfg = dict(g["scfg"], vision_config=dict(g["vis"]), text_encoder=None)
report["nlvr"] = compare(mn.EffXVLMForNLVR(cfg), build_with_tiny_bert(EffXVLMForNLVR, ours_cfg, g["bert"]), ckpt, cfg)
report["nlvr_domain"] = compare(mn.EffXVLMForNLVR(cfg), build_with_tiny_bert(EffXVLMForNLVR, ours_cfg, g["bert"]), ckpt, cfg, load_nlvr_pretrain=True)
# captioning student: text_encoder -> text_decoder
g = load_golden("caption_kd_tiny")
ckpt = os.path.join(tmp, "pre_cap.th"); pretrain_checkpoint(g, ckpt, 6)
vj, td = make_config_dir(dict(g["vis"]), dict(g["bert"]))
base = os.path.dirname(td)
os.makedirs(os.path.join(base, "data"), exist_ok=True)
os.symlink(td, os.path.join(base, "data", "bert-base-uncased"))
cwd = os.getcwd(); os.chdir(base)
ref_cap = mg.EffXVLMForCaptioning(dict(g["scfg"], vision_config=vj, text_encoder="data/bert-base-uncased"))
os.chdir(cwd)
tok = FakeTokenizer(g["bert"]["vocab_size"])
import efficientvlm_b200.eff_bert as eb
orig = eb.BertConfig.__init__
def patched(self, **k2):
    m = dict(g["bert"]); m.update(k2); orig(self, **m)
eb.BertConfig.__init__ = patched
our_cap = EffXVLMForCaptioning(dict(g["scfg"], vision_config=dict(g["vis"]), text_encoder=None), tokenizer=tok)
eb.BertConfig.__init__ = orig
cfg = dict(g["scfg"], vision_config=vj, text_encoder="data/bert-base-uncased")
report["caption"] = compare(ref_cap, our_cap, ckpt, cfg)
report["caption_domain"] = compare(ref_cap, our_cap, ckpt, cfg, load_capt_pretrain=True)
# retrieval student: bert. prefix removed
g = load_golden("itr_kd_tiny")
ckpt = os.path.join(tmp, "pre_itr.th"); pretrain_checkpoint(g, ckpt, 6)
vj, td = make_config_dir(dict(g["vis"]), dict(g["bert"]))
cfg = dict(g["scfg"], vision_config=vj, text_encoder=td)
report["itr"] = compare(mr.EffXVLMforRetrieval(cfg), build_with_tiny_bert(EffXVLMforRetrieval, dict(g["scfg"], vision_config=dict(g["vis"]), text_encoder=None), g["bert"]), ckpt, cfg)
print("load_pretrained: (tensors loaded, tensors total)", report)
assert all(v[0] > 0.5 * v[1] for k, v in report.items() if not k.endswith("_domain")), report
''',
    "itr_eval": r'''
# Eff_Retrieval.py imports ruamel / the dataset package at module level, so its two evaluation functions are lifted out with `ast`
# (exactly what oracle/make_golden_itr_eval.py did on the reference side) and run, unmodified, on OUR model
g = load_golden("itr_eval_tiny")
model, loader, tokenizer = itr_eval_setup(g, "cpu")
src = open(os.path.join(REF, "Eff_Retrieval.py")).read()
fns = [n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name in ("evaluation", "itm_eval")]
class Logger:
    def __init__(self, delimiter=""): pass
    def log_every(self, it, freq, header=None): return it
utils = types.SimpleNamespace(MetricLogger=Logger, get_world_size=lambda: 1, get_rank=lambda: 0)
ns = {"torch": torch, "np": np, "time": time, "datetime": datetime, "utils": utils, "dist": torch.distributed,
      "args": types.SimpleNamespace(distributed=False)}
exec(compile(ast.Module(body=fns, type_ignores=[]), "Eff_Retrieval.py", "exec"), ns)
a, b, sparsity = ns["evaluation"](model, loader, tokenizer, "cpu", g["config"])
e = [rel_err(torch.from_numpy(a), g["score_i2t"]), rel_err(torch.from_numpy(b), g["score_t2i"])]
print("itr eval errs", e)
assert max(e) < 1e-5 and abs(float(sparsity) - g["sparsity"]) < 1e-6
assert ns["itm_eval"](a, b, g["txt2img"], g["img2txt"]) == g["result"]
''',
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_reference_files_run_unchanged_on_our_core(case):
    """`models/model_pretrain.py` + the GeneralDistill.py train-loop statements (GD, the headline), `efficient_models/model_generation.py`
    (VQA, captioning), `efficient_models/model_nlvr.py` and `Eff_Retrieval.py`'s evaluation, unmodified, on top of the compat shims: losses / logits / answer ids / captions / score matrices of the reference-generated goldens.
    `gd_train_loop`: the unmodified `GeneralDistill.py::train()` for 4 iterations (image + region steps, clip, AdamW, schedule, checkpoint
    hand-over) against the same iterations on the product API: same logged losses, same parameters."""
    r = subprocess.run([sys.executable, "-c", PREAMBLE + CASES[case] + "\nprint('OK')\n", ROOT, REF], capture_output=True, text=True, timeout=600,
                       cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert "OK" in r.stdout


def test_drivers_own_loss_statements_on_our_outputs(monkeypatch):
    """The loss sections of the four pruning drivers' train() loops — Eff_Retrieval.py:101-178, Eff_VQA.py:105-176, Eff_NLVR.py:100-157,
    Eff_Captioning.py:99-148, lifted from the unmodified files with `ast` (oracle/driver_code.py) — executed on the outputs of OUR student /
    teacher models reproduce the fixtures' totals.  This pins the output-dict layout the drivers index into, and ties both the fixture
    generators' statement-by-statement restatements and our `*_loss` helpers to the drivers' actual code."""
    import torch
    from oracle.driver_code import lift_train_loss
    from tests import helpers as H
    from tests import ref_ops
    ref_ops.install(monkeypatch)
    out = {}
    # ITR
    g = H.load_golden("itr_kd_tiny")
    student, teacher = H.itr_models(g)
    student.sample_itm_negatives, teacher.sample_itm_negatives = H.argmax_negatives(student), H.argmax_negatives(teacher)
    H.arm_eps(student.l0_module, g["eps"])
    args, kw = (g["image"], g["text_ids"], g["text_atts"]), dict(idx=g["idx"], output_attentions=True, output_hidden_states=True)
    so = student(*args, **kw)
    with torch.no_grad():
        to = teacher(*args, **kw)
    run, lines = lift_train_loss("Eff_Retrieval.py")
    ns = run(so, to, student, g["step"])
    out["itr"] = (lines, H.rel_err(ns["loss"], g["total"]))
    for ours, theirs in (("text_hidden", "text_hidden_loss"), ("itm_neg_cross", "itm_neg_cross_loss"), ("itm_logits", "itm_logits_loss")):
        H.assert_close(ns[theirs], g["parts"][ours], 1e-5, theirs)
    # VQA
    g = H.load_golden("vqa_tiny")
    student, teacher = H.vqa_models(g)
    q, a = H.Tokens(g["q_ids"], g["q_atts"]), H.Tokens(g["a_ids"], g["a_atts"])
    H.arm_eps(student.l0_module, g["eps"])
    kw = dict(train=True, k=g["k"], weights=g["weights"], output_attentions=True, output_hidden_states=True)
    so = student(g["image"], q, a, **kw)
    with torch.no_grad():
        to = teacher(g["image"], q, a, **kw)
    run, lines = lift_train_loss("Eff_VQA.py")
    out["vqa"] = (lines, H.rel_err(run(so, to, student, g["step"])["loss"], g["total"]))
    # NLVR2
    g = H.load_golden("nlvr_kd_tiny")
    student, teacher = H.nlvr_models(g)
    H.arm_eps(student.l0_module, g["eps"])
    args, kw = (g["image"], g["text_ids"], g["text_atts"]), dict(targets=g["targets"], train=True, output_attentions=True, output_hidden_states=True)
    so = student(*args, **kw)
    with torch.no_grad():
        to = teacher(*args, **kw)
    run, lines = lift_train_loss("Eff_NLVR.py")
    out["nlvr"] = (lines, H.rel_err(run(so, to, student, g["step"])["loss"], g["total"]))
    # captioning
    g = H.load_golden("caption_kd_tiny")
    student, teacher = H.caption_models(g)
    H.arm_eps(student.l0_module, g["eps"])
    so = student(g["image"], g["captions"], output_attentions=True, output_hidden_states=True)
    with torch.no_grad():
        to = teacher(g["image"], g["captions"], output_attentions=True, output_hidden_states=True)
    run, lines = lift_train_loss("Eff_Captioning.py")
    out["caption"] = (lines, H.rel_err(run(so, to, student, g["step"])["loss"], g["total"]))
    print(out)
    assert {k: v[0] for k, v in out.items()} == {"itr": (101, 178), "vqa": (105, 176), "nlvr": (100, 157), "caption": (99, 148)}
    assert max(v[1] for v in out.values()) < 1e-5, out


def test_reference_optimizer_grouping_and_schedule_on_our_models(monkeypatch):
    """`optim.py::create_optimizer` / `create_L0_optimizer` (lifted with `ast`: the file imports an AdamW that transformers 5.x no longer
    ships) run on OUR models: the parameter groups they build from our parameter names — weight-decay / no-decay by name substring,
    `init_params` at lr x lr_mult, gate parameters vs Lagrange multipliers with the negated learning rate — are the groups
    `efficientvlm_b200.optim.group_parameters` / `create_L0_optimizer` build.  `scheduler.py::create_scheduler` (imported as is) and
    `LinearWarmupDecay` produce the same learning-rate sequence."""
    import ast
    import importlib.util
    import types

    import torch
    from efficientvlm_b200 import optim as our_optim
    from tests import helpers as H
    from tests import ref_ops
    ref_ops.install(monkeypatch)
    tree = ast.parse(open(os.path.join(REF, "optim.py")).read())
    fns = [n for n in tree.body if isinstance(n, ast.FunctionDef)]

    class Recorder:          # stands in for transformers 4.12.5's AdamW: keeps what the reference passes to it
        def __init__(self, groups, **kw):
            self.groups, self.kw = groups, kw
    ns = {"AdamW": Recorder, "print": lambda *a, **k: None}
    exec(compile(ast.Module(body=fns, type_ignores=[]), "optim.py", "exec"), ns)
    args = types.SimpleNamespace(lr=3e-4, weight_decay=0.01, lr_mult=2, reg_learning_rate=0.1)
    g = H.load_golden("vqa_tiny")
    student, _ = H.vqa_models(g)
    gd_student, _ = H.gd_models(H.load_golden("gd_kd_tiny"))
    student.init_params = ["text_decoder.bert.encoder.layer.0.crossattention.self.key.weight", "text_decoder.bert.encoder.layer.0.crossattention.self.key.bias"]
    for model in (student, gd_student):
        names = {id(p): n for n, p in model.named_parameters()}
        theirs = ns["create_optimizer"](args, model)
        ours = our_optim.group_parameters(model, args.lr, args.weight_decay, args.lr_mult)
        assert theirs.kw == dict(lr=args.lr, eps=1e-8, betas=(0.9, 0.98))
        for a, b in zip(theirs.groups, ours):
            assert (a["weight_decay"], a["lr"]) == (b["weight_decay"], b["lr"])
            assert [names[id(p)] for p in a["params"]] == b["names"]
        assert sum(len(b["names"]) for b in ours) == len(names)
    assert len(our_optim.group_parameters(student, args.lr, args.weight_decay, args.lr_mult)[2]["names"]) == 1      # key.weight: decay, large lr
    assert len(our_optim.group_parameters(student, args.lr, args.weight_decay, args.lr_mult)[3]["names"]) == 1      # key.bias: no decay, large lr
    l0_t, lag_t = ns["create_L0_optimizer"](args, student.l0_module)
    gates = [n for n, _ in student.l0_module.named_parameters() if "lambda" not in n]
    lams = [n for n, _ in student.l0_module.named_parameters() if "lambda" in n]
    names = {id(p): n for n, p in student.l0_module.named_parameters()}
    assert [names[id(p)] for p in l0_t.groups[0]["params"]] == gates and l0_t.groups[0]["lr"] == args.reg_learning_rate
    assert [names[id(p)] for p in lag_t.groups[0]["params"]] == lams and lag_t.groups[0]["lr"] == -args.reg_learning_rate
    assert l0_t.kw == lag_t.kw == dict(eps=1e-8, betas=(0.9, 0.98))
    # scheduler.py as is
    spec = importlib.util.spec_from_file_location("ref_scheduler", os.path.join(REF, "scheduler.py"))
    sched = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(sched)

    class Args(dict):
        __getattr__ = dict.__getitem__
    for total, warm in ((50, 0.1), (37, 5), (10, 0)):
        w = torch.nn.Parameter(torch.zeros(1))
        opt = torch.optim.SGD([{"params": [w], "lr": 0.5}, {"params": [torch.nn.Parameter(torch.zeros(1))], "lr": 0.02}], lr=0.5)
        monkeypatch.setattr("builtins.print", lambda *a, **k: None)
        ref = sched.create_scheduler(Args(sched="linear", num_training_steps=total, num_warmup_steps=warm), opt)
        mine_opt = types.SimpleNamespace(param_groups=[{"lr": 0.5, "initial_lr": 0.5}, {"lr": 0.02, "initial_lr": 0.02}])
        mine = our_optim.LinearWarmupDecay(mine_opt, total, warm)
        for _ in range(total + 3):
            assert [gp["lr"] for gp in opt.param_groups] == [gp["lr"] for gp in mine_opt.param_groups]
            opt.step()
            ref.step()
            mine.step()


def test_checkpoint_key_surgery_matches_reference(tmp_path, monkeypatch):
    """Checkpoints are loaded with `load_state_dict(strict=False)` after key surgery (SURVEY 8b "Ownership" i): the reference's
    `load_pretrained`, `load_params_choose_layers`, `load_params_change_prefix` (efficient_models/xvlm.py:24-52,183-208) and
    `interpolate_pos_embed` (models/vit.py:222-247), lifted with `ast` from the unmodified files, against ours on synthetic checkpoints:
    same keys in the same order, bit-identical tensors (bicubic position-grid resize 224 -> 384 px, layer picking 12 -> 6, `bert.` prefix
    removal)."""
    import ast

    import torch
    import torch.nn.functional as F
    from efficientvlm_b200 import xvlm as ours
    monkeypatch.setattr("builtins.print", lambda *a, **k: None)

    def lift(path, names, ns):
        tree = ast.parse(open(os.path.join(REF, path)).read())
        fns = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name in names]
        assert len(fns) == len(names), (path, names)
        exec(compile(ast.Module(body=fns, type_ignores=[]), path, "exec"), ns)
        return ns
    ns = {"torch": torch, "F": F}
    lift("models/vit.py", ["interpolate_pos_embed"], ns)
    lift("efficient_models/xvlm.py", ["load_pretrained", "load_params_choose_layers", "load_params_change_prefix"], ns)
    g = torch.Generator().manual_seed(0)
    W = 32

    def checkpoint():
        sd = {"vision_encoder.position_ids": torch.arange(197)[None], "vision_encoder.pos_embed.weight": torch.randn(197, W, generator=g),
              "vision_encoder.class_embedding": torch.randn(W, generator=g), "temp": torch.tensor(0.07),
              "itm_head.0.weight": torch.randn(4, W, generator=g), "text_encoder.cls.predictions.bias": torch.randn(7, generator=g)}
        for i in range(12):
            sd["vision_encoder.encoder.layers.%d.mlp.fc1.weight" % i] = torch.randn(3, W, generator=g)
            sd["text_encoder.bert.encoder.layer.%d.attention.self.query.weight" % i] = torch.randn(3, W, generator=g)
            sd["text_encoder.bert.encoder.layer.%d.output.LayerNorm.bias" % i] = torch.randn(W, generator=g)
        return sd
    path = str(tmp_path / "ckpt.th")
    torch.save({"model": checkpoint()}, path)
    raw = str(tmp_path / "raw.th")
    torch.save(checkpoint(), raw)                                  # a checkpoint without the {"model": ...} wrapper

    def same(a, b):
        assert list(a.keys()) == list(b.keys())
        for k in a:
            assert torch.equal(a[k], b[k]), k
    for res in (224, 384, 480):
        cfg = {"image_res": res, "patch_size": 16, "use_clip_vit": True, "use_swin": False}
        for kw in (dict(is_eval=True), dict(), dict(load_text=True)):
            for p in (path, raw):
                a, b = ns["load_pretrained"](p, cfg, **kw), ours.load_pretrained(p, cfg, **kw)
                same(a, b)
                if not kw.get("is_eval"):
                    assert b["vision_encoder.pos_embed.weight"].shape == (1 + (res // 16) ** 2, W)
    for n_patches in (196, 576, 900, 4):
        pe = torch.randn(1, 197, W, generator=g)
        assert torch.equal(ns["interpolate_pos_embed"](pe, n_patches), ours.interpolate_pos_embed(pe, n_patches))
    mapper = {1: 0, 3: 1, 5: 2, 7: 3, 9: 4, 11: 5}
    for prefix in ("vision_encoder.encoder.layers", "text_encoder.bert.encoder.layer"):
        a, b = checkpoint(), None
        b = {k: v.clone() for k, v in a.items()}
        ns["load_params_choose_layers"](prefix, a, mapper)
        ours.load_params_choose_layers(prefix, b, mapper)
        same(a, b)
        assert sum(k.startswith(prefix) for k in b) == 6 * (1 if "vision" in prefix else 2)


ACCEL_SCRIPT = r'''
import os, sys, types
ROOT, REF = sys.argv[1], sys.argv[2]
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "efficientvlm_b200", "compat"))   # our drop-in packages / modules win ...
sys.path.append(REF)                                                    # ... the reference supplies everything else
import torch
# what GeneralDistill.py:33-36 imports, by the same names
from optim import create_optimizer
from scheduler import create_scheduler
from accelerators.apex_ddp_accelerator import ApexDDPAccelerator
import optim, scheduler, accelerators.apex_ddp_accelerator as acc
for m in (optim, scheduler, acc):
    assert "efficientvlm_b200" in m.__file__, m.__file__
import utils                                        # the reference's utils package (AttrDict) is untouched
assert utils.__file__.startswith(REF)
cfg = utils.AttrDict(dict(RNG_SEED=42, SYNCBN=False, FP16_OPT_LEVEL="O1", FP16_LOSS_SCALE="dynamic", CLIP_GRAD_NORM=1.0))
a = ApexDDPAccelerator(cfg, logger=None)
assert (a.accelerator_rng_seed, a.accelerator_syncbn, a.accelerator_fp16_opt_level, a.accelerator_fp16_loss_scale) == (42, False, "O1", "dynamic")
net = torch.nn.Linear(3, 2)
try:
    a.set_up(net, None, None, 0, 1, 0)
    raise SystemExit("set_up must refuse to run without a CUDA device")
except RuntimeError as e:
    assert "no CPU path" in str(e)
w = torch.nn.Parameter(torch.ones(2))
loss = (w * torch.tensor([2.0, 3.0])).sum()
a.backward_step(loss, optimizer=None)               # GeneralDistill.py:261 passes the optimizer positionally
assert torch.equal(w.grad, torch.tensor([2.0, 3.0]))
armed = types.SimpleNamespace(clip_grad_norm=0.0, grad_norm=lambda: torch.tensor(0.5))
assert float(a.optimizer_step(armed, net, 1.0)) == 0.5 and armed.clip_grad_norm == 1.0      # arms FlatAdamW's clip for the step() that follows
net.weight.grad = torch.full_like(net.weight, 10.0); net.bias.grad = torch.zeros_like(net.bias)
total = a.optimizer_step(torch.optim.SGD(net.parameters(), lr=0.1), net, 1.0)             # a plain torch optimizer: the base-class clip
assert abs(total - (6 * 100.0) ** 0.5) < 1e-4 and abs(float(net.weight.grad.norm()) - 1.0) < 1e-4
# scheduler: same argument handling and sequence as the reference's LambdaLR; resumable
fake = types.SimpleNamespace(param_groups=[{"lr": 0.5, "initial_lr": 0.5}, {"lr": 0.02, "initial_lr": 0.02}])
args = utils.AttrDict(dict(sched="linear", epochs=3, step_per_epoch=7, num_warmup_steps=0.2))
s = create_scheduler(args, fake)
assert (args["num_training_steps"], args["num_warmup_steps"]) == (21, 4)
seq = []
for _ in range(9):
    seq.append(fake.param_groups[0]["lr"]); s.step()
state = s.state_dict()
fake2 = types.SimpleNamespace(param_groups=[{"lr": 0.5, "initial_lr": 0.5}, {"lr": 0.02, "initial_lr": 0.02}])
s2 = create_scheduler(utils.AttrDict(dict(sched="linear", num_training_steps=21, num_warmup_steps=4)), fake2)
s2.load_state_dict(state)
assert fake2.param_groups == fake.param_groups
ref_opt = torch.optim.SGD([{"params": [torch.nn.Parameter(torch.zeros(1))], "lr": 0.5}], lr=0.5)
import importlib.util
spec = importlib.util.spec_from_file_location("ref_scheduler", os.path.join(REF, "scheduler.py"))
rs = importlib.util.module_from_spec(spec); spec.loader.exec_module(rs)
r = rs.create_scheduler(utils.AttrDict(dict(sched="linear", epochs=3, step_per_epoch=7, num_warmup_steps=0.2)), ref_opt)
ref_seq = []
for _ in range(9):
    ref_seq.append(ref_opt.param_groups[0]["lr"]); ref_opt.step(); r.step()
assert seq == ref_seq, (seq, ref_seq)
print("OK")
'''


def test_accelerator_optim_scheduler_shims():
    """`from accelerators.apex_ddp_accelerator import ApexDDPAccelerator`, `from optim import create_optimizer`, `from scheduler import
    create_scheduler` (GeneralDistill.py:33-36) resolve to the drop-ins with compat first on sys.path; the accelerator keeps the reference's
    interface (set_up / backward_step / optimizer_step), refuses to run without a CUDA device, and arms FlatAdamW's post-allreduce clip."""
    r = subprocess.run([sys.executable, "-c", ACCEL_SCRIPT, ROOT, REF], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert "OK" in r.stdout


def test_vqa_driver_evaluation_on_our_model(monkeypatch):
    """`Eff_VQA.py:216-239` (`evaluation`: answer-list tokenisation, `model(..., train=False, k=k_test)`, arg-max over the re-ranked
    candidates), lifted unmodified, on OUR EffXVLMForVQA: the predicted answers are the ones the reference model's own ranking gives
    (tests/golden/vqa_tiny.pt)."""
    import ast
    import types

    import torch
    from tests import helpers as H
    from tests import ref_ops
    ref_ops.install(monkeypatch)
    g = H.load_golden("vqa_tiny")
    student, _ = H.vqa_models(g)
    tree = ast.parse(open(os.path.join(REF, "Eff_VQA.py")).read())
    fn = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "evaluation"]

    class Logger:
        def __init__(self, delimiter=""):
            pass

        def log_every(self, it, freq, header=None):
            return it
    ns = {"torch": torch, "utils": types.SimpleNamespace(MetricLogger=Logger)}
    exec(compile(ast.Module(body=fn, type_ignores=[]), "Eff_VQA.py", "exec"), ns)
    n_q, n_a = g["q_ids"].shape[0], g["l_ids"].shape[0]
    answer_list = ["answer %d" % i for i in range(n_a)]
    questions = ["question %d" % i for i in range(n_q)]

    def tokenizer(text, **kw):          # the fixture holds token ids; the strings are only handles for its rows
        if text and text[0].startswith("answer"):
            return H.Tokens(g["l_ids"], g["l_atts"])
        rows = torch.tensor([int(t.split()[1]) for t in text])
        return H.Tokens(g["q_ids"][rows], g["q_atts"][rows])

    class Loader(list):
        dataset = types.SimpleNamespace(answer_list=answer_list)
    half = n_q // 2 or 1
    loader = Loader([(g["image"][:half], questions[:half], torch.arange(100, 100 + half)),
                     (g["image"][half:], questions[half:], torch.arange(100 + half, 100 + n_q))][:2 if n_q > half else 1])
    result = ns["evaluation"](student, loader, tokenizer, "cpu", {"k_test": g["k_test"]})
    want = [answer_list[int(ids[p.argmax()])] for ids, p in zip(g["topk_ids"], g["topk_probs"])]
    assert [r["question_id"] for r in result] == list(range(100, 100 + n_q))
    assert [r["answer"] for r in result] == want
