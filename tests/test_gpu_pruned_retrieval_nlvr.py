"""Materialised retrieval and NLVR2 students on the device: the ITR re-rank evaluation and the NLVR prediction of the physically pruned,
gate-free models (ragged per-layer head counts and FFN widths, 1-head cross-attention layers, the two copies of an NLVR fusion layer with
different head counts) against the masked targets at the bf16 bars, every re-rank batching mode against the resident K|V path, FP8
against an fp32 emulation of the quantised arithmetic, and the cross-attention kernel over K|V row pitches of 2 * h * 64 for h = 1 ... 12."""
import pytest
import torch

from efficientvlm_b200 import fp8, ops
from efficientvlm_b200 import retrieval_eval as RE
from tests import helpers
from tests.helpers import assert_close, itr_eval_setup, load_golden, rel_err, with_reference_bf16_noise
from tests.test_gpu_fp8 import _emulation, _emulation_copy
from tests.test_pruned_retrieval_nlvr import ITR_RAGGED_SEED, cross_pairs, materialised, nlvr_batch, nlvr_predict, nlvr_student, seed_logas

pytestmark = pytest.mark.gpu
ACT_TOL = 1e-2      # the project's bf16 bar (tests/test_gpu_models.py)
# FP8 against its fp32 emulation: the device's attention, LayerNorm and residual adds run in bf16 where the emulation runs fp32, so an
# activation within a bf16 step of an e4m3 rounding boundary rounds one e4m3 step (2^-4 relative) apart, and every later layer quantises
# the already different activations again.  Over the 9-layer NLVR encoder and the ViT + text + fusion stack of the ITR model this
# compounds to 4 - 8 % relative on a B200.  So the bar is 1e-1, and the discriminating check is that the device's FP8 outputs are closer
# to the emulation than the same model's bf16 outputs are: it computes the quantised arithmetic, not the unquantised one.
FP8_TOL = 1e-1


@with_reference_bf16_noise
def test_materialised_itr_evaluation_on_device_vs_masked_golden(monkeypatch):
    """The fixture's student, materialised on the device, against the reference's MASKED evaluation: similarities, candidates (swaps only
    where the fixture's own similarities cannot separate them), scores, every re-rank batching mode and the two-rank split."""
    monkeypatch.setattr(helpers, "itr_eval_setup", lambda g, device: (materialised(itr_eval_setup(g, device)[0]),) + itr_eval_setup(g, device)[1:])
    helpers.run_itr_eval(load_golden("itr_eval_tiny"), "cuda", ACT_TOL, ACT_TOL, exact_candidates=False)


def _ragged_itr(device):
    g = load_golden("itr_eval_tiny")
    model, loader, tokenizer = itr_eval_setup(g, device)
    return g, seed_logas(model, ITR_RAGGED_SEED), loader, tokenizer


def _evaluate(model, loader, tokenizer, g):
    details = {}
    out = RE.evaluation(model, loader, tokenizer, "cuda", g["config"], details=details)
    return out, details


def test_ragged_materialised_itr_evaluation_vs_masked_on_device():
    """Pruned heads (1-head vision, text and cross layers) and FFN widths that are not multiples of 8: masked and materialised evaluation
    on the device agree at the bf16 bar; the resident K|V is sized and cached at the ragged per-layer widths; every batching mode of
    rerank_scores equals the resident path."""
    g, masked, loader, tokenizer = _ragged_itr("cuda")
    (mi, mt, ms), md = _evaluate(masked, loader, tokenizer, g)
    model = materialised(_ragged_itr("cuda")[1])
    (fi, ft, fs), fd = _evaluate(model, loader, tokenizer, g)
    assert ms == fs
    assert_close(fd["sims_matrix"], md["sims_matrix"], ACT_TOL, "similarities")
    both = (mi != -100) & (fi != -100)
    assert both.sum() >= 0.9 * (mi != -100).sum()
    assert_close(torch.from_numpy(fi[both]), torch.from_numpy(mi[both]), ACT_TOL, "image->text scores")
    both = (mt != -100) & (ft != -100)
    assert both.sum() >= 0.9 * (mt != -100).sum()
    assert_close(torch.from_numpy(ft[both]), torch.from_numpy(mt[both]), ACT_TOL, "text->image scores")
    # resident K|V at the ragged widths
    bert = model._bert()
    heads = [blk.crossattention.self.num_attention_heads for blk in bert.encoder.layer if blk.has_cross_attention]
    assert 1 in heads
    feats, sims, k = fd["image_feats"], fd["sims_matrix"], g["config"]["k_test"]
    n_tok, width = feats.shape[0] * feats.shape[1], feats.shape[2]
    assert RE._fusion_kv_bytes(model, feats) == n_tok * width * 2 + sum(n_tok * 2 * 64 * h * 2 for h in heads)
    ops._cross_kv.clear()
    args = (model, feats, fd["text_feats"], fd["text_atts"], sims, k)
    a, b = RE.rerank_scores(*args, rank=0, world=1)
    cached = sorted(e[2].shape[1] for e in ops._cross_kv.values() if e[2].shape[0] == n_tok)
    assert cached == sorted(2 * 64 * h for h in heads), (cached, heads)
    for kw in (dict(queries_per_pass=1, group_rows=1), dict(queries_per_pass=3, group_rows=2), dict(group_rows=5),
               dict(queries_per_pass=4, group_rows=3, kv_cache_bytes=0), dict(queries_per_pass=1, share_image_kv=False),
               dict(queries_per_pass=5, share_image_kv=False)):
        a2, b2 = RE.rerank_scores(*args, rank=0, world=1, **kw)
        for ours, want in ((a2, a), (b2, b)):
            assert torch.equal(ours == -100.0, want == -100.0), kw
            assert_close(ours[want != -100.0], want[want != -100.0], ACT_TOL, "batching mode %r" % (kw,))
    total = [torch.zeros_like(a), torch.zeros_like(b)]
    for r in range(2):
        for j, t in enumerate(RE.rerank_scores(*args, queries_per_pass=2, group_rows=3, rank=r, world=2)):
            total[j] += t
    for t, want in zip(total, (a, b)):
        assert torch.equal(t == -200.0, want == -100.0)
        assert_close(t[want != -100.0] + 100.0, want[want != -100.0], ACT_TOL, "two-rank split")
    ops._cross_kv.clear()


@with_reference_bf16_noise
def test_materialised_nlvr_prediction_on_device_vs_masked():
    """Ragged NLVR student (1-head self and cross layers, fusion copies with different cross-attention head counts): the materialised
    model's eval logits on the device against the gated model's fp32 logits on the CPU."""
    g = load_golden("nlvr_kd_tiny")
    with helpers.reference_ops_fp32():
        want = nlvr_predict(nlvr_student(g), nlvr_batch(g))
    model = materialised(nlvr_student(g).cuda())
    assert any(a.crossattention.self.num_attention_heads != b.crossattention.self.num_attention_heads for a, b in cross_pairs(model))
    got = nlvr_predict(model, nlvr_batch(g, "cuda"))
    assert_close(got, want, ACT_TOL, "materialised NLVR logits")
    masked = nlvr_student(g).cuda()
    assert_close(nlvr_predict(masked, nlvr_batch(g, "cuda")), want, ACT_TOL, "masked NLVR logits")


def test_fp8_materialised_nlvr_vs_emulation(monkeypatch):
    g = load_golden("nlvr_kd_tiny")
    model = materialised(nlvr_student(g).cuda())
    emu = _emulation_copy(model)
    bf16 = nlvr_predict(model, nlvr_batch(g, "cuda")).cpu()
    fp8.enable(model)
    got = nlvr_predict(model, nlvr_batch(g, "cuda")).cpu()
    with _emulation(monkeypatch):
        want = nlvr_predict(emu, nlvr_batch(g))
    assert_close(got, want, FP8_TOL, "FP8 NLVR logits vs emulation")
    assert rel_err(got, want) < rel_err(bf16, want)


def test_fp8_materialised_itr_evaluation_vs_emulation(monkeypatch):
    """FP8 ITR evaluation (resident K|V included) against the emulation: similarities, and the scores of every pair both rank."""
    g, _, loader, tokenizer = _ragged_itr("cuda")
    model = materialised(_ragged_itr("cuda")[1])
    emu = _emulation_copy(model)
    _, bd = _evaluate(model, loader, tokenizer, g)
    fp8.enable(model)
    (fi, ft, _), fd = _evaluate(model, loader, tokenizer, g)
    with _emulation(monkeypatch):
        ed = {}
        ei, et, _ = RE.evaluation(emu, loader, tokenizer, "cpu", g["config"], details=ed)
    for key in ("image_feats", "text_feats", "sims_matrix"):
        assert_close(fd[key], ed[key], FP8_TOL, "FP8 %s vs emulation" % key)
        assert rel_err(fd[key], ed[key]) < rel_err(bd[key], ed[key]), key
    for ours, want, what in ((fi, ei, "image->text"), (ft, et, "text->image")):
        both = (ours != -100) & (want != -100)
        assert both.sum() >= 0.8 * (want != -100).sum(), what
        assert_close(torch.from_numpy(ours[both]), torch.from_numpy(want[both]), FP8_TOL, "FP8 %s scores vs emulation" % what)


def test_cached_cross_kv_is_never_shared_between_bf16_and_fp8():
    """A re-rank over the same image-token tensor, before and after fp8.enable: the FP8 pass projects its own K|V (equal, bit for bit, to
    an FP8 pass from an empty cache) and does not serve the bf16 one."""
    g, _, loader, tokenizer = _ragged_itr("cuda")
    model = materialised(_ragged_itr("cuda")[1])
    _, d = _evaluate(model, loader, tokenizer, g)
    args = (model, d["image_feats"], d["text_feats"], d["text_atts"], d["sims_matrix"], g["config"]["k_test"])
    ops._cross_kv.clear()
    a16, _ = RE.rerank_scores(*args, rank=0, world=1)
    kv16 = {k: v[2].clone() for k, v in ops._cross_kv.items()}
    assert kv16
    fp8.enable(model)
    a8, _ = RE.rerank_scores(*args, rank=0, world=1)
    assert not torch.equal(a8, a16)
    new = [v for k, v in ops._cross_kv.items() if k not in kv16]
    assert len(new) == len(kv16) and all(isinstance(v[1], ops.Fp8Weight) for v in new)
    assert all(torch.equal(ops._cross_kv[k][2], v) for k, v in kv16.items())
    ops._cross_kv.clear()
    fresh, _ = RE.rerank_scores(*args, rank=0, world=1)
    assert torch.equal(a8, fresh)
    ops._cross_kv.clear()


@pytest.mark.parametrize("heads", list(range(1, 13)))
def test_uniform_group_cross_attention_at_every_head_count(heads):
    """The long-key attention kernel as the re-rank runs it: 577 image tokens, K and V as the two halves of one [rows, 2 * h * 64] K|V
    buffer, groups of 16 captions x 40 tokens indexing a resident image batch out of order (UniformGroups(items=)).  Against fp32
    softmax(q k^T / 8) v on the same bf16 operands."""
    from efficientvlm_b200 import kernels as K
    gen = torch.Generator().manual_seed(heads)
    E, Nn, L, k, n_img = 64 * heads, 577, 40, 16, 4
    items = torch.tensor([3, 0, 3, 1, 2], dtype=torch.int32)
    G = items.numel()
    q = torch.randn(G * k * L, E, generator=gen).to(torch.bfloat16)
    kv = (torch.randn(n_img * Nn, 2 * E, generator=gen) * 2.0).to(torch.bfloat16)
    qd, kvd = q.cuda(), kv.cuda()
    ctx, _, _ = K.attention_fwd(qd, kvd[:, :E], kvd[:, E:], G, heads, k * L, Nn, 0.125, want_probs=False, kv_index=items.cuda())
    torch.cuda.synchronize()
    qf = q.float().view(G, k * L, heads, 64).transpose(1, 2)
    kf = kv.float().view(n_img, Nn, 2, heads, 64)[items.long()]
    s = torch.einsum("ghqd,gkhd->ghqk", qf, kf[:, :, 0]) * 0.125
    want = torch.einsum("ghqk,gkhd->gqhd", torch.softmax(s, -1), kf[:, :, 1]).reshape(G * k * L, E)
    assert ctx.shape == (G * k * L, E)
    assert_close(ctx.float().cpu(), want, 1e-2, "h=%d" % heads)
