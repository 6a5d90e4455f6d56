"""prune.materialize on the captioning student (host logic, CPU, through the oracle operators of tests/ref_ops.py): which gate rows are
folded into which decoder layer, the pruned shapes, and that the physically smaller, gate-free model decodes what the gated model
decodes (teacher-forced logits, greedy, sampling and beam search).  The reference's caption_utils.py is not available, so the gated
model's own decode is the target."""
import pytest
import torch

from tests import ref_ops
from tests.helpers import caption_models, load_golden

# Log-alphas from this seed (x 3.0 + 1.5, like bench.py's synthetic gates) prune heads and FFN columns in the decoder layers the
# gate table reads; with the fixture's own log-alphas only cross_head_z[5] loses a head, and no decoder layer reads that row.
RAGGED_SEED = 0
# This seed zeroes both heads of cross_head_z[2], the cross-attention gate of decoder layer 5.
EMPTY_CROSS_SEED = 6


@pytest.fixture(scope="module")
def golden():
    return load_golden("caption_kd_tiny")


def _student(g, seed):
    student, _ = caption_models(g)
    gen = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, la in student.l0_module.named_parameters():
            if name.endswith("_loga"):
                la.copy_(torch.randn(la.shape, generator=gen) * 3.0 + 1.5)
    student.tokenizer(g["captions"])          # the whitespace tokenizer learns id -> word from the training captions
    return student


def _zs(student):
    with torch.no_grad():
        return student.l0_module.forward(training=False)


def _decoder_gates(zs):
    return dict(head_z=torch.cat((zs["text_head_z"], zs["cross_head_z"]), dim=0),
                mlp_z=torch.cat((zs["text_intermediate_z"], zs["cross_intermediate_z"]), dim=0))


def _image_embeds(student, image, zs=None):
    with torch.no_grad():
        if zs is None:
            return student.vision_encoder(image)[0]
        return student.vision_encoder(image, head_z=zs["vision_head_z"], mlp_z=zs["vision_intermediate_z"])[0]


def _teacher_forced_logits(student, g, image_embeds, gates):
    with torch.no_grad():
        return student.text_decoder(g["input_ids"], attention_mask=torch.ones_like(g["input_ids"]), encoder_hidden_states=image_embeds,
                                    encoder_attention_mask=None, return_dict=True, **gates).logits


def _materialised(g, seed=RAGGED_SEED):
    from efficientvlm_b200 import prune
    model = _student(g, seed)
    zs = _zs(model)
    prune.materialize(model, zs)
    return model, zs


def test_decoder_gate_table_follows_quirk_q1(monkeypatch, golden):
    """Layer i < F takes head_z[i] / mlp_z[i]; layer i >= F takes self head_z[2(i - F)], cross head_z[2(i - F) + 1], mlp_z[i - F]."""
    from efficientvlm_b200 import prune
    from efficientvlm_b200.eff_bert import layer_gate_rows
    ref_ops.install(monkeypatch)
    assert [layer_gate_rows(i, 3) for i in range(6)] == [(0, None, 0), (1, None, 1), (2, None, 2), (0, 1, 0), (2, 3, 1), (4, 5, 2)]
    student = _student(golden, RAGGED_SEED)
    zs = _zs(student)
    th, ch = [r.reshape(-1) for r in zs["text_head_z"]], [r.reshape(-1) for r in zs["cross_head_z"]]
    ti = [r.reshape(-1) for r in zs["text_intermediate_z"]]
    want = [(th[0], None, ti[0]), (th[1], None, ti[1]), (th[2], None, ti[2]),
            (th[0], th[1], ti[0]), (th[2], ch[0], ti[1]), (ch[1], ch[2], ti[2])]
    got = prune.caption_decoder_gates(zs, student.text_decoder.bert)
    assert len(got) == len(want) == golden["bert"]["num_hidden_layers"]
    for (s, c, m), (ws, wc, wm) in zip(got, want):
        assert torch.equal(s, ws) and torch.equal(m, wm)
        assert (c is None and wc is None) or torch.equal(c, wc)


def test_pruned_shapes_follow_the_gate_table(monkeypatch, golden):
    from efficientvlm_b200 import prune
    ref_ops.install(monkeypatch)
    model, zs = _materialised(golden)
    gates = prune.caption_decoder_gates(zs, model.text_decoder.bert)
    self_heads, cross_heads, widths = [], [], []
    for blk, (s, c, m) in zip(model.text_decoder.bert.encoder.layer, gates):
        n_self, n_ffn = int((s != 0).sum()), int((m != 0).sum())
        assert blk.attention.self.num_attention_heads == n_self
        assert blk.attention.self.query.weight.shape[0] == blk.attention.self.value.weight.shape[0] == 64 * n_self
        assert blk.attention.output.dense.weight.shape[1] == 64 * n_self
        if c is not None:
            n_cross = int((c != 0).sum())
            assert blk.crossattention.self.num_attention_heads == n_cross
            assert blk.crossattention.self.key.weight.shape[0] == blk.crossattention.output.dense.weight.shape[1] == 64 * n_cross
            cross_heads.append(n_cross)
            self_heads.append(n_self)
        assert blk.intermediate.dense.weight.shape[0] == blk.output.dense.weight.shape[1] == n_ffn
        widths.append(n_ffn)
    assert any(blk.attention.self.num_attention_heads == 1 for blk in model.text_decoder.bert.encoder.layer)
    assert any(w % 8 for w in widths)
    assert any(a != b for a, b in zip(self_heads, cross_heads))
    assert model.gates_folded and not type(model).gates_folded


def test_only_rows_the_gated_decoder_reads_matter(monkeypatch, golden):
    """cross_head_z[3] is never read (quirk Q1): changing it changes neither the gated logits nor the materialised weights;
    changing cross_head_z[2] (layer 5 cross-attention) changes the gated logits."""
    from efficientvlm_b200 import prune
    ref_ops.install(monkeypatch)
    student = _student(golden, RAGGED_SEED)
    zs = _zs(student)
    image_embeds = _image_embeds(student, golden["image"], zs)
    base = _teacher_forced_logits(student, golden, image_embeds, _decoder_gates(zs))
    for row, read in ((3, False), (2, True)):
        zs2 = dict(zs, cross_head_z=zs["cross_head_z"].clone())
        zs2["cross_head_z"][row] = zs2["cross_head_z"][row] * 0.5
        got = _teacher_forced_logits(student, golden, image_embeds, _decoder_gates(zs2))
        assert torch.equal(got, base) != read, row
    a, b = _student(golden, RAGGED_SEED), _student(golden, RAGGED_SEED)
    zs_b = dict(zs, cross_head_z=zs["cross_head_z"].clone())
    zs_b["cross_head_z"][3] = torch.rand_like(zs_b["cross_head_z"][3])
    prune.materialize(a, zs)
    prune.materialize(b, zs_b)
    sa, sb = a.state_dict(), b.state_dict()
    assert sa.keys() == sb.keys()
    assert all(torch.equal(sa[k], sb[k]) for k in sa if not k.startswith("l0_module."))


def test_materialised_teacher_forced_logits_match_gated(monkeypatch, golden):
    ref_ops.install(monkeypatch)
    gated = _student(golden, RAGGED_SEED)
    zs = _zs(gated)
    want = _teacher_forced_logits(gated, golden, _image_embeds(gated, golden["image"], zs), _decoder_gates(zs))
    model, _ = _materialised(golden)
    got = _teacher_forced_logits(model, golden, _image_embeds(model, golden["image"]), {})
    assert got.shape == want.shape
    assert (got - want).abs().max().item() <= 1e-5 * max(1.0, want.abs().max().item())


def test_materialised_decodes_match_gated(monkeypatch, golden):
    """Greedy (eager and sync_free), sampling and beam search of the materialised model against the gated model's host loops with the
    decoder gates applied."""
    ref_ops.install(monkeypatch)
    gated = _student(golden, RAGGED_SEED)
    zs = _zs(gated)
    image = golden["image"]
    enc = _image_embeds(gated, image, zs)
    model, _ = _materialised(golden)
    tok = gated.tokenizer
    prompt = tok([gated.prompt] * image.shape[0], return_tensors="pt").input_ids[:, :-1]

    def gated_no_beam(max_length, do_sample=False, repetition_penalty=1.0):
        return gated.text_decoder._generate_no_beam_search(
            input_ids=prompt.clone(), cur_len=prompt.shape[1], max_length=max_length, do_sample=do_sample, temperature=1, top_k=0, top_p=1,
            repetition_penalty=repetition_penalty, pad_token_id=tok.pad_token_id, eos_token_ids=[tok.sep_token_id], batch_size=image.shape[0],
            encoder_hidden_states=enc, encoder_attention_mask=None, **_decoder_gates(zs))

    for kw in (dict(max_length=10), dict(max_length=12, repetition_penalty=1.3)):
        want, _ = gated_no_beam(**kw)
        for sync_free in (False, True):
            _, ids = model.generate(image, greedy=True, return_ids=True, sync_free=sync_free, **kw)
            assert torch.equal(ids, want), (kw, sync_free)
    torch.manual_seed(golden["sample_seed"])
    want, want_lp = gated_no_beam(12, do_sample=True, repetition_penalty=1.1)
    torch.manual_seed(golden["sample_seed"])
    _, lp, ids = model.generate(image, sample=True, max_length=12, repetition_penalty=1.1, return_ids=True)
    assert torch.equal(ids, want)
    assert torch.allclose(lp, want_lp, rtol=0, atol=1e-5)
    for beams, min_length, rp in ((3, 5, 1.0), (2, 0, 1.3)):
        kw = dict(sample=False, num_beams=beams, max_length=12, min_length=min_length, repetition_penalty=rp, return_ids=True)
        want_caps, want = gated.generate(image, **kw)
        caps, ids = model.generate(image, **kw)
        assert torch.equal(ids, want) and caps == want_caps, (beams, min_length, rp)


def test_empty_layers_are_refused_before_any_weight_changes(monkeypatch, golden):
    from efficientvlm_b200 import prune
    ref_ops.install(monkeypatch)
    model = _student(golden, EMPTY_CROSS_SEED)
    zs = _zs(model)
    assert int((zs["cross_head_z"][2] != 0).sum()) == 0
    before = {k: v.clone() for k, v in model.state_dict().items()}
    with pytest.raises(NotImplementedError, match="decoder cross layer 5: every head is pruned"):
        prune.materialize(model, zs)
    after = model.state_dict()
    assert before.keys() == after.keys() and all(torch.equal(before[k], after[k]) for k in before)
    model = _student(golden, RAGGED_SEED)
    zs = _zs(model)
    zs["text_intermediate_z"] = zs["text_intermediate_z"].clone()
    zs["text_intermediate_z"][1] = 0
    with pytest.raises(NotImplementedError, match="decoder layer 1: every FFN column is pruned"):
        prune.materialize(model, zs)


def test_forward_after_materialise_raises(monkeypatch, golden):
    ref_ops.install(monkeypatch)
    model, _ = _materialised(golden)
    with pytest.raises(RuntimeError, match="materialised"):
        model(golden["image"], golden["captions"])
