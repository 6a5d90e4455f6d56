"""prune.materialize on the retrieval and NLVR2 students (host logic, CPU, through the oracle operators of tests/ref_ops.py): the
physically smaller, gate-free models compute what the gated models compute.

Retrieval (text / fusion modes, separate gates): the materialised fixture student reproduces the REFERENCE's masked evaluation
(tests/golden/itr_eval_tiny.pt), and with ragged seeded log-alphas the materialised evaluation equals the masked one.  NLVR2 (multi_modal
mode with concatenated gates, quirk Q1, and key / value projections tied across the two per-image copies of a fusion layer): the
materialised model's eval prediction equals the gated model's own."""
import pytest
import torch

from tests import helpers, ref_ops
from tests.helpers import assert_close, itr_eval_setup, load_golden, nlvr_models

# Log-alphas from these seeds (x 3.0 + 1.5, like bench.py's synthetic gates) leave 1-head vision, self and cross-attention layers and FFN
# widths that are not multiples of 8; in NLVR the two copies of fusion layers 3 / 4 and 7 / 8 get different cross-attention head counts.
RAGGED_SEED = 10
ITR_RAGGED_SEED = 12
# With this seed the gated NLVR forward reads an all-zero cross-attention head row in encoder layer 6.
EMPTY_CROSS_SEED = 26


def seed_logas(model, seed):
    gen = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, la in model.l0_module.named_parameters():
            if name.endswith("_loga"):
                la.copy_(torch.randn(la.shape, generator=gen) * 3.0 + 1.5)
    return model


def det_gates(model):
    with torch.no_grad():
        return model.l0_module.forward(training=False)


def materialised(model):
    from efficientvlm_b200 import prune
    prune.materialize(model)
    return model


def nlvr_student(g, seed=RAGGED_SEED):
    student, _ = nlvr_models(g)
    return seed_logas(student, seed)


def nlvr_batch(g, device="cpu"):
    return tuple(g[k].to(device) for k in ("image", "text_ids", "text_atts", "targets"))


def nlvr_predict(model, batch):
    with torch.no_grad():
        return model(*batch, train=False)


def cross_pairs(model):
    """(first copy, second copy) BertLayer of every NLVR fusion layer."""
    layers = model._bert().encoder.layer
    return [(layers[model.num_text_layers + 2 * i], layers[model.num_text_layers + 2 * i + 1]) for i in range(model.num_cross_layers)]


@pytest.fixture(scope="module")
def nlvr_golden():
    return load_golden("nlvr_kd_tiny")


def test_materialised_retrieval_evaluation_reproduces_masked_golden(monkeypatch):
    """retrieval_eval.evaluation on a materialised copy of the fixture's student: similarities, candidate sets, scores, recalls, the
    two-rank split and every re-rank batching mode against the reference's MASKED evaluation."""
    ref_ops.install(monkeypatch)
    monkeypatch.setattr(helpers, "itr_eval_setup", lambda g, device: (materialised(itr_eval_setup(g, device)[0]),) + itr_eval_setup(g, device)[1:])
    helpers.run_itr_eval(load_golden("itr_eval_tiny"), "cpu", 1e-5, 1e-4, exact_candidates=True)


def test_materialised_retrieval_evaluation_with_pruned_heads_equals_masked(monkeypatch):
    from efficientvlm_b200 import retrieval_eval as RE
    ref_ops.install(monkeypatch)
    g = load_golden("itr_eval_tiny")
    runs = []
    for fold in (False, True):
        model, loader, tokenizer = itr_eval_setup(g, "cpu")
        seed_logas(model, ITR_RAGGED_SEED)
        if fold:
            zs = det_gates(model)
            materialised(model)
            cross = [blk.crossattention.self.num_attention_heads for blk in model._bert().encoder.layer[3:]]
            assert cross == [int((r != 0).sum()) for r in zs["cross_head_z"].reshape(6, 2)[1::2]] and 1 in cross
            assert min(a.self_attn.num_heads for a in model.vision_encoder.encoder.layers) == 1
        details = {}
        runs.append(RE.evaluation(model, loader, tokenizer, "cpu", g["config"], details=details) + (details,))
    (mi, mt, ms, md), (fi, ft, fs, fd) = runs
    assert ms == fs
    assert all(v is None for v in fd["zs"].values())
    assert_close(fd["sims_matrix"], md["sims_matrix"], 1e-5, "similarities")
    assert ((mi == -100) == (fi == -100)).all() and ((mt == -100) == (ft == -100)).all()
    assert_close(torch.from_numpy(fi), torch.from_numpy(mi), 1e-4, "image->text scores")
    assert_close(torch.from_numpy(ft), torch.from_numpy(mt), 1e-4, "text->image scores")


def test_nlvr_gate_table_follows_quirk_q1(monkeypatch, nlvr_golden):
    """Text layer i < F reads head_z[i] / mlp_z[i] of cat(text_*, cross_*); fusion copy i >= F reads self 2(i - F), cross 2(i - F) + 1
    and FFN i - F, so the first fusion copies re-use the text rows and cross_head_z[9..11] are never read."""
    from efficientvlm_b200 import prune
    ref_ops.install(monkeypatch)
    student = nlvr_student(nlvr_golden)
    zs = det_gates(student)
    heads = [r.reshape(-1) for r in torch.cat((zs["text_head_z"], zs["cross_head_z"]))]
    mlps = [r.reshape(-1) for r in torch.cat((zs["text_intermediate_z"], zs["cross_intermediate_z"]))]
    got = prune.concat_gate_rows(zs, student._bert())
    assert len(got) == 9
    for i, (s, c, m) in enumerate(got):
        if i < 3:
            assert torch.equal(s, heads[i]) and c is None and torch.equal(m, mlps[i])
        else:
            assert torch.equal(s, heads[2 * (i - 3)]) and torch.equal(c, heads[2 * (i - 3) + 1]) and torch.equal(m, mlps[i - 3])


def test_materialised_nlvr_prediction_equals_masked(monkeypatch, nlvr_golden):
    ref_ops.install(monkeypatch)
    batch = nlvr_batch(nlvr_golden)
    gated = nlvr_student(nlvr_golden)
    want = nlvr_predict(gated, batch)
    model = materialised(nlvr_student(nlvr_golden))
    assert model.gates_folded and not type(model).gates_folded
    widths = [blk.intermediate.dense.weight.shape[0] for blk in model._bert().encoder.layer]
    assert any(w % 8 for w in widths)
    assert any(blk.attention.self.num_attention_heads == 1 for blk in model._bert().encoder.layer)
    assert any(a.crossattention.self.num_attention_heads == 1 for a, _ in cross_pairs(model))
    got = nlvr_predict(model, batch)
    assert got.shape == want.shape
    assert (got - want).abs().max().item() <= 1e-5 * max(1.0, want.abs().max().item())
    assert torch.equal(got.argmax(1), want.argmax(1))


def test_nlvr_fusion_copies_own_their_key_value(monkeypatch, nlvr_golden):
    """The tie of share_cross_attention is undone before folding: every copy folds and prunes its own cross-head gate row."""
    from efficientvlm_b200 import prune
    ref_ops.install(monkeypatch)
    gated = nlvr_student(nlvr_golden)
    assert all(a.crossattention.self.value.weight is b.crossattention.self.value.weight for a, b in cross_pairs(gated))
    zs = det_gates(gated)
    rows = prune.concat_gate_rows(zs, gated._bert())
    model = materialised(nlvr_student(nlvr_golden))
    differ = 0
    for i, (a, b) in enumerate(cross_pairs(model)):
        sa, sb = a.crossattention.self, b.crossattention.self
        for name in ("key", "value"):
            la, lb = getattr(sa, name), getattr(sb, name)
            assert la.weight is not lb.weight and la.bias is not lb.bias
            assert la.weight.data_ptr() != lb.weight.data_ptr()
        for blk, (_, c, _) in ((a, rows[3 + 2 * i]), (b, rows[4 + 2 * i])):
            n = int((c != 0).sum())
            assert blk.crossattention.self.num_attention_heads == n
            assert blk.crossattention.self.key.weight.shape[0] == blk.crossattention.self.value.weight.shape[0] == 64 * n
            assert blk.crossattention.output.dense.weight.shape[1] == 64 * n
        differ += sa.num_attention_heads != sb.num_attention_heads
    assert differ >= 1
    names = [n for n, _ in model.named_parameters()]
    assert all(any(n.endswith("layer.%d.crossattention.self.%s.weight" % (j, kv)) for n in names) for j in range(3, 9) for kv in ("key", "value"))


def test_refused_nlvr_plan_leaves_the_model_untouched(monkeypatch, nlvr_golden):
    from efficientvlm_b200 import prune
    ref_ops.install(monkeypatch)
    for seed, tweak, msg in ((EMPTY_CROSS_SEED, None, "encoder cross layer 6: every head is pruned"),
                             (RAGGED_SEED, ("text_intermediate_z", 1), "encoder layer 1: every FFN column is pruned"),
                             (RAGGED_SEED, ("vision_head_z", 0), "vision layer 0: every head is pruned")):
        model = nlvr_student(nlvr_golden, seed)
        zs = det_gates(model)
        if tweak is not None:
            zs[tweak[0]] = zs[tweak[0]].clone()
            zs[tweak[0]][tweak[1]] = 0
        before = {k: v.clone() for k, v in model.state_dict().items()}
        params = [id(p) for p in model.parameters()]
        with pytest.raises(NotImplementedError, match=msg):
            prune.materialize(model, zs)
        after = model.state_dict()
        assert before.keys() == after.keys() and all(torch.equal(before[k], after[k]) for k in before), msg
        assert [id(p) for p in model.parameters()] == params and not model.gates_folded


def test_training_forwards_refuse_a_materialised_model(monkeypatch, nlvr_golden):
    ref_ops.install(monkeypatch)
    model = materialised(nlvr_student(nlvr_golden))
    batch = nlvr_batch(nlvr_golden)
    with pytest.raises(RuntimeError, match="materialised"):
        model(*batch, train=True)
    with pytest.raises(RuntimeError, match="materialised"):
        model(*batch, train=False, output_attentions=True, output_hidden_states=True)
    g = load_golden("itr_eval_tiny")
    itr = materialised(itr_eval_setup(g, "cpu")[0])
    with pytest.raises(RuntimeError, match="materialised"):
        itr(g["images"][:2], g["text_ids"][:2], g["text_atts"][:2])
    with pytest.raises(RuntimeError, match="materialised"):
        itr(g["images"][:2], g["text_ids"][:2], g["text_atts"][:2], output_attentions=True, output_hidden_states=True)
