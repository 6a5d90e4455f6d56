"""Beam search on the device (`evlm_beam_step`, `evlm_beam_finalize`, `evlm_kv_beam_reorder` and `BertLMHeadModel._beam_search_device`)
against the scorer's own statements (oracle/beam_search_oracle.py's BeamHypotheses) and against the host loop `_beam_search`."""
import math

import pytest
import torch

from oracle.beam_search_oracle import BeamHypotheses
from tests.helpers import caption_models, load_golden

pytestmark = pytest.mark.gpu


def _close(a, b):
    return abs(a - b) <= 1e-6 * max(1.0, abs(b))


class _Mirror:
    """Plain-Python restatement of one beam-search item set: `_beam_search`'s per-step statements, with finished items frozen the way
    the device loop freezes them (identity source, pad token, score 0)."""

    def __init__(self, prompt, batch, beams, width, pad, lp, early):
        self.beams, self.width, self.pad, self.lp, self.early = beams, width, pad, lp, early
        self.tokens = [list(prompt[r // beams]) for r in range(batch * beams)]
        self.scores = [0.0 if r % beams == 0 else -1e9 for r in range(batch * beams)]
        self.src = [0] * (batch * beams)
        self.done = [False] * batch
        self.hyps = [BeamHypotheses(beams, lp, early) for _ in range(batch)]
        self.eos_kept = self.eos_skipped = 0

    def step(self, logits, cur_len, min_length, rp, eos):
        beams, V = self.beams, logits.shape[1]
        # the exact log-softmax rounded to fp32 (the framework's fp32 CPU log_softmax is off by up to ~1e-5 on 30 k-entry rows)
        logp = torch.log_softmax(logits.double(), dim=-1).float()
        if rp != 1.0:
            hist = torch.tensor([t[:cur_len] for t in self.tokens])
            seen = torch.gather(logp, 1, hist)
            logp.scatter_(1, hist, torch.where(seen < 0, seen * rp, seen / rp))
        if cur_len < min_length:
            logp[:, eos] = -float("inf")
        scores = logp + torch.tensor(self.scores, dtype=torch.float32)[:, None]
        new_tokens, new_scores, new_src = [], [], []
        for b in range(len(self.done)):
            if self.done[b]:
                new_tokens += [self.pad] * beams
                new_scores += [0.0] * beams
                new_src += list(range(beams))
                continue
            flat = scores[b * beams:(b + 1) * beams].reshape(-1)
            vals, idx = torch.topk(flat, min(flat.numel(), 2 * beams + 32))
            cand = sorted(zip(vals.tolist(), idx.tolist()), key=lambda t: (-t[0], t[1]))
            if cand[-1][0] >= cand[2 * beams - 1][0]:                     # ties run past the window: order the whole item
                cand = sorted(zip(flat.tolist(), range(flat.numel())), key=lambda t: (-t[0], t[1]))
            top = cand[:2 * beams]
            kept = 0
            for rank, (sc, fi) in enumerate(top):
                tok, k = fi % V, fi // V
                if tok == eos:
                    if rank >= beams:
                        self.eos_skipped += 1
                        continue
                    self.eos_kept += 1
                    self.hyps[b].add(self.tokens[b * beams + k][:cur_len], sc)
                else:
                    new_tokens.append(tok)
                    new_scores.append(sc)
                    new_src.append(k)
                    kept += 1
                if kept == beams:
                    break
            self.done[b] = self.hyps[b].is_done(top[0][0], cur_len)
        self.tokens = [self.tokens[(r // beams) * beams + new_src[r]][:cur_len] + [new_tokens[r]] for r in range(len(self.tokens))]
        self.scores, self.src = new_scores, new_src

    def finalize(self, max_length, eos):
        out = []
        for b, h in enumerate(self.hyps):
            if not self.done[b]:
                for k in range(self.beams):
                    h.add(self.tokens[b * self.beams + k], self.scores[b * self.beams + k])
            best = sorted(h.beams, key=lambda t: t[0])[-1][1]
            row = [self.pad] * max_length
            row[:len(best)] = best[:max_length]
            if len(best) < max_length:
                row[len(best)] = eos
            out.append((row, len(best)))
        return out


def _state(batch, beams, width, prompt, pad, dev):
    rows = batch * beams
    tokens = torch.full((rows, width), pad, dtype=torch.int64, device=dev)
    tokens[:, :len(prompt[0])] = torch.tensor(prompt, device=dev).repeat_interleave(beams, 0)
    scores = torch.zeros(batch, beams, device=dev)
    scores[:, 1:] = -1e9
    return dict(tokens=tokens, beam_scores=scores.view(-1), beam_src=torch.zeros(rows, dtype=torch.int32, device=dev),
                done=torch.zeros(batch, dtype=torch.int32, device=dev), hyp_tokens=torch.zeros(batch, beams, width, dtype=torch.int64, device=dev),
                hyp_len=torch.zeros(batch, beams, dtype=torch.int32, device=dev), hyp_score=torch.zeros(batch, beams, dtype=torch.float64, device=dev),
                hyp_count=torch.zeros(batch, dtype=torch.int32, device=dev), hyp_worst=torch.full((batch,), 1e9, dtype=torch.float64, device=dev))


def _assert_state(st, m, beams, cur_len):
    assert st["tokens"][:, :cur_len + 1].tolist() == [t[:cur_len + 1] for t in m.tokens]
    assert st["beam_src"].tolist() == m.src
    assert st["done"].tolist() == [int(d) for d in m.done]
    for a, b in zip(st["beam_scores"].tolist(), m.scores):
        assert _close(a, b), (a, b)
    for b, h in enumerate(m.hyps):
        n = int(st["hyp_count"][b])
        assert n == len(h.beams), (b, n, len(h.beams))
        for j, (sc, toks) in enumerate(h.beams):
            L = int(st["hyp_len"][b, j])
            assert L == len(toks) and st["hyp_tokens"][b, j, :L].tolist() == toks, (b, j)
            assert _close(float(st["hyp_score"][b, j]), sc), (b, j)
        assert _close(float(st["hyp_worst"][b]), h.worst_score)


@pytest.mark.parametrize("V,ld,rp,early", [(30522, 30524, 1.0, False), (30522, 30524, 1.3, True), (37, 37, 1.3, False), (37, 40, 1.0, True)])
def test_beam_step_matches_the_scorer_statements(V, ld, rp, early):
    from efficientvlm_b200 import kernels as K
    dev = "cuda"
    batch, beams, width, eos, pad, min_length, lp = 5, 3, 13, 2, 0, 5, 1.0
    prompt = [[5, 7, 5]] * batch                                          # a repeated prompt token: penalised once
    st = _state(batch, beams, width, prompt, pad, dev)
    m = _Mirror(prompt, batch, beams, width, pad, lp, early)
    g = torch.Generator().manual_seed(V + int(rp * 10) + early)
    rows = batch * beams
    for cur_len in range(3, width):
        x = torch.randn(rows, V, generator=g) * 3.0
        M = float(x.max())
        x[0, 9] = x[0, 11] = M + 4.0                                       # planted exact tie inside one row (item 0)
        x[2 * beams + 1:3 * beams] = 0.5                                   # item 2: flat rows, exact ties between their tokens
        x[3 * beams, eos] = M + 30.0                                       # item 3: eos at rank 0 (a hypothesis once cur_len >= min_length)
        # item 4: every row has eos 1 above one other token; with beam scores -1, -1.5, -3 the candidates rank
        # eos0, eos1, tok0, tok1, eos2, tok2: eos2 is visited at rank 4 >= beams with two beams still open and must be skipped
        r = 4 * beams
        for k in range(beams):
            x[r + k, eos] = M + 30.0
            x[r + k, 20 + k] = M + 29.0
        planted = [-1.0, -1.5, -3.0]
        st["beam_scores"][r:r + beams] = torch.tensor(planted, device=dev)
        m.scores[r:r + beams] = planted
        buf = torch.zeros(rows, ld)
        buf[:, :V] = x
        logits = buf.to(dev)[:, :V]
        K.beam_step(logits, beams, cur_len, min_length, rp, lp, early, eos, pad, **st)
        m.step(x, cur_len, min_length, rp, eos)
        _assert_state(st, m, beams, cur_len)
    assert m.eos_kept > 0 and m.eos_skipped > 0
    if early:
        assert any(m.done)
    out, lengths = K.beam_finalize(beams, width, width, lp, eos, pad, st["tokens"], st["beam_scores"], st["done"], st["hyp_tokens"],
                                   st["hyp_len"], st["hyp_score"], st["hyp_count"], st["hyp_worst"])
    want = m.finalize(width, eos)
    assert out.tolist() == [w[0] for w in want] and lengths.tolist() == [w[1] for w in want]


def test_beam_finalize_tie_rule_and_layout():
    """The best hypothesis is the LAST of the maximal scores in list order (stable sort, [-1]); out = hypothesis, eos if shorter than
    max_length, pad."""
    from efficientvlm_b200 import kernels as K
    dev, batch, beams, width, eos, pad, lp = "cuda", 3, 3, 8, 2, 0, 1.0
    st = _state(batch, beams, width, [[1, 1, 1]] * batch, pad, dev)
    g = torch.Generator().manual_seed(3)
    st["tokens"].copy_(torch.randint(3, 50, (batch * beams, width), generator=g).to(dev))
    m = _Mirror([[1]] * batch, batch, beams, width, pad, lp, False)
    m.tokens = st["tokens"].tolist()
    hyps = {0: [(-1.0, 4), (-0.5, 5), (-0.5, 6)], 1: [(-2.0, 3)], 2: []}
    beam_scores = [0.0, 0.0, 0.0, -4.0, -4.0, -100.0, -3.0, -1.0, -2.0]
    m.done = [True, False, False]
    for b, hs in hyps.items():
        for j, (sc, L) in enumerate(hs):
            toks = torch.randint(3, 50, (L,), generator=g)
            st["hyp_tokens"][b, j, :L] = toks.to(dev)
            st["hyp_len"][b, j] = L
            st["hyp_score"][b, j] = sc
            m.hyps[b].beams.append((sc, toks.tolist()))
        st["hyp_count"][b] = len(hs)
        w = min([sc for sc, _ in hs], default=1e9)
        st["hyp_worst"][b] = w
        m.hyps[b].worst_score = w
    st["done"].copy_(torch.tensor([1, 0, 0], dtype=torch.int32))
    st["beam_scores"].copy_(torch.tensor(beam_scores))
    m.scores = beam_scores
    out, lengths = K.beam_finalize(beams, width, width, lp, eos, pad, st["tokens"], st["beam_scores"], st["done"], st["hyp_tokens"],
                                   st["hyp_len"], st["hyp_score"], st["hyp_count"], st["hyp_worst"])
    want = m.finalize(width, eos)
    assert out.tolist() == [w[0] for w in want] and lengths.tolist() == [w[1] for w in want]
    assert lengths.tolist() == [6, 8, 8]                                   # item 0: the last of the two -0.5 scores; item 1: beam 1
    assert out[1].tolist() == st["tokens"][4].tolist() and out[2].tolist() == st["tokens"][7].tolist()
    assert out[0, 6].item() == eos and out[0, 7].item() == pad


@pytest.mark.parametrize("row_elems", [256, 1536, 4096])
def test_kv_beam_reorder_in_place_matches_index_select(row_elems):
    from efficientvlm_b200 import kernels as K
    dev, cap, length = "cuda", 11, 7
    for beams, src in ((3, [[1, 1, 0], [0, 1, 2], [2, 1, 0]]), (4, [[3, 3, 3, 3], [1, 0, 3, 2]])):
        batch = len(src)
        rows = batch * beams
        caches = [torch.randn(rows, cap, row_elems, device=dev).to(torch.bfloat16) for _ in range(3)]
        before = [c.clone() for c in caches]
        bs = torch.tensor(src, dtype=torch.int32, device=dev).view(-1)
        idx = (torch.arange(rows, device=dev) // beams * beams + bs).long()
        K.kv_beam_reorder(caches, bs, beams, length)
        for c, c0 in zip(caches, before):
            assert torch.equal(c[:, :length], c0[:, :length].index_select(0, idx))
            assert torch.equal(c[:, length:], c0[:, length:])
    with pytest.raises(ValueError):
        K.kv_beam_reorder(caches, bs, 9, length)


def test_beam_wrappers_reject_bad_arguments():
    from efficientvlm_b200 import kernels as K
    st = _state(2, 3, 6, [[1, 2]] * 2, 0, "cuda")
    logits = torch.zeros(6, 37, device="cuda")
    with pytest.raises(ValueError):
        K.beam_step(logits, 1, 2, 0, 1.0, 1.0, False, 2, 0, **st)                              # num_beams outside 2..8
    with pytest.raises(ValueError):
        K.beam_step(logits[:, :6], 3, 2, 0, 1.0, 1.0, False, 2, 0, **st)                       # vocab <= 2 * num_beams
    with pytest.raises(ValueError):
        K.beam_step(logits, 3, 6, 0, 1.0, 1.0, False, 2, 0, **st)                              # no column left for the new token
    with pytest.raises(ValueError):
        K.beam_finalize(3, 6, 7, 1.0, 2, 0, st["tokens"], st["beam_scores"], st["done"], st["hyp_tokens"], st["hyp_len"], st["hyp_score"],
                        st["hyp_count"], st["hyp_worst"])                                      # max_length beyond the history width


def _tiny_student():
    g = load_golden("caption_kd_tiny")
    student, _ = caption_models(g)
    return g, student.cuda().eval()


def _host_top_scores(fn):
    """Runs fn() and returns the host loop's top 2 * num_beams scores of every step (torch.topk inside `_beam_search`)."""
    rec, orig = [], torch.topk

    def spy(*a, **k):
        r = orig(*a, **k)
        if r[0].dim() == 2:
            rec.append(r[0].float().cpu())
        return r
    torch.topk = spy
    try:
        out = fn()
    finally:
        torch.topk = orig
    return out, rec


def _compare_with_tie_rule(dev_ids, host_ids, host_tops):
    """Rows must be identical, unless the host loop's own top-2*beams scores of that item hold a near-tie (within 1e-5 relative) at some
    step: an order that torch.topk and the device kernel may break differently."""
    assert dev_ids.shape == host_ids.shape, (dev_ids.shape, host_ids.shape)
    for b in range(dev_ids.shape[0]):
        if torch.equal(dev_ids[b], host_ids[b]):
            continue
        tie = False
        for t in host_tops:
            s = t[b].tolist()
            tie |= any(abs(s[i] - s[i + 1]) <= 1e-5 * max(1.0, abs(s[i])) for i in range(len(s) - 1))
        assert tie, ("row %d differs without a near-tie in the host loop's candidates" % b, dev_ids[b].tolist(), host_ids[b].tolist())


def test_device_loop_equals_host_loop_on_the_caption_student():
    from efficientvlm_b200 import eff_bert as EB
    from efficientvlm_b200 import ops
    g, student = _tiny_student()
    image = g["image"].cuda()
    prompt_len = student.tokenizer([student.prompt], return_tensors="pt").input_ids.shape[1] - 1
    calls = [0]
    orig_reorder = EB.BertLMHeadModel._reorder_cache

    def counting(self, past, idx):
        calls[0] += 1
        return orig_reorder(self, past, idx)
    EB.BertLMHeadModel._reorder_cache = counting
    try:
        for num_beams, max_length, min_length, rp in ((3, 12, 5, 1.0), (2, 9, 0, 1.0), (4, 14, 7, 1.3), (3, prompt_len + 1, 0, 1.0)):
            kw = dict(sample=False, num_beams=num_beams, max_length=max_length, min_length=min_length, repetition_penalty=rp, return_ids=True)
            EB.BEAM_SEARCH_ON_DEVICE = False
            (caps_h, ids_h), tops = _host_top_scores(lambda: student.generate(image, **kw))
            EB.BEAM_SEARCH_ON_DEVICE = True
            calls[0] = 0
            caps_d, ids_d = student.generate(image, **kw)
            assert calls[0] == 0                                           # in-place re-order at every step: no copying fallback
            _compare_with_tie_rule(ids_d, ids_h, tops)
            if torch.equal(ids_d, ids_h):
                assert caps_d == caps_h
        spare = ops.KV_CACHE_SPARE
        ops.KV_CACHE_SPARE = 3                                             # the cache runs out mid-loop: copying re-order from there on
        try:
            kw = dict(sample=False, num_beams=3, max_length=12, min_length=5, return_ids=True)
            calls[0] = 0
            _, ids_s = student.generate(image, **kw)
            assert calls[0] > 0
            EB.BEAM_SEARCH_ON_DEVICE = False
            (_, ids_h), tops = _host_top_scores(lambda: student.generate(image, **kw))
            _compare_with_tie_rule(ids_s, ids_h, tops)
        finally:
            ops.KV_CACHE_SPARE = spare
    finally:
        EB.BEAM_SEARCH_ON_DEVICE = True
        EB.BertLMHeadModel._reorder_cache = orig_reorder


def test_device_loop_launches_fewer_kernels_than_the_host_loop():
    from efficientvlm_b200 import eff_bert as EB
    g, student = _tiny_student()
    image = g["image"].cuda()
    kw = dict(sample=False, num_beams=3, max_length=12, min_length=5, return_ids=True)

    def kernels(flag):
        EB.BEAM_SEARCH_ON_DEVICE = flag
        try:
            student.generate(image, **kw)
            torch.cuda.synchronize()
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as p:
                student.generate(image, **kw)
                torch.cuda.synchronize()
            return sum(1 for e in p.events() if e.device_type == torch.autograd.DeviceType.CUDA)
        finally:
            EB.BEAM_SEARCH_ON_DEVICE = True
    n_dev, n_host = kernels(True), kernels(False)
    assert 0 < n_dev < n_host, (n_dev, n_host)


def test_beam_search_graph_capture_replays_on_new_encoder_states():
    g, student = _tiny_student()
    dec = student.text_decoder
    tok = student.tokenizer
    image = g["image"].cuda()
    zs = student._zs(False)
    gates = dict(head_z=torch.cat((zs["text_head_z"], zs["cross_head_z"]), dim=0),
                 mlp_z=torch.cat((zs["text_intermediate_z"], zs["cross_intermediate_z"]), dim=0))
    with torch.no_grad():
        enc_a = student.vision_encoder(image, head_z=zs["vision_head_z"], mlp_z=zs["vision_intermediate_z"])[0].repeat_interleave(3, dim=0)
    enc_b = torch.flip(enc_a, dims=[0]).contiguous() * 0.9
    prompt = tok([student.prompt] * image.size(0), return_tensors="pt").input_ids[:, :-1].cuda()
    kw = dict(max_length=12, min_length=5, num_beams=3, eos_token_id=tok.sep_token_id, pad_token_id=tok.pad_token_id, **gates)

    def run(enc, sync_free):
        return dec.generate(input_ids=prompt.clone(), encoder_hidden_states=enc, encoder_attention_mask=None, sync_free=sync_free, **kw)
    static_enc = enc_a.clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        run(static_enc, True)                                              # warm-up
    torch.cuda.current_stream().wait_stream(side)
    static_enc.copy_(enc_a)                                                # new version: the capture projects the encoder states itself
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static_out = run(static_enc, True)
    static_enc.copy_(enc_b)
    graph.replay()
    torch.cuda.synchronize()
    eager_b = run(enc_b.clone(), True)
    assert torch.equal(static_out, eager_b)
    trimmed = run(enc_b.clone(), False)
    n = trimmed.shape[1]
    assert torch.equal(eager_b[:, :n], trimmed)
    assert bool((eager_b[:, n:] == tok.pad_token_id).all())


def test_device_loop_equals_host_loop_at_full_width():
    """The caption student at the benchmark's BERT-base / ViT-B widths, 224 px, batch 4, 3 beams, max_length 20, min_length 5."""
    import bench
    from efficientvlm_b200 import eff_bert as EB
    from efficientvlm_b200.captioning import EffXVLMForCaptioning
    torch.manual_seed(42)
    cfg = dict(bench.itr_cfg("student", 224, sparsity=0.35), prompt="a picture of ", max_tokens=40, label_smoothing=0.1)
    model = EffXVLMForCaptioning(cfg, tokenizer=bench.PromptTokenizer()).cuda().eval()
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():
        for la in model.l0_module.z_logas.values():
            la.copy_((torch.randn(la.shape, generator=g) * 3.0 + 1.5).cuda())
    image = torch.randn(4, 3, 224, 224, generator=torch.Generator().manual_seed(42)).cuda()
    kw = dict(sample=False, num_beams=3, max_length=20, min_length=5, return_ids=True)
    try:
        EB.BEAM_SEARCH_ON_DEVICE = False
        (_, ids_h), tops = _host_top_scores(lambda: model.generate(image, **kw))
    finally:
        EB.BEAM_SEARCH_ON_DEVICE = True
    _, ids_d = model.generate(image, **kw)
    _compare_with_tie_rule(ids_d, ids_h, tops)
    assert not math.isnan(float(ids_d.float().sum()))
