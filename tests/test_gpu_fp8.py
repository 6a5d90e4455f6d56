"""FP8 inference on the device: the quantise kernel bit for bit against its host mirror, evlm_gemm_fp8 against fp64 on the dequantised
operands (weight-stream and tcgen05 paths, tile edges, ragged K, every epilogue it supports), the arguments it refuses, and the
materialised VQA / captioning students with fp8.enable against an fp32 emulation of the same quantised arithmetic."""
import copy
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from efficientvlm_b200 import _lib, fp8
from efficientvlm_b200 import kernels as K
from efficientvlm_b200._lib import ACT_GELU_ERF, ACT_NONE, ACT_QUICK_GELU
from tests.helpers import load_golden, sd_from_spec
from tests.test_gpu_caption_materialize import full_width  # noqa: F401  (fixture: bench.py's materialised caption_infer student)

pytestmark = pytest.mark.gpu
bf16, f32 = torch.bfloat16, torch.float32


def _rows(R, Kd, dtype, seed, pitch=0):
    """[R, Kd] view of a [R, Kd + pitch] buffer (NaN in the pitch padding) with per-row magnitudes over six decades, one outlier row,
    one all-zero row."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(R, Kd, generator=g) * torch.logspace(-3, 3, R)[:, None]
    if R > 2:
        x[1, Kd // 2] = 3e4
        x[2] = 0
    buf = torch.full((R, Kd + pitch), float("nan"), dtype=dtype)
    buf[:, :Kd] = x.to(dtype)
    return buf.cuda()[:, :Kd]


@pytest.mark.parametrize("dtype", [bf16, f32])
@pytest.mark.parametrize("Kd", [1, 15, 16, 17, 768, 2493, 3072])
@pytest.mark.parametrize("pitch", [0, 3, 8])
def test_quant_rows_bit_exact_against_mirror(dtype, Kd, pitch):
    x = _rows(37, Kd, dtype, Kd + pitch)
    q, s = K.quant_rows_e4m3(x)
    torch.cuda.synchronize()
    wq, ws = fp8.quant_rows_reference(x.cpu())
    assert q.stride(0) % 16 == 0
    assert torch.equal(q.cpu().view(torch.uint8), wq.view(torch.uint8))
    assert torch.equal(s.cpu().view(torch.int32), ws.view(torch.int32))
    full = q.as_strided((q.shape[0], q.stride(0)), (q.stride(0), 1)).cpu().view(torch.uint8)
    assert int(full[:, Kd:].abs().sum()) == 0, "pad bytes must be zero"


# ---------------------------------------------------------------------------------------------------------------------------------
def _operands(M, N, Kd, seed):
    g = torch.Generator().manual_seed(seed)
    a = (torch.randn(M, Kd, generator=g) * torch.rand(M, 1, generator=g) * 4).to(bf16).cuda()
    b = (torch.randn(N, Kd, generator=g) * 0.05).cuda()
    qa, sa = K.quant_rows_e4m3(a)
    qb, sb = K.quant_rows_e4m3(b)
    return qa, sa, qb, sb


def _reference(qa, sa, qb, sb):
    """(fp64 sa[m] sb[n] sum_k qa qb, fp64 sa sb sum_k |qa qb|) on the device."""
    A, B = qa.double(), qb.double()
    sc = sa.double()[:, None] * sb.double()[None, :]
    return (A @ B.t()) * sc, (A.abs() @ B.abs().t()) * sc


def _check(D, want, mag, bf16_out, what):
    err = (D.double() - want).abs()
    bound = 1e-5 * mag + 1e-6
    if bf16_out:
        bound = bound + 2.0 ** -8 * want.abs()
    assert bool(torch.isfinite(D).all()), what
    worst = float((err / bound).max())
    assert worst <= 1.0, (what, worst, float(err.max()))


_SHAPES = [(M, N, Kd) for M in (1, 24, 32, 33, 127, 129, 12288) for N in (64, 200, 768, 2304, 30522) for Kd in (16, 768, 2493, 3072)
           if M * N * Kd <= 12288 * 30522 * 768]


@pytest.mark.parametrize("M,N,Kd", _SHAPES)
def test_gemm_fp8_against_fp64(M, N, Kd):
    qa, sa, qb, sb = _operands(M, N, Kd, M + 7 * N + 13 * Kd)
    bias = torch.randn(N, generator=torch.Generator().manual_seed(N)).cuda()
    D = torch.full((M, (N + 3) // 4 * 4), float("nan"), dtype=f32, device="cuda")[:, :N]
    K.gemm_fp8(qa, sa, qb, sb, D, M, N, Kd, bias=bias)
    want, mag = _reference(qa, sa, qb, sb)
    _check(D, want + bias.double(), mag + bias.double().abs(), False, (M, N, Kd))


def _gelu_erf(x):
    return 0.5 * x * (1 + torch.erf(x / 2 ** 0.5))


@pytest.mark.parametrize("M,N,Kd", [(24, 768, 768), (129, 2304, 768), (1024, 3072, 768), (33, 768, 2493), (512, 768, 3072)])
@pytest.mark.parametrize("flavour", ["alpha", "quick_gelu", "gelu_erf", "res_f32", "res_bf16", "d_bf16"])
def test_gemm_fp8_epilogues(M, N, Kd, flavour):
    qa, sa, qb, sb = _operands(M, N, Kd, 3 * M + N)
    g = torch.Generator().manual_seed(Kd)
    bias = torch.randn(N, generator=g).cuda()
    want, mag = _reference(qa, sa, qb, sb)
    want, mag = want + bias.double(), mag + bias.double().abs()
    d_bf16 = flavour in ("d_bf16", "quick_gelu", "gelu_erf")
    D = torch.empty(M, N, dtype=bf16 if d_bf16 else f32, device="cuda")
    kw = dict(bias=bias)
    if flavour == "alpha":
        kw.update(alpha=0.125, alpha_cols=N // 3)
        cols = torch.arange(N, device="cuda") < N // 3
        want = torch.where(cols, want * 0.125, want)
        mag = torch.where(cols, mag * 0.125, mag)
    elif flavour in ("quick_gelu", "gelu_erf"):
        aux = torch.empty(M, N, dtype=bf16, device="cuda")
        kw.update(act=ACT_QUICK_GELU if flavour == "quick_gelu" else ACT_GELU_ERF, aux_out=aux)
    elif flavour.startswith("res"):
        res = torch.randn(M, N, generator=g).to(f32 if flavour == "res_f32" else bf16).cuda()
        kw.update(residual=res)
    K.gemm_fp8(qa, sa, qb, sb, D, M, N, Kd, **kw)
    if flavour in ("quick_gelu", "gelu_erf"):
        _check(aux, want, mag, True, "aux_out")
        act = (lambda x: x * torch.sigmoid(1.702 * x)) if flavour == "quick_gelu" else _gelu_erf
        # the activation's slope is below 1.13: the pre-activation bound carries over, plus the fast formulations' 2e-6 absolute
        err = (D.double() - act(want)).abs()
        bound = 1.13 * (1e-5 * mag + 1e-6) + 2e-6 + 2.0 ** -8 * act(want).abs()
        assert bool((err <= bound).all()), float((err / bound).max())
        return
    if flavour.startswith("res"):
        want, mag = want + res.double(), mag + res.double().abs()
    _check(D, want, mag, d_bf16, flavour)


def _args(M=64, N=64, Kd=64):
    a = torch.zeros(M, Kd, dtype=torch.uint8, device="cuda")
    b = torch.zeros(N, Kd, dtype=torch.uint8, device="cuda")
    d = torch.empty(M, N, dtype=f32, device="cuda")
    s = torch.ones(max(M, N), dtype=f32, device="cuda")
    g = _lib.GemmArgs()
    g.M, g.N, g.K = M, N, Kd
    g.A, g.lda, g.B, g.ldb = a.data_ptr(), Kd, b.data_ptr(), Kd
    g.D, g.ldd, g.d_dtype = d.data_ptr(), N, _lib.F32
    g.alpha, g.splits = 1.0, 1
    return g, (a, b, d, s)


@pytest.mark.parametrize("M", [8, 256])
@pytest.mark.parametrize("bad", ["epi_mode", "dropout", "splits", "accumulate", "gate", "m_limit", "k_limit", "a_mn", "b_mn", "pitch",
                                 "aux_without_act"])
def test_gemm_fp8_rejects(M, bad):
    g, keep = _args(M=M)
    lim = torch.ones(1, dtype=torch.int32, device="cuda")
    if bad == "epi_mode":
        g.epi_mode = _lib.EPI_ACT_BACKWARD
        g.aux_in, g.ld_aux_in = keep[2].data_ptr(), 64
    elif bad == "dropout":
        g.dropout_p = 0.1
    elif bad == "splits":
        g.splits = 2
    elif bad == "accumulate":
        g.accumulate = 1
    elif bad == "gate":
        g.gate, g.gate_mode = keep[3].data_ptr(), _lib.GATE_POST_ACT
    elif bad in ("m_limit", "k_limit"):
        setattr(g, bad, lim.data_ptr())
    elif bad in ("a_mn", "b_mn"):
        setattr(g, bad, 1)
    elif bad == "pitch":
        g.K, g.lda = 40, 40
    elif bad == "aux_without_act":
        g.aux_out, g.ld_aux_out = keep[2].data_ptr(), 64
    s = keep[3]
    rc = _lib.load().evlm_gemm_fp8(C.byref(g), C.c_void_p(s.data_ptr()), C.c_void_p(s.data_ptr()), K._stream())
    assert rc < 0
    with pytest.raises(ValueError):
        _lib.check(rc, "evlm_gemm_fp8")
    g2, keep2 = _args(M=M)
    assert _lib.load().evlm_gemm_fp8(C.byref(g2), C.c_void_p(keep2[3].data_ptr()), C.c_void_p(keep2[3].data_ptr()), K._stream()) == 0
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------------------------------------
# Model level: the fp32 emulation is the oracle operators (tests/ref_ops.py) with every covered product replaced by quantise -> dequantise
# of both operands (the activation first rounded to bf16, as the device path hands it over).
def _qdq(t):
    q, s = fp8.quant_rows_reference(t.reshape(-1, t.shape[-1]))
    return (q.float() * s[:, None]).reshape(t.shape)


def _emulation_copy(model):
    """CPU copy of a materialised model whose covered layers take the FP8 paths (then swapped for the emulation by _emulation)."""
    emu = copy.deepcopy(model).cpu()
    for m in emu.modules():
        if fp8._weight_groups(m) is not None:
            m.evlm_fp8 = True
    return emu


class _emulation:
    def __init__(self, monkeypatch):
        self.mp = monkeypatch

    def __enter__(self):
        from efficientvlm_b200 import ops
        from oracle import xvlm_oracle as O
        from tests import ref_ops
        ref_ops.install(self.mp)

        def o_linear(x, sd, name):
            return F.linear(_qdq(x.to(bf16)), _qdq(sd[name + ".weight"]), sd.get(name + ".bias"))

        def linear_fp8(x, w, b=None, act=ACT_NONE):
            return ref_ops.linear(_qdq(x.to(bf16)), _qdq(w), b, act)
        self.mp.setattr(O, "linear", o_linear)
        self.mp.setattr(ops, "linear_fp8", linear_fp8)
        return self

    def __exit__(self, *exc):
        self.mp.undo()
        return False


def _tiny_vqa():
    from tests.helpers import Tokens, build_with_tiny_bert
    from efficientvlm_b200 import prune
    from efficientvlm_b200.vqa import EffXVLMForVQA
    g, v = load_golden("vqa_pruned_tiny"), load_golden("vqa_tiny")
    m = build_with_tiny_bert(EffXVLMForVQA, dict(v["scfg"], vision_config=dict(g["vis"]), text_encoder=None), v["bert"])
    sd = sd_from_spec(g["sd_spec"])
    sd["text_decoder.cls.predictions.decoder.weight"] = sd["text_decoder.bert.embeddings.word_embeddings.weight"]
    m.load_state_dict(sd, strict=True)
    m.eval()
    prune.materialize(m, g["zs"])
    inputs = (v["image"], Tokens(v["q_ids"], v["q_atts"]), Tokens(v["l_ids"], v["l_atts"]))
    return m.cuda(), inputs, v["k_test"]


def _baseline_vqa(batch=2):
    import bench
    from efficientvlm_b200 import prune
    from efficientvlm_b200.vqa import EffXVLMForVQA
    torch.manual_seed(42)
    m = EffXVLMForVQA(bench.vqa_cfg("student", 480, sparsity=0.35)).cuda().eval()
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():
        for la in m.l0_module.z_logas.values():
            la.copy_((torch.randn(la.shape, generator=g) * 3.0 + 1.5).cuda())
        prune.materialize(m, m.l0_module(training=False))
    from tests.helpers import Tokens
    l_ids, l_atts = bench.make_answer_list()
    image, q_ids, q_atts = bench.make_vqa_batch(batch, 480, 42)[:3]
    return m, (image, Tokens(q_ids, q_atts), Tokens(l_ids, l_atts)), 128


def _vqa_vs_emulation(monkeypatch, model, inputs, k):
    """inputs: (image, question, answer list) on the CPU."""
    emu = _emulation_copy(model)
    fp8.enable(model)
    image, q, a = inputs
    ids, probs, _ = model.fake_forward(image.cuda(), q.to("cuda"), a.to("cuda"), k=k)
    with _emulation(monkeypatch):
        wids, wprobs, _ = emu.fake_forward(image, q, a, k=k)
    ids, probs, wids, wprobs = ids.cpu(), probs.float().cpu(), wids.cpu(), wprobs.float().cpu()
    for r in range(ids.shape[0]):
        if int(ids[r, 0]) != int(wids[r, 0]):
            # a tie: the emulation ranks our answer within the tolerance of its own first choice
            hit = (wids[r] == ids[r, 0]).nonzero()
            assert hit.numel() == 1, (r, ids[r, :4], wids[r, :4])
            assert float(wprobs[r, 0] - wprobs[r, int(hit)]) <= 2e-2, (r, float(wprobs[r, 0]), float(wprobs[r, int(hit)]))
        # probabilities of the answers both rank, matched by id
        common = {int(a): float(p) for a, p in zip(wids[r], wprobs[r])}
        for a, p in zip(ids[r].tolist(), probs[r].tolist()):
            if a in common:
                assert abs(p - common[a]) <= 1e-2, (r, a, p, common[a])


def test_tiny_materialised_vqa_fp8_vs_emulation(monkeypatch):
    model, inputs, k = _tiny_vqa()
    _vqa_vs_emulation(monkeypatch, model, inputs, k)


def test_baseline_width_materialised_vqa_fp8_vs_emulation(monkeypatch):
    model, inputs, k = _baseline_vqa()
    _vqa_vs_emulation(monkeypatch, model, inputs, k)


def _tiny_captioner():
    from tests.test_caption_materialize import RAGGED_SEED, _student
    from efficientvlm_b200 import prune
    g = load_golden("caption_kd_tiny")
    model = _student(g, RAGGED_SEED).cuda().eval()
    prune.materialize(model, model.l0_module.forward(training=False))
    return model, g["image"]


@pytest.mark.parametrize("beams", [1, 3])
def test_tiny_materialised_caption_fp8_vs_emulation(monkeypatch, beams):
    """Greedy and 3-beam ids against the emulation.  Where a row differs, the emulation's own margin between its token and ours at the first
    differing position must be below 2 x 1e-2 x max|logit| (greedy), or the two sequences must score within 1e-1 under it (beams).  The
    beam bound is wider: the device's attention runs in bf16 and the emulation's in fp32, and where their activations differ by a bf16 step
    the e4m3 quantisation that follows can round one element a whole e4m3 step (2^-4 relative) apart; over the 3 x 12 decoder passes of a
    beam search that moved a length-normalised score by 5e-2 on this fixture."""
    model, image = _tiny_captioner()
    emu = _emulation_copy(model)
    fp8.enable(model)
    kw = dict(greedy=True) if beams == 1 else dict(sample=False, num_beams=3, min_length=5)
    got = model.generate(image.cuda(), max_length=12, return_ids=True, sync_free=True, **kw)[1].cpu()
    with _emulation(monkeypatch):
        want = emu.generate(image, max_length=12, return_ids=True, **kw)[1].cpu()
        got = got[:, :want.shape[1]]
        d = emu.text_decoder
        with torch.no_grad():
            enc = emu.vision_encoder(image)[0]

            def logits_after(r, prefix):
                inp = d.prepare_inputs_for_generation(prefix[None], past=None, encoder_hidden_states=enc[r:r + 1],
                                                      encoder_attention_mask=None)
                return d(**inp, return_dict=True).logits[0].double().cpu()
            pad = emu.tokenizer.pad_token_id
            prompt_len = emu.tokenizer([emu.prompt], return_tensors="pt").input_ids.shape[1] - 1
            same = 0
            for r in range(got.shape[0]):
                if torch.equal(got[r], want[r]):
                    same += 1
                    continue
                if beams == 1:
                    t = int((got[r] != want[r]).nonzero()[0])
                    lg = logits_after(r, want[r, :t])[-1]
                    a, b = int(got[r, t]), int(want[r, t])
                    assert 0 <= float(lg[b] - lg[a]) <= 2 * 1e-2 * float(lg.abs().max()), (r, t, a, b)
                else:
                    def score(seq):
                        n = len(seq)
                        while n > prompt_len and seq[n - 1] == pad:
                            n -= 1
                        logp = torch.log_softmax(logits_after(r, torch.tensor(seq[:n])), dim=-1)
                        return float(sum(logp[i - 1, seq[i]] for i in range(prompt_len, n))) / n
                    sx, sy = score(got[r].tolist()), score(want[r].tolist())
                    assert abs(sx - sy) <= 1e-1 * max(1.0, abs(sy)), (r, sx, sy)
    assert same >= 1


@pytest.mark.parametrize("beams", [1, 3])
def test_fp8_generate_captured_graph_replays_on_new_images(full_width, beams):
    """bench.py's materialised caption_infer student with FP8: generate(sync_free=True) captured once, replayed on new images, equals the
    eager FP8 ids."""
    model, images = full_width
    if not fp8.enabled(model):
        fp8.enable(model)
    kw = dict(greedy=True) if beams == 1 else dict(sample=False, num_beams=beams, min_length=5)

    def run(x):
        return model.generate(x, max_length=20, return_ids=True, sync_free=True, **kw)[1]
    image = images[0]
    images = [images[1], images[0]]
    static = image.clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            run(static)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = run(static)
    for x in images:
        static.copy_(x)
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(out.clone(), run(x.clone()))


def test_fp8_refuses_a_forward_that_needs_a_backward():
    model, image = _tiny_captioner()
    image = image.cuda()
    fp8.enable(model)
    with pytest.raises(RuntimeError, match="no backward"):
        model.vision_encoder(image)           # grad mode on, parameters require grad
    model.train()
    with pytest.raises(RuntimeError, match="no backward"):
        with torch.no_grad():
            model.vision_encoder(image)


def test_fp8_on_one_model_leaves_another_bitwise_unchanged():
    model, image = _tiny_captioner()
    image = image.cuda()
    other = copy.deepcopy(model)
    kw = dict(max_length=12, return_ids=True)
    with torch.no_grad():
        before = (other.generate(image, greedy=True, **kw)[1], other.generate(image, sample=False, num_beams=3, **kw)[1],
                  other.vision_encoder(image)[0].clone())
    fp8.enable(model)
    assert fp8.enabled(model) and not fp8.enabled(other)
    model.generate(image, greedy=True, **kw)
    with torch.no_grad():
        after = (other.generate(image, greedy=True, **kw)[1], other.generate(image, sample=False, num_beams=3, **kw)[1],
                 other.vision_encoder(image)[0])
    for a, b in zip(before, after):
        assert torch.equal(a, b)
