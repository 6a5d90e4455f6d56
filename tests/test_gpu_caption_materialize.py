"""Caption generation on the materialised (physically pruned) captioning student, on the device: the weight-stream GEMM at ragged K,
greedy and beam decoding of the tiny fixture model against the fp32 CPU reference and the gated device loop, and the full-width model's
single-token steps and captured decode graphs."""
import pytest
import torch

from tests.helpers import load_golden, reference_ops_fp32
from tests.test_caption_materialize import RAGGED_SEED, _decoder_gates, _student, _zs

pytestmark = pytest.mark.gpu


def _gemm_kernel_names(fn):
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "gemm" in e.name.lower()]


def _nan_padded(rows, cols, gen):
    """bf16 [rows, cols] view of a [rows, pitch] buffer whose pitch padding (at least 8 elements) is NaN."""
    pitch = (cols + 7) // 8 * 8 + 8
    buf = torch.full((rows, pitch), float("nan"), dtype=torch.bfloat16, device="cuda")
    view = buf[:, :cols]
    view.copy_(torch.randn(rows, cols, generator=gen).to(torch.bfloat16))
    return view


@pytest.mark.parametrize("M", [1, 17, 32])
@pytest.mark.parametrize("K", [13, 221, 769, 1851, 3072])
@pytest.mark.parametrize("N", [64, 221, 768])
def test_weight_stream_gemm_takes_any_k(M, K, N):
    """D = A B^T + bias on the small-M weight-stream kernel, element by element against an fp64 product of the same bf16 inputs.
    Bound: every product of two bf16 values is exact in fp32 (8 + 8 significant bits), so the only error is the fp32 accumulation of
    the K products, of the 2 x ks <= 16 per-slice partial sums and of the bias: at most n = K + 17 additions in any order, each of
    relative error <= 2u with u = 2^-24 (2u allows for a tensor-core adder that truncates instead of rounding).  Recursive summation
    then errs by at most n * 2u * (sum_k |a_k b_k| + |bias|) to first order."""
    from efficientvlm_b200 import kernels as K_
    gen = torch.Generator().manual_seed(1000 * M + 10 * K + N)
    A, B = _nan_padded(M, K, gen), _nan_padded(N, K, gen)
    bias = torch.randn(N, generator=gen).cuda()
    D = torch.full((M, N), float("nan"), dtype=torch.float32, device="cuda")
    names = _gemm_kernel_names(lambda: K_.gemm(A, B, D, M, N, K, bias=bias))
    assert names and all("gemm_skinny_kernel" in n for n in names), names
    a, b = A.double().cpu(), B.double().cpu()
    want = a @ b.t() + bias.double().cpu()
    bound = (K + 17) * 2.0 ** -23 * ((a.abs() @ b.abs().t()) + bias.double().cpu().abs())
    err = (D.double().cpu() - want).abs()
    assert bool(torch.isfinite(D).all())
    assert bool((err <= bound).all()), (float(err.max()), float((err / bound).max()))


def _tiny_pair():
    """(device materialised model, CPU fp32 materialised reference model, fixture)."""
    from efficientvlm_b200 import prune
    g = load_golden("caption_kd_tiny")
    model = _student(g, RAGGED_SEED).cuda().eval()
    prune.materialize(model, model.l0_module.forward(training=False))
    ref = _student(g, RAGGED_SEED)
    with reference_ops_fp32():
        prune.materialize(ref, _zs(ref))
    for a, b in zip(model.text_decoder.bert.encoder.layer, ref.text_decoder.bert.encoder.layer):
        assert a.intermediate.dense.weight.shape == b.intermediate.dense.weight.shape
        assert a.attention.self.num_attention_heads == b.attention.self.num_attention_heads
    return model, ref, g


def test_tiny_materialised_greedy_on_device_vs_fp32_reference():
    """Greedy ids, eager and sync_free, against the CPU fp32 materialised model.  At the first position where a row differs, the
    reference's own margin between its token and ours must be below 2 x 1e-2 x max|logit| (a tie inside the bf16 logit tolerance)."""
    model, ref, g = _tiny_pair()
    image = g["image"].cuda()
    kinds = (dict(greedy=True, max_length=10), dict(greedy=True, max_length=12, repetition_penalty=1.3))
    with reference_ops_fp32():
        want = [ref.generate(g["image"], return_ids=True, **kw)[1] for kw in kinds]
        ref_img = ref.vision_encoder(g["image"])[0]
        rows, flips = 0, 0
        for kw, w in zip(kinds, want):
            for sync_free in (False, True):
                ids = model.generate(image, return_ids=True, sync_free=sync_free, **kw)[1].cpu()
                assert ids.shape == w.shape
                for r in range(ids.shape[0]):
                    rows += 1
                    if torch.equal(ids[r], w[r]):
                        continue
                    flips += 1
                    t = int((ids[r] != w[r]).nonzero()[0])
                    with torch.no_grad():
                        d = ref.text_decoder
                        inp = d.prepare_inputs_for_generation(w[r, :t][None], past=None, encoder_hidden_states=ref_img[r:r + 1],
                                                              encoder_attention_mask=None)
                        logits = d(**inp, return_dict=True).logits[0, -1].float()
                    rp = kw.get("repetition_penalty", 1.0)
                    for tok in set(w[r, :t].tolist()):
                        logits[tok] = logits[tok] * rp if logits[tok] < 0 else logits[tok] / rp
                    a, b = int(ids[r, t]), int(w[r, t])
                    assert b == int(logits.argmax())
                    assert 0 <= float(logits[b] - logits[a]) <= 2 * 1e-2 * float(logits.abs().max()), (kw, r, t, a, b)
    assert flips <= rows // 2


def test_tiny_materialised_beam_search_vs_gated_device_loop():
    """Device beam search of the materialised model against the gated model's device loop: identical ids, or a sequence that scores
    within 1e-2 of the gated model's choice under the gated model."""
    model, _, g = _tiny_pair()
    gated = _student(g, RAGGED_SEED).cuda().eval()
    image = g["image"].cuda()
    zs = gated._zs(False)
    gates = _decoder_gates(zs)
    with torch.no_grad():
        enc = gated.vision_encoder(image, head_z=zs["vision_head_z"], mlp_z=zs["vision_intermediate_z"])[0]
    pad = gated.tokenizer.pad_token_id
    prompt_len = gated.tokenizer([gated.prompt], return_tensors="pt").input_ids.shape[1] - 1

    def score(item, seq):
        n = len(seq)
        while n > prompt_len and seq[n - 1] == pad:
            n -= 1
        t = torch.tensor([seq[:n]], device="cuda")
        with torch.no_grad():
            out = gated.text_decoder(input_ids=t, attention_mask=torch.ones_like(t), encoder_hidden_states=enc[item:item + 1],
                                     encoder_attention_mask=None, return_dict=True, **gates)
        logp = torch.log_softmax(out.logits[0].double(), dim=-1)
        return float(sum(logp[i - 1, seq[i]] for i in range(prompt_len, n))) / n

    same = 0
    for beams, min_length, rp in ((3, 5, 1.0), (2, 0, 1.3)):
        kw = dict(sample=False, num_beams=beams, max_length=12, min_length=min_length, repetition_penalty=rp, return_ids=True)
        w = gated.generate(image, sync_free=True, **kw)[1]
        for sync_free in (False, True):
            got = model.generate(image, sync_free=sync_free, **kw)[1]
            got = torch.cat([got, got.new_full((got.shape[0], 12 - got.shape[1]), pad)], 1)        # sync_free=False trims the padding
            for b, (x, y) in enumerate(zip(got.tolist(), w.tolist())):
                if x == y:
                    same += 1
                    continue
                sx, sy = score(b, x), score(b, y)
                assert abs(sx - sy) <= 1e-2 * max(1.0, abs(sy)), (beams, b, x, y, sx, sy)
    assert same >= 1


@pytest.fixture(scope="module")
def full_width():
    """bench.py's caption_infer student (768 wide, 12 heads, FFN 3072, 384 px, batch 32, log-alphas x 3.0 + 1.5 from seed 5),
    materialised."""
    import bench
    from efficientvlm_b200 import prune
    from efficientvlm_b200.captioning import EffXVLMForCaptioning
    torch.manual_seed(42)
    cfg = dict(bench.itr_cfg("student", 384, sparsity=0.35), prompt="a picture of ", max_tokens=40, label_smoothing=0.1)
    model = EffXVLMForCaptioning(cfg, tokenizer=bench.PromptTokenizer()).cuda().eval()
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():
        for la in model.l0_module.z_logas.values():
            la.copy_((torch.randn(la.shape, generator=g) * 3.0 + 1.5).cuda())
    prune.materialize(model, model.l0_module.forward(training=False))
    widths = [blk.intermediate.dense.weight.shape[0] for blk in model.text_decoder.bert.encoder.layer]
    assert any(w % 8 for w in widths), widths
    images = [torch.randn(32, 3, 384, 384, generator=torch.Generator().manual_seed(s)).cuda() for s in (42, 43)]
    return model, images


def test_full_width_single_token_step_runs_every_gemm_on_the_weight_stream_kernel(full_width):
    model, images = full_width
    dec = model.text_decoder
    with torch.no_grad():
        enc = model.vision_encoder(images[0])[0]
        ids = model.tokenizer([model.prompt] * 32, return_tensors="pt").input_ids.cuda()[:, :-1].contiguous()
        out = dec(**dec.prepare_inputs_for_generation(ids, past=None, encoder_hidden_states=enc, encoder_attention_mask=None),
                  return_dict=True, use_cache=True)
        nxt = torch.cat([ids, out.logits[:, -1].argmax(-1, keepdim=True)], 1)
        past = out.past_key_values

        def step():
            dec(**dec.prepare_inputs_for_generation(nxt, past=past, encoder_hidden_states=enc, encoder_attention_mask=None),
                return_dict=True, use_cache=True)
        step()
        names = _gemm_kernel_names(step)
    assert names and all("gemm_skinny_kernel" in n for n in names), sorted(set(names))


@pytest.mark.parametrize("beams", [1, 3])
def test_full_width_captured_decode_replays_on_new_images(full_width, beams):
    model, images = full_width
    kw = dict(greedy=True) if beams == 1 else dict(sample=False, num_beams=beams, min_length=5)

    def run(image):
        return model.generate(image, max_length=20, return_ids=True, sync_free=True, **kw)[1]
    static = images[0].clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            run(static)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = run(static)
    for image in (images[1], images[0]):
        static.copy_(image)
        graph.replay()
        torch.cuda.synchronize()
        replayed = out.clone()
        assert torch.equal(replayed, run(image.clone()))
