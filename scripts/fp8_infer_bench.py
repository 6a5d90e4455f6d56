"""FP8 inference against bf16 on the materialised (physically pruned) students: time per batch, GEMM share, GEMM rates, agreement.

Workloads are bench.py's: vqa_infer --materialize (batch 24, 480 px, fake_forward over the 3129-answer list with k_test 128, synthetic
log-alphas x 3.0 + 1.5 from seed 5) and caption_infer on the materialised captioner (batch 32, 384 px, greedy and num_beams 3 with
max_length 20 / min_length 5 for beams, one captured graph of generate(sync_free=True) per arm).  The FP8 arm is a deep copy of the bf16
model after fp8.enable.  In one process, after a warm-up, the arms alternate over --batches timed batches (host clock around work that
ends in a device synchronise).  A separate torch.profiler pass per arm splits kernel time into GEMM (kernels whose name contains "gemm")
and the rest; the FP8 arm's activation quantisation launches are listed on their own.  The vocabulary product (12288 x 30522 x 768) and
two projections are timed alone with CUDA events (operands larger than L2 are not rotated: the rates are for warm operands).
Agreement with bf16: fraction of identical top-1 answers, largest change of a ranked answer's probability, fraction of caption rows
with identical ids.  Writes <out>/fp8_infer_bench.json.

    python scripts/fp8_infer_bench.py --out profiles/tmp
"""
import argparse
import copy
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        out = ""
    return out or "unknown"


def stats(ms):
    ms = sorted(ms)
    return dict(median_ms=ms[len(ms) // 2], min_ms=ms[0], max_ms=ms[-1], n=len(ms))


def kernel_split(fn):
    """(GEMM kernel ms, other kernel ms, quantise kernel ms) of one call of fn."""
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    gemm = other = quant = 0.0
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        t = e.device_time_total / 1000.0 if hasattr(e, "device_time_total") else e.cuda_time_total / 1000.0
        if "gemm" in e.name.lower():
            gemm += t
        else:
            other += t
            if "quant_rows" in e.name:
                quant += t
    return dict(gemm_ms=gemm, other_ms=other, quant_ms=quant)


def alternate(fns, batches):
    times = {k: [] for k in fns}
    for _ in range(batches):
        for k, fn in fns.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            times[k].append((time.perf_counter() - t0) * 1e3)
    return {k: stats(v) for k, v in times.items()}


def materialised(model):
    from efficientvlm_b200 import prune
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():
        for la in model.l0_module.z_logas.values():
            la.copy_((torch.randn(la.shape, generator=g) * 3.0 + 1.5).to(la.device))
        prune.materialize(model, model.l0_module(training=False))
    return model


def vqa_arm(args, dev, res):
    import bench
    from efficientvlm_b200 import fp8
    from efficientvlm_b200.vqa import EffXVLMForVQA
    torch.manual_seed(42)
    bf = materialised(EffXVLMForVQA(bench.vqa_cfg("student", 480, sparsity=0.35)).to(dev).eval())
    f8 = fp8.enable(copy.deepcopy(bf))
    l_ids, l_atts = (t.to(dev) for t in bench.make_answer_list())
    image, q_ids, q_atts = (t.to(dev) for t in bench.make_vqa_batch(24, 480, 42)[:3])
    q, a = bench.Tok(q_ids, q_atts), bench.Tok(l_ids, l_atts)
    out = {}

    def run(name, m):
        def fn():
            with torch.no_grad():
                out[name] = m.fake_forward(image, q, a, k=128)[:2]
        return fn
    fns = {"bf16": run("bf16", bf), "fp8": run("fp8", f8)}
    for fn in fns.values():
        fn()
        fn()
    res["vqa"] = dict(time=alternate(fns, args.batches), kernels={k: kernel_split(fn) for k, fn in fns.items()})
    (bi, bp), (fi, fp) = out["bf16"], out["fp8"]
    top1 = float((bi[:, 0] == fi[:, 0]).float().mean())
    dmax = 0.0
    for r in range(bi.shape[0]):
        pb = dict(zip(bi[r].tolist(), bp[r].float().tolist()))
        for i, p in zip(fi[r].tolist(), fp[r].float().tolist()):
            if i in pb:
                dmax = max(dmax, abs(p - pb[i]))
    res["vqa"]["agreement"] = dict(top1_equal_fraction=top1, max_abs_prob_change=dmax)
    del bf, f8
    torch.cuda.empty_cache()


def capture(fn, image):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            fn(image)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = fn(image)
    return graph, out


def caption_arm(args, dev, res):
    import bench
    from efficientvlm_b200 import fp8
    from efficientvlm_b200.captioning import EffXVLMForCaptioning
    torch.manual_seed(42)
    cfg = dict(bench.itr_cfg("student", 384, sparsity=0.35), prompt="a picture of ", max_tokens=40, label_smoothing=0.1)
    bf = materialised(EffXVLMForCaptioning(cfg, tokenizer=bench.PromptTokenizer()).to(dev).eval())
    f8 = fp8.enable(copy.deepcopy(bf))
    image = torch.randn(32, 3, 384, 384, generator=torch.Generator().manual_seed(42)).to(dev)
    for beams in (1, 3):
        kw = dict(greedy=True) if beams == 1 else dict(sample=False, num_beams=3, min_length=5)
        graphs, outs = {}, {}
        for name, m in (("bf16", bf), ("fp8", f8)):
            static = image.clone()
            graphs[name], outs[name] = capture(lambda x, m=m: m.generate(x, max_length=20, return_ids=True, sync_free=True, **kw)[1], static)
        fns = {k: g.replay for k, g in graphs.items()}
        for fn in fns.values():
            fn()
        key = "caption_greedy" if beams == 1 else "caption_beams3"
        res[key] = dict(time=alternate(fns, args.batches), kernels={k: kernel_split(fn) for k, fn in fns.items()})
        res[key]["agreement"] = dict(identical_rows_fraction=float((outs["bf16"] == outs["fp8"]).all(1).float().mean()))
        del graphs, outs
    del bf, f8
    torch.cuda.empty_cache()


def gemm_rates(dev, res, iters=50):
    from efficientvlm_b200 import kernels as K
    out = {}
    for name, (M, N, Kd) in {"vocab_12288x30522x768": (12288, 30522, 768), "proj_12288x3072x768": (12288, 3072, 768),
                             "proj_12288x768x3072": (12288, 768, 3072)}.items():
        a = (torch.randn(M, Kd, device=dev) * 0.5).to(torch.bfloat16)
        w = torch.randn(N, Kd, device=dev) * 0.05
        w16 = w.to(torch.bfloat16)
        D = torch.empty(M, (N + 3) // 4 * 4, device=dev)[:, :N]
        qa, sa = K.quant_rows_e4m3(a)
        qw, sw = K.quant_rows_e4m3(w)
        arms = {"bf16": lambda: K.gemm(a, w16, D, M, N, Kd), "fp8": lambda: K.gemm_fp8(qa, sa, qw, sw, D, M, N, Kd),
                "fp8_with_activation_quant": lambda: K.gemm_fp8(*K.quant_rows_e4m3(a), qw, sw, D, M, N, Kd)}
        row = {}
        for arm, fn in arms.items():
            for _ in range(5):
                fn()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                fn()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / iters
            row[arm] = dict(ms=ms, tflops=2.0 * M * N * Kd / ms / 1e9)
        out[name] = row
    res["gemm"] = out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--batches", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("fp8_infer_bench.py measures the GPU: no CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = dict(gpu=gpu_info(), batches=args.batches)
    gemm_rates(dev, res)
    vqa_arm(args, dev, res)
    caption_arm(args, dev, res)
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "fp8_infer_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
