"""Caption generation throughput of the masked student vs the materialised (physically pruned) one.

The model and inputs are bench.py's caption_infer workload: the pruned student with synthetic log-alphas (x 3.0 + 1.5, generator seed 5),
batch 32 at 384 px, the same seeds.  The materialised arm is a second copy of that model after prune.materialize.  Each arm is ONE captured
CUDA graph of generate(sync_free=True), greedy and num_beams 3 (max_length 20, min_length 5 for beams).  In one process, after a warm-up,
the arms alternate over --batches timed batches each (host clock around work that ends in a device synchronise).  A separate
torch.profiler pass per arm splits kernel time into GEMM and the rest.  Writes <out>/caption_materialized_bench.json.

The masked greedy arm runs the decoder WITHOUT gates (the reference's greedy call passes none) while the materialised decoder carries the
folded beam-search gates, so only the beam arms are expected to pick the same ids; the JSON says whether they do.

    python scripts/caption_materialized_bench.py --out profiles/tmp
"""
import argparse
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


def n_params(model):
    return sum(p.numel() for n, p in model.named_parameters() if not n.startswith("l0_module."))


def build(args, dev):
    """bench.build_caption_infer's model, gates and image."""
    import bench
    from efficientvlm_b200.captioning import EffXVLMForCaptioning
    torch.manual_seed(42)
    cfg = dict(bench.itr_cfg("student", args.image_res, sparsity=0.35), prompt="a picture of ", max_tokens=40, label_smoothing=0.1)
    model = EffXVLMForCaptioning(cfg, tokenizer=bench.PromptTokenizer()).to(dev).eval()
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():
        for la in model.l0_module.z_logas.values():
            la.copy_((torch.randn(la.shape, generator=g) * 3.0 + 1.5).to(dev))
    return model


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


def kernel_split(fn):
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    gemm = other = 0.0
    top = {}
    for e in prof.key_averages():
        if e.device_type != torch.autograd.DeviceType.CUDA:          # kernels only (CPU ops would count their kernels again)
            continue
        t = e.device_time_total
        if t <= 0:
            continue
        if "gemm" in e.key.lower():
            gemm += t
        else:
            other += t
        top[e.key] = t
    return dict(gemm_ms=gemm / 1e3, non_gemm_ms=other / 1e3,
                top_kernels_ms={k: v / 1e3 for k, v in sorted(top.items(), key=lambda kv: -kv[1])[:12]})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--batches", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--image-res", type=int, default=384)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    from efficientvlm_b200 import prune
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    masked, materialised = build(args, dev), build(args, dev)
    with torch.no_grad():
        zs = materialised.l0_module.forward(training=False)
        kept = {k[:-2]: float((v > 0).float().mean()) for k, v in zs.items()}
    params_before = n_params(materialised)
    prune.materialize(materialised, zs)
    params_after = n_params(materialised)
    dec = materialised.text_decoder.bert.encoder.layer
    shapes = dict(decoder_self_heads=[b.attention.self.num_attention_heads for b in dec],
                  decoder_cross_heads=[b.crossattention.self.num_attention_heads if b.has_cross_attention else None for b in dec],
                  decoder_ffn_widths=[b.intermediate.dense.weight.shape[0] for b in dec],
                  vision_ffn_widths=[lay.mlp.fc1.weight.shape[0] for lay in materialised.vision_encoder.encoder.layers])
    image = torch.randn(args.batch, 3, args.image_res, args.image_res, generator=torch.Generator().manual_seed(42)).to(dev)
    decodes = {"greedy": dict(greedy=True, max_length=20), "beams3": dict(sample=False, num_beams=3, max_length=20, min_length=5)}
    arms, outs = {}, {}
    for mname, model in (("masked", masked), ("materialized", materialised)):
        for dname, kw in decodes.items():
            graph, out = capture(lambda im, m=model, kw=kw: m.generate(im, return_ids=True, sync_free=True, **kw)[1], image)
            arms[mname + "_" + dname] = graph.replay
            outs[mname + "_" + dname] = out
    for name, fn in arms.items():
        for _ in range(args.warmup):
            fn()
    torch.cuda.synchronize()
    ids_agree = {d: bool(torch.equal(outs["masked_" + d], outs["materialized_" + d])) for d in decodes}
    times = {name: [] for name in arms}
    for _ in range(args.batches):
        for name, fn in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            times[name].append((time.perf_counter() - t0) * 1e3)
    split = {name: kernel_split(fn) for name, fn in arms.items()}
    res = dict(gpu=gpu_info(), batch=args.batch, image_res=args.image_res, max_length=20, beams_min_length=5, timed_batches=args.batches,
               params_before=params_before, params_after=params_after, kept_fraction=kept, materialized_shapes=shapes,
               ids_agree_masked_vs_materialized=ids_agree, arms={})
    for name in arms:
        t = sorted(times[name])
        med = t[len(t) // 2]
        res["arms"][name] = dict(ms_per_batch_median=med, ms_per_batch_min=t[0], ms_per_batch_max=t[-1],
                                 captions_per_s=args.batch / med * 1e3, kernel_time_split=split[name])
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "caption_materialized_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: (v if k != "arms" else {a: {x: y for x, y in d.items() if x != "kernel_time_split"} for a, d in v.items()})
                      for k, v in res.items() if k != "materialized_shapes"}))
    for a, d in res["arms"].items():
        print(a, "gemm %.2f ms, non-gemm %.2f ms" % (d["kernel_time_split"]["gemm_ms"], d["kernel_time_split"]["non_gemm_ms"]))


if __name__ == "__main__":
    main()
