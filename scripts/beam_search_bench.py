"""Beam-search captioning throughput: the host loop vs the device loop (eager) vs one captured CUDA graph of generate(sync_free=True).

The model and inputs are bench.py's caption_infer workload (pruned student, batch 32 at 384 px, the same seeds); the decode is the
reference evaluation's (num_beams 3, max_length 20, min_length 5).  In one process, after a warm-up, the three arms alternate over
--batches timed batches each (host clock around work that ends in a device synchronise).  A separate torch.profiler pass per arm splits
kernel time into GEMM and non-GEMM.  All arms must produce identical ids.  Writes <out>/beam_search_bench.json.

    python scripts/beam_search_bench.py --out profiles/tmp
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


def power_limit():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                              timeout=30).stdout.strip() or "unknown"
    except Exception:
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--batches", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--image-res", type=int, default=384)
    ap.add_argument("--beams", type=int, default=3)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    import bench
    from efficientvlm_b200 import eff_bert as EB
    from efficientvlm_b200 import kernels as K
    from efficientvlm_b200.captioning import EffXVLMForCaptioning
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    torch.manual_seed(42)                                          # bench.build_caption_infer's model, gates and image
    cfg = dict(bench.itr_cfg("student", args.image_res, sparsity=0.35), prompt="a picture of ", max_tokens=40, label_smoothing=0.1)
    model = EffXVLMForCaptioning(cfg, tokenizer=bench.PromptTokenizer()).to(dev).eval()
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():
        for la in model.l0_module.z_logas.values():
            la.copy_((torch.randn(la.shape, generator=g) * 3.0 + 1.5).to(dev))
    image = torch.randn(args.batch, 3, args.image_res, args.image_res, generator=torch.Generator().manual_seed(42)).to(dev)
    kw = dict(sample=False, num_beams=args.beams, max_length=20, min_length=5, return_ids=True)

    def host():
        EB.BEAM_SEARCH_ON_DEVICE = False
        try:
            return model.generate(image, **kw)[1]
        finally:
            EB.BEAM_SEARCH_ON_DEVICE = True

    def device():
        return model.generate(image, **kw)[1]

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            model.generate(image, sync_free=True, **kw)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    n0 = K.launch_count()
    with torch.cuda.graph(graph):
        graph_ids = model.generate(image, sync_free=True, **kw)[1]
    graph_launches = K.launch_count() - n0

    def graphed():
        graph.replay()
        return graph_ids

    arms = {"host_loop": host, "device_loop_eager": device, "device_loop_graph": graphed}
    ids = {}
    launches = {"device_loop_graph": graph_launches}
    for name, fn in arms.items():
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        n0 = K.launch_count()
        ids[name] = fn().clone()
        torch.cuda.synchronize()
        if name != "device_loop_graph":
            launches[name] = K.launch_count() - n0
    ref = ids["host_loop"]
    n = ref.shape[1]
    assert torch.equal(ids["device_loop_eager"], ref), "device loop ids differ from the host loop"
    assert torch.equal(ids["device_loop_graph"][:, :n], ref), "graph ids differ from the host loop"
    assert bool((ids["device_loop_graph"][:, n:] == 0).all())
    times = {name: [] for name in arms}
    for _ in range(args.batches):
        for name, fn in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            times[name].append((time.perf_counter() - t0) * 1e3)
    split = {}
    for name, fn in arms.items():
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
        split[name] = dict(gemm_ms=gemm / 1e3, non_gemm_ms=other / 1e3,
                           top_kernels_ms={k: v / 1e3 for k, v in sorted(top.items(), key=lambda kv: -kv[1])[:12]})
    res = dict(gpu=torch.cuda.get_device_name(0), power_limit=power_limit(), batch=args.batch, image_res=args.image_res, num_beams=args.beams,
               max_length=20, min_length=5, timed_batches=args.batches, ids_identical=True, arms={})
    for name in arms:
        t = sorted(times[name])
        med = t[len(t) // 2]
        res["arms"][name] = dict(ms_per_batch_median=med, ms_per_batch_min=t[0], ms_per_batch_max=t[-1],
                                 captions_per_s=args.batch / med * 1e3, evlm_launches_per_batch=launches[name],
                                 kernel_time_split=split[name])
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "beam_search_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: (v if k != "arms" else {a: {x: y for x, y in d.items() if x != "kernel_time_split"} for a, d in v.items()})
                      for k, v in res.items()}))
    for a, d in res["arms"].items():
        print(a, "gemm %.2f ms, non-gemm %.2f ms" % (d["kernel_time_split"]["gemm_ms"], d["kernel_time_split"]["non_gemm_ms"]))


if __name__ == "__main__":
    main()
