"""Retrieval and NLVR2 inference on the physically pruned students: masked against materialised against materialised + FP8.

Arms, one process, alternating over --reps timed repetitions after a warm-up (host clock around work that ends in a device synchronise):
  masked        the L0-gated student, deterministic gates applied in the GEMM / attention epilogues;
  materialised  a deep copy after prune.materialize (ragged head counts / FFN widths, no gates);
  fp8           a deep copy of the materialised model after fp8.enable.
Workloads:
  (a) ITR re-rank evaluation at the r01 configuration (scripts/itr_eval_bench.py): x-vlm-small student, 512 synthetic images at 384 px,
      2 560 captions of 40 tokens, k_test 128, log-alphas x 3.0 + 1.5 from seed 5 (bench.py's synthetic gates).  One repetition is what
      retrieval_eval.evaluation runs on the device: text and image features, similarities, both re-rank loops from an empty K|V cache.
  (b) NLVR2 prediction at bench.py's nlvr_step shape (10 pairs, 384 px, 40 tokens) in eval mode, forward(train=False); one repetition is
      --nlvr-calls calls.
A separate torch.profiler pass per arm and workload splits kernel time into GEMM, attention and the rest, with the largest kernels.
Agreement with the masked arm: candidate sets, relative difference of the scores / logits both arms produce, top-1 agreement.
Writes <out>/r03_pruned_retrieval_nlvr_bench.json.

    python scripts/pruned_retrieval_bench.py --out profiles
"""
import argparse
import copy
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "scripts")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

from fp8_infer_bench import alternate, gpu_info  # noqa: E402

ARMS = ("masked", "materialised", "fp8")


def kernel_split(fn, top=8):
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    per = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            n, c = per.get(e.name, (0.0, 0))
            per[e.name] = (n + e.device_time_total / 1000.0, c + 1)
    split = dict(gemm_ms=0.0, attention_ms=0.0, other_ms=0.0, launches=sum(c for _, c in per.values()))
    for name, (ms, _) in per.items():
        low = name.lower()
        split["gemm_ms" if "gemm" in low else "attention_ms" if "attn" in low or "attention" in low else "other_ms"] += ms
    split["top"] = [dict(name=n[:120], ms=ms, launches=c) for n, (ms, c) in sorted(per.items(), key=lambda kv: -kv[1][0])[:top]]
    return split


def seeded(model, dev):
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():
        for la in model.l0_module.z_logas.values():
            la.copy_((torch.randn(la.shape, generator=g) * 3.0 + 1.5).to(dev))
    return model


def arms_of(masked):
    from efficientvlm_b200 import fp8, prune
    mat = copy.deepcopy(masked)
    prune.materialize(mat)
    f8 = fp8.enable(copy.deepcopy(mat))
    return dict(masked=masked, materialised=mat, fp8=f8)


def n_params(m):
    return sum(p.numel() for n, p in m.named_parameters() if not n.startswith("l0_module."))


def rel(a, b):
    return float((a.float() - b.float()).norm() / b.float().norm())


def itr_workload(args, dev):
    from bench import itr_cfg
    from efficientvlm_b200 import ops
    from efficientvlm_b200 import retrieval_eval as RE
    from efficientvlm_b200.distill import EffXVLMforRetrieval
    torch.manual_seed(42)
    models = arms_of(seeded(EffXVLMforRetrieval(itr_cfg("student", args.image_res)).to(dev).eval(), dev))
    g = torch.Generator().manual_seed(5)
    n_img, n_txt, k = args.images, args.images * 5, args.k_test
    images = torch.randn(n_img, 3, args.image_res, args.image_res, generator=g).to(dev)
    text_ids = torch.randint(1000, 30522, (n_txt, 40), generator=g)
    text_ids[:, 0] = 101
    lens = torch.randint(8, 41, (n_txt,), generator=g)
    text_ids, text_atts = text_ids.to(dev), (torch.arange(40)[None, :] < lens[:, None]).long().to(dev)
    out = {}

    def run(name):
        """retrieval_eval.evaluation's device work (features, similarities, both re-rank loops from an empty K|V cache)."""
        m = models[name]
        with torch.no_grad():
            zs = m.l0_module.forward(training=False)
            if getattr(m, "gates_folded", False):
                zs = {key: None for key in zs}
            tf, te, vf, ve = [], [], [], []
            for i in range(0, n_txt, 256):
                f = m.get_text_embeds(text_ids[i:i + 256], text_atts[i:i + 256], head_z=zs["text_head_z"], mlp_z=zs["text_intermediate_z"])
                tf.append(f)
                te.append(m.get_features(text_embeds=f))
            for i in range(0, n_img, 64):
                f, _ = m.get_vision_embeds(images[i:i + 64], head_z=zs["vision_head_z"], mlp_z=zs["vision_intermediate_z"])
                vf.append(f)
                ve.append(m.get_features(image_embeds=f))
            image_feats = torch.cat(vf)
            sims = torch.cat(ve).float() @ torch.cat(te).float().t()
            ops._cross_kv.clear()
            a, b = RE.rerank_scores(m, image_feats, torch.cat(tf), text_atts, sims, k, zs["cross_head_z"], zs["cross_intermediate_z"])
            ops._cross_kv.clear()
        out[name] = (a, b, RE._fusion_kv_bytes(m, image_feats))

    fns = {name: (lambda name=name: run(name)) for name in ARMS}
    for fn in fns.values():
        fn()
    times = alternate(fns, args.reps)
    res = {}
    ma, mb, _ = out["masked"]
    for name in ARMS:
        a, b, kv = out[name]
        r = dict(time=times[name], queries_per_s=(n_img + n_txt) / (times[name]["median_ms"] / 1e3), resident_kv_gb=kv / 1e9,
                 params_m=n_params(models[name]) / 1e6, kernels=kernel_split(fns[name]))
        if name != "masked":
            agree = {}
            for what, x, y in (("i2t", a, ma), ("t2i", b, mb)):
                cx, cy = x != -100.0, y != -100.0
                both = cx & cy
                agree[what] = dict(same_candidates=float((both.sum() / cy.sum()).item()), score_rel_diff=rel(x[both], y[both]),
                                   top1_agreement=float((x.argmax(1) == y.argmax(1)).float().mean().item()))
            r["agreement_with_masked"] = agree
        res[name] = r
    with torch.no_grad():
        zs = models["masked"].l0_module.forward(training=False)
        sparsity = models["masked"].l0_module.calculate_model_size(zs)["pruned_model_sparsity"]
    return dict(workload="ITR re-rank evaluation: x-vlm-small student, %d images at %d px, %d captions of 40 tokens, k_test %d; one repetition = "
                         "features + similarities + both re-rank loops from an empty K|V cache" % (n_img, args.image_res, n_txt, k),
                pruned_model_sparsity=float(sparsity), arms=res)


def nlvr_workload(args, dev):
    from bench import WORKLOADS, itr_cfg, make_nlvr_batch
    from efficientvlm_b200.nlvr import EffXVLMForNLVR
    torch.manual_seed(42)
    models = arms_of(seeded(EffXVLMForNLVR(itr_cfg("student", args.image_res)).to(dev).eval(), dev))
    B = WORKLOADS["nlvr_step"][2]
    image, text_ids, text_atts, targets = (t.to(dev) for t in make_nlvr_batch(B, args.image_res, 42))
    out = {}

    def run(name):
        with torch.no_grad():
            for _ in range(args.nlvr_calls):
                out[name] = models[name](image, text_ids, text_atts, targets=targets, train=False)

    fns = {name: (lambda name=name: run(name)) for name in ARMS}
    for fn in fns.values():
        fn()
    times = alternate(fns, args.reps)
    res = {}
    for name in ARMS:
        per_call = times[name]["median_ms"] / args.nlvr_calls
        r = dict(time=times[name], ms_per_call=per_call, samples_per_s=B / (per_call / 1e3), params_m=n_params(models[name]) / 1e6)
        with torch.no_grad():
            r["kernels"] = kernel_split(lambda name=name: models[name](image, text_ids, text_atts, targets=targets, train=False))
        if name != "masked":
            r["agreement_with_masked"] = dict(logit_rel_diff=rel(out[name], out["masked"]),
                                              top1_agreement=float((out[name].argmax(1) == out["masked"].argmax(1)).float().mean().item()))
        res[name] = r
    return dict(workload="NLVR2 prediction: x-vlm-small student, forward(train=False) on %d pairs (two %d px images each, 40 tokens); "
                         "one repetition = %d calls" % (B, args.image_res, args.nlvr_calls), arms=res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles")
    ap.add_argument("--images", type=int, default=512)
    ap.add_argument("--k-test", type=int, default=128)
    ap.add_argument("--image-res", type=int, default=384)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--nlvr-calls", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("pruned_retrieval_bench.py measures the B200 path and needs a CUDA device")
    dev = torch.device("cuda:0")
    result = dict(gpu=gpu_info(), torch=torch.__version__, reps=args.reps,
                  itr=itr_workload(args, dev), nlvr=nlvr_workload(args, dev))
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "r03_pruned_retrieval_nlvr_bench.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    summary = {w: {a: (v["time"]["median_ms"], v.get("agreement_with_masked")) for a, v in result[w]["arms"].items()} for w in ("itr", "nlvr")}
    print(json.dumps(dict(gpu=result["gpu"], summary=summary)))


if __name__ == "__main__":
    main()
