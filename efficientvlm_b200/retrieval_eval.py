"""ITR re-rank evaluation (SURVEY §8f row 4): `evaluation` / `itm_eval` of `Eff_Retrieval.py:216-378`, same signatures and results.

The reference scores one query at a time: per image it repeats the image k_test times and runs the fusion encoder on its k_test best
texts (`Eff_Retrieval.py:277-291`), per text it gathers the k_test best images (`:300-314`) — every one of the 2·k_test·N candidate rows
re-projects the K|V of its 577-token image in every fusion layer (about half of the FLOPs of a row: the text side is 40 tokens) and runs
its cross-attention as a 40-row problem.

Here, B200-first:
  * the per-layer cross-attention K|V of EVERY test image is projected once and stays resident in HBM (COCO-5k at 384 px: 5 000 x 577
    tokens x 1 536 bf16 = 8.9 GB per fusion layer, three layers on the student — the 180 GB part holds it); the fusion passes only
    index it (`get_cross_embeds(..., image_index=)`, `ops._cross_kv`).  When it does not fit `kv_cache_bytes`, a pass projects the K|V
    of the images it touches (once per image and pass);
  * both directions are sets of (image, text) pairs, so both run IMAGE-major: pairs sorted by image, `group_rows` text rows of one image
    form one cross-attention problem (`ops.UniformGroups(.., items=)`: full 128-row tiles, the image's K|V read once per tile), and a
    fusion pass takes ~16k text rows instead of k_test.

Scores, the -100 fill, the `size // world + 1` row split and the SUM all-reduce are the reference's.  Nothing here has a CPU path: the
model calls go through the CUDA extension like every other forward.
"""
import numpy as np
import torch

from . import ops


def _is_dist():
    return torch.distributed.is_available() and torch.distributed.is_initialized()


def _rank_world():
    if _is_dist():
        return torch.distributed.get_rank(), torch.distributed.get_world_size()
    return 0, 1


def _fusion_kv_bytes(model, image_feats):
    """bf16 K|V of all images in every cross-attention layer + the bf16 copy of the image tokens."""
    bert = model._bert()
    n_tok = image_feats.shape[0] * image_feats.shape[1]
    total = n_tok * image_feats.shape[2] * 2
    for layer in bert.encoder.layer:
        if getattr(layer, "has_cross_attention", False):
            total += n_tok * 2 * layer.crossattention.self.key.weight.shape[0] * 2
    return total


@torch.no_grad()
def rerank_scores(model, image_feats, text_feats, text_atts, sims_matrix, k_test, cross_head_z=None, cross_mlp_z=None, queries_per_pass=None,
                  kv_cache_bytes=64 << 30, rank=None, world=None, share_image_kv=True, group_rows=16):
    """The two re-rank loops of `Eff_Retrieval.py:265-314` for this rank's rows.  Returns (score_matrix_i2t [n_img, n_txt],
    score_matrix_t2i [n_txt, n_img]), -100 where a pair was not scored (before any cross-rank reduction).

    Both directions score (image, text) PAIRS, so both run image-major: the pairs are sorted by image and cut into groups of `group_rows`
    text rows that share one image (the last group of an image is padded by repeating its last pair); a group is ONE
    cross-attention problem with group_rows * L query rows against the image's resident K|V (`ops.UniformGroups(.., items=)`), i.e. full
    128-row tensor-core tiles instead of one 40-row tile per pair, and a fusion pass takes `queries_per_pass * k_test` pairs.
    `share_image_kv=False` keeps the reference's pass structure instead (query-major, every candidate row gets its own copy of the
    image tokens: `.repeat(k_test, 1, 1)` / `image_feats[topk_idx]`): same scores, kept for A/B timing (scripts/itr_eval_bench.py)."""
    if rank is None or world is None:
        rank, world = _rank_world()
    dev = image_feats.device
    n_img, n_txt = sims_matrix.shape
    L = text_feats.shape[1]
    if queries_per_pass is None:
        queries_per_pass = max(1, 16384 // max(1, k_test * L))             # ~16k text rows per fusion pass
    Q = int(queries_per_pass)
    image_feats = image_feats.contiguous()
    resident = share_image_kv and _fusion_kv_bytes(model, image_feats) <= kv_cache_bytes

    def itm_score(out):
        return model.itm_head(out[:, 0, :])[:, 1].float()

    def fusion(img, index, txt_rows):
        return itm_score(model.get_cross_embeds(image_embeds=img, image_atts=None, text_embeds=text_feats.index_select(0, txt_rows),
                                                text_atts=text_atts.index_select(0, txt_rows), head_z=cross_head_z, head_layer_z=None,
                                                mlp_z=cross_mlp_z, image_index=index))

    def score_pairs(img_ids, txt_ids):
        """ITM scores of the pairs (img_ids[p], txt_ids[p]), image-major."""
        P, g = img_ids.numel(), max(1, int(group_rows))
        out = torch.empty(P, device=dev)
        if P == 0:
            return out
        img_sorted, order = torch.sort(img_ids, stable=True)
        counts = torch.bincount(img_sorted, minlength=n_img)
        n_groups = (counts + g - 1) // g                                    # groups per image
        first_group = torch.cumsum(n_groups, 0) - n_groups
        first_pair = torch.cumsum(counts, 0) - counts
        group_img = torch.repeat_interleave(torch.arange(n_img, device=dev), n_groups)            # [G] image of every group
        G = group_img.numel()
        # slot s of group j holds sorted pair  first_pair[img] + (j - first_group[img]) * g + s, clamped to the image's last pair (padding)
        base = first_pair[group_img] + (torch.arange(G, device=dev) - first_group[group_img]) * g
        slot = base[:, None] + torch.arange(g, device=dev)[None, :]
        last = (first_pair + counts - 1)[group_img][:, None]
        slot = torch.minimum(slot, last)                                       # [G, g] indices into the sorted pair list
        groups_per_pass = max(1, (Q * k_test) // g)
        for a in range(0, G, groups_per_pass):
            b = min(G, a + groups_per_pass)
            sl = slot[a:b].reshape(-1)
            txt_rows = txt_ids[order[sl]]
            if resident:   # the same image_feats object every pass: its bf16 copy and per-layer K|V are projected once and stay cached
                items = group_img[a:b].to(torch.int32)
                sc = fusion(image_feats, ops.UniformGroups(g, items.repeat_interleave(g), items=items), txt_rows)
            else:          # the pass's images only: K|V projected once per (image, pass)
                uniq, inv = torch.unique_consecutive(group_img[a:b], return_inverse=True)
                items = inv.to(torch.int32)
                sc = fusion(image_feats.index_select(0, uniq), ops.UniformGroups(g, items.repeat_interleave(g), items=items), txt_rows)
            out[order[sl]] = sc      # a padding slot repeats its image's last pair: same rows, same kernels, the same value written twice
        return out

    # ---- image -> text (Eff_Retrieval.py:265-291) ----
    score_i2t = torch.full((n_img, n_txt), -100.0, device=dev)
    step = n_img // world + 1
    start, end = rank * step, min(n_img, rank * step + step)
    if share_image_kv and end > start:
        topk_idx = sims_matrix[start:end].topk(k=k_test, dim=1)[1]            # [rows, k] text ids
        img_ids = torch.arange(start, end, device=dev).repeat_interleave(k_test)
        score_i2t[start:end].scatter_(1, topk_idx, score_pairs(img_ids, topk_idx.reshape(-1)).view(end - start, k_test))
    else:
        for a in range(start, end, Q):
            b = min(end, a + Q)
            topk_idx = sims_matrix[a:b].topk(k=k_test, dim=1)[1]
            sc = fusion(image_feats[a:b].repeat_interleave(k_test, 0), None, topk_idx.reshape(-1))
            score_i2t[a:b].scatter_(1, topk_idx, sc.view(b - a, k_test))
    # ---- text -> image (Eff_Retrieval.py:293-314) ----
    score_t2i = torch.full((n_txt, n_img), -100.0, device=dev)
    sims_t = sims_matrix.t()
    step = n_txt // world + 1
    start, end = rank * step, min(n_txt, rank * step + step)
    if share_image_kv and end > start:
        topk_idx = sims_t[start:end].topk(k=k_test, dim=1)[1]                 # [rows, k] image ids
        txt_ids = torch.arange(start, end, device=dev).repeat_interleave(k_test)
        score_t2i[start:end].scatter_(1, topk_idx, score_pairs(topk_idx.reshape(-1), txt_ids).view(end - start, k_test))
    else:
        for a in range(start, end, Q):
            b = min(end, a + Q)
            topk_idx = sims_t[a:b].topk(k=k_test, dim=1)[1]
            txt_rows = torch.arange(a, b, device=dev).repeat_interleave(k_test)
            sc = fusion(image_feats.index_select(0, topk_idx.reshape(-1)), None, txt_rows)
            score_t2i[a:b].scatter_(1, topk_idx, sc.view(b - a, k_test))
    return score_i2t, score_t2i


@torch.no_grad()
def evaluation(model, data_loader, tokenizer, device, config, queries_per_pass=None, kv_cache_bytes=64 << 30, details=None, group_rows=16):
    """`Eff_Retrieval.py:216-332`.  Returns (score_matrix_i2t ndarray, score_matrix_t2i ndarray, pruned_model_sparsity).
    `details` (optional dict) receives the intermediate tensors (sims_matrix, image_feats, text_feats, text_atts, zs).
    On a materialised model (prune.materialize: its gates live in the pruned weights) every encoder and the re-rank run without gates;
    the sparsity is still that of the deterministic masks, which materialize leaves in `l0_module`."""
    model.eval()
    texts = data_loader.dataset.text
    num_text = len(texts)
    text_bs = config["batch_size_test_text"]
    zs = model.l0_module.forward(training=False)
    pruned_model_size_info = model.l0_module.calculate_model_size(zs)
    if getattr(model, "gates_folded", False):
        zs = {k: None for k in zs}
    text_feats, text_embeds, text_atts = [], [], []
    for i in range(0, num_text, text_bs):
        text_input = tokenizer(texts[i:min(num_text, i + text_bs)], padding="max_length", truncation=True, max_length=config["max_tokens"],
                               return_tensors="pt").to(device)
        text_feat = model.get_text_embeds(text_input.input_ids, text_input.attention_mask, head_z=zs["text_head_z"], head_layer_z=None,
                                          mlp_z=zs["text_intermediate_z"])
        text_embeds.append(model.get_features(text_embeds=text_feat))
        text_feats.append(text_feat)
        text_atts.append(text_input.attention_mask)
    text_embeds, text_feats, text_atts = torch.cat(text_embeds, 0), torch.cat(text_feats, 0), torch.cat(text_atts, 0)
    image_feats, image_embeds = [], []
    for image, _img_id in data_loader:
        image_feat, _ = model.get_vision_embeds(image.to(device), head_z=zs["vision_head_z"], head_layer_z=None, mlp_z=zs["vision_intermediate_z"])
        image_embeds.append(model.get_features(image_embeds=image_feat))
        image_feats.append(image_feat)
    image_feats, image_embeds = torch.cat(image_feats, 0), torch.cat(image_embeds, 0)
    sims_matrix = image_embeds.float() @ text_embeds.float().t()
    if details is not None:
        details.update(sims_matrix=sims_matrix, image_feats=image_feats, text_feats=text_feats, text_atts=text_atts, zs=zs)
    score_i2t, score_t2i = rerank_scores(model, image_feats, text_feats, text_atts, sims_matrix, config["k_test"], zs["cross_head_z"],
                                         zs["cross_intermediate_z"], queries_per_pass, kv_cache_bytes, group_rows=group_rows)
    ops._cross_kv.clear()          # the resident per-layer K|V of the gallery (GBs at COCO-5k scale) is not needed past this point
    if _is_dist() and torch.distributed.get_world_size() > 1:
        torch.distributed.barrier()
        torch.distributed.all_reduce(score_i2t, op=torch.distributed.ReduceOp.SUM)
        torch.distributed.all_reduce(score_t2i, op=torch.distributed.ReduceOp.SUM)
    return score_i2t.cpu().numpy(), score_t2i.cpu().numpy(), pruned_model_size_info["pruned_model_sparsity"]


def itm_eval(scores_i2t, scores_t2i, txt2img, img2txt):
    """`Eff_Retrieval.py:335-378`: recall@1/5/10 of both directions from the score matrices (host side, numpy like the reference)."""
    def recalls(ranks):
        return tuple(100.0 * float(np.count_nonzero(ranks < n)) / len(ranks) for n in (1, 5, 10))
    order = np.argsort(scores_i2t, axis=1)[:, ::-1]
    position = np.empty_like(order)
    np.put_along_axis(position, order, np.arange(order.shape[1])[None, :], axis=1)      # position[i, t] = rank of text t for image i
    ranks = np.array([min(position[i, t] for t in img2txt[i]) for i in range(scores_i2t.shape[0])], dtype=np.float64)
    tr1, tr5, tr10 = recalls(ranks)
    order = np.argsort(scores_t2i, axis=1)[:, ::-1]
    ranks = np.array([np.where(order[t] == txt2img[t])[0][0] for t in range(scores_t2i.shape[0])], dtype=np.float64)
    ir1, ir5, ir10 = recalls(ranks)
    tr_mean, ir_mean = (tr1 + tr5 + tr10) / 3, (ir1 + ir5 + ir10) / 3
    return {"txt_r1": tr1, "txt_r5": tr5, "txt_r10": tr10, "txt_r_mean": tr_mean, "img_r1": ir1, "img_r5": ir5, "img_r10": ir10,
            "img_r_mean": ir_mean, "r_mean": (tr_mean + ir_mean) / 2}
