"""N>1 parity ON THE DEVICE (VERDICT r1 item 6 / SURVEY 4 "DDP pin"): two processes, two GPUs, NCCL.

What the reference does at N>1 (accelerators/apex_ddp_accelerator.py:74-101, efficient_models/xvlm.py:54-74): parameters broadcast from
rank 0, every rank runs the step on its shard, the ITC features are all_gather'ed (backward = LOCAL slice, quirk Q3) so every rank
computes the SAME full-batch ITC loss, gradients are mean-allreduced, every rank applies the same update.

Checked here on the CUDA product over NCCL:
  1. broadcast: parameters bit-identical on both ranks even though rank 1 started from different weights;
  2. the ITC loss of every rank == the oracle's contrastive loss on the concatenated batch's features (fp32), and == the 1-process
     run on the concatenated batch; the batch-mean terms (ITM, MLM, every KD term) of the 1-process run on the concatenated batch ==
     the mean over ranks of the per-rank terms;
  3. the reduced gradient arena == the mean over ranks of the local arenas (the NCCL AVG over the flat arenas did what DDP does) AND
     == the mean over shards of single-process per-shard gradients in which the gathered features of the OTHER shard are constants
     (Q3: no gradient crosses ranks) — i.e. the two-GPU step is the reference's DDP step, not merely self-consistent;
  4. after `FlatAdamW.step()` the parameters are bit-identical across ranks;
  5. the overlapped exchange (`FlatAdamW.enable_overlap`: the non-vision part of every arena leaves on a side stream under the vision
     tower's backward) produces the blocking exchange's gradients.
Skipped with fewer than two GPUs (the driver's round-end `-m gpu` box has one; `gpurun --gpus 2` runs it: profiles/r02_ddp_parity_2gpu.log).
"""
import os
import socket
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _batch(world, B, L=9):
    g = torch.Generator().manual_seed(31)
    n = world * B
    image = torch.randn(n, 3, 32, 32, generator=g)
    text_ids = torch.randint(1, 211, (n, L), generator=g)
    text_atts = torch.ones(n, L, dtype=torch.long)
    text_atts[1, 6:] = 0
    text_atts[B + 2, 5:] = 0
    masked_pos = torch.stack([torch.randperm(L - 1, generator=g)[:3].sort().values + 1 for _ in range(n)])
    masked_ids = torch.gather(text_ids, 1, masked_pos)           # no ignored labels: equal counts per shard, so means compose
    text_ids_masked = text_ids.clone().scatter_(1, masked_pos, 103)
    return [image, text_ids, text_atts, text_ids_masked, masked_pos, masked_ids]


def _worker(rank, world, port, q):
    try:
        sys.path.insert(0, ROOT)
        os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
        torch.cuda.set_device(rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
        from efficientvlm_b200 import xvlm as X
        from efficientvlm_b200.distill import gd_kd_losses, gd_loss
        from efficientvlm_b200.optim import create_optimizer
        from oracle import xvlm_oracle as O
        from tests.helpers import rel_err
        from tests.test_gpu_models import _tiny_gd_models
        B = 4
        student, teacher = _tiny_gd_models()
        student.cuda()
        teacher.cuda()
        if rank == 1:                                   # rank 1 starts elsewhere: the broadcast has to bring it back
            with torch.no_grad():
                for p in student.parameters():
                    p.add_(0.01)
        opt = create_optimizer(dict(lr=1e-3, weight_decay=0.01, lr_mult=1), student, clip_grad_norm=1.0)
        opt.broadcast_parameters(0)

        def gathered(t):
            out = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(out, t.contiguous())
            return out
        for gp in opt.param_groups:
            both = gathered(gp["p"])
            assert torch.equal(both[0], both[1]), "1. parameters identical after broadcast"
        full = [t.cuda() for t in _batch(world, B)]
        shard = [t[rank * B:(rank + 1) * B] for t in full]
        local_negs = (torch.roll(torch.arange(B), 1).cuda(), torch.roll(torch.arange(B), -1).cuda())
        student.sample_itm_negatives = teacher.sample_itm_negatives = lambda image_feat, text_feat, idx=None: local_negs
        feats = {}
        orig_itc = student.get_contrastive_loss

        def recording_itc(image_feat, text_feat, idx=None):
            feats["i"], feats["t"] = image_feat.detach().clone(), text_feat.detach().clone()
            return orig_itc(image_feat, text_feat, idx=idx)
        student.get_contrastive_loss = recording_itc
        so = student(*shard, output_attentions=True, output_hidden_states=True)
        with torch.no_grad():
            to = teacher(*shard, output_attentions=True, output_hidden_states=True)
        total, parts = gd_loss(so, to, 1.0)
        kd = gd_kd_losses(so, to, 1.0)
        opt.zero_grad()
        total.backward()
        # 2. ITC: same value on both ranks, equal to the oracle on the gathered features
        fi, ft = torch.cat(gathered(feats["i"])), torch.cat(gathered(feats["t"]))
        ref_itc = O.contrastive_loss(fi.cpu(), ft.cpu(), student.temp.detach().cpu())
        assert abs(float(so["loss"]["loss_itc"]) - float(ref_itc)) < 1e-4 * abs(float(ref_itc)), (float(so["loss"]["loss_itc"]), float(ref_itc))
        itcs = gathered(so["loss"]["loss_itc"].detach().reshape(1))
        assert torch.equal(itcs[0], itcs[1])
        # 3a. reduced arena == mean over ranks of the local arenas
        local = [gp["g"].clone() for gp in opt.param_groups]
        opt.allreduce_gradients()
        for gp, l in zip(opt.param_groups, local):
            both = gathered(l)
            assert rel_err(gp["g"], (both[0] + both[1]) / world) < 1e-6, "3a. NCCL AVG over the flat arena"
        reduced = [gp["g"].clone() for gp in opt.param_groups]
        mean_terms = {}
        for k in ("loss_itm", "loss_mlm"):
            both = gathered(so["loss"][k].detach().reshape(1))
            mean_terms[k] = float((both[0] + both[1]) / world)
        for k, v in kd.items():
            both = gathered(v.detach().reshape(1))
            mean_terms[k] = float((both[0] + both[1]) / world)
        # 4. identical parameters after the update
        opt.step(allreduce=False)
        for gp in opt.param_groups:
            both = gathered(gp["p"])
            assert torch.equal(both[0], both[1]), "4. parameters identical after the step"
        other_i, other_t = fi, ft
        dist.barrier()
        # 5. overlapped exchange (FlatAdamW.enable_overlap): the part of every arena outside the vision tower is all-reduced on a side
        #    stream as soon as autograd reaches the vision tower's output; the result must be the blocking exchange's
        student3, teacher3 = _tiny_gd_models()
        student3.cuda()
        teacher3.cuda()
        opt3 = create_optimizer(dict(lr=1e-3, weight_decay=0.01, lr_mult=1), student3, clip_grad_norm=1.0)
        student3.sample_itm_negatives = teacher3.sample_itm_negatives = lambda image_feat, text_feat, idx=None: local_negs
        opt3.enable_overlap(student3, "vision_encoder.")
        splits = [(gp["split"], gp["size"]) for gp in opt3.param_groups]
        assert any(0 < a < b for a, b in splits), splits
        so4 = student3(*shard, output_attentions=True, output_hidden_states=True)
        with torch.no_grad():
            to4 = teacher3(*shard, output_attentions=True, output_hidden_states=True)
        opt3.zero_grad()
        gd_loss(so4, to4, 1.0)[0].backward()
        assert opt3._early["done"], "the early exchange started during the backward"
        opt3.allreduce_gradients()
        assert not opt3._early["done"]
        torch.cuda.synchronize()
        worst = max(rel_err(gp["g"], r) for gp, r in zip(opt3.param_groups, reduced))
        assert worst < 1e-4, "5. overlapped exchange == blocking exchange (%.3e)" % worst
        dist.barrier()
        # ---- single-process comparators on rank 0 (no collectives below this line on either rank) ----
        if rank == 0:
            student2, teacher2 = _tiny_gd_models()
            student2.cuda()
            teacher2.cuda()
            opt2 = create_optimizer(dict(lr=1e-3, weight_decay=0.01, lr_mult=1), student2, clip_grad_norm=1.0)
            student2.sample_itm_negatives = teacher2.sample_itm_negatives = lambda image_feat, text_feat, idx=None: local_negs
            saved = X._dist_rank_world
            expected = [torch.zeros_like(gp["g"]) for gp in opt2.param_groups]
            try:
                for r in range(world):
                    # shard r as a 1-process step whose "all_gather" returns the other shard's features as constants (Q3)
                    X._dist_rank_world = lambda: (0, 1)

                    def emulated_itc(image_feat, text_feat, idx=None, r=r):
                        s = slice(r * B, (r + 1) * B)
                        ia = torch.cat([image_feat if j == r else other_i[j * B:(j + 1) * B] for j in range(world)])
                        ta = torch.cat([text_feat if j == r else other_t[j * B:(j + 1) * B] for j in range(world)])
                        assert rel_err(image_feat, other_i[s]) < 1e-6     # same weights, same shard, same kernels
                        return X.XVLMBase.get_contrastive_loss(student2, ia, ta, idx=None)
                    student2.get_contrastive_loss = emulated_itc
                    sh = [t[r * B:(r + 1) * B] for t in full]
                    so2 = student2(*sh, output_attentions=True, output_hidden_states=True)
                    with torch.no_grad():
                        to2 = teacher2(*sh, output_attentions=True, output_hidden_states=True)
                    opt2.zero_grad()
                    gd_loss(so2, to2, 1.0)[0].backward()
                    for e, gp in zip(expected, opt2.param_groups):
                        e.add_(gp["g"] / world)
                worst = max(rel_err(a, e) for a, e in zip(reduced, expected))
                assert worst < 2e-3, "3b. two-GPU gradients vs the mean of per-shard single-process gradients: %.3e" % worst
                # the 1-process run on the CONCATENATED batch: ITC is the same number, batch-mean terms are the mean over ranks
                del student2.get_contrastive_loss
                cat_negs = (torch.cat([local_negs[0] + r * B for r in range(world)]), torch.cat([local_negs[1] + r * B for r in range(world)]))
                student2.sample_itm_negatives = teacher2.sample_itm_negatives = lambda image_feat, text_feat, idx=None: cat_negs
                with torch.no_grad():
                    so3 = student2(*full, output_attentions=True, output_hidden_states=True)
                    to3 = teacher2(*full, output_attentions=True, output_hidden_states=True)
                    kd3 = gd_kd_losses(so3, to3, 1.0)
                assert abs(float(so3["loss"]["loss_itc"]) - float(itcs[0])) < 2e-3 * abs(float(itcs[0])), "2. ITC: concatenated batch"
                for k in ("loss_itm", "loss_mlm"):
                    assert abs(float(so3["loss"][k]) - mean_terms[k]) < 2e-3 * abs(mean_terms[k]), (k, float(so3["loss"][k]), mean_terms[k])
                for k, v in kd3.items():
                    assert abs(float(v) - mean_terms[k]) < 2e-3 * max(abs(mean_terms[k]), 1e-6), (k, float(v), mean_terms[k])
            finally:
                X._dist_rank_world = saved
        dist.barrier()
        dist.destroy_process_group()
        q.put((rank, "ok"))
    except Exception as e:  # pragma: no cover
        import traceback
        q.put((rank, "FAIL: " + repr(e) + "\n" + traceback.format_exc()))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_gpu_nccl_step_matches_single_process():
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=600) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
    for rank, msg in results:
        assert msg == "ok", "rank %d: %s" % (rank, msg)
