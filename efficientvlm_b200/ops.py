"""Differentiable operators of the hot path.  Each autograd Function below orchestrates calls into libevlm_b200.so
(kernels.py) for a whole transformer layer / head / loss, forward AND backward, so that no implicit PyTorch compute
kernels (adds for residual gradients, dtype casts, elementwise gates) are issued on the hot path.

Conventions: public tensors (hidden states, attention maps, logits, losses) are fp32 like the reference returns;
GEMM operands are bf16 internally with fp32 accumulation; parameters stay the reference's fp32 nn.Parameters and
are shadowed in bf16 once per optimizer step.
"""
import math
import os
import weakref

import torch

from . import kernels as K
from ._lib import (ACT_GELU_ERF, ACT_NONE, ACT_QUICK_GELU, EPI_ACT_BACKWARD, GATE_POST_ACT, GATE_PRE_ACT)

bf16 = torch.bfloat16
f32 = torch.float32

# ----------------------------------------------------------------------------------------------------------------------
# RNG for dropout (counter-based on the device; the host only hands out 63-bit seeds)
# ----------------------------------------------------------------------------------------------------------------------
_seed = [0x2545F4914F6CDD1D]


def manual_seed(s):
    _seed[0] = (int(s) * 0x9E3779B97F4A7C15 + 0x632BE59BD9B4E019) & 0x7FFFFFFFFFFFFFFF


def next_seed():
    _seed[0] = (_seed[0] * 6364136223846793005 + 1442695040888963407) & 0x7FFFFFFFFFFFFFFF
    return _seed[0]


# ----------------------------------------------------------------------------------------------------------------------
# bf16 weight shadows
# ----------------------------------------------------------------------------------------------------------------------
_w16 = {}
_w8 = {}
_cat = {}
_epoch = [0]
_pepoch = {}


def invalidate_weight_cache(params=None):
    """Call after parameters were modified behind autograd's back (our fused optimizer / arena re-pointing): all shadows, or
    only those of `params` (the optimizer's own: a frozen teacher keeps its shadows across steps)."""
    if params is None:
        _epoch[0] += 1
    else:
        for p in params:
            k = id(p)
            _pepoch[k] = _pepoch.get(k, 0) + 1


def clear_weight_cache():
    _w16.clear()
    _w8.clear()
    _cat.clear()


def _torch_optimizer_stepped(optimizer, args, kwargs):
    """Global `torch.optim.Optimizer` post-step hook.  A shadow's validity is keyed on `w._version` / `data_ptr()`, and an optimizer that
    updates through `p.data.add_()` — exactly what transformers-4.12.5's AdamW, the reference's optimizer (optim.py:1,67), does — bumps
    neither, so its shadows would silently go stale.  Every torch optimizer (HF AdamW subclasses `torch.optim.Optimizer`) therefore
    invalidates the shadows of its own parameters when its step() returns; `FlatAdamW` does the same itself.  Code that edits
    `p.data` outside any optimizer has to call `invalidate_weight_cache()`."""
    for g in optimizer.param_groups:
        for p in g["params"]:
            k = id(p)
            _pepoch[k] = _pepoch.get(k, 0) + 1


try:
    from torch.optim.optimizer import register_optimizer_step_post_hook as _register_post_hook
    _register_post_hook(_torch_optimizer_stepped)
except ImportError:  # pragma: no cover  (torch < 2.0)
    pass


def alloc16(rows, cols, device):
    """bf16 [rows, cols] view whose row pitch is a multiple of 8 elements (16 bytes: TMA / vector-access requirement)."""
    ld = (cols + 7) // 8 * 8
    if ld == cols:
        return torch.empty(rows, cols, dtype=bf16, device=device)
    return torch.zeros(rows, ld, dtype=bf16, device=device)[:, :cols]


def weight_bf16(*ws):
    """bf16 shadow of one or several fp32 [out, in...] weights stacked along dim 0 (cached per parameter version)."""
    key = tuple(id(w) for w in ws)
    ver = (tuple((w._version, w.data_ptr(), _pepoch.get(id(w), 0)) for w in ws), _epoch[0])
    ent = _w16.get(key)
    # identity is checked through weak references: id() / data_ptr() values are recycled once a model is freed
    alive = ent is not None and all(r() is w for r, w in zip(ent[2], ws))
    if alive and ent[0] == ver:
        return ent[1]
    rows = sum(w.shape[0] for w in ws)
    cols = ws[0][0].numel()
    out = ent[1] if alive and ent[1].shape == (rows, cols) else alloc16(rows, cols, ws[0].device)
    r = 0
    for w in ws:
        K.cast_bf16(w.detach().reshape(w.shape[0], cols), out[r:r + w.shape[0]])
        r += w.shape[0]
    if len(_w16) > 4096:
        for k in [k for k, e in _w16.items() if any(rf() is None for rf in e[2])]:
            del _w16[k]
    _w16[key] = (ver, out, tuple(weakref.ref(w) for w in ws))
    return out


class Fp8Weight:
    """e4m3 shadow of one or several stacked fp32 weights [N, K]: q [N, K] (16-byte row pitch) and one fp32 scale per output channel."""
    __slots__ = ("q", "scale")

    def __init__(self, q, scale):
        self.q, self.scale = q, scale

    def data_ptr(self):
        return self.q.data_ptr()


def weight_e4m3(*ws):
    """Fp8Weight of the fp32 weights `ws` stacked along dim 0, cached and invalidated exactly like weight_bf16.  Rows are quantised
    independently (K.quant_rows_e4m3, one launch per weight), so the stacked shadow equals the quantisation of the stacked matrix."""
    key = tuple(id(w) for w in ws)
    ver = (tuple((w._version, w.data_ptr(), _pepoch.get(id(w), 0)) for w in ws), _epoch[0])
    ent = _w8.get(key)
    alive = ent is not None and all(r() is w for r, w in zip(ent[2], ws))
    if alive and ent[0] == ver:
        return ent[1]
    rows = sum(w.shape[0] for w in ws)
    cols = ws[0][0].numel()
    out = Fp8Weight(torch.empty(rows, (cols + 15) // 16 * 16, dtype=K.e4m3, device=ws[0].device)[:, :cols],
                    torch.empty(rows, dtype=f32, device=ws[0].device))
    r = 0
    for w in ws:
        if w.shape[0]:
            K.quant_rows_e4m3(w.detach().reshape(w.shape[0], cols), out.q[r:r + w.shape[0]], out.scale[r:r + w.shape[0]])
        r += w.shape[0]
    if len(_w8) > 4096:
        for k in [k for k, e in _w8.items() if any(rf() is None for rf in e[2])]:
            del _w8[k]
    _w8[key] = (ver, out, tuple(weakref.ref(w) for w in ws))
    return out


def weight_fwd(fp8, *ws):
    """The forward operand of a covered Linear: the bf16 shadow, or the e4m3 one when the layer runs FP8 inference (fp8.enable)."""
    return weight_e4m3(*ws) if fp8 else weight_bf16(*ws)


def gemm_fwd(a16, W, D, M, N, Kd, dropout_p=0.0, seed=0, stream_id=0, gate=None, gate_mode=0, **epi):
    """Forward product D = epilogue(a16 W^T) of a covered Linear with the operand weight_fwd returned.  bf16: K.gemm.  FP8: the bf16
    activation is quantised per row (K.quant_rows_e4m3) and multiplied by the e4m3 weight (K.gemm_fp8); the epilogue is the same."""
    if not isinstance(W, Fp8Weight):
        return K.gemm(a16, W, D, M, N, Kd, dropout_p=dropout_p, seed=seed, stream_id=stream_id, gate=gate, gate_mode=gate_mode, **epi)
    if dropout_p > 0.0 or gate is not None:
        raise ValueError("FP8 inference has no dropout and no gates (it runs a model that prune.materialize has pruned, in eval mode)")
    qa, sa = K.quant_rows_e4m3(a16)
    return K.gemm_fp8(qa, sa, W.q, W.scale, D, M, N, Kd, **epi)


def _fp8_inference_only(fp8, training, need_grad, *gates):
    if not fp8:
        return
    if training or need_grad:
        raise RuntimeError("efficientvlm_b200: this model runs FP8 inference (fp8.enable), which has no backward: call it in eval mode "
                           "under torch.no_grad() / torch.inference_mode()")
    if any(z is not None for z in gates):
        raise ValueError("efficientvlm_b200: FP8 inference runs without gates (the gates of a materialised model live in its weights)")


_refresh_tables = {}


def refresh_weight_shadows(params):
    """Rebuild, with ONE launch, every existing bf16 shadow that contains one of `params` (called by FlatAdamW right after its update,
    instead of ~100 lazy per-weight casts during the next forward).  The (src, dst) table is cached in device memory while the set of
    shadows is unchanged, so a captured step graph replays it."""
    ids = {id(p) for p in params}
    entries, touched = [], []
    for key, ent in _w16.items():
        ws = [r() for r in ent[2]]
        if any(w is None for w in ws) or not any(id(w) in ids for w in ws) or not ws[0].is_cuda:
            continue
        out, r = ent[1], 0
        cols = ws[0][0].numel()
        for w in ws:
            entries.append((w.detach().reshape(w.shape[0], cols), out[r:r + w.shape[0]]))
            r += w.shape[0]
        touched.append((key, ws))
    if not entries:
        return 0
    sig = tuple((s.data_ptr(), d.data_ptr(), s.shape[0], s.shape[1], d.stride(0)) for s, d in entries)
    cached = _refresh_tables.get(id(params))
    if cached is None or cached[0] != sig:
        cached = _refresh_tables[id(params)] = (sig, K.cast_table_build(entries, entries[0][0].device))
    K.cast_table_run(cached[1])
    for key, ws in touched:
        ent = _w16[key]
        ver = (tuple((w._version, w.data_ptr(), _pepoch.get(id(w), 0)) for w in ws), _epoch[0])
        _w16[key] = (ver, ent[1], ent[2])
    return len(entries)


def bias_cat(*bs):
    if len(bs) == 1:
        return bs[0].detach()
    key = tuple(id(b) for b in bs)
    ver = (tuple((b._version, b.data_ptr(), _pepoch.get(id(b), 0)) for b in bs), _epoch[0])
    ent = _cat.get(key)
    if ent is not None and ent[0] == ver and all(r() is b for r, b in zip(ent[2], bs)):
        return ent[1]
    out = torch.cat([b.detach() for b in bs])
    if len(_cat) > 4096:
        for k in [k for k, e in _cat.items() if any(rf() is None for rf in e[2])]:
            del _cat[k]
    _cat[key] = (ver, out, tuple(weakref.ref(b) for b in bs))
    return out


def _join_rowdots(out, grads, bounds, shape):
    """Attention-map gradients carry `_evlm_rowdot` (see MSEPairsFn.backward): keep it when slices are joined back together."""
    if len(shape) != 4 or not all(g is None or getattr(g, "_evlm_rowdot", None) is not None for g in grads) or all(g is None for g in grads):
        return
    per_item = shape[1] * shape[2]
    parts = [g._evlm_rowdot if g is not None else torch.zeros((b - a) * per_item, dtype=f32, device=out.device)
             for g, a, b in zip(grads, bounds[:-1], bounds[1:])]
    out._evlm_rowdot = torch.cat(parts)


class SplitRowsFn(torch.autograd.Function):
    """x -> (x[b0:b1], x[b1:b2], ...) as views.  Plain slicing would make autograd zero-fill a full-size gradient per slice
    and add them up (three passes over a 145 MB attention map per slice); here the backward is ONE concatenation."""

    @staticmethod
    def forward(ctx, x, *bounds):
        ctx.set_materialize_grads(False)      # slices nobody differentiates through arrive as None (handled below), not as zero tensors
        ctx.bounds, ctx.meta = bounds, (x.shape, x.dtype, x.device)
        ctx.pitch = K.row_pitch(x) if x.dim() >= 2 and x.dtype == f32 else None
        return tuple(x[a:b] for a, b in zip(bounds[:-1], bounds[1:]))

    @staticmethod
    def backward(ctx, *grads):
        shape, dtype, device = ctx.meta
        pitch = ctx.pitch
        if pitch is not None and pitch != shape[-1] and all(g is None or K.row_pitch(g) == pitch for g in grads):
            # attention maps with padded rows: the gradient keeps the pitch (the attention backward reads it in place)
            # (whole padded row blocks are copied: dense, vectorised copies; the pad columns of the parts are exact zeros)
            base = torch.empty(tuple(shape[:-1]) + (pitch,), dtype=dtype, device=device)
            for g, a, b in zip(grads, ctx.bounds[:-1], ctx.bounds[1:]):
                if g is None:
                    base[a:b].zero_()
                else:
                    base[a:b].copy_(K.padded_base(g))
            out = base[..., :shape[-1]]
            _join_rowdots(out, grads, ctx.bounds, shape)
            return (out,) + (None,) * len(ctx.bounds)
        parts = []
        for g, a, b in zip(grads, ctx.bounds[:-1], ctx.bounds[1:]):
            parts.append(g if g is not None else torch.zeros((b - a,) + tuple(shape[1:]), dtype=dtype, device=device))
        out = torch.cat(parts, 0)
        _join_rowdots(out, grads, ctx.bounds, shape)
        return (out,) + (None,) * len(ctx.bounds)


def split_rows(x, bounds):
    """Slices of x along dim 0 at `bounds` (b0=0, ..., bn=len(x)); None passes through (maps skipped by attention_stride)."""
    if x is None:
        return (None,) * (len(bounds) - 1)
    if not (torch.is_grad_enabled() and x.requires_grad):
        return tuple(x[a:b] for a, b in zip(bounds[:-1], bounds[1:]))
    return SplitRowsFn.apply(x, *bounds)


class UniformGroups:
    """`encoder_batch_index` for rows that come in equal, consecutive groups: row r cross-attends to encoder item r // k
    (VQA rank_answer: k answer candidates per question).  Carries the explicit int32 index as well, for the paths that need it.
    In inference the layer then runs the cross-attention as ONE problem per encoder item with k * L query rows (query rows never
    interact in cross-attention), i.e. full 128-row tiles instead of one nearly empty tile per candidate."""

    def __init__(self, k, index, items=None):
        """items (int32 [rows // k], optional): encoder item of every group, for groups that index a larger resident encoder batch
        (ITR re-rank: several groups per image, images not in batch order); None = group j belongs to encoder item j."""
        self.k, self.index, self.items = int(k), index, items


_cross_kv = {}     # inference-only cache of cross-attention K|V projections (see BertLayerFn.forward)
_self_packs = {}
PACK_SELF_ATTENTION = os.environ.get("EVLM_NO_SELF_PACK") is None      # profiling knob


def self_attention_pack(B, L, device):
    """Pack table for the self-attention of short sequences: up to three consecutive batch items share one 128-row attention
    tile as a block-diagonal problem (evlm_attn_args.pack_own_kv).  None when the shape does not qualify."""
    if not PACK_SELF_ATTENTION or L % 8 != 0 or 2 * L > 128 or B < 2:
        return None
    width = min(3, 128 // L)
    key = (B, width, device)
    t = _self_packs.get(key)
    if t is None:
        groups = (B + width - 1) // width
        idx = torch.arange(groups * width, dtype=torch.int32).view(groups, width)
        idx = torch.where(idx < B, idx, torch.full_like(idx, -1))
        t = _self_packs[key] = idx.to(device).contiguous()
    return t


_act16 = {}


def act_bf16(x2):
    """bf16 [rows, width] copy of a contiguous fp32 activation [..., width], cached per tensor object: the image tokens feed the cross-attention K/V projection of
    every fusion layer, so one cast per forward pass replaces one per layer."""
    key = id(x2)
    ent = _act16.get(key)
    if ent is not None and ent[0]() is x2 and ent[1] == (x2._version, x2.data_ptr()):
        return ent[2]
    out = K.cast_bf16(x2.view(-1, x2.shape[-1]))
    for k in [k for k, e in _act16.items() if e[0]() is None]:
        del _act16[k]
    _act16[key] = (weakref.ref(x2), (x2._version, x2.data_ptr()), out)
    return out


# bf16 twins of layer outputs: a post-LN BERT layer ends in a LayerNorm whose fp32 output is the next layer's input, which that layer
# needs in bf16 for its QKV GEMM.  The LayerNorm writes both; the twin is found again through the identity (and version) of the fp32
# tensor object the caller passes on, so the per-layer fp32 -> bf16 cast kernel disappears.  A tensor that was sliced, concatenated or
# modified in between simply misses and is cast as before.
_twins = {}


def _register_twin(t, t16):
    for k in [k for k, e in _twins.items() if e[0]() is None]:      # (a handful of live entries: the twins die with their tensors)
        del _twins[k]
    _twins[id(t)] = (weakref.ref(t), t._version, t.data_ptr(), t16)


def _twin_of(x, rows, width):
    ent = _twins.get(id(x))
    if ent is not None and ent[0]() is x and ent[1] == x._version and ent[2] == x.data_ptr() and tuple(ent[3].shape) == (rows, width):
        return ent[3]
    return None


def _flat_gate(z, n):
    """[1,h,1,1] / [1,1,I] / ... gate -> contiguous fp32 [n] (detached)."""
    if z is None:
        return None
    z = z.detach().reshape(-1)
    if z.numel() != n:
        raise ValueError("gate has %d entries, expected %d" % (z.numel(), n))
    return z.to(f32).contiguous()


def _wgrad(dy16, x16, n_out, n_in, T):
    """dW[n_out, n_in] (fp32) = dy^T x over T rows; both operands are read in place (MN-major UMMA operands)."""
    dW = torch.zeros(n_out, n_in, dtype=f32, device=dy16.device)
    K.gemm(dy16, x16, dW, n_out, n_in, T, a_mn=True, b_mn=True, splits=K.wgrad_splits(n_out, n_in, T), accumulate=True)
    return dW


def _zeros(n, dev):
    return torch.zeros(n, dtype=f32, device=dev)


# ----------------------------------------------------------------------------------------------------------------------
# Fused gradient accumulation.  FlatAdamW keeps every parameter's gradient as a view into one fp32 arena and tags the parameter
# with it (`_evlm_main_grad`).  The backward passes below then accumulate weight / bias / LayerNorm gradients STRAIGHT into
# that view (split-K wgrad GEMM with accumulate, column sums with accumulate) and hand autograd `None` for the parameter:
# no per-parameter zero-fill, no temporary dW, no AccumulateGrad `add` launch (about 700 tiny launches per GD step).
# `loss.backward()` still leaves `p.grad` populated - it IS that view.  `torch.autograd.grad(...)` callers, who want the
# gradients returned instead, wrap the call in `with ops.returned_grads():`.
# ----------------------------------------------------------------------------------------------------------------------
_FUSED_GRADS = [os.environ.get("EVLM_RETURNED_GRADS") is None]      # EVLM_RETURNED_GRADS=1: gradients always go through autograd (a driver
#                                                                      that keeps its own torch DDP wrapper needs its per-parameter hooks to fire)


class returned_grads:
    """Context manager: parameter gradients are returned through autograd (no in-place accumulation into the arena)."""

    def __enter__(self):
        self.prev = _FUSED_GRADS[0]
        _FUSED_GRADS[0] = False

    def __exit__(self, *exc):
        _FUSED_GRADS[0] = self.prev


def accumulating_into_main_grads():
    """False inside `returned_grads()` (gradients then travel through autograd, not straight into the optimizer's arenas)."""
    return bool(_FUSED_GRADS[0])


def main_grad(p):
    if p is None or not _FUSED_GRADS[0]:
        return None
    return getattr(p, "_evlm_main_grad", None)


def _wgrad_to(param, dy16, x16, n_out, n_in, T):
    """dW[n_out, n_in] += dy^T x: into the parameter's arena gradient (returns None) or, without one, a fresh tensor."""
    mg = main_grad(param)
    if mg is None:
        return _wgrad(dy16, x16, n_out, n_in, T).view(param.shape)
    K.gemm(dy16, x16, mg.view(n_out, n_in), n_out, n_in, T, a_mn=True, b_mn=True, splits=K.wgrad_splits(n_out, n_in, T), accumulate=True)
    return None


def _bgrad_to(param, d16):
    """db += column sums of d16 (a 2-D bf16 view, rows may be strided)."""
    if param is None:
        return None
    mg = main_grad(param)
    if mg is None:
        return K.colsum(d16)
    K.colsum(d16, out=mg.view(-1), accumulate=True)
    return None


def _ln_bwd_for_linear(dout, x, lnw, mean, rstd, bg, bb, H, bias_param, p_out=0.0, seed=0, sid_out=0, dres=None):
    """LayerNorm backward + everything the Linear in front of it (dense -> dropout -> + residual -> LayerNorm) needs from the same pass:
    returns (dx fp32, that Linear's output gradient in bf16 = dx with the Linear's dropout mask replayed, its bias gradient or None when
    it was accumulated into the parameter's arena view).  One kernel instead of LayerNorm-backward + cast + column-sum."""
    if K.layernorm_bwd_can_fuse(H) and dout.is_cuda:
        mg = main_grad(bias_param)
        dcol = mg.view(-1) if mg is not None else torch.zeros(H, dtype=f32, device=dout.device)
        d32, d16 = K.layernorm_bwd(dout, x, lnw, mean, rstd, dres=dres, want_f32=True, want_bf16=True, dgamma=bg, dbeta=bb, seed=seed,
                                   out_dropout_p=p_out, out_stream_id=sid_out, dcolsum=dcol)
        return d32, d16, (None if mg is not None else dcol.view(bias_param.shape))
    d32, _ = K.layernorm_bwd(dout, x, lnw, mean, rstd, dres=dres, want_f32=True, dgamma=bg, dbeta=bb)
    d16 = K.cast_bf16(d32, dropout_p=p_out, seed=seed, stream_id=sid_out)
    return d32, d16, _bgrad_to(bias_param, d16)


def _stacked_grads(wparams, bparams, d16, x16, sizes, n_in, T):
    """Gradients of several Linear layers that share the input x16 and whose outputs are column blocks of d16 (fused QKV / KV
    projections): per-parameter accumulation into the arena when every one of them has an arena gradient, otherwise one stacked
    wgrad GEMM + column sum, split into views.  Returns ([dW...], [db...])."""
    if all(main_grad(w) is not None for w in wparams) and all(main_grad(b) is not None for b in bparams):
        c = 0
        for w, b, n in zip(wparams, bparams, sizes):
            blk = d16[:, c:c + n]
            _wgrad_to(w, blk, x16, n, n_in, T)
            _bgrad_to(b, blk)
            c += n
        return [None] * len(wparams), [None] * len(bparams)
    tot = sum(sizes)
    with returned_grads():
        dW = _wgrad(d16, x16, tot, n_in, T)
        db = K.colsum(d16)
    gw, gb, c = [], [], 0
    for n in sizes:
        gw.append(dW[c:c + n])
        gb.append(db[c:c + n])
        c += n
    return gw, gb


def _ln_grad_bufs(wparam, bparam, H, dev):
    """(dgamma buffer, dbeta buffer, grad to return for gamma, for beta): the kernels accumulate into the buffers."""
    mw, mb = main_grad(wparam), main_grad(bparam)
    if mw is not None and mb is not None:
        return mw.view(-1), mb.view(-1), None, None
    dw, db = _zeros(H, dev), _zeros(H, dev)
    return dw, db, dw, db


def _vec_grad_buf(param, shape, dev):
    """(accumulation buffer, grad to return) for kernels that accumulate into a dense fp32 gradient (embedding tables, cls, pos)."""
    mg = main_grad(param)
    if mg is not None:
        return mg, None
    z = torch.zeros(shape, dtype=f32, device=dev)
    return z, z


_GRAD_MODE = [True]


def _apply(fn, *args):
    """Function.forward always runs with grad mode off, so the caller's grad mode is captured here: under torch.no_grad()
    (teacher forward, evaluation, generation) nothing is saved and no backward-only buffers are written."""
    _GRAD_MODE[0] = torch.is_grad_enabled()
    return fn.apply(*args)


def _saved_or_raise(ctx, attr="saved"):
    """The Functions here keep their backward operands as plain ctx attributes and drop them after the first backward (the buffers of a
    layer are hundreds of MB).  A second backward through the same graph (retain_graph=True, double backward) therefore has nothing to read:
    say so instead of failing on a None unpack (ADVICE r1)."""
    v = getattr(ctx, attr, None)
    if v is None:
        raise RuntimeError("efficientvlm_b200: backward through this graph a second time — the layer buffers were freed after the first "
                           "backward (these Functions do not support retain_graph / double backward); re-run the forward")
    return v


def _needs_grad(ctx):
    return _GRAD_MODE[0] and any(ctx.needs_input_grad)


# ----------------------------------------------------------------------------------------------------------------------
# Zero-skip of pruned FFN columns (north star: "apply the gates in the epilogue AND skip fully-zeroed heads and columns")
# ----------------------------------------------------------------------------------------------------------------------
# The reference multiplies by z (eff_vit.py:214-219 before quick-GELU, eff_bert.py:553-557 after GELU).  A column with z == 0 produces
# an exact 0 activation (quick_gelu(0) = 0; 0 * gelu(u) = 0), so fc2 never sees it, and its weight / bias gradients are exact zeros.
# The kept columns are compacted to the front ON THE DEVICE (K.compact_index -> gathered bf16 weight rows / columns, bias, gate) and the
# four FFN GEMMs + two wgrads run with a device-side column limit: no host read-back, so the step graph replays with fresh masks.
# The gradient w.r.t. z ITSELF at z == 0 is the one thing that differs (the reference's is non-zero): it never reaches a parameter when
# z comes from the hard-concrete sampler, whose clamp has zero slope there (xvlm_l0_module.py:239-271), and is not needed at all for
# constant gates; a hand-made gate that requires grad keeps the dense path.
ZERO_SKIP = True
ZERO_SKIP_MIN_WIDTH = 256
SKIP_STATS = {"skip": 0, "dense_gated": 0}      # layer calls that took the compacted / the dense gated FFN path (tests, bench)


def _comes_from_l0(z, depth=8):
    """True when z is (a view / reshape / slice of) the hard-concrete sampler's output."""
    fn, seen = z.grad_fn, 0
    stack = [fn]
    while stack and seen < 64:
        fn = stack.pop()
        seen += 1
        if fn is None:
            continue
        if "L0SampleFn" in type(fn).__name__:
            return True
        name = type(fn).__name__
        if any(k in name for k in ("View", "Reshape", "Slice", "Select", "Squeeze", "Unsqueeze", "Expand", "Alias", "Index", "Permute",
                                   "Transpose", "Clone", "Split", "Unbind", "Cat", "Stack", "Narrow", "AsStrided", "Unsafe")):
            stack.extend(f for f, _ in fn.next_functions)
    return False


def ffn_skip_ok(mlp_z):
    if mlp_z is None:
        return False
    ok = ZERO_SKIP and mlp_z.numel() >= ZERO_SKIP_MIN_WIDTH and (
        not (torch.is_grad_enabled() and mlp_z.requires_grad) or _comes_from_l0(mlp_z))
    SKIP_STATS["skip" if ok else "dense_gated"] += 1
    return ok


class _Compact:
    """Kept-column index of one gate vector + the gathered fc1 rows / bias / gate and fc2 columns."""

    def __init__(self, mz, W1, b1, W2):
        self.idx, self.count = K.compact_index(mz)
        self.W1 = K.gather_rows(W1, self.idx, self.count)
        self.b1 = K.gather_rows(b1.detach().to(f32), self.idx, self.count)
        self.z = K.gather_rows(mz, self.idx, self.count)
        self.W2 = K.gather_cols(W2, self.idx, self.count)


# Inference with STATIC gates (the deterministic masks l0_module caches per log-alpha version): the compacted weights are a function of
# (mask, weights) only, so they are built once and re-used by every batch — masked inference then runs the kept columns at no per-batch
# index cost, like a physically pruned model (prune.materialize) but without touching the checkpoint layout.
_static_gates = {}     # data_ptr of a registered gate tensor -> (nbytes, token)
_compact_cache = {}


def register_static_gate(t, token):
    _static_gates[t.data_ptr()] = (t.numel() * t.element_size(), token)
    if len(_static_gates) > 256:
        for k in list(_static_gates)[:128]:
            del _static_gates[k]


def _static_gate_token(mz):
    p = mz.data_ptr()
    for base, (nbytes, token) in _static_gates.items():
        if base <= p < base + nbytes:
            return (base, token)
    return None


def _compact_for(mz, W1, w1p, b1, W2, w2p):
    """_Compact of this layer; cached when the gate is a registered static mask and autograd is off."""
    tok = None if torch.is_grad_enabled() else _static_gate_token(mz)
    if tok is None:
        return _Compact(mz, W1, b1, W2)
    key = (mz.data_ptr(), mz.numel(), id(w1p), id(w2p))
    ver = (tok, w1p._version, w1p.data_ptr(), _pepoch.get(id(w1p), 0), w2p._version, w2p.data_ptr(), _pepoch.get(id(w2p), 0),
           b1._version, _pepoch.get(id(b1), 0), _epoch[0])
    ent = _compact_cache.get(key)
    if ent is not None and ent[0] == ver and ent[2]() is w1p and ent[3]() is w2p:
        return ent[1]
    c = _Compact(mz, W1, b1, W2)
    _compact_cache[key] = (ver, c, weakref.ref(w1p), weakref.ref(w2p))
    return c


def _wgrad_compact(param, dy16, x16, n_out, n_in, T, cp, rows):
    """Weight gradient over the kept rows (`rows`: n_out is the gated dimension, fc1) or kept columns (fc2), scattered into the
    parameter's arena gradient (returns None) or a fresh dense tensor."""
    splits = K.wgrad_splits(n_out, n_in, T)
    tmp = (torch.zeros if splits > 1 else torch.empty)(n_out, n_in, dtype=f32, device=dy16.device)   # only the kept part is ever read
    lim = dict(m_limit=cp.count) if rows else dict(n_limit=cp.count)
    K.gemm(dy16, x16, tmp, n_out, n_in, T, a_mn=True, b_mn=True, splits=splits, accumulate=splits > 1, **lim)
    mg = main_grad(param)
    dst = mg.view(n_out, n_in) if mg is not None else torch.zeros(n_out, n_in, dtype=f32, device=dy16.device)
    (K.scatter_rows_add if rows else K.scatter_cols_add)(tmp, cp.idx, cp.count, dst, accumulate=True)
    return None if mg is not None else dst.view(param.shape)


def _vecgrad_compact(param, compact_vec, cp):
    """A [I] gradient computed on compacted columns -> the parameter's arena gradient (None) or a dense vector."""
    mg = main_grad(param) if param is not None else None
    if mg is not None:
        K.scatter_rows_add(compact_vec, cp.idx, cp.count, mg.view(-1), accumulate=True)
        return None
    out = torch.empty_like(compact_vec)
    K.scatter_rows_add(compact_vec, cp.idx, cp.count, out, accumulate=False)
    return out


class LayerCfg:
    """Static (non-tensor) configuration of one transformer layer call."""

    def __init__(self, num_heads, eps, want_probs=False, training=False, attn_dropout=0.0, hidden_dropout=0.0, causal=False,
                 has_cross=False, cross_heads=0, past_len=0, fp16_prescale=False, fp8=False):
        self.num_heads = num_heads
        self.eps = eps
        self.want_probs = want_probs
        self.training = training
        self.attn_dropout = attn_dropout
        self.hidden_dropout = hidden_dropout
        self.causal = causal
        self.has_cross = has_cross
        self.cross_heads = cross_heads
        self.past_len = past_len
        self.fp16_prescale = fp16_prescale
        self.fp8 = fp8                 # forward products in e4m3 (fp8.enable): inference only


# ----------------------------------------------------------------------------------------------------------------------
# ViT layer (pre-LN)  — eff_vit.py:231-273 / Appendix A.1
# ----------------------------------------------------------------------------------------------------------------------
# Attention-map distillation without a materialised gradient.  The KD loss is scale * mean((P_s - P_t)^2) per layer
# (GeneralDistill.py:60-82); its gradient c (P_s - P_t) is as large as the map itself (ViT-224: 242 MB per layer, ViT-384: 2 GB).
# For the maps of the ViT layers (no attention dropout) the loss backward writes nothing: the attention backward re-computes P_s anyway
# and reads the TEACHER map where it would read dP (evlm_attn_args.dp_kd_coef), the row sums it needs come out of the loss FORWARD
# (both maps are in registers there).  What autograd carries from MSEPairsFn.backward to VitLayerFn.backward is a NaN-filled,
# zero-stride placeholder of the map's shape with the real operands attached (`_evlm_kd`): any other consumer of that gradient — a map
# that also feeds another loss — would accumulate NaN and fail loudly instead of silently using a wrong gradient.
FUSED_ATTN_KD = os.environ.get("EVLM_NO_FUSED_ATTN_KD") is None
_kd_maps = {}              # data_ptr of a ViT layer's returned map -> weakref(map): the maps whose backward understands the placeholder
KD_STATS = {"fused_pairs": 0}


def _register_kd_map(probs):
    if len(_kd_maps) > 256:
        for key in [key for key, r in _kd_maps.items() if r() is None]:
            del _kd_maps[key]
    _kd_maps[probs.data_ptr()] = weakref.ref(probs)


def _is_kd_map(s):
    ref = _kd_maps.get(s.data_ptr())
    t = ref() if ref is not None else None
    return t is not None and t.shape == s.shape and t.stride() == s.stride() and t.dtype == s.dtype


class VitLayerFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, h, key_mask, head_z, head_layer_z, mlp_z, cfg, ln1w, ln1b, qw, qb, kw, kb, vw, vb, ow, ob, ln2w, ln2b, f1w, f1b,
                f2w, f2b):
        # an attention map nobody differentiates through must arrive as None in backward, not as a materialised zero tensor (which
        # would be filled, densified and streamed through the softmax backward for nothing)
        ctx.set_materialize_grads(False)
        B, N, H = h.shape
        T = B * N
        dev = h.device
        nh = cfg.num_heads
        E = qw.shape[0]
        I = f1w.shape[0]
        if E != nh * 64:
            raise ValueError("head_dim must be 64 (embed %d, heads %d)" % (E, nh))
        if head_layer_z is not None and _needs_grad(ctx):
            raise NotImplementedError("head_layer_z is forward-only (never produced by the reference's live L0 modules)")
        _fp8_inference_only(cfg.fp8, cfg.training, _needs_grad(ctx), head_z, head_layer_z, mlp_z)
        x2 = h.contiguous().reshape(T, H)
        _, a16, mean1, rstd1 = K.layernorm_fwd(x2, ln1w, ln1b, cfg.eps, want_f32=False, want_bf16=True)
        Wqkv = weight_fwd(cfg.fp8, qw, kw, vw)
        qkv = alloc16(T, 3 * E, dev)
        gemm_fwd(a16, Wqkv, qkv, T, 3 * E, H, bias=bias_cat(qb, kb, vb))
        hz = _flat_gate(head_z, nh)
        p_att = cfg.attn_dropout if cfg.training else 0.0
        seed = next_seed() if p_att > 0 else 0
        # (q W^T + b) * 64^-0.5 (eff_vit.py:137): the power-of-two scale commutes exactly with bf16 rounding
        c16, probs, lse = K.attention_fwd(qkv[:, :E], qkv[:, E:2 * E], qkv[:, 2 * E:], B, nh, N, N, 0.125, key_mask=key_mask, head_z=hz,
                                          want_probs=cfg.want_probs, dropout_p=p_att, seed=seed, stream_id=0)
        Wo = weight_fwd(cfg.fp8, ow)
        h1 = torch.empty(T, H, dtype=f32, device=dev)
        hlz = _flat_gate(head_layer_z.expand(1, 1, H) if head_layer_z is not None and head_layer_z.numel() == 1 else head_layer_z, H)
        gemm_fwd(c16, Wo, h1, T, H, E, bias=ob.detach(), gate=hlz, gate_mode=GATE_POST_ACT, residual=x2)
        _, m16, mean2, rstd2 = K.layernorm_fwd(h1, ln2w, ln2b, cfg.eps, want_f32=False, want_bf16=True)
        W1 = weight_fwd(cfg.fp8, f1w)
        W2 = weight_fwd(cfg.fp8, f2w)
        need_grad = _needs_grad(ctx)
        g16 = alloc16(T, I, dev)
        u16 = alloc16(T, I, dev) if need_grad else None
        mz = _flat_gate(mlp_z, I)
        cpk = _compact_for(mz, W1, f1w, f1b, W2, f2w) if getattr(cfg, "ffn_skip", False) else None
        h2 = torch.empty(T, H, dtype=f32, device=dev)
        if cpk is None:
            gemm_fwd(m16, W1, g16, T, I, H, bias=f1b.detach(), act=ACT_QUICK_GELU, gate=mz, gate_mode=GATE_PRE_ACT, aux_out=u16)
            gemm_fwd(g16, W2, h2, T, H, I, bias=f2b.detach(), residual=h1)
        else:     # kept columns only (device-side limit)
            K.gemm(m16, cpk.W1, g16, T, I, H, bias=cpk.b1, act=ACT_QUICK_GELU, gate=cpk.z, gate_mode=GATE_PRE_ACT, aux_out=u16, n_limit=cpk.count)
            K.gemm(g16, cpk.W2, h2, T, H, I, bias=f2b.detach(), residual=h1, k_limit=cpk.count)
            W1, W2, mz = cpk.W1, cpk.W2, cpk.z
        if need_grad:
            ctx.cfg = cfg
            ctx.dims = (B, N, H, E, I)
            ctx.seed = seed
            ctx.gate_shapes = (None if head_z is None else head_z.shape, None if mlp_z is None else mlp_z.shape)
            ctx.saved = (x2, a16, mean1, rstd1, qkv, c16, lse, probs, h1, m16, mean2, rstd2, u16, g16, Wqkv, Wo, W1, W2, hz, mz, key_mask)
            ctx.cpk = cpk
            ctx.params = (ln1w, ln1b, qw, qb, kw, kb, vw, vb, ow, ob, ln2w, ln2b, f1w, f1b, f2w, f2b)
        out = h2.view(B, N, H)
        if probs is None:
            return out, None
        if need_grad and p_att == 0.0 and N <= 1024:      # (the tcgen05 backward kernels: the tiled one reads a materialised dP only)
            _register_kd_map(probs)
        return out, probs

    @staticmethod
    def backward(ctx, dh2, dprobs):
        cfg = ctx.cfg
        B, N, H, E, I = ctx.dims
        T = B * N
        if dh2 is None:
            dh2 = torch.zeros(B, N, H, dtype=f32, device=ctx.saved[0].device)
        (x2, a16, mean1, rstd1, qkv, c16, lse, probs, h1, m16, mean2, rstd2, u16, g16, Wqkv, Wo, W1, W2, hz, mz, key_mask) = _saved_or_raise(ctx)
        ln1w, ln1b, qw, qb, kw, kb, vw, vb, ow, ob, ln2w, ln2b, f1w, f1b, f2w, f2b = ctx.params
        ctx.saved = None
        dev = x2.device
        nh = cfg.num_heads
        dh2 = dh2.contiguous().reshape(T, H)
        dy16 = K.cast_bf16(dh2)
        # ---- MLP ----
        cpk = ctx.cpk
        ctx.cpk = None
        need_mz = mz is not None and ctx.needs_input_grad[4]
        du16 = alloc16(T, I, dev)
        e16 = alloc16(T, I, dev) if need_mz else None
        dm16 = alloc16(T, H, dev)
        df2b = _bgrad_to(f2b, dy16)
        if cpk is None:
            df2w = _wgrad_to(f2w, dy16, g16, H, I, T)
            K.gemm(dy16, W2, du16, T, I, H, b_mn=True, epi_mode=EPI_ACT_BACKWARD, act=ACT_QUICK_GELU, gate=mz, gate_mode=GATE_PRE_ACT,
                   aux_in=u16, aux_out=e16)
            dmz = K.colsum(e16).reshape(ctx.gate_shapes[1]) if need_mz else None
            del e16, u16, g16
            df1w = _wgrad_to(f1w, du16, m16, I, H, T)
            df1b = _bgrad_to(f1b, du16)
            K.gemm(du16, W1, dm16, T, H, I, b_mn=True)
        else:     # the same products on the kept columns (W1 / W2 / mz are the compacted copies), gradients scattered back
            df2w = _wgrad_compact(f2w, dy16, g16, H, I, T, cpk, rows=False)
            K.gemm(dy16, W2, du16, T, I, H, b_mn=True, epi_mode=EPI_ACT_BACKWARD, act=ACT_QUICK_GELU, gate=mz, gate_mode=GATE_PRE_ACT,
                   aux_in=u16, aux_out=e16, n_limit=cpk.count)
            dmz = None
            if need_mz:
                dmz = torch.empty(I, dtype=f32, device=dev)
                K.scatter_rows_add(K.colsum(e16), cpk.idx, cpk.count, dmz, accumulate=False)
                dmz = dmz.reshape(ctx.gate_shapes[1])
            del e16, u16, g16
            df1w = _wgrad_compact(f1w, du16, m16, I, H, T, cpk, rows=True)
            df1b = _vecgrad_compact(f1b, K.colsum(du16), cpk)
            K.gemm(du16, W1, dm16, T, H, I, b_mn=True, k_limit=cpk.count)
        del du16
        bg2, bb2, dln2w, dln2b = _ln_grad_bufs(ln2w, ln2b, H, dev)
        dh1_32, dh1_16, dob = _ln_bwd_for_linear(dm16, h1, ln2w, mean2, rstd2, bg2, bb2, H, ob, dres=dh2)
        # ---- attention ----
        dow = _wgrad_to(ow, dh1_16, c16, H, E, T)
        dc16 = alloc16(T, E, dev)
        K.gemm(dh1_16, Wo, dc16, T, E, H, b_mn=True)
        dqkv = alloc16(T, 3 * E, dev)
        need_hz = hz is not None and ctx.needs_input_grad[2]
        dhz = _zeros(nh, dev) if need_hz else None
        rowdot, kd_coef = None, None
        if dprobs is not None:
            kd = getattr(dprobs, "_evlm_kd", None)
            if kd is not None:          # placeholder from MSEPairsFn.backward: (teacher map, coefficient, unscaled row sums), see FUSED_ATTN_KD
                dprobs, kd_coef, rowdot = kd
            else:
                rowdot = getattr(dprobs, "_evlm_rowdot", None)
                dprobs = K.pitched(dprobs)
        p_att = cfg.attn_dropout if cfg.training else 0.0
        K.attention_bwd(qkv[:, :E], qkv[:, E:2 * E], qkv[:, 2 * E:], c16, lse, dc16, dqkv[:, :E], dqkv[:, E:2 * E], dqkv[:, 2 * E:], B, nh, N,
                        N, 0.125, probs=probs, dprobs=dprobs, dp_rowdot=rowdot, dp_kd_coef=kd_coef, key_mask=key_mask, head_z=hz, dhead_z=dhz,
                        dropout_p=p_att, seed=ctx.seed, stream_id=0)
        (dqw, dkw, dvw), (dqb, dkb, dvb) = _stacked_grads((qw, kw, vw), (qb, kb, vb), dqkv, a16, (E, E, E), H, T)
        da16 = alloc16(T, H, dev)
        K.gemm(dqkv, Wqkv, da16, T, H, 3 * E, b_mn=True)
        bg1, bb1, dln1w, dln1b = _ln_grad_bufs(ln1w, ln1b, H, dev)
        dh, _ = K.layernorm_bwd(da16, x2, ln1w, mean1, rstd1, dres=dh1_32, want_f32=True, dgamma=bg1, dbeta=bb1)
        dhz_out = dhz.reshape(ctx.gate_shapes[0]) if need_hz else None
        return (dh.view(B, N, H), None, dhz_out, None, dmz, None, dln1w, dln1b, dqw, dqb, dkw, dkb, dvw, dvb, dow, dob, dln2w, dln2b,
                df1w, df1b, df2w, df2b)


def vit_layer(h, key_mask, head_z, head_layer_z, mlp_z, cfg, params):
    """params: (ln1w, ln1b, qw, qb, kw, kb, vw, vb, ow, ob, ln2w, ln2b, f1w, f1b, f2w, f2b). Returns (h_out, probs|None)."""
    cfg.ffn_skip = ffn_skip_ok(mlp_z)
    return _apply(VitLayerFn, h, key_mask, head_z, head_layer_z, mlp_z, cfg, *params)


# ----------------------------------------------------------------------------------------------------------------------
# ViT embeddings: patch conv (as im2col + GEMM) + cls + pos + pre-LN  — eff_vit.py:444-452
# ----------------------------------------------------------------------------------------------------------------------
class VitEmbedFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, patch_w, cls, pos, lnw, lnb, eps):
        B = x.shape[0]
        H = patch_w.shape[0]
        P = patch_w.shape[-1]
        N = pos.shape[0]
        if x.shape[2] != x.shape[3] or (x.shape[2] // P) ** 2 + 1 != N:
            raise ValueError("image %s does not match %d position embeddings (patch %d)" % (tuple(x.shape), N, P))
        patches = K.im2col_patch(x.detach().to(f32), P)
        Wp = weight_bf16(patch_w)
        pe = alloc16(patches.shape[0], H, x.device)
        K.gemm(patches, Wp, pe, patches.shape[0], H, patches.shape[1])
        asm = K.vit_assemble_fwd(pe, cls.detach(), pos.detach(), B, N, H)
        y, _, mean, rstd = K.layernorm_fwd(asm.view(B * N, H), lnw, lnb, eps, want_f32=True)
        if _needs_grad(ctx):
            ctx.saved = (patches, asm, mean, rstd, lnw)
            ctx.params = (patch_w, cls, pos, lnw, lnb)
            ctx.dims = (B, N, H, tuple(patch_w.shape))
        return y.view(B, N, H)

    @staticmethod
    def backward(ctx, dy):
        patches, asm, mean, rstd, lnw = _saved_or_raise(ctx)
        ctx.saved = None
        B, N, H, wshape = ctx.dims
        dev = dy.device
        patch_w, cls, pos, lnw_p, lnb_p = ctx.params
        bg, bb, dlnw, dlnb = _ln_grad_bufs(lnw_p, lnb_p, H, dev)
        dasm, _ = K.layernorm_bwd(dy.contiguous().view(B * N, H), asm.view(B * N, H), lnw, mean, rstd, want_f32=True, dgamma=bg, dbeta=bb)
        bcls, dcls = _vec_grad_buf(cls, (H,), dev)
        bpos, dpos = _vec_grad_buf(pos, (N, H), dev)
        dpatch = K.vit_assemble_bwd(dasm, bcls.view(-1), bpos.view(N, H), B, N, H)
        dW = _wgrad_to(patch_w, dpatch, patches, H, patches.shape[1], patches.shape[0])
        return None, dW, dcls, dpos, dlnw, dlnb, None


def vit_embed(x, patch_w, cls, pos, lnw, lnb, eps=1e-5):
    return _apply(VitEmbedFn, x, patch_w, cls, pos, lnw, lnb, eps)


# ----------------------------------------------------------------------------------------------------------------------
# generic pieces: LayerNorm, Linear(+act), activation
# ----------------------------------------------------------------------------------------------------------------------
class LayerNormFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w, b, eps):
        shape = x.shape
        x2 = x.contiguous().view(-1, shape[-1]).to(f32)
        y, _, mean, rstd = K.layernorm_fwd(x2, w, b, eps, want_f32=True)
        if _needs_grad(ctx):
            ctx.saved = (x2, mean, rstd, w)
            ctx.params = (w, b)
        return y.view(shape)

    @staticmethod
    def backward(ctx, dy):
        x2, mean, rstd, w = _saved_or_raise(ctx)
        ctx.saved = None
        H = x2.shape[-1]
        bg, bb, dw, db = _ln_grad_bufs(ctx.params[0], ctx.params[1], H, dy.device)
        dx, _ = K.layernorm_bwd(dy.contiguous().view(-1, H), x2, w, mean, rstd, want_f32=True, dgamma=bg, dbeta=bb)
        return dx.view(dy.shape), dw, db, None


def layer_norm(x, w, b, eps):
    return _apply(LayerNormFn, x, w, b, eps)


class LinearFn(torch.autograd.Function):
    """y = act(x W^T + b), fp32 in / fp32 out, bf16 tensor-core GEMM inside."""

    @staticmethod
    def forward(ctx, x, w, b, act, fp8):
        shape = x.shape
        Kin = shape[-1]
        Nout = w.shape[0]
        x2 = x.contiguous().view(-1, Kin).to(f32)
        M = x2.shape[0]
        dev = x.device
        x16 = alloc16(M, Kin, dev)
        K.cast_bf16(x2, x16)
        need = _needs_grad(ctx)
        _fp8_inference_only(fp8, False, need)
        W16 = weight_fwd(fp8, w)
        # row pitch padded to 16 bytes: the epilogue's TMA box stores need it (vocabulary 30522 -> pitch 30524; without it the
        # [1024, 30522] MLM logits fall back to scalar stores: 146 us instead of ~40 us per launch)
        y = torch.empty(M, Nout, dtype=f32, device=dev) if Nout % 4 == 0 else torch.empty(M, (Nout + 3) // 4 * 4, dtype=f32, device=dev)[:, :Nout]
        u16 = alloc16(M, Nout, dev) if (need and act != ACT_NONE) else None
        gemm_fwd(x16, W16, y, M, Nout, Kin, bias=None if b is None else b.detach(), act=act, aux_out=u16)
        if need:
            ctx.saved = (x16, W16, u16)
            ctx.params = (w, b)
            ctx.meta = (M, Nout, Kin, act, b is not None, tuple(w.shape))
        return y.view(*shape[:-1], Nout)

    @staticmethod
    def backward(ctx, dy):
        x16, W16, u16 = _saved_or_raise(ctx)
        ctx.saved = None
        M, Nout, Kin, act, has_b, wshape = ctx.meta
        dev = dy.device
        dy2 = dy.contiguous().view(M, Nout)
        d16 = alloc16(M, Nout, dev)
        if act != ACT_NONE:
            if d16.is_contiguous() and u16.is_contiguous():
                check_d = K.act_bwd(dy2, u16, act, out_dtype=bf16)
                d16 = check_d
            else:
                tmp = K.act_bwd(dy2, K.cast_f32(u16), act, out_dtype=f32)
                K.cast_bf16(tmp, d16)
        else:
            K.cast_bf16(dy2, d16)
        dW = _wgrad_to(ctx.params[0], d16, x16, Nout, Kin, M) if ctx.needs_input_grad[1] else None
        db = _bgrad_to(ctx.params[1], d16) if has_b and ctx.needs_input_grad[2] else None
        dx = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty(M, Kin, dtype=f32, device=dev)
            K.gemm(d16, W16, dx, M, Kin, Nout, b_mn=True)
            dx = dx.view(*dy.shape[:-1], Kin)
        return dx, dW, db, None, None


def linear(x, w, b=None, act=ACT_NONE):
    return _apply(LinearFn, x, w, b, act, False)


def linear_fp8(x, w, b=None, act=ACT_NONE):
    """linear() with the product in e4m3: the LM head of a model that fp8.enable has switched (inference only)."""
    return _apply(LinearFn, x, w, b, act, True)


class ActFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, act):
        x = x.contiguous()
        ctx.save_for_backward(x)
        ctx.act = act
        return K.act_fwd(x, act)

    @staticmethod
    def backward(ctx, dy):
        (x,) = ctx.saved_tensors
        return K.act_bwd(dy.contiguous(), x, ctx.act), None


def gelu(x):
    return _apply(ActFn, x, ACT_GELU_ERF)


# ----------------------------------------------------------------------------------------------------------------------
# BERT embeddings — eff_bert.py:188-215
# ----------------------------------------------------------------------------------------------------------------------
class BertEmbedFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, ids, type_ids, pos_ids, word, type_emb, pos_emb, lnw, lnb, eps, p_drop, past_len, padding_idx):
        B, L = ids.shape
        H = word.shape[1]
        ids = ids.contiguous()
        type_ids = None if type_ids is None else type_ids.contiguous()
        pos_ids = None if pos_ids is None else pos_ids.expand(B, L).contiguous()
        e = K.bert_embed_fwd(ids, type_ids, pos_ids, word.detach(), type_emb.detach(), pos_emb.detach(), past_len)
        seed = next_seed() if p_drop > 0 else 0
        y, _, mean, rstd = K.layernorm_fwd(e.view(B * L, H), lnw, lnb, eps, want_f32=True, dropout_p=p_drop, seed=seed, stream_id=7)
        if _needs_grad(ctx):
            ctx.saved = (ids, type_ids, pos_ids, e, mean, rstd, lnw)
            ctx.params = (word, type_emb, pos_emb, lnw, lnb)
            ctx.meta = (B, L, H, p_drop, seed, past_len, tuple(word.shape), tuple(type_emb.shape), tuple(pos_emb.shape), padding_idx)
        return y.view(B, L, H)

    @staticmethod
    def backward(ctx, dy):
        ids, type_ids, pos_ids, e, mean, rstd, lnw = _saved_or_raise(ctx)
        ctx.saved = None
        B, L, H, p_drop, seed, past_len, wsh, tsh, psh, padding_idx = ctx.meta
        dev = dy.device
        word, type_emb, pos_emb, lnw_p, lnb_p = ctx.params
        bg, bb, dlnw, dlnb = _ln_grad_bufs(lnw_p, lnb_p, H, dev)
        de, _ = K.layernorm_bwd(dy.contiguous().view(B * L, H), e.view(B * L, H), lnw, mean, rstd, want_f32=True, dgamma=bg, dbeta=bb,
                                dropout_p=p_drop, seed=seed, stream_id=7)
        bword, dword = _vec_grad_buf(word, wsh, dev) if ctx.needs_input_grad[3] else (None, None)
        btype, dtype_e = _vec_grad_buf(type_emb, tsh, dev) if ctx.needs_input_grad[4] else (None, None)
        bpos, dpos = _vec_grad_buf(pos_emb, psh, dev) if ctx.needs_input_grad[5] else (None, None)
        K.bert_embed_bwd(de, ids, type_ids, pos_ids, bword, btype, bpos, past_len, padding_idx)
        return None, None, None, dword, dtype_e, dpos, dlnw, dlnb, None, None, None, None


def bert_embed(ids, type_ids, pos_ids, word, type_emb, pos_emb, lnw, lnb, eps, p_drop, past_len=0, padding_idx=None):
    """padding_idx: the word row that gets no look-up gradient (nn.Embedding(padding_idx=pad_token_id), eff_bert.py:173)."""
    return _apply(BertEmbedFn, ids, type_ids, pos_ids, word, type_emb, pos_emb, lnw, lnb, eps, p_drop, past_len, padding_idx)


# ----------------------------------------------------------------------------------------------------------------------
# BERT layer (post-LN; self-attention [+ cross-attention to image tokens] + FFN) — eff_bert.py:480-560 / Appendix A.2
# ----------------------------------------------------------------------------------------------------------------------
N_SELF, N_CROSS, N_FFN = 10, 10, 6


KV_CACHE = os.environ.get("EVLM_NO_KV_CACHE") is None     # profiling knob: concatenating KV "cache" of the reference loop
KV_CACHE_SPARE = 32                                       # decode steps a cache holds beyond its prompt before the loop falls back to cat


_kv_caches = {}                                           # data_ptr -> weakref(cache buffer)


def _kv_cache_of(past_k, past_v, B, nh, E):
    """The live cache buffer [B, capacity, 2E] that `past_k` / `past_v` ([B, heads, Lp, 64]) are the K and V views of, else None."""
    ref = _kv_caches.get(past_k.data_ptr())
    cache = ref() if ref is not None else None
    if cache is None:
        if ref is not None:
            del _kv_caches[past_k.data_ptr()]
        return None
    cap = cache.shape[1]
    want = (cap * 2 * E, 64, 2 * E, 1)
    if (cache.shape[0] != B or cache.shape[2] != 2 * E or past_k.dtype != bf16 or past_k.shape[0] != B or past_k.shape[1] != nh
            or tuple(past_k.stride()) != want or tuple(past_v.stride()) != want or past_v.shape != past_k.shape
            or past_v.data_ptr() != cache.data_ptr() + 2 * E or past_k.shape[2] > cap):
        return None
    if len(_kv_caches) > 256:
        for key in [key for key, r in _kv_caches.items() if r() is None]:
            del _kv_caches[key]
    return cache


def kv_beam_reorder(past, beam_src, num_beams):
    """Beam search: re-order a decode loop's `past` IN PLACE (row r takes the row of its item's beam beam_src[r], int32 [rows]) when every
    layer's K / V are views of a live cache buffer; `past` then stays recognised by _kv_cache_of, so the next step keeps appending in
    place.  One launch per distinct cache shape (one for an unpruned decoder).  Returns False, touching nothing, when some layer's
    `past` is not a live cache (KV_CACHE off, or a cache that ran out of spare rows): the caller re-orders by copying."""
    if not KV_CACHE:
        return False
    groups = {}
    for layer in past:
        pk, pv = layer[0], layer[1]
        B, nh, Lp, _ = pk.shape
        cache = _kv_cache_of(pk, pv, B, nh, nh * 64)
        if cache is None:
            return False
        groups.setdefault((tuple(cache.shape), Lp), []).append(cache)
    for (_, Lp), caches in groups.items():
        for i in range(0, len(caches), 32):
            K.kv_beam_reorder(caches[i:i + 32], beam_src, num_beams, Lp)
    return True


class BertLayerFn(torch.autograd.Function):
    """args: x, key_mask, enc, enc_mask, enc_index, self_head_z, cross_head_z, mlp_z, past_k, past_v, cfg,
             [self: qw,qb,kw,kb,vw,vb,ow,ob,lnw,lnb] [cross: same 10 | omitted] [ffn: w1,b1,w2,b2,lnw,lnb]
    enc_index (int32 [B] or None): text row b cross-attends to encoder item enc_index[b] — the K/V projection of the image
    tokens then runs once per IMAGE (enc has fewer items than x) instead of once per text row.  It may also be a tuple
    (enc_index, pack_items): pack_items int32 [groups, <=3] lists text rows that attend to the same image and share one
    128-row attention tile (include/evlm.h, evlm_attn_args.pack_items)."""

    @staticmethod
    def forward(ctx, x, key_mask, enc, enc_mask, enc_index, shz, chz, mlp_z, past_k, past_v, cfg, *P):
        ctx.set_materialize_grads(False)     # unused attention maps: None in backward (see VitLayerFn)
        B, L, H = x.shape
        T = B * L
        dev = x.device
        sp = P[:N_SELF]
        cp = P[N_SELF:N_SELF + N_CROSS] if cfg.has_cross else None
        fp = P[-N_FFN:]
        nh = cfg.num_heads
        E = sp[0].shape[0]
        if E != nh * 64:
            raise ValueError("head_dim must be 64 (all_head_size %d, heads %d)" % (E, nh))
        need = _needs_grad(ctx)
        if need and past_k is not None:
            raise NotImplementedError("KV-cache decoding is inference-only")
        _fp8_inference_only(cfg.fp8, cfg.training, need, shz, chz, mlp_z)
        train = cfg.training
        p_att = cfg.attn_dropout if train else 0.0
        p_hid = cfg.hidden_dropout if train else 0.0
        seed = next_seed() if (p_att > 0 or p_hid > 0) else 0
        scale = 1.0 / math.sqrt(64.0)  # eff_bert.py:330-331 (or the fp16 pre-scale :297-302: same power of two)
        x2 = x.contiguous().view(T, H).to(f32)
        x16 = _twin_of(x, T, H)
        if x16 is None:
            x16 = K.cast_bf16(x2)
        # ---- self attention ----
        Wqkv = weight_fwd(cfg.fp8, sp[0], sp[2], sp[4])
        qkv = alloc16(T, 3 * E, dev)
        gemm_fwd(x16, Wqkv, qkv, T, 3 * E, H, bias=bias_cat(sp[1], sp[3], sp[5]))
        q, k, v = qkv[:, :E], qkv[:, E:2 * E], qkv[:, 2 * E:]
        Lk = L
        k_new, v_new = k, v
        # KV cache of a decode loop (inference): ONE pre-allocated [B, capacity, K | V] buffer per layer.  The prompt step creates it, every
        # single-token step writes its K | V row in place (one strided copy instead of two growing torch.cat) and the single-query
        # attention kernel reads the first Lk rows per item (kv_item_rows).  The `present` tensors handed to the reference-style loop are
        # VIEWS of the buffer in the reference's [B, heads, Lk, 64] layout, tagged with it; anything else that comes back as `past`
        # (re-ordered beams, user tensors) takes the concatenating path.
        cache, kv_rows = None, 0
        if past_k is not None:
            Lp = past_k.shape[2]
            cache = _kv_cache_of(past_k, past_v, B, nh, E) if KV_CACHE else None
            if cache is not None and L == 1 and not cfg.want_probs and p_att == 0.0 and Lp + 1 <= cache.shape[1]:
                cache[:, Lp] = qkv[:, E:]
                Lk, kv_rows = Lp + 1, cache.shape[1]
                flat = cache.view(B * kv_rows, 2 * E)
                k, v = flat[:, :E], flat[:, E:]
            else:
                cache = None
                kk = torch.cat([past_k.permute(0, 2, 1, 3).reshape(B, Lp, E).to(bf16), k.reshape(B, L, E)], 1).reshape(B * (Lp + L), E)
                vv = torch.cat([past_v.permute(0, 2, 1, 3).reshape(B, Lp, E).to(bf16), v.reshape(B, L, E)], 1).reshape(B * (Lp + L), E)
                k, v, Lk = kk, vv, Lp + L
        elif KV_CACHE and cfg.causal and not need:
            cache = torch.empty(B, L + KV_CACHE_SPARE, 2 * E, dtype=bf16, device=dev)
            cache[:, :L] = qkv[:, E:].view(B, L, 2 * E)
        hz = _flat_gate(shz, nh)
        spack = self_attention_pack(B, L, dev) if (past_k is None and not cfg.causal) else None
        c16, probs, lse = K.attention_fwd(q, k, v, B, nh, L, Lk, scale, key_mask=key_mask, causal=cfg.causal, causal_offset=Lk - L,
                                          head_z=hz, want_probs=cfg.want_probs, dropout_p=p_att, seed=seed, stream_id=0,
                                          pack_items=spack, pack_own_kv=spack is not None, kv_item_rows=kv_rows)
        Wo = weight_fwd(cfg.fp8, sp[6])
        s1 = torch.empty(T, H, dtype=f32, device=dev)
        gemm_fwd(c16, Wo, s1, T, H, E, bias=sp[7].detach(), dropout_p=p_hid, seed=seed, stream_id=1, residual=x2)
        h1_32, h1_16, mean_a, rstd_a = K.layernorm_fwd(s1, sp[8], sp[9], cfg.eps, want_f32=True, want_bf16=True)
        # ---- cross attention ----
        cross_saved = None
        probs_x = None
        h2_32, h2_16 = h1_32, h1_16
        if cfg.has_cross:
            if enc is None:
                raise ValueError("encoder_hidden_states must be given for cross-attention layers")
            nhx = cfg.cross_heads
            Ex = cp[0].shape[0]
            Bn, Nn, He = enc.shape
            enc_pack = None
            uniform_k = 0
            uniform_items = None
            if isinstance(enc_index, UniformGroups):
                groups = Bn if enc_index.items is None else enc_index.items.numel()
                if not need and not cfg.want_probs and p_att == 0.0 and B == groups * enc_index.k:
                    uniform_k, uniform_items = enc_index.k, enc_index.items
                enc_index = enc_index.index
            if isinstance(enc_index, tuple):
                enc_index, enc_pack = enc_index
            if enc_index is None and Bn != B:
                raise ValueError("encoder batch %d != text batch %d" % (Bn, B))
            if enc_index is not None and (enc_index.dtype != torch.int32 or enc_index.numel() != B):
                raise ValueError("encoder_batch_index must be int32 with one entry per text row")
            enc16_obj = act_bf16(enc) if (enc.dtype == f32 and enc.is_contiguous()) else K.cast_bf16(enc.contiguous().to(f32).view(Bn * Nn, He))
            enc16 = enc16_obj.view(Bn * Nn, He)       # a NEW tensor object every call: cache identity is checked on enc16_obj
            Wq = weight_fwd(cfg.fp8, cp[0])
            Wkv = weight_fwd(cfg.fp8, cp[2], cp[4])
            qx = alloc16(T, Ex, dev)
            gemm_fwd(h1_16, Wq, qx, T, Ex, H, bias=cp[1].detach())
            # Inference (nothing saved for a backward): the K|V projection of the encoder states is the same at every step of a
            # decode loop and in both decoder passes of rank_answer — keep the last few (keyed by the bf16 activation copy, which
            # act_bf16 caches per tensor version, and by the weight shadow, which changes with every optimizer step).
            kv_key = None
            if not need:
                kv_key = (enc16.data_ptr(), Bn * Nn, Wkv.data_ptr(), _epoch[0], _pepoch.get(id(cp[2]), 0), _pepoch.get(id(cp[4]), 0),
                          cp[2]._version, cp[4]._version, cp[3]._version, cp[5]._version)
            hit = _cross_kv.get(kv_key) if kv_key is not None else None
            if hit is not None and hit[0] is enc16_obj and hit[1] is Wkv:
                kvx = hit[2]
            else:
                kvx = alloc16(Bn * Nn, 2 * Ex, dev)
                gemm_fwd(enc16, Wkv, kvx, Bn * Nn, 2 * Ex, He, bias=bias_cat(cp[3], cp[5]))
                if kv_key is not None:
                    if len(_cross_kv) >= 8:
                        _cross_kv.clear()
                    _cross_kv[kv_key] = (enc16_obj, Wkv, kvx)
            cz = _flat_gate(chz, nhx)
            if uniform_k:
                # k consecutive text rows per encoder item: one attention problem per item with k * L query rows
                gmask = None if enc_mask is None else enc_mask[::uniform_k].contiguous()
                cx16, probs_x, lse_x = K.attention_fwd(qx, kvx[:, :Ex], kvx[:, Ex:], B // uniform_k, nhx, L * uniform_k, Nn, scale,
                                                       key_mask=gmask, head_z=cz, want_probs=False, kv_index=uniform_items)
            else:
                cx16, probs_x, lse_x = K.attention_fwd(qx, kvx[:, :Ex], kvx[:, Ex:], B, nhx, L, Nn, scale, key_mask=enc_mask, head_z=cz,
                                                       want_probs=cfg.want_probs, dropout_p=p_att, seed=seed, stream_id=4,
                                                       kv_index=enc_index, pack_items=enc_pack)
            # K/V item every dK / dV row block belongs to: per text row, or per packed group (its first member's image)
            fold_index = enc_index
            if enc_pack is not None and need:
                fold_index = enc_index.index_select(0, enc_pack[:, 0].long()).contiguous()
            Wox = weight_fwd(cfg.fp8, cp[6])
            s2 = torch.empty(T, H, dtype=f32, device=dev)
            gemm_fwd(cx16, Wox, s2, T, H, Ex, bias=cp[7].detach(), dropout_p=p_hid, seed=seed, stream_id=2, residual=h1_32)
            h2_32, h2_16, mean_x, rstd_x = K.layernorm_fwd(s2, cp[8], cp[9], cfg.eps, want_f32=True, want_bf16=True)
            cross_saved = (enc16, Wq, Wkv, qx, kvx, cz, cx16, lse_x, probs_x, Wox, s2, mean_x, rstd_x, Nn, He, Ex, nhx, enc_mask, enc_index, Bn,
                           enc_pack, fold_index)
        # ---- FFN ----
        I = fp[0].shape[0]
        W1 = weight_fwd(cfg.fp8, fp[0])
        W2 = weight_fwd(cfg.fp8, fp[2])
        g16 = alloc16(T, I, dev)
        u16 = alloc16(T, I, dev) if need else None
        mz = _flat_gate(mlp_z, I)
        cpk = _compact_for(mz, W1, fp[0], fp[1], W2, fp[2]) if getattr(cfg, "ffn_skip", False) else None
        s3 = torch.empty(T, H, dtype=f32, device=dev)
        if cpk is None:
            gemm_fwd(h2_16, W1, g16, T, I, H, bias=fp[1].detach(), act=ACT_GELU_ERF, gate=mz, gate_mode=GATE_POST_ACT, aux_out=u16)
            gemm_fwd(g16, W2, s3, T, H, I, bias=fp[3].detach(), dropout_p=p_hid, seed=seed, stream_id=3, residual=h2_32)
        else:     # kept columns only (device-side limit)
            K.gemm(h2_16, cpk.W1, g16, T, I, H, bias=cpk.b1, act=ACT_GELU_ERF, gate=cpk.z, gate_mode=GATE_POST_ACT, aux_out=u16, n_limit=cpk.count)
            K.gemm(g16, cpk.W2, s3, T, H, I, bias=fp[3].detach(), dropout_p=p_hid, seed=seed, stream_id=3, residual=h2_32, k_limit=cpk.count)
            W1, W2, mz = cpk.W1, cpk.W2, cpk.z
        out, out16, mean_o, rstd_o = K.layernorm_fwd(s3, fp[4], fp[5], cfg.eps, want_f32=True, want_bf16=True)
        out = out.view(B, L, H)
        _register_twin(out, out16)
        if need:
            ctx.cfg = cfg
            ctx.dims = (B, L, H, E, I)
            ctx.seed = seed
            ctx.gate_shapes = tuple(None if z is None else z.shape for z in (shz, chz, mlp_z))
            ctx.saved = (x16, Wqkv, qkv, hz, c16, lse, probs, Wo, s1, mean_a, rstd_a, h1_16, h2_16, cross_saved, W1, W2, g16, u16, mz, s3,
                         mean_o, rstd_o, key_mask)
            ctx.lnw = (sp[8], cp[8] if cfg.has_cross else None, fp[4])
            ctx.cpk = cpk
            ctx.params = (sp, cp, fp)
            ctx.nP = len(P)
        if cache is not None:
            present_k = cache[:, :Lk, :E].view(B, Lk, nh, 64).permute(0, 2, 1, 3)
            present_v = cache[:, :Lk, E:].view(B, Lk, nh, 64).permute(0, 2, 1, 3)
            _kv_caches[cache.data_ptr()] = weakref.ref(cache)
        else:
            present_k = k_new.reshape(B, L, nh, 64).permute(0, 2, 1, 3) if past_k is None else k.reshape(B, Lk, nh, 64).permute(0, 2, 1, 3)
            present_v = v_new.reshape(B, L, nh, 64).permute(0, 2, 1, 3) if past_k is None else v.reshape(B, Lk, nh, 64).permute(0, 2, 1, 3)
        ctx.mark_non_differentiable(present_k, present_v)
        return out, probs, probs_x, present_k, present_v

    @staticmethod
    def backward(ctx, dout, dprobs, dprobs_x, _dk, _dv):
        cfg = ctx.cfg
        B, L, H, E, I = ctx.dims
        T = B * L
        if dout is None:
            dout = torch.zeros(B, L, H, dtype=f32, device=ctx.saved[0].device)
        (x16, Wqkv, qkv, hz, c16, lse, probs, Wo, s1, mean_a, rstd_a, h1_16, h2_16, cross_saved, W1, W2, g16, u16, mz, s3, mean_o, rstd_o,
         key_mask) = _saved_or_raise(ctx)
        ctx.saved = None
        ln_a_w, ln_x_w, ln_o_w = ctx.lnw
        sp, cp, fp = ctx.params
        dev = dout.device
        nh = cfg.num_heads
        seed = ctx.seed
        p_att = cfg.attn_dropout if cfg.training else 0.0
        p_hid = cfg.hidden_dropout if cfg.training else 0.0
        scale = 1.0 / math.sqrt(64.0)
        nig = ctx.needs_input_grad
        # ---- FFN ----
        bgo, bbo, dlnow, dlnob = _ln_grad_bufs(fp[4], fp[5], H, dev)
        ds3, dy3, db2 = _ln_bwd_for_linear(dout.contiguous().view(T, H), s3, ln_o_w, mean_o, rstd_o, bgo, bbo, H, fp[3], p_hid, seed, 3)
        cpk = ctx.cpk
        ctx.cpk = None
        need_mz = mz is not None and nig[7]
        du16 = alloc16(T, I, dev)
        e16 = alloc16(T, I, dev) if need_mz else None
        dh2 = torch.empty(T, H, dtype=f32, device=dev)
        if cpk is None:
            dw2 = _wgrad_to(fp[2], dy3, g16, H, I, T)
            K.gemm(dy3, W2, du16, T, I, H, b_mn=True, epi_mode=EPI_ACT_BACKWARD, act=ACT_GELU_ERF, gate=mz, gate_mode=GATE_POST_ACT, aux_in=u16,
                   aux_out=e16)
            dmz = K.colsum(e16).reshape(ctx.gate_shapes[2]) if need_mz else None
            del e16, u16, g16
            dw1 = _wgrad_to(fp[0], du16, h2_16, I, H, T)
            db1 = _bgrad_to(fp[1], du16)
            K.gemm(du16, W1, dh2, T, H, I, b_mn=True, residual=ds3)  # grad wrt h2 = FFN path + residual path
        else:     # kept columns only (W1 / W2 / mz are the compacted copies), gradients scattered back
            dw2 = _wgrad_compact(fp[2], dy3, g16, H, I, T, cpk, rows=False)
            K.gemm(dy3, W2, du16, T, I, H, b_mn=True, epi_mode=EPI_ACT_BACKWARD, act=ACT_GELU_ERF, gate=mz, gate_mode=GATE_POST_ACT, aux_in=u16,
                   aux_out=e16, n_limit=cpk.count)
            dmz = None
            if need_mz:
                dmz = torch.empty(I, dtype=f32, device=dev)
                K.scatter_rows_add(K.colsum(e16), cpk.idx, cpk.count, dmz, accumulate=False)
                dmz = dmz.reshape(ctx.gate_shapes[2])
            del e16, u16, g16
            dw1 = _wgrad_compact(fp[0], du16, h2_16, I, H, T, cpk, rows=True)
            db1 = _vecgrad_compact(fp[1], K.colsum(du16), cpk)
            K.gemm(du16, W1, dh2, T, H, I, b_mn=True, residual=ds3, k_limit=cpk.count)
        del du16
        gcross = [None] * N_CROSS
        denc = None
        dchz_out = None
        dh1 = dh2
        if cfg.has_cross:
            (enc16, Wq, Wkv, qx, kvx, cz, cx16, lse_x, probs_x, Wox, s2, mean_x, rstd_x, Nn, He, Ex, nhx, enc_mask, enc_index, Bn, enc_pack,
             fold_index) = cross_saved
            bgx, bbx, dlnxw, dlnxb = _ln_grad_bufs(cp[8], cp[9], H, dev)
            ds2, dy2, dbox = _ln_bwd_for_linear(dh2, s2, ln_x_w, mean_x, rstd_x, bgx, bbx, H, cp[7], p_hid, seed, 2)
            dwox = _wgrad_to(cp[6], dy2, cx16, H, Ex, T)
            dcx = alloc16(T, Ex, dev)
            K.gemm(dy2, Wox, dcx, T, Ex, H, b_mn=True)
            dqx = alloc16(T, Ex, dev)
            n_blocks = enc_pack.shape[0] if enc_pack is not None else B      # dK / dV row blocks: per packed group or per text row
            dkvx = alloc16(n_blocks * Nn, 2 * Ex, dev)
            need_cz = cz is not None and nig[6]
            dcz = _zeros(nhx, dev) if need_cz else None
            rowdot_x = None
            if dprobs_x is not None:
                rowdot_x = getattr(dprobs_x, "_evlm_rowdot", None)
                dprobs_x = K.pitched(dprobs_x)
            K.attention_bwd(qx, kvx[:, :Ex], kvx[:, Ex:], cx16, lse_x, dcx, dqx, dkvx[:, :Ex], dkvx[:, Ex:], B, nhx, L, Nn, scale,
                            probs=probs_x, dprobs=dprobs_x, dp_rowdot=rowdot_x, key_mask=enc_mask, head_z=cz, dhead_z=dcz, dropout_p=p_att, seed=seed,
                            stream_id=4, kv_index=enc_index, pack_items=enc_pack)
            if enc_index is not None:
                # dk / dv came out per text row (or per packed group): fold the blocks that share an image
                dkvx = K.index_fold_rows(dkvx.view(n_blocks, Nn * 2 * Ex), fold_index, Bn).view(Bn * Nn, 2 * Ex)
            dwq = _wgrad_to(cp[0], dqx, h1_16, Ex, H, T)
            dbq = _bgrad_to(cp[1], dqx)
            (dwk, dwv), (dbk, dbv) = _stacked_grads((cp[2], cp[4]), (cp[3], cp[5]), dkvx, enc16, (Ex, Ex), He, Bn * Nn)
            if nig[2]:
                denc = torch.empty(Bn * Nn, He, dtype=f32, device=dev)
                K.gemm(dkvx, Wkv, denc, Bn * Nn, He, 2 * Ex, b_mn=True)
                denc = denc.view(Bn, Nn, He)
            dh1 = torch.empty(T, H, dtype=f32, device=dev)
            K.gemm(dqx, Wq, dh1, T, H, Ex, b_mn=True, residual=ds2)
            gcross = [dwq, dbq, dwk, dbk, dwv, dbv, dwox, dbox, dlnxw, dlnxb]
            dchz_out = dcz.reshape(ctx.gate_shapes[1]) if need_cz else None
        # ---- self attention ----
        bga, bba, dlnaw, dlnab = _ln_grad_bufs(sp[8], sp[9], H, dev)
        ds1, dy1, dbo = _ln_bwd_for_linear(dh1, s1, ln_a_w, mean_a, rstd_a, bga, bba, H, sp[7], p_hid, seed, 1)
        dwo = _wgrad_to(sp[6], dy1, c16, H, E, T)
        dc = alloc16(T, E, dev)
        K.gemm(dy1, Wo, dc, T, E, H, b_mn=True)
        dqkv = alloc16(T, 3 * E, dev)
        need_hz = hz is not None and nig[5]
        dhz = _zeros(nh, dev) if need_hz else None
        rowdot = None
        if dprobs is not None:
            rowdot = getattr(dprobs, "_evlm_rowdot", None)
            dprobs = K.pitched(dprobs)
        spack = self_attention_pack(B, L, dev) if not cfg.causal else None      # same geometry as the forward (dropout replay)
        K.attention_bwd(qkv[:, :E], qkv[:, E:2 * E], qkv[:, 2 * E:], c16, lse, dc, dqkv[:, :E], dqkv[:, E:2 * E], dqkv[:, 2 * E:], B, nh, L, L,
                        scale, probs=probs, dprobs=dprobs, dp_rowdot=rowdot, key_mask=key_mask, causal=cfg.causal, causal_offset=0, head_z=hz, dhead_z=dhz,
                        dropout_p=p_att, seed=seed, stream_id=0, pack_items=spack, pack_own_kv=spack is not None)
        (dwq_s, dwk_s, dwv_s), (dbq_s, dbk_s, dbv_s) = _stacked_grads((sp[0], sp[2], sp[4]), (sp[1], sp[3], sp[5]), dqkv, x16, (E, E, E), H, T)
        dx = None
        if nig[0]:
            dx = torch.empty(T, H, dtype=f32, device=dev)
            K.gemm(dqkv, Wqkv, dx, T, H, 3 * E, b_mn=True, residual=ds1)
            dx = dx.view(B, L, H)
        gself = [dwq_s, dbq_s, dwk_s, dbk_s, dwv_s, dbv_s, dwo, dbo, dlnaw, dlnab]
        gffn = [dw1, db1, dw2, db2, dlnow, dlnob]
        dhz_out = dhz.reshape(ctx.gate_shapes[0]) if need_hz else None
        grads = gself + (gcross if cfg.has_cross else []) + gffn
        return (dx, None, denc, None, None, dhz_out, dchz_out, dmz, None, None, None) + tuple(grads)


def bert_layer(x, key_mask, enc, enc_mask, self_head_z, cross_head_z, mlp_z, past_kv, cfg, params, enc_index=None):
    """Returns (out, self_probs|None, cross_probs|None, (present_k, present_v))."""
    pk, pv = (past_kv[0], past_kv[1]) if past_kv is not None else (None, None)
    cfg.ffn_skip = ffn_skip_ok(mlp_z)
    out, probs, probs_x, k, v = _apply(BertLayerFn, x, key_mask, enc, enc_mask, enc_index, self_head_z, cross_head_z, mlp_z, pk, pv, cfg,
                                       *params)
    return out, probs, probs_x, (k, v)


# ----------------------------------------------------------------------------------------------------------------------
# losses
# ----------------------------------------------------------------------------------------------------------------------
class MSEPairsFn(torch.autograd.Function):
    """out[p] = scale[p] * mean((s_p - t_p)^2) for all pairs in ONE launch (GeneralDistill.py:60-82)."""

    @staticmethod
    def forward(ctx, scales, n, *tensors):
        # Attention maps arrive as [..., :Lk] views of rows padded to 16 bytes (kernels.probs_pitch) with exact zeros in the pad
        # columns of BOTH maps: the kernel then runs over the padded storage in place (the pads contribute (0 - 0)^2) and the mean is
        # rescaled to the logical element count.  Anything else is densified as before.
        students, teachers, scales, logical, fused = [], [], list(scales), [], []
        grad_on = _GRAD_MODE[0]
        for i in range(n):
            s, t = tensors[i], tensors[n + i].detach()
            ps, pt = K.row_pitch(s), K.row_pitch(t)
            kd_map = s.dim() == 4 and _is_kd_map(s)
            if ps is not None and ps == pt and s.shape == t.shape and (ps != s.shape[-1] or kd_map):
                sb, tb = K.padded_base(s.detach()), K.padded_base(t)
                scales[i] = scales[i] * (sb.numel() / float(s.numel()))
                logical.append(s.shape[-1])
                # a ViT layer's own map (see FUSED_ATTN_KD): its gradient is never written, the loss forward leaves the row sums
                fused.append(FUSED_ATTN_KD and grad_on and ctx.needs_input_grad[2 + i] and kd_map and s.dtype == f32 and t.dtype == f32
                             and ps % 4 == 0)
            else:
                sb, tb = s.detach().contiguous(), t.contiguous()
                logical.append(None)
                fused.append(False)
            students.append(sb)
            teachers.append(tb)
        ctx.rowdots = None
        if any(fused):
            out, ctx.rowdots = K.mse_pairs_fwd(students, teachers, scales, want_rowdot=fused)
            fused = [f and rd is not None for f, rd in zip(fused, ctx.rowdots)]
            KD_STATS["fused_pairs"] += sum(fused)
        else:
            out = K.mse_pairs_fwd(students, teachers, scales)
        ctx.scales, ctx.n, ctx.logical, ctx.fused = tuple(scales), n, logical, fused
        ctx.students, ctx.teachers = students, teachers
        return out

    @staticmethod
    def backward(ctx, dout):
        need = [ctx.needs_input_grad[2 + i] and not f for i, f in enumerate(ctx.fused)]
        # 4-D pairs are attention maps: their gradient carries the per-row sums  sum_j dP_ij P_ij  along (`_evlm_rowdot`), which the
        # softmax backward needs and would otherwise recompute by re-reading both maps (attn_bwd_delta_kernel)
        _saved_or_raise(ctx, "students")
        is_map = [s.dim() == 4 for s in ctx.students]
        dout = dout.contiguous()
        if any(need):
            grads, rowdots = K.mse_pairs_bwd(ctx.students, ctx.teachers, ctx.scales, dout, need, want_rowdot=is_map)
        else:
            grads, rowdots = [None] * ctx.n, [None] * ctx.n
        grads = [g if (g is None or lk is None) else g[..., :lk] for g, lk in zip(grads, ctx.logical)]
        for g, rd in zip(grads, rowdots):
            if g is not None and rd is not None:
                g._evlm_rowdot = rd
        if any(ctx.fused):
            # d/dP_s of scale * mean((P_s - P_t)^2) = coef (P_s - P_t), coef = dout * 2 scale / numel (a device scalar per pair)
            nan = torch.full((1,), float("nan"), dtype=f32, device=dout.device)
            for i, f in enumerate(ctx.fused):
                if f:
                    s, t, lk = ctx.students[i], ctx.teachers[i], ctx.logical[i]
                    g = nan.expand(tuple(s.shape[:-1]) + (lk,))
                    g._evlm_kd = (t[..., :lk], dout[i:i + 1] * (2.0 * ctx.scales[i] / float(s.numel())), ctx.rowdots[i])
                    grads[i] = g
        ctx.students = ctx.teachers = ctx.rowdots = None
        return (None, None) + tuple(grads) + (None,) * ctx.n


def mse_pairs(students, teachers, scales):
    """Vector [len(students)] of scaled mean-squared errors."""
    return _apply(MSEPairsFn, tuple(float(s) for s in scales), len(students), *students, *teachers)


def _rows2d(t):
    """2-D tensors whose rows are dense (any row pitch) go to the loss kernels as they are: those take a leading dimension.  The MLM
    logits come out of the vocabulary GEMM with a 16-byte row pitch (30522 -> 30524); densifying them was a 125 MB copy per use."""
    return t if (t.dim() == 2 and t.stride(1) == 1 and t.stride(0) >= t.shape[1]) else t.contiguous()


class XentFn(torch.autograd.Function):
    """Per-row softmax CE (ignore_index rows -> 0), optional label smoothing.  logits fp32 [rows, V]."""

    @staticmethod
    def forward(ctx, logits, labels, ignore_index, label_smoothing):
        logits = _rows2d(logits)
        labels = labels.contiguous()
        loss, lse = K.xent_fwd(logits.detach(), labels, ignore_index, label_smoothing)
        ctx.saved = (logits.detach(), labels, lse)
        ctx.meta = (ignore_index, label_smoothing)
        return loss

    @staticmethod
    def backward(ctx, g):
        logits, labels, lse = _saved_or_raise(ctx)
        ctx.saved = None
        return K.xent_bwd(logits, labels, lse, g.contiguous(), ctx.meta[0], ctx.meta[1]), None, None, None


def xent_rows(logits, labels, ignore_index=-100, label_smoothing=0.0):
    return _apply(XentFn, logits, labels, ignore_index, label_smoothing)


class KLFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, s, t, inv_temp):
        s, t = _rows2d(s), _rows2d(t.detach())
        kl, ls, lt = K.kl_fwd(s.detach(), t, inv_temp)
        ctx.saved = (s.detach(), t, ls, lt)
        ctx.inv_temp = inv_temp
        return kl

    @staticmethod
    def backward(ctx, g):
        s, t, ls, lt = _saved_or_raise(ctx)
        ctx.saved = None
        return K.kl_bwd(s, t, ls, lt, g.contiguous(), ctx.inv_temp), None, None


def kl_rows(s_logits, t_logits, inv_temp=1.0):
    return _apply(KLFn, s_logits, t_logits, inv_temp)


class SoftXentFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, labels):
        logits, labels = logits.contiguous(), labels.detach().contiguous()
        loss, lse = K.soft_xent_fwd(logits.detach(), labels)
        ctx.saved = (logits.detach(), labels, lse)
        return loss

    @staticmethod
    def backward(ctx, g):
        logits, labels, lse = _saved_or_raise(ctx)
        ctx.saved = None
        return K.soft_xent_bwd(logits, labels, lse, g.contiguous()), None


def soft_xent_rows(logits, labels):
    return _apply(SoftXentFn, logits, labels)


class SumFn(torch.autograd.Function):
    """scale * sum(x) as a 0-dim tensor."""

    @staticmethod
    def forward(ctx, x, scale):
        ctx.shape, ctx.scale = x.shape, scale
        return K.reduce_sum(x.contiguous().to(f32), scale)

    @staticmethod
    def backward(ctx, g):
        return (g * ctx.scale).expand(ctx.shape), None


def sum_scaled(x, scale=1.0):
    return _apply(SumFn, x, scale)


class L2NormFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        x = x.contiguous().to(f32)
        y, inv = K.l2norm_fwd(x)
        ctx.saved = (y, inv)
        return y

    @staticmethod
    def backward(ctx, dy):
        y, inv = _saved_or_raise(ctx)
        ctx.saved = None
        return K.l2norm_bwd(dy.contiguous(), y, inv)


def l2_normalize(x):
    return _apply(L2NormFn, x)


class SimFn(torch.autograd.Function):
    """logits = a @ b^T / temp in fp32 (ITC, xvlm.py:397-399); temp is a device scalar parameter."""

    @staticmethod
    def forward(ctx, a, b, temp):
        a, b = a.contiguous().to(f32), b.contiguous().to(f32)
        M, Kd = a.shape
        N = b.shape[0]
        out = torch.empty(M, N, dtype=f32, device=a.device)
        K.sgemm(a, b, out, M, N, Kd, b_trans=True, alpha_dev=temp.detach(), alpha_dev_inv=True)
        ctx.saved = (a, b, temp.detach(), out)
        return out

    @staticmethod
    def backward(ctx, g):
        a, b, temp, out = _saved_or_raise(ctx)
        ctx.saved = None
        g = g.contiguous()
        M, Kd = a.shape
        N = b.shape[0]
        da = db = dt = None
        if ctx.needs_input_grad[0]:
            da = torch.empty_like(a)
            K.sgemm(g, b, da, M, Kd, N, alpha_dev=temp, alpha_dev_inv=True)               # (g / temp) @ b
        if ctx.needs_input_grad[1]:
            db = torch.empty_like(b)
            K.sgemm(g, a, db, N, Kd, M, a_trans=True, alpha_dev=temp, alpha_dev_inv=True)  # (g / temp)^T @ a
        if ctx.needs_input_grad[2]:
            # d/dtemp (x / temp) = -logits / temp
            dt = torch.empty((), dtype=f32, device=a.device)
            K.dot(g, out, dt, scale=-1.0)
            dt = dt / temp
        return da, db, dt


def sim_over_temp(a, b, temp):
    return _apply(SimFn, a, b, temp)


# ----------------------------------------------------------------------------------------------------------------------
# L0
# ----------------------------------------------------------------------------------------------------------------------
class L0SampleFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, loga, u, temperature):
        loga_c = loga.detach().contiguous()
        u = u.contiguous()
        ctx.saved = (loga_c, u)
        ctx.temperature = temperature
        return K.l0_sample_fwd(loga_c, u, temperature)

    @staticmethod
    def backward(ctx, dz):
        loga, u = _saved_or_raise(ctx)
        ctx.saved = None
        return K.l0_sample_bwd(loga, u, dz.contiguous(), ctx.temperature), None, None


def l0_sample(loga, u, temperature):
    return _apply(L0SampleFn, loga, u, temperature)


class L0ExpectedFn(torch.autograd.Function):
    """sum_k weight_k * sum(1 - cdf_qz(0, loga_k))  (get_num_parameters_and_constraint, xvlm_l0_module.py:198-216)."""

    @staticmethod
    def forward(ctx, temperature, weights, *logas):
        out = torch.zeros((), dtype=f32, device=logas[0].device)
        cs = [la.detach().contiguous() for la in logas]
        for la, w in zip(cs, weights):
            K.l0_expected_fwd(la, temperature, float(w), out, True)
        ctx.saved = cs
        ctx.meta = (temperature, weights)
        return out

    @staticmethod
    def backward(ctx, g):
        temperature, weights = ctx.meta
        g = g.contiguous()
        grads = []
        for la, w in zip(ctx.saved, weights):
            d = torch.zeros_like(la)
            K.l0_expected_bwd(la, temperature, float(w), g, d)
            grads.append(d)
        ctx.saved = None
        return (None, None) + tuple(grads)


def l0_expected_size(logas, weights, temperature):
    return _apply(L0ExpectedFn, temperature, tuple(weights), *logas)
