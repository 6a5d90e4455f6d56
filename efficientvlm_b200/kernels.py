"""Thin Python wrappers (one per C-ABI entry point) that take torch CUDA tensors, pass raw device pointers and the
CURRENT torch stream to libevlm_b200.so and return/fill torch tensors.  No math happens here; PyTorch only owns the
memory and the stream.  Every wrapper raises if a tensor is not on a CUDA device — there is no CPU path.
"""
import ctypes as C
import os

import torch

from . import _lib
from ._lib import BF16, F32, GemmArgs, AttnArgs, check

bf16 = torch.bfloat16
f32 = torch.float32


_raw_stream = torch._C._cuda_getCurrentRawStream   # ~0.1 us; torch.cuda.current_stream() costs ~3 us per launch
_dev_index = [None]


def _stream():
    d = _dev_index[0]
    if d is None:
        d = _dev_index[0] = torch.cuda.current_device()   # one process per GPU: the device never changes after the first launch
    return _raw_stream(d)


def _p(t):
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("efficientvlm_b200 kernels need CUDA tensors (no CPU fallback); got a %s tensor" % t.device)
    return C.c_void_p(t.data_ptr())


def _dt(t):
    if t.dtype == bf16:
        return BF16
    if t.dtype == f32:
        return F32
    raise ValueError("unsupported dtype %s" % t.dtype)


def launch_count():
    return int(_lib.load().evlm_launch_count())


def reset_launch_count():
    _lib.load().evlm_reset_launch_count()


_NUM_SMS = None


def num_sms():
    global _NUM_SMS
    if _NUM_SMS is None:
        _NUM_SMS = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    return _NUM_SMS


# ------------------------------------------------------------------------------------------------------------------
# GEMM
# ------------------------------------------------------------------------------------------------------------------
def gemm(A, B, D, M, N, K, *, a_mn=False, b_mn=False, epi_mode=0, bias=None, alpha=1.0, alpha_cols=0, act=0, gate=None,
         gate_mode=0, aux_out=None, aux_in=None, residual=None, dropout_p=0.0, seed=0, stream_id=0, splits=1, accumulate=False,
         m_limit=None, n_limit=None, k_limit=None):
    """D[M,N] = epilogue(A x B^T); A/B are 2-D bf16 tensors (rows may be strided), see include/evlm.h.
    m_limit / n_limit / k_limit: int32 device scalars (zero-skip: only the leading rows / columns / k are scheduled)."""
    assert A.dtype == bf16 and B.dtype == bf16 and A.dim() == 2 and B.dim() == 2 and D.dim() == 2
    assert A.stride(1) == 1 and B.stride(1) == 1 and D.stride(1) == 1
    g = GemmArgs()
    g.M, g.N, g.K = M, N, K
    g.A, g.lda, g.a_mn = _p(A), A.stride(0), int(a_mn)
    g.B, g.ldb, g.b_mn = _p(B), B.stride(0), int(b_mn)
    g.D, g.ldd, g.d_dtype = _p(D), D.stride(0), _dt(D)
    g.epi_mode = epi_mode
    g.bias = _p(bias)
    g.alpha, g.alpha_cols = alpha, alpha_cols
    g.act = act
    g.gate, g.gate_mode = _p(gate), (gate_mode if gate is not None else 0)
    if aux_out is not None:
        g.aux_out, g.ld_aux_out = _p(aux_out), aux_out.stride(0)
    if aux_in is not None:
        g.aux_in, g.ld_aux_in = _p(aux_in), aux_in.stride(0)
    if residual is not None:
        assert residual.dim() == 2 and residual.stride(1) == 1
        g.residual, g.ldr, g.res_dtype = _p(residual), residual.stride(0), _dt(residual)
    g.dropout_p, g.dropout_seed, g.dropout_stream = float(dropout_p), int(seed), int(stream_id)
    g.splits, g.accumulate, g.max_ctas = int(splits), int(accumulate), GEMM_MAX_CTAS
    g.m_limit, g.n_limit, g.k_limit = _p(m_limit), _p(n_limit), _p(k_limit)
    lim = [(d, t) for d, t in ((M, m_limit), (N, n_limit), (K, k_limit)) if t is not None]
    if GEMM_PROFILE is not None:   # bench.py: per-launch CUDA-event timing of the dominant kernel on the launching stream
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        check(_lib.load().evlm_gemm_bf16(C.byref(g), _stream()), "evlm_gemm_bf16")
        e1.record()
        # (executed FLOPs of a zero-skip launch: resolved from the device counts when the profile is read: bench.py)
        GEMM_PROFILE.append((e0, e1, 2.0 * M * N * K, (M, N, K, int(a_mn), int(b_mn))) + ((lim,) if lim else ()))
        return D
    check(_lib.load().evlm_gemm_bf16(C.byref(g), _stream()), "evlm_gemm_bf16")
    return D


e4m3 = torch.float8_e4m3fn


def quant_rows_e4m3(x, out=None, scale=None):
    """Rows of x (bf16 / fp32 [R, K], any row pitch) -> (q e4m3 [R, K] view of a [R, ldq] buffer with ldq % 16 == 0 and zero pad bytes,
    scale fp32 [R]).  q = satfinite_rn(x * (448 / amax_row)), scale = amax_row / 448 (include/evlm.h)."""
    assert x.dim() == 2 and x.stride(1) == 1
    R, Kd = x.shape
    if out is None:
        out = torch.empty(R, (Kd + 15) // 16 * 16, dtype=e4m3, device=x.device)[:, :Kd]
    if scale is None:
        scale = torch.empty(R, dtype=f32, device=x.device)
    assert out.dtype == e4m3 and out.shape == (R, Kd) and out.stride(1) == 1 and scale.dtype == f32 and scale.numel() == R
    check(_lib.load().evlm_quant_rows_e4m3(_p(x), _dt(x), x.stride(0), R, Kd, _p(out), out.stride(0), _p(scale), _stream()),
          "evlm_quant_rows_e4m3")
    return out, scale


def gemm_fp8(A, a_scale, B, b_scale, D, M, N, K, *, bias=None, alpha=1.0, alpha_cols=0, act=0, aux_out=None, residual=None):
    """D[M,N] = epilogue(a_scale[m] b_scale[n] sum_k A[m,k] B[n,k]); A / B e4m3 [rows, K] views with 16-byte row pitches (as
    quant_rows_e4m3 leaves them).  The forward epilogue of gemm() without gates, dropout, splits or limits."""
    assert A.dtype == e4m3 and B.dtype == e4m3 and A.dim() == 2 and B.dim() == 2 and D.dim() == 2
    assert A.stride(1) == 1 and B.stride(1) == 1 and D.stride(1) == 1
    assert a_scale.dtype == f32 and b_scale.dtype == f32
    g = GemmArgs()
    g.M, g.N, g.K = M, N, K
    g.A, g.lda = _p(A), A.stride(0)
    g.B, g.ldb = _p(B), B.stride(0)
    g.D, g.ldd, g.d_dtype = _p(D), D.stride(0), _dt(D)
    g.bias = _p(bias)
    g.alpha, g.alpha_cols = alpha, alpha_cols
    g.act = act
    if aux_out is not None:
        g.aux_out, g.ld_aux_out = _p(aux_out), aux_out.stride(0)
    if residual is not None:
        assert residual.dim() == 2 and residual.stride(1) == 1
        g.residual, g.ldr, g.res_dtype = _p(residual), residual.stride(0), _dt(residual)
    g.splits, g.max_ctas = 1, GEMM_MAX_CTAS
    check(_lib.load().evlm_gemm_fp8(C.byref(g), _p(a_scale), _p(b_scale), _stream()), "evlm_gemm_fp8")
    return D


GEMM_PROFILE = None
GEMM_MAX_CTAS = 0      # persistent-grid width of the tcgen05 GEMM (0 = every SM); profiling knob
HBM_PROFILE = None      # bench.py: list of (kernel name, start event, end event, algorithmic bytes) for the HBM-bound kernels


def _esz(t):
    return 0 if t is None else t.numel() * t.element_size()


def _hbm(name, nbytes, call):
    """Run `call()`; when bench.py has armed HBM_PROFILE, bracket it with CUDA events on the launching stream and record the
    ALGORITHMIC bytes of the launch (every operand read once, every result written once)."""
    if HBM_PROFILE is None:
        return call()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    r = call()
    e1.record()
    HBM_PROFILE.append((name, e0, e1, int(nbytes)))
    return r


def wgrad_splits(M, N, K):
    """Reduction-dimension split for weight gradients (few output tiles, very long K)."""
    # 128 x 256 output tiles when N allows (the kernel picks them when tiles x splits fill the machine): fewer, longer k ranges
    # per work item than 128 x 128 tiles with half the splits
    tiles = ((M + 127) // 128) * ((N + 255) // 256 if (N >= 256 and not os.environ.get("EVLM_GEMM_NARROW_SPLITK")) else (N + 127) // 128)
    kb = (K + 63) // 64
    s = max(1, min(num_sms() // max(tiles, 1), kb // 8))
    return s


def sgemm(A, B, D, M, N, K, *, alpha=1.0, a_trans=False, b_trans=False, beta=0.0, alpha_dev=None, alpha_dev_inv=False):
    assert A.dtype == f32 and B.dtype == f32 and D.dtype == f32
    check(_lib.load().evlm_sgemm(M, N, K, alpha, _p(A), A.stride(0), int(a_trans), _p(B), B.stride(0), int(b_trans), beta, _p(D),
                                 D.stride(0), _p(alpha_dev), int(alpha_dev_inv), _stream()), "evlm_sgemm")
    return D


def dot(x, y, out, scale=1.0, accumulate=False):
    check(_lib.load().evlm_dot(_p(x), _p(y), x.numel(), scale, _p(out), int(accumulate), _stream()), "evlm_dot")
    return out


# ------------------------------------------------------------------------------------------------------------------
# elementwise / layout
# ------------------------------------------------------------------------------------------------------------------
def cast_bf16(src, dst=None, dropout_p=0.0, seed=0, stream_id=0):
    """fp32 [rows, cols] (row-strided ok) -> bf16; optional dropout-mask replay."""
    assert src.dtype == f32 and src.dim() == 2 and src.stride(1) == 1
    if dst is None:
        dst = torch.empty(src.shape, dtype=bf16, device=src.device)
    _hbm("cast_f32_bf16", src.numel() * 6, lambda: check(
        _lib.load().evlm_cast_f32_to_bf16(_p(src), src.stride(0), _p(dst), dst.stride(0), src.shape[0], src.shape[1], dropout_p,
                                          int(seed), int(stream_id), _stream()), "evlm_cast_f32_to_bf16"))
    return dst


def cast_f32(src, dst=None):
    assert src.dtype == bf16 and src.dim() == 2 and src.stride(1) == 1
    if dst is None:
        dst = torch.empty(src.shape, dtype=f32, device=src.device)
    check(_lib.load().evlm_cast_bf16_to_f32(_p(src), src.stride(0), _p(dst), dst.stride(0), src.shape[0], src.shape[1], _stream()),
          "evlm_cast_bf16_to_f32")
    return dst


def colsum(X, out=None, accumulate=False):
    assert X.dim() == 2 and X.stride(1) == 1
    if out is None:
        out = torch.empty(X.shape[1], dtype=f32, device=X.device)
        accumulate = False
    check(_lib.load().evlm_colsum(_p(X), _dt(X), X.stride(0), X.shape[0], X.shape[1], _p(out), int(accumulate), _stream()), "evlm_colsum")
    return out


def cast_table_build(entries, device):
    """entries: [(src fp32 dense 2-D, dst bf16 2-D row-pitched)] -> device table for cast_table_run (kept by the caller)."""
    n = len(entries)
    arr = (_lib.CastEntry * n)()
    for i, (src, dst) in enumerate(entries):
        assert src.dtype == f32 and src.is_contiguous() and dst.dtype == bf16 and dst.stride(-1) == 1 and src.shape == dst.shape
        arr[i].src, arr[i].dst = src.data_ptr(), dst.data_ptr()
        arr[i].rows, arr[i].cols, arr[i].ldd = src.shape[0], src.shape[1], dst.stride(0)
    host = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).pin_memory()
    return host.to(device, non_blocking=True), n, host          # (the pinned buffer lives as long as the table: a captured copy re-reads it)


def cast_table_run(table):
    tab, n = table[0], table[1]
    check(_lib.load().evlm_cast_table(_p(tab), n, _stream()), "evlm_cast_table")


# ------------------------------------------------------------------------------------------------------------------
# zero-skip index work (include/evlm.h)
# ------------------------------------------------------------------------------------------------------------------
def compact_index(z):
    """(idx int32 [n]: kept positions first, then the dropped ones; count int32 [1]) of a gate vector, on the device."""
    z = z.reshape(-1)
    assert z.dtype == f32 and z.is_contiguous()
    idx = torch.empty(z.numel(), dtype=torch.int32, device=z.device)
    count = torch.empty(1, dtype=torch.int32, device=z.device)
    check(_lib.load().evlm_compact_index(_p(z), z.numel(), _p(idx), _p(count), _stream()), "evlm_compact_index")
    return idx, count


def gather_rows(src, idx, count, out=None):
    """out[j] = src[idx[j]] for j < count, 0 after; src 1-D or 2-D (bf16 / fp32)."""
    s2 = src if src.dim() == 2 else src.reshape(-1, 1)
    assert s2.stride(1) == 1 or s2.shape[1] == 1
    if out is None:
        out = torch.empty_like(s2, memory_format=torch.contiguous_format) if s2.dtype != bf16 else _alloc16_like(s2)
    check(_lib.load().evlm_gather_rows(_p(s2), s2.stride(0), _dt(s2), _p(idx), _p(count), _p(out), out.stride(0), s2.shape[0], s2.shape[1],
                                       _stream()), "evlm_gather_rows")
    return out if src.dim() == 2 else out.reshape(-1)


def _alloc16_like(x):
    ld = (x.shape[1] + 7) // 8 * 8
    return torch.empty(x.shape[0], ld, dtype=bf16, device=x.device)[:, :x.shape[1]] if ld != x.shape[1] else torch.empty(
        x.shape[0], ld, dtype=bf16, device=x.device)


def gather_cols(src, idx, count):
    assert src.dim() == 2 and src.dtype == bf16 and src.stride(1) == 1
    out = _alloc16_like(src)
    check(_lib.load().evlm_gather_cols_bf16(_p(src), src.stride(0), _p(idx), _p(count), _p(out), out.stride(0), src.shape[0], src.shape[1],
                                            _stream()), "evlm_gather_cols_bf16")
    return out


def scatter_rows_add(src, idx, count, dst, accumulate=True):
    """dst[idx[j]] (+)= src[j] for j < count (fp32, 1-D or 2-D); accumulate=False also zeroes the rows that were not kept."""
    s2 = src if src.dim() == 2 else src.reshape(-1, 1)
    d2 = dst if dst.dim() == 2 else dst.reshape(-1, 1)
    assert s2.dtype == f32 and d2.dtype == f32 and s2.shape == d2.shape
    check(_lib.load().evlm_scatter_rows_add(_p(s2), s2.stride(0), _p(idx), _p(count), _p(d2), d2.stride(0), s2.shape[0], s2.shape[1],
                                            int(accumulate), _stream()), "evlm_scatter_rows_add")
    return dst


def scatter_cols_add(src, idx, count, dst, accumulate=True):
    assert src.dim() == 2 and dst.dim() == 2 and src.dtype == f32 and dst.dtype == f32 and src.shape == dst.shape
    check(_lib.load().evlm_scatter_cols_add(_p(src), src.stride(0), _p(idx), _p(count), _p(dst), dst.stride(0), src.shape[0], src.shape[1],
                                            int(accumulate), _stream()), "evlm_scatter_cols_add")
    return dst


def coldot(X, Y):
    assert X.shape == Y.shape and X.dtype == bf16 and Y.dtype == bf16 and X.stride(0) == Y.stride(0)
    out = torch.empty(X.shape[1], dtype=f32, device=X.device)
    check(_lib.load().evlm_coldot(_p(X), _p(Y), X.stride(0), X.shape[0], X.shape[1], _p(out), _stream()), "evlm_coldot")
    return out


def act_fwd(x, act, out_dtype=None):
    assert x.is_contiguous()
    y = torch.empty(x.shape, dtype=out_dtype or x.dtype, device=x.device)
    check(_lib.load().evlm_act_fwd(_p(x), _dt(x), _p(y), _dt(y), x.numel(), act, _stream()), "evlm_act_fwd")
    return y


def act_bwd(dy, x, act, out_dtype=None):
    assert dy.is_contiguous() and x.is_contiguous() and dy.numel() == x.numel()
    dx = torch.empty(x.shape, dtype=out_dtype or dy.dtype, device=x.device)
    check(_lib.load().evlm_act_bwd(_p(dy), _dt(dy), _p(x), _dt(x), _p(dx), _dt(dx), x.numel(), act, _stream()), "evlm_act_bwd")
    return dx


def im2col_patch(image, P):
    B, Cc, R, _ = image.shape
    image = image.contiguous()
    G = R // P
    out = torch.empty(B * G * G, Cc * P * P, dtype=bf16, device=image.device)
    check(_lib.load().evlm_im2col_patch(_p(image), _p(out), B, Cc, R, P, _stream()), "evlm_im2col_patch")
    return out


def vit_assemble_fwd(patch_emb, cls, pos, B, N, H):
    out = torch.empty(B, N, H, dtype=f32, device=patch_emb.device)
    check(_lib.load().evlm_vit_assemble_fwd(_p(patch_emb), _p(cls), _p(pos), _p(out), B, N, H, _stream()), "evlm_vit_assemble_fwd")
    return out


def vit_assemble_bwd(dh, dcls, dpos, B, N, H):
    dpatch = torch.empty(B * (N - 1), H, dtype=bf16, device=dh.device)
    check(_lib.load().evlm_vit_assemble_bwd(_p(dh), _p(dpatch), _p(dcls), _p(dpos), B, N, H, _stream()), "evlm_vit_assemble_bwd")
    return dpatch


def bert_embed_fwd(ids, type_ids, pos_ids, word, type_emb, pos_emb, past_len):
    B, L = ids.shape
    H = word.shape[1]
    out = torch.empty(B, L, H, dtype=f32, device=word.device)
    check(_lib.load().evlm_bert_embed_fwd(_p(ids), _p(type_ids), _p(pos_ids), _p(word), _p(type_emb), _p(pos_emb), _p(out), B * L, L, H,
                                          past_len, word.shape[0], _stream()), "evlm_bert_embed_fwd")
    return out


def bert_embed_bwd(dout, ids, type_ids, pos_ids, dword, dtype_emb, dpos, past_len, padding_idx=-1):
    B, L = ids.shape
    H = dout.shape[-1]
    check(_lib.load().evlm_bert_embed_bwd(_p(dout), _p(ids), _p(type_ids), _p(pos_ids), _p(dword), _p(dtype_emb), _p(dpos), B * L, L, H,
                                          past_len, -1 if padding_idx is None else int(padding_idx), _stream()), "evlm_bert_embed_bwd")


# ------------------------------------------------------------------------------------------------------------------
# LayerNorm
# ------------------------------------------------------------------------------------------------------------------
def layernorm_fwd(x, gamma, beta, eps, want_f32=True, want_bf16=False, save_stats=True, dropout_p=0.0, seed=0, stream_id=0):
    """x: [rows, H] contiguous (fp32 / bf16). Returns (y_f32|None, y_bf16|None, mean|None, rstd|None)."""
    assert x.is_contiguous()
    H = x.shape[-1]
    rows = x.numel() // H
    y32 = torch.empty(x.shape, dtype=f32, device=x.device) if want_f32 else None
    y16 = torch.empty(x.shape, dtype=bf16, device=x.device) if want_bf16 else None
    mean = torch.empty(rows, dtype=f32, device=x.device) if save_stats else None
    rstd = torch.empty(rows, dtype=f32, device=x.device) if save_stats else None
    _hbm("layernorm_fwd", _esz(x) + _esz(y32) + _esz(y16), lambda: check(
        _lib.load().evlm_layernorm_fwd(_p(x), _dt(x), _p(gamma), _p(beta), eps, _p(y32), _p(y16), _p(mean), _p(rstd), rows, H,
                                       dropout_p, int(seed), int(stream_id), _stream()), "evlm_layernorm_fwd"))
    return y32, y16, mean, rstd


def layernorm_bwd_can_fuse(H):
    """Widths for which layernorm_bwd can also replay a dropout mask on its bf16 output and emit that output's column sums."""
    return H % 128 == 0 and H <= 1024


def layernorm_bwd(dy, x, gamma, mean, rstd, dres=None, want_f32=True, want_bf16=False, dgamma=None, dbeta=None, dropout_p=0.0, seed=0,
                  stream_id=0, out_dropout_p=0.0, out_stream_id=0, dcolsum=None):
    """Returns (dx_f32|None, dx_bf16|None); dgamma/dbeta (fp32 [H]) are accumulated into.
    out_dropout_p / out_stream_id / dcolsum (evlm_layernorm_bwd_ex, widths `layernorm_bwd_can_fuse`): dx_bf16 carries the dropout mask
    of stream `out_stream_id` (same seed) and dcolsum [H] += its column sums."""
    assert dy.is_contiguous() and x.is_contiguous()
    H = x.shape[-1]
    rows = x.numel() // H
    dx32 = torch.empty(x.shape, dtype=f32, device=x.device) if want_f32 else None
    dx16 = torch.empty(x.shape, dtype=bf16, device=x.device) if want_bf16 else None
    if out_dropout_p > 0.0 or dcolsum is not None:
        assert want_bf16 and layernorm_bwd_can_fuse(H)
        _hbm("layernorm_bwd", _esz(dy) + _esz(x) + _esz(dres) + _esz(dx32) + _esz(dx16), lambda: check(
            _lib.load().evlm_layernorm_bwd_ex(_p(dy), _dt(dy), _p(x), _dt(x), _p(gamma), _p(mean), _p(rstd), _p(dres), _p(dx32), _p(dx16),
                                              _p(dgamma), _p(dbeta), rows, H, dropout_p, int(seed), int(stream_id), float(out_dropout_p),
                                              int(out_stream_id), _p(dcolsum), _stream()), "evlm_layernorm_bwd_ex"))
        return dx32, dx16
    _hbm("layernorm_bwd", _esz(dy) + _esz(x) + _esz(dres) + _esz(dx32) + _esz(dx16), lambda: check(
        _lib.load().evlm_layernorm_bwd(_p(dy), _dt(dy), _p(x), _dt(x), _p(gamma), _p(mean), _p(rstd), _p(dres), _p(dx32), _p(dx16),
                                       _p(dgamma), _p(dbeta), rows, H, dropout_p, int(seed), int(stream_id), _stream()),
        "evlm_layernorm_bwd"))
    return dx32, dx16


# ------------------------------------------------------------------------------------------------------------------
# attention
# ------------------------------------------------------------------------------------------------------------------
def _attn_args(q, k, v, B, H, Lq, Lk, scale, key_mask, full_mask, causal, causal_offset, head_z, dropout_p, seed, stream_id,
               kv_index=None, pack_items=None, pack_own_kv=False):
    a = AttnArgs()
    if pack_items is not None:
        assert pack_items.dtype == torch.int32 and pack_items.dim() == 2 and pack_items.is_contiguous()
        a.pack_items, a.pack_groups, a.pack_width = _p(pack_items), pack_items.shape[0], pack_items.shape[1]
        a.pack_own_kv = 1 if pack_own_kv else 0
    if kv_index is not None:
        assert kv_index.dtype == torch.int32 and kv_index.numel() == B and kv_index.is_contiguous()
        assert k.shape[0] % Lk == 0
        a.kv_index, a.kv_batches = _p(kv_index), k.shape[0] // Lk
    a.B, a.H, a.Lq, a.Lk = B, H, Lq, Lk
    a.q, a.ldq = _p(q), q.stride(0)
    a.k, a.ldk = _p(k), k.stride(0)
    a.v, a.ldv = _p(v), v.stride(0)
    a.key_mask, a.full_mask = _p(key_mask), _p(full_mask)
    a.causal, a.causal_offset, a.scale = int(causal), int(causal_offset), float(scale)
    a.head_z = _p(head_z)
    a.dropout_p, a.dropout_seed, a.dropout_stream = float(dropout_p), int(seed), int(stream_id)
    return a


def probs_pitch(Lk):
    """Row pitch (floats) of the attention maps this library allocates: rounded up to 16 bytes so the forward can leave the rows as
    TMA box stores (197 keys -> 200).  The reference API sees the `[..., :Lk]` view; the pad columns hold exact zeros."""
    return (Lk + 3) // 4 * 4


def row_pitch(t):
    """Pitch of the last-but-one dimension when `t` is a [..., rows, cols] fp32 tensor whose rows are `pitch` floats apart and whose
    leading dimensions are dense over that pitch (a dense tensor, or a `[..., :cols]` view of one with padded rows); else None."""
    if t is None or t.dim() < 2 or t.stride(-1) != 1:
        return None
    ld = t.stride(-2) if t.shape[-2] > 1 else max(t.shape[-1], t.stride(-2))
    if ld < t.shape[-1]:
        return None
    exp = ld * t.shape[-2]
    for d in range(t.dim() - 3, -1, -1):
        if t.shape[d] != 1 and t.stride(d) != exp:
            return None
        exp *= t.shape[d]
    return ld


def pitched(t):
    """`t` itself when `row_pitch(t)` exists (no copy), else a dense copy."""
    return t if row_pitch(t) is not None else t.contiguous()


def padded_base(t):
    """The [..., rows, pitch] tensor over the memory of a row-pitched view (pad columns included)."""
    ld = row_pitch(t)
    if ld is None:
        return None
    return t if ld == t.shape[-1] else t.as_strided(tuple(t.shape[:-1]) + (ld,), t.stride(), t.storage_offset())


def attention_fwd(q, k, v, B, H, Lq, Lk, scale, *, key_mask=None, full_mask=None, causal=False, causal_offset=0, head_z=None,
                  want_probs=False, dropout_p=0.0, seed=0, stream_id=0, kv_index=None, pack_items=None, pack_own_kv=False,
                  kv_item_rows=0):
    """q: [B*Lq, *] bf16 view (row stride = ld), k/v: [B*Lk, *] (or [n_kv*Lk, *] with kv_index int32 [B]: query item b attends
    to K/V item kv_index[b]). Returns (ctx bf16 [B*Lq, H*64], probs|None, lse).
    kv_item_rows (Lq == 1, no map): k / v hold that many rows per item (a pre-allocated KV cache), the first Lk of them valid."""
    dev = q.device
    ctx = torch.empty(B * Lq, H * 64, dtype=bf16, device=dev)
    ldp = probs_pitch(Lk)
    probs = torch.empty(B, H, Lq, ldp, dtype=f32, device=dev) if want_probs else None
    lse = torch.empty(B, H, Lq, dtype=f32, device=dev)
    a = _attn_args(q, k, v, B, H, Lq, Lk, scale, key_mask, full_mask, causal, causal_offset, head_z, dropout_p, seed, stream_id, kv_index,
                   pack_items, pack_own_kv)
    a.ctx, a.ldc = _p(ctx), ctx.stride(0)
    a.probs, a.lse, a.ldp = _p(probs), _p(lse), ldp
    a.kv_item_rows = int(kv_item_rows)
    check(_lib.load().evlm_attention_fwd(C.byref(a), _stream()), "evlm_attention_fwd")
    if probs is not None and ldp != Lk:
        probs = probs[..., :Lk]
    return ctx, probs, lse


def attention_bwd(q, k, v, ctx, lse, dctx, dq, dk, dv, B, H, Lq, Lk, scale, *, probs=None, dprobs=None, key_mask=None, full_mask=None,
                  causal=False, causal_offset=0, head_z=None, dhead_z=None, dropout_p=0.0, seed=0, stream_id=0, kv_index=None,
                  pack_items=None, pack_own_kv=False, dp_rowdot=None, dp_kd_coef=None):
    """Writes dq/dk/dv (bf16 2-D views with row strides; dk/dv always have B*Lk rows, one block per QUERY item);
    dhead_z [H] fp32 is accumulated into.
    dp_kd_coef (device fp32 scalar): `dprobs` is the distillation TARGET map and the gradient on the returned map is
    dp_kd_coef * (P - target), formed inside the kernel; dp_rowdot then holds the unscaled sums of (P - target) * P per row."""
    a = _attn_args(q, k, v, B, H, Lq, Lk, scale, key_mask, full_mask, causal, causal_offset, head_z, dropout_p, seed, stream_id, kv_index,
                   pack_items, pack_own_kv)
    a.ctx, a.ldc = _p(ctx), ctx.stride(0)
    a.lse = _p(lse)
    if dp_kd_coef is not None:
        ld = row_pitch(dprobs)
        assert ld is not None and dp_rowdot is not None and dp_rowdot.numel() == B * H * Lq and dp_rowdot.dtype == f32
        assert dp_kd_coef.dtype == f32 and dp_kd_coef.numel() == 1
        a.ldp, a.dp_rowdot, a.dp_kd_coef = ld, _p(dp_rowdot), _p(dp_kd_coef)
    elif dprobs is not None:
        # the saved map and the incoming gradient share one row pitch (both are [..., :Lk] views of padded rows when they come from
        # attention_fwd / the KD loss backward); anything else is densified
        lp, ld = row_pitch(probs), row_pitch(dprobs)
        if lp is None or ld is None or lp != ld:
            probs, dprobs = probs.contiguous(), dprobs.contiguous()
            lp = Lk
        a.ldp = lp
        if dp_rowdot is not None and dp_rowdot.numel() == B * H * Lq and dp_rowdot.dtype == f32 and dp_rowdot.is_contiguous():
            a.dp_rowdot = _p(dp_rowdot)
    a.probs = _p(probs)
    a.dprobs_ext = _p(dprobs)
    a.dctx, a.lddc = _p(dctx), dctx.stride(0)
    a.dq, a.lddq = _p(dq), dq.stride(0)
    a.dk, a.lddk = _p(dk), dk.stride(0)
    a.dv, a.lddv = _p(dv), dv.stride(0)
    a.dhead_z = _p(dhead_z)
    lib = _lib.load()
    ws = torch.empty((int(lib.evlm_attention_bwd_workspace(C.byref(a))) + 3) // 4, dtype=f32, device=q.device)
    a.dkv_accum = _p(ws)
    check(lib.evlm_attention_bwd(C.byref(a), _stream()), "evlm_attention_bwd")


def index_add_rows(src16, index, n_dst):
    """out[index[i]] += src16[i] over rows; src16 bf16 [n_src, row_elems] contiguous, index int32 [n_src]; returns fp32 [n_dst, row_elems]."""
    assert src16.dtype == bf16 and src16.is_contiguous() and index.dtype == torch.int32 and index.numel() == src16.shape[0]
    out = torch.zeros(n_dst, src16.shape[1], dtype=f32, device=src16.device)
    check(_lib.load().evlm_index_add_rows(_p(src16), _p(index), _p(out), src16.shape[0], src16.shape[1], _stream()), "evlm_index_add_rows")
    return out


def index_fold_rows(src16, index, n_dst):
    """out[u] = sum of the rows src16[i] with index[i] == u (bf16 in / fp32 accumulate / bf16 out, deterministic)."""
    assert src16.dtype == bf16 and src16.is_contiguous() and index.dtype == torch.int32 and index.numel() == src16.shape[0]
    out = torch.empty(n_dst, src16.shape[1], dtype=bf16, device=src16.device)
    ws = torch.empty(2 * n_dst + 1 + src16.shape[0], dtype=torch.int32, device=src16.device)
    check(_lib.load().evlm_index_fold_rows(_p(src16), _p(index), src16.shape[0], n_dst, src16.shape[1], _p(out), _p(ws), _stream()),
          "evlm_index_fold_rows")
    return out


# ------------------------------------------------------------------------------------------------------------------
# losses
# ------------------------------------------------------------------------------------------------------------------
_CAPTURED_HOST_BUFFERS = []


def _pair_table(students, teachers, scales, grads=None, rowdots=None):
    n = len(students)
    arr = (_lib.MsePair * n)()
    for i, (s, t) in enumerate(zip(students, teachers)):
        assert s.is_contiguous() and t.is_contiguous() and s.numel() == t.numel()
        arr[i].s, arr[i].t = s.data_ptr(), t.data_ptr()
        arr[i].ds = grads[i].data_ptr() if grads is not None and grads[i] is not None else None
        if rowdots is not None and rowdots[i] is not None and (arr[i].ds or grads is None):
            arr[i].rowdot, arr[i].row_len = rowdots[i].data_ptr(), s.shape[-1]
        arr[i].n, arr[i].scale = s.numel(), float(scales[i])
        arr[i].s_dtype, arr[i].t_dtype = _dt(s), _dt(t)
    host = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).pin_memory()
    if torch.cuda.is_current_stream_capturing():
        # a captured H2D copy re-reads this pinned buffer at every replay: it must outlive the graph
        _CAPTURED_HOST_BUFFERS.append(host)
    return host.to(students[0].device, non_blocking=True), host


def mse_pairs_fwd(students, teachers, scales, want_rowdot=None):
    """want_rowdot[i]: also leave rowdot[i] = sum_j (s_ij - t_ij) s_ij per row of pair i (fp32 [numel / row_len], UNSCALED): what the
    attention backward needs when it forms the map gradient itself (attention_bwd(dp_kd_coef=...)).  Returns out or (out, rowdots)."""
    rowdots = None
    if want_rowdot is not None:
        rowdots = [torch.zeros(s.numel() // s.shape[-1], dtype=f32, device=s.device)
                   if (w and s.shape[-1] % 4 == 0 and s.dtype == f32 and t.dtype == f32) else None
                   for s, t, w in zip(students, teachers, want_rowdot)]
    tab, keep = _pair_table(students, teachers, scales, None, rowdots)
    out = torch.empty(len(students), dtype=f32, device=students[0].device)
    _hbm("mse_pairs_fwd", sum(_esz(a) + _esz(b) for a, b in zip(students, teachers)),
         lambda: check(_lib.load().evlm_mse_pairs_fwd(_p(tab), len(students), _p(out), _stream()), "evlm_mse_pairs_fwd"))
    out._evlm_keep = (tab, keep)
    if rowdots is not None:
        return out, rowdots
    return out


def mse_pairs_bwd(students, teachers, scales, dout, need, want_rowdot=None):
    """want_rowdot[i]: pair i is an attention map [..., rows, row_len]; also return rowdot[i] = sum_j ds_ij s_ij per row (fp32
    [numel / row_len]), the term the attention backward otherwise recomputes by re-reading both maps."""
    grads = [torch.empty(s.shape, dtype=f32, device=s.device) if nd else None for s, nd in zip(students, need)]
    rowdots = None
    if want_rowdot is not None:
        rowdots = [torch.zeros(s.numel() // s.shape[-1], dtype=f32, device=s.device)
                   if (w and g is not None and s.shape[-1] % 4 == 0 and s.dtype == f32) else None
                   for s, g, w in zip(students, grads, want_rowdot)]
    tab, keep = _pair_table(students, teachers, scales, grads, rowdots)
    _hbm("mse_pairs_bwd", sum(_esz(a) + _esz(b) + _esz(gr) for a, b, gr in zip(students, teachers, grads) if gr is not None),
         lambda: check(_lib.load().evlm_mse_pairs_bwd(_p(tab), len(students), _p(dout), _stream()), "evlm_mse_pairs_bwd"))
    if grads:
        for gten in grads:
            if gten is not None:
                gten._evlm_keep = (tab, keep)
                break
    if rowdots is not None:
        return grads, rowdots
    return grads


def xent_fwd(logits, labels, ignore_index=-100, label_smoothing=0.0):
    rows, V = logits.shape
    loss = torch.empty(rows, dtype=f32, device=logits.device)
    lse = torch.empty(rows, dtype=f32, device=logits.device)
    _hbm("xent_fwd", _esz(logits), lambda: check(
        _lib.load().evlm_xent_fwd(_p(logits), logits.stride(0), rows, V, _p(labels), ignore_index, label_smoothing, _p(loss), _p(lse),
                                  _stream()), "evlm_xent_fwd"))
    return loss, lse


def xent_bwd(logits, labels, lse, g_rows, ignore_index=-100, label_smoothing=0.0, out=None, accumulate=False):
    rows, V = logits.shape
    if out is None:
        out = torch.empty(rows, V, dtype=f32, device=logits.device)
        accumulate = False
    check(_lib.load().evlm_xent_bwd(_p(logits), logits.stride(0), rows, V, _p(labels), ignore_index, label_smoothing, _p(lse),
                                    _p(g_rows), _p(out), out.stride(0), int(accumulate), _stream()), "evlm_xent_bwd")
    return out


def kl_fwd(s, t, inv_temp=1.0):
    rows, V = s.shape
    kl = torch.empty(rows, dtype=f32, device=s.device)
    ls = torch.empty(rows, dtype=f32, device=s.device)
    lt = torch.empty(rows, dtype=f32, device=s.device)
    _hbm("kl_fwd", _esz(s) + _esz(t), lambda: check(
        _lib.load().evlm_kl_fwd(_p(s), _p(t), s.stride(0), t.stride(0), rows, V, inv_temp, _p(kl), _p(ls), _p(lt), _stream()), "evlm_kl_fwd"))
    return kl, ls, lt


def kl_bwd(s, t, ls, lt, g_rows, inv_temp=1.0, out=None, accumulate=False):
    rows, V = s.shape
    if out is None:
        out = torch.empty(rows, V, dtype=f32, device=s.device)
        accumulate = False
    check(_lib.load().evlm_kl_bwd(_p(s), _p(t), s.stride(0), t.stride(0), rows, V, inv_temp, _p(ls), _p(lt), _p(g_rows), _p(out),
                                  out.stride(0), int(accumulate), _stream()), "evlm_kl_bwd")
    return out


def soft_xent_fwd(logits, labels):
    rows, V = logits.shape
    loss = torch.empty(rows, dtype=f32, device=logits.device)
    lse = torch.empty(rows, dtype=f32, device=logits.device)
    check(_lib.load().evlm_soft_xent_fwd(_p(logits), logits.stride(0), _p(labels), labels.stride(0), rows, V, _p(loss), _p(lse), _stream()),
          "evlm_soft_xent_fwd")
    return loss, lse


def soft_xent_bwd(logits, labels, lse, g_rows):
    rows, V = logits.shape
    out = torch.empty(rows, V, dtype=f32, device=logits.device)
    check(_lib.load().evlm_soft_xent_bwd(_p(logits), logits.stride(0), _p(labels), labels.stride(0), rows, V, _p(lse), _p(g_rows), _p(out),
                                         out.stride(0), 0, _stream()), "evlm_soft_xent_bwd")
    return out


def reduce_sum(x, scale=1.0, out=None, accumulate=False):
    if out is None:
        out = torch.empty((), dtype=f32, device=x.device)
        accumulate = False
    check(_lib.load().evlm_reduce_sum(_p(x), x.numel(), scale, _p(out), int(accumulate), _stream()), "evlm_reduce_sum")
    return out


def l2norm_fwd(x):
    rows, D = x.shape
    y = torch.empty_like(x)
    inv = torch.empty(rows, dtype=f32, device=x.device)
    check(_lib.load().evlm_l2norm_fwd(_p(x), _p(y), _p(inv), rows, D, _stream()), "evlm_l2norm_fwd")
    return y, inv


def l2norm_bwd(dy, y, inv):
    rows, D = y.shape
    dx = torch.empty_like(y)
    check(_lib.load().evlm_l2norm_bwd(_p(dy), _p(y), _p(inv), _p(dx), rows, D, _stream()), "evlm_l2norm_bwd")
    return dx


def itm_sample_neg(sim, idx, u):
    B = sim.shape[0]
    out = torch.empty(B, dtype=torch.int64, device=sim.device)
    check(_lib.load().evlm_itm_sample_neg(_p(sim), sim.stride(0), _p(idx), _p(u), _p(out), B, _stream()), "evlm_itm_sample_neg")
    return out


# ------------------------------------------------------------------------------------------------------------------
# L0 / optimizer
# ------------------------------------------------------------------------------------------------------------------
def l0_sample_fwd(loga, u, temperature):
    z = torch.empty_like(loga)
    check(_lib.load().evlm_l0_sample_fwd(_p(loga), _p(u), _p(z), loga.numel(), temperature, _stream()), "evlm_l0_sample_fwd")
    return z


def l0_sample_bwd(loga, u, dz, temperature):
    d = torch.empty_like(loga)
    check(_lib.load().evlm_l0_sample_bwd(_p(loga), _p(u), _p(dz), _p(d), loga.numel(), temperature, _stream()), "evlm_l0_sample_bwd")
    return d


def l0_expected_fwd(loga, temperature, weight, out, accumulate):
    check(_lib.load().evlm_l0_expected_fwd(_p(loga), loga.numel(), temperature, weight, _p(out), int(accumulate), _stream()),
          "evlm_l0_expected_fwd")


def l0_expected_bwd(loga, temperature, weight, g, dloga):
    check(_lib.load().evlm_l0_expected_bwd(_p(loga), loga.numel(), temperature, weight, _p(g), _p(dloga), _stream()), "evlm_l0_expected_bwd")


def l0_deterministic(loga, temperature, magical_number):
    layers, size = loga.shape
    mask = torch.empty_like(loga)
    kept = torch.empty(layers, dtype=torch.int32, device=loga.device)
    check(_lib.load().evlm_l0_deterministic(_p(loga), _p(mask), _p(kept), layers, size, temperature, magical_number, _stream()),
          "evlm_l0_deterministic")
    return mask, kept


def clamp_(x, lo, hi):
    check(_lib.load().evlm_clamp_(_p(x), x.numel(), lo, hi, _stream()), "evlm_clamp_")


def sumsq(x, out):
    check(_lib.load().evlm_sumsq(_p(x), x.numel(), _p(out), _stream()), "evlm_sumsq")


def clip_coef(sumsq_t, max_norm, coef):
    check(_lib.load().evlm_clip_coef(_p(sumsq_t), max_norm, _p(coef), _stream()), "evlm_clip_coef")


def adamw_step(groups, grad_scale=None, hyper_dev=None):
    """groups: list of dicts(p, g, m, v, p_bf16|None, lr, beta1, beta2, eps, weight_decay, step); with `hyper_dev` (device
    fp32 [ngroups, 2] = step_size, lr*wd) the per-step scalars come from device memory (CUDA-graph replay)."""
    n = len(groups)
    arr = (_lib.AdamWGroup * n)()
    for i, gr in enumerate(groups):
        arr[i].p, arr[i].g, arr[i].m, arr[i].v = gr["p"].data_ptr(), gr["g"].data_ptr(), gr["m"].data_ptr(), gr["v"].data_ptr()
        arr[i].p_bf16 = gr["p_bf16"].data_ptr() if gr.get("p_bf16") is not None else None
        arr[i].n = gr["p"].numel()
        arr[i].lr, arr[i].beta1, arr[i].beta2, arr[i].eps = gr["lr"], gr["beta1"], gr["beta2"], gr["eps"]
        arr[i].weight_decay, arr[i].step = gr["weight_decay"], gr["step"]
    nbytes = sum(gr["p"].numel() for gr in groups) * 28        # read p, g, m, v (16 B) + write p, m, v (12 B) per parameter
    if hyper_dev is not None:
        assert hyper_dev.dtype == f32 and hyper_dev.numel() >= 2 * n
        _hbm("adamw", nbytes, lambda: check(_lib.load().evlm_adamw_step_dev(arr, n, _p(grad_scale), _p(hyper_dev), _stream()),
                                            "evlm_adamw_step_dev"))
    else:
        _hbm("adamw", nbytes, lambda: check(_lib.load().evlm_adamw_step(arr, n, _p(grad_scale), _stream()), "evlm_adamw_step"))


def store_f32(dst, values):
    """dst[:len(values)] = values (<= 32 host floats, passed as launch arguments; stream ordered)."""
    n = len(values)
    arr = (C.c_float * n)(*values)
    check(_lib.load().evlm_store_f32(_p(dst), arr, n, _stream()), "evlm_store_f32")


def greedy_select(logits, unfinished, pad_token_id, eos_token_ids):
    """One decode step's token selection (eff_bert.py:1510-1538, greedy branch) in one launch.
    logits fp32 [rows, vocab] (rows may be strided), unfinished int64 [rows].
    Returns (next_token int64 [rows], score fp32 [rows, 1], tokens_to_add int64 [rows], unfinished_out int64 [rows])."""
    assert logits.dtype == f32 and logits.dim() == 2 and logits.stride(1) == 1 and unfinished.dtype == torch.int64
    rows, vocab = logits.shape
    dev = logits.device
    out = torch.empty(3, rows, dtype=torch.int64, device=dev)
    score = torch.empty(rows, 1, dtype=f32, device=dev)
    eos = (C.c_int64 * max(1, len(eos_token_ids)))(*[int(e) for e in eos_token_ids])
    check(_lib.load().evlm_greedy_select(_p(logits), logits.stride(0), rows, vocab, _p(unfinished.contiguous()), int(pad_token_id), eos,
                                         len(eos_token_ids), out[0].data_ptr(), _p(score), out[1].data_ptr(), out[2].data_ptr(), _stream()),
          "evlm_greedy_select")
    return out[0], score, out[1], out[2]


def _beam_check(cond, what, msg):
    if not cond:
        check(-1, "%s: %s" % (what, msg))


def beam_step(logits, num_beams, cur_len, min_length, repetition_penalty, length_penalty, early_stopping, eos_token_id, pad_token_id,
              tokens, beam_scores, beam_src, done, hyp_tokens, hyp_len, hyp_score, hyp_count, hyp_worst):
    """One beam-search decode position for all items in one launch (include/evlm.h, evlm_beam_step).  logits fp32 [rows, vocab] with
    rows = batch * num_beams (row pitch may exceed vocab); the loop state tensors are updated in place: tokens int64 [rows, width]
    (history; column cur_len receives the new token), beam_scores fp32 [rows], beam_src int32 [rows], done int32 [batch], hyp_tokens
    int64 [batch, num_beams, width], hyp_len int32 [batch, num_beams], hyp_score fp64 [batch, num_beams], hyp_count int32 [batch],
    hyp_worst fp64 [batch]."""
    what = "evlm_beam_step"
    _beam_check(2 <= num_beams <= 8, what, "num_beams must be in 2..8")
    _beam_check(logits.dtype == f32 and logits.dim() == 2 and logits.stride(1) == 1, what, "logits must be fp32 [rows, vocab] with unit stride")
    rows, vocab = logits.shape
    _beam_check(rows % num_beams == 0, what, "rows must be batch * num_beams")
    batch = rows // num_beams
    _beam_check(vocab > 2 * num_beams, what, "vocab must exceed 2 * num_beams")
    _beam_check(tokens.dtype == torch.int64 and tokens.dim() == 2 and tokens.shape[0] == rows and tokens.is_contiguous(), what,
                "tokens must be contiguous int64 [rows, width]")
    width = tokens.shape[1]
    _beam_check(1 <= cur_len < width, what, "cur_len must be inside the history width")
    _beam_check(0 <= eos_token_id < vocab, what, "eos id outside the vocabulary")
    _state_check(what, num_beams, batch, width, beam_scores, beam_src, done, hyp_tokens, hyp_len, hyp_score, hyp_count, hyp_worst)
    check(_lib.load().evlm_beam_step(_p(logits), logits.stride(0), batch, num_beams, vocab, int(cur_len), int(min_length), float(repetition_penalty),
                                     float(cur_len ** length_penalty), 1 if early_stopping else 0, int(eos_token_id), int(pad_token_id),
                                     _p(tokens), width, _p(beam_scores), _p(beam_src), _p(done), _p(hyp_tokens), _p(hyp_len), _p(hyp_score),
                                     _p(hyp_count), _p(hyp_worst), _stream()), what)


def _state_check(what, num_beams, batch, width, beam_scores, beam_src, done, hyp_tokens, hyp_len, hyp_score, hyp_count, hyp_worst):
    rows = batch * num_beams
    for t, dt, shape in ((beam_scores, f32, (rows,)), (beam_src, torch.int32, (rows,)), (done, torch.int32, (batch,)),
                         (hyp_tokens, torch.int64, (batch, num_beams, width)), (hyp_len, torch.int32, (batch, num_beams)),
                         (hyp_score, torch.float64, (batch, num_beams)), (hyp_count, torch.int32, (batch,)), (hyp_worst, torch.float64, (batch,))):
        if t is None:
            continue
        _beam_check(t.dtype == dt and tuple(t.shape) == shape and t.is_contiguous(), what, "beam state tensor must be contiguous %s %s" % (dt, shape))


def beam_finalize(num_beams, cur_len, max_length, length_penalty, eos_token_id, pad_token_id, tokens, beam_scores, done, hyp_tokens, hyp_len,
                  hyp_score, hyp_count, hyp_worst):
    """BeamSearchScorer.finalize after the last step (history length cur_len).  Returns (out int64 [batch, max_length]: best hypothesis,
    eos if shorter than max_length, pad; lengths int32 [batch])."""
    what = "evlm_beam_finalize"
    _beam_check(2 <= num_beams <= 8, what, "num_beams must be in 2..8")
    _beam_check(tokens.dtype == torch.int64 and tokens.dim() == 2 and tokens.shape[0] % num_beams == 0 and tokens.is_contiguous(), what,
                "tokens must be contiguous int64 [batch * num_beams, width]")
    rows, width = tokens.shape
    batch = rows // num_beams
    _beam_check(1 <= cur_len <= width, what, "cur_len must be inside the history width")
    _beam_check(1 <= max_length <= width, what, "max_length must not exceed the history width")
    _state_check(what, num_beams, batch, width, beam_scores, None, done, hyp_tokens, hyp_len, hyp_score,
                 hyp_count, hyp_worst)
    out = torch.empty(batch, max_length, dtype=torch.int64, device=tokens.device)
    lengths = torch.empty(batch, dtype=torch.int32, device=tokens.device)
    check(_lib.load().evlm_beam_finalize(_p(tokens), width, _p(beam_scores), _p(done), batch, num_beams, int(cur_len), int(max_length),
                                         float(cur_len ** length_penalty), int(eos_token_id), int(pad_token_id), _p(hyp_tokens), _p(hyp_len),
                                         _p(hyp_score), _p(hyp_count), _p(hyp_worst), _p(out), _p(lengths), _stream()), what)
    return out, lengths


def kv_beam_reorder(caches, beam_src, num_beams, length):
    """In place, ONE launch: for every cache (bf16 [batch * num_beams, capacity, row_elems], contiguous) and position < length, row r
    takes the row of item(r) * num_beams + beam_src[r] (int32 [rows], 0 <= beam_src < num_beams)."""
    what = "evlm_kv_beam_reorder"
    _beam_check(2 <= num_beams <= 8, what, "num_beams must be in 2..8")
    _beam_check(1 <= len(caches) <= 32, what, "1..32 caches")
    shape = tuple(caches[0].shape)
    _beam_check(len(shape) == 3 and shape[0] % num_beams == 0, what, "caches must be [batch * num_beams, capacity, row_elems]")
    for c in caches:
        _beam_check(c.dtype == bf16 and tuple(c.shape) == shape and c.is_contiguous(), what, "caches must be contiguous bf16 of one shape")
    _beam_check(beam_src.dtype == torch.int32 and beam_src.numel() == shape[0] and beam_src.is_contiguous(), what, "beam_src must be int32 [rows]")
    _beam_check(0 <= length <= shape[1], what, "length exceeds the cache capacity")
    table = (C.c_void_p * len(caches))(*[_p(c).value for c in caches])
    check(_lib.load().evlm_kv_beam_reorder(table, len(caches), shape[0] // num_beams, num_beams, shape[1], shape[2], int(length), _p(beam_src),
                                           _stream()), what)


def rng_bind(state):
    """Bind (or with None unbind) the device uint64 word every dropout site adds to its seed."""
    if state is not None:
        assert state.dtype == torch.int64 and state.numel() == 1 and state.is_cuda
    check(_lib.load().evlm_rng_bind(_p(state)), "evlm_rng_bind")


def rng_advance(state, delta, set_value=False):
    check(_lib.load().evlm_rng_advance(_p(state), int(delta) & 0xFFFFFFFFFFFFFFFF, 1 if set_value else 0, _stream()), "evlm_rng_advance")
