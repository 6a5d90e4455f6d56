"""GPU parity tests, kernel level: every C-ABI entry point against a plain torch fp32 reference of the same op on the
same seeded inputs (tolerances: 2e-2 relative for bf16-operand tensor-core paths, 1e-4 for fp32 paths; bit-exact for masks
and indices; BF_TOL is for KERNEL-level checks against torch on bf16-rounded inputs, the model-level bar is 1e-2 + the measured
reference noise, tests/helpers.py).  All calls go through efficientvlm_b200.kernels -> ctypes -> libevlm_b200.so."""
import math

import pytest
import torch
import torch.nn.functional as F

from tests.helpers import assert_close, load_golden

pytestmark = pytest.mark.gpu
bf16, f32 = torch.bfloat16, torch.float32
BF_TOL = 2e-2


@pytest.fixture(scope="module")
def K():
    from efficientvlm_b200 import kernels
    return kernels


def _rand(*shape, scale=1.0, dtype=f32, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(*shape, generator=g, device="cuda") * scale).to(dtype)


# ------------------------------------------------------------------------------------------------ GEMM
@pytest.mark.parametrize("M,N,K_", [(256, 256, 128), (300, 200, 136), (1000, 768, 768), (64, 2, 1536), (1024, 30522, 128)])
def test_gemm_forward_bias(K, M, N, K_):
    A = _rand(M, K_, dtype=bf16, seed=1)
    B = _rand(N, K_, dtype=bf16, seed=2)
    bias = _rand(N, seed=3)
    D = torch.empty(M, N, dtype=f32, device="cuda")
    K.gemm(A, B, D, M, N, K_, bias=bias)
    ref = A.float() @ B.float().t() + bias
    assert_close(D, ref, 1e-4, "gemm fwd fp32 out")
    D16 = torch.empty(M, (N + 7) // 8 * 8, dtype=bf16, device="cuda")[:, :N]
    K.gemm(A, B, D16, M, N, K_, bias=bias)
    assert_close(D16, ref, 6e-3, "gemm fwd bf16 out")


def test_gemm_dgrad_wgrad_layouts(K):
    T, O, I = 777, 328, 200   # ragged sizes: exercises TMA OOB fill and partial tiles
    dy = _rand(T, O, dtype=bf16, seed=4)
    W = _rand(O, I, dtype=bf16, seed=5)
    x = _rand(T, I, dtype=bf16, seed=6)
    dx = torch.empty(T, I, dtype=f32, device="cuda")
    K.gemm(dy, W, dx, T, I, O, b_mn=True)
    assert_close(dx, dy.float() @ W.float(), 1e-4, "dgrad (B MN-major)")
    dW = torch.zeros(O, I, dtype=f32, device="cuda")
    K.gemm(dy, x, dW, O, I, T, a_mn=True, b_mn=True, splits=3, accumulate=True)
    assert_close(dW, dy.float().t() @ x.float(), 1e-4, "wgrad (A,B MN-major, split-K)")
    K.gemm(dy, x, dW, O, I, T, a_mn=True, b_mn=True, splits=1, accumulate=True)
    assert_close(dW, 2 * (dy.float().t() @ x.float()), 1e-4, "wgrad accumulate")


def test_gemm_epilogues(K):
    from efficientvlm_b200._lib import ACT_GELU_ERF, ACT_QUICK_GELU, EPI_ACT_BACKWARD, GATE_POST_ACT, GATE_PRE_ACT
    M, N, K_ = 384, 512, 256
    A = _rand(M, K_, dtype=bf16, seed=1, scale=0.2)
    B = _rand(N, K_, dtype=bf16, seed=2, scale=0.2)
    bias, gate = _rand(N, seed=3), torch.rand(N, device="cuda")
    gate[::7] = 0
    res = _rand(M, N, seed=4)
    acc = A.float() @ B.float().t()
    # ViT: quick_gelu((acc+b)*z) + residual, pre-activation saved
    D = torch.empty(M, N, dtype=f32, device="cuda")
    aux = torch.empty(M, N, dtype=bf16, device="cuda")
    K.gemm(A, B, D, M, N, K_, bias=bias, act=ACT_QUICK_GELU, gate=gate, gate_mode=GATE_PRE_ACT, aux_out=aux, residual=res)
    u = acc + bias
    ref = (u * gate) * torch.sigmoid(1.702 * u * gate) + res
    assert_close(D, ref, 1e-4, "vit fc1 epilogue")
    assert_close(aux, u, 6e-3, "pre-activation")
    # BERT: gelu(acc+b)*z + bf16 residual
    K.gemm(A, B, D, M, N, K_, bias=bias, act=ACT_GELU_ERF, gate=gate, gate_mode=GATE_POST_ACT, residual=res.to(bf16))
    assert_close(D, F.gelu(u) * gate + res.to(bf16).float(), 1e-4, "bert ffn epilogue")
    # activation backward (dgrad of fc2 fused with act' and the gate-grad integrand)
    dy = _rand(M, K_, dtype=bf16, seed=7, scale=0.2)
    W2 = _rand(K_, N, dtype=bf16, seed=8, scale=0.2)      # [out=K_, in=N]
    dg = dy.float() @ W2.float()
    uu = aux.float().requires_grad_()
    zz = gate.clone().requires_grad_()
    du16, e16 = torch.empty(M, N, dtype=bf16, device="cuda"), torch.empty(M, N, dtype=bf16, device="cuda")
    K.gemm(dy, W2, du16, M, N, K_, b_mn=True, epi_mode=EPI_ACT_BACKWARD, act=ACT_QUICK_GELU, gate=gate, gate_mode=GATE_PRE_ACT, aux_in=aux,
           aux_out=e16)
    y = (uu * zz) * torch.sigmoid(1.702 * uu * zz)
    gu, gz = torch.autograd.grad(y, [uu, zz], dg)
    assert_close(du16, gu, 8e-3, "act-backward du (pre gate)")
    assert_close(K.colsum(e16), gz, 8e-3, "gate gradient (pre gate)")
    K.gemm(dy, W2, du16, M, N, K_, b_mn=True, epi_mode=EPI_ACT_BACKWARD, act=ACT_GELU_ERF, gate=gate, gate_mode=GATE_POST_ACT, aux_in=aux,
           aux_out=e16)
    y = F.gelu(uu) * zz
    gu, gz = torch.autograd.grad(y, [uu, zz], dg)
    assert_close(du16, gu, 8e-3, "act-backward du (post gate)")
    assert_close(K.colsum(e16), gz, 8e-3, "gate gradient (post gate)")


def test_gemm_dropout_replay_and_rate(K):
    M, N, K_ = 512, 768, 64
    A, B = _rand(M, K_, dtype=bf16, seed=1), _rand(N, K_, dtype=bf16, seed=2)
    D0 = torch.empty(M, N, dtype=f32, device="cuda")
    D1 = torch.empty(M, N, dtype=f32, device="cuda")
    K.gemm(A, B, D0, M, N, K_)
    K.gemm(A, B, D1, M, N, K_, dropout_p=0.1, seed=1234, stream_id=3)
    kept = D1 != 0
    rate = 1.0 - kept.float().mean().item()
    assert abs(rate - 0.1) < 0.01, rate
    assert_close(D1[kept], (D0 / 0.9)[kept], 1e-5, "kept values scaled by 1/(1-p)")
    # the cast kernel replays the same mask from (seed, stream, index)
    rep = K.cast_bf16(torch.ones(M, N, device="cuda"), dropout_p=0.1, seed=1234, stream_id=3)
    assert torch.equal(rep != 0, kept)
    rep2 = K.cast_bf16(torch.ones(M, N, device="cuda"), dropout_p=0.1, seed=1235, stream_id=3)
    assert not torch.equal(rep2 != 0, kept)


def test_gemm_rejects_bad_arguments(K):
    A, B = _rand(8, 12, dtype=bf16), _rand(8, 12, dtype=bf16)   # 12 elements = 24-byte pitch: not TMA-able
    with pytest.raises(ValueError):
        K.gemm(A, B, torch.empty(8, 8, device="cuda"), 8, 8, 12)


def test_sgemm_and_dot(K):
    a, b = _rand(37, 50, seed=1), _rand(29, 50, seed=2)
    temp = torch.tensor(0.07, device="cuda")
    out = torch.empty(37, 29, device="cuda")
    K.sgemm(a, b, out, 37, 29, 50, b_trans=True, alpha_dev=temp, alpha_dev_inv=True)
    assert_close(out, a @ b.t() / 0.07, 1e-5, "sgemm nt / temp")
    g = _rand(37, 29, seed=3)
    da = torch.empty_like(a)
    K.sgemm(g, b, da, 37, 50, 29)
    assert_close(da, g @ b, 1e-5, "sgemm nn")
    db = torch.empty_like(b)
    K.sgemm(g, a, db, 29, 50, 37, a_trans=True)
    assert_close(db, g.t() @ a, 1e-5, "sgemm tn")
    d = torch.empty((), device="cuda")
    K.dot(g, out, d, scale=-1.0)
    assert_close(d, -(g * out).sum(), 1e-5, "dot")


# ------------------------------------------------------------------------------------------------ LayerNorm / elementwise
@pytest.mark.parametrize("H", [128, 768, 1536])
@pytest.mark.parametrize("xdt", [f32, bf16])
def test_layernorm(K, H, xdt):
    rows = 333
    x = _rand(rows, H, seed=1, scale=2.0).to(xdt)
    w, b = 1 + 0.1 * _rand(H, seed=2), 0.1 * _rand(H, seed=3)
    eps = 1e-12 if H == 768 else 1e-5
    y32, y16, mean, rstd = K.layernorm_fwd(x, w, b, eps, want_f32=True, want_bf16=True)
    xr = x.float().requires_grad_()
    wr, br = w.clone().requires_grad_(), b.clone().requires_grad_()
    ref = F.layer_norm(xr, (H,), wr, br, eps)
    assert_close(y32, ref, 1e-5, "ln fwd")
    assert_close(y16, ref, 5e-3, "ln fwd bf16")
    dy = _rand(rows, H, seed=4)
    dres = _rand(rows, H, seed=5)
    gx, gw, gb = torch.autograd.grad(ref, [xr, wr, br], dy)
    dgam, dbet = torch.zeros(H, device="cuda"), torch.zeros(H, device="cuda")
    dx32, dx16 = K.layernorm_bwd(dy, x, w, mean, rstd, dres=dres, want_f32=True, want_bf16=True, dgamma=dgam, dbeta=dbet)
    assert_close(dx32, gx + dres, 1e-4, "ln dx (+dres)")
    assert_close(dx16, gx + dres, 5e-3, "ln dx bf16")
    assert_close(dgam, gw, 1e-4, "ln dgamma")
    assert_close(dbet, gb, 1e-4, "ln dbeta")
    dxb, _ = K.layernorm_bwd(dy.to(bf16), x, w, mean, rstd, want_f32=True)
    assert_close(dxb, gx, 8e-3, "ln dx from bf16 dy")


def test_layernorm_dropout_consistency(K):
    rows, H = 64, 768
    x, w, b = _rand(rows, H), torch.ones(H, device="cuda"), torch.zeros(H, device="cuda")
    y0, _, mean, rstd = K.layernorm_fwd(x, w, b, 1e-12)
    y1, _, _, _ = K.layernorm_fwd(x, w, b, 1e-12, dropout_p=0.1, seed=99, stream_id=7)
    kept = y1 != 0
    assert abs(1 - kept.float().mean().item() - 0.1) < 0.02
    assert_close(y1[kept], (y0 / 0.9)[kept], 1e-5, "ln dropout scale")
    dy = torch.ones(rows, H, device="cuda")
    d1, _ = K.layernorm_bwd(dy, x, w, mean, rstd, dropout_p=0.1, seed=99, stream_id=7)
    d0, _ = K.layernorm_bwd(dy * kept / 0.9, x, w, mean, rstd)
    assert_close(d1, d0, 1e-5, "ln bwd replays the forward mask")


def test_casts_colsum_act(K):
    from efficientvlm_b200._lib import ACT_GELU_ERF, ACT_QUICK_GELU
    x = _rand(301, 203, seed=1)
    x16 = K.cast_bf16(x)
    assert torch.equal(x16, x.to(bf16))
    assert torch.equal(K.cast_f32(x16), x16.float())
    # contiguous fast path (flat kernel) vs the generic strided kernel: same rounding, same dropout mask for the same (row, column)
    for rows, cols in ((300, 768), (25216, 768), (7, 8)):
        xc = _rand(rows, cols, seed=5)
        assert torch.equal(K.cast_bf16(xc), xc.to(bf16))
        wide = torch.zeros(rows, cols + 4, device="cuda")
        wide[:, :cols] = xc
        d_flat = K.cast_bf16(xc, dropout_p=0.25, seed=1234, stream_id=3)
        d_strided = K.cast_bf16(wide[:, :cols], dropout_p=0.25, seed=1234, stream_id=3)
        assert torch.equal(d_flat, d_strided)
        if rows * cols > 10000:
            assert abs((d_flat == 0).float().mean().item() - 0.25) < 0.01
    assert_close(K.colsum(x), x.sum(0), 1e-5, "colsum f32")
    assert_close(K.colsum(x16), x16.float().sum(0), 1e-5, "colsum bf16")
    y16 = _rand(301, 203, seed=2, dtype=bf16)
    assert_close(K.coldot(x16, y16), (x16.float() * y16.float()).sum(0), 1e-5, "coldot")
    for act, fn in ((ACT_GELU_ERF, F.gelu), (ACT_QUICK_GELU, lambda t: t * torch.sigmoid(1.702 * t))):
        xr = x.clone().requires_grad_()
        ref = fn(xr)
        assert_close(K.act_fwd(x.contiguous(), act), ref, 1e-5, "act fwd")
        dy = _rand(301, 203, seed=3)
        (gx,) = torch.autograd.grad(ref, xr, dy)
        assert_close(K.act_bwd(dy, x.contiguous(), act), gx, 1e-4, "act bwd")


def test_vit_patchify_and_assemble(K):
    B, R, P, H = 3, 64, 16, 128
    img = _rand(B, 3, R, R, seed=1)
    W = _rand(H, 3, P, P, seed=2, scale=0.05)
    patches = K.im2col_patch(img, P)
    ref = F.conv2d(img.to(bf16).float(), W.to(bf16).float(), stride=P).flatten(2).transpose(1, 2)     # [B, G*G, H]
    got = patches.float() @ W.to(bf16).float().view(H, -1).t()
    assert_close(got.view(B, -1, H), ref, 1e-4, "im2col ordering == conv2d")
    N = (R // P) ** 2 + 1
    cls, pos = _rand(H, seed=3), _rand(N, H, seed=4)
    pe16 = ref.reshape(-1, H).to(bf16).contiguous()
    out = K.vit_assemble_fwd(pe16, cls, pos, B, N, H)
    exp = torch.cat([cls.expand(B, 1, H), pe16.float().view(B, N - 1, H)], 1) + pos[None]
    assert_close(out, exp, 1e-6, "assemble fwd")
    dh = _rand(B, N, H, seed=5)
    dcls, dpos = torch.zeros(H, device="cuda"), torch.zeros(N, H, device="cuda")
    dpatch = K.vit_assemble_bwd(dh, dcls, dpos, B, N, H)
    assert_close(dcls, dh[:, 0].sum(0), 1e-5, "dcls")
    assert_close(dpos, dh.sum(0), 1e-5, "dpos")
    assert torch.equal(dpatch.view(B, N - 1, H), dh[:, 1:].to(bf16))


def test_bert_embed(K):
    V, H, B, L = 211, 128, 4, 9
    word, typ, pos = _rand(V, H, seed=1), _rand(2, H, seed=2), _rand(40, H, seed=3)
    ids = torch.randint(0, V, (B, L), device="cuda")
    tt = torch.randint(0, 2, (B, L), device="cuda")
    out = K.bert_embed_fwd(ids, tt, None, word, typ, pos, 3)
    exp = word[ids] + typ[tt] + pos[3:3 + L][None]
    assert_close(out, exp, 1e-6, "embed fwd (past offset)")
    dout = _rand(B, L, H, seed=4)
    dw, dt, dp = torch.zeros_like(word), torch.zeros_like(typ), torch.zeros_like(pos)
    K.bert_embed_bwd(dout, ids, tt, None, dw, dt, dp, 3)
    ew = torch.zeros_like(word).index_add_(0, ids.view(-1), dout.view(-1, H))
    assert_close(dw, ew, 1e-5, "dword")
    assert_close(dp[3:3 + L], dout.sum(0), 1e-5, "dpos")
    # nn.Embedding(padding_idx=0) semantics (eff_bert.py:173): look-ups of the padding row contribute no gradient
    ids[0, -2:] = 0
    dw2, dt2, dp2 = torch.zeros_like(word), torch.zeros_like(typ), torch.zeros_like(pos)
    K.bert_embed_bwd(dout, ids, tt, None, dw2, dt2, dp2, 3, padding_idx=0)
    emb = torch.nn.Embedding(V, H, padding_idx=0).cuda()
    with torch.no_grad():
        emb.weight.copy_(word)
    emb(ids).backward(dout)
    assert_close(dw2, emb.weight.grad, 1e-5, "dword with padding_idx")
    assert float(dw2[0].abs().max()) == 0.0
    assert_close(dp2, dp, 1e-6, "dpos unaffected by padding_idx")


# ------------------------------------------------------------------------------------------------ attention
def _ref_attention(q, k, v, B, H, Lq, Lk, scale, key_mask=None, causal=False, offset=0, head_z=None):
    qh = q.float().view(B, Lq, H, 64).transpose(1, 2)
    kh = k.float().view(B, Lk, H, 64).transpose(1, 2)
    vh = v.float().view(B, Lk, H, 64).transpose(1, 2)
    s = qh @ kh.transpose(-1, -2) * scale
    if key_mask is not None:
        s = s + key_mask[:, None, None, :]
    if causal:
        i = torch.arange(Lq, device=q.device)[:, None]
        j = torch.arange(Lk, device=q.device)[None, :]
        s = s + (j > i + offset).float() * -10000.0
    p = torch.softmax(s, -1)
    ctx = p @ vh
    if head_z is not None:
        ctx = ctx * head_z.view(1, H, 1, 1)
    return ctx.transpose(1, 2).reshape(B * Lq, H * 64), p


@pytest.mark.parametrize("B,H,Lq,Lk,causal,masked", [(2, 2, 5, 5, False, False), (3, 12, 197, 197, False, False), (2, 4, 40, 197, False, True),
                                                     (2, 3, 40, 40, True, True), (1, 2, 130, 77, False, True), (2, 2, 1, 9, True, False),
                                                     (2, 2, 256, 256, False, False), (1, 2, 40, 577, False, True),
                                                     (1, 2, 300, 300, True, False),
                                                     # 256 < Lk <= 1024: the two-sweep tcgen05 kernel (attention_tc_long.cu)
                                                     (2, 12, 901, 901, False, False), (2, 3, 16, 901, False, True),
                                                     (1, 2, 577, 577, False, True), (1, 2, 300, 1024, False, False),
                                                     (1, 1, 129, 257, False, True),
                                                     # tiny problems with many (item, head) pairs: the warp-per-pair forward (answer decoders)
                                                     (300, 4, 4, 4, True, False), (200, 6, 1, 9, True, False), (128, 12, 16, 16, False, True),
                                                     (90, 12, 4, 16, False, True),
                                                     # beyond every tcgen05 envelope (Lk > 1024): the tiled mma.sync kernels still serve it
                                                     (1, 1, 70, 1100, False, True)])
def test_attention_forward_backward(K, B, H, Lq, Lk, causal, masked):
    E = H * 64
    qkv = _rand(B * max(Lq, Lk), 3 * E, dtype=bf16, seed=1, scale=0.7)
    q = qkv[:B * Lq, :E]
    k = qkv[:B * Lk, E:2 * E]
    v = qkv[:B * Lk, 2 * E:]
    key_mask = None
    if masked:
        key_mask = torch.zeros(B, Lk, device="cuda")
        key_mask[:, Lk - 3:] = -10000.0
    head_z = torch.rand(H, device="cuda")
    head_z[0] = 0.0
    offset = Lk - Lq if causal else 0
    ctx, probs, lse = K.attention_fwd(q, k, v, B, H, Lq, Lk, 0.125, key_mask=key_mask, causal=causal, causal_offset=offset, head_z=head_z,
                                      want_probs=True)
    qr, kr, vr = (t.float().detach().clone().requires_grad_() for t in (q, k, v))
    zr = head_z.clone().requires_grad_()
    rctx, rp = _ref_attention(qr, kr, vr, B, H, Lq, Lk, 0.125, key_mask, causal, offset, zr)
    assert_close(probs, rp, 3e-3, "probs")
    assert_close(ctx, rctx, 1e-2, "ctx")
    ctx2, none_probs, lse2 = K.attention_fwd(q, k, v, B, H, Lq, Lk, 0.125, key_mask=key_mask, causal=causal, causal_offset=offset,
                                             head_z=head_z, want_probs=False)
    assert none_probs is None
    if Lk <= 256 and Lq != 1:
        assert torch.equal(ctx2, ctx)
    else:   # single query without a map: the K/V stream kernel (attention_decode.cu), another summation order;  long keys: the row sum is accumulated in sweep 1 (with P output) or sweep 2 (without) -> last-bit differences
        assert_close(ctx2, rctx, 1e-2, "ctx (no probs)")
        assert_close(lse2, lse, 1e-5, "lse (no probs)")
    # backward with a gradient arriving on the returned probabilities too (attention-map distillation)
    dctx = _rand(B * Lq, E, seed=2, scale=0.5).to(bf16)
    dprobs = _rand(B, H, Lq, Lk, seed=3, scale=0.3)
    gq, gk, gv, gz = torch.autograd.grad([rctx, rp], [qr, kr, vr, zr], [dctx.float(), dprobs], retain_graph=True)
    dqkv = torch.zeros(B * max(Lq, Lk), 3 * E, dtype=bf16, device="cuda")
    dz = torch.zeros(H, device="cuda")
    K.attention_bwd(q, k, v, ctx, lse, dctx, dqkv[:B * Lq, :E], dqkv[:B * Lk, E:2 * E], dqkv[:B * Lk, 2 * E:], B, H, Lq, Lk, 0.125,
                    probs=probs, dprobs=dprobs, key_mask=key_mask, causal=causal, causal_offset=offset, head_z=head_z, dhead_z=dz)
    assert_close(dqkv[:B * Lq, :E], gq, BF_TOL, "dq")
    assert_close(dqkv[:B * Lk, E:2 * E], gk, BF_TOL, "dk")
    assert_close(dqkv[:B * Lk, 2 * E:], gv, BF_TOL, "dv")
    assert_close(dz, gz, BF_TOL, "dhead_z")
    # and without it (recompute-from-lse path only)
    gq2, gk2, gv2 = torch.autograd.grad(rctx, [qr, kr, vr], dctx.float())
    K.attention_bwd(q, k, v, ctx, lse, dctx, dqkv[:B * Lq, :E], dqkv[:B * Lk, E:2 * E], dqkv[:B * Lk, 2 * E:], B, H, Lq, Lk, 0.125,
                    key_mask=key_mask, causal=causal, causal_offset=offset, head_z=head_z)
    assert_close(dqkv[:B * Lq, :E], gq2, BF_TOL, "dq (no dprobs)")
    assert_close(dqkv[:B * Lk, 2 * E:], gv2, BF_TOL, "dv (no dprobs)")


@pytest.mark.parametrize("L", [128, 512])
def test_attention_dropout_statistics_and_replay(K, L):
    B, H = 2, 2
    E = H * 64
    q, k = _rand(B * L, E, dtype=bf16, seed=1, scale=0.1), _rand(B * L, E, dtype=bf16, seed=2, scale=0.1)
    v = torch.ones(B * L, E, dtype=bf16, device="cuda")
    ctx0, _, lse = K.attention_fwd(q, k, v, B, H, L, L, 0.125)
    ctx1, _, _ = K.attention_fwd(q, k, v, B, H, L, L, 0.125, dropout_p=0.1, seed=77, stream_id=0)
    # E[dropout(P) @ 1] = 1; per-row deviation is small but non-zero
    assert abs(ctx1.float().mean().item() - 1.0) < 0.02
    assert (ctx1.float() - ctx0.float()).abs().max().item() > 1e-3
    ctx2, _, _ = K.attention_fwd(q, k, v, B, H, L, L, 0.125, dropout_p=0.1, seed=77, stream_id=0)
    assert torch.equal(ctx1, ctx2)
    # backward replays the same mask: dV = (D o P)^T dO, so with dO = 1, sum_j dV_j = sum_i ctx-row sums
    dctx = torch.ones(B * L, E, dtype=bf16, device="cuda")
    dq, dk, dv = (torch.zeros(B * L, E, dtype=bf16, device="cuda") for _ in range(3))
    K.attention_bwd(q, k, v, ctx1, lse, dctx, dq, dk, dv, B, H, L, L, 0.125, dropout_p=0.1, seed=77, stream_id=0)
    assert abs(dv.float().view(B, L, E).sum(1).mean().item() - ctx1.float().view(B, L, E).sum(1).mean().item()) < 0.5


# ------------------------------------------------------------------------------------------------ losses
def test_mse_pairs(K):
    S = [_rand(4, 197, 64, seed=i) for i in range(3)] + [_rand(2, 12, 33, 33, seed=9)]
    T = [_rand(4, 197, 64, seed=10 + i) for i in range(3)] + [_rand(2, 12, 33, 33, seed=19)]
    S[1] = S[1].to(bf16)
    T[2] = T[2].to(bf16)
    W = [1.0, 0.5, 2.0, 33.0]
    out = K.mse_pairs_fwd(S, T, W)
    ref = torch.stack([F.mse_loss(s.float(), t.float()) * w for s, t, w in zip(S, T, W)])
    assert_close(out, ref, 1e-5, "mse pairs")
    dout = torch.tensor([1.0, 2.0, 0.5, 0.25], device="cuda")
    grads = K.mse_pairs_bwd(S, T, W, dout, [True, True, False, True])
    assert grads[2] is None
    for i in (0, 1, 3):
        exp = dout[i] * W[i] * 2 * (S[i].float() - T[i].float()) / S[i].numel()
        assert_close(grads[i], exp, 1e-5, "mse grad %d" % i)


def test_softmax_losses(K):
    rows, V = 37, 30522
    logits = _rand(rows, V, seed=1, scale=3.0)
    labels = torch.randint(0, V, (rows,), device="cuda")
    labels[::5] = -100
    for ls in (0.0, 0.1):
        lr = logits.clone().requires_grad_()
        loss, lse = K.xent_fwd(logits, labels, -100, ls)
        ref = F.cross_entropy(lr, labels, reduction="none", ignore_index=-100, label_smoothing=0.0)
        if ls > 0:
            logp = F.log_softmax(lr, 1)
            oh = torch.full_like(logp, ls / V).scatter_(1, labels.clamp(min=0).unsqueeze(1), 1 - ls)
            ref = -(logp * oh).sum(1) * (labels != -100)
        assert_close(loss, ref, 1e-5, "xent rows ls=%g" % ls)
        g = _rand(rows, seed=2)
        (gref,) = torch.autograd.grad(ref, lr, g)
        assert_close(K.xent_bwd(logits, labels, lse, g, -100, ls), gref, 1e-4, "xent grad")
    t = _rand(rows, V, seed=3, scale=3.0)
    for inv_t in (1.0, 0.5):
        sr = logits.clone().requires_grad_()
        kl, ls_, lt = K.kl_fwd(logits, t, inv_t)
        ref = F.kl_div(F.log_softmax(sr * inv_t, -1), F.softmax(t * inv_t, -1), reduction="none").sum(-1)
        assert_close(kl, ref, 1e-4, "kl rows")
        g = _rand(rows, seed=4)
        (gref,) = torch.autograd.grad(ref, sr, g)
        assert_close(K.kl_bwd(logits, t, ls_, lt, g, inv_t), gref, 1e-4, "kl grad")
    small = _rand(16, 16, seed=5, scale=4.0)
    lab = torch.rand(16, 16, device="cuda")
    lab = lab / lab.sum(1, keepdim=True)
    sr = small.clone().requires_grad_()
    loss, lse = K.soft_xent_fwd(small, lab)
    ref = -(F.log_softmax(sr, 1) * lab).sum(1)
    assert_close(loss, ref, 1e-5, "soft xent")
    g = _rand(16, seed=6)
    (gref,) = torch.autograd.grad(ref, sr, g)
    assert_close(K.soft_xent_bwd(small, lab, lse, g), gref, 1e-4, "soft xent grad")


def test_reduce_l2norm_itm_sampling(K):
    x = _rand(100003, seed=1)
    assert_close(K.reduce_sum(x, 0.5), 0.5 * x.sum(), 1e-4, "reduce sum")
    f = _rand(33, 256, seed=2)
    fr = f.clone().requires_grad_()
    y, inv = K.l2norm_fwd(f)
    ref = F.normalize(fr, dim=-1)
    assert_close(y, ref, 1e-6, "l2norm")
    dy = _rand(33, 256, seed=3)
    (g,) = torch.autograd.grad(ref, fr, dy)
    assert_close(K.l2norm_bwd(dy, y, inv), g, 1e-5, "l2norm grad")
    # ITM negatives: never the positive / same-idx entry, distribution follows softmax + 1e-5
    B = 64
    sim = _rand(B, B, seed=4, scale=2.0)
    idx = torch.arange(B, device="cuda") // 2
    for ids in (None, idx):
        u = torch.rand(B, device="cuda")
        neg = K.itm_sample_neg(sim, ids, u)
        assert neg.min() >= 0 and neg.max() < B
        if ids is None:
            assert (neg != torch.arange(B, device="cuda")).all()
        else:
            assert (ids[neg] != ids).all()
        w = torch.softmax(sim, 1) + 1e-5
        ex = torch.eye(B, device="cuda", dtype=torch.bool) if ids is None else ids[:, None] == ids[None, :]
        w = w.masked_fill(ex, 0)
        c = torch.cumsum(w, 1)
        exp = (c > (u * c[:, -1])[:, None]).float().argmax(1)
        assert (neg == exp).float().mean() > 0.95     # identical inverse-CDF draw up to fp32 rounding at bin edges


# ------------------------------------------------------------------------------------------------ L0 / optimizer
def test_l0_kernels_against_golden(K):
    from oracle import xvlm_oracle as O
    g = load_golden("l0_tiny")
    for t in g["types"]:
        loga = g["logas"][t].cuda()
        u = g["eps"][t].cuda()
        z = K.l0_sample_fwd(loga, u, 2.0 / 3.0)
        assert_close(z.view(g["shapes"][t]), g["zs_train"][t + "_z"], 1e-5, "z " + t)
        assert torch.equal(z == 0, g["zs_train"][t + "_z"].cuda().view_as(z) == 0)
        mask, kept = K.l0_deterministic(loga, 2.0 / 3.0, 0.8)
        assert torch.equal(mask.cpu().view(g["zs_eval"][t + "_z"].shape), g["zs_eval"][t + "_z"]), "deterministic mask bit-exact: " + t
        assert torch.equal(kept.cpu().long(), g["zs_eval"][t + "_z"].view(loga.shape[0], -1).sum(1).long())
        lr = g["logas"][t].clone().requires_grad_()
        zr = O.l0_sample_z(lr, g["eps"][t])
        dz = torch.rand(zr.shape)
        (gr,) = torch.autograd.grad(zr, lr, dz)
        assert_close(K.l0_sample_bwd(loga, u, dz.cuda(), 2.0 / 3.0), gr, 1e-4, "dloga " + t)
    out = torch.zeros((), device="cuda")
    for t in g["types"]:
        K.l0_expected_fwd(g["logas"][t].cuda().contiguous(), 2.0 / 3.0, float(g["params_per_dim"][t]), out, True)
    es = 1 - out / g["prunable_model_size"]
    assert_close(es, g["expected_sparsity"], 1e-5, "expected sparsity")
    x = _rand(1000, seed=1, scale=10)
    K.clamp_(x, math.log(1e-2), math.log(1e2))
    assert x.min() >= math.log(1e-2) - 1e-6 and x.max() <= math.log(1e2) + 1e-6


def test_adamw_matches_hf_semantics(K):
    n = 10007
    p, g = _rand(n, seed=1), _rand(n, seed=2)
    m, v = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    p_ref, m_ref, v_ref = p.clone(), m.clone(), v.clone()
    p16 = torch.empty(n, dtype=bf16, device="cuda")
    lr, b1, b2, eps, wd = 1e-3, 0.9, 0.999, 1e-6, 0.01
    coef = torch.tensor(0.5, device="cuda")
    for step in (1, 2, 3):
        K.adamw_step([dict(p=p, g=g, m=m, v=v, p_bf16=p16, lr=lr, beta1=b1, beta2=b2, eps=eps, weight_decay=wd, step=step)], coef)
        gg = g * 0.5
        m_ref.mul_(b1).add_(gg, alpha=1 - b1)
        v_ref.mul_(b2).addcmul_(gg, gg, value=1 - b2)
        step_size = lr * math.sqrt(1 - b2 ** step) / (1 - b1 ** step)
        p_ref.addcdiv_(m_ref, v_ref.sqrt().add_(eps), value=-step_size)
        p_ref.add_(p_ref, alpha=-lr * wd)
    assert_close(p, p_ref, 1e-5, "adamw params")
    assert torch.equal(p16, p.to(bf16))
    ss = torch.zeros(1, device="cuda")
    K.sumsq(g, ss)
    assert_close(ss, (g * g).sum(), 1e-4, "sumsq")
    c = torch.empty(1, device="cuda")
    K.clip_coef(ss, 1.0, c)
    assert_close(c, torch.clamp(1.0 / (g.norm() + 1e-6), max=1.0), 1e-5, "clip coef")


def test_attention_shared_kv_and_packed_query_items(K):
    """kv_index (query item -> K/V item) and pack_items (query items that share a K/V item share one 128-row tile) must give the
    same forward outputs and gradients as materialising K/V per query item; dK/dV of a group fold back per K/V item."""
    torch.manual_seed(0)
    B, H, Lq, Lk, nkv = 8, 2, 40, 197, 3
    E = H * 64
    dev = "cuda"
    q = torch.randn(B * Lq, E, device=dev).to(bf16)
    kk = torch.randn(nkv * Lk, E, device=dev).to(bf16)
    vv = torch.randn(nkv * Lk, E, device=dev).to(bf16)
    kv_index = torch.tensor([0, 1, 0, 2, 0, 1, 2, 2], device=dev, dtype=torch.int32)
    mask = torch.zeros(B, Lk, device=dev)
    mask[:, 190:] = -10000.0
    idx = kv_index.long()
    k_full = kk.view(nkv, Lk, E).index_select(0, idx).reshape(B * Lk, E).contiguous()
    v_full = vv.view(nkv, Lk, E).index_select(0, idx).reshape(B * Lk, E).contiguous()
    ctx0, P0, lse0 = K.attention_fwd(q, k_full, v_full, B, H, Lq, Lk, 0.125, key_mask=mask, want_probs=True)
    # groups: kv 0 -> items (0, 2, 4); kv 1 -> (1, 5); kv 2 -> (3, 6, 7)
    pack = torch.tensor([[0, 2, 4], [1, 5, -1], [3, 6, 7]], device=dev, dtype=torch.int32)
    for kwargs in (dict(kv_index=kv_index), dict(kv_index=kv_index, pack_items=pack)):
        ctx1, P1, lse1 = K.attention_fwd(q, kk, vv, B, H, Lq, Lk, 0.125, key_mask=mask, want_probs=True, **kwargs)
        assert_close(ctx1.float(), ctx0.float(), 1e-2, "ctx %s" % list(kwargs))
        assert_close(P1, P0, 1e-4, "probs %s" % list(kwargs))
        assert_close(lse1, lse0, 1e-4, "lse %s" % list(kwargs))
    dctx = torch.randn(B * Lq, E, device=dev).to(bf16)
    dP = torch.randn(B, H, Lq, Lk, device=dev) * 1e-2
    dq0, dk0, dv0 = torch.empty_like(q), torch.empty_like(k_full), torch.empty_like(v_full)
    K.attention_bwd(q, k_full, v_full, ctx0, lse0, dctx, dq0, dk0, dv0, B, H, Lq, Lk, 0.125, probs=P0, dprobs=dP, key_mask=mask)
    ref_dk = torch.zeros(nkv, Lk * E, device=dev).index_add_(0, idx, dk0.float().view(B, Lk * E))
    ref_dv = torch.zeros(nkv, Lk * E, device=dev).index_add_(0, idx, dv0.float().view(B, Lk * E))
    # (a) shared K/V, one CTA per query item: dk/dv per item, folded by kv_index
    dq1, dk1, dv1 = torch.empty_like(q), torch.empty_like(k_full), torch.empty_like(v_full)
    K.attention_bwd(q, kk, vv, ctx0, lse0, dctx, dq1, dk1, dv1, B, H, Lq, Lk, 0.125, probs=P0, dprobs=dP, key_mask=mask, kv_index=kv_index)
    assert_close(dq1.float(), dq0.float(), 2e-2, "dq shared kv")
    assert_close(K.index_fold_rows(dk1.view(B, Lk * E), kv_index, nkv).float(), ref_dk, 2e-2, "dk folded")
    assert_close(K.index_fold_rows(dv1.view(B, Lk * E), kv_index, nkv).float(), ref_dv, 2e-2, "dv folded")
    # (b) packed: dk/dv per group
    G = pack.shape[0]
    dq2 = torch.empty_like(q)
    dk2, dv2 = torch.empty(G * Lk, E, device=dev, dtype=bf16), torch.empty(G * Lk, E, device=dev, dtype=bf16)
    K.attention_bwd(q, kk, vv, ctx0, lse0, dctx, dq2, dk2, dv2, B, H, Lq, Lk, 0.125, probs=P0, dprobs=dP, key_mask=mask, kv_index=kv_index,
                    pack_items=pack)
    assert_close(dq2.float(), dq0.float(), 2e-2, "dq packed")
    group_kv = kv_index.index_select(0, pack[:, 0].long()).contiguous()
    assert_close(K.index_fold_rows(dk2.view(G, Lk * E), group_kv, nkv).float(), ref_dk, 2e-2, "dk packed+folded")
    assert_close(K.index_fold_rows(dv2.view(G, Lk * E), group_kv, nkv).float(), ref_dv, 2e-2, "dv packed+folded")


@pytest.mark.parametrize("p_drop", [0.0, 0.1])
def test_attention_block_diagonal_pack(K, p_drop):
    """pack_own_kv: three short self-attention problems share one 128 x 128 tile (block-diagonal mask); forward outputs,
    dq, dk, dv must equal the one-CTA-per-item launch (dropout: both draw each item's mask by its own keys, so the masks match)."""
    torch.manual_seed(1)
    B, H, L = 8, 2, 40
    E = H * 64
    dev = "cuda"
    qkv = torch.randn(B * L, 3 * E, device=dev).to(bf16)
    q, k, v = qkv[:, :E], qkv[:, E:2 * E], qkv[:, 2 * E:]
    mask = torch.zeros(B, L, device=dev)
    mask[2, 30:] = -10000.0
    pack = torch.tensor([[0, 1, 2], [3, 4, 5], [6, 7, -1]], device=dev, dtype=torch.int32)
    ctx0, P0, lse0 = K.attention_fwd(q, k, v, B, H, L, L, 0.125, key_mask=mask, want_probs=True)
    ctx1, P1, lse1 = K.attention_fwd(q, k, v, B, H, L, L, 0.125, key_mask=mask, want_probs=True, pack_items=pack, pack_own_kv=True)
    assert_close(ctx1.float(), ctx0.float(), 1e-2, "ctx")
    assert_close(P1, P0, 1e-4, "probs")
    assert_close(lse1, lse0, 1e-4, "lse")
    dctx = torch.randn(B * L, E, device=dev).to(bf16)
    dP = torch.randn(B, H, L, L, device=dev) * 1e-2
    outs = []
    for kw in (dict(), dict(pack_items=pack, pack_own_kv=True)):
        c, P, lse = K.attention_fwd(q, k, v, B, H, L, L, 0.125, key_mask=mask, want_probs=True, dropout_p=p_drop, seed=77, stream_id=3, **kw)
        dqkv = torch.zeros(B * L, 3 * E, device=dev, dtype=bf16)
        K.attention_bwd(q, k, v, c, lse, dctx, dqkv[:, :E], dqkv[:, E:2 * E], dqkv[:, 2 * E:], B, H, L, L, 0.125, probs=P, dprobs=dP,
                        key_mask=mask, dropout_p=p_drop, seed=77, stream_id=3, **kw)
        outs.append((c, dqkv))
    assert_close(outs[1][0].float(), outs[0][0].float(), 1e-2, "ctx (bwd run)")
    assert_close(outs[1][1].float(), outs[0][1].float(), 2e-2, "dq|dk|dv")


def test_weight_shadow_follows_data_inplace_optimizer():
    """An optimizer that updates through `p.data.add_()` (transformers-4.12.5 AdamW, the reference's optim.py:1,67) changes neither
    `_version` nor `data_ptr()`; the global optimizer post-step hook (ops._torch_optimizer_stepped) must still refresh the bf16 shadow."""
    from efficientvlm_b200 import ops

    class DataSGD(torch.optim.Optimizer):
        def __init__(self, params):
            super().__init__(params, dict(lr=0.5))

        def step(self, closure=None):
            for g in self.param_groups:
                for p in g["params"]:
                    p.data.add_(p.grad.data, alpha=-g["lr"])
    w = torch.nn.Parameter(torch.randn(16, 32, device="cuda"))
    s0 = ops.weight_bf16(w).clone()
    assert torch.equal(s0, w.detach().to(torch.bfloat16))
    w.grad = torch.ones_like(w)
    DataSGD([w]).step()
    s1 = ops.weight_bf16(w)
    assert torch.equal(s1, w.detach().to(torch.bfloat16)) and not torch.equal(s1, s0)


# ------------------------------------------------------------------------------------------------ zero-skip (north star bullet 1)
def test_compact_index_gather_scatter_are_exact(K):
    """Index work of the zero-skip path: bit-exact against torch.nonzero / index_select / index_add."""
    g = torch.Generator().manual_seed(5)
    for n, frac in ((3072, 0.17), (3072, 0.6), (256, 0.35), (1000, 0.0), (512, 1.0), (70000 // 2, 0.5)):
        z = torch.rand(n, generator=g)
        z[torch.rand(n, generator=g) < frac] = 0
        zc = z.cuda()
        idx, cnt = K.compact_index(zc)
        kept = torch.nonzero(z != 0).flatten()
        drop = torch.nonzero(z == 0).flatten()
        assert int(cnt) == kept.numel()
        assert torch.equal(idx.cpu().long(), torch.cat([kept, drop])), "kept positions first (ascending), dropped after (ascending)"
        W = torch.randn(n, 40, generator=g).to(torch.bfloat16).cuda()
        Wc = K.gather_rows(W, idx, cnt)
        ref = torch.zeros_like(W)
        ref[:kept.numel()] = W[kept.cuda()]
        assert torch.equal(Wc, ref)
        v = torch.randn(n, generator=g).cuda()
        vc = K.gather_rows(v, idx, cnt)
        assert torch.equal(vc[:kept.numel()], v[kept.cuda()]) and float(vc[kept.numel():].abs().sum()) == 0
        W2 = torch.randn(24, n, generator=g).to(torch.bfloat16).cuda()
        W2c = K.gather_cols(W2, idx, cnt)
        ref2 = torch.zeros_like(W2)
        ref2[:, :kept.numel()] = W2[:, kept.cuda()]
        assert torch.equal(W2c, ref2)
        src = torch.randn(n, 40, generator=g).cuda()
        dst0 = torch.randn(n, 40, generator=g).cuda()
        dst = dst0.clone()
        K.scatter_rows_add(src, idx, cnt, dst, accumulate=True)
        want = dst0.clone()
        want[kept.cuda()] += src[:kept.numel()]
        assert torch.equal(dst, want)
        K.scatter_rows_add(src, idx, cnt, dst, accumulate=False)
        want = torch.zeros_like(dst0)
        want[kept.cuda()] = src[:kept.numel()]
        assert torch.equal(dst, want)
        srcc = torch.randn(24, n, generator=g).cuda()
        d2 = torch.zeros(24, n).cuda()
        K.scatter_cols_add(srcc, idx, cnt, d2, accumulate=True)
        want2 = torch.zeros(24, n).cuda()
        want2[:, kept.cuda()] = srcc[:, :kept.numel()]
        assert torch.equal(d2, want2)


def test_greedy_select_matches_the_loop_statements(K):
    """`evlm_greedy_select` against the decode loop's own statements (eff_bert.py:1510-1538, greedy branch): argmax (first maximal
    index on ties), log_softmax gathered at it, the padded token for finished sentences and the end-of-sequence bookkeeping —
    ids bit-exact, score to fp32 rounding; strided logits rows (the [B, L, V] logits' last position)."""
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(11)
    for rows, vocab, eos in ((32, 30522, [102]), (5, 97, [3, 7]), (1, 1, []), (9, 1000, [0, 1, 2, 3])):
        full = (torch.randn(rows, 2, vocab, generator=g) * 4).cuda()
        logits = full[:, -1, :]
        if vocab > 10:
            logits[0, 5] = logits[0, 9] = logits[0].max() + 1          # a tie: the first index wins
            logits[rows - 1, eos[0] if eos else 0] = 100.0             # a sentence that ends now
        unfinished = (torch.rand(rows, generator=g) < 0.7).long().cuda()
        pad = 0
        nt, sc, add, un = K.greedy_select(logits, unfinished, pad, eos)
        want_nt = torch.argmax(logits, dim=-1)
        want_sc = torch.gather(F.log_softmax(logits, dim=-1), -1, want_nt.unsqueeze(-1))
        want_add = want_nt * unfinished + pad * (1 - unfinished)
        want_un = unfinished
        for e in eos:
            want_un = want_un.mul(want_add.ne(e).long())
        assert torch.equal(nt, want_nt) and torch.equal(add, want_add) and torch.equal(un, want_un)
        assert sc.shape == want_sc.shape
        assert_close(sc, want_sc, 1e-5, "log-softmax score")


def test_attention_single_query_decode_kernel(K):
    """Lq == 1 without a returned map (decode steps) runs on `attn_fwd_decode_kernel` (csrc/attention_decode.cu): context and row
    log-sum-exp against an fp32 torch statement for self-attention cache lengths (1..20), the caption decoder's 577 image keys and
    VQA-480's 901, with key masks, head gates, shared K/V items (kv_index) and a KV cache with spare rows (kv_item_rows)."""
    g = torch.Generator().manual_seed(5)
    H, scale = 12, 0.125
    for B, Lk, n_kv, cap in ((32, 577, 32, 0), (3, 1, 3, 0), (5, 20, 5, 36), (24, 901, 6, 0), (7, 33, 7, 64)):
        rows = cap or Lk
        q = torch.randn(B, H * 64, generator=g).to(torch.bfloat16).cuda()
        kc = torch.randn(n_kv, rows, H * 64, generator=g).to(torch.bfloat16).cuda()
        vc = torch.randn(n_kv, rows, H * 64, generator=g).to(torch.bfloat16).cuda()
        mask = torch.zeros(B, Lk)
        mask[torch.rand(B, Lk, generator=g) < 0.2] = -10000.0
        mask[:, 0] = 0
        mask = mask.cuda()
        hz = torch.rand(H, generator=g).cuda()
        kv_index = (torch.arange(B) % n_kv).int().cuda() if n_kv != B else None
        ctx, probs, lse = K.attention_fwd(q, kc.view(n_kv * rows, H * 64), vc.view(n_kv * rows, H * 64), B, H, 1, Lk, scale, key_mask=mask,
                                          head_z=hz, kv_index=kv_index, kv_item_rows=cap)
        assert probs is None
        item = kv_index.long() if kv_index is not None else torch.arange(B).cuda()
        kf = kc[item, :Lk].float().view(B, Lk, H, 64).permute(0, 2, 1, 3)
        vf = vc[item, :Lk].float().view(B, Lk, H, 64).permute(0, 2, 1, 3)
        s = torch.einsum("bhd,bhkd->bhk", q.float().view(B, H, 64), kf) * scale + mask[:, None, :]
        want = torch.einsum("bhk,bhkd->bhd", torch.softmax(s, -1), vf) * hz[None, :, None]
        assert_close(ctx.float().view(B, H, 64), want, 8e-3, "decode context B %d Lk %d" % (B, Lk))
        assert_close(lse.view(B, H), torch.logsumexp(s, -1), 1e-4, "decode lse")
    # the same problem through the tile kernels (profiling knob off in a subprocess is overkill: compare with the map-returning call)
    B, Lk = 4, 50
    q = torch.randn(B, H * 64, generator=g).to(torch.bfloat16).cuda()
    k = torch.randn(B * Lk, H * 64, generator=g).to(torch.bfloat16).cuda()
    v = torch.randn(B * Lk, H * 64, generator=g).to(torch.bfloat16).cuda()
    c1, _, l1 = K.attention_fwd(q, k, v, B, H, 1, Lk, scale)
    c2, p2, l2 = K.attention_fwd(q, k, v, B, H, 1, Lk, scale, want_probs=True)
    assert_close(c1.float(), c2.float(), 8e-3, "decode kernel vs tile kernel")
    assert_close(l1, l2, 1e-4, "lse")


def test_gemm_small_m_weight_stream_path(K):
    """M <= 32 forward products (the single-token decode steps) run on `gemm_skinny_kernel` (csrc/gemm_skinny.cu): every forward
    epilogue option against an fp32 torch statement, ragged M / N / K (K only needs to be a multiple of 8), strided rows, and
    against the tcgen05 kernel on the same operands (M padded past the switch-over)."""
    g = torch.Generator().manual_seed(31)
    for M, N, Kd in ((32, 768, 768), (32, 768, 3072), (32, 3072, 768), (24, 2304, 768), (1, 768, 768), (17, 30522, 768), (32, 100, 40),
                     (5, 9, 8)):
        Afull = torch.randn(40, Kd + 8, generator=g).to(torch.bfloat16).cuda()
        A = Afull[:M, :Kd]                                            # strided rows (lda = Kd + 8)
        B = (torch.randn(N, Kd, generator=g) * 0.05).to(torch.bfloat16).cuda()
        bias = torch.randn(N, generator=g).cuda()
        res = torch.randn(M, N, generator=g).cuda()
        gate = torch.rand(N, generator=g).cuda()
        ref0 = A.float() @ B.float().t()
        for dt in (torch.float32, torch.bfloat16):
            tol = 1e-4 if dt == torch.float32 else 8e-3
            D = torch.full((M, N), float("nan"), device="cuda", dtype=dt)
            K.gemm(A, B, D, M, N, Kd)
            assert_close(D.float(), ref0, tol, "plain %s %s" % ((M, N, Kd), dt))
            D = torch.full((M, N), float("nan"), device="cuda", dtype=dt)
            K.gemm(A, B, D, M, N, Kd, bias=bias, residual=res, alpha=0.125, alpha_cols=N // 3)
            want = ref0 + bias
            want[:, :N // 3] *= 0.125
            assert_close(D.float(), want + res, tol, "bias + q-scale + residual %s %s" % ((M, N, Kd), dt))
        for act, fn in ((1, lambda x: x * torch.sigmoid(1.702 * x)), (2, lambda x: torch.nn.functional.gelu(x))):
            for gate_mode in (0, 1, 2):
                D = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
                aux = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
                K.gemm(A, B, D, M, N, Kd, bias=bias, act=act, gate=gate if gate_mode else None, gate_mode=gate_mode, aux_out=aux)
                u = ref0 + bias
                want = fn(u * gate) if gate_mode == 1 else (fn(u) * gate if gate_mode == 2 else fn(u))
                assert_close(aux.float(), u, 8e-3, "saved pre-activation")
                assert_close(D.float(), want, 8e-3, "act %d gate mode %d %s" % (act, gate_mode, (M, N, Kd)))
        # the tcgen05 kernel on the same operands (33 rows: past the small-M switch-over)
        if Kd % 64 == 0 and N % 8 == 0:
            A33 = torch.zeros(33, Kd, dtype=torch.bfloat16, device="cuda")
            A33[:M] = A
            D33 = torch.empty(33, N, device="cuda")
            K.gemm(A33, B, D33, 33, N, Kd, bias=bias)
            D = torch.empty(M, N, device="cuda")
            K.gemm(A, B, D, M, N, Kd, bias=bias)
            assert_close(D, D33[:M], 1e-5, "same as the tcgen05 path up to fp32 summation order")


def test_gemm_device_side_limits(K):
    """m / n / k limits read from device memory: the scheduled part equals the dense product on the leading rows / columns / k; a
    k limit of 0 leaves D = epilogue(0) = bias + residual."""
    g = torch.Generator().manual_seed(9)
    M, N, Kd = 700, 640, 520
    A = torch.randn(M, Kd, generator=g).to(torch.bfloat16).cuda()
    B = torch.randn(N, Kd, generator=g).to(torch.bfloat16).cuda()
    bias = torch.randn(N, generator=g).cuda()
    res = torch.randn(M, N, generator=g).cuda()
    for lim in (1, 129, 300, 513, 640):
        cnt = torch.tensor([lim], dtype=torch.int32, device="cuda")
        D = torch.full((M, N), float("nan"), device="cuda")
        K.gemm(A, B, D, M, N, Kd, bias=bias, n_limit=cnt)
        ref = A.float() @ B.float().t() + bias
        assert_close(D[:, :lim], ref[:, :lim], 1e-4, "n_limit %d" % lim)
        if lim < 512:
            assert bool(torch.isnan(D[:, 512:]).all()), "tiles beyond the limit are not touched"
        D = torch.full((M, N), float("nan"), device="cuda")
        K.gemm(A, B, D, M, N, Kd, m_limit=cnt)
        assert_close(D[:lim], (A.float() @ B.float().t())[:lim], 1e-4, "m_limit %d" % lim)
    for lim in (0, 1, 64, 65, 300, 520):
        cnt = torch.tensor([lim], dtype=torch.int32, device="cuda")
        A0 = A.clone()
        k_up = min(Kd, (lim + 63) // 64 * 64)
        A0[:, lim:] = 0          # the compacted operands are zero beyond the count (up to the 64-wide k block the kernel reads)
        D = torch.empty(M, N, device="cuda")
        K.gemm(A0, B, D, M, N, Kd, bias=bias, residual=res, k_limit=cnt)
        ref = A.float()[:, :lim] @ B.float()[:, :lim].t() + bias + res
        assert_close(D, ref, 1e-4, "k_limit %d (reads k < %d)" % (lim, k_up))


@pytest.mark.parametrize("zero_frac", [0.17, 0.35, 0.6, 1.0])
def test_ffn_zero_skip_equals_dense_gated_path(K, zero_frac):
    """VERDICT r1 row N1: the skip path == the dense gated path — layer output, every parameter gradient and d log-alpha through the
    hard-concrete sampler — at CLIP-ViT-B / BERT-base FFN width with 17 / 35 / 60 / 100 % of the columns gated to exactly 0."""
    from efficientvlm_b200 import ops
    from efficientvlm_b200.eff_bert import BertConfig, BertLayer
    from efficientvlm_b200.eff_vit import CLIPEncoderLayer
    from oracle.det_init import det_init_module_
    H, I, nh, B, N = 768, 3072, 12, 4, 50
    g = torch.Generator().manual_seed(17)
    vit = CLIPEncoderLayer(H, "quick_gelu", nh, 0.0, I).eval()
    det_init_module_(vit)
    cfg = BertConfig(vocab_size=64, hidden_size=H, num_hidden_layers=1, num_attention_heads=nh, intermediate_size=I, max_position_embeddings=64)
    cfg.fusion_layer, cfg.encoder_width = 1, H
    bert = BertLayer(cfg, 0).eval()
    det_init_module_(bert)
    vit.cuda()
    bert.cuda()
    x = torch.randn(B, N, H, generator=g).cuda()
    u = torch.rand(2, I, generator=g).clamp(1e-4, 1 - 1e-4).cuda()
    # log-alphas: a `zero_frac` share far enough below 0 that the stretched hard-concrete sample clamps to exactly 0
    loga0 = torch.randn(2, I, generator=g) * 0.5 + 2.0
    loga0[torch.rand(2, I, generator=g) < zero_frac] = -12.0

    def run(skip):
        ops.ZERO_SKIP = skip
        try:
            for m in (vit, bert):
                for p in m.parameters():
                    p.grad = None
            loga = loga0.clone().cuda().requires_grad_()
            z = ops.l0_sample(loga, u, 2.0 / 3.0)
            assert abs(float((z == 0).float().mean()) - zero_frac) < 0.03
            xin = x.clone().requires_grad_()
            # both layers read the SAME input: chained, the 2e-7 summation-order difference of the first layer's output flips bf16
            # roundings inside the second one and shows up as 4e-4 (measured) — rounding chaos, not a property of the skip
            hv = vit(xin, None, False, mlp_z=z[0].view(1, 1, I))[0]
            hb = bert(xin, attention_mask=None, mlp_z=z[1].view(1, 1, I))[0]
            loss = hb.pow(2).mean() + hv.pow(2).mean()
            loss.backward()
            return (loss.detach(), torch.cat([hv, hb]).detach(), loga.grad.clone(), xin.grad.clone(),
                    {n: p.grad.clone() for m in (vit, bert) for n, p in m.named_parameters()})
        finally:
            ops.ZERO_SKIP = True
    K.reset_launch_count()
    l_d, h_d, dla_d, dx_d, g_d = run(False)
    l_s, h_s, dla_s, dx_s, g_s = run(True)
    # fp32 accumulation noise only: the kept columns are summed in compacted order (forward 2e-7 measured); the backward adds
    # split-K atomics and bf16 roundings of intermediate gradients that sit next to a rounding boundary
    assert_close(l_s, l_d, 1e-6, "loss")
    assert_close(h_s, h_d, 2e-6, "layer outputs")
    assert_close(dla_s, dla_d, 1e-3, "d log-alpha")
    assert torch.equal(dla_s == 0, dla_d == 0), "the same log-alphas receive no gradient"
    assert_close(dx_s, dx_d, 1e-3, "d input")
    for n in g_d:
        if n.endswith("k_proj.bias") or n.endswith("key.bias"):
            continue    # exactly 0 in exact arithmetic (softmax ignores a per-query constant): both sides are rounding noise
        # FFN parameters: the products themselves.  Attention-side parameters sit behind the FFN's bf16 input gradient, where a
        # 1e-7 difference flips roundings; the query / key projection gradients (small differences of large terms: softmax is
        # invariant to a per-query shift) show it most: 1.0e-3 - 1.3e-3 measured
        ffn = any(k in n for k in ("mlp.fc", "intermediate.dense", "output.dense", "output.LayerNorm")) and "attention" not in n
        assert_close(g_s[n], g_d[n], 1e-3 if ffn else 3e-3, "grad " + n)


@pytest.mark.parametrize("N", [197, 577])
def test_attention_map_kd_gradient_formed_inside_the_attention_backward(K, N):
    """Attention-map distillation of a ViT layer without a materialised gradient (ops.FUSED_ATTN_KD): the loss backward writes no dP,
    the attention backward reads the teacher map and forms coef * (P - P_t) from its re-computed P, the row sums come from the loss
    forward.  Loss, input gradient and every parameter gradient equal the materialised path (N = 197: one-CTA-per-head kernel, N = 577:
    the key-range LONG kernel); a map that ALSO feeds another loss gets NaN gradients (loud), never silently wrong ones."""
    from efficientvlm_b200 import ops
    from efficientvlm_b200.eff_vit import CLIPEncoderLayer
    from oracle.det_init import det_init_module_
    H, I, nh, B = 768, 3072, 12, 2
    layer = CLIPEncoderLayer(H, "quick_gelu", nh, 0.0, I).cuda().train()
    det_init_module_(layer)
    g = torch.Generator().manual_seed(N)
    x0 = torch.randn(B, N, H, generator=g).cuda()
    teacher = torch.softmax(torch.randn(B, nh, N, N, generator=g) * 2, -1).cuda()
    ld = K.probs_pitch(N)
    tpad = torch.zeros(B, nh, N, ld, device="cuda")
    tpad[..., :N] = teacher
    tmap = tpad[..., :N]
    wout = torch.randn(B, N, H, generator=g).cuda() * 0.01

    def run(fused, extra_consumer=False):
        ops.FUSED_ATTN_KD = fused
        try:
            x = x0.clone().requires_grad_()
            n0 = ops.KD_STATS["fused_pairs"]
            out, probs = layer(x, output_attentions=True)[:2]
            loss = 5.0 * ops.mse_pairs([probs], [tmap], [1.0]).sum() + (out * wout).sum()
            if extra_consumer:
                loss = loss + probs.sum()
            params = [p for _, p in sorted(layer.named_parameters())]
            grads = torch.autograd.grad(loss, [x] + params)
            return loss.detach(), grads, ops.KD_STATS["fused_pairs"] - n0
        finally:
            ops.FUSED_ATTN_KD = True
    loss_m, grads_m, n_m = run(False)
    loss_f, grads_f, n_f = run(True)
    assert n_m == 0 and n_f == 1
    assert_close(loss_f, loss_m, 1e-6, "loss")
    names = ["dx"] + [n for n, _ in sorted(layer.named_parameters())]
    for n, a, b in zip(names, grads_f, grads_m):
        if n.endswith("k_proj.bias"):
            continue                                    # identically zero up to rounding noise (softmax shift invariance)
        assert_close(a, b, 3e-3, n)
    _, grads_x, _ = run(True, extra_consumer=True)
    assert bool(torch.isnan(grads_x[0]).any()), "a second consumer of a fused map must fail loudly"


def test_mse_backward_row_dots_feed_the_attention_backward(K):
    """The KD MSE backward hands the softmax backward its  sum_j dP_ij P_ij  term (evlm_mse_pair.rowdot -> evlm_attn_args.dp_rowdot)
    instead of the pre-kernel re-reading both maps: the values equal the direct sum, on dense and on row-padded maps, and the
    attention backward produces the same dq / dk / dv with and without them."""
    from efficientvlm_b200 import ops
    g = torch.Generator().manual_seed(4)
    B, H, Lq, Lk = 3, 2, 40, 197
    q = (torch.randn(B * Lq, H * 64, generator=g) * 0.5).to(bf16).cuda()
    k = (torch.randn(B * Lk, H * 64, generator=g) * 0.5).to(bf16).cuda()
    v = (torch.randn(B * Lk, H * 64, generator=g) * 0.5).to(bf16).cuda()
    ctx, probs, lse = K.attention_fwd(q, k, v, B, H, Lq, Lk, 0.125, want_probs=True)
    assert K.row_pitch(probs) == 200 and probs.shape[-1] == Lk
    assert float(K.padded_base(probs)[..., Lk:].abs().sum()) == 0.0, "pad columns are exact zeros"
    teacher = torch.softmax(torch.randn(B, H, Lq, Lk, generator=g), -1).cuda()
    tpad = torch.zeros(B, H, Lq, 200, device="cuda")
    tpad[..., :Lk] = teacher
    s_in = probs.detach().requires_grad_()
    loss = ops.mse_pairs([s_in], [tpad[..., :Lk]], [3.0]).sum()
    (dp,) = torch.autograd.grad(loss, [s_in])
    ref_dp = 3.0 * 2 * (probs - teacher) / probs.numel()
    assert_close(dp, ref_dp, 1e-5, "dP from the padded storage, mean over the LOGICAL element count")
    rd = dp._evlm_rowdot
    assert_close(rd.view(B, H, Lq), (ref_dp * probs).sum(-1), 1e-4, "row dots")
    dctx = (torch.randn(B * Lq, H * 64, generator=g) * 0.1).to(bf16).cuda()
    outs = []
    for rowdot in (None, rd):
        dq, dk, dv = (torch.zeros_like(q), torch.zeros_like(k), torch.zeros_like(v))
        K.attention_bwd(q, k, v, ctx, lse, dctx, dq, dk, dv, B, H, Lq, Lk, 0.125, probs=probs, dprobs=dp, dp_rowdot=rowdot)
        outs.append((dq.float(), dk.float(), dv.float()))
    for a, b, n in zip(outs[0], outs[1], ("dq", "dk", "dv")):
        assert_close(b, a, 2e-3, n + " with the supplied row dots")
    # dense map (Lk % 4 == 0): same contract
    s2 = torch.softmax(torch.randn(2, 2, 8, 40, generator=g), -1).cuda().requires_grad_()
    t2 = torch.softmax(torch.randn(2, 2, 8, 40, generator=g), -1).cuda()
    (dp2,) = torch.autograd.grad(ops.mse_pairs([s2], [t2], [1.0]).sum(), [s2])
    assert_close(dp2._evlm_rowdot.view(2, 2, 8), (dp2 * s2.detach()).sum(-1), 1e-4, "row dots (dense map)")


def test_weight_shadows_refreshed_by_one_multi_tensor_cast(K):
    """FlatAdamW.step() rebuilds every bf16 shadow of its weights with one evlm_cast_table launch (stacked Q|K|V shadows and padded-pitch
    shadows included); the shadows then equal a fresh cast and the next forward issues no per-weight cast."""
    from efficientvlm_b200 import ops
    from efficientvlm_b200.optim import FlatAdamW
    g = torch.Generator().manual_seed(0)
    ws = [torch.nn.Parameter(torch.randn(*shape, generator=g).cuda()) for shape in ((64, 128), (64, 128), (64, 128), (40, 36), (256, 64))]
    opt = FlatAdamW([{"params": ws, "lr": 1e-2, "weight_decay": 0.0}])
    stacked = ops.weight_bf16(ws[0], ws[1], ws[2])
    odd = ops.weight_bf16(ws[3])                      # 36 columns: row pitch padded to 40
    single = ops.weight_bf16(ws[4])
    for w in ws:
        w.grad.copy_(torch.randn(w.shape, generator=g).cuda())
    n0 = K.launch_count()
    opt.step(allreduce=False)
    launches = K.launch_count() - n0
    n1 = K.launch_count()
    s2, o2, g2 = ops.weight_bf16(ws[0], ws[1], ws[2]), ops.weight_bf16(ws[3]), ops.weight_bf16(ws[4])
    assert K.launch_count() == n1, "shadows are valid right after the step: no lazy cast"
    assert s2.data_ptr() == stacked.data_ptr() and o2.data_ptr() == odd.data_ptr() and g2.data_ptr() == single.data_ptr()
    assert torch.equal(s2, torch.cat([w.detach() for w in ws[:3]]).to(bf16))
    assert torch.equal(o2, ws[3].detach().to(bf16)) and o2.stride(0) == 40
    assert torch.equal(g2, ws[4].detach().to(bf16))
    assert launches <= 4, launches                    # hyper-parameter store + AdamW + ONE cast (+ nothing per weight)
