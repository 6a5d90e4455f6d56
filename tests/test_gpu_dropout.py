"""Dropout masks, exactly.  Every dropout site of the library draws its keep/drop decisions from one counter-based stream
(Philox2x32-10 on a 64-bit element index, evlm_common.cuh); `dropout_uniform` below mirrors that stream in plain numpy on the host.
Each site documents the element index it draws:

    attention          ((b*H + h)*Lq + i) * round_up4(Lk) + j      b = the query item, j = the item's own key
    GEMM epilogue      row*N + col
    cast_f32_to_bf16   r*cols + c
    LayerNorm          row*H + col (forward output, backward replay and the bwd_ex output mask alike)

and keeps an element iff u >= p, scaling it by 1/(1-p).  The tests read each kernel's mask back and compare it with the mirror bit for
bit, and compare attention gradients under dropout with an fp64 autograd reference that applies the mirror's mask, per (item, head)
block and per 128-row tile, so that one wrong pack slot, query tile or kernel variant cannot hide behind the rest of the tensor."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.helpers import assert_close

bf16, f32 = torch.bfloat16, torch.float32
gpu = pytest.mark.gpu
BF_TOL = 2e-2          # kernel-level bf16 tolerance of tests/test_gpu_kernels.py
P = 0.1                # the training workloads' dropout rate (eff_bert.py)
SEEDS = (0, 1234, 2 ** 32 + 7, 0xDEADBEEF12345678)    # the high word reaches the key through the rotate
STREAMS = (0, 1, 2, 3, 4, 7, 2 ** 31)

# ------------------------------------------------------------------------------------------------ the host mirror
M32 = np.uint64(0xFFFFFFFF)


def _philox(seed, stream, i4):
    """(x, y) words of Philox2x32-10 for counters i4 (== evlm_common.cuh dropout_bits(seed, stream, i4))."""
    i4 = np.asarray(i4, dtype=np.uint64)
    seed &= 0xFFFFFFFFFFFFFFFF
    hi = (seed >> 32) & 0xFFFFFFFF
    key = np.uint64(((seed & 0xFFFFFFFF) ^ (((hi << 13) | (hi >> 19)) & 0xFFFFFFFF) ^ 0x65766C6D) & 0xFFFFFFFF)
    x = i4 & M32
    y = (i4 >> np.uint64(32)) ^ np.uint64((stream * 0x85EBCA6B + 0xC2B2AE35) & 0xFFFFFFFF)
    for _ in range(10):
        prod = np.uint64(0xD256D193) * x
        x, y = ((prod >> np.uint64(32)) ^ key ^ y) & M32, prod & M32
        key = (key + np.uint64(0x9E3779B9)) & M32
    return x, y


def dropout_uniform(seed, stream, idx):
    """== evlm_common.cuh dropout_uniform(seed, stream, idx): the uniform in [0, 1) of element `idx`."""
    idx = np.asarray(idx, dtype=np.uint64)
    x, y = _philox(seed, stream, idx >> np.uint64(2))
    w = np.where((idx & np.uint64(2)) != 0, y, x)
    h = np.where((idx & np.uint64(1)) != 0, w >> np.uint64(16), w & np.uint64(0xFFFF))
    return h.astype(np.float32) / np.float32(65536.0)


def keep_grid(seed, stream, base, ncols, p=P):
    """Keep mask (bool torch tensor [len(base), ncols]) of the elements base[r] + c.  Bases that are multiples of 4 take one Philox
    call per 4 elements, as the kernels do; the values are those of `dropout_uniform` either way."""
    base = np.asarray(base, dtype=np.uint64).reshape(-1)
    if np.all(base % np.uint64(4) == 0):
        c4 = np.arange((ncols + 3) // 4, dtype=np.uint64)
        x, y = _philox(seed, stream, (base[:, None] >> np.uint64(2)) + c4[None, :])
        w = np.stack([x & np.uint64(0xFFFF), x >> np.uint64(16), y & np.uint64(0xFFFF), y >> np.uint64(16)], -1)
        u = (w.reshape(len(base), -1)[:, :ncols].astype(np.float32) / np.float32(65536.0))
    else:
        u = dropout_uniform(seed, stream, base[:, None] + np.arange(ncols, dtype=np.uint64)[None, :])
    return torch.from_numpy(u >= np.float32(p))


def keep_rows(seed, stream, rows, cols, p=P):
    """Keep mask of a row-major [rows, cols] site (index row*cols + col) on the device."""
    return keep_grid(seed, stream, np.arange(rows, dtype=np.uint64) * np.uint64(cols), cols, p).cuda()


def test_mirror_known_answer():
    """First uniforms of seed 0x123456789, stream 3, from a line-by-line C++ host port of dropout_bits / dropout_uniform."""
    assert (dropout_uniform(0x123456789, 3, np.arange(4)) * 65536).astype(np.int64).tolist() == [60991, 22988, 15504, 4052]


def _mismatch(got, exp, names):
    bad = (got != exp).nonzero()
    return "%d of %d mask bits differ, first at %s" % (bad.shape[0], got.numel(), dict(zip(names, bad[0].tolist()))) if bad.numel() else ""


# ------------------------------------------------------------------------------------------------ fixtures
@pytest.fixture(scope="module")
def rng_word():
    """A zero seed-offset word bound for this module: the masks are mirrored at exactly the seeds the calls pass, even when an earlier
    test left graph.rng_state's word bound at some offset.  That word (or none) is bound again afterwards."""
    from efficientvlm_b200 import graph, kernels
    zero = torch.zeros(1, dtype=torch.int64, device="cuda")
    kernels.rng_bind(zero)
    yield zero
    torch.cuda.synchronize()
    kernels.rng_bind(graph._rng_state.get(("cuda", torch.cuda.current_device())))


@pytest.fixture(scope="module")
def K(rng_word):
    from efficientvlm_b200 import kernels
    return kernels


def _rand(*shape, scale=1.0, dtype=f32, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(*shape, generator=g, device="cuda") * scale).to(dtype)


# ------------------------------------------------------------------------------------------------ elementwise sites
def _check_cast(K, rows, cols, seed, stream, eff=None):
    """cast_bf16 of ones: out != 0 is the mask; flat (dense) and strided (padded source rows) launches alike."""
    eff = seed if eff is None else eff
    exp = keep_rows(eff, stream, rows, cols)
    wide = torch.ones(rows, cols + 4, device="cuda")
    for what, src in (("dense", wide[:, :cols].contiguous()), ("strided", wide[:, :cols])):
        out = K.cast_bf16(src, dropout_p=P, seed=seed, stream_id=stream)
        got = out != 0
        assert torch.equal(got, exp), "cast %s %dx%d seed %#x stream %d: %s" % (what, rows, cols, seed, stream,
                                                                                  _mismatch(got, exp, ("row", "col")))
        assert torch.equal(out[got].float().unique(), torch.tensor([1 / (1 - P)], device="cuda").to(bf16).float())


@gpu
@pytest.mark.parametrize("rows,cols", [(7, 8), (300, 768), (37, 203)])
def test_cast_dropout_mask_equals_mirror(K, rows, cols):
    for seed in SEEDS:
        for stream in STREAMS:
            _check_cast(K, rows, cols, seed, stream)


@gpu
def test_cast_dropout_mask_equals_mirror_large(K):
    _check_cast(K, 25216, 768, 0xDEADBEEF12345678, 2 ** 31)


# (id, M, N, K, residual dtype or None, D dtype, D / residual row pitch or None)
GEMM_CASES = [
    ("single-buffer", 300, 768, 256, None, f32, None),
    ("double-buffer-f32-residual", 300, 768, 768, f32, f32, None),
    ("double-buffer-bf16-residual", 300, 768, 1024, bf16, f32, None),
    ("single-buffer-residual-k3072", 300, 768, 3072, f32, f32, None),
    ("bf16-D", 300, 768, 768, bf16, bf16, None),
    ("m20-not-skinny", 20, 768, 256, None, f32, None),
    ("n770-single-buffer", 300, 770, 256, None, f32, 776),
    ("n770-double-buffer", 300, 770, 768, f32, f32, 776),
]


def _check_gemm(K, case, seed, stream, eff=None):
    """GEMM with dropout (and a bias far from 0, so no product is 0): D - residual != 0 is the mask, kept values are the fp32
    product x 1/(1-p).  Dropout comes before the residual (include/evlm.h), so dropped elements equal the residual exactly."""
    what, M, N, K_, rdt, ddt, ld = case
    eff = seed if eff is None else eff
    A = _rand(M, K_, dtype=bf16, seed=1, scale=0.1)
    B = _rand(N, K_, dtype=bf16, seed=2, scale=0.1)
    bias = 3.0 + 0.1 * _rand(N, seed=3)
    pitch = ld or N
    res = None
    if rdt is not None:
        res = _rand(M, pitch, seed=4).to(rdt)[:, :N]
    D = torch.empty(M, pitch, dtype=ddt, device="cuda")[:, :N]
    K.gemm(A, B, D, M, N, K_, bias=bias, residual=res, dropout_p=P, seed=seed, stream_id=stream)
    out = D.float() - (res.float() if res is not None else 0.0)
    got = out != 0
    exp = keep_rows(eff, stream, M, N)
    assert torch.equal(got, exp), "gemm %s seed %#x stream %d: %s" % (what, seed, stream, _mismatch(got, exp, ("row", "col")))
    ref = (A.float() @ B.float().t() + bias) / (1 - P)
    assert_close(out[exp], ref[exp], 1e-4 if ddt == f32 else 6e-3, "gemm %s kept values" % what)


@gpu
@pytest.mark.parametrize("case", GEMM_CASES, ids=[c[0] for c in GEMM_CASES])
def test_gemm_dropout_mask_equals_mirror(K, case):
    for seed, stream in ((1234, 3), (2 ** 32 + 7, 1), (0xDEADBEEF12345678, 2 ** 31)):
        _check_gemm(K, case, seed, stream)


def _ln_inputs(H, rows=333):
    x = _rand(rows, H, seed=1, scale=2.0)
    w, b = 0.1 + 0.02 * _rand(H, seed=2), 3.0 + 0.1 * _rand(H, seed=3)     # |y - 3| < 1: no output is 0
    return x, w, b


def _ln_ref_grads(x, w, b, dy, eps=1e-12):
    xr, wr, br = (t.double().requires_grad_() for t in (x, w, b))
    y = F.layer_norm(xr, (x.shape[-1],), wr, br, eps)
    return torch.autograd.grad(y, [xr, wr, br], dy.double())


def _check_ln_fwd(K, H, seed, eff=None):
    """LayerNorm forward with output dropout (stream 7), then the backward replaying that mask on dy."""
    eff = seed if eff is None else eff
    x, w, b = _ln_inputs(H)
    rows = x.shape[0]
    y32, y16, mean, rstd = K.layernorm_fwd(x, w, b, 1e-12, want_f32=True, want_bf16=True, dropout_p=P, seed=seed, stream_id=7)
    exp = keep_rows(eff, 7, rows, H)
    for what, y in (("fp32", y32), ("bf16", y16)):
        got = y != 0
        assert torch.equal(got, exp), "ln fwd %s H %d seed %#x: %s" % (what, H, seed, _mismatch(got, exp, ("row", "col")))
    ref = F.layer_norm(x.double(), (H,), w.double(), b.double(), 1e-12) * exp / (1 - P)
    assert_close(y32, ref, 1e-5, "ln fwd dropout values")
    dy = _rand(rows, H, seed=4)
    dx, _ = K.layernorm_bwd(dy, x, w, mean, rstd, dropout_p=P, seed=seed, stream_id=7)
    gx, _, _ = _ln_ref_grads(x, w, b, dy * exp / (1 - P))
    assert_close(dx, gx, 1e-4, "ln bwd replays the forward mask")


@gpu
@pytest.mark.parametrize("H", [768, 1536])
def test_layernorm_dropout_mask_equals_mirror(K, H):
    for seed in SEEDS:
        _check_ln_fwd(K, H, seed)


def _check_ln_bwd_ex(K, H, seed, eff=None):
    """evlm_layernorm_bwd_ex: replay of the input mask (stream 7) on dy, the output mask of another stream (5) on dx_bf16 only,
    dcolsum += column sums of dx_bf16, dgamma / dbeta accumulated."""
    eff = seed if eff is None else eff
    x, w, b = _ln_inputs(H)
    rows = x.shape[0]
    _, _, mean, rstd = K.layernorm_fwd(x, w, b, 1e-12)
    dy, dres = _rand(rows, H, seed=5), _rand(rows, H, seed=6, scale=0.5)
    dg0, db0, cs0 = _rand(H, seed=7), _rand(H, seed=8), _rand(H, seed=9)
    dg, db, cs = dg0.clone(), db0.clone(), cs0.clone()
    dx32, dx16 = K.layernorm_bwd(dy, x, w, mean, rstd, dres=dres, want_f32=True, want_bf16=True, dgamma=dg, dbeta=db, dropout_p=P,
                                 seed=seed, stream_id=7, out_dropout_p=P, out_stream_id=5, dcolsum=cs)
    keep_in, keep_out = keep_rows(eff, 7, rows, H), keep_rows(eff, 5, rows, H)
    gx, gw, gb = _ln_ref_grads(x, w, b, dy * keep_in / (1 - P))
    ref = gx + dres.double()
    assert_close(dx32, ref, 1e-4, "ln bwd_ex dx fp32 (no output mask)")
    got = dx16 != 0
    assert torch.equal(got, keep_out), "ln bwd_ex output mask H %d seed %#x: %s" % (H, seed, _mismatch(got, keep_out, ("row", "col")))
    assert_close(dx16, ref * keep_out / (1 - P), 8e-3, "ln bwd_ex dx bf16 (output mask)")
    assert_close(cs, cs0 + dx16.float().sum(0), 1e-5, "ln bwd_ex dcolsum")
    assert_close(dg, dg0 + gw, 1e-4, "ln bwd_ex dgamma")
    assert_close(db, db0 + gb, 1e-4, "ln bwd_ex dbeta")


@gpu
@pytest.mark.parametrize("H", [128, 768, 1024])
def test_layernorm_bwd_ex_output_mask_equals_mirror(K, H):
    for seed in (1234, 0xDEADBEEF12345678):
        _check_ln_bwd_ex(K, H, seed)


# ------------------------------------------------------------------------------------------------ attention
SCALE = 0.125
KV_INDEX = [0, 1, 0, 2, 0, 1, 2, 2]
# (id, B, H, Lq, Lk, options); the kernel each case reaches (attention.cu evlm_attention_fwd / evlm_attention_bwd):
ATTN_CASES = [
    ("tc", 2, 2, 40, 197, {}),                                               # tcgen05 forward / backward, Lq, Lk <= 256
    ("tc-two-query-tiles", 1, 2, 197, 197, {}),                              # two 128-row query tiles
    ("tc-lk77", 2, 2, 40, 77, {}),                                           # round_up4(Lk) = 80 != Lk
    ("tc-256", 1, 2, 256, 256, {}),
    ("tc-causal", 2, 2, 40, 40, dict(causal=True)),
    ("tc-key-mask", 2, 2, 40, 197, dict(masked=True)),
    ("kv-index", 8, 2, 40, 197, dict(kv=KV_INDEX)),                          # shared K/V, one CTA per query item
    ("pack-shared-kv", 8, 2, 40, 197, dict(kv=KV_INDEX, pack=[[0, 2, 4], [1, 5, -1], [3, 6, 7]])),
    ("pack-own-kv-40", 8, 2, 40, 40, dict(pack=[[0, 1, 2], [3, 4, 5], [6, 7, -1]], own=True, masked=True)),
    ("pack-own-kv-56", 5, 2, 56, 56, dict(pack=[[0, 1], [2, 3], [4, -1]], own=True)),
    ("long-16x901", 2, 2, 16, 901, {}),                                      # two-sweep tcgen05 forward, LONG backward
    ("long-577-key-mask", 1, 2, 577, 577, dict(masked=True)),
    ("long-129x300", 1, 1, 129, 300, {}),
    ("tiled-70x1100", 1, 1, 70, 1100, dict(masked=True)),                    # Lk > 1024: tiled mma.sync forward / backward
]


class _Attn:
    """One attention configuration: inputs, the kernel keyword arguments and the reference's view of K / V."""

    def __init__(self, case, masked=None):
        self.name, self.B, self.H, self.Lq, self.Lk, o = case
        B, H, Lq, Lk = self.B, self.H, self.Lq, self.Lk
        self.E = H * 64
        self.causal = bool(o.get("causal"))
        self.kv = torch.tensor(o["kv"], dtype=torch.int32, device="cuda") if "kv" in o else None
        self.nkv = 3 if self.kv is not None else B
        self.pack = torch.tensor(o["pack"], dtype=torch.int32, device="cuda") if "pack" in o else None
        self.own = bool(o.get("own"))
        # dk / dv rows: one block per query item, or per pack group when the group shares one K/V item
        self.shared_pack = self.pack is not None and not self.own
        self.n_dkv = self.pack.shape[0] if self.shared_pack else B
        self.group = {}
        if self.shared_pack:
            for gi, row in enumerate(o["pack"]):
                for b in row:
                    if b >= 0:
                        self.group[b] = gi
        self.key_mask = None
        if masked is None:
            masked = bool(o.get("masked"))
        if masked:
            self.key_mask = torch.zeros(B, Lk, device="cuda")
            for b in range(B):
                self.key_mask[b, Lk - 3 - b % 3:] = -10000.0
        self.kw = dict(key_mask=self.key_mask, causal=self.causal, causal_offset=Lk - Lq if self.causal else 0, kv_index=self.kv,
                       pack_items=self.pack, pack_own_kv=self.own)

    def per_item(self, t):
        """K / V rows as each QUERY item sees them ([B*Lk, E])."""
        if self.kv is None:
            return t
        return t.view(self.nkv, self.Lk, self.E).index_select(0, self.kv.long()).reshape(self.B * self.Lk, self.E)

    def valid(self):
        """[B, 1|H, Lq, Lk] bool: the (query, key) pairs that carry probability (not masked, not above the causal diagonal)."""
        v = torch.ones(self.B, 1, self.Lq, self.Lk, dtype=torch.bool, device="cuda")
        if self.key_mask is not None:
            v &= (self.key_mask == 0)[:, None, None, :]
        if self.causal:
            i = torch.arange(self.Lq, device="cuda")[:, None]
            j = torch.arange(self.Lk, device="cuda")[None, :]
            v &= j <= i + (self.Lk - self.Lq)
        return v

    def keep(self, seed, stream):
        """The documented attention mask: element ((b*H + h)*Lq + i) * round_up4(Lk) + j, b the query item. [B, H, Lq, Lk]"""
        lkp4 = (self.Lk + 3) // 4 * 4
        base = np.arange(self.B * self.H * self.Lq, dtype=np.uint64) * np.uint64(lkp4)
        return keep_grid(seed, stream, base, self.Lk).view(self.B, self.H, self.Lq, self.Lk).cuda()

    def scores(self, q, k_items):
        B, H, Lq, Lk = self.B, self.H, self.Lq, self.Lk
        qh = q.double().reshape(B, Lq, H, 64).transpose(1, 2)
        kh = k_items.double().reshape(B, Lk, H, 64).transpose(1, 2)
        s = qh @ kh.transpose(-1, -2) * SCALE
        if self.key_mask is not None:
            s = s + self.key_mask.double()[:, None, None, :]
        if self.causal:
            i = torch.arange(Lq, device="cuda")[:, None]
            j = torch.arange(Lk, device="cuda")[None, :]
            s = s + (j > i + (Lk - Lq)).double() * -10000.0
        return s


def _fwd_dropped_probs(K, c, q, k, seed, stream):
    """(D o P) / (1-p) as the forward applied it, read back through V one-hot over a 64-key window w: v[j, h*64 + d] = 1 iff
    j == 64w + d, so ctx[i, h*64 + d] is the dropped probability of key 64w + d.  [B, H, Lq, Lk] fp32."""
    B, H, Lq, Lk = c.B, c.H, c.Lq, c.Lk
    out = torch.zeros(B, H, Lq, Lk, device="cuda")
    for w0 in range(0, Lk, 64):
        n = min(64, Lk - w0)
        d = torch.arange(n, device="cuda")
        v = torch.zeros(c.nkv, Lk, H, 64, dtype=bf16, device="cuda")
        v[:, w0 + d, :, d] = 1
        ctx, _, _ = K.attention_fwd(q, k, v.view(c.nkv * Lk, c.E), B, H, Lq, Lk, SCALE, dropout_p=P, seed=seed, stream_id=stream, **c.kw)
        out[..., w0:w0 + n] = ctx.float().view(B, Lq, H, 64)[..., :n].permute(0, 2, 1, 3)
    return out


def _bwd_dropped_probs(K, c, q, k, v, seed, stream):
    """(D o P) / (1-p) as the backward replayed it, read back through dctx one-hot over a 64-query window w: then
    dv[j, h*64 + d] is the dropped probability of query 64w + d and key j.  Where a pack group shares one K/V item (dv per
    group), one member's window is driven at a time.  [B, H, Lq, Lk] fp32."""
    B, H, Lq, Lk, E = c.B, c.H, c.Lq, c.Lk, c.E
    ctx, _, lse = K.attention_fwd(q, k, v, B, H, Lq, Lk, SCALE, dropout_p=P, seed=seed, stream_id=stream, **c.kw)
    out = torch.zeros(B, H, Lq, Lk, device="cuda")
    drives = [[b] for b in range(B)] if c.shared_pack else [list(range(B))]
    for w0 in range(0, Lq, 64):
        n = min(64, Lq - w0)
        d = torch.arange(n, device="cuda")
        for items in drives:
            dctx = torch.zeros(B, Lq, H, 64, dtype=bf16, device="cuda")
            for b in items:
                dctx[b, w0 + d, :, d] = 1
            dq = torch.zeros(B * Lq, E, dtype=bf16, device="cuda")
            dk, dv = (torch.zeros(c.n_dkv * Lk, E, dtype=bf16, device="cuda") for _ in range(2))
            K.attention_bwd(q, k, v, ctx, lse, dctx.view(B * Lq, E), dq, dk, dv, B, H, Lq, Lk, SCALE, dropout_p=P, seed=seed, stream_id=stream,
                            **c.kw)
            got = dv.float().view(c.n_dkv, Lk, H, 64)[..., :n].permute(0, 2, 3, 1)      # [n_dkv, H, n, Lk]
            if c.shared_pack:
                out[items[0], :, w0:w0 + n] = got[c.group[items[0]]]
            else:
                out[:, :, w0:w0 + n] = got
    return out


def _attn_inputs(c):
    """Small q and k (every unmasked probability is ~ 1 / Lk and never rounds to 0) and a random v."""
    q = _rand(c.B * c.Lq, c.E, dtype=bf16, seed=1, scale=0.1)
    k = _rand(c.nkv * c.Lk, c.E, dtype=bf16, seed=2, scale=0.1)
    v = _rand(c.nkv * c.Lk, c.E, dtype=bf16, seed=3)
    return q, k, v


def _check_attention_masks(K, c, seed, stream, eff=None, fwd=True, bwd=True):
    eff = seed if eff is None else eff
    q, k, v = _attn_inputs(c)
    p_ref = torch.softmax(c.scores(q, c.per_item(k)), -1)
    keep = c.keep(eff, stream)
    valid = c.valid().expand_as(keep)
    names = ("item", "head", "query", "key")
    runs = ([("forward", _fwd_dropped_probs(K, c, q, k, seed, stream))] if fwd else []) + \
           ([("backward", _bwd_dropped_probs(K, c, q, k, v, seed, stream))] if bwd else [])
    for what, got in runs:
        nz = (got != 0) & valid
        exp = keep & valid
        assert torch.equal(nz, exp), "attention %s %s seed %#x stream %d: %s" % (c.name, what, seed, stream, _mismatch(nz, exp, names))
        ref = (p_ref / (1 - P))[exp]
        err = ((got[exp].double() - ref).abs() / ref).max().item()
        assert err < 1e-2, "attention %s %s: kept values differ from P / (1-p) by %.2e (relative)" % (c.name, what, err)


@gpu
@pytest.mark.parametrize("case", ATTN_CASES, ids=[c[0] for c in ATTN_CASES])
def test_attention_mask_reads_back_exactly(K, case):
    """Each forward draws the documented stream and each backward replays it, on every kernel path."""
    _check_attention_masks(K, _Attn(case), 0xDEADBEEF12345678, 3)


def _assert_blocks(got, ref, tol, what):
    """assert_close per (item, head) block and per 128-row tile of tensors viewed as [items, rows, H, cols]."""
    for it in range(got.shape[0]):
        for h in range(got.shape[2]):
            for r0 in range(0, got.shape[1], 128):
                assert_close(got[it, r0:r0 + 128, h], ref[it, r0:r0 + 128, h], tol, "%s item %d head %d rows %d+" % (what, it, h, r0))


@gpu
@pytest.mark.parametrize("case", ATTN_CASES, ids=[c[0] for c in ATTN_CASES])
def test_attention_gradients_under_dropout(K, case):
    """ctx = z ((P o D) / (1-p)) V with the mirror's mask D, differentiated in fp64, against the kernels' forward and backward
    (gradient on ctx and on the returned, pre-dropout map; head_z with one head at 0)."""
    c = _Attn(case, masked=True)
    B, H, Lq, Lk, E = c.B, c.H, c.Lq, c.Lk, c.E
    seed, stream = 0x5EED0000ABCD, 3
    q = _rand(B * Lq, E, dtype=bf16, seed=11, scale=0.7)
    k = _rand(c.nkv * Lk, E, dtype=bf16, seed=12, scale=0.7)
    v = _rand(c.nkv * Lk, E, dtype=bf16, seed=13, scale=0.7)
    head_z = torch.rand(H, device="cuda")
    head_z[0] = 0.0
    ctx, probs, lse = K.attention_fwd(q, k, v, B, H, Lq, Lk, SCALE, head_z=head_z, want_probs=True, dropout_p=P, seed=seed, stream_id=stream,
                                      **c.kw)
    dctx = _rand(B * Lq, E, seed=14, scale=0.5).to(bf16)
    dprobs = _rand(B, H, Lq, Lk, seed=15, scale=0.3)
    dq = torch.zeros(B * Lq, E, dtype=bf16, device="cuda")
    dk, dv = (torch.zeros(c.n_dkv * Lk, E, dtype=bf16, device="cuda") for _ in range(2))
    dz = torch.zeros(H, device="cuda")
    K.attention_bwd(q, k, v, ctx, lse, dctx, dq, dk, dv, B, H, Lq, Lk, SCALE, probs=probs, dprobs=dprobs, head_z=head_z, dhead_z=dz,
                    dropout_p=P, seed=seed, stream_id=stream, **c.kw)
    # fp64 reference on the K / V each query item sees
    qr, kr, vr = (t.double().requires_grad_() for t in (q, c.per_item(k), c.per_item(v)))
    zr = head_z.double().requires_grad_()
    s = c.scores(qr, kr)
    p = torch.softmax(s, -1)
    drop = c.keep(seed, stream).double() / (1 - P)
    rctx = ((p * drop) @ vr.view(B, Lk, H, 64).transpose(1, 2)) * zr.view(1, H, 1, 1)
    rctx = rctx.transpose(1, 2).reshape(B * Lq, E)
    gq, gk, gv, gz = torch.autograd.grad([rctx, p], [qr, kr, vr, zr], [dctx.double(), dprobs.double()])
    if c.shared_pack:     # dk / dv per pack group: the sum over its members
        idx = torch.tensor([c.group[b] for b in range(B)], device="cuda")
        gk = torch.zeros(c.n_dkv, Lk * E, dtype=gk.dtype, device="cuda").index_add_(0, idx, gk.view(B, Lk * E))
        gv = torch.zeros(c.n_dkv, Lk * E, dtype=gv.dtype, device="cuda").index_add_(0, idx, gv.view(B, Lk * E))

    def rows(t, n, L):
        return t.reshape(n, L, H, -1)

    _assert_blocks(rows(ctx.float(), B, Lq), rows(rctx.detach(), B, Lq), 1e-2, "%s ctx" % c.name)
    _assert_blocks(probs.permute(0, 2, 1, 3), p.detach().permute(0, 2, 1, 3), 3e-3, "%s probs" % c.name)
    _assert_blocks(lse.permute(0, 2, 1)[..., None], torch.logsumexp(s.detach(), -1).permute(0, 2, 1)[..., None], 1e-4, "%s lse" % c.name)
    _assert_blocks(rows(dq.float(), B, Lq), rows(gq, B, Lq), BF_TOL, "%s dq" % c.name)
    _assert_blocks(rows(dk.float(), c.n_dkv, Lk), rows(gk, c.n_dkv, Lk), BF_TOL, "%s dk" % c.name)
    _assert_blocks(rows(dv.float(), c.n_dkv, Lk), rows(gv, c.n_dkv, Lk), BF_TOL, "%s dv" % c.name)
    assert_close(dz, gz, BF_TOL, "%s dhead_z" % c.name)


# ------------------------------------------------------------------------------------------------ the device seed offset
@gpu
def test_rng_bind_offset_reaches_every_site(K, rng_word):
    """evlm_rng_bind sets the seed-offset pointer of every translation unit: under a bound word each site draws the mirror's mask at
    seed + offset, and after rng_advance(delta) at seed + offset + delta (how a replayed CUDA graph gets fresh masks)."""
    seed, offset, delta = 1234, 2 ** 40 + 3, 0x9E3779B97F4A7C15
    cases = {c[0]: c for c in ATTN_CASES}
    state = torch.tensor([offset], dtype=torch.int64, device="cuda")
    K.rng_bind(state)
    try:
        for eff in (seed + offset, seed + offset + delta):
            _check_cast(K, 300, 768, seed, 3, eff)
            _check_gemm(K, GEMM_CASES[0], seed, 3, eff)          # single-buffer epilogue
            _check_gemm(K, GEMM_CASES[1], seed, 3, eff)          # double-buffered epilogue
            _check_ln_fwd(K, 768, seed, eff)
            _check_ln_bwd_ex(K, 768, seed, eff)
            for name in ("tc-lk77", "long-129x300", "tiled-70x1100"):   # forward and backward of each attention kernel family
                _check_attention_masks(K, _Attn(cases[name]), seed, 3, eff)
            K.rng_advance(state, delta)
    finally:
        torch.cuda.synchronize()
        K.rng_bind(rng_word)
