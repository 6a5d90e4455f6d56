"""The loss, L0-gate and optimizer kernels (csrc/losses.cu, csrc/l0_optim.cu) against fp64 restatements of the same formulas, at the
shapes, row pitches, dtypes and alignments training reaches them with.

Every float check is element-wise against a bound derived next to it from the kernel's own arithmetic: U = 2^-24 is the unit roundoff
of fp32, and a sum of k terms accumulated in fp32 (serially, or through a tree of depth k) is off by at most k U times the sum of the
terms' magnitudes.  Masks, indices, counts, the bf16 shadow and run-to-run repeats are compared exactly.  Pad columns and unused
storage around the strided views are NaN, so a kernel that reads outside a row returns NaN and fails."""
import json
import math
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
f32, f64, bf16 = torch.float32, torch.float64, torch.bfloat16
U = 2.0 ** -24
NAN = float("nan")


@pytest.fixture(scope="module")
def K():
    from efficientvlm_b200 import kernels
    return kernels


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _randn(*shape, seed, scale=1.0):
    return torch.randn(*shape, generator=_gen(seed), device="cuda") * scale


def _rand(*shape, seed):
    return torch.rand(*shape, generator=_gen(seed), device="cuda")


def _within(got, want, tol, what):
    """|got - want| <= tol element-wise (fp64); NaN anywhere fails.  With EVLM_CALIBRATE_LOG set, the largest error and the largest
    error / bound ratio of every check are appended there (as tests/helpers.assert_close does)."""
    err = (got.double() - want).abs()
    tol = torch.as_tensor(tol, dtype=f64, device=err.device).expand_as(err)
    ratio = torch.nan_to_num(err / tol, nan=float("inf"), posinf=float("inf"))
    ratio = torch.where(err == 0, torch.zeros_like(ratio), ratio)
    log = os.environ.get("EVLM_CALIBRATE_LOG")
    if log:
        with open(log, "a") as f:
            f.write(json.dumps({"test": os.environ.get("PYTEST_CURRENT_TEST", ""), "what": what, "max_err": float(err.max()),
                                "max_err_over_bound": float(ratio.max())}) + "\n")
    bad = ~(err <= tol)
    if bool(bad.any()):
        i = int(ratio.flatten().argmax())
        raise AssertionError("%s: %d of %d elements outside the bound; worst: error %.3e, bound %.3e, got %r, want %r" % (
            what, int(bad.sum()), bad.numel(), float(err.flatten()[i]), float(tol.flatten()[i]), float(got.flatten()[i]),
            float(want.flatten()[i])))


def _row_view(x, pitch, offset):
    """x [rows, V] copied into a NaN-filled buffer as a view with row pitch `pitch` and storage offset `offset` (floats)."""
    rows, V = x.shape
    buf = torch.full((offset + rows * pitch + pitch,), NAN, device="cuda")
    v = buf[offset:offset + rows * pitch].view(rows, pitch)[:, :V]
    v.copy_(x)
    assert v.stride(0) == pitch and v.storage_offset() == offset
    return v


# ------------------------------------------------------------------------------------------------ row softmax losses
# (pitch, storage offset) of the logits rows.  "pitch+2" is the MLM logits' layout (30522 columns on a 30524 pitch); "odd-pitch" makes
# consecutive rows alternate between the 8-byte-aligned float2 path of row_lse and its scalar path; "offset1" starts every row (V even)
# or every other row (V odd) off the 8-byte grid.
LAYOUTS = {"dense": lambda V: (V, 0), "pitch+2": lambda V: (V + 2, 0), "odd-pitch": lambda V: (V + 2 if V % 2 else V + 1, 0),
           "offset1": lambda V: (V, 1)}
VOCABS = [2, 3, 511, 512, 1001, 2047, 30522]


def _logits(rows, V, seed):
    """Per-row scales 3 .. 10 (what the MLM and ITM heads produce); row 3 has one maximum 60 above the rest in its LAST column (the
    scalar tail of row_lse) and row 4 one in its first column, so the online max / rescale paths both start from a far outlier."""
    scale = torch.linspace(3.0, 10.0, rows, device="cuda")[:, None]
    x = _randn(rows, V, seed=seed) * scale
    if rows > 4:
        x[3, V - 1] = x[3].max() + 60.0
        x[4, 0] = x[4].max() + 60.0
    return x


def _lse_tol(y):
    """Bound on |lse_kernel - lse| for one fp64 row y = x * inv_temp (rows of a [rows, V] tensor).
    row_lse rounds x * inv_temp (shifts lse by <= U max|y|); every thread sums its <= V/256 exponentials and rescales <= V/2048 times,
    then an 8-level block tree combines them: <= V/256 + V/2048 + 8 roundings of a positive sum.  __expf is within (2 + 1.17 |a|) ulp
    of exp(a) for a <= 0; weighted by the softmax that is <= 2 + 1.17 (entropy + lse - max) <= 2 + 2.4 ln V ulp of the sum.  logf and
    the final add round once each (<= 2 U |lse|).  The counts are doubled to cover the ulp-level slack of __expf / logf."""
    V = y.shape[-1]
    lse = torch.logsumexp(y, -1)
    steps = V / 256 + V / 2048 + 8 + 2 + 2.4 * math.log(V) + 2
    return U * (y.abs().amax(-1) + 2 * lse.abs() + 2 * steps), lse


def _p_rel(lp, ltol, y):
    """Relative error bound of __expf(y - l) with l off by <= ltol: ltol, the rounding of y and of y - l, and __expf's (2 + 1.17|a|) ulp."""
    return ltol[:, None] + U * (y.abs() + lp.abs() + 3 + 1.2 * lp.abs())


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("V", VOCABS)
def test_xent_rows(K, V, layout):
    rows = 37
    pitch, off = LAYOUTS[layout](V)
    x = _logits(rows, V, seed=V)
    xv = _row_view(x, pitch, off)
    labels = torch.randint(0, V, (rows,), generator=_gen(V + 1), device="cuda")
    labels[1], labels[2] = 0, V - 1
    labels[::5] = -100
    x64 = x.double()
    ltol, lse64 = _lse_tol(x64)
    g = _randn(rows, seed=V + 2)
    keep = (labels != -100).double()
    for ls in (0.0, 0.1):
        loss, lse = K.xent_fwd(xv, labels, -100, ls)
        _within(lse, lse64, ltol, "lse V=%d %s" % (V, layout))
        # target: (1 - ls) on the label, ls / V elsewhere (eff_bert.py label smoothing through scatter_)
        neg = ls / V
        tgt = torch.full((rows, V), neg, dtype=f64, device="cuda").scatter_(1, labels.clamp(min=0)[:, None], 1.0 - ls)
        xr = x64.clone().requires_grad_()
        logp = torch.log_softmax(xr, 1)
        ref = -(tgt * logp).sum(1) * keep
        # loss = lse - x[lab] (+ ls / V (V lse - sum x) terms): lse's bound (times 1 + ls: the smoothing term carries V * lse * ls / V),
        # the roundings of x[lab] - lse and of the result, and for ls > 0 the 256-thread sum of x (V/256 + 8 levels) and V * lse
        xl = x64.gather(1, labels.clamp(min=0)[:, None])[:, 0]
        tol = (1 + ls) * ltol + 2 * U * (xl.abs() + lse64.abs() + ref.detach().abs())
        if ls > 0:
            tol = tol + neg * U * ((V / 256 + 10) * x64.abs().sum(1) + 2 * (x64.sum(1).abs() + V * lse64.abs()))
        _within(loss, ref.detach(), tol * keep, "xent rows V=%d %s ls=%g" % (V, layout, ls))
        (gref,) = torch.autograd.grad(ref, xr, g.double())
        d = K.xent_bwd(xv, labels, lse, g, -100, ls)
        # d_v = g (tsum p_v - tgt_v): p_v = __expf(x_v - lse) carries lse's error and __expf's; two roundings on each product
        p64 = torch.exp(logp.detach())
        tsum = tgt.sum(1, keepdim=True)
        tol = g.double().abs()[:, None] * keep[:, None] * (tsum * p64 * _p_rel(logp.detach(), ltol, x64) + 3 * U * (tsum * p64 + tgt))
        _within(d, gref, tol, "xent grad V=%d %s ls=%g" % (V, layout, ls))


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("V", VOCABS)
def test_kl_rows(K, V, layout):
    rows = 37
    pitch, off = LAYOUTS[layout](V)
    s = _logits(rows, V, seed=2 * V)
    t = _logits(rows, V, seed=2 * V + 1)
    sv = _row_view(s, pitch, off)
    tv = _row_view(t, pitch + 4, 0)          # the teacher's rows on a different pitch: ld_s != ld_t
    g = _randn(rows, seed=V + 3)
    for it in (1.0, 0.5, 0.25):
        ys, yt = s.double() * it, t.double() * it
        tol_s, lse_s = _lse_tol(ys)
        tol_t, lse_t = _lse_tol(yt)
        kl, ls_, lt_ = K.kl_fwd(sv, tv, it)
        _within(ls_, lse_s, tol_s, "kl student lse V=%d %s T=%g" % (V, layout, 1 / it))
        _within(lt_, lse_t, tol_t, "kl teacher lse V=%d %s T=%g" % (V, layout, 1 / it))
        sr = s.double().clone().requires_grad_()
        lps = torch.log_softmax(sr * it, 1)
        lpt = torch.log_softmax(yt, 1)
        pt = torch.exp(lpt)
        ref = (pt * (lpt - lps)).sum(1)
        # term_v = pt (lpt - lps): lpt / lps are off by the lse bound plus the roundings of y and y - lse; pt by that plus __expf's
        # error; the 256-thread sum of the terms adds V/256 + 8 roundings of sum |term|
        e_t = tol_t[:, None] + U * (yt.abs() + lpt.abs())
        e_s = tol_s[:, None] + U * (ys.abs() + lps.detach().abs())
        dl = (lpt - lps.detach()).abs()
        term = pt * dl
        tol = (term * _p_rel(lpt, tol_t, yt) + pt * (e_t + e_s) + 2 * U * term).sum(1) + U * (V / 256 + 10) * term.sum(1)
        _within(kl, ref.detach(), tol, "kl rows V=%d %s T=%g" % (V, layout, 1 / it))
        (gref,) = torch.autograd.grad(ref, sr, g.double())
        d = K.kl_bwd(sv, tv, ls_, lt_, g, it)
        # d_v = g it (ps_v - pt_v): each probability within its __expf bound, three roundings on the products
        ps = torch.exp(lps.detach())
        tol = (g.double() * it).abs()[:, None] * (ps * _p_rel(lps.detach(), tol_s, ys) + pt * _p_rel(lpt, tol_t, yt) + 3 * U * (ps + pt))
        _within(d, gref, tol, "kl grad V=%d %s T=%g" % (V, layout, 1 / it))


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("V", VOCABS)
def test_soft_xent_rows(K, V, layout):
    rows = 37
    pitch, off = LAYOUTS[layout](V)
    x = _logits(rows, V, seed=3 * V)
    # soft labels: ITC targets with idx are 1 / group size on a few entries; the other rows are dense distributions
    y = _rand(rows, V, seed=3 * V + 1)
    y[:rows // 2] = (y[:rows // 2] < min(0.5, 3.0 / V)).float()
    y[:rows // 2, 0] = 1.0
    y = y / y.sum(1, keepdim=True)
    xv = _row_view(x, pitch, off)
    yv = _row_view(y, pitch + 3, 0)
    x64, y64 = x.double(), y.double()
    ltol, lse64 = _lse_tol(x64)
    loss, lse = K.soft_xent_fwd(xv, yv)
    _within(lse, lse64, ltol, "soft xent lse V=%d %s" % (V, layout))
    xr = x64.clone().requires_grad_()
    logp = torch.log_softmax(xr, 1)
    ref = -(y64 * logp).sum(1)
    # -sum y (x - lse): (x - lse) off by the lse bound and two roundings; the 256-thread sum adds V/256 + 8 roundings
    lp = logp.detach()
    tol = (y64 * (ltol[:, None] + 2 * U * (x64.abs() + lp.abs()))).sum(1) + U * (V / 256 + 10) * (y64 * lp.abs()).sum(1)
    _within(loss, ref.detach(), tol, "soft xent rows V=%d %s" % (V, layout))
    g = _randn(rows, seed=V + 4)
    (gref,) = torch.autograd.grad(ref, xr, g.double())
    d = K.soft_xent_bwd(xv, yv, lse, g)
    # d_v = g (sum(y) p_v - y_v): sum(y) is a 256-thread sum (V/256 + 8 roundings), p_v within its __expf bound
    p64 = torch.exp(lp)
    ys = y64.sum(1, keepdim=True)
    tol = g.double().abs()[:, None] * (ys * p64 * (_p_rel(lp, ltol, x64) + U * (V / 256 + 10)) + 3 * U * (ys * p64 + y64))
    _within(d, gref, tol, "soft xent grad V=%d %s" % (V, layout))


# ------------------------------------------------------------------------------------------------ multi-pair MSE
def _probs(shape, Lk, seed):
    """Attention-map-like rows: [..., pitch] with the first Lk columns a probability distribution and exact zeros in the pad."""
    p = _rand(*shape, seed=seed)
    p[..., Lk:] = 0
    return p / p.sum(-1, keepdim=True)


def _mse_table():
    """(students, teachers, scales, want_rowdot) shaped like distill.gd_kd_losses at batch 128 (ViT and cross maps at smaller batches):
    hidden states in every fp32 / bf16 combination, text maps (row_len 40), ViT maps on the 200-float pitch (row_len 200), cross maps
    40 x 197 on the same pitch, 577-token ViT maps on the 580 pitch, odd element counts, and one fp32 map that starts one float past an
    allocation (every vector path refused: the scalar path)."""
    S, T, W, R = [], [], [], []
    dts = [(f32, f32), (bf16, f32), (f32, bf16), (bf16, bf16)]

    def add(s, t, w, r):
        S.append(s)
        T.append(t)
        W.append(w)
        R.append(r)
    seed = 100
    for i in range(13):
        ds, dt = dts[i % 4]
        add(_randn(128, 40, 768, seed=seed).to(ds), _randn(128, 40, 768, seed=seed + 1).to(dt), 1.0, False)
        seed += 2
    for i in range(12):
        dt = bf16 if i == 11 else f32
        add(_probs((128, 12, 40, 40), 40, seed), _probs((128, 12, 40, 40), 40, seed + 1).to(dt), 40.0, True)
        seed += 2
    for i in range(12):
        add(_probs((8, 12, 197, 200), 197, seed), _probs((8, 12, 197, 200), 197, seed + 1), 197.0 * 200 / 197, True)
        seed += 2
    for i in range(6):
        add(_probs((32, 12, 40, 200), 197, seed), _probs((32, 12, 40, 200), 197, seed + 1), 197.0 * 200 / 197, True)
        seed += 2
    for i in range(2):
        add(_probs((2, 12, 577, 580), 577, seed), _probs((2, 12, 577, 580), 577, seed + 1), 577.0 * 580 / 577, True)
        seed += 2
    shifted = torch.full((1 + 8 * 12 * 40 * 200,), NAN, device="cuda")
    s = shifted[1:].view(8, 12, 40, 200)
    s.copy_(_probs((8, 12, 40, 200), 197, seed))
    assert s.data_ptr() % 16 == 4
    add(s, _probs((8, 12, 40, 200), 197, seed + 1), 197.0, True)
    add(_randn(3, 7, 13, seed=seed + 2), _randn(3, 7, 13, seed=seed + 3).to(bf16), 1.0, False)
    add(_randn(5, 1001, seed=seed + 4).to(bf16), _randn(5, 1001, seed=seed + 5).to(bf16), 0.5, False)
    add(_randn(1, 1, 3, seed=seed + 6).to(bf16), _randn(1, 1, 3, seed=seed + 7), 2.0, False)
    add(_randn(4, 40, 42, seed=seed + 8), _randn(4, 40, 42, seed=seed + 9), 3.0, True)     # row_len % 4 != 0: no rowdot
    return S, T, W, R


def test_mse_pairs_table(K):
    S, T, W, R = _mse_table()
    n_pairs = len(S)
    assert n_pairs >= 50
    out, rd_f = K.mse_pairs_fwd(S, T, W, want_rowdot=R)
    dout = _randn(n_pairs, seed=7)
    need = [i != 5 for i in range(n_pairs)]
    grads, rd_b = K.mse_pairs_bwd(S, T, W, dout, need, want_rowdot=[s.dim() == 4 for s in S])
    assert grads[5] is None
    for i, (s, t, w) in enumerate(zip(S, T, W)):
        what = "pair %d %s %s/%s" % (i, tuple(s.shape), str(s.dtype)[6:], str(t.dtype)[6:])
        s64, t64 = s.double(), t.double()
        n = s.numel()
        d = s64 - t64
        ref = w * (d * d).sum() / n
        # positive terms: each thread sums <= n / (888 * 256) + 4 of them, a block tree of 8 levels, 888 atomics into the slot,
        # 3 roundings per squared difference and 3 on scale / n
        chunk = n / (888 * 256) + 4
        _within(out[i], ref, U * (chunk + 8 + 888 + 6) * ref, "mse loss " + what)
        row_len = s.shape[-1]
        if R[i] and s.dtype == f32 and t.dtype == f32 and row_len % 4 == 0:
            assert rd_f[i] is not None, what
            # a row's sum of (s - t) s over row_len terms of mixed sign: <= row_len + 16 roundings of sum |term|, whichever path
            # (warp per row, or one atomic per element) the pair takes
            term = (d * s64).view(-1, row_len)
            _within(rd_f[i], term.sum(1), U * (row_len + 16) * term.abs().sum(1), "mse rowdot fwd " + what)
        else:
            assert rd_f[i] is None, what
        if not need[i]:
            continue
        k = float(dout[i]) * w * 2.0 / n
        gref = k * d
        # k = dout scale 2 / n rounds 3 times, k (s - t) twice
        _within(grads[i], gref, 6 * U * gref.abs(), "mse grad " + what)
        if s.dim() == 4 and s.dtype == f32 and row_len % 4 == 0:
            assert rd_b[i] is not None, what
            term = (gref * s64).view(-1, row_len)
            # ds carries 6 U; the row sum <= row_len + 16 roundings (float4 dot, segmented warp sums, one atomic per warp or element)
            _within(rd_b[i], term.sum(1), U * (row_len + 22) * term.abs().sum(1), "mse rowdot bwd " + what)
        else:
            assert rd_b[i] is None, what


# ------------------------------------------------------------------------------------------------ reduce_sum, l2norm, ITM sampling
@pytest.mark.parametrize("n", [1, 1023, 100003, 5_000_000])
def test_reduce_sum(K, n):
    x = _randn(n, seed=n)
    x64 = x.double()
    blocks = min(592, max(1, (n + 255) // 256))
    # per thread <= n / (blocks 256) + 1 terms, 8 tree levels, `blocks` atomics, the scale and the accumulated start value
    steps = n / (blocks * 256) + 1 + 8 + blocks + 2
    for acc, start in ((False, 0.0), (True, 3.25)):
        out = torch.full((), start, device="cuda")
        K.reduce_sum(x, 0.5, out, acc)
        ref = start + 0.5 * x64.sum()
        _within(out, ref, U * (steps * 0.5 * x64.abs().sum() + 2 * abs(start)), "reduce_sum n=%d accumulate=%s" % (n, acc))


@pytest.mark.parametrize("D", [256, 100])
def test_l2norm(K, D):
    rows = 1023                                   # not a multiple of the 4 rows per 128-thread block
    x = _randn(rows, D, seed=D, scale=3.0)
    x[17] = 0.0
    y, inv = K.l2norm_fwd(x)
    x64 = x.double()
    xr = x64.clone().requires_grad_()
    ref = torch.nn.functional.normalize(xr, dim=-1, eps=1e-12)
    nrm = x64.norm(dim=1)
    # sum of squares: each lane D/32 terms, 5 shuffle levels, 1 rounding per square: relative (D/32 + 6) U; sqrt and the reciprocal
    # add 2 U, the product 1 U
    rel = U * ((D / 32 + 6) / 2 + 4)
    _within(y, ref.detach(), rel * ref.detach().abs(), "l2norm y D=%d" % D)
    inv_ref = 1.0 / torch.clamp(nrm, min=float(torch.tensor(1e-12, dtype=f32)))
    _within(inv, inv_ref, rel * inv_ref, "l2norm inv D=%d" % D)
    assert float(y[17].abs().max()) == 0.0 and float(inv[17]) == float(1.0 / torch.tensor(1e-12, dtype=f32))
    dy = _randn(rows, D, seed=D + 1)
    (gref,) = torch.autograd.grad(ref, xr, dy.double())
    dx = K.l2norm_bwd(dy, y, inv)
    # dx = inv (dy - y <dy, y>): <dy, y> is a D-term warp sum (D/32 + 6 roundings of sum |dy y|) over a y that carries `rel`, which
    # enters again through y <dy, y>; the difference and the products round 3 times; inv's `rel` scales the whole result
    y64, dy64 = ref.detach(), dy.double()
    s_abs = (dy64 * y64).abs().sum(1, keepdim=True)
    s = (dy64 * y64).sum(1, keepdim=True)
    tol = inv_ref[:, None] * (y64.abs() * s_abs * (U * (D / 32 + 6) + 2 * rel) + 3 * U * (dy64.abs() + (y64 * s).abs())) + rel * gref.abs()
    _within(dx, gref, tol, "l2norm grad D=%d" % D)


@pytest.mark.parametrize("grouped", [False, True])
@pytest.mark.parametrize("B", [64, 128])
def test_itm_sample_neg(K, B, grouped):
    sim = _randn(B, B, seed=B, scale=4.0)
    if grouped:
        idx = torch.randint(0, B // 3, (B,), generator=_gen(B + 1), device="cuda")
        idx[0] = idx[1] = idx[2]
    else:
        idx = None
    u = _rand(B, seed=B + 2)
    u[0], u[1], u[2], u[3] = 0.0, 1e-7, 1.0 - 2.0 ** -24, 0.5
    # very peaked rows: one allowed entry carries ~all of the softmax, and u lands in the part of the CDF that only the +1e-5 floor
    # of every other allowed entry makes up: the draw must fall past the peak
    ex = torch.eye(B, dtype=torch.bool, device="cuda") if idx is None else idx[:, None] == idx[None, :]
    for r in (4, 5):
        j0 = int((~ex[r]).nonzero()[0]) if r == 4 else int((~ex[r]).nonzero()[-1])
        sim[r] = -20.0
        sim[r, j0] = 60.0
        u[r] = 0.99995 if r == 4 else 1e-6
    neg = K.itm_sample_neg(sim, idx, u).long()
    assert bool(((neg >= 0) & (neg < B)).all())
    assert not bool(ex.gather(1, neg[:, None]).any()), "drew an excluded (positive or same-idx) entry"
    w = (torch.softmax(sim.double(), 1) + 1e-5).masked_fill(ex, 0.0)
    C = torch.cumsum(w, 1)
    tot = C[:, -1]
    target = u.double() * tot
    # the kernel's running sum and total are off by <= B + 16 roundings of the (positive) total: each weight is __expf (2 ulp) / s
    # (a 32-lane sum: B/32 + 5 roundings) + 1e-5, the running sum adds <= B terms, the total is a warp sum, target one product
    tol = U * (B + 16) * tot
    c_hi = C.gather(1, neg[:, None])[:, 0]
    c_lo = c_hi - w.gather(1, neg[:, None])[:, 0]
    ok = (c_lo - tol <= target) & (target <= c_hi + tol)
    assert bool(ok.all()), "inverse-CDF draw outside its bin on rows %s" % ok.logical_not().nonzero()[:, 0].tolist()
    j4 = int((~ex[4]).nonzero()[0])
    assert int(neg[4]) > j4, "the +1e-5 floor must carry the draw past the peak"
    assert int(neg[5]) == int((~ex[5]).nonzero()[0])


# ------------------------------------------------------------------------------------------------ L0 gates
L0_L, L0_R, BETA, MAGIC = -0.1, 1.1, 2.0 / 3.0, 0.8
LOGIT0 = math.log(1.0 / 12.0) - math.log(11.0 / 12.0)        # log(xn / (1 - xn)), xn = (0 - l) / (r - l)
B32 = float(torch.tensor(BETA, dtype=f32))                     # the kernels see beta (and logit0) as fp32
LOGIT0_32 = float(torch.tensor(LOGIT0, dtype=f32))


def _l0_inputs(L, size, seed):
    loga = torch.empty(L, size, device="cuda").uniform_(-6.0, 6.0, generator=_gen(seed))
    u = _rand(L, size, seed=seed + 1).clamp(1e-6, 1 - 1e-6)   # l0_module.get_eps clamps the same way
    u.view(-1)[:64] = 1e-6                                     # the hardtanh clamps at both ends
    u.view(-1)[64:128] = 1 - 1e-6
    return loga, u


@pytest.mark.parametrize("size", [12, 3072])
@pytest.mark.parametrize("L", [6, 12])
def test_l0_sample(K, L, size):
    loga, u = _l0_inputs(L, size, seed=L * size)
    lr = loga.double().clone().requires_grad_()
    u64 = u.double()
    lu, l1u = torch.log(u64), torch.log1p(-u64)
    x = (lu - l1u + lr) / B32
    y = torch.sigmoid(x)
    zz = y * (L0_R - L0_L) + L0_L
    z64 = torch.nn.functional.hardtanh(zz, 0.0, 1.0)
    # x = (logf(u) - logf(1 - u) + loga) / beta: 1 ulp per logf, 1 - u rounds once (<= U absolute on its log), two adds and a
    # division; y = 1 / (1 + expf(-x)) adds 3 U y; z = y (r - l) + l: the clamped affine map is 1.2-Lipschitz, plus 2 roundings
    ex = (U * (2 * lu.abs() + 3 * l1u.abs() + 2 * loga.double().abs() + 2) / B32 + U * x.detach().abs())
    ey = y.detach() * (1 - y.detach()) * ex + 3 * U * y.detach()
    ez = 1.2 * ey + 2 * U
    z = K.l0_sample_fwd(loga, u, BETA)
    _within(z, z64.detach(), ez, "l0 z [%d, %d]" % (L, size))
    clear = ((zz.detach() < -ez) | (zz.detach() > ez))
    assert torch.equal((z == 0)[clear], (z64.detach() == 0)[clear])
    clear1 = ((zz.detach() - 1).abs() > ez)
    assert torch.equal((z == 1)[clear1], (z64.detach() >= 1)[clear1])
    assert int((z == 0).sum()) > 0 and int((z == 1).sum()) > 0
    dz = _rand(L, size, seed=L + size + 7)
    (gref,) = torch.autograd.grad(z64, lr, dz.double())
    d = K.l0_sample_bwd(loga, u, dz, BETA)
    # where the hardtanh passes, y is in (1/12, 11/12): y and 1 - y are each within 12 ey relatively, 1 - y rounds once, and
    # dz (r - l) y (1 - y) / beta four more times; entries within ez of a clamp edge may fall either way and are skipped
    inner = clear & clear1
    tol = gref.abs() * (24 * ey + 6 * U)
    _within(d[inner], gref[inner], tol[inner], "l0 dloga [%d, %d]" % (L, size))
    assert bool((d[~(zz.detach() > -ez) | ~(zz.detach() < 1 + ez)] == 0).all())


def _cdf64(loga64):
    s = torch.sigmoid(LOGIT0_32 * B32 - loga64)
    return s, s.clamp(1e-6, 1 - 1e-6)


@pytest.mark.parametrize("size", [12, 3072])
@pytest.mark.parametrize("L", [6, 12])
def test_l0_expected(K, L, size):
    loga = torch.empty(L, size, device="cuda").uniform_(-10.0, 10.0, generator=_gen(L * size + 3))
    # a few entries deep inside the eps clamp of the CDF (zero gradient) at both ends; the rest stay clear of its edges at
    # logit0 * beta -+ 13.8
    c = LOGIT0_32 * B32
    loga.view(-1)[:5] = c + 20.0
    loga.view(-1)[5:10] = c - 20.0
    weight = _fp32(0.37 * size)
    lr = loga.double().clone().requires_grad_()
    _, cdf = _cdf64(lr)
    e = weight * (1 - cdf).sum()
    start = 11.5
    out = torch.full((), start, device="cuda")
    K.l0_expected_fwd(loga, BETA, weight, out, True)
    n = loga.numel()
    blocks = min(148, (n + 255) // 256)
    # each term 1 - cdf is within 6 U (absolute: the argument's rounding moves s by <= 0.5 U, expf / add / division 4 U s, the
    # subtraction U); positive sum: per thread <= n / (blocks 256) + 1 terms, 8 tree levels, `blocks` atomics; weight and the start
    # value round twice more
    tol = weight * U * (6 * n + (n / (blocks * 256) + 1 + 8 + blocks + 2) * float(e.detach()) / weight) + 2 * U * abs(start)
    _within(out, start + e.detach(), tol, "l0 expected (accumulated)")
    gval = _fp32(1.7)
    g = torch.tensor([gval], device="cuda")
    (gref,) = torch.autograd.grad(e, lr, torch.tensor(gval, dtype=f64, device="cuda"))
    d0 = _randn(L, size, seed=5)
    d = d0.clone()
    K.l0_expected_bwd(loga, BETA, weight, g, d)
    # d += g weight s (1 - s): s within 5 U (as above), so s (1 - s) within 6 U absolutely; the products and the accumulate round
    # 3 times more
    _within(d, d0.double() + gref, 6 * U * abs(gval * weight) + 4 * U * (d0.double().abs() + gref.abs()), "l0 expected dloga (+=)")
    assert bool((d.view(-1)[:10] == d0.view(-1)[:10]).all())


def _det_loga(L, size, seed):
    """Rows of distinct log-alphas on a grid (spacing 8 / 3072, |loga| <= 6.5: the fp32 soft scores keep their fp64 order), rows of
    planted ties (each value three times), one row with every entry far above the CDF edge (n0 = 0) and one far below (n0 = size)."""
    g = _gen(seed)
    rows = []
    for r in range(L):
        shift = -2.5 + 5.0 * r / max(L - 1, 1)
        if r % 3 == 1:
            vals = torch.linspace(-4.0, 4.0, (size + 2) // 3, device="cuda").repeat(3)[:size]
        else:
            vals = torch.linspace(-4.0, 4.0, size, device="cuda")
        rows.append(vals[torch.randperm(size, generator=g, device="cuda")] + shift)
    loga = torch.stack(rows)
    c = LOGIT0_32 * B32
    loga[L - 2] = c + 25.0 + torch.linspace(0, 1, size, device="cuda")
    loga[L - 1] = c - 25.0 - torch.linspace(0, 1, size, device="cuda")
    return loga


@pytest.mark.parametrize("size", [12, 3072])
@pytest.mark.parametrize("L", [6, 12])
def test_l0_deterministic(K, L, size):
    loga = _det_loga(L, size, seed=L + size)
    mask, kept = K.l0_deterministic(loga, BETA, MAGIC)
    m = mask.cpu().numpy()
    assert set(np.unique(m).tolist()) <= {0.0, 1.0}
    assert torch.equal(kept.cpu().long(), mask.cpu().sum(1).long()), "kept = row sums of the mask"
    l64 = loga.double()
    _, cdf = _cdf64(l64)
    E = (size - (1 - cdf).sum(1)).cpu().numpy()                 # expected number of zeros per row
    # fp32: each 1 - cdf within 6 U (test_l0_expected), a 256-thread sum (size / 256 + 8 roundings of a sum <= size), size - acc
    # rounds once
    delta = U * (6 * size + (size / 256 + 8) * size + size)
    soft = torch.sigmoid(l64 / B32 * MAGIC).cpu().numpy()
    ambiguous = 0
    for r in range(L):
        n0 = int(size - m[r].sum())
        want = round(float(E[r]))
        near_half = abs((E[r] - math.floor(E[r])) - 0.5) <= delta
        if near_half:
            ambiguous += 1
            assert n0 in (math.floor(E[r]), math.ceil(E[r])), (r, n0, E[r])
        else:
            assert n0 == want, "row %d: %d zeros, round(%.6f) = %d" % (r, n0, E[r], want)
        if r < L - 2:
            s = np.sort(np.unique(soft[r]))
            # distinct scores differ by >= 1.2e-6, far beyond the few-ulp (< 3e-7) error of the kernel's fp32 sigmoid: its order is
            # the fp64 order
            assert s.size < 2 or np.diff(s).min() > 1e-6, "the grid must keep distinct soft scores apart in fp32"
        order = np.lexsort((np.arange(size), soft[r]))         # ascending soft score, ties -> lower index first
        want_mask = np.ones(size)
        want_mask[order[:n0]] = 0.0
        assert np.array_equal(m[r], want_mask), "row %d: zeroed set is not the %d smallest soft scores (ties to the lower index)" % (r, n0)
    assert ambiguous <= max(1, L // 4)
    assert m[L - 2].sum() == size and m[L - 1].sum() == 0        # n0 == 0 and n0 == size
    assert any(0 < m[r].sum() < size for r in range(L - 2))


# ------------------------------------------------------------------------------------------------ optimizer
B1, B2, EPS = 0.9, 0.999, 1e-6


def _fp32(x):
    return float(np.float32(x))


def _adamw_groups():
    """Three groups inside one 256-byte-aligned arena, each padded to 64 floats like optim.py's ARENA_ALIGN, different lr and
    weight decay (one without decay); a bf16 shadow arena beside it."""
    sizes = [64 * 1000, 64 * 37, 64 * 4099]
    hp = [(1e-3, 0.01), (5e-4, 0.0), (2e-5, 0.1)]
    n = sum(sizes)
    arena = {k: torch.zeros(n, device="cuda") for k in ("p", "g", "m", "v")}
    arena["p"].copy_(_randn(n, seed=11))
    shadow = torch.zeros(n, dtype=bf16, device="cuda")
    groups, o = [], 0
    for sz, (lr, wd) in zip(sizes, hp):
        gr = {k: arena[k][o:o + sz] for k in arena}
        gr.update(p_bf16=shadow[o:o + sz], lr=lr, beta1=B1, beta2=B2, eps=EPS, weight_decay=wd)
        assert gr["p"].data_ptr() % 256 == 0 and gr["p_bf16"].data_ptr() % 128 == 0
        groups.append(gr)
        o += sz
    return groups, arena, shadow


def _hyper(groups, t):
    """(step_size, lr * weight_decay) per group as the host half of adamw_step computes them (fp32 parameters, fp64 bias correction)."""
    vals = []
    for gr in groups:
        lr, b1, b2 = _fp32(gr["lr"]), _fp32(gr["beta1"]), _fp32(gr["beta2"])
        ss = lr * math.sqrt(1.0 - math.pow(b2, float(t))) / (1.0 - math.pow(b1, float(t)))
        vals += [_fp32(ss), float(np.float32(gr["lr"]) * np.float32(gr["weight_decay"]))]
    return vals


@pytest.mark.parametrize("scaled", [False, True])
def test_adamw_float4_path(K, scaled):
    groups, arena, shadow = _adamw_groups()
    twin = {k: v.clone() for k, v in arena.items()}
    twin_shadow = shadow.clone()
    tgroups = []
    o = 0
    for gr in groups:
        sz = gr["p"].numel()
        tg = dict(gr, **{k: twin[k][o:o + sz] for k in twin}, p_bf16=twin_shadow[o:o + sz])
        tgroups.append(tg)
        o += sz
    hyper = torch.zeros(2 * len(groups), device="cuda")
    gs = torch.tensor([0.37], device="cuda") if scaled else None
    gs64 = _fp32(0.37) if scaled else 1.0
    ref = [{k: gr[k].double().clone() for k in ("p", "m", "v")} for gr in groups]
    err = [{k: torch.zeros_like(r["p"]) for k in ("p", "m", "v")} for r in ref]
    for i, t in enumerate((1, 2, 10, 1000)):
        arena["g"].copy_(_randn(arena["g"].numel(), seed=20 + i, scale=1e-2))
        twin["g"].copy_(arena["g"])
        for gr, tg in zip(groups, tgroups):
            gr["step"] = tg["step"] = t
        K.adamw_step(groups, gs)
        K.store_f32(hyper, _hyper(groups, t))
        K.adamw_step(tgroups, gs, hyper_dev=hyper)
        for gr, r, e in zip(groups, ref, err):
            lr, b1, b2, eps, wd = (_fp32(gr[k]) for k in ("lr", "beta1", "beta2", "eps", "weight_decay"))
            g = gr["g"].double() * gs64
            # HF AdamW (transformers.optimization.AdamW): EMAs, bias-corrected step size, then decoupled decay p -= lr wd p
            mag_m = b1 * r["m"].abs() + (1 - b1) * g.abs()
            r["m"] = b1 * r["m"] + (1 - b1) * g
            r["v"] = b2 * r["v"] + (1 - b2) * g * g
            ss = lr * math.sqrt(1 - b2 ** t) / (1 - b1 ** t)
            den = r["v"].sqrt() + eps
            upd = ss * r["m"] / den
            p_mid = r["p"] - upd
            r["p"] = p_mid - (lr * wd) * p_mid if wd != 0 else p_mid
            # running error bounds of the fp32 state: m and v contract by beta and pick up 4 / 5 roundings (grad scale, two
            # products, the sum; g^2 once more) of their terms' magnitudes; the update carries m's error, v's through sqrt (half
            # the relative error), 4 roundings (fp32 step size, sqrt, add, divide, multiply); p picks up the update's error and two
            # roundings (subtract, decay), the decay term one more
            e["m"] = b1 * e["m"] + 4 * U * mag_m
            e["v"] = b2 * e["v"] + 5 * U * r["v"]
            e_upd = ss * e["m"] / den + upd.abs() * (e["v"] / r["v"].clamp_min(1e-300) / 2 + 6 * U)
            e["p"] = e["p"] + e_upd + 2 * U * p_mid.abs() + 2 * U * (lr * wd) * p_mid.abs()
            what = "adamw step %d lr=%g wd=%g scaled=%s" % (t, lr, wd, scaled)
            _within(gr["m"], r["m"], e["m"], what + " m")
            _within(gr["v"], r["v"], e["v"], what + " v")
            _within(gr["p"], r["p"], e["p"], what + " p")
        assert torch.equal(shadow, arena["p"].to(bf16)), "bf16 shadow != p.to(bf16) after step %d" % t
        for k in ("p", "m", "v"):
            assert torch.equal(twin[k], arena[k]), "adamw_step_dev (device hyper) differs from adamw_step in %s at step %d" % (k, t)
        assert torch.equal(twin_shadow, shadow)


@pytest.mark.parametrize("offset", [0, 1])
@pytest.mark.parametrize("n", [3, 4, 10007, 2_500_000])
def test_sumsq(K, n, offset):
    buf = _randn(n + 4, seed=n)
    x = buf[offset:offset + n]
    assert (x.data_ptr() % 16 == 0) == (offset == 0)
    blocks = min(592, max(1, (n // 4 + 255) // 256))
    start = 1.25
    outs = []
    for _ in range(2):
        out = torch.full((1,), start, device="cuda")
        K.sumsq(x, out)
        outs.append(out)
    assert torch.equal(outs[0], outs[1]), "sumsq is not bit-identical between two runs"
    x64 = x.double()
    ref = start + (x64 * x64).sum()
    # positive terms: per thread <= n / (blocks 256) + 4 of them (4 per float4, plus the scalar tail), 8 tree levels, the last block's
    # strided sum over `blocks` partials (blocks / 256 + 1) and its 8 tree levels, one rounding per square, the accumulate into `out`
    steps = n / (blocks * 256) + 4 + 8 + blocks / 256 + 1 + 8 + 1 + 1
    _within(outs[0], ref.view(1), U * steps * ref.view(1), "sumsq n=%d offset=%d" % (n, offset))


def test_clip_coef(K):
    c = torch.empty(1, device="cuda")
    for ss, max_norm in ((0.25, 1.0), (100.0, 1.0), (3.9, 2.0), (4.1, 2.0)):
        K.clip_coef(torch.tensor([ss], device="cuda"), max_norm, c)
        want = min(1.0, max_norm / (math.sqrt(ss) + 1e-6))
        if want == 1.0:
            assert float(c) == 1.0, (ss, max_norm, float(c))
        else:
            assert abs(float(c) - want) <= 4 * U * want, (ss, max_norm, float(c), want)   # sqrt, add, divide, fp32 1e-6


# ------------------------------------------------------------------------------------------------ ITC sgemm / dot
@pytest.mark.parametrize("MN", [128, 1024])
@pytest.mark.parametrize("Kd", [256, 250])
@pytest.mark.parametrize("a_trans,b_trans", [(False, False), (False, True), (True, False), (True, True)])
def test_sgemm(K, MN, Kd, a_trans, b_trans):
    M = N = MN
    A = _randn(*((Kd, M) if a_trans else (M, Kd)), seed=M + Kd)
    B = _randn(*((N, Kd) if b_trans else (Kd, N)), seed=M + Kd + 1)
    opA = A.double().t() if a_trans else A.double()
    opB = B.double().t() if b_trans else B.double()
    prod = opA @ opB
    mag = opA.abs() @ opB.abs()
    temp = torch.tensor([0.07], device="cuda")
    D0 = _randn(M, N, seed=3)
    for beta in (0.0, 0.5):
        for alpha_dev, inv in ((None, False), (temp, False), (temp, True)):
            a = _fp32(1.3)
            if alpha_dev is not None:
                a = a / _fp32(0.07) if inv else a * _fp32(0.07)
            D = D0.clone() if beta else torch.full((M, N), NAN, device="cuda")     # beta = 0 must not read D
            K.sgemm(A, B, D, M, N, Kd, alpha=1.3, a_trans=a_trans, b_trans=b_trans, beta=beta, alpha_dev=alpha_dev, alpha_dev_inv=inv)
            ref = a * prod + (beta * D0.double() if beta else 0.0)
            # a K-term fp32 dot product is within K U sum |a b|; the effective alpha rounds once, alpha acc and beta D once each and
            # their sum once
            tol = U * ((Kd + 3) * abs(a) * mag + 3 * abs(beta) * D0.double().abs() + 2 * ref.abs())
            _within(D, ref, tol, "sgemm %dx%dx%d trans=%d%d beta=%g alpha_dev=%s inv=%d" % (
                M, N, Kd, a_trans, b_trans, beta, alpha_dev is not None, inv))


def test_dot(K):
    n = 1024 * 1024
    x, y = _randn(n, seed=1), _randn(n, seed=2)
    p = x.double() * y.double()
    blocks = 592
    steps = n / (blocks * 256) + 1 + 8 + blocks + 2      # per-thread terms, tree, atomics, scale and accumulate
    out = torch.full((), 2.0, device="cuda")
    K.dot(x, y, out, scale=-1.0, accumulate=True)
    ref = 2.0 - p.sum()
    _within(out, ref, U * (steps * p.abs().sum() + 2 * 2.0), "dot accumulate")
    K.dot(x, y, out, scale=0.25)
    _within(out, 0.25 * p.sum(), U * steps * 0.25 * p.abs().sum(), "dot")
