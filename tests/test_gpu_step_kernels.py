"""Kernel-level tests of the training step's scorer, loss, user-pooling, reduction, small-table, optimizer and streaming
recurrence entry points (score.cu, userpool.cu, attn.cu lstur_colsum, gather.cu, optim.cu, gru.cu) against float64
references of the same operation.

Every output is filled with NaN before the call, so an element the kernel does not write fails.  Strided arguments get
a leading dimension larger than the width, with NaN in the pad columns of inputs (a read past the width shows) and of
outputs (a write past the width shows).  Bounds, with u = 2^-23:
  element-wise results   a few u of the magnitude of the terms;
  sums of n terms        n u sum|terms| (several of these sums cancel, so a bound relative to the result is wrong);
  recurrences            the 2e-5 norm-wise bound of test_gpu_gru.py.
Sums the kernels do in a fixed order are run twice and compared byte for byte."""
import ctypes
import dataclasses
import itertools

import numpy as np
import pytest
import torch

from oracle import lstur_torch as ot
from oracle.lstur_numpy import adam_step
from test_gpu_gru import make as gru_make, oracle as gru_oracle
from tolerances import rel

pytestmark = pytest.mark.gpu

U32 = 2.0 ** -23
ERR_ARG = -1
NAN = float('nan')
F32 = lambda x: float(np.float32(x))


# Device tensors whose addresses were handed to a kernel.  A temporary such as P_(dev(x)) would otherwise go back to the
# caching allocator before the kernel is even enqueued, and the next allocation would reuse its memory; they are
# released only after the device has finished with them (sync()).
_in_flight = []


def P_(t):
    if t is None:
        return None
    _in_flight.append(t)
    return ctypes.c_void_p(t.data_ptr())


def sync():
    torch.cuda.synchronize()
    _in_flight.clear()


@pytest.fixture(autouse=True)
def _release_in_flight():
    yield
    sync()


def st():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def ok(lib, rc):
    assert rc == 0, lib.lstur_last_error().decode()


def dev(a, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(a)).to(dtype).cuda()


def nans(*shape):
    return torch.full(shape, NAN, device='cuda')


def host(t):
    sync()
    return t.detach().cpu().numpy().astype(np.float64)


def strided(a, ld, dtype=torch.float32):
    """(rows, w) array -> (rows, ld) device buffer: the rows in the first w columns, NaN in the pad."""
    a = np.asarray(a)
    out = np.full((a.shape[0], ld), np.nan, dtype=np.float64)
    out[:, :a.shape[1]] = a
    return dev(out, dtype)


def within(got, ref, bound, what=''):
    got, ref, bound = (np.asarray(x, dtype=np.float64) for x in (got, ref, bound))
    assert np.isfinite(got).all(), '%s: %d non-finite elements' % (what, int((~np.isfinite(got)).sum()))
    err = np.abs(got - ref)
    bad = err > np.broadcast_to(bound, err.shape)
    if bad.any():
        i = np.unravel_index(np.argmax(err - bound), err.shape)
        raise AssertionError('%s: %d elements out of bound; worst at %s: got %r ref %r bound %r'
                             % (what, int(bad.sum()), i, got[i], ref[i], np.broadcast_to(bound, err.shape)[i]))


def pad_untouched(buf, w, what=''):
    """the columns beyond the width of an ld-strided output are still NaN"""
    assert torch.isnan(buf[:, w:]).all().item(), what + ': wrote past the row width'


def rng(seed):
    return np.random.default_rng(seed)


def f32(a):
    return np.asarray(a, dtype=np.float32).astype(np.float64)


# ============================================================================================ 1. loss heads
def softmax_ce_ref(s, y, scale):
    """(1+K)-way softmax + Keras categorical cross-entropy (probabilities renormalised, clipped to [1e-7, 1 - 1e-7]
    in float32, zero gradient through a saturated clip) from float64 logits s (B, C)."""
    lo, hi = F32(1e-7), F32(1 - 1e-7)
    e = np.exp(s - s.max(1, keepdims=True))
    p = e / e.sum(1, keepdims=True)
    q = p / p.sum(1, keepdims=True)
    inr = (q >= lo) & (q <= hi)
    loss = -(y * np.log(np.clip(q, lo, hi))).sum(1)
    g = np.where(inr & (y != 0), -y / q, 0.0)
    gp = (g * p).sum(1, keepdims=True)
    ds = p * (g - gp) * scale
    ds_abs = p * (np.abs(g) + np.abs(gp)) * abs(scale)   # magnitude of the terms of ds (ds itself cancels)
    return p, loss, ds, ds_abs


def label_rows(kind, B, C, g):
    if kind == 'none':
        return None
    y = np.zeros((B, C), np.float32)
    if kind == 'onehot':                     # the positive anywhere, the last column included
        col = g.integers(0, C, B)
        col[0] = C - 1
        y[np.arange(B), col] = 1
    else:                                    # two positives per row
        for b in range(B):
            y[b, g.choice(C, size=min(2, C), replace=False)] = 1
    return y


def run_softmax_ce(lib, u, d, y, scale, pad=(3, 5, 2, 7), mean=False, grads=True):
    B, D = u.shape
    C = d.shape[0] // B
    ldu, ldd, lddu, lddd = D + pad[0], D + pad[1], D + pad[2], D + pad[3]
    ud, dd_in = strided(u, ldu), strided(d, ldd)
    yd = dev(y) if y is not None else None
    logits, probs, loss_rows = nans(B, C), nans(B, C), nans(B)
    loss_mean = nans(1) if mean else None
    du, dd = (nans(B, lddu), nans(B * C, lddd)) if grads else (None, None)
    ok(lib, lib.lstur_score_softmax_ce(B, C, D, P_(ud), ldu, P_(dd_in), ldd, P_(yd), P_(logits), P_(probs), P_(loss_rows),
                                       P_(loss_mean), P_(du), lddu, P_(dd), lddd, scale, st()))
    sync()
    if grads:
        pad_untouched(du, D, 'du')
        pad_untouched(dd, D, 'dd')
        du, dd = du[:, :D], dd[:, :D]
    return logits, probs, loss_rows, loss_mean, du, dd


def check_softmax_ce(u, d, y, scale, out):
    logits, probs, loss_rows, loss_mean, du, dd = [host(t) if t is not None else None for t in out]
    B, D = u.shape
    C = d.shape[0] // B
    u64, d64 = f32(u), f32(d).reshape(B, C, D)
    s = np.einsum('bk,bck->bc', u64, d64)
    s_abs = np.einsum('bk,bck->bc', np.abs(u64), np.abs(d64))
    within(logits, s, D * U32 * s_abs + 1e-37, 'logits')
    y64 = np.zeros((B, C)) if y is None else f32(y)
    if y is None:
        y64[:, 0] = 1
    # the softmax from the kernel's own logits: isolates it from the dot products checked above
    p, loss, ds, ds_abs = softmax_ce_ref(logits, y64, scale)
    k = C + 8
    within(probs, p, k * U32 * p + 1e-37, 'probs')
    within(loss_rows, loss, k * U32 * (y64.sum(1) + np.abs(loss)), 'loss_rows')
    if loss_mean is not None:
        within(loss_mean[0], loss_rows.mean(), (B + 2) * U32 * np.abs(loss_rows).mean(), 'loss_mean')
    if du is not None:
        eds = (k + 8) * U32 * ds_abs                  # error of the kernel's ds
        within(du, np.einsum('bc,bck->bk', ds, d64),
               np.einsum('bc,bck->bk', eds, np.abs(d64)) + (C + 1) * U32 * np.einsum('bc,bck->bk', np.abs(ds), np.abs(d64)) + 1e-37,
               'du')
        ddr = ds[:, :, None] * u64[:, None, :]
        within(dd, ddr.reshape(B * C, D), ((eds[:, :, None] + U32 * np.abs(ds)[:, :, None]) * np.abs(u64)[:, None, :]).reshape(B * C, D)
               + 1e-37, 'dd')
    return logits, ds


@pytest.mark.parametrize('B,C,D,label,scale,mean', [
    (6, 3, 8, 'none', 1 / 6, False),                  # tiny
    (7, 5, 1, 'onehot', 1.0, False),
    (7, 5, 31, 'two', 0.37, False),
    (7, 5, 32, 'onehot', 1 / 7, False),
    (7, 5, 33, 'none', 1 / 7, True),                   # the k0 loop runs twice, the second time with one live lane
    (9, 1, 33, 'none', 1.0, False),                    # C = 1: p = 1 is saturated, zero gradient
    (9, 32, 33, 'onehot', 1.0, True),                  # every lane owns a candidate
    (9, 32, 70, 'two', -0.5, False),
    (2048, 5, 200, 'none', 1 / 2048, True),            # C3-like batch, loss mean over 2048 rows
    (1024, 5, 400, 'onehot', 1 / 1024, True),
])
def test_score_softmax_ce(lib, B, C, D, label, scale, mean):
    g = rng(B * 1000 + C * 10 + D)
    u = (g.standard_normal((B, D)) / np.sqrt(D)).astype(np.float32)
    d = g.standard_normal((B * C, D)).astype(np.float32)
    y = label_rows(label, B, C, g)
    out = run_softmax_ce(lib, u, d, y, scale, mean=mean)
    check_softmax_ce(u, d, y, scale, out)
    a = run_softmax_ce(lib, u, d, y, scale, mean=mean)
    for x, z in zip(out, a):                           # fixed-order sums: bit-reproducible
        if x is not None:
            assert torch.equal(x.view(torch.int32), z.view(torch.int32))
    # forward only (du = dd = NULL) gives the same forward bits
    f = run_softmax_ce(lib, u, d, y, scale, mean=mean, grads=False)
    for x, z in zip(out[:3], f[:3]):
        assert torch.equal(x.view(torch.int32), z.view(torch.int32))


def test_score_softmax_ce_saturated_rows(lib):
    """logit gaps >= 40: q clips at 1 - 1e-7 (the positive wins) or 1e-7 (the positive loses); the loss is the clipped
    value and the gradient is exactly zero, as Keras' clip has zero gradient outside its range."""
    B, C, D = 4, 5, 40
    g = rng(5)
    u = np.zeros((B, D), np.float32)
    d = g.standard_normal((B * C, D)).astype(np.float32)
    u[:, 0] = 1
    d.reshape(B, C, D)[:, :, 0] = 0
    d.reshape(B, C, D)[0, 0, 0] = 50                    # row 0: positive 50 above the rest
    d.reshape(B, C, D)[1, 3, 0] = 45                    # row 1: a negative 45 above the positive
    d.reshape(B, C, D)[2, 0, 0] = 40
    d.reshape(B, C, D)[3, :, 0] = g.standard_normal(C)  # row 3: an ordinary row next to them
    out = run_softmax_ce(lib, u, d, None, 1.0)
    logits, ds = check_softmax_ce(u, d, None, 1.0, out)
    loss, du, dd = host(out[2]), host(out[4]), host(out[5]).reshape(B, C, D)
    hi, lo = -np.log(F32(1 - 1e-7)), -np.log(F32(1e-7))
    assert abs(loss[0] - hi) <= 4 * U32 * hi and loss[2] == loss[0]
    assert abs(loss[1] - lo) <= 4 * U32 * lo
    for b in range(3):
        assert np.all(du[b] == 0) and np.all(dd[b] == 0), b
    assert np.abs(du[3]).max() > 0


def test_score_softmax_ce_rejects_more_than_32_candidates(lib):
    t = nans(4, 64)
    assert lib.lstur_score_softmax_ce(1, 33, 2, P_(t), 2, P_(t), 2, None, P_(t), P_(t), P_(t), None, None, 2, None, 2,
                                      1.0, st()) == ERR_ARG


def bce_ref(s, y, gain, K, gs, p=None):
    p = 1 / (1 + np.exp(-s)) if p is None else p
    loss = -0.5 * (1 + K) * (y * np.log(p + 1e-8) * gain + (1 - y) * np.log(1 - p + 1e-8) / K)
    dp = -0.5 * (1 + K) * (y * gain / (p + 1e-8) - (1 - y) / (K * (1 - p + 1e-8)))
    return p, loss, gs * dp * p * (1 - p)


def bce_bound(s, y, gain, K, gs, k=8):
    """How far the float32 kernel may be from bce_ref: its p is within k u of sigmoid(s), and 1 - p, p + 1e-8 are
    ill-conditioned near p = 1 and p = 0, so the bound is the spread of the reference over that interval of p, plus
    k u of the magnitude of every output."""
    p, loss, ds = bce_ref(s, y, gain, K, gs)
    lo = bce_ref(s, y, gain, K, gs, p=np.clip(p * (1 - k * U32), 0, 1))
    hi = bce_ref(s, y, gain, K, gs, p=np.clip(p * (1 + k * U32), 0, 1))
    # the float32 sums p + 1e-8 and (1 - p) + 1e-8 carry 2 u of relative rounding (1 - p is exact for p >= 1/2), which
    # enters log() in the loss as an absolute error and the reciprocal in the gradient as a relative one
    r = 2 * U32
    c = 0.5 * (1 + K)
    arg = [np.zeros_like(p), c * (y * gain + (1 - y) / K) * r,
           abs(gs) * c * (y * gain / (p + 1e-8) + (1 - y) / (K * (1 - p + 1e-8))) * r * p * (1 - p) + U32 * np.abs(ds)]
    out = []
    for i, r in enumerate((p, loss, ds)):
        spread = np.maximum(np.abs(lo[i] - r), np.abs(hi[i] - r))
        out.append(spread + arg[i] + k * U32 * np.abs(r) + 1e-37)
    return (p, loss, ds), out


@pytest.mark.parametrize('n,K,gain', [(7, 1, 1.0), (300, 4, 2.5), (10240, 4, 0.3)])
def test_bce_loss(lib, n, K, gain):
    g = rng(n + K)
    s = (g.standard_normal(n) * 6).astype(np.float32)
    s[:4] = [40, -40, 40, -40]
    y = (g.random(n) < 0.3).astype(np.float32)
    y[:4] = [1, 1, 0, 0]
    gs = 1.0 / n
    sd, yd = dev(s), dev(y)
    ref, bound = bce_bound(f32(s), f32(y), F32(gain), float(K), F32(gs))
    first = None
    for mask in itertools.product([0, 1], repeat=4):
        probs, rows, mean, ds = [nans(n) if m else None for m in mask[:2]] + [nans(1) if mask[2] else None] + \
                                [nans(n) if mask[3] else None]
        rc = lib.lstur_bce_loss(n, P_(sd), P_(yd), gain, K, P_(probs), P_(rows), P_(mean), P_(ds), gs, st())
        if mean is not None and rows is None:
            assert rc == ERR_ARG
            continue
        ok(lib, rc)
        if probs is not None:
            within(host(probs), ref[0], bound[0], 'probs')
        if rows is not None:
            within(host(rows), ref[1], bound[1], 'loss_rows')
        if mean is not None:
            r = host(rows)
            within(host(mean)[0], r.mean(), (n + 2) * U32 * np.abs(r).mean(), 'loss_mean')
        if ds is not None:
            within(host(ds), ref[2], bound[2], 'dscores')
            if first is None:
                first = host(ds)
            assert np.array_equal(first, host(ds))    # the same gradient whichever forward outputs are asked for


def softmax_labels_ref(x, lab, scale):
    nc = x.shape[1]
    y = np.where((lab < 0) | (lab >= nc), 0, lab)
    e = np.exp(x - x.max(1, keepdims=True))
    p = e / e.sum(1, keepdims=True)
    q = p[np.arange(len(y)), y] / p.sum(1)
    lo, hi = F32(1e-7), F32(1 - 1e-7)
    loss = -np.log(np.clip(q, lo, hi))
    gq = np.where((q >= lo) & (q <= hi), -1 / q, 0.0)
    py = p[np.arange(len(y)), y]
    onehot = np.zeros_like(p)
    onehot[np.arange(len(y)), y] = 1
    dl = scale * p * (onehot * gq[:, None] - (gq * py)[:, None])
    dl_abs = abs(scale) * p * (onehot * np.abs(gq)[:, None] + np.abs(gq * py)[:, None])
    return p, loss, dl, dl_abs


@pytest.mark.parametrize('nc', [1, 15, 32, 33, 300])
def test_softmax_ce_labels(lib, nc):
    """Logits around +100 and -100 (exp overflows float32 without the max subtraction), labels 0 and nc - 1, and labels
    outside [0, nc), which the kernel reads as class 0."""
    n = 64
    g = rng(nc)
    x = (g.standard_normal((n, nc)) * 3).astype(np.float32)
    x[: n // 2] += 100
    x[n // 2:] -= 100
    lab = g.integers(0, nc, n).astype(np.int32)
    lab[:4] = [0, nc - 1, nc, -1]
    lab[-4:] = [0, nc - 1, nc + 7, -5]
    scale = 1.0 / n
    xd, ld = dev(x), dev(lab, torch.int32)
    probs, rows, mean, dl = nans(n, nc), nans(n), nans(1), nans(n, nc)
    ok(lib, lib.lstur_softmax_ce_labels(n, nc, P_(xd), P_(ld), P_(probs), P_(rows), P_(mean), P_(dl), scale, st()))
    p, loss, dlr, dl_abs = softmax_labels_ref(f32(x), lab, scale)
    k = nc + 8
    within(host(probs), p, k * U32 * p + 1e-37, 'probs')
    within(host(rows), loss, k * U32 * (1 + np.abs(loss)), 'loss_rows')
    r = host(rows)
    within(host(mean)[0], r.mean(), (n + 2) * U32 * np.abs(r).mean(), 'loss_mean')
    within(host(dl), dlr, (k + 8) * U32 * dl_abs + 1e-37, 'dlogits')
    # an out-of-range label is class 0: those rows are bit-identical to the same logits labelled 0
    lab0 = lab.copy()
    lab0[[2, 3, n - 2, n - 1]] = 0
    rows0, dl0 = nans(n), nans(n, nc)
    ok(lib, lib.lstur_softmax_ce_labels(n, nc, P_(xd), P_(dev(lab0, torch.int32)), None, P_(rows0), None, P_(dl0), scale, st()))
    assert torch.equal(rows.view(torch.int32), rows0.view(torch.int32)) and torch.equal(dl.view(torch.int32), dl0.view(torch.int32))
    if nc == 1:      # one class: q = 1 is saturated, the gradient is zero
        assert np.all(host(dl) == 0)
    # optional outputs: each alone gives the same bits
    dl2 = nans(n, nc)
    ok(lib, lib.lstur_softmax_ce_labels(n, nc, P_(xd), P_(ld), None, None, None, P_(dl2), scale, st()))
    assert torch.equal(dl.view(torch.int32), dl2.view(torch.int32))
    assert lib.lstur_softmax_ce_labels(n, nc, P_(xd), P_(ld), None, None, P_(mean), None, scale, st()) == ERR_ARG


# ============================================================================================ 2. scorer pieces
@pytest.mark.parametrize('B,C,D', [(6, 3, 8), (5, 5, 1), (5, 5, 31), (5, 5, 32), (5, 5, 33), (2048, 5, 200), (1024, 5, 400)])
def test_dot_score_bwd(lib, B, C, D):
    g = rng(B + C + D)
    u = g.standard_normal((B, D)).astype(np.float32)
    d = g.standard_normal((B * C, D)).astype(np.float32)
    ds = g.standard_normal((B, C)).astype(np.float32)
    ldu, ldd, lddu, lddd = D + 1, D + 3, D + 2, D + 5
    ud, ddi, dsd = strided(u, ldu), strided(d, ldd), dev(ds)
    du, dd = nans(B, lddu), nans(B * C, lddd)
    ok(lib, lib.lstur_dot_score_bwd(B, C, D, P_(ud), ldu, P_(ddi), ldd, P_(dsd), P_(du), lddu, P_(dd), lddd, st()))
    pad_untouched(du, D, 'du')
    pad_untouched(dd, D, 'dd')
    d3, ds64, u64 = f32(d).reshape(B, C, D), f32(ds), f32(u)
    within(host(du[:, :D]), np.einsum('bc,bck->bk', ds64, d3), C * U32 * np.einsum('bc,bck->bk', np.abs(ds64), np.abs(d3)) + 1e-37, 'du')
    ddr = (ds64[:, :, None] * u64[:, None, :]).reshape(B * C, D)
    within(host(dd[:, :D]), ddr, U32 * np.abs(ddr), 'dd')


@pytest.mark.parametrize('U,D', [(8, 8), (1, 31), (32, 33), (200, 200)])
@pytest.mark.parametrize('ragged', [False, True])
def test_pair_concat(lib, U, D, ragged):
    g = rng(U * D + ragged)
    B, C = 37, 5
    n = B * C
    u = g.standard_normal((B, U)).astype(np.float32)
    d = g.standard_normal((n, D)).astype(np.float32)
    ldu, ldd = U + 3, D + 2
    pr = np.sort(g.integers(0, B, n)).astype(np.int32) if ragged else None
    out = nans(n + 1, U + D)                           # one spare row: nothing past n_pairs is written
    ok(lib, lib.lstur_pair_concat(n, C, U, D, P_(strided(u, ldu)), ldu, P_(strided(d, ldd)), ldd, P_(out),
                                  P_(dev(pr, torch.int32)) if ragged else None, st()))
    rows = pr if ragged else np.arange(n) // C
    want = np.concatenate([u[rows], d], 1)
    assert np.array_equal(host(out[:n]), want.astype(np.float64))
    assert torch.isnan(out[n]).all()


@pytest.mark.parametrize('B,C,U,D', [(6, 3, 8, 8), (5, 1, 1, 33), (5, 5, 31, 32), (2048, 5, 200, 200)])
def test_pair_split(lib, B, C, U, D):
    g = rng(B + U)
    dcat = g.standard_normal((B * C, U + D)).astype(np.float32)
    lddu, lddd = U + 2, D + 3
    outs = []
    for _ in range(2):
        du, dd = nans(B, lddu), nans(B * C, lddd)
        ok(lib, lib.lstur_pair_split(B, C, U, D, P_(dev(dcat)), P_(du), lddu, P_(dd), lddd, st()))
        pad_untouched(du, U, 'du')
        pad_untouched(dd, D, 'dd')
        outs.append((host(du[:, :U]), host(dd[:, :D])))
    x = f32(dcat).reshape(B, C, U + D)
    within(outs[0][0], x[:, :, :U].sum(1), C * U32 * np.abs(x[:, :, :U]).sum(1) + 1e-37, 'du')
    assert np.array_equal(outs[0][1], x[:, :, U:].reshape(B * C, D))
    assert np.array_equal(outs[0][0], outs[1][0]) and np.array_equal(outs[0][1], outs[1][1])


@pytest.mark.parametrize('H', [1, 8, 31, 32, 33, 400])
@pytest.mark.parametrize('bias', [False, True])
def test_rowdot_bias(lib, H, bias):
    g = rng(H)
    n = 1029
    h = g.standard_normal((n, H)).astype(np.float32)
    w = g.standard_normal(H).astype(np.float32)
    b = np.array([0.75], np.float32)
    out = nans(n)
    ok(lib, lib.lstur_rowdot_bias(n, H, P_(dev(h)), P_(dev(w)), P_(dev(b)) if bias else None, P_(out), st()))
    h64, w64 = f32(h), f32(w)
    ref = h64 @ w64 + (0.75 if bias else 0)
    within(host(out), ref, (H + 1) * U32 * (np.abs(h64) @ np.abs(w64) + (0.75 if bias else 0)) + 1e-37, 'rowdot')


@pytest.mark.parametrize('H', [1, 33, 200])
def test_dnn_out_bwd(lib, H):
    g = rng(H)
    n = 517
    hid = np.maximum(g.standard_normal((n, H)), 0).astype(np.float32)   # relu output: about half exactly 0
    hid[0] = 0
    w2 = g.standard_normal(H).astype(np.float32)
    dl = g.standard_normal(n).astype(np.float32)
    dhid, whid = nans(n, H), nans(n, H)
    ok(lib, lib.lstur_dnn_out_bwd(n, H, P_(dev(hid)), P_(dev(w2)), P_(dev(dl)), P_(dhid), P_(whid), st()))
    h64, w64, g64 = f32(hid), f32(w2), f32(dl)
    rd = np.where(h64 > 0, g64[:, None] * w64[None, :], 0.0)
    rw = g64[:, None] * h64
    within(host(dhid), rd, U32 * np.abs(rd), 'dhid')
    within(host(whid), rw, U32 * np.abs(rw), 'whid')
    assert np.all(host(dhid)[hid == 0] == 0) and np.all(host(whid)[hid == 0] == 0)


def test_tanh_relu_fill(lib):
    g = rng(11)
    n = 100003
    x = (g.standard_normal(n) * 3).astype(np.float32)
    x[:6] = [0, -0.0, 20, -20, 1e-30, 9]
    t = dev(x)
    ok(lib, lib.lstur_tanh_fwd(n, P_(t), st()))
    y = host(t)
    within(y, np.tanh(f32(x)), 2 * U32 * np.abs(np.tanh(f32(x))) + 1e-37, 'tanh')
    gr = g.standard_normal(n).astype(np.float32)
    gd = dev(gr)
    ok(lib, lib.lstur_tanh_bwd(n, P_(t), P_(gd), st()))
    within(host(gd), f32(gr) * (1 - y * y), 3 * U32 * np.abs(f32(gr)) * (1 + y * y), 'tanh_bwd')
    yr = g.standard_normal(n).astype(np.float32)
    yr[:4] = [0, -0.0, 1e-38, -1e-38]
    gd = dev(gr)
    ok(lib, lib.lstur_relu_bwd(n, P_(dev(yr)), P_(gd), st()))
    assert np.array_equal(host(gd), np.where(yr > 0, f32(gr), 0.0))
    assert host(gd)[:2].tolist() == [0.0, 0.0]
    buf = nans(n + 1)
    ok(lib, lib.lstur_fill(n, -2.5, P_(buf), st()))
    assert np.all(host(buf[:n]) == -2.5) and torch.isnan(buf[n]).item()


# ============================================================================================ 3. user pooling
@pytest.mark.parametrize('B,W,D', [(6, 5, 8), (5, 3, 1), (5, 7, 31), (5, 7, 33), (1024, 50, 200), (2048, 200, 400)])
def test_masked_mean(lib, B, W, D):
    g = rng(B + W + D)
    m = (g.random((B, W)) < 0.6).astype(np.float32)
    m[0] = 0                                            # all masked: 0, not NaN
    keep = (g.random((B, W)) < 0.5).astype(np.float32)  # keep != mask
    H = (g.standard_normal((B, W, D)) * m[:, :, None]).astype(np.float32)
    ldo = D + 3
    out = nans(B, ldo)
    ok(lib, lib.lstur_masked_mean_fwd(B, W, D, P_(dev(H)), P_(dev(m)), P_(out), ldo, st()))
    pad_untouched(out, D, 'out')
    cnt = f32(m).sum(1)[:, None] + F32(1e-7)
    within(host(out[:, :D]), f32(H).sum(1) / cnt, (W + 2) * U32 * np.abs(f32(H)).sum(1) / cnt, 'fwd')
    assert np.all(host(out[0, :D]) == 0)
    dout = g.standard_normal((B, D)).astype(np.float32)
    dH = nans(B, W, D)
    ok(lib, lib.lstur_masked_mean_bwd(B, W, D, P_(strided(dout, ldo)), ldo, P_(dev(m)), P_(dev(keep)), P_(dH), st()))
    ref = f32(keep)[:, :, None] * (f32(dout) / cnt)[:, None, :]
    within(host(dH), ref, (W + 3) * U32 * np.abs(ref), 'bwd')


def seq_attn_ref(H, m, kw, kb, dout, keep):
    """float64 autograd of the layer the kernels implement: x = H * keep (the mask multiplied in before the layer),
    a = tanh(x.k + b), e = exp(a) mask, w = e / (sum e + 1e-7), out = sum_t w_t x_t."""
    X = torch.tensor(f32(H), requires_grad=True)
    k = torch.tensor(f32(kw), requires_grad=True)
    b = torch.tensor(f32(kb), requires_grad=True)
    mt = torch.tensor(f32(m))
    x = X * torch.tensor(f32(keep))[:, :, None]
    a = torch.tanh(x @ k + b[0])
    e = torch.exp(a) * mt
    w = e / (e.sum(-1, keepdim=True) + ot.EPS)
    out = (x * w[:, :, None]).sum(1)
    (out * torch.tensor(f32(dout))).sum().backward()
    return out.detach().numpy(), a.detach().numpy(), w.detach().numpy(), X.grad.numpy(), k.grad.numpy(), b.grad.numpy()


@pytest.mark.parametrize('B,W,D', [(6, 5, 8), (9, 1, 33), (9, 2, 1), (7, 5, 400), (64, 200, 33), (64, 200, 400),
                                   (3, 4096, 1), (3, 4096, 33)])
@pytest.mark.parametrize('with_keep', [False, True])
def test_seq_attn(lib, B, W, D, with_keep):
    """SimpleAttentionMaskSupport over W steps: forward, backward and the colsum-folded parameter gradients vs float64
    autograd; row 0 has every step masked with non-zero inputs (sum e = 0: the 1e-7 keeps it finite)."""
    g = rng(B * W + D + with_keep)
    H = g.standard_normal((B, W, D)).astype(np.float32)
    m = (g.random((B, W)) < 0.7).astype(np.float32)
    m[0] = 0
    m[1] = 1
    keep = (g.random((B, W)) < 0.8).astype(np.float32) if with_keep else np.ones((B, W), np.float32)
    Hin = H * keep[:, :, None]                          # exact in float32 (keep is 0 / 1)
    kw = (g.standard_normal(D) / np.sqrt(D)).astype(np.float32)
    kb = np.array([0.1], np.float32)
    dout = g.standard_normal((B, D)).astype(np.float32)
    ldo = D + 2
    Hd, md, kwd, kbd = dev(Hin), dev(m), dev(kw), dev(kb)
    out, a, w = nans(B, ldo), nans(B, W), nans(B, W)
    ok(lib, lib.lstur_seq_attn_fwd(B, W, D, P_(Hd), P_(md), P_(kwd), P_(kbd), P_(out), ldo, P_(a), P_(w), st()))
    pad_untouched(out, D, 'out')
    out2 = nans(B, ldo)
    ok(lib, lib.lstur_seq_attn_fwd(B, W, D, P_(Hd), P_(md), P_(kwd), P_(kbd), P_(out2), ldo, None, None, st()))
    assert torch.equal(out[:, :D].view(torch.int32), out2[:, :D].view(torch.int32))
    ro, ra, rw, rdH, rdk, rdb = seq_attn_ref(H, m, kw, kb, dout, keep)
    # running error bound: the score of step t carries (D + 4) u sum_k |x k| of error, which moves w_t relatively by
    # as much (through exp and the normalisation, twice); every later sum adds its own n u sum|terms|.
    x64 = f32(Hin)
    da = (D + 4) * U32 * (np.abs(x64) @ np.abs(f32(kw)) + 0.1) + 4 * U32
    rel_w = 2 * da.max(1, keepdims=True) + (W + 4) * U32
    within(host(a), ra, da, 'a')
    within(host(w), rw, rel_w * rw + 1e-37, 'w')
    within(host(out[:, :D]), ro, np.einsum('bt,btk->bk', rel_w * rw + (W + 2) * U32 * rw, np.abs(x64)) + 1e-37, 'out')
    assert np.all(host(out[0, :D]) == 0) and np.all(host(w)[0] == 0)
    dH, part = nans(B, W, D), nans(B, D + 1)
    kp = dev(keep) if with_keep else None
    ok(lib, lib.lstur_seq_attn_bwd(B, W, D, P_(Hd), P_(kwd), P_(a), P_(w), P_(strided(dout, ldo)), ldo, P_(kp), P_(dH),
                                   P_(part), st()))
    # magnitude of the backward's terms: |d w_t| <= sum_k |x dout|, |c| <= sum_t w |d w|, |d pre| <= (|d w| + |c|) w
    dw_abs = np.einsum('btk,bk->bt', np.abs(x64), np.abs(f32(dout)))
    c_abs = (rw * dw_abs).sum(1, keepdims=True)
    dpre_abs = (dw_abs + c_abs) * rw
    kk = (W + D + 16) * U32 + 4 * rel_w[:, :, None]
    dH_abs = f32(keep)[:, :, None] * (rw[:, :, None] * np.abs(f32(dout))[:, None, :] + dpre_abs[:, :, None] * np.abs(f32(kw)))
    within(host(dH), rdH, kk * dH_abs + 1e-37, 'dH')
    assert np.all(host(dH)[0] == 0)
    ws_rows = 1024
    ws = nans(ws_rows * (D + 1))
    dk, db = nans(D), nans(1)
    ok(lib, lib.lstur_colsum(B, D, P_(part), D + 1, P_(dk), 0, P_(ws), ws.numel() * 4, st()))
    ok(lib, lib.lstur_colsum(B, 1, P_(part[:, D:]), D + 1, P_(db), 0, P_(ws), ws.numel() * 4, st()))
    kb_ = (W + D + B + 16) * U32 + 4 * rel_w.max()
    within(host(dk), rdk, kb_ * np.einsum('bt,btk->k', dpre_abs, np.abs(x64)) + 1e-37, 'd att_w')
    within(host(db), rdb, kb_ * dpre_abs.sum() + 1e-37, 'd att_b')


def test_seq_attn_rejects_long_sequences(lib):
    t = nans(8)
    assert lib.lstur_seq_attn_fwd(1, 4097, 1, P_(t), P_(t), P_(t), P_(t), P_(t), 1, None, None, st()) == ERR_ARG


@pytest.mark.parametrize('D', [1, 33, 200])
def test_alpha_add(lib, D):
    g = rng(D)
    R = 301
    a = g.standard_normal((R, D)).astype(np.float32)
    b = g.standard_normal((R, D)).astype(np.float32)
    dout = g.standard_normal((R, D)).astype(np.float32)
    al = np.array([0.3], np.float32)
    lda, ldb, ldo = D + 1, D + 2, D + 3
    ad, bd, ald = strided(a, lda), strided(b, ldb), dev(al)
    out = nans(R, ldo)
    ok(lib, lib.lstur_alpha_add_fwd(R, D, P_(ald), P_(ad), lda, P_(bd), ldb, P_(out), ldo, st()))
    pad_untouched(out, D, 'out')
    A, Bv, al64, g64 = f32(a), f32(b), F32(0.3), f32(dout)
    within(host(out[:, :D]), al64 * A + (1 - al64) * Bv, 3 * U32 * (np.abs(al64 * A) + np.abs((1 - al64) * Bv)), 'fwd')
    da, db, rp = nans(R, ldo), nans(R, ldo), nans(R)
    ok(lib, lib.lstur_alpha_add_bwd(R, D, P_(ald), P_(ad), lda, P_(bd), ldb, P_(strided(dout, ldo)), ldo, P_(da), ldo,
                                    P_(db), ldo, P_(rp), st()))
    pad_untouched(da, D, 'da')
    pad_untouched(db, D, 'db')
    within(host(da[:, :D]), al64 * g64, U32 * np.abs(al64 * g64), 'da')
    within(host(db[:, :D]), (1 - al64) * g64, 2 * U32 * np.abs((1 - al64) * g64), 'db')
    within(host(rp), (g64 * (A - Bv)).sum(1), (D + 2) * U32 * (np.abs(g64) * (np.abs(A) + np.abs(Bv))).sum(1) + 1e-37, 'partial')


@pytest.mark.parametrize('lo,hi', [(0.0, 1.0), (0.5, 1.0), (0.2, 0.3)])
def test_minmaxnorm(lib, lo, hi):
    w = np.array([0, -0.0, 0.05, -0.05, 0.25, -0.25, 0.7, -0.7, 3, -3, 1e-9, lo, hi], np.float32)
    t = dev(w)
    ok(lib, lib.lstur_minmaxnorm(len(w), lo, hi, P_(t), st()))
    x = f32(w)
    ref = x * (np.clip(np.abs(x), F32(lo), F32(hi)) / (F32(1e-7) + np.abs(x)))
    within(host(t), ref, 4 * U32 * np.abs(ref), 'minmaxnorm')


def test_add_rows(lib):
    g = rng(3)
    R, D = 77, 33
    ldx, ldy = D + 4, D + 7
    x = g.standard_normal((R, D)).astype(np.float32)
    y = g.standard_normal((R, D)).astype(np.float32)
    y[5] = np.nan
    yd = strided(y, ldy)
    ok(lib, lib.lstur_add_rows(R, D, 1.5, P_(strided(x, ldx)), ldx, 0.0, P_(yd), ldy, st()))
    pad_untouched(yd, D, 'y')
    within(host(yd[:, :D]), 1.5 * f32(x), U32 * np.abs(1.5 * f32(x)), 'ay = 0')     # NaN in y does not propagate
    y[5] = 0
    yd = strided(y, ldy)
    ok(lib, lib.lstur_add_rows(R, D, -0.5, P_(strided(x, ldx)), ldx, 2.0, P_(yd), ldy, st()))
    ref = -0.5 * f32(x) + 2.0 * f32(y)
    within(host(yd[:, :D]), ref, 2 * U32 * (np.abs(0.5 * f32(x)) + np.abs(2 * f32(y))), 'add')


@pytest.mark.parametrize('D', [1, 31, 32, 33, 401])
def test_rows_nonzero(lib, D):
    g = rng(D)
    R, ld = 41, D + 3
    x = np.zeros((R, D), np.float32)
    x[1] = -0.0                                         # -0.0 counts as zero
    x[2, D - 1] = 1e-30                                 # one non-zero in the last column
    x[3, 0] = -2
    x[4:20] = g.standard_normal((16, D))
    xd = strided(x, ld)                                 # NaN pad: a read past D would count as non-zero
    mask = nans(R)
    ok(lib, lib.lstur_rows_nonzero(R, D, P_(xd), ld, P_(mask), st()))
    assert np.array_equal(host(mask), (x != 0).any(1).astype(np.float64))


@pytest.mark.parametrize('W', [1, 31, 32, 33, 200])
def test_first_live_step(lib, W):
    g = rng(W)
    B = 37
    m = (g.random((B, W)) < 0.1).astype(np.float32)
    m[0] = 0                                            # none live -> W
    for b, t in enumerate([31, 32, 199, 0, W - 1], start=1):
        m[b] = 0
        m[b, min(t, W - 1):] = 1
    key = torch.full((B,), -7, dtype=torch.int32, device='cuda')
    ok(lib, lib.lstur_first_live_step(B, W, P_(dev(m)), P_(key), st()))
    ref = np.where(m.any(1), np.argmax(m != 0, 1), W)
    assert np.array_equal(key.cpu().numpy(), ref)


@pytest.mark.parametrize('cols', [1, 33, 200])
@pytest.mark.parametrize('bias', [False, True])
def test_fill_rows_where(lib, cols, bias):
    g = rng(cols)
    R, ld = 53, cols + 2
    flags = g.integers(0, 3, R).astype(np.int32)
    bv = g.standard_normal(cols).astype(np.float32)
    out = nans(R, ld)
    ok(lib, lib.lstur_fill_rows_where(R, cols, P_(dev(flags, torch.int32)), 1, P_(dev(bv)) if bias else None, P_(out), ld, st()))
    o = host(out)
    sel = flags == 1
    assert np.array_equal(o[sel, :cols], np.broadcast_to(f32(bv) if bias else 0.0, (int(sel.sum()), cols)))
    assert np.isnan(o[~sel]).all() and np.isnan(o[:, cols:]).all()


# ============================================================================================ 4. reductions, small tables
def colsum_ws_bytes(rows, cols):
    return min(max((rows + 255) // 256, 1), 1024) * cols * 4


@pytest.mark.parametrize('rows', [0, 1, 3, 255, 256, 257, 409_600, 1024 * 256 + 1])
@pytest.mark.parametrize('cols', [1, 33, 1200])
def test_colsum(lib, rows, cols):
    """out[c] (+)= sum_r in[r, c] in two fixed-order stages; 409 600 = C5's B W, 1024 * 256 + 1 is the first row count
    at which the 1024-chunk cap makes the chunks longer than 256 rows."""
    torch.manual_seed(rows + cols)
    ld = cols + 3
    x = torch.randn(max(rows, 1), ld, device='cuda')
    x[:, cols:] = NAN
    wsb = colsum_ws_bytes(rows, cols)
    ws = nans(wsb // 4)
    ref = x[:rows, :cols].double().sum(0)
    bound = max(rows, 1) * U32 * x[:rows, :cols].double().abs().sum(0) + 1e-37
    outs = []
    for _ in range(2):
        out = nans(cols)
        ok(lib, lib.lstur_colsum(rows, cols, P_(x), ld, P_(out), 0, P_(ws), wsb, st()))
        outs.append(out)
    assert torch.equal(outs[0].view(torch.int32), outs[1].view(torch.int32))
    within(host(outs[0]), ref.cpu().numpy(), bound.cpu().numpy(), 'colsum')
    acc = torch.linspace(-3, 3, cols, device='cuda')
    out = acc.clone()
    ok(lib, lib.lstur_colsum(rows, cols, P_(x), ld, P_(out), 1, P_(ws), wsb, st()))
    within(host(out), (ref + acc.double()).cpu().numpy(), (bound + 2 * U32 * (acc.double().abs() + ref.abs())).cpu().numpy(),
           'accumulate')
    assert lib.lstur_colsum(rows, cols, P_(x), ld, P_(out), 0, P_(ws), wsb - 4, st()) == ERR_ARG


@pytest.mark.parametrize('n,col0,n_vert,pile', [(37, 0, 1, False), (1000, 8, 300, False), (419_840, 400, 16, False),
                                                (419_840, 400, 300, True)])
def test_vert_concat_and_small_table_grad(lib, n, col0, n_vert, pile):
    """Cook.get_doc_encoder's [title | Vemb[vert] | Semb[subvert]] and the Embedding backward of the small tables, at up
    to C5's 2048 (200 + 5) titles; ids out of range read (and credit) row 0 in the forward."""
    g = rng(n + n_vert)
    dv, ds = 15, 35
    D = col0 + dv + ds + 3
    n_docs = 5000
    n_sub = 307
    doc_vert = g.integers(0, n_vert, n_docs).astype(np.int32)
    doc_vert[:3] = [-1, n_vert, n_vert + 5]
    if pile:
        doc_vert[3:] = 3 % n_vert
    doc_sub = g.integers(0, n_sub, n_docs).astype(np.int32)
    doc_ids = g.integers(0, n_docs, n).astype(np.int32)
    doc_ids[:3] = [0, 1, 2]
    ve = g.standard_normal((n_vert, dv)).astype(np.float32)
    se = g.standard_normal((n_sub, ds)).astype(np.float32)
    docv = nans(n, D)
    tv = torch.full((n,), -9, dtype=torch.int32, device='cuda')
    ts = torch.full((n,), -9, dtype=torch.int32, device='cuda')
    ok(lib, lib.lstur_vert_concat(n, D, col0, dv, ds, n_docs, n_vert, n_sub, P_(dev(doc_ids, torch.int32)),
                                  P_(dev(doc_vert, torch.int32)), P_(dev(doc_sub, torch.int32)), P_(dev(ve)), P_(dev(se)),
                                  P_(docv), P_(tv), P_(ts), st()))
    v = doc_vert[doc_ids]
    v = np.where((v < 0) | (v >= n_vert), 0, v)
    s = doc_sub[doc_ids]
    assert np.array_equal(tv.cpu().numpy(), v) and np.array_equal(ts.cpu().numpy(), s)
    o = host(docv)
    assert np.array_equal(o[:, col0:col0 + dv], f32(ve)[v]) and np.array_equal(o[:, col0 + dv:col0 + dv + ds], f32(se)[s])
    assert np.isnan(o[:, :col0]).all() and np.isnan(o[:, col0 + dv + ds:]).all()
    dd = torch.randn(n, D, device='cuda')
    for ids, c0, dim, nr in ((tv, col0, dv, n_vert), (ts, col0 + dv, ds, n_sub)):
        wsb = lib.lstur_small_table_grad_workspace_bytes(nr, dim)
        ws = nans(wsb // 4)
        outs = []
        for _ in range(2):
            out = nans(nr, dim)
            ok(lib, lib.lstur_small_table_grad(n, D, c0, dim, nr, P_(ids), P_(dd), P_(out), P_(ws), wsb, st()))
            outs.append(out)
        assert torch.equal(outs[0].view(torch.int32), outs[1].view(torch.int32))
        cols = dd[:, c0:c0 + dim].double()
        ref = torch.zeros(nr, dim, dtype=torch.float64, device='cuda').index_add_(0, ids.long(), cols)
        absr = torch.zeros(nr, dim, dtype=torch.float64, device='cuda').index_add_(0, ids.long(), cols.abs())
        cnt = torch.bincount(ids.long(), minlength=nr).double()[:, None]
        within(host(outs[0]), ref.cpu().numpy(), (cnt * U32 * absr + 1e-37).cpu().numpy(), 'd table')
        assert lib.lstur_small_table_grad(n, D, c0, dim, nr, P_(ids), P_(dd), P_(outs[0]), P_(ws), wsb - 4, st()) == ERR_ARG


def test_scale_rows(lib):
    g = rng(4)
    B, D = 2049, 200
    ld = D + 5
    x = g.standard_normal((B, D)).astype(np.float32)
    sc = g.standard_normal(B).astype(np.float32)
    sc[:2] = [0, 1 / 0.7]
    xd = strided(x, ld)
    ok(lib, lib.lstur_scale_rows(B, D, P_(dev(sc)), P_(xd), ld, st()))
    pad_untouched(xd, D, 'x')
    ref = f32(x) * f32(sc)[:, None]
    within(host(xd[:, :D]), ref, U32 * np.abs(ref), 'scale_rows')


@pytest.mark.parametrize('D', [1, 33, 200])
def test_rows_add(lib, D):
    g = rng(D)
    n_tab, max_rows, n_live = 500, 64, 41
    table = g.standard_normal((n_tab, D)).astype(np.float32)
    rows = g.permutation(n_tab)[:max_rows].astype(np.int32)        # unique, unsorted
    gr = g.standard_normal((max_rows, D)).astype(np.float32)
    td = dev(table)
    ok(lib, lib.lstur_rows_add(max_rows, P_(dev(np.array([n_live], np.int32), torch.int32)), D,
                               P_(dev(rows, torch.int32)), P_(dev(gr)), P_(td), st()))
    t = host(td)
    want = f32(table)
    want[rows[:n_live]] += f32(gr[:n_live])
    hit = np.zeros(n_tab, bool)
    hit[rows[:n_live]] = True
    assert np.array_equal(t[~hit], f32(table)[~hit])                 # rows beyond *n_rows and unlisted rows: bit-identical
    within(t[hit], want[hit], U32 * np.abs(want[hit]), 'rows_add')


# ============================================================================================ 5. optimizer
B1, B2, EPS = F32(0.9), F32(0.999), F32(1e-7)
C3_DENSE = 681_604     # the dense arena of the C3 'igru' plan: conv 3x300x400 + 400 + 400 + 1, dense 400x200 + 200, GRU
                       # 200x600 + 200x600 + 600, each tensor starting on a multiple of 4 floats


def adam_check(p0, g, m0, v0, t, lr, gs, p, m, v):
    lr32 = F32(lr)
    rp, rm, rv = adam_step(f32(p0), f32(g) * F32(gs), f32(m0), f32(v0), t, lr32, b1=B1, b2=B2, eps=EPS)
    lr_t = lr32 * np.sqrt(1 - B2 ** t) / (1 - B1 ** t)
    gi = f32(g) * F32(gs)
    m_abs = np.abs(B1 * f32(m0)) + np.abs((1 - B1) * gi)
    within(m, rm, 4 * U32 * m_abs + 1e-37, 'm')
    within(v, rv, 5 * U32 * rv + 1e-37, 'v')
    den = np.sqrt(rv) + EPS
    within(p, rp, 2 * U32 * np.abs(rp) + 12 * U32 * lr_t * m_abs / den + 1e-37, 'p')


@pytest.mark.parametrize('n', [5, 606_207, 606_208, 606_209, C3_DENSE])
@pytest.mark.parametrize('t,gs', [(1, 1.0), (2, 1 / 1024), (10_000, 3.0)])
def test_adam_dense(lib, n, t, gs):
    """Keras-2.2 Adam against oracle.lstur_numpy.adam_step; 148 * 16 * 256 = 606 208 is the grid-stride cap, beyond
    which the loop wraps."""
    g = rng(n + t)
    p0 = g.standard_normal(n).astype(np.float32)
    gr = g.standard_normal(n).astype(np.float32)
    m0 = (g.standard_normal(n) * 0.1).astype(np.float32) if t > 1 else np.zeros(n, np.float32)
    v0 = (g.random(n) * 0.01).astype(np.float32) if t > 1 else np.zeros(n, np.float32)
    p, m, v = dev(p0), dev(m0), dev(v0)
    ok(lib, lib.lstur_adam_dense(n, P_(p), P_(dev(gr)), P_(m), P_(v), 1e-3, t, B1, B2, EPS, gs, st()))
    adam_check(p0, gr, m0, v0, t, 1e-3, gs, host(p), host(m), host(v))


@pytest.mark.parametrize('D', [1, 33, 200])
def test_adam_rows(lib, D):
    g = rng(D)
    n_tab, max_rows, n_live, t = 300, 50, 37, 3
    p0 = g.standard_normal((n_tab, D)).astype(np.float32)
    m0 = (g.standard_normal((n_tab, D)) * 0.1).astype(np.float32)
    v0 = (g.random((n_tab, D)) * 0.01).astype(np.float32)
    rows = g.permutation(n_tab)[:max_rows].astype(np.int32)
    gr = g.standard_normal((max_rows, D)).astype(np.float32)
    p, m, v = dev(p0), dev(m0), dev(v0)
    ok(lib, lib.lstur_adam_rows(max_rows, P_(dev(np.array([n_live], np.int32), torch.int32)), D, P_(dev(rows, torch.int32)),
                                P_(dev(gr)), P_(p), P_(m), P_(v), 1e-3, t, B1, B2, EPS, 0.5, st()))
    P, M, V = host(p), host(m), host(v)
    hit = np.zeros(n_tab, bool)
    hit[rows[:n_live]] = True
    for got, x0 in ((P, p0), (M, m0), (V, v0)):
        assert np.array_equal(got[~hit], f32(x0)[~hit])
    r = rows[:n_live]
    adam_check(p0[r], gr[:n_live], m0[r], v0[r], t, 1e-3, 0.5, P[r], M[r], V[r])


@pytest.mark.parametrize('n', [7, 606_209])
def test_axpby(lib, n):
    g = rng(n)
    x = g.standard_normal(n).astype(np.float32)
    y = g.standard_normal(n).astype(np.float32)
    y[::97] = np.nan
    yd = dev(y)
    ok(lib, lib.lstur_axpby(n, 0.25, P_(dev(x)), 0.0, P_(yd), st()))     # b = 0: y is not read
    within(host(yd), 0.25 * f32(x), U32 * np.abs(0.25 * f32(x)), 'b = 0')
    y[::97] = 1
    yd = dev(y)
    ok(lib, lib.lstur_axpby(n, -1.5, P_(dev(x)), 0.75, P_(yd), st()))
    ref = -1.5 * f32(x) + 0.75 * f32(y)
    within(host(yd), ref, 2 * U32 * (np.abs(1.5 * f32(x)) + np.abs(0.75 * f32(y))), 'axpby')


# ============================================================================================ 6. streaming recurrences
WIDTHS = [200, 215, 448, 449, 544, 545, 672, 673, 736, 737, 1000, 1024]
TOL = 2e-5


@pytest.mark.parametrize('G', WIDTHS)
@pytest.mark.parametrize('act', ['hard_sigmoid', 'sigmoid'])
@pytest.mark.parametrize('entry', ['streaming', 'dispatch'])
def test_gru_every_accepted_width(lib, G, act, entry):
    """lstur_gru_{fwd,bwd}_streaming and the lstur_gru_fwd/bwd dispatchers run every G <= 1024 (one thread per unit:
    the widths past what the 8-row instance's registers allow take the 4-row instance) and match the float64 oracle."""
    B, W = 13, 6
    XW, gm, Wh, h0, dhT = gru_make(B, W, G, seed=G + 7, ini=True, pad='holes')
    hT_ref, dA_ref, dh0_ref = gru_oracle(XW, Wh, h0, dhT, act)
    f = lambda a: dev(a)
    XWd, gmd, Whd, dhTd, h0d = f(XW), f(gm), f(Wh), f(dhT), f(h0)
    WhT = Whd.t().contiguous()
    a = 0 if act == 'hard_sigmoid' else 1
    ldh = G + 3
    hT, dh0 = nans(B, ldh), nans(B, ldh)
    sv = [nans(B, W, G) for _ in range(5)]
    dA = nans(B, W, 3 * G)
    if entry == 'streaming':
        ok(lib, lib.lstur_gru_fwd_streaming(B, W, G, P_(XWd), P_(gmd), P_(h0d), G, P_(Whd), a, P_(hT), ldh,
                                            *[P_(s) for s in sv], st()))
        ok(lib, lib.lstur_gru_bwd_streaming(B, W, G, P_(gmd), *[P_(s) for s in sv[:4]], P_(WhT), a, P_(dhTd), G, P_(dA),
                                            P_(dh0), ldh, st()))
    else:
        ok(lib, lib.lstur_gru_fwd(B, W, G, P_(XWd), P_(gmd), P_(h0d), G, P_(Whd), a, P_(hT), ldh, *[P_(s) for s in sv],
                                  None, st()))
        ok(lib, lib.lstur_gru_bwd(B, W, G, P_(gmd), *[P_(s) for s in sv[:4]], P_(WhT), a, P_(dhTd), G, P_(dA), P_(dh0),
                                  ldh, None, st()))
    pad_untouched(hT, G, 'hT')
    pad_untouched(dh0, G, 'dh0')
    assert rel(host(hT[:, :G]), hT_ref) < TOL
    assert rel(host(dA), dA_ref) < 5 * TOL
    assert rel(host(dh0[:, :G]), dh0_ref) < 5 * TOL
    assert all(np.isfinite(host(s)).all() for s in sv)
    assert np.all(host(dA)[gm == 0] == 0)


def lstm_oracle(XW, Wh, gm, dh, act):
    """keras LSTM recurrence (gate order i, f, c, o; masked steps carry h and c) in float64 autograd."""
    B, W, G4 = XW.shape
    G = G4 // 4
    sig = ot.hard_sigmoid if act == 'hard_sigmoid' else torch.sigmoid
    x = torch.tensor(f32(XW), requires_grad=True)
    w = torch.tensor(f32(Wh))
    m = torch.tensor(gm) != 0
    h, c = torch.zeros(B, G, dtype=torch.float64), torch.zeros(B, G, dtype=torch.float64)
    for s in range(W):
        a = x[:, s] + h @ w
        i, f, gg, o = sig(a[:, :G]), sig(a[:, G:2 * G]), torch.tanh(a[:, 2 * G:3 * G]), sig(a[:, 3 * G:])
        cn = f * c + i * gg
        hn = o * torch.tanh(cn)
        c = torch.where(m[:, s:s + 1], cn, c)
        h = torch.where(m[:, s:s + 1], hn, h)
    (h * torch.tensor(f32(dh))).sum().backward()
    return h.detach().numpy(), x.grad.numpy()


@pytest.mark.parametrize('G', WIDTHS)
@pytest.mark.parametrize('act', ['hard_sigmoid', 'sigmoid'])
def test_lstm_every_accepted_width(lib, G, act):
    B, W = 13, 6
    g = rng(G)
    XW = g.standard_normal((B, W, 4 * G)).astype(np.float32)
    Wh = (g.standard_normal((G, 4 * G)) / np.sqrt(G)).astype(np.float32)
    gm = (g.random((B, W)) < 0.7).astype(np.float32)
    gm[1] = 0
    gm[0] = 1
    dh = g.standard_normal((B, G)).astype(np.float32)
    a = 0 if act == 'hard_sigmoid' else 1
    XWd, gmd, Whd, dhd = dev(XW), dev(gm), dev(Wh), dev(dh)
    ldo = G + 5
    hT = nans(B, ldo)
    S = [nans(B, W, G) for _ in range(7)]
    ok(lib, lib.lstur_lstm_fwd(B, W, G, P_(XWd), P_(gmd), P_(Whd), a, P_(hT), ldo, *[P_(s) for s in S], st()))
    pad_untouched(hT, G, 'hT')
    SI, SF, SG, SO, SCP, SHP, STC = S
    dA = nans(B, W, 4 * G)
    ok(lib, lib.lstur_lstm_bwd(B, W, G, P_(gmd), P_(SI), P_(SF), P_(SG), P_(SO), P_(SCP), P_(STC), P_(Whd.t().contiguous()), a,
                               P_(dhd), G, P_(dA), st()))
    h_ref, dA_ref = lstm_oracle(XW, Wh, gm, dh, act)
    assert rel(host(hT[:, :G]), h_ref) < TOL
    assert rel(host(dA), dA_ref) < 5 * TOL
    assert all(np.isfinite(host(s)).all() for s in S)
    assert np.all(host(dA)[gm == 0] == 0)


def test_igru_engine_at_a_width_off_the_cluster_geometry(lib):
    """An fp32 'igru' model with user_embedding_dim = 502 (no multiple of 4, so the recurrence runs on the streaming
    kernels, on the wide instance) trains: gradients within the fp32 bounds of test_gpu_cook_archs.py, and the step's
    loss equals the oracle's."""
    from mnexp_b200 import synth
    from mnexp_b200.engine import LsturEngine
    sh = dataclasses.replace(synth.SHAPES['tiny'], U=502)
    tok, _, _ = synth.make_docs(sh.n_news, sh.L, sh.vocab)
    P = synth.make_weights(sh, arch='igru', bias_noise=0.05, seed=77)
    (b,), _ = synth.make_batches(sh, 1, seed=78)
    assert lib.lstur_gru_cluster_supported(sh.B, sh.W, 502) == 0
    eng = LsturEngine(P, sh.B, sh.W, 1 + sh.K, sh.L, arch='igru', doc_tokens=tok, lr=1e-3)
    db = eng.to_device_batch(b)
    eng.forward(db, training=True, seed=1)
    eng.backward(db)
    torch.cuda.synchronize()
    got = eng.get_grads_dict()
    ora = ot.LsturOracle(P, arch='igru', lr=1e-3)
    u, c, d = ora._ints(b['user'], tok[b['hist_doc']], tok[b['cand_doc']])
    loss = ot.loss_fn(ora.P, u, c, d, arch='igru')
    ref = dict(zip(ora.trainable, torch.autograd.grad(loss, [ora.P[k] for k in ora.trainable], allow_unused=True)))
    for k in ('gru_wh', 'gru_wx', 'gru_b', 'dense_w', 'conv_w', 'user_emb'):
        assert rel(got[k], ref[k].numpy()) < 5e-5, k
    l_eng = float(eng.train_step(db)[0])
    torch.cuda.synchronize()
    l_ora = ora.train_step(b['user'], tok[b['hist_doc']], tok[b['cand_doc']], training=False)
    assert abs(l_eng - l_ora) <= 5e-5 * max(1.0, abs(l_ora))
