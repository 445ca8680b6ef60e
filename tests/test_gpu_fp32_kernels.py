"""Kernel-level tests of the fp32 (verification-mode) news encoder's gather, attention-pooling and word-table gradient
kernels (gather.cu, attn.cu, wordgrad.cu), of the small row kernels of the user side (gather.cu lstur_hist_mask_apply /
lstur_row_gather, gru.cu lstur_transpose) and of the evaluation heads (score.cu), each against a float64 reference of
the same operation.

The conventions of test_gpu_step_kernels.py hold: every output is NaN before the call, strided arguments have NaN pad
columns, sums of n terms are bounded by n u sum|terms| (u = 2^-23) and fixed-order sums are run twice and compared byte
for byte.  Dropout masks are replayed from the rng_u32 stream (mnexp_b200.rng).  Where a kernel consumes another kernel's
output, its reference starts from the device output of that stage, so no ReLU, mask or dropout decision can differ
between kernel and reference."""
import ctypes
import functools

import numpy as np
import pytest
import torch

from mnexp_b200 import _lib, rng as drng
from test_gpu_step_kernels import (ERR_ARG, U32, P_, _release_in_flight, dev, f32, host, nans, ok, pad_untouched, rng,  # noqa: F401
                                   st, strided, sync, within)

pytestmark = pytest.mark.gpu

NAN = float('nan')


@functools.lru_cache(maxsize=8)
def keep_mult(seed, n, p):
    """float32-valued inverted-dropout multipliers (1/(1-p) or 0) of the rng_u32 stream, flat indices 0..n-1"""
    return drng.dropout_multiplier(seed, n, p, dtype=np.float32)


def bits_equal(a, b):
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def within_t(got, ref, bound, what=''):
    """within() on device tensors (float64): the large cases would be slow on the host"""
    got, ref = got.double(), ref.double()
    assert torch.isfinite(got).all().item(), '%s: %d non-finite elements' % (what, int((~torch.isfinite(got)).sum()))
    err = (got - ref).abs()
    bound = torch.broadcast_to(torch.as_tensor(bound, dtype=torch.float64, device=got.device), err.shape)
    bad = err > bound
    if bad.any().item():
        i = int(torch.argmax((err - bound).reshape(-1)))
        raise AssertionError('%s: %d elements out of bound; worst at flat %d: got %r ref %r bound %r'
                             % (what, int(bad.sum()), i, got.reshape(-1)[i].item(), ref.reshape(-1)[i].item(),
                                bound.reshape(-1)[i].item()))


def titles(g, N, L, V, pad_frac=0.3):
    """(N, L) int32 tokens: right-padded titles of random length (some all-pad, some full), ids in [1, V) with a few
    out-of-range ids (-1, V, V + 7) among the real tokens"""
    tok = g.integers(1, V, (N, L)).astype(np.int32)
    length = g.integers(0, L + 1, N)
    length[g.random(N) < pad_frac] = 0
    tok[np.arange(L)[None, :] >= length[:, None]] = 0
    odd = (g.random((N, L)) < 0.03) & (tok != 0)
    tok[odd] = g.choice(np.array([-1, V, V + 7], np.int32), int(odd.sum()))
    return tok


# ============================================================================================ a. lstur_embed_gather_pad
@pytest.mark.parametrize('KS', [1, 2, 3, 4, 5])
@pytest.mark.parametrize('E', [4, 12, 300, 1, 7, 33])
@pytest.mark.parametrize('p', [0.0, 0.2])
def test_embed_gather_pad(lib, KS, E, p):
    """Embedding + Dropout into the zero-haloed title buffer: bit-exact, halo rows exactly 0, ids -1 and >= V read
    row 0, the X-dropout mask replayed from its stream"""
    g = rng(KS * 100 + E + int(p * 10))
    N, L, V, seed = 9, 11, 50, 7
    tok = titles(g, N, L, V)
    tok[0, :4] = [-1, V, V + 3, 0]
    emb = g.standard_normal((V, E)).astype(np.float32)
    pl, Lp = (KS - 1) // 2, L + KS - 1
    Xp = nans(N, Lp, E)
    ok(lib, lib.lstur_embed_gather_pad(N, L, E, V, KS, P_(dev(emb)), P_(dev(tok, torch.int32)), P_(Xp), p, seed, st()))
    got = Xp.cpu().numpy()
    ids = np.where((tok < 0) | (tok >= V), 0, tok)
    mult = keep_mult(seed, N * L * E, p).reshape(N, L, E)
    want = np.where(mult != 0, emb[ids] * mult, np.float32(0)).astype(np.float32) if p > 0 else emb[ids]
    assert np.array_equal(got[:, pl:pl + L], want)
    assert np.all(got[:, :pl] == 0) and np.all(got[:, pl + L:] == 0)       # the halo: exactly 0, no NaN left


# ============================================================================================ b. lstur_attn_pool_fwd
def attn_inputs(g, N, L, F, extra_rows=2):
    """conv+bias+relu output C in a buffer of title stride (L + extra_rows) F (rows beyond L NaN), tokens with the
    special titles: 0 all-pad, 1 one real token at position 0, 2 one real token at L-1, 3 a real token whose conv row is
    all zero"""
    C = np.maximum(g.standard_normal((N, L, F)) + 0.2, 0).astype(np.float32)
    tok = titles(g, N, L, 40, pad_frac=0.1)
    if N > 1:
        tok[0] = 0
        C[0] = np.abs(C[0]) + 1                       # all-pad title with non-zero conv output: masked away
    if N > 3:
        tok[1] = 0
        tok[1, 0] = 5
        tok[2] = 0
        tok[2, L - 1] = 6
        tok[3, 0] = 7
        C[3, 0] = 0
    if N == 1:
        tok[0] = 0
        tok[0, 0] = 3
        C[0] = np.abs(C[0]) + 0.5
    Cbuf = np.full((N, L + extra_rows, F), np.nan, np.float32)
    Cbuf[:, :L] = C
    return Cbuf, tok


def attn_fwd(lib, Cbuf, tok, kw, kb, p, seed, ldp, with_aw=True):
    N, Lr, F = Cbuf.shape
    L = tok.shape[1]
    Cd = dev(Cbuf)
    pooled = nans(N, ldp)
    a, w = (nans(N, L), nans(N, L)) if with_aw else (None, None)
    ok(lib, lib.lstur_attn_pool_fwd(N, L, F, P_(Cd), Lr * F, P_(dev(tok, torch.int32)), P_(dev(kw)), P_(dev(kb)), P_(pooled),
                                    ldp, P_(a), P_(w), p, seed, st()))
    sync()
    return Cd, pooled, a, w


def attn_fwd_ref(Cw, tok, kw, kb, m):
    """a, w, pooled and their bounds in float64 from the written-back C (device), on the device"""
    kw64, C64 = torch.as_tensor(kw, dtype=torch.float64, device='cuda'), Cw.double()
    F, L = C64.shape[2], C64.shape[1]
    z = C64 @ kw64 + float(kb[0])
    a = torch.tanh(z)
    e = torch.exp(a) * m
    w = e / (e.sum(1, keepdim=True) + float(np.float32(1e-7)))
    pooled = (w[:, :, None] * C64).sum(1)
    # the score of step t carries (F + 4) u sum_f |C k| of error, which moves w_t relatively by as much (through exp and
    # the normalisation, twice); every later sum adds its own n u sum|terms|
    da = (F + 4) * U32 * (C64.abs() @ kw64.abs() + abs(float(kb[0]))) + 4 * U32
    rel_w = 2 * da.max(1, keepdim=True).values + (L + 4) * U32
    return a, w, pooled, da, rel_w


@pytest.mark.parametrize('N,L,F', [(1, 1, 1), (37, 30, 400), (5, 256, 33), (700, 7, 16)])
@pytest.mark.parametrize('p', [0.0, 0.2])
def test_attn_pool_fwd(lib, N, L, F, p):
    """pad mask + Masking + Dropout + attention pooling: the written-back C bit-exact, masked rows w == 0 exactly, a / w /
    pooled within bounds propagated through tanh and exp; the same C and pooled without a_out / w_out"""
    g = rng(N + L + F + int(p * 10))
    seed, ldp = 11, F + 3
    Cbuf, tok = attn_inputs(g, N, L, F)
    kw = (g.standard_normal(F) / np.sqrt(F)).astype(np.float32)
    kb = np.array([0.1], np.float32)
    Cd, pooled, a, w = attn_fwd(lib, Cbuf, tok, kw, kb, p, seed, ldp)
    Cd2, pooled2, _, _ = attn_fwd(lib, Cbuf, tok, kw, kb, p, seed, ldp, with_aw=False)
    assert bits_equal(Cd, Cd2)
    assert bits_equal(pooled[:, :F], pooled2[:, :F])
    pad_untouched(pooled, F, 'pooled')
    assert torch.isnan(Cd[:, L:]).all().item(), 'wrote C rows beyond L'
    # the written-back C: pad mask, then the dropout multiply (bit-exact)
    C = Cbuf[:, :L] * (tok != 0)[:, :, None].astype(np.float32)
    m = (C != 0).any(-1)
    if p > 0:
        mult = keep_mult(seed, N * L * F, p).reshape(N, L, F)
        C = np.where(mult != 0, C * mult, np.float32(0)).astype(np.float32)
    Cw = Cd[:, :L]
    assert np.array_equal(Cw.cpu().numpy(), C)
    mt = torch.as_tensor(m, dtype=torch.float64, device='cuda')
    ra, rw, rp, da, rel_w = attn_fwd_ref(Cw, tok, kw, kb, mt)
    within_t(a, ra, da, 'a')
    assert torch.all(w[~torch.as_tensor(m, device='cuda')] == 0).item(), 'masked rows must have w == 0 exactly'
    within_t(w, rw, rel_w * rw + 1e-37, 'w')
    pb = ((rel_w * rw + (L + 2) * U32 * rw)[:, :, None] * Cw.double().abs()).sum(1) + 1e-37
    within_t(pooled[:, :F], rp, pb, 'pooled')
    if N > 1:
        assert torch.all(pooled[0, :F] == 0).item() and torch.all(w[0] == 0).item()


# ============================================================================================ c. lstur_attn_pool_bwd
def attn_bwd(lib, N, L, Lrows, F, Cd, title_stride, a, w, dp, lddp, kw, p, dpre, dpre_stride, outs, accumulate,
             partial_bytes=None):
    grid = lib.lstur_attn_bwd_grid(N)
    part = nans(grid * (2 * F + 1))
    nb = part.numel() * 4 if partial_bytes is None else partial_bytes
    dw, dcb, dab = outs
    return lib.lstur_attn_pool_bwd(N, L, Lrows, F, P_(Cd), title_stride, P_(a), P_(w), P_(dp), lddp, P_(kw), P_(dpre),
                                   dpre_stride, p, P_(dw), P_(dcb), P_(dab), accumulate, P_(part), nb, st())


@pytest.mark.parametrize('N,L,F', [(1, 1, 1), (592, 256, 1), (593, 30, 128), (2000, 7, 129), (37, 256, 256),
                                   (1, 30, 257), (593, 1, 512), (5, 256, 513), (2000, 30, 1024)])
@pytest.mark.parametrize('p', [0.0, 0.2])
def test_attn_pool_bwd(lib, N, L, F, p):
    """attention / ReLU / mask / dropout backward from the forward's written-back C, a and w: dPre vs float64 (rows
    L..Lrows-1 exactly 0, rows beyond Lrows untouched), d att_w / d conv_b / d att_b vs float64 with accumulate 0 and 1,
    a second run byte-identical.  Covers every FPT instantiation and the grid-strided title loop (N > 592)."""
    g = rng(N * 7 + L + F + int(p * 10))
    seed, Lrows = 5, L + 2
    title_stride = (Lrows + 1) * F            # the conv output buffer: Lp rows per title, rows beyond L unread
    Cbuf, tok = attn_inputs(g, N, L, F, extra_rows=Lrows + 1 - L)
    kw = (g.standard_normal(F) / np.sqrt(F)).astype(np.float32)
    kb = np.array([-0.05], np.float32)
    Cd, _, a, w = attn_fwd(lib, Cbuf, tok, kw, kb, p, seed, F + 1)
    lddp = F + 3
    dpo = g.standard_normal((N, F)).astype(np.float32)
    dp, kwd = strided(dpo, lddp), dev(kw)
    dpre_stride = (Lrows + 1) * F + 3
    runs = []
    for accumulate in (0, 1):
        dpre = nans(N * dpre_stride).reshape(N, dpre_stride)
        if accumulate:
            base = [torch.full((F,), 0.25, device='cuda'), torch.full((F,), -0.5, device='cuda'),
                    torch.full((1,), 2.0, device='cuda')]
        else:
            base = [nans(F), nans(F), nans(1)]
        outs = [b.clone() for b in base]
        ok(lib, attn_bwd(lib, N, L, Lrows, F, Cd, title_stride, a, w, dp, lddp, kwd, p, dpre, dpre_stride, outs, accumulate))
        sync()
        runs.append((dpre, base, outs))
    (dpre, _, outs), (dpre1, base1, outs1) = runs
    assert bits_equal(dpre[:, :Lrows * F], dpre1[:, :Lrows * F])            # byte-identical run to run
    for b, o0, o1 in zip(base1, outs, outs1):                                 # accumulate = 1 adds the same sums
        assert np.array_equal(o1.cpu().numpy(), (b.cpu().numpy() + o0.cpu().numpy()).astype(np.float32))
    assert torch.isnan(dpre[:, Lrows * F:]).all().item(), 'wrote dPre beyond Lrows rows'
    assert torch.all(dpre[:, L * F:Lrows * F] == 0).item(), 'rows L..Lrows-1 of dPre must be 0'
    # float64 reference from the device C, a, w
    C64 = Cd.reshape(N, -1)[:, :L * F].reshape(N, L, F).double()
    a64, w64 = a.double(), w.double()
    dp64, kw64 = torch.as_tensor(dpo, dtype=torch.float64, device='cuda'), kwd.double()
    inv = float(np.float32(1) / (np.float32(1) - np.float32(p)))
    dwt = torch.einsum('ntf,nf->nt', C64, dp64)
    q = (dwt * w64).sum(1, keepdim=True)
    one_a2 = 1 - a64 * a64
    dz = (dwt - q) * w64 * one_a2
    gg = w64[:, :, None] * dp64[:, None, :] + dz[:, :, None] * kw64
    ref = torch.where(C64 > 0, gg * inv, torch.zeros_like(gg))
    # magnitudes: |d w_t| <= sum_f |C dp|, |q| <= sum_t w |d w|, |dz| <= (|d w| + |q|) w
    dw_abs = torch.einsum('ntf,nf->nt', C64.abs(), dp64.abs())
    q_abs = (dw_abs * w64).sum(1, keepdim=True)
    dz_abs = (dw_abs + q_abs) * w64
    dz_err = (F + L + 16) * U32 * dz_abs
    g_abs = w64[:, :, None] * dp64.abs()[:, None, :] + dz_abs[:, :, None] * kw64.abs()
    gate = (C64 > 0).double()
    dpre_err = gate * inv * (dz_err[:, :, None] * kw64.abs() + 4 * U32 * g_abs)
    within_t(dpre[:, :L * F].reshape(N, L, F), ref, dpre_err + 1e-37, 'dPre')
    grid = lib.lstur_attn_bwd_grid(N)
    n_add = -(-N // grid) * L + -(-grid // 8) + 10                          # longest fixed-order chain of one sum
    d_kw = torch.einsum('nt,ntf->f', dz, C64)
    d_kw_err = torch.einsum('nt,ntf->f', dz_err + n_add * U32 * dz_abs, C64.abs())
    within_t(outs[0], d_kw, d_kw_err + 1e-37, 'd att_w')
    within_t(outs[1], ref.sum((0, 1)), (dpre_err + n_add * U32 * gate * inv * g_abs).sum((0, 1)) + 1e-37, 'd conv_b')
    within_t(outs[2], dz.sum().reshape(1), (dz_err + n_add * U32 * dz_abs).sum().reshape(1) + 1e-37, 'd att_b')


def test_attn_pool_bwd_empty_and_refused(lib):
    """N = 0 zeroes the parameter gradients (accumulate 0) or leaves them alone (1); a partials buffer one float short
    and F = 1025 are refused before any launch"""
    F = 33
    t = nans(64)
    for accumulate in (0, 1):
        outs = [torch.full((F,), 3.0, device='cuda'), torch.full((F,), 4.0, device='cuda'), torch.full((1,), 5.0, device='cuda')]
        ok(lib, attn_bwd(lib, 0, 4, 4, F, t, 4 * F, t, t, t, F, t, 0.0, t, 4 * F, outs, accumulate))
        sync()
        for o, v in zip(outs, (3.0, 4.0, 5.0)):
            assert torch.all(o == (v if accumulate else 0.0)).item()
    N, L = 3, 4
    need = lib.lstur_attn_bwd_grid(N) * (2 * F + 1) * 4
    outs = [nans(F), nans(F), nans(1)]
    assert attn_bwd(lib, N, L, L, F, t, L * F, t, t, t, F, t, 0.0, t, L * F, outs, 0, partial_bytes=need - 4) == ERR_ARG
    big = nans(N * L * 1025)
    outs = [nans(1025), nans(1025), nans(1)]
    assert attn_bwd(lib, N, L, L, 1025, big, L * 1025, t, t, big, 1025, big, 0.0, big, L * 1025, outs, 0) == ERR_ARG


# ============================================================================================ d. lstur_word_grad_scatter_f32
def zipf_titles(g, N, L, V):
    """right-padded titles of Zipf-drawn tokens: token 1 owns ~25 % of the real positions; ids -1 and >= V among them"""
    tok = np.minimum(g.zipf(1.3, (N, L)), V - 1).astype(np.int32)
    length = g.integers(0, L + 1, N)
    length[g.random(N) < 0.1] = 0
    length[g.random(N) < 0.1] = L
    tok[np.arange(L)[None, :] >= length[:, None]] = 0
    hole = (g.random((N, L)) < 0.05)
    tok[hole] = 0                                                       # pad tokens inside a title
    odd = (g.random((N, L)) < 0.02) & (tok != 0)
    tok[odd] = g.choice(np.array([-1, -5, V, V + 7], np.int32), int(odd.sum()))
    return tok


@pytest.mark.parametrize('KS', [1, 2, 3, 4, 5, 7])
@pytest.mark.parametrize('N,L,E,V,p', [
    (1, 1, 4, 511, 0.0),               # one position; one 9-bit radix pass
    (8, 8, 12, 512, 0.2),              # 64 positions: one level-1 chunk; two passes
    (5, 13, 132, 513, 0.0),            # 65: two chunks; two pieces per lane, the second partial
    (64, 32, 300, 300000, 0.2),        # 2048: one level-2 chunk; three passes
    (683, 3, 128, 512, 0.0),           # 2049: three levels
    (2200, 30, 512, 300000, 0.2),      # 66000 > 65536: four levels, four pieces per lane
])
def test_word_grad_scatter_f32(lib, KS, N, L, E, V, p):
    """d word_emb = sum over positions of dXp * keep * scale / (1-p) grouped by (clamped) token, from the dXp that the
    conv input gradient produces: pad positions that a conv output over a real token reads are included at every filter
    width (the conv window reaches KS-1-pl positions back and pl forward).  Absent tokens' rows exactly 0, byte-identical
    run to run."""
    g = rng(KS * 1000 + N + E)
    seed, scale = 3, 0.37
    tok = zipf_titles(g, N, L, V)
    pl, Lp = (KS - 1) // 2, L + KS - 1
    # dPre projected to the input width: one row per conv output, zero at pad outputs; dXp = its KS-tap sum
    tok_d = torch.as_tensor(tok, device='cuda')
    D = torch.as_tensor(g.standard_normal((N, L, E)), device='cuda') * (tok_d != 0)[:, :, None]
    taps = g.standard_normal(KS)
    X = torch.zeros((N, Lp, E), dtype=torch.float64, device='cuda')
    for j in range(KS):
        X[:, j:j + L] += float(taps[j]) * D
    X = X.float()
    X[:, :pl] = NAN                                                     # the halo rows: never read
    X[:, pl + L:] = NAN
    nb = lib.lstur_word_grad_workspace_bytes(N * L, V, E)
    ws = torch.empty(nb, dtype=torch.uint8, device='cuda')
    tokd = dev(tok, torch.int32)
    outs = []
    for _ in range(2):
        out = nans(V, E)
        ok(lib, lib.lstur_word_grad_scatter_f32(N, L, KS, E, V, P_(tokd), P_(X), p, seed, scale, P_(out), P_(ws), nb, st()))
        sync()
        outs.append(out)
    assert bits_equal(outs[0], outs[1])
    got = outs[0]
    # reference: every position, grouped by clamped token, in float64
    ids = torch.where((tok_d < 0) | (tok_d >= V), 0, tok_d).reshape(-1).long()
    rows = X[:, pl:pl + L].double().reshape(N * L, E)
    if p > 0:
        rows = rows * torch.as_tensor(keep_mult(seed, N * L * E, p) != 0, device='cuda').reshape(N * L, E)
    fac = float(np.float32(scale) / (np.float32(1) - np.float32(p)))       # the kernel's scale / (1 - p), in float32
    ref = torch.zeros((V, E), dtype=torch.float64, device='cuda').index_add_(0, ids, rows) * fac
    mag = torch.zeros((V, E), dtype=torch.float64, device='cuda').index_add_(0, ids, rows.abs()) * fac
    cnt = torch.zeros(V, dtype=torch.float64, device='cuda').index_add_(0, ids, torch.ones_like(ids, dtype=torch.float64))
    within_t(got, ref, (cnt[:, None] + 8) * U32 * mag + 1e-37, 'd word_emb')
    absent = cnt == 0
    assert torch.all(got[absent] == 0).item(), 'rows of absent tokens must be exactly 0'


def test_word_grad_scatter_f32_refused(lib):
    """a workspace one byte short and E % 4 != 0 are refused before any launch"""
    N, L, E, V = 4, 5, 12, 100
    tok = dev(np.ones((N, L), np.int32), torch.int32)
    X, out = nans(N, L + 2, E), nans(V, E)
    nb = lib.lstur_word_grad_workspace_bytes(N * L, V, E)
    ws = torch.empty(nb, dtype=torch.uint8, device='cuda')
    assert lib.lstur_word_grad_scatter_f32(N, L, 3, E, V, P_(tok), P_(X), 0.0, 1, 1.0, P_(out), P_(ws), nb - 1, st()) == ERR_ARG
    nb6 = lib.lstur_word_grad_workspace_bytes(N * L, V, 6)
    ws6 = torch.empty(nb6, dtype=torch.uint8, device='cuda')
    assert lib.lstur_word_grad_scatter_f32(N, L, 3, 6, V, P_(tok), P_(X), 0.0, 1, 1.0, P_(out), P_(ws6), nb6, st()) == ERR_ARG
    sync()
    assert torch.isnan(out).all().item()                                  # refused: nothing written


# ============================================================================================ e. user-side row kernels
@pytest.mark.parametrize('D', [1, 33, 400])
@pytest.mark.parametrize('with_tokens', [True, False])
@pytest.mark.parametrize('with_hm', [True, False])
def test_hist_mask_apply(lib, D, with_tokens, with_hm):
    """ComputeMasking(0) + multiply + Masking(): bit-exact; an all-pad title with non-zero H is zeroed (hm = gm = 0),
    real tokens with H all zero give hm = 1, gm = 0; without tokens hm = gm = any(H != 0); the pad of H stays NaN"""
    g = rng(D * 4 + with_tokens * 2 + with_hm)
    rows, L, ldh = 50, 40, D + 5
    tok = titles(g, rows, L, 30, pad_frac=0.3)
    H = g.standard_normal((rows, D)).astype(np.float32)
    tok[0] = 0                                                          # all-pad, non-zero H
    tok[1] = 0
    tok[1, L - 1] = 4                                                   # the only real token beyond lane 31
    H[2] = 0
    tok[2, 0] = 9                                                       # real tokens, H all zero
    H[3] = 0
    tok[3] = 0                                                          # all-pad, H all zero
    if D > 1:
        H[4, :D - 1] = 0                                                # only the last column non-zero
    Hd = strided(H, ldh)
    hm, gm = (nans(rows) if with_hm else None), nans(rows)
    tk = dev(tok, torch.int32) if with_tokens else None
    ok(lib, lib.lstur_hist_mask_apply(rows, L, D, P_(tk), P_(Hd), ldh, P_(hm), P_(gm), st()))
    sync()
    pad_untouched(Hd, D, 'H')
    live = (tok != 0).any(1) if with_tokens else np.ones(rows, bool)
    Hw = np.where(live[:, None], H, np.float32(0))
    assert np.array_equal(Hd[:, :D].cpu().numpy(), Hw)
    anyh = (Hw != 0).any(1)
    assert np.array_equal(gm.cpu().numpy(), anyh.astype(np.float32))
    if with_hm:
        assert np.array_equal(hm.cpu().numpy(), (live if with_tokens else anyh).astype(np.float32))
    if with_tokens:
        assert gm[0].item() == 0 and (not with_hm or hm[0].item() == 0)
        assert gm[2].item() == 0 and (not with_hm or hm[2].item() == 1)


@pytest.mark.parametrize('D', [1, 33, 400])
@pytest.mark.parametrize('with_scale', [False, True])
def test_row_gather(lib, D, with_scale):
    """user-ID lookup: bit-exact, ids -1 and n_rows read row 0, optional per-row scale, the pad of out untouched"""
    g = rng(D + with_scale)
    B, n_rows, ldo = 70, 40, D + 3
    table = g.standard_normal((n_rows, D)).astype(np.float32)
    ids = g.integers(0, n_rows, B).astype(np.int32)
    ids[:3] = [-1, n_rows, n_rows + 100]
    sc = g.random(B).astype(np.float32) if with_scale else None
    out = nans(B, ldo)
    ok(lib, lib.lstur_row_gather(B, D, n_rows, P_(dev(table)), P_(dev(ids, torch.int32)), P_(dev(sc) if with_scale else None),
                                 P_(out), ldo, st()))
    sync()
    pad_untouched(out, D, 'out')
    want = table[np.where((ids < 0) | (ids >= n_rows), 0, ids)]
    if with_scale:
        want = (want * sc[:, None]).astype(np.float32)
    assert np.array_equal(out[:, :D].cpu().numpy(), want)


@pytest.mark.parametrize('rows,cols', [(1, 1), (33, 99), (400, 1200)])
def test_transpose(lib, rows, cols):
    x = rng(rows + cols).standard_normal((rows, cols)).astype(np.float32)
    out = nans(cols, rows)
    ok(lib, lib.lstur_transpose(rows, cols, P_(dev(x)), P_(out), st()))
    sync()
    assert np.array_equal(out.cpu().numpy(), x.T)


# ============================================================================================ f. evaluation heads
def sigmoid_inputs(g, B, C, D):
    u = g.standard_normal((B, D)).astype(np.float32)
    d = g.standard_normal((B * C, D)).astype(np.float32)
    u[:2] = 0
    u[:2, 0] = 10
    d[:C] = 0
    d[:C, 0] = 10                                                       # row 0: logits +100
    d[C:2 * C] = 0
    d[C:2 * C, 0] = -10                                                 # row 1: logits -100
    return u, d


def check_sigmoid(got, u64, d64, rows, docs, apply_sigmoid, what):
    s = np.einsum('jk,jk->j', u64[rows], d64[docs])
    s_err = u64.shape[1] * U32 * np.einsum('jk,jk->j', np.abs(u64[rows]), np.abs(d64[docs])) + 1e-37
    if not apply_sigmoid:
        within(got, s, s_err, what)
        return
    with np.errstate(over='ignore'):
        sg = 1 / (1 + np.exp(-s))
    # below float32's normal range the kernel's exp overflows to a sigmoid of exactly 0
    within(got, sg, sg * (1 - sg) * s_err * 1.001 + 4 * U32 * sg + np.finfo(np.float32).tiny, what)


@pytest.mark.parametrize('C', [1, 5])
@pytest.mark.parametrize('D', [1, 31, 33, 400])
@pytest.mark.parametrize('apply_sigmoid', [0, 1])
def test_score_sigmoid(lib, C, D, apply_sigmoid):
    """test head: u[i / C] . d[i] (and its sigmoid) within D u sum|u d|; logits of +-100 give exactly 1 / 0"""
    g = rng(C * 10 + D + apply_sigmoid)
    B = 9
    u, d = sigmoid_inputs(g, B, C, D)
    ldu, ldd = D + 2, D + 5
    out = nans(B * C)
    ok(lib, lib.lstur_score_sigmoid(B * C, C, D, P_(strided(u, ldu)), ldu, P_(strided(d, ldd)), ldd, P_(out), apply_sigmoid, st()))
    got = host(out)
    check_sigmoid(got, f32(u), f32(d), np.arange(B * C) // C, np.arange(B * C), apply_sigmoid, 'out')
    if apply_sigmoid:
        assert np.all(got[:C] == 1) and np.all(got[C:2 * C] == 0)
    else:
        assert np.all(got[:C] == 100) and np.all(got[C:2 * C] == -100)


@pytest.mark.parametrize('D', [1, 33, 400])
@pytest.mark.parametrize('with_doc', [False, True])
def test_score_sigmoid_ragged(lib, D, with_doc):
    """ragged test head: unsorted, repeated pair_row and repeated pair_doc within bounds; with pair_row = j / C and no
    pair_doc it is lstur_score_sigmoid bit for bit"""
    g = rng(D + with_doc)
    B, C, n = 9, 5, 200
    u, d = sigmoid_inputs(g, B, C, D)
    ldu, ldd = D + 2, D + 5
    ud, dd = strided(u, ldu), strided(d, ldd)
    row = g.integers(0, B, n).astype(np.int32)
    doc = g.integers(0, B * C, n).astype(np.int32) if with_doc else None
    if not with_doc:
        n = B * C
        row = g.permutation(np.arange(n) // C).astype(np.int32)         # unsorted, every row C times
    out = nans(n)
    ok(lib, lib.lstur_score_sigmoid_ragged(n, D, P_(dev(row, torch.int32)), P_(ud), ldu,
                                           P_(dev(doc, torch.int32) if with_doc else None), P_(dd), ldd, P_(out), st()))
    check_sigmoid(host(out), f32(u), f32(d), row, doc if with_doc else np.arange(n), 1, 'out')
    # the promise of its comment: the same lane order as lstur_score_sigmoid
    a, b = nans(B * C), nans(B * C)
    ok(lib, lib.lstur_score_sigmoid_ragged(B * C, D, P_(dev(np.arange(B * C) // C, torch.int32)), P_(ud), ldu, None, P_(dd), ldd,
                                           P_(a), st()))
    ok(lib, lib.lstur_score_sigmoid(B * C, C, D, P_(ud), ldu, P_(dd), ldd, P_(b), 1, st()))
    sync()
    assert bits_equal(a, b)


def test_csr_rows(lib):
    """CSR offsets from a non-zero base, empty rows and rows of 1 .. 1000 pairs -> the row of every pair; entries past
    the last pair untouched; n_rows = 0 touches nothing"""
    counts = np.array([0, 1, 31, 32, 0, 33, 1000, 0, 5, 64])
    base = 17
    off = (base + np.concatenate([[0], np.cumsum(counts)])).astype(np.int32)
    total = int(counts.sum())
    row_of = torch.full((total + 40,), -7, dtype=torch.int32, device='cuda')
    offd = dev(off, torch.int32)
    ok(lib, lib.lstur_csr_rows(len(counts), P_(offd), P_(row_of), st()))
    sync()
    got = row_of.cpu().numpy()
    assert np.array_equal(got[:total], np.repeat(np.arange(len(counts)), counts))
    assert np.all(got[total:] == -7)
    row_of.fill_(-7)
    ok(lib, lib.lstur_csr_rows(0, P_(offd), P_(row_of), st()))
    sync()
    assert torch.all(row_of == -7).item()


def ranking_ref(s, y):
    """the host formulas of test_gpu_ranking_metrics_match_host (utils.py:106-124, sklearn roc_auc_score); NaN where they
    divide by zero or the AUC is undefined (one class only)"""
    from sklearn.metrics import roc_auc_score
    s64, y64 = s.astype(np.float64), y.astype(np.float64)
    n = len(s)
    order = np.lexsort((-np.arange(n), -s64))                           # descending score, ties by descending index
    yo = y64[order]
    disc = np.log2(np.arange(n) + 2)
    ideal = np.sort(y64)[::-1]
    with np.errstate(invalid='ignore', divide='ignore'):
        ndcg = lambda k: np.sum((2 ** yo[:k] - 1) / disc[:k]) / np.sum((2 ** ideal[:k] - 1) / disc[:k])
        mrr = np.sum(yo / (np.arange(n) + 1)) / np.sum(yo)
        auc = roc_auc_score(y, s) if 0 < (y > 0).sum() < n else np.nan
        return np.array([auc, ndcg(10), ndcg(5), mrr])


def test_ranking_metrics_edges(lib):
    """AUC / nDCG@10 / nDCG@5 / MRR at the edges: C = 1 (AUC NaN, nDCG 1, MRR 1), no positive (all NaN), no negative
    (AUC NaN, the rest finite), C = 0 (all NaN), all scores tied, C = 1000 (several passes of the 128-thread loop), and
    offsets starting at a non-zero base with NaN before it"""
    g = rng(41)
    imps = []
    imps.append((np.array([0.3], np.float32), np.array([1], np.float32)))                    # C = 1
    imps.append((g.random(7).astype(np.float32), np.zeros(7, np.float32)))                   # no positive
    imps.append((g.random(6).astype(np.float32), np.ones(6, np.float32)))                    # no negative
    imps.append((np.zeros(0, np.float32), np.zeros(0, np.float32)))                          # C = 0
    y = np.zeros(12, np.float32)
    y[[2, 5, 11]] = 1
    imps.append((np.full(12, 0.5, np.float32), y))                                           # all tied
    y = (g.random(1000) < 0.1).astype(np.float32)
    y[0], y[1] = 1, 0
    imps.append((g.random(1000).astype(np.float32), y))                                      # C = 1000
    s = np.round(g.random(300), 1).astype(np.float32)
    y = (g.random(300) < 0.2).astype(np.float32)
    y[0], y[1] = 1, 0
    imps.append((s, y))                                                                      # many ties, C = 300
    base = 13
    counts = [len(s) for s, _ in imps]
    off = (base + np.concatenate([[0], np.cumsum(counts)])).astype(np.int32)
    sc = np.concatenate([np.full(base, np.nan, np.float32)] + [s for s, _ in imps])
    lb = np.concatenate([np.full(base, np.nan, np.float32)] + [y for _, y in imps])
    out = nans(len(imps), 4)
    ok(lib, lib.lstur_ranking_metrics(len(imps), P_(dev(off, torch.int32)), P_(dev(sc)), P_(dev(lb)), P_(out), st()))
    got = host(out)
    for i, (s, y) in enumerate(imps):
        want = ranking_ref(s, y)
        assert np.array_equal(np.isnan(got[i]), np.isnan(want)), (i, got[i], want)
        fin = ~np.isnan(want)
        assert np.abs(got[i][fin] - want[fin]).max(initial=0) < 2e-6, (i, got[i], want)
    assert np.isnan(got[0, 0]) and got[0, 1] == 1 and got[0, 2] == 1 and got[0, 3] == 1
    assert np.all(np.isnan(got[1])) and np.all(np.isnan(got[3]))
    assert np.isnan(got[2, 0]) and np.all(np.isfinite(got[2, 1:]))


# ============================================================================================ g. plan refusal
def test_plan_refuses_fp32_training_beyond_attention_backward_width(lib):
    """an fp32 training plan with F = 1025 would fail at its first backward (the attention backward takes F <= 1024):
    lstur_plan_create refuses it; F = 1024, and F = 1025 for inference, are accepted"""
    def create(F, bw):
        cfg = dict(B=8, W=5, C=3, L=7, E=12, F=F, KS=3, use_dense=1, Dd=16, dv=0, ds=0, G=16, Ue=16, U=16, arch=0,
                   score_model=0, rec_act=0, precision=0, V=120, n_users=50, n_docs=81, dropout=0.0, save_for_backward=bw,
                   n_vert=0, n_subvert=0, Hs=0, loss_model=0, bce_neg=0, gain=0.0, trainable_word_emb=0, aux_nv=0,
                   aux_hidden=0, aux_gain=0.0, cls_nv=0)
        c = _lib.lstur_config(**cfg)
        plan = ctypes.c_void_p()
        rc = lib.lstur_plan_create(ctypes.byref(c), ctypes.byref(plan))
        if rc == 0:
            lib.lstur_plan_destroy(plan)
        return rc
    assert create(1025, 1) == ERR_ARG
    assert b'1024' in lib.lstur_last_error()
    assert create(1024, 1) == 0
    assert create(1025, 0) == 0
