"""Tensor-core news-encoder backward, kernel by kernel, against float64 references.

The engine's tensor-core backward (csrc/engine.cu, encoder_backward) is a chain over the compacted list of live titles
(device-side count n_live, original indices live_idx):
  lstur_attn_pool_bwd_img      attention / ReLU / mask / dropout backward -> dPre as a swizzled 16-bit image, x img_scale
  lstur_conv_wgrad_tc_m        conv weight gradient from that image (forward keep bits or hash replay, dpre_scale)
  lstur_conv_dgrad_tc          conv input gradient from that image (trainable word table)
  lstur_word_grad_scatter_16   scatter of the input gradient into the word table
Every check here is stage-isolated: a kernel's reference is built in float64 from the DEVICE output of the stage before
it (the forward's saved C16, a, w; the decoded dPre image; dx16), never from an oracle forward of its own.  No ReLU gate
can flip between kernel and reference, so the bounds are set by the 16-bit rounding of the outputs and by fp32
accumulation.  The references run in torch float64 on the device (the C3-sized weight gradient is ~1e12 FLOP).
"""
import ctypes
import types

import numpy as np
import pytest
import torch

from mnexp_b200 import rng
from test_gpu_tc import P_, dpre_image, keep_bytes, make_enc_case, round16, stream
from tolerances import rel

pytestmark = pytest.mark.gpu
F64 = torch.float64
DEV = 'cuda'
CHUNK = 4096                     # titles per slice of the float64 references (bounds their device memory)


# ---------------------------------------------------------------- the dPre image layout (csrc/attn.cu, attn_bwd_img_kernel)
def _slot(L):
    return 32 if L <= 31 else 64


def image_words(img, N, L, F):
    """Raw 16-bit words of the first N title blocks of a dPre image, un-swizzled: (N, slot, 2, ngh * 64) int16, indexed
    [title][row t][half h][column within the half].  A title block is [half][64-column group][slot rows][128 B] and the
    16-byte piece p of row t is stored at piece p ^ (t & 7).  img: numpy array or torch tensor of any 1- or 2-byte dtype."""
    slot, ngh = _slot(L), (F // 2 + 63) // 64
    u = torch.from_numpy(np.ascontiguousarray(img).view(np.int16)) if isinstance(img, np.ndarray) else img.view(torch.int16)
    u = u.reshape(-1)[:N * 2 * ngh * slot * 64].reshape(N, 2, ngh, slot, 8, 8)
    t = torch.arange(slot, device=u.device)
    phys = torch.arange(8, device=u.device)[None, :] ^ (t[:, None] & 7)
    u = u[:, :, :, t[:, None], phys, :]
    return u.permute(0, 3, 1, 2, 4, 5).reshape(N, slot, 2, ngh * 64)


def words_to_f64(u, fp16):
    return u.view(torch.float16 if fp16 else torch.bfloat16).to(F64)


def decode_dpre_image(img, N, L, F, fp16):
    """Inverse of the image layout: (N, L, F) float64 values (numpy in, numpy out; a torch tensor stays on its device)."""
    v = words_to_f64(image_words(img, N, L, F), fp16)
    Fh = F // 2
    out = torch.cat([v[:, :L, 0, :Fh], v[:, :L, 1, :Fh]], -1)
    return out.numpy() if isinstance(img, np.ndarray) else out


# ---------------------------------------------------------------- helpers
def ok(lib, rc):
    assert rc == 0, lib.lstur_last_error()


def PN(t):
    return P_(t) if t is not None else None


def inv_keep(p):
    """1 / (1 - p) as the kernels compute it (fp32)"""
    return float(np.float32(1) / (np.float32(1) - np.float32(p)))


def i32(shape, fill=0):
    return torch.full((int(shape),) if np.ndim(shape) == 0 else tuple(shape), fill, dtype=torch.int32, device=DEV)


def unpack_keep(xm, rows, Ep):
    """forward keep bytes (rows, Ep / 8) -> (rows, Ep) bool: bit j = element 2j, bit 4+j = element 2j+1 of a piece"""
    shifts = torch.tensor([0, 4, 1, 5, 2, 6, 3, 7], device=xm.device, dtype=torch.uint8)
    b = xm.reshape(-1)[:rows * (Ep // 8)].reshape(rows, Ep // 8, 1)
    return ((b >> shifts) & 1).reshape(rows, Ep).bool()


def encoder_state(lib, N, L, E, F, fp16, p=0.0, seed=7, case_seed=0, dead=0.5, live_only=None, compact=True):
    """Tokens, weights and the REAL tensor-core forward (lstur_news_conv_tc_fwd_m) over the compacted title list, as the
    engine runs it: returns the forward's saved state (C16, a, w at the compacted index), keep bytes, tokens_c, live_idx.
    dead: fraction of titles >= 2 made all-pad (title 1 is all-pad already, so compacted and original indices differ);
    live_only: indices of the only live titles.  Rows of tokens_c past n_live hold the valid but wrong id V - 1, which no
    live title uses."""
    tok, P = make_enc_case(N, L, E, F, seed=case_seed)
    V = P['word_emb'].shape[0]
    tok[tok == V - 1] = V - 2
    g = np.random.default_rng(case_seed + 17)
    if live_only is not None:
        keep = np.zeros(N, bool)
        keep[list(live_only)] = True
        tok[~keep] = 0
        tok[keep & ~(tok != 0).any(-1)] = 1 + np.arange(L)[None] % (V - 2)
    elif dead > 0 and N > 2:
        tok[2:][g.random(N - 2) < dead] = 0
    Ep = lib.lstur_tc_padded_e(E)
    dt16 = torch.float16 if fp16 else torch.bfloat16
    dev = lambda x, dt: torch.as_tensor(np.ascontiguousarray(x)).to(dt).to(DEV)
    emb = torch.zeros((V, Ep), dtype=dt16, device=DEV)
    wimg = torch.zeros(lib.lstur_tc_wimg_elems(E, F), dtype=dt16, device=DEV)
    we, cw = dev(P['word_emb'], torch.float32), dev(P['conv_w'], torch.float32)
    ok(lib, lib.lstur_pack_word_emb_16(V, E, P_(we), P_(emb), fp16, stream()))
    ok(lib, lib.lstur_pack_conv_w_tc(E, F, P_(cw), P_(wimg), fp16, stream()))
    t = dev(tok, torch.int32)
    if compact:
        flags, idx, n_live, tok_c = i32(lib.lstur_compact_titles_scratch_ints(N)), i32(N), i32(1), i32((N, L), V - 1)
        ok(lib, lib.lstur_compact_titles(N, L, P_(t), P_(flags), P_(idx), P_(n_live), P_(tok_c), stream()))
    else:
        idx, n_live, tok_c = None, None, t
    cb, aw, ab = dev(P['conv_b'], torch.float32), dev(P['att_w'].reshape(-1), torch.float32), dev(np.asarray(P['att_b']).reshape(1), torch.float32)
    c16 = torch.zeros((N, L, F), dtype=dt16, device=DEV)
    pooled = torch.zeros((N, F), device=DEV)
    a, w = torch.zeros((N, L), device=DEV), torch.zeros((N, L), device=DEV)
    xm = torch.zeros(lib.lstur_tc_xmask_bytes(N, L, E), dtype=torch.uint8, device=DEV) if p > 0 else None
    ok(lib, lib.lstur_news_conv_tc_fwd_m(N, L, E, F, V, P_(tok_c), P_(emb), P_(wimg), P_(cb), P_(aw), P_(ab), P_(c16),
                                         P_(pooled), P_(a), P_(w), ctypes.c_float(p), seed, fp16, 0, PN(xm), PN(n_live),
                                         PN(idx), stream()))
    torch.cuda.synchronize()
    live = np.where((tok != 0).any(-1))[0]
    nl = int(n_live.item()) if compact else N
    if compact:
        assert nl == len(live) and np.array_equal(idx[:nl].cpu().numpy(), live)
    return types.SimpleNamespace(N=N, L=L, E=E, F=F, V=V, Ep=Ep, fp16=fp16, p=p, seed=seed, tok=tok, P=P, live=live,
                                 nl=nl, n_live=n_live, idx=idx if compact else torch.arange(N, dtype=torch.int32, device=DEV),
                                 idx_arg=idx, tok_c=tok_c, emb=emb, cw=cw, aw=aw, c16=c16, a=a, w=w, xm=xm)


def make_d_pooled(st, lddp, seed=3):
    """d pooled (N, lddp): live rows random; the rows of dead titles and the columns past F hold large distinct values, so
    reading a row at the compacted index instead of the original one (or reading past F) shows.  Everything is linear in
    d pooled: it is scaled by a power of two (exactly) so that max |dPre| is in [1/8, 1/4), which keeps 2^17 * dPre inside
    the fp16 range."""
    g = np.random.default_rng(seed)
    dp = (1000.0 + np.arange(st.N * lddp).reshape(st.N, lddp) % 977).astype(np.float32)
    dp[st.live, :st.F] = (g.standard_normal((len(st.live), st.F)) * 0.05).astype(np.float32)
    dp = torch.as_tensor(dp).to(DEV)
    vmax = max([float(attn_reference_chunk(st, dp, n0, min(st.nl, n0 + CHUNK))[0].abs().max()) for n0 in range(0, st.nl, CHUNK)] + [0.0])
    if vmax > 0:
        dp *= 2.0 ** int(np.floor(np.log2(0.25 / vmax)))
    return dp


def run_attn(lib, st, dp, img_scale, accumulate=0, grads=None):
    """lstur_attn_pool_bwd_img as the engine calls it, into an image pre-filled with 0xFF bytes"""
    N, L, F = st.N, st.L, st.F
    img = torch.full((lib.lstur_tc_dpre_img_bytes(N, L, F),), 0xFF, dtype=torch.uint8, device=DEV)
    if grads is None:
        grads = [torch.full((F,), float('nan'), device=DEV), torch.full((F,), float('nan'), device=DEV),
                 torch.full((1,), float('nan'), device=DEV)]
    nb = lib.lstur_attn_bwd_grid(N) * (2 * F + 1) * 4
    part = torch.empty(nb // 4, dtype=torch.float32, device=DEV)
    ok(lib, lib.lstur_attn_pool_bwd_img(st.fp16, N, L, F, P_(st.c16), P_(st.a), P_(st.w), P_(dp), dp.shape[1], P_(st.aw),
                                        P_(img), ctypes.c_float(st.p), ctypes.c_float(img_scale), P_(grads[0]),
                                        P_(grads[1]), P_(grads[2]), accumulate, P_(part), nb, PN(st.n_live),
                                        PN(st.idx_arg), stream()))
    torch.cuda.synchronize()
    return types.SimpleNamespace(img=img, d_att_w=grads[0], d_conv_b=grads[1], d_att_b=grads[2], scale=img_scale)


def attn_reference_chunk(st, dp, n0, n1):
    """float64 attention backward of compacted titles [n0, n1) from the forward's saved C, a, w:
         dw_t = c_t . dp,  q = sum_t w_t dw_t,  dz_t = (dw_t - q) w_t (1 - a_t^2),
         dPre = [c > 0] inv_keep (w_t dp + dz_t att_w)"""
    C = st.c16[n0:n1].to(F64)
    a, w = st.a[n0:n1].to(F64), st.w[n0:n1].to(F64)
    d = dp[st.idx[n0:n1].long(), :st.F].to(F64)          # d pooled rows live at the ORIGINAL title index
    dw = torch.einsum('ntf,nf->nt', C, d)
    q = (w * dw).sum(1, keepdim=True)
    dz = (dw - q) * w * (1 - a * a)
    dpre = (C > 0) * inv_keep(st.p) * (w[..., None] * d[:, None, :] + dz[..., None] * st.aw.to(F64))
    # dw_t - q cancels (the softmax constraint; exactly so for L = 1, where w_0 = 1 up to the 1e-7 guard): the fp32 kernel
    # can only get dz to within rounding of |dw_t| + |q|, so d att_w and d att_b are bounded against the same sums taken
    # over the absolute values of their terms
    dw_abs = torch.einsum('ntf,nf->nt', C.abs(), d.abs())
    dz_abs = (dw_abs + (w * dw_abs).sum(1, keepdim=True)) * w * (1 - a * a)
    return (dpre, torch.einsum('nt,ntf->f', dz, C), dpre.sum((0, 1)), dz.sum(),
            torch.einsum('nt,ntf->f', dz_abs, C.abs()), dz_abs.sum())


def block_slice(img, st, n0, n1):
    blk = img.numel() // st.N
    return img[n0 * blk:n1 * blk]


def check_attn(st, dp, out, check_pad=True):
    """dPre image (element-wise, 16-bit output rounding), its pad rows / pad pieces (exactly zero), untouched blocks past
    n_live, d conv_b (norm-wise 1e-5), and d att_w / d att_b, sums of the cancelling dz_t, to 1e-5 of the same sums over
    the absolute values of their terms."""
    L, F, fp16, nl = st.L, st.F, st.fp16, st.nl
    Fh = F // 2
    c32 = (Fh + 31) // 32 * 32
    # the image holds img_scale * dPre rounded to 16 bits (fp16: round to nearest, |err| <= 2^-11 |x| for normal values,
    # the 1e-6 floor covers subnormal outputs and fp32 rounding of cancelling terms w_t dp + dz_t att_w)
    tol = 2.0 ** -10 if fp16 else 2.0 ** -7
    g_aw = torch.zeros(F, dtype=F64, device=DEV)
    g_cb, g_ab = torch.zeros_like(g_aw), torch.zeros((), dtype=F64, device=DEV)
    s_aw, s_ab = torch.zeros_like(g_aw), torch.zeros((), dtype=F64, device=DEV)
    refs = []
    for n0 in range(0, nl, CHUNK):
        n1 = min(nl, n0 + CHUNK)
        dpre, aw, cb, ab, aw_abs, ab_abs = attn_reference_chunk(st, dp, n0, n1)
        g_aw += aw; g_cb += cb; g_ab += ab; s_aw += aw_abs; s_ab += ab_abs
        words = image_words(block_slice(out.img, st, n0, n1), n1 - n0, L, F)
        got = torch.cat([words_to_f64(words[:, :L, 0, :Fh], fp16), words_to_f64(words[:, :L, 1, :Fh], fp16)], -1) / out.scale
        refs.append((got, dpre))
        if check_pad:
            assert int(torch.count_nonzero(words[:, L:, :, :c32])) == 0, 'pad rows t >= L of a written title are not zero'
            assert int(torch.count_nonzero(words[:, :, :, Fh:c32])) == 0, 'pad pieces F/2 .. next 32 columns are not zero'
    vmax = max([float(r.abs().max()) for _, r in refs] + [1e-30])
    for got, dpre in refs:
        excess = float(((got - dpre).abs() / (tol * dpre.abs() + 1e-6 * vmax)).max()) if dpre.numel() else 0.0
        assert excess <= 1.0, 'dPre image: element-wise bound exceeded by a factor %.3f' % excess
    if check_pad:
        rest = out.img.reshape(st.N, -1)[nl:]
        assert bool((rest == 0xFF).all()), 'image blocks at or past n_live were written'
    ref = dict(att_w=g_aw, conv_b=g_cb, att_b=g_ab)
    if nl == 0:
        assert float(out.d_att_w.abs().max()) == 0 and float(out.d_conv_b.abs().max()) == 0 and float(out.d_att_b[0]) == 0
    else:
        err_aw = float((out.d_att_w.to(F64) - g_aw).abs().max())
        assert err_aw <= 1e-5 * float(s_aw.max()), 'd att_w: %.3e vs scale %.3e (max |ref| %.3e)' % (err_aw, float(s_aw.max()), float(g_aw.abs().max()))
        assert rel(out.d_conv_b.cpu().numpy(), g_cb.cpu().numpy()) <= 1e-5, 'd conv_b'
        err_ab = abs(float(out.d_att_b[0]) - float(g_ab))
        assert err_ab <= 1e-5 * float(s_ab), 'd att_b: %.3e vs scale %.3e' % (err_ab, float(s_ab))
    return ref


def dpre_from_image(st, img, n0, n1, scale):
    """stage-isolated dPre of compacted titles [n0, n1): the decoded device image / img_scale"""
    return decode_dpre_image(block_slice(img, st, n0, n1), n1 - n0, st.L, st.F, st.fp16) / scale


# ---------------------------------------------------------------- 1. lstur_attn_pool_bwd_img alone
ATTN_CASES = [  # N, L, F, dropout, compacted title list
    (1, 1, 16, 0.0, True),
    (3, 7, 48, 0.2, True),
    (37, 30, 400, 0.2, True),
    (37, 30, 400, 0.2, False),          # no device count / index list (NULL arguments)
    (5, 31, 496, 0.0, True),            # F/8 + 2 * pad_pieces = 64: the idle chunk threads exactly cover the pad pieces
    (9, 32, 512, 0.2, True),            # 64-row slot, no pad pieces
    (593, 30, 400, 0.2, True),          # grid capped at 148 x 4 = 592 CTAs: one CTA handles two titles
    (2000, 50, 400, 0.2, True),         # several titles per CTA through both bulk-copy buffers
    (2000, 30, 400, 0.2, True),         # the same with 32-row slots
    (300, 63, 272, 0.0, True),
]


@pytest.mark.parametrize('N,L,F,p,compact', ATTN_CASES)
@pytest.mark.parametrize('fp16', [1, 0])
def test_attn_bwd_img(lib, N, L, F, p, compact, fp16):
    st = encoder_state(lib, N, L, 64, F, fp16, p=p, case_seed=N + L + F, compact=compact)
    if N == 2000:
        assert lib.lstur_attn_bwd_grid(N) < st.nl, 'the grid must be smaller than the live count: CTAs loop over titles'
    dp = make_d_pooled(st, F + 24)
    outs = {}
    for s in (1.0, 2.0 ** 10, 2.0 ** 17):
        outs[s] = run_attn(lib, st, dp, s)
        check_attn(st, dp, outs[s])
    # a power-of-two image scale is exact: d att_w does not see it, d conv_b is summed from the scaled fp32 values and
    # unscaled once at the end, so both (and d att_b) are bit-identical across scales
    for s in (2.0 ** 10, 2.0 ** 17):
        for k in ('d_att_w', 'd_conv_b', 'd_att_b'):
            assert torch.equal(getattr(outs[s], k), getattr(outs[1.0], k)), (s, k)
    # reproducible: a second call gives the same image and gradients, bit for bit
    again = run_attn(lib, st, dp, 2.0 ** 10)
    for k in ('img', 'd_att_w', 'd_conv_b', 'd_att_b'):
        assert torch.equal(getattr(again, k), getattr(outs[2.0 ** 10], k)), k
    # accumulate=1: prior contents + the same new sums (one fp32 add)
    g = torch.Generator(device=DEV).manual_seed(5)
    prior = [torch.randn(F, device=DEV, generator=g), torch.randn(F, device=DEV, generator=g),
             torch.randn(1, device=DEV, generator=g)]
    acc = run_attn(lib, st, dp, 2.0 ** 10, accumulate=1, grads=[x.clone() for x in prior])
    for x, k in zip(prior, ('d_att_w', 'd_conv_b', 'd_att_b')):
        assert torch.equal(getattr(acc, k), x + getattr(outs[1.0], k)), k
    if fp16 and st.nl:
        # a scale that pushes values past the fp16 range: the image saturates to +-65504 (never inf), d conv_b is summed
        # before the 16-bit conversion and is still bit-identical
        vmax = max(float(attn_reference_chunk(st, dp, n0, min(st.nl, n0 + CHUNK))[0].abs().max()) for n0 in range(0, st.nl, CHUNK))
        big = 2.0 ** int(np.ceil(np.log2(4 * 65504.0 / vmax)))
        sat = run_attn(lib, st, dp, big)
        v = decode_dpre_image(sat.img[:st.nl * (sat.img.numel() // st.N)], st.nl, L, F, 1)
        ref = torch.cat([attn_reference_chunk(st, dp, n0, min(st.nl, n0 + CHUNK))[0] for n0 in range(0, st.nl, CHUNK)]) * big
        assert bool(torch.isfinite(v).all())
        over = ref.abs() >= 65520
        assert int(over.sum()) > 0 and torch.equal(v[over], torch.sign(ref[over]) * 65504)
        assert torch.equal(sat.d_conv_b, outs[1.0].d_conv_b) and torch.equal(sat.d_att_w, outs[1.0].d_att_w)


@pytest.mark.parametrize('fp16', [1, 0])
def test_attn_bwd_img_no_live_title(lib, fp16):
    """n_live = 0 on the device (every title all-pad): gradients zeroed with accumulate=0, unchanged with accumulate=1,
    no image byte written"""
    st = encoder_state(lib, 40, 30, 64, 400, fp16, p=0.2, live_only=[])
    assert st.nl == 0
    dp = make_d_pooled(st, 424)
    out = run_attn(lib, st, dp, 2.0 ** 10)
    check_attn(st, dp, out)
    prior = [torch.randn(400, device=DEV), torch.randn(400, device=DEV), torch.randn(1, device=DEV)]
    acc = run_attn(lib, st, dp, 2.0 ** 10, accumulate=1, grads=[x.clone() for x in prior])
    for x, k in zip(prior, ('d_att_w', 'd_conv_b', 'd_att_b')):
        assert torch.equal(getattr(acc, k), x), k
    assert bool((acc.img == 0xFF).all())


@pytest.mark.parametrize('L', [30, 50])
@pytest.mark.parametrize('fp16', [1, 0])
def test_attn_bwd_img_one_live_title(lib, L, fp16):
    """n_live = 1: the only live title sits at original index 6 (its d pooled row is read there)"""
    st = encoder_state(lib, 40, L, 64, 400, fp16, p=0.2, live_only=[6])
    assert st.nl == 1 and int(st.idx[0]) == 6
    dp = make_d_pooled(st, 424)
    check_attn(st, dp, run_attn(lib, st, dp, 2.0 ** 10))


# ---------------------------------------------------------------- 2. the consumers, fed the producer's image
def wgrad_reference(st, dpre_of, keep=None):
    """dW[j] = sum over live titles of X_shift_j (.) mx . dPre, X = the forward's 16-bit table rows of tokens_c,
    mx = keep / (1 - p); chunked over titles.  dpre_of(n0, n1) -> float64 dPre of compacted titles [n0, n1)."""
    L, E = st.L, st.E
    ref = torch.zeros((3, E, st.F), dtype=F64, device=DEV)
    for n0 in range(0, st.nl, CHUNK):
        n1 = min(st.nl, n0 + CHUNK)
        X = st.emb[st.tok_c[n0:n1].long()][:, :, :E].to(F64)
        if st.p > 0:
            X = X * keep[n0 * L:n1 * L, :E].reshape(n1 - n0, L, E) * inv_keep(st.p)
        Xp = torch.nn.functional.pad(X, (0, 0, 1, 1))
        d = dpre_of(n0, n1)
        for j in range(3):
            ref[j] += torch.einsum('nte,ntf->ef', Xp[:, j:j + L], d)
    return ref


def run_wgrad(lib, st, img, scale, xmask):
    nb = lib.lstur_tc_wgrad_partial_bytes(st.N, st.E, st.F)
    ws = torch.empty(nb, dtype=torch.uint8, device=DEV)
    dW = torch.full((3, st.E, st.F), float('nan'), device=DEV)
    ok(lib, lib.lstur_conv_wgrad_tc_m(st.N, st.L, st.E, st.F, st.V, P_(st.tok_c), P_(st.emb), P_(img), P_(dW),
                                      ctypes.c_float(st.p), st.seed, st.fp16, P_(ws), nb, PN(xmask), ctypes.c_float(scale),
                                      PN(st.n_live), stream()))
    torch.cuda.synchronize()
    return dW


def run_dgrad(lib, st, img):
    dt16 = torch.float16 if st.fp16 else torch.bfloat16
    wd = torch.zeros(lib.lstur_tc_wimg_dgrad_elems(st.E, st.F), dtype=dt16, device=DEV)
    ok(lib, lib.lstur_pack_conv_w_dgrad_tc(st.E, st.F, P_(st.cw), P_(wd), st.fp16, stream()))
    dx = torch.full((st.N, st.L, st.Ep), -1, dtype=torch.int16, device=DEV)     # 0xFFFF: NaN in fp16 and bf16
    ok(lib, lib.lstur_conv_dgrad_tc(st.N, st.L, st.E, st.F, P_(img), P_(wd), P_(dx), ctypes.c_float(1.0), st.fp16, 0,
                                    PN(st.n_live), stream()))
    torch.cuda.synchronize()
    return dx


def check_dgrad(st, dx, dpre_img_of):
    """dx16 = sum_j dPre_img[t+1-j] . W16[j]^T (out_scale 1: the image's own scale multiplies through); rows at or past
    n_live untouched, pad columns E..Ep zero"""
    L, E, nl = st.L, st.E, st.nl
    assert bool((dx[nl:] == -1).all()), 'dx16 rows at or past n_live were written'
    got = words_to_f64(dx[:nl], st.fp16)
    assert int(torch.count_nonzero(got[:, :, E:])) == 0
    W16 = torch.as_tensor(round16(st.P['conv_w'], st.fp16)).to(F64).to(DEV)
    tol = 2.0 ** -10 if st.fp16 else 2.0 ** -7
    refs = []
    for n0 in range(0, nl, CHUNK):
        n1 = min(nl, n0 + CHUNK)
        dp = torch.nn.functional.pad(dpre_img_of(n0, n1), (0, 0, 1, 1))
        refs.append(sum(torch.einsum('ntf,ef->nte', dp[:, 2 - j:2 - j + L], W16[j]) for j in range(3)))
    if not nl:
        return None
    ref = torch.cat(refs)
    vmax = float(ref.abs().max())
    # the output is rounded to 16 bits; the floor covers the fp32 accumulation over 3F terms of cancelling sums
    excess = float(((got[:, :, :E] - ref).abs() / (tol * ref.abs() + 1e-4 * vmax)).max())
    assert excess <= 1.0, 'dx16: element-wise bound exceeded by a factor %.3f' % excess
    return ref


def run_scatter(lib, st, dx, scale):
    nb = lib.lstur_word_grad_workspace_bytes(st.N * st.L, st.V, st.E)
    ws = torch.empty(nb, dtype=torch.uint8, device=DEV)
    out = torch.full((st.V, st.E), float('nan'), device=DEV)
    ok(lib, lib.lstur_word_grad_scatter_16(st.N, st.L, st.E, st.V, P_(st.tok_c), P_(dx), st.fp16, ctypes.c_float(scale),
                                           PN(st.xm), P_(out), P_(ws), nb, PN(st.n_live), stream()))
    torch.cuda.synchronize()
    return out


def scatter_reference(st, rows, keep, scale):
    """np.add.at over the live positions of tokens_c of rows (n_live * L, E) (x) keep, times scale"""
    nl, L, E = st.nl, st.L, st.E
    r = rows.reshape(nl * L, rows.shape[-1])[:, :E].to(F64)
    if st.p > 0:
        r = r * keep[:nl * L, :E]
    ref = torch.zeros((st.V, E), dtype=F64, device=DEV)
    ref.index_add_(0, st.tok_c[:nl].reshape(-1).long(), r)
    return ref * scale


def check_scatter(st, out, ref):
    if st.nl:
        assert rel(out.cpu().numpy(), ref.cpu().numpy()) < 2e-6
    else:
        assert float(out.abs().max()) == 0
    # rows no live position touches (the id past n_live among them) are exactly 0
    tc = st.tok_c[:st.nl].cpu().numpy()
    tp = np.pad(tc, ((0, 0), (1, 1)))
    live = (tp[:, :-2] != 0) | (tp[:, 1:-1] != 0) | (tp[:, 2:] != 0)
    absent = np.setdiff1d(np.arange(st.V), np.unique(tc[live]))
    assert st.V - 1 in absent
    assert float(out[torch.as_tensor(absent).to(DEV)].abs().max()) == 0


def engine_img_scale(B):
    """the engine's loss scale of the dPre image for grad_scale = 1/B (csrc/engine.cu, encoder_backward)"""
    _, ex = np.frexp(np.float32(B))
    return 2.0 ** (int(ex) - 1 + 4)


def x_keep(st):
    """X-dropout keep flags (n_live * L, Ep) of the forward: the replicated quad stream, indexed by compacted title"""
    k = rng.quad_keep(st.seed * 2, st.nl * st.L * st.Ep, st.p).reshape(st.nl * st.L, st.Ep)
    return torch.as_tensor(k).to(DEV)


CONSUMER_CASES = [  # live titles, L, E, fp16
    ('odd', 30, 300, 1), ('odd', 30, 300, 0), ('odd', 50, 300, 1), ('none', 30, 300, 1), ('one', 30, 300, 1),
    ('all', 30, 300, 1), ('all', 50, 300, 0), ('odd', 30, 4, 1), ('odd', 30, 'max', 1), ('odd', 50, 'max', 0),
]


@pytest.mark.parametrize('live,L,E,fp16', CONSUMER_CASES)
def test_consumers_fed_producer_image(lib, live, L, E, fp16):
    """wgrad (keep bits and hash replay), dgrad and the word-table scatter on the image lstur_attn_pool_bwd_img wrote,
    with exactly the arguments the engine passes: dropout 0.2, compacted titles (n_titles_dev), img_scale != 1."""
    N, F, p = 37, 400, 0.2
    if E == 'max':        # the widest embedding the tensor-core kernels accept at this L and F
        E = max(e for e in range(4, 1025, 4) if lib.lstur_tc_supported(L, e, F, 3))
    live_only = {'none': [], 'one': [9], 'all': list(range(N)), 'odd': None}[live]
    st = encoder_state(lib, N, L, E, F, fp16, p=p, seed=13, case_seed=N + L + E, live_only=live_only)
    if live == 'odd' and st.nl % 2 == 0:
        st = encoder_state(lib, N, L, E, F, fp16, p=p, seed=13, case_seed=N + L + E, live_only=st.live[:-1])
    assert st.nl == {'none': 0, 'one': 1, 'all': N}.get(live, st.nl) and (live != 'odd' or st.nl % 2 == 1)
    scale = engine_img_scale(256)
    dp = make_d_pooled(st, F)
    att = run_attn(lib, st, dp, scale)
    check_attn(st, dp, att)
    keep = x_keep(st)
    if st.nl:
        assert torch.equal(st.xm[:st.nl * L * (st.Ep // 8)].cpu(),
                           torch.as_tensor(keep_bytes(keep.cpu().numpy())).reshape(-1)), 'forward keep bytes != quad stream'
    dpre_of = lambda n0, n1: dpre_from_image(st, att.img, n0, n1, scale)
    ref = wgrad_reference(st, dpre_of, keep)
    for xmask in (st.xm, None):            # the forward's keep bits, and the replay of the dropout hash
        dW = run_wgrad(lib, st, att.img, scale, xmask)
        if st.nl == 0:
            assert float(dW.abs().max()) == 0
        else:
            assert rel(dW.cpu().numpy(), ref.cpu().numpy()) < 2e-5, 'wgrad (xmask %s)' % ('bits' if xmask is not None else 'replay')
    dx = run_dgrad(lib, st, att.img)
    check_dgrad(st, dx, lambda n0, n1: dpre_from_image(st, att.img, n0, n1, 1.0))
    wscale = float(np.float32(1) / ((np.float32(1) - np.float32(p)) * np.float32(scale)))
    out = run_scatter(lib, st, dx, wscale)
    check_scatter(st, out, scatter_reference(st, words_to_f64(dx[:st.nl], fp16), keep, wscale))


# ---------------------------------------------------------------- 3. the chain at the benchmark's widths, and at C3's title count
@pytest.mark.parametrize('N,L', [(4096, 30), (1024, 50)])
def test_chain_bench_widths(lib, N, L):
    """forward -> attention backward -> wgrad -> dgrad -> scatter at E 300, F 400, fp16, dropout 0.2, ~50 % all-pad
    titles and the engine's image scale for B = 1024.  Each stage against the reference built from the previous stage's
    device output (a failure names one kernel), then the end results against one float64 chain from the forward's
    saved state."""
    E, F, p = 300, 400, 0.2
    st = encoder_state(lib, N, L, E, F, 1, p=p, seed=21, case_seed=N + L)
    scale = engine_img_scale(1024)
    dp = make_d_pooled(st, F)
    att = run_attn(lib, st, dp, scale)
    check_attn(st, dp, att)
    keep = unpack_keep(st.xm, st.nl * L, st.Ep)
    assert torch.equal(keep.cpu(), x_keep(st).cpu())
    dW = run_wgrad(lib, st, att.img, scale, st.xm)
    ref_w = wgrad_reference(st, lambda n0, n1: dpre_from_image(st, att.img, n0, n1, scale), keep)
    assert rel(dW.cpu().numpy(), ref_w.cpu().numpy()) < 2e-5, 'wgrad'
    dx = run_dgrad(lib, st, att.img)
    check_dgrad(st, dx, lambda n0, n1: dpre_from_image(st, att.img, n0, n1, 1.0))
    wscale = float(np.float32(1) / ((np.float32(1) - np.float32(p)) * np.float32(scale)))
    wg = run_scatter(lib, st, dx, wscale)
    check_scatter(st, wg, scatter_reference(st, words_to_f64(dx[:st.nl], 1), keep, wscale))
    # end to end: float64 from the forward's saved state, no 16-bit image in between (bounds: the 16-bit rounding of
    # dPre and of dx16, ~2^-11 per element)
    dpre64 = lambda n0, n1: attn_reference_chunk(st, dp, n0, n1)[0]
    ref_w64 = wgrad_reference(st, dpre64, keep)
    assert rel(dW.cpu().numpy(), ref_w64.cpu().numpy()) < 2e-3, 'wgrad vs the float64 chain'
    W64 = torch.as_tensor(round16(st.P['conv_w'], 1)).to(F64).to(DEV)
    dx64 = []
    for n0 in range(0, st.nl, CHUNK):
        d = torch.nn.functional.pad(dpre64(n0, min(st.nl, n0 + CHUNK)), (0, 0, 1, 1))
        dx64.append(sum(torch.einsum('ntf,ef->nte', d[:, 2 - j:2 - j + L], W64[j]) for j in range(3)))
    dx64 = torch.cat(dx64)
    assert rel((words_to_f64(dx[:st.nl], 1)[:, :, :E] / scale).cpu().numpy(), dx64.cpu().numpy()) < 2e-3, 'dgrad vs the float64 chain'
    ref_wg64 = scatter_reference(st, dx64, keep, inv_keep(p))
    assert rel(wg.cpu().numpy(), ref_wg64.cpu().numpy()) < 3e-3, 'word-table gradient vs the float64 chain'


def test_c3_title_count(lib):
    """56 320 titles at L = 30 (BASELINE config C3: B = 1024, W = 50, K = 4), about half of them live: the attention
    backward over the whole compacted list and the full weight gradient, both against float64 references on the device."""
    N, L, E, F, p = 56320, 30, 300, 400, 0.2
    st = encoder_state(lib, N, L, E, F, 1, p=p, seed=31, case_seed=3)
    assert 0.4 * N < st.nl < 0.6 * N
    scale = engine_img_scale(1024)
    dp = make_d_pooled(st, F)
    att = run_attn(lib, st, dp, scale)
    check_attn(st, dp, att)
    keep = unpack_keep(st.xm, st.nl * L, st.Ep)
    # the keep bytes against the replicated stream on a sample of titles (the whole stream is 2.7e8 flags)
    k0 = rng.quad_keep(st.seed * 2, 64 * L * st.Ep, p).reshape(64 * L, st.Ep)
    assert np.array_equal(keep[:64 * L].cpu().numpy(), k0)
    dW = run_wgrad(lib, st, att.img, scale, st.xm)
    ref = wgrad_reference(st, lambda n0, n1: dpre_from_image(st, att.img, n0, n1, scale), keep)
    # each CTA pair accumulates the token rows of its split (here ~47 000, 18 splits) in fp32 in tensor memory: the
    # rounding grows with the square root of that length, ~5x the 1 700 rows per split of the 1001-title case where 2e-5
    # holds (measured on a B200 at 1000 W: 3.8e-5).  A missing dropout or loss-scale factor is an error of 25 % or more.
    assert rel(dW.cpu().numpy(), ref.cpu().numpy()) < 1e-4
