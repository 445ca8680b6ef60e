"""GPU parity tests for the tensor-core (tcgen05/TMEM, bf16) news encoder and the bf16_tc engine mode.

Tolerance: north_star's 1e-3 relative (max|a-b| / max|b|) on encoder outputs, scores and loss against the
float64 oracle; a tighter check against the oracle fed with bf16-rounded operands isolates kernel bugs from
the (expected) bf16 input rounding.
"""
import ctypes

import numpy as np
import pytest
import torch

from mnexp_b200 import rng, synth
from tolerances import assert_close
from oracle import lstur_numpy as on
from oracle import lstur_torch as ot

pytestmark = pytest.mark.gpu
TOL_SPEC = 1e-3


def rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def P_(t):
    return ctypes.c_void_p(t.data_ptr())


def round16(x, fp16):
    return torch.as_tensor(np.asarray(x, dtype=np.float32)).to(torch.float16 if fp16 else torch.bfloat16).to(torch.float32).numpy()


def stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def run_tc_encoder(lib, tok, P, dropout=0.0, seed=0, max_ctas=0, fp16=1):
    N, L = tok.shape
    ks, E, F = P['conv_w'].shape
    V = P['word_emb'].shape[0]
    Ep = lib.lstur_tc_padded_e(E)
    dev = lambda x, dt: torch.as_tensor(np.ascontiguousarray(x)).to(dt).cuda()
    dt16 = torch.float16 if fp16 else torch.bfloat16
    emb = torch.zeros((V, Ep), dtype=dt16, device='cuda')
    wimg = torch.zeros(lib.lstur_tc_wimg_elems(E, F), dtype=dt16, device='cuda')
    we, cw = dev(P['word_emb'], torch.float32), dev(P['conv_w'], torch.float32)
    assert lib.lstur_pack_word_emb_16(V, E, P_(we), P_(emb), fp16, stream()) == 0
    assert lib.lstur_pack_conv_w_tc(E, F, P_(cw), P_(wimg), fp16, stream()) == 0
    t = dev(tok, torch.int32)
    cb, aw, ab = dev(P['conv_b'], torch.float32), dev(P['att_w'].reshape(-1), torch.float32), dev(np.asarray(P['att_b']).reshape(1), torch.float32)
    c_out = torch.full((N, L, F), float('nan'), dtype=dt16, device='cuda')
    pooled = torch.full((N, F), float('nan'), device='cuda')
    a = torch.full((N, L), float('nan'), device='cuda')
    w = torch.full((N, L), float('nan'), device='cuda')
    rc = lib.lstur_news_conv_tc_fwd(N, L, E, F, V, P_(t), P_(emb), P_(wimg), P_(cb), P_(aw), P_(ab), P_(c_out), P_(pooled),
                                    P_(a), P_(w), ctypes.c_float(dropout), seed, fp16, max_ctas, stream())
    assert rc == 0, lib.lstur_last_error()
    torch.cuda.synchronize()
    return c_out.float().cpu().numpy(), pooled.cpu().numpy(), a.cpu().numpy(), w.cpu().numpy()


def check_attention_given_c(tok, P, c, pooled, a, w):
    """Attention pooling must be exact (fp32 rounding only) given the kernel's own saved bf16 C."""
    m = (c != 0).any(-1).astype(np.float64)
    p_ref, att = on.attention_pool(c.astype(np.float64), m, P['att_w'].astype(np.float64).reshape(-1),
                                   float(np.asarray(P['att_b']).reshape(-1)[0]))
    assert rel(a, att['a']) < 1e-5
    assert rel(w, att['w']) < 1e-5
    assert rel(pooled, p_ref) < 1e-5


def make_enc_case(N, L, E, F, V=500, seed=0, bias=0.05):
    g = np.random.default_rng(seed)
    sh = synth.Shape('t', 10, 10, V, L=L, E=E, F=F, U=8)
    P = synth.make_weights(sh, arch='nigru', seed=seed, bias_noise=bias)
    P['word_emb'] = (g.standard_normal((V, E)) * 0.1).astype(np.float32)   # row 0 is a normal row (mask_zero=False)
    length = g.integers(1, L + 1, N)
    tok = g.integers(1, V, (N, L)).astype(np.int32)
    tok[np.arange(L)[None] >= length[:, None]] = 0
    if N > 2:
        tok[1] = 0                     # an all-pad title
    return tok, P


@pytest.mark.parametrize('N,L,E,F', [(4, 30, 64, 16), (1, 30, 64, 64), (5, 7, 12, 32), (9, 31, 128, 256),
                                     (130, 30, 300, 400), (7, 30, 300, 272), (1500, 30, 300, 400),
                                     # 64-row title slots (L > 31; BASELINE config C5 has L = 50)
                                     (5, 32, 64, 64), (1, 50, 64, 16), (131, 50, 300, 400), (9, 63, 128, 256), (700, 50, 300, 400)])
@pytest.mark.parametrize('fp16', [1, 0])
def test_tc_news_encoder_forward(lib, N, L, E, F, fp16):
    tok, P = make_enc_case(N, L, E, F, seed=N + L + E + F)
    c, pooled, a, w = run_tc_encoder(lib, tok, P, fp16=fp16)
    # (1) kernel exactness: oracle fed the same 16-bit-rounded operands; C itself is stored in 16 bits
    Pq = dict(P, word_emb=round16(P['word_emb'], fp16), conv_w=round16(P['conv_w'], fp16))
    _, aux = on.news_encoder(tok, Pq, use_dense=False, aux=True)
    assert rel(c, aux['C']) < (8e-4 if fp16 else 6e-3)
    check_attention_given_c(tok, P, c, pooled, a, w)
    # (2) spec tolerance vs the true fp32-weights oracle (fp16 operands meet 1e-3; bf16 does not)
    _, aux32 = on.news_encoder(tok, P, use_dense=False, aux=True)
    assert rel(pooled, aux32['p']) < (1e-3 if fp16 else 6e-3)
    # all-pad title pools to exactly 0
    if N > 2:
        assert np.all(pooled[1] == 0)


@pytest.mark.parametrize('L', [30, 50])
def test_tc_matches_across_grid_sizes(lib, L):
    """Persistent-CTA tile scheduling: 1 CTA looping over all tiles == one tile per CTA (bitwise)."""
    tok, P = make_enc_case(300, L, 300, 400, seed=3)
    r1 = run_tc_encoder(lib, tok, P, max_ctas=1)
    r2 = run_tc_encoder(lib, tok, P, max_ctas=0)
    for x, y in zip(r1, r2):
        assert np.array_equal(x, y)


def tc_dropout_masks(seed, N, L, E, Ep, F, p):
    inv = np.float32(1) / (np.float32(1) - np.float32(p))
    def mask(sd, rows, width, used):
        m = rng.quad_keep(sd, rows * width, p).reshape(rows, width)[:, :used]
        return np.where(m, np.float64(inv), 0.0)
    return mask(seed * 2, N * L, Ep, E).reshape(N, L, E), mask(seed * 2 + 1, N * L, F, F).reshape(N, L, F)


@pytest.mark.parametrize('L', [30, 50])
def test_tc_dropout_replay(lib, L):
    N, E, F = 37, 300, 400
    tok, P = make_enc_case(N, L, E, F, seed=11)
    p, seed = 0.2, 5
    c, pooled, a, w = run_tc_encoder(lib, tok, P, dropout=p, seed=seed)
    dx, dc = tc_dropout_masks(seed, N, L, E, lib.lstur_tc_padded_e(E), F, p)
    Pq = dict(P, word_emb=round16(P['word_emb'], 1), conv_w=round16(P['conv_w'], 1))
    _, aux = on.news_encoder(tok, Pq, use_dense=False, aux=True, drop_x=dx, drop_c=dc)
    assert rel(c, aux['C']) < 8e-4
    check_attention_given_c(tok, P, c, pooled, a, w)
    assert abs(float((dx == 0).mean()) - p) < 0.01 and abs(float((dc == 0).mean()) - p) < 0.01


def make_case(shape_name='tiny', arch='igru', seed=0):
    sh = synth.SHAPES[shape_name]
    tok, _, _ = synth.make_docs(sh.n_news, sh.L, sh.vocab)
    P = synth.make_weights(sh, arch=arch, bias_noise=0.05, seed=1237 + seed)
    (b,), _ = synth.make_batches(sh, 1, seed=1236 + seed)
    return sh, tok, P, b


@pytest.mark.parametrize('shape,arch', [('tiny', 'igru'), ('C1', 'igru'), ('C1', 'gru')])
@pytest.mark.parametrize('relu_open', [False, True])
def test_engine_fp16_tc_forward_and_grads(lib, shape, arch, relu_open):
    """relu_open=True shifts the conv bias by +1 so every pre-activation is positive: then no ReLU gate can flip
    between the fp16 forward and the float64 oracle and gradients must agree to rounding (2e-2 incl. cancellation-heavy sums).  With live gates a
    ~1e-3 fraction of near-zero pre-activations flips, which perturbs d(conv_w) by a few % in max-norm — the usual
    ReLU discontinuity, bounded here by cosine > 0.995."""
    from mnexp_b200.engine import LsturEngine
    sh, tok, P, b = make_case(shape, arch)
    if relu_open:
        P = dict(P, conv_b=P['conv_b'] + np.float32(1.0))
    eng = LsturEngine(P, sh.B, sh.W, 1 + sh.K, sh.L, arch=arch, doc_tokens=tok, precision='fp16_tc')
    db = eng.to_device_batch(b)
    eng.forward(db, training=True, seed=1)
    eng.backward(db)
    torch.cuda.synchronize()
    ora = ot.LsturOracle(P, arch=arch)
    out = ora.forward(b['user'], tok[b['hist_doc']], tok[b['cand_doc']], aux=True)
    nh = sh.B * sh.W
    dv = eng.view('doc_vec').reshape(-1, eng.D).cpu().numpy()
    # both readings of the 1e-3 bound: norm-wise and element-wise with an rms floor (tests/tolerances.py)
    assert_close(dv[:nh], out['hist_vec'].detach().numpy().reshape(nh, -1), TOL_SPEC, 'history vectors')
    assert_close(dv[nh:], out['cand_vec'].detach().numpy().reshape(-1, eng.D), TOL_SPEC, 'candidate vectors')
    assert_close(eng.view('user_vec').reshape(sh.B, -1).cpu().numpy(), out['user_vec'].detach().numpy(), TOL_SPEC, 'user vectors')
    assert_close(eng.view('logits').reshape(sh.B, -1).cpu().numpy(), out['logits'].detach().numpy(), TOL_SPEC, 'scores')
    assert_close(eng.view('probs').reshape(sh.B, -1).cpu().numpy(), out['probs'].detach().numpy(), TOL_SPEC, 'probabilities')
    loss, ref = ora.loss_and_grads(b['user'], tok[b['hist_doc']], tok[b['cand_doc']])
    assert abs(eng.loss() - float(loss)) < TOL_SPEC * max(1.0, abs(float(loss)))
    got = eng.get_grads_dict()
    for k, g in ref.items():
        g = g.numpy().astype(np.float64).ravel()
        h = got[k].astype(np.float64).ravel()
        if relu_open:
            assert rel(h, g) < 2e-2, k      # att_w / att_b grads are cancellation-heavy sums (sum_t dz_t ~ 0)
        else:
            cos = float(h @ g / max(np.linalg.norm(h) * np.linalg.norm(g), 1e-300))
            assert cos > 0.995, (k, cos)
            assert abs(np.linalg.norm(h) / np.linalg.norm(g) - 1.0) < 0.02, k


def dpre_image(dpre, fp16=1):
    """numpy restatement of the K-block image layout documented in csrc/attn.cu (attn_bwd_img_kernel)."""
    N, L, F = dpre.shape
    Fh = F // 2
    ngh = (Fh + 63) // 64
    gb = (32 if L <= 31 else 64) * 128           # bytes of one 64-column group of one title slot
    img = np.zeros(N * 2 * ngh * gb // 2, dtype=np.float16 if fp16 else np.uint16)
    n, t, f = np.meshgrid(np.arange(N), np.arange(L), np.arange(F), indexing='ij')
    h = (f >= Fh).astype(np.int64)
    fl = f - h * Fh
    byte = n * (2 * ngh * gb) + (h * ngh + (fl >> 6)) * gb + t * 128 + ((((fl & 63) >> 3) ^ (t & 7)) << 4) + (fl & 7) * 2
    if fp16:
        img[byte.ravel() // 2] = dpre.astype(np.float16).ravel()
    else:
        img[byte.ravel() // 2] = torch.as_tensor(dpre.ravel()).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)
    return img


@pytest.mark.parametrize('N,L,E,F', [(2, 30, 64, 64), (5, 7, 12, 32), (3, 31, 128, 256), (64, 30, 300, 400),
                                     (1001, 30, 300, 400), (3, 32, 64, 64), (65, 50, 300, 400), (9, 63, 128, 256)])
@pytest.mark.parametrize('fp16', [1, 0])
def test_tc_conv_wgrad(lib, N, L, E, F, fp16):
    tok, P = make_enc_case(N, L, E, F, seed=N + E)
    g = np.random.default_rng(N)
    dpre = (g.standard_normal((N, L, F)) * (g.random((N, L, F)) < 0.5)).astype(np.float32)
    V = P['word_emb'].shape[0]
    Ep = lib.lstur_tc_padded_e(E)
    dt16 = torch.float16 if fp16 else torch.bfloat16
    emb = torch.zeros((V, Ep), dtype=dt16, device='cuda')
    we = torch.as_tensor(P['word_emb']).cuda()
    assert lib.lstur_pack_word_emb_16(V, E, P_(we), P_(emb), fp16, stream()) == 0
    img = torch.as_tensor(dpre_image(dpre, fp16).view(np.int16)).cuda()
    assert img.numel() * 2 == lib.lstur_tc_dpre_img_bytes(N, L, F)
    nb = lib.lstur_tc_wgrad_partial_bytes(N, E, F)
    ws = torch.empty(nb, dtype=torch.uint8, device='cuda')
    dW = torch.full((3, E, F), float('nan'), device='cuda')
    t = torch.as_tensor(tok).cuda()
    rc = lib.lstur_conv_wgrad_tc(N, L, E, F, V, P_(t), P_(emb), P_(img), P_(dW), ctypes.c_float(0.0), 0, fp16, P_(ws), nb, stream())
    assert rc == 0, lib.lstur_last_error()
    torch.cuda.synchronize()
    X = round16(P['word_emb'], fp16).astype(np.float64)[tok]                 # (N,L,E)
    Xp = np.zeros((N, L + 2, E)); Xp[:, 1:L + 1] = X
    d16 = round16(dpre, fp16).astype(np.float64)
    ref = np.stack([np.einsum('nte,ntf->ef', Xp[:, j:j + L], d16) for j in range(3)])
    assert rel(dW.cpu().numpy(), ref) < 2e-5


@pytest.mark.parametrize('ta,tb', [(0, 0), (1, 0), (0, 1), (1, 1)])
@pytest.mark.parametrize('M,N,K', [(1, 1, 1), (130, 72, 33), (400, 200, 56320), (200, 600, 5000), (51200, 600, 200),
                                   (257, 304, 200), (128, 256, 64), (1000, 400, 200)])
def test_gemm_tc(lib, ta, tb, M, N, K):
    if M * K > 3e7 and ta:
        pytest.skip('covered by the non-transposed case')
    g = np.random.default_rng(M * 7 + N * 3 + K + ta * 2 + tb)
    A = g.standard_normal((K, M) if ta else (M, K)).astype(np.float32)
    Bm = g.standard_normal((N, K) if tb else (K, N)).astype(np.float32)
    bias = g.standard_normal(N).astype(np.float32)
    C = torch.full((M, N), float('nan'), device='cuda')
    nb = lib.lstur_gemm_tc_workspace_bytes(M, N, K)
    ws = torch.empty(max(nb, 4), dtype=torch.uint8, device='cuda')
    a_d, b_d, bias_d = torch.as_tensor(A).cuda(), torch.as_tensor(Bm).cuda(), torch.as_tensor(bias).cuda()
    rc = lib.lstur_gemm_tc(ta, tb, M, N, K, P_(a_d), A.shape[1], P_(b_d), Bm.shape[1], P_(C), N, P_(bias_d), 1, P_(ws), nb, stream())
    assert rc == 0, lib.lstur_last_error()
    torch.cuda.synchronize()
    A16, B16 = round16(A, 1).astype(np.float64), round16(Bm, 1).astype(np.float64)
    ref = np.maximum((A16.T if ta else A16) @ (B16.T if tb else B16) + bias, 0)
    assert rel(C.cpu().numpy(), ref) < 2e-5
    # 3-term split mode (LSTUR_GEMM_PRECISE): close to the un-rounded fp32 operands
    C.fill_(float('nan'))
    rc = lib.lstur_gemm_tc(ta, tb, M, N, K, P_(a_d), A.shape[1], P_(b_d), Bm.shape[1], P_(C), N, P_(bias_d), 1 | 4, P_(ws), nb, stream())
    assert rc == 0, lib.lstur_last_error()
    torch.cuda.synchronize()
    A64, B64 = A.astype(np.float64), Bm.astype(np.float64)
    ref = np.maximum((A64.T if ta else A64) @ (B64.T if tb else B64) + bias, 0)
    assert rel(C.cpu().numpy(), ref) < (5e-6 if K < 10000 else 3e-5)      # fp32 accumulation over K terms


@pytest.mark.parametrize('N,L,E,F', [(5, 7, 12, 32), (64, 30, 300, 400), (333, 30, 300, 400), (77, 50, 300, 400)])
def test_keep_bits_from_forward_equal_hash_replay(lib, N, L, E, F):
    """The weight-gradient kernel either replays the X-dropout hash or reads the keep bits the forward left behind
    (one byte per 16-byte piece): both must give bit-identical gradients, and the bytes must equal the replicated stream."""
    from mnexp_b200 import rng
    tok, P = make_enc_case(N, L, E, F, seed=N + F)
    g = np.random.default_rng(N)
    dpre = (g.standard_normal((N, L, F)) * (g.random((N, L, F)) < 0.5)).astype(np.float32)
    V = P['word_emb'].shape[0]
    Ep = lib.lstur_tc_padded_e(E)
    emb = torch.zeros((V, Ep), dtype=torch.float16, device='cuda')
    wimg = torch.zeros(lib.lstur_tc_wimg_elems(E, F), dtype=torch.float16, device='cuda')
    f32 = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float32)).cuda()
    we, cw, cb, aw, ab = (f32(P[k]) for k in ('word_emb', 'conv_w', 'conv_b', 'att_w', 'att_b'))
    assert lib.lstur_pack_word_emb_16(V, E, P_(we), P_(emb), 1, stream()) == 0
    assert lib.lstur_pack_conv_w_tc(E, F, P_(cw), P_(wimg), 1, stream()) == 0
    t = torch.as_tensor(tok).cuda()
    c_out = torch.empty((N, L, F), dtype=torch.float16, device='cuda')
    pooled = torch.empty((N, F), device='cuda')
    nbm = lib.lstur_tc_xmask_bytes(N, L, E)
    xm = torch.full((nbm,), 0xAA, dtype=torch.uint8, device='cuda')
    seed, drop = 11, 0.2
    rc = lib.lstur_news_conv_tc_fwd_m(N, L, E, F, V, P_(t), P_(emb), P_(wimg), P_(cb), P_(aw), P_(ab), P_(c_out), P_(pooled),
                                      None, None, ctypes.c_float(drop), seed, 1, 0, P_(xm), None, None, stream())
    assert rc == 0, lib.lstur_last_error()
    # bytes == the replicated quad stream of the X dropout (seed * 2, elements indexed (title, token, column of Ep))
    keep = rng.quad_keep(seed * 2, N * L * Ep, drop).reshape(N, L, Ep // 8, 4, 2)
    want = np.zeros((N, L, Ep // 8), dtype=np.uint8)
    for j in range(4):
        want |= (keep[..., j, 0].astype(np.uint8) << j) | (keep[..., j, 1].astype(np.uint8) << (4 + j))
    assert np.array_equal(xm.cpu().numpy().reshape(N, L, Ep // 8), want)
    img = torch.as_tensor(dpre_image(dpre, 1).view(np.int16)).cuda()
    nb = lib.lstur_tc_wgrad_partial_bytes(N, E, F)
    ws = torch.empty(nb, dtype=torch.uint8, device='cuda')
    outs = []
    for mask in (None, xm):
        dW = torch.full((3, E, F), float('nan'), device='cuda')
        rc = lib.lstur_conv_wgrad_tc_m(N, L, E, F, V, P_(t), P_(emb), P_(img), P_(dW), ctypes.c_float(drop), seed, 1, P_(ws), nb,
                                       P_(mask) if mask is not None else None, ctypes.c_float(1.0), None, stream())
        assert rc == 0, lib.lstur_last_error()
        torch.cuda.synchronize()
        outs.append(dW.cpu().numpy())
    assert np.isfinite(outs[0]).all() and np.array_equal(outs[0], outs[1])


# ---------------------------------------------------------------- word-table training path (task/paper.py:136)
@pytest.mark.parametrize('N,L,E,F', [(2, 30, 64, 64), (5, 7, 12, 32), (3, 31, 128, 256), (64, 30, 300, 400), (601, 30, 300, 400),
                                     (3, 32, 64, 64), (65, 50, 300, 400), (9, 63, 128, 256)])
@pytest.mark.parametrize('fp16', [1, 0])
def test_tc_conv_dgrad(lib, N, L, E, F, fp16):
    """Conv1D input gradient on tcgen05: dX[m, e] = sum_j sum_f dPre[m+1-j, f] * Wc[j, e, f] within each title."""
    g = np.random.default_rng(N + L + E + F)
    dpre = (g.standard_normal((N, L, F)) * (g.random((N, L, F)) < 0.5)).astype(np.float32)
    Wc = (g.standard_normal((3, E, F)) * 0.05).astype(np.float32)
    Ep = lib.lstur_tc_padded_e(E)
    dt16 = torch.float16 if fp16 else torch.bfloat16
    # the pad columns of the image hold garbage in the workspace of a real run (here: NaN) except where the producer
    # kernel zeroes them; build the image over NaN to prove that no unwritten byte is consumed
    img_np = dpre_image(dpre, fp16)
    if fp16:
        Fh, slot = F // 2, (32 if L <= 31 else 64)
        ngh, c32 = (Fh + 63) // 64, (Fh + 31) // 32 * 32
        n, t, h, fl = np.meshgrid(np.arange(N), np.arange(slot), np.arange(2), np.arange(c32, ngh * 64), indexing='ij')
        if fl.size:
            gb = slot * 128
            byte = n * (2 * ngh * gb) + (h * ngh + (fl >> 6)) * gb + t * 128 + ((((fl & 63) >> 3) ^ (t & 7)) << 4) + (fl & 7) * 2
            img_np[byte.ravel() // 2] = np.nan
    img = torch.as_tensor(img_np.view(np.int16)).cuda()
    wd = torch.zeros(lib.lstur_tc_wimg_dgrad_elems(E, F), dtype=dt16, device='cuda')
    cw = torch.as_tensor(Wc).cuda()
    assert lib.lstur_pack_conv_w_dgrad_tc(E, F, P_(cw), P_(wd), fp16, stream()) == 0
    dx = torch.full((N, L, Ep), float('nan'), dtype=dt16, device='cuda')
    rc = lib.lstur_conv_dgrad_tc(N, L, E, F, P_(img), P_(wd), P_(dx), ctypes.c_float(0.5), fp16, 0, None, stream())
    assert rc == 0, lib.lstur_last_error()
    torch.cuda.synchronize()
    d16 = round16(dpre, fp16).astype(np.float64)
    W16 = round16(Wc, fp16).astype(np.float64)
    dp = np.zeros((N, L + 2, F)); dp[:, 1:L + 1] = d16
    # dX[t] = sum_j dPre[t+1-j] . Wc[j]^T  ->  padded index (t+1-j)+1 = t+2-j
    ref = 0.5 * sum(np.einsum('ntf,ef->nte', dp[:, 2 - j:2 - j + L], W16[j]) for j in range(3))
    got = dx.float().cpu().numpy()
    assert np.all(got[:, :, E:] == 0)
    assert rel(got[:, :, :E], ref) < (1.5e-3 if fp16 else 1e-2)          # the output itself is rounded to 16 bits


def keep_bytes(keep):
    """(rows, Ep) bool -> the forward's keep bytes (rows, Ep/8): bit j = element 2j, bit 4+j = element 2j+1 of a 16-byte piece"""
    k = keep.reshape(keep.shape[0], -1, 4, 2).astype(np.uint8)
    return (k[..., 0] << np.arange(4, dtype=np.uint8)).sum(-1).astype(np.uint8) | ((k[..., 1] << (4 + np.arange(4, dtype=np.uint8))).sum(-1).astype(np.uint8))


@pytest.mark.parametrize('N,L,E,V,hot', [(3, 7, 12, 40, 0.0), (50, 30, 300, 1000, 0.3), (2000, 30, 64, 500, 0.6), (7000, 50, 32, 100000, 0.9),
                                         (1, 1, 4, 1, 0.0)])
@pytest.mark.parametrize('masked', [False, True])
def test_word_grad_scatter_16(lib, N, L, E, V, hot, masked):
    """Segment-sorted scatter-add of the token rows into the word table: exact grouping, fixed summation order
    (bit-reproducible), heavy tokens (one token owning up to 90 % of the positions: > R^2 rows -> all three levels)."""
    g = np.random.default_rng(N * 31 + L + E)
    Ep = lib.lstur_tc_padded_e(E)
    tok = g.integers(1, V, (N, L)).astype(np.int32) if V > 1 else np.zeros((N, L), np.int32)
    if hot > 0:
        tok[g.random((N, L)) < hot] = min(3, V - 1)
    length = g.integers(1, L + 1, N)
    tok[np.arange(L)[None] >= length[:, None]] = 0
    if N > 2:
        tok[1] = 0
    dx = g.standard_normal((N * L, Ep)).astype(np.float16)
    dx[:, E:] = 0
    keep = g.random((N * L, Ep)) < 0.8 if masked else np.ones((N * L, Ep), bool)
    t_d = torch.as_tensor(tok).cuda()
    dx_d = torch.as_tensor(dx).cuda()
    km = torch.as_tensor(keep_bytes(keep)).cuda() if masked else None
    nb = lib.lstur_word_grad_workspace_bytes(N * L, V, E)
    ws = torch.empty(nb, dtype=torch.uint8, device='cuda')
    outs = []
    for _ in range(2):
        out = torch.full((V, E), float('nan'), device='cuda')
        rc = lib.lstur_word_grad_scatter_16(N, L, E, V, P_(t_d), P_(dx_d), 1, ctypes.c_float(0.25), P_(km) if masked else None,
                                            P_(out), P_(ws), nb, None, stream())
        assert rc == 0, lib.lstur_last_error()
        torch.cuda.synchronize()
        outs.append(out.cpu().numpy())
    assert np.array_equal(outs[0], outs[1])                       # bit-reproducible
    # positions whose conv window holds no real token carry an exactly-zero gradient in the real pipeline and are
    # dropped by the kernel; zero them in the reference input too
    tp = np.pad(tok, ((0, 0), (1, 1)))
    live = ((tp[:, :-2] != 0) | (tp[:, 1:-1] != 0) | (tp[:, 2:] != 0)).reshape(-1)
    rows = dx.astype(np.float64)[:, :E] * keep[:, :E] * live[:, None]
    ref = np.zeros((V, E))
    np.add.at(ref, tok.reshape(-1), rows)
    ref *= 0.25
    assert rel(outs[0], ref) < 2e-6
    absent = np.setdiff1d(np.arange(V), np.unique(tok[live.reshape(N, L)]))
    assert np.all(outs[0][absent] == 0)


# ---------------------------------------------------------------- live-title compaction
@pytest.mark.parametrize('N,L', [(1, 7), (1000, 30), (5000, 50), (3, 1), (51200, 1), (1025, 1)])
def test_compact_titles_bit_exact(lib, N, L):
    g = np.random.default_rng(N + L)
    tok = g.integers(0, 5, (N, L)).astype(np.int32)
    tok[g.random(N) < 0.45] = 0                      # all-pad titles
    t = torch.as_tensor(tok).cuda()
    flags = torch.full((lib.lstur_compact_titles_scratch_ints(N),), -7, dtype=torch.int32, device='cuda')
    idx = torch.full((N,), -7, dtype=torch.int32, device='cuda')
    n_live, tc_ = torch.full((1,), -7, dtype=torch.int32, device='cuda'), torch.full((N, L), -7, dtype=torch.int32, device='cuda')
    assert lib.lstur_compact_titles(N, L, P_(t), P_(flags), P_(idx), P_(n_live), P_(tc_), stream()) == 0
    torch.cuda.synchronize()
    live = np.where((tok != 0).any(-1))[0]
    assert int(n_live[0]) == len(live)
    assert np.array_equal(idx.cpu().numpy()[:len(live)], live)
    assert np.array_equal(tc_.cpu().numpy()[:len(live)], tok[live])


@pytest.mark.parametrize('L', [30, 50])
def test_tc_forward_over_compacted_titles(lib, L):
    """the kernel over the compacted live-title list (device-side count, pooled rows written at the original index)
    == the kernel over all titles, bit for bit; dead titles pool to exactly 0 either way"""
    N, E, F = 301, 300, 400
    tok, P = make_enc_case(N, L, E, F, seed=5)
    tok[np.random.default_rng(1).random(N) < 0.5] = 0
    c0, pooled0, a0, w0 = run_tc_encoder(lib, tok, P)
    V, Ep = P['word_emb'].shape[0], lib.lstur_tc_padded_e(E)
    dev = lambda x, dt: torch.as_tensor(np.ascontiguousarray(x)).to(dt).cuda()
    emb = torch.zeros((V, Ep), dtype=torch.float16, device='cuda')
    wimg = torch.zeros(lib.lstur_tc_wimg_elems(E, F), dtype=torch.float16, device='cuda')
    we, cw = dev(P['word_emb'], torch.float32), dev(P['conv_w'], torch.float32)
    assert lib.lstur_pack_word_emb_16(V, E, P_(we), P_(emb), 1, stream()) == 0
    assert lib.lstur_pack_conv_w_tc(E, F, P_(cw), P_(wimg), 1, stream()) == 0
    t = dev(tok, torch.int32)
    i32 = lambda *s: torch.zeros(s, dtype=torch.int32, device='cuda')
    flags, idx, n_live, tok_c = i32(lib.lstur_compact_titles_scratch_ints(N)), i32(N), i32(1), i32(N, L)
    assert lib.lstur_compact_titles(N, L, P_(t), P_(flags), P_(idx), P_(n_live), P_(tok_c), stream()) == 0
    cb, aw, ab = dev(P['conv_b'], torch.float32), dev(P['att_w'].reshape(-1), torch.float32), dev(np.asarray(P['att_b']).reshape(1), torch.float32)
    c_out = torch.zeros((N, L, F), dtype=torch.float16, device='cuda')
    pooled = torch.zeros((N, F), device='cuda')
    a, w = torch.zeros((N, L), device='cuda'), torch.zeros((N, L), device='cuda')
    rc = lib.lstur_news_conv_tc_fwd_m(N, L, E, F, V, P_(tok_c), P_(emb), P_(wimg), P_(cb), P_(aw), P_(ab), P_(c_out), P_(pooled),
                                      P_(a), P_(w), ctypes.c_float(0.0), 0, 1, 0, None, P_(n_live), P_(idx), stream())
    assert rc == 0, lib.lstur_last_error()
    torch.cuda.synchronize()
    live = np.where((tok != 0).any(-1))[0]
    assert np.array_equal(pooled.cpu().numpy(), pooled0)
    assert np.all(pooled0[np.setdiff1d(np.arange(N), live)] == 0)
    assert np.array_equal(c_out.float().cpu().numpy()[:len(live)], c0[live])
    assert np.array_equal(w.cpu().numpy()[:len(live)], w0[live])
