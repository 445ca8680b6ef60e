"""Word-table training (reference: keras Embedding(trainable=config.textual_embedding_trainable), task/paper.py:132-138,
main.py:36): conv input gradient + deterministic segment-sorted scatter-add + dense Keras-Adam on the table, checked
against autograd of the oracle — with the X / C dropout masks of the device streams replayed into it."""
import numpy as np
import pytest
import torch

from mnexp_b200 import rng, synth
from oracle import lstur_torch as ot
from tolerances import rel

pytestmark = pytest.mark.gpu


def oracle_grads(P, arch, b, tok, masks=None, dtype=torch.float64):
    """loss and gradients (word table included) of the oracle graph, optionally under given dropout multipliers"""
    ora = ot.LsturOracle(P, arch=arch, dtype=dtype, trainable_word_emb=True)
    Pt = ora.P
    user = torch.as_tensor(b['user']).long()
    ht, ct = torch.as_tensor(tok[b['hist_doc']]).long(), torch.as_tensor(tok[b['cand_doc']]).long()
    B, W, Lt = ht.shape
    C = ct.shape[1]
    toks = torch.cat([ht.reshape(B * W, Lt), ct.reshape(B * C, Lt)])
    dx, dc = (None, None) if masks is None else [torch.as_tensor(m, dtype=dtype) for m in masks]
    d = ot.news_encoder(toks, Pt, drop_x=dx, drop_c=dc)
    H = d[:B * W].reshape(B, W, -1) * (ht != 0).any(-1).to(d.dtype).unsqueeze(-1)
    u = ot.user_encoder(arch, user, H, Pt)
    probs = torch.softmax(ot.score(u, d[B * W:].reshape(B, C, -1)), -1)
    y = torch.zeros_like(probs)
    y[:, 0] = 1.0
    loss = ot.categorical_crossentropy(y, probs)
    gs = torch.autograd.grad(loss, [Pt[k] for k in ora.trainable], allow_unused=True)
    return float(loss), {k: (None if g is None else g.numpy()) for k, g in zip(ora.trainable, gs)}


def case(sh, arch='igru', seed=0, relu_open=False):
    tok, _, _ = synth.make_docs(sh.n_news, sh.L, sh.vocab)
    P = synth.make_weights(sh, arch=arch, bias_noise=0.05, seed=1237 + seed)
    P['word_emb'] = P['word_emb'].copy()
    P['word_emb'][0] = 0.03                 # row 0 is looked up like any row (mask_zero=False) and is trained too
    if relu_open:
        P['conv_b'] = P['conv_b'] + np.float32(1.0)
    (b,), _ = synth.make_batches(sh, 1, seed=1236 + seed)
    return tok, P, b


@pytest.mark.parametrize('k', [3, 2, 4, 5])
@pytest.mark.parametrize('dropout', [0.0, 0.2])
def test_word_table_gradient_fp32(lib, dropout, k):
    """fp32 mode: d word_emb == autograd to <= 5e-5, bit-reproducible run to run, at filter widths 2 .. 5 (an even
    width's 'same' halo reaches one more position back than forward)"""
    from mnexp_b200.engine import LsturEngine
    sh = synth.Shape('wt', 50, 80, 120, L=7, W=5, K=2, B=6, E=12, F=16, U=8, k=k)
    tok, P, b = case(sh)
    eng = LsturEngine(P, sh.B, sh.W, 1 + sh.K, sh.L, arch='igru', doc_tokens=tok, dropout=dropout, trainable_word_emb=True)
    db = eng.to_device_batch(b)
    seed = 9
    grads = []
    for _ in range(2):
        eng.forward(db, training=True, seed=seed)
        eng.backward(db)
        torch.cuda.synchronize()
        grads.append(eng.get_grads_dict())
    assert np.array_equal(grads[0]['word_emb'], grads[1]['word_emb'])
    masks = None
    if dropout > 0:
        N = sh.B * (sh.W + 1 + sh.K)
        masks = (rng.dropout_multiplier(seed * 2, N * sh.L * sh.E, dropout).reshape(N, sh.L, sh.E),
                 rng.dropout_multiplier(seed * 2 + 1, N * sh.L * sh.F, dropout).reshape(N, sh.L, sh.F))
    loss, ref = oracle_grads(P, 'igru', b, tok, masks)
    assert abs(eng.loss() - loss) < 2e-5 * max(1.0, abs(loss))
    assert rel(grads[0]['word_emb'], ref['word_emb']) < 5e-5
    assert rel(grads[0]['conv_w'], ref['conv_w']) < 5e-5
    used = np.unique(np.concatenate([tok[b['hist_doc']].ravel(), tok[b['cand_doc']].ravel()]))
    absent = np.setdiff1d(np.arange(sh.vocab), used)
    assert np.all(grads[0]['word_emb'][absent] == 0)
    assert np.abs(grads[0]['word_emb'][0]).max() > 0            # the pad token's row gets the halo contributions


@pytest.mark.parametrize('L_,dropout', [(30, 0.0), (30, 0.2), (50, 0.0)])
def test_word_table_gradient_fp16_tc(lib, L_, dropout):
    """tensor-core mode at full width (E300 F400 U200), both title-slot heights.  The conv bias is shifted so that no
    ReLU gate can flip between the 16-bit forward and the float64 oracle (see test_engine_fp16_tc_forward_and_grads)."""
    from mnexp_b200.engine import LsturEngine
    sh = synth.Shape('wt16', 40, 300, 2000, L=L_, W=20, K=4, B=8, E=300, F=400, U=200)
    tok, P, b = case(sh, seed=3, relu_open=True)
    eng = LsturEngine(P, sh.B, sh.W, 1 + sh.K, sh.L, arch='igru', doc_tokens=tok, dropout=dropout, precision='fp16_tc',
                      trainable_word_emb=True)
    db = eng.to_device_batch(b)
    seed = 4
    grads = []
    for _ in range(2):
        eng.forward(db, training=True, seed=seed)
        eng.backward(db)
        torch.cuda.synchronize()
        grads.append(eng.get_grads_dict())
    assert np.array_equal(grads[0]['word_emb'], grads[1]['word_emb'])      # deterministic
    masks = None
    if dropout > 0:
        toks = np.concatenate([tok[b['hist_doc']].reshape(-1, sh.L), tok[b['cand_doc']].reshape(-1, sh.L)])
        masks = rng.tc_dropout_multipliers(seed, toks, sh.E, lib.lstur_tc_padded_e(sh.E), sh.F, dropout)
    loss, ref = oracle_grads(P, 'igru', b, tok, masks)
    assert abs(eng.loss() - loss) < 1e-3 * max(1.0, abs(loss))
    g, r = grads[0]['word_emb'].astype(np.float64), ref['word_emb']
    assert rel(g, r) < 2e-2
    cos = float((g * r).sum() / (np.linalg.norm(g) * np.linalg.norm(r)))
    assert cos > 0.9995, cos
    assert rel(grads[0]['conv_w'], ref['conv_w']) < 2e-2


@pytest.mark.parametrize('precision', ['fp32', 'fp16_tc'])
def test_word_table_train_steps_match_oracle_adam(lib, precision):
    """three training steps with the table trainable: dense Keras-Adam on it (reference semantics)"""
    from mnexp_b200.engine import LsturEngine
    sh = synth.Shape('wt', 50, 80, 120, L=7, W=5, K=2, B=6, E=12, F=16, U=8) if precision == 'fp32' else \
        synth.Shape('wt16', 40, 300, 2000, L=30, W=20, K=4, B=8, E=300, F=400, U=200)
    tok, P, _ = case(sh, seed=5, relu_open=precision != 'fp32')
    batches, _ = synth.make_batches(sh, 3, seed=77)
    eng = LsturEngine(P, sh.B, sh.W, 1 + sh.K, sh.L, arch='igru', doc_tokens=tok, lr=1e-3, sparse_user_adam=False,
                      precision=precision, trainable_word_emb=True)
    ora = ot.LsturOracle(P, arch='igru', lr=1e-3, trainable_word_emb=True)
    for b in batches:
        lg = float(eng.train_step(eng.to_device_batch(b))[0])
        lo = ora.train_step(b['user'], tok[b['hist_doc']], tok[b['cand_doc']], training=False)
        assert abs(lg - lo) < (1e-4 if precision == 'fp32' else 1e-3) * max(1, abs(lo))
    w = eng.get_weights_dict()
    moved = np.abs(w['word_emb'] - P['word_emb']).max()
    assert moved > 1e-3                       # three Adam steps of ~lr each
    if precision == 'fp32':
        for k in ora.trainable:
            assert np.abs(w[k] - ora.P[k].detach().numpy()).max() < 2e-5, k
    else:
        # Adam normalises every gradient to ~lr, so elements whose gradient is tiny flip sign under 16-bit rounding; the
        # bulk of the table must still move with the oracle
        d_e, d_o = w['word_emb'] - P['word_emb'], ora.P['word_emb'].detach().numpy() - P['word_emb']
        sel = np.abs(d_o) > 2e-3
        assert sel.sum() > 1000 and np.mean(np.sign(d_e[sel]) == np.sign(d_o[sel])) > 0.98
