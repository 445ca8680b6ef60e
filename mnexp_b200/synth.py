"""Seeded synthetic Vocab / DocMeta / ClickData / weights / batches (SURVEY.md §8d).

The reference's datasets are private (README.md:8), so every measurement and
parity run uses data of the reference's shapes generated here:

* Vocab     : (V,E) fp32 N(0,0.1²), row 0 = zeros — what
              ``utils.load_textual_embedding`` yields for a missing index
              (utils.py:43-49).
* DocMeta   : doc ids 1..n_news (+ pad doc 0 = all-zero title,
              task/seq2vec.py:104-108); title tokens Zipf(1.1) over 1..V-1,
              right-zero-padded to L (document.py:37-54); vertical in 1..15,
              subvertical in 1..306 (utils.py:153-228).
* ClickData : per-sample history of h clicks, left-padded with doc 0 to W
              (task/seq2vec.py:17-49); 1 positive + K negatives sampled with
              replacement (task/paper.py:17-18), positive first (:529).
* weights   : Keras initialisers (SURVEY §9.8).
"""
from dataclasses import dataclass, asdict

import numpy as np


@dataclass
class Shape:
    name: str
    n_users: int
    n_news: int
    vocab: int
    L: int = 30           # title_shape
    W: int = 50           # window_size
    K: int = 4            # negative_samples
    B: int = 64           # batch_size
    E: int = 300          # textual_embedding_dim
    F: int = 400          # title_filter_shape[0]
    k: int = 3            # title_filter_shape[1]
    U: int = 200          # user_embedding_dim
    arch: str = 'igru'

    def dict(self):
        return asdict(self)


# BASELINE.json configs[0..4]
SHAPES = {
    'C1': Shape('C1', 1_000, 5_000, 30_000, B=64, arch='igru'),
    'C2': Shape('C2', 50_000, 50_000, 30_000, B=1024, arch='gru'),
    'C3': Shape('C3', 1_000_000, 130_000, 100_000, B=1024, arch='igru'),
    'C4': Shape('C4', 1_000_000, 130_000, 100_000, B=1024, arch='igru'),
    'C5': Shape('C5', 1_000_000, 130_000, 100_000, L=50, W=200, B=2048, arch='igru'),
    'tiny': Shape('tiny', 50, 80, 120, L=7, W=5, K=2, B=6, E=12, F=16, U=8),
}


def _zipf_cdf(n, s):
    p = 1.0 / np.arange(1, n + 1, dtype=np.float64) ** s
    c = np.cumsum(p)
    return c / c[-1]


def _zipf_sample(rng, cdf, size):
    return np.searchsorted(cdf, rng.random(size), side='left').astype(np.int64)


def make_vocab(V, E, seed=1234):
    rng = np.random.default_rng(seed)
    emb = (rng.standard_normal((V, E)) * 0.1).astype(np.float32)
    emb[0] = 0.0
    return emb


def make_docs(n_news, L, V, seed=1235):
    """-> tokens (n_news+1, L) int32 (row 0 = pad doc), vert (n_news+1,), subvert (n_news+1,)."""
    rng = np.random.default_rng(seed)
    n = n_news + 1
    length = np.clip(np.rint(rng.normal(0.6 * L, 0.2 * L, n)), min(3, L), L).astype(np.int64)
    cdf = _zipf_cdf(V - 1, 1.1)
    tok = (_zipf_sample(rng, cdf, (n, L)) + 1).astype(np.int32)
    tok[np.arange(L)[None, :] >= length[:, None]] = 0
    tok[0] = 0
    vert = rng.integers(1, 16, n).astype(np.int32)
    subvert = rng.integers(1, 307, n).astype(np.int32)
    vert[0] = 0
    subvert[0] = 0
    return tok, vert, subvert


def make_batches(shape, n_batches, seed=1236, B=None, full_history=False):
    """Pre-tensorised int32 batches: user (B,), hist_doc (B,W) left-padded with 0,
    cand_doc (B,1+K) positive first.  Returns a list of dicts plus the realised
    fraction of left-padded history slots.  full_history: every user has W clicks (no padding at all)."""
    rng = np.random.default_rng(seed)
    B = B or shape.B
    W, K = shape.W, shape.K
    cdf = _zipf_cdf(shape.n_news, 1.05)
    out, pad = [], 0
    for _ in range(n_batches):
        user = rng.integers(0, shape.n_users, B).astype(np.int32)
        h = np.clip(rng.geometric(1.0 / (0.6 * W), B), 1, 3 * W)
        h = np.minimum(h, W)
        if full_history:
            h[:] = W
        hist = (_zipf_sample(rng, cdf, (B, W)) + 1).astype(np.int32)
        hist[np.arange(W)[None, :] < (W - h)[:, None]] = 0          # left padding
        cand = (_zipf_sample(rng, cdf, (B, 1 + K)) + 1).astype(np.int32)
        pad += int((hist == 0).sum())
        out.append(dict(user=user, hist_doc=hist, cand_doc=cand))
    return out, pad / float(n_batches * B * W)


def _glorot(rng, shape, fan_in, fan_out):
    lim = np.sqrt(6.0 / (fan_in + fan_out))
    return rng.uniform(-lim, lim, shape).astype(np.float32)


def _orthogonal(rng, rows, cols):
    a = rng.standard_normal((rows, cols))
    u, _, vt = np.linalg.svd(a, full_matrices=False)
    q = u if u.shape == (rows, cols) else vt
    return q.astype(np.float32)


def make_weights(shape, arch=None, seed=1237, word_emb=None, score_model='dot', cook=False,
                 dv=15, ds=35, bias_noise=0.0, paper_vert=0, vertsup=None, vertalt=0, keras_orthogonal=False):
    """Keras-initialised parameter dict (names: oracle/lstur_numpy.py docstring).

    bias_noise > 0 replaces the all-zero bias initialisers by small normals so
    parity tests exercise the bias paths.  keras_orthogonal: draw the recurrent kernels as ONE (G, 3G) / (G, 4G)
    orthogonal matrix (orthonormal rows), as keras.initializers.Orthogonal does for the GRU / LSTM recurrent_kernel; the
    default (one orthogonal G x G block per gate) is what the committed golden fixtures were generated with."""
    arch = arch or shape.arch
    rng = np.random.default_rng(seed)
    E, F, k, U = shape.E, shape.F, shape.k, shape.U
    bz = lambda n: (rng.standard_normal(n) * bias_noise).astype(np.float32)
    P = {}
    P['word_emb'] = make_vocab(shape.vocab, E) if word_emb is None else word_emb
    P['conv_w'] = _glorot(rng, (k, E, F), k * E, k * F)
    P['conv_b'] = bz(F)
    P['att_w'] = _glorot(rng, (F,), F, 1)
    P['att_b'] = bz(1)
    if cook:
        D = F + dv + ds
        P['vert_emb'] = rng.uniform(-0.05, 0.05, (16, dv)).astype(np.float32)
        P['subvert_emb'] = rng.uniform(-0.05, 0.05, (307, ds)).astype(np.float32)
    else:
        D = U
        P['dense_w'] = _glorot(rng, (F, U), F, U)
        P['dense_b'] = bz(U)
        if paper_vert:      # Seq2VecPaperSoftmaxDaysIdVert (task/paper.py:1205-1232): [Dense(U)(title) ‖ Vemb[vertical]], and
            D = U + paper_vert          # the user encoder is built with user_embedding_dim + vertical_embedding_dim
            P['vert_emb'] = rng.uniform(-0.05, 0.05, (16, paper_vert)).astype(np.float32)
            U = U + paper_vert
    Hs = shape.U        # scorer hidden width = config.user_embedding_dim: score_encoder runs outside the temporary
                        # user_embedding_dim += vertical_embedding_dim of ...DaysIdVert.get_user_encoder (task/paper.py:1204-1208)
    G = U // 2 if arch == 'hgru' else U
    Ue = U // 2 if arch == 'hgru' else U
    if arch not in ('nigru', 'niavg', 'att'):
        P['user_emb'] = rng.uniform(-0.05, 0.05, (shape.n_users, Ue)).astype(np.float32)
    if arch not in ('vo', 'niavg', 'iavg', 'att', 'iatt', 'ilstm'):
        P['gru_wx'] = _glorot(rng, (D, 3 * G), D, 3 * G)
        P['gru_wh'] = _orthogonal(rng, G, 3 * G) if keras_orthogonal else np.concatenate([_orthogonal(rng, G, G) for _ in range(3)], 1)
        P['gru_b'] = bz(3 * G)
    if arch == 'ilstm':                                         # keras LSTM (task/cook.py:161-163), unit_forget_bias
        P['lstm_wx'] = _glorot(rng, (D, 4 * G), D, 4 * G)
        P['lstm_wh'] = _orthogonal(rng, G, 4 * G) if keras_orthogonal else np.concatenate([_orthogonal(rng, G, G) for _ in range(4)], 1)
        P['lstm_b'] = bz(4 * G)
        P['lstm_b'][G:2 * G] += 1.0
    if arch in ('att', 'iatt', 'atgru'):                        # SimpleAttentionMaskSupport kernel (Da, 1) + bias (models.py:456-468)
        Da = 1 if arch == 'atgru' else D           # atgru pools 2U one-feature steps: kernel (1, 1) (task/cook.py:184-190)
        P['uatt_w'] = _glorot(rng, (Da,), Da, 1)
        P['uatt_b'] = bz(1)
    if arch == 'algru':                                         # models.AlphaAdd: Constant(0.5) (models.py:541-545)
        P['alpha'] = (np.float32(0.5) + bz(1)).astype(np.float32)
    if arch in ('gru', 'iigru'):
        P['con_w'] = _glorot(rng, (G + Ue, U), G + Ue, U)
        P['con_b'] = bz(U)
    if arch in ('iigru', 'iicat', 'inagru'):                    # second user table, task/paper.py:616 / :340, task/cook.py:178
        P['user_emb2'] = rng.uniform(-0.05, 0.05, (shape.n_users, Ue)).astype(np.float32)
    if score_model == 'dnn':                                   # task/paper.py:448-451
        Du = 2 * U if arch in ('ngru', 'dgru', 'iicat', 'ilstm') else (D if arch in ('niavg', 'att') else (D + U if arch in ('iavg', 'iatt') else (1 if arch == 'atgru' else U)))
        P['sh_w'] = _glorot(rng, (Du + D, Hs), Du + D, Hs)
        P['sh_b'] = bz(Hs)
        P['so_w'] = _glorot(rng, (Hs, 1), Hs, 1)
        P['so_b'] = bz(1)
    if score_model == 'ddot':
        Du = 2 * U if arch in ('ngru', 'dgru', 'iicat', 'ilstm') else (D if arch in ('niavg', 'att') else (D + U if arch in ('iavg', 'iatt') else (1 if arch == 'atgru' else U)))
        P['su_w'] = _glorot(rng, (Du, Hs), Du, Hs)
        P['su_b'] = bz(Hs)
        P['sd_w'] = _glorot(rng, (D, Hs), D, Hs)
        P['sd_b'] = bz(Hs)
    if vertsup:      # (n_vert, hidden_dim): vertical classifier of ...VertSup, task/paper.py:948-952
        nv, hd = vertsup
        P['vs_w1'] = _glorot(rng, (D, hd), D, hd)
        P['vs_b1'] = bz(hd)
        P['vs_w2'] = _glorot(rng, (hd, nv), hd, nv)
        P['vs_b2'] = bz(nv)
    if vertalt:      # n_vert: Dense(len(self.verticals), softmax) of ...VertAlt's vertical model, task/paper.py:1131
        P['vcls_w'] = _glorot(rng, (D, vertalt), D, vertalt)
        P['vcls_b'] = bz(vertalt)
    return P


# ---- TSV writers in the reference's on-disk formats (README.md:7-23) -------------------------
def write_vocab_tsv(path, emb):
    """Vocab.tsv rows ``…\\t<index>\\t<space-separated floats>`` (utils.py:37-41); index 0 omitted."""
    with open(path, 'w') as f:
        for i in range(1, emb.shape[0]):
            f.write('w%d\t%d\t%s\n' % (i, i, ' '.join(repr(float(x)) for x in emb[i])))


def write_docmeta_tsv(path, tok, vert=None, subvert=None):
    """DocMeta.tsv: col1 = doc id, col4 = title tokens, col5 = body tokens (task/seq2vec.py:96-101);
    cols 2,3 carry vertical / subvertical names in the DaysId variants (task/paper.py:803-820)."""
    with open(path, 'w') as f:
        for i in range(1, tok.shape[0]):
            t = ' '.join(str(int(x)) for x in tok[i] if x != 0)
            from .utils import VERTICAL_NAMES
            f.write('d%d\t%d\t%s\ts%d\t%s\t%s\n' % (i, i, VERTICAL_NAMES[0 if vert is None else int(vert[i])],
                                                      0 if subvert is None else subvert[i], t, t))


def write_clickdata_tsv(path, n_users, n_news, rng, max_imp=4, n_neg=8):
    """ClickData.tsv: column 2 = training impressions, column 3 = validation impressions, each
    ``pos#TAB#neg#TAB#time`` joined by ``#N#`` (task/paper.py:7-35)."""
    cdf = _zipf_cdf(n_news, 1.05)

    def distinct(k):
        """k different documents (Zipf draws, first occurrences): the candidates of one impression.  A document listed
        twice gets two identical scores, and the order numpy's argsort leaves ties in — which utils.mrr_score / ndcg_score
        depend on (utils.py:106-124) — changed between numpy releases (stable insertion sort for short arrays in 1.x, SIMD
        sorts in 2.x), so impressions with repeated documents have no well-defined reference value."""
        out = []
        while len(out) < k:
            for d in _zipf_sample(rng, cdf, 2 * k) + 1:
                if d not in out:
                    out.append(int(d))
                    if len(out) == k:
                        break
        return out

    def imps(k):
        out = []
        for i in range(k):
            n_pos = int(rng.integers(1, 3))
            docs = distinct(n_pos + n_neg)
            pos, neg = docs[:n_pos], docs[n_pos:]
            out.append('%s#TAB#%s#TAB#01/%02d/2019 %02d:%02d:00 PM' % (' '.join(map(str, pos)), ' '.join(map(str, neg)),
                                                                    1 + i % 28, 1 + i % 12, i % 60))
        return '#N#'.join(out)
    with open(path, 'w') as f:
        for u in range(n_users):
            f.write('u%d\tx\t%s\t%s\n' % (u, imps(rng.integers(1, max_imp + 1)), imps(rng.integers(0, 3))))


def write_dataset(dirname, shape, seed=7):
    """Small on-disk dataset in the reference formats: Vocab.tsv(.npy), DocMeta.tsv, ClickData.tsv."""
    import os
    rng = np.random.default_rng(seed)
    os.makedirs(dirname, exist_ok=True)
    emb = make_vocab(shape.vocab, shape.E, seed)
    tok, vert, subvert = make_docs(shape.n_news, shape.L, shape.vocab, seed + 1)
    write_vocab_tsv(os.path.join(dirname, 'Vocab.tsv'), emb)
    np.save(os.path.join(dirname, 'Vocab.tsv.npy'), emb)
    write_docmeta_tsv(os.path.join(dirname, 'DocMeta.tsv'), tok, vert, subvert)
    write_clickdata_tsv(os.path.join(dirname, 'ClickData.tsv'), shape.n_users, shape.n_news, rng)
    return emb, tok


def write_pipeline_files(dirname, tok, W, n_docs=40, n_users=11, seed=3):
    """docs.tsv / UserClick.tsv / userDocPair.tsv of the decomposed scoring pipeline (settings.py pipeline_inputs,
    task/test_pipeline.py:18-24, 72-79, 152-160): `doc \\t title tokens`, `user id \\t user type \\t clicks joined by #N#`,
    `user id \\t user type \\t doc`.  One user clicks a document that is not in docs.tsv (stays a zero vector), one pair names
    an unknown user (skipped)."""
    import os
    g = np.random.default_rng(seed)
    os.makedirs(dirname, exist_ok=True)
    docs = list(range(1, min(n_docs, tok.shape[0] - 1) + 1))
    with open(os.path.join(dirname, 'docs.tsv'), 'w') as f:
        for d in docs:
            toks = [int(x) for x in tok[d] if x != 0] or [1]
            f.write('d%d\t%s\n' % (d, ' '.join(map(str, toks))))
    with open(os.path.join(dirname, 'UserClick.tsv'), 'w') as f:
        for u in range(n_users):
            clicks = ['d%d' % docs[i] for i in g.integers(0, len(docs), g.integers(1, W + 3))]
            if u == 3:
                clicks.append('d_unknown')
            f.write('%d\tx\t%s\n' % (u, '#N#'.join(clicks)))
    with open(os.path.join(dirname, 'userDocPair.tsv'), 'w') as f:
        for u in range(n_users):
            for d in g.integers(0, len(docs), 3):
                f.write('%d\tx\td%d\n' % (u, docs[d]))
        f.write('999\tx\td%d\n' % docs[0])


def write_cook_npz(dirname, shape, n_train=24, n_test=30, seed=0, days=30):
    """train / test .npz in the reference's cook layout (task/cook.py:14-28, settings.py train_npz_input / test_npz_input)
    + Vocab.tsv.npy: idx, idx_mask (n,1); ch_title (n,W,L), ch_vert, ch_subvert (n,W); cd_title (n,5,L), cd_vert, cd_subvert
    (n,5), cd_label (n,5) — the test file carries one candidate per row plus label / user / impr."""
    import os
    g = np.random.default_rng(seed)
    tok, _, _ = make_docs(shape.n_news, shape.L, shape.vocab)

    def block(n, C):
        hd = g.integers(0, shape.n_news + 1, (n, shape.W))
        hd[:, :2] = 0                                            # left padding
        cd = g.integers(1, shape.n_news + 1, (n, C))
        return dict(idx=g.integers(0, 50, (n, 1)), idx_mask=(g.random((n, 1)) < 0.8).astype(np.float32),
                    ch_title=tok[hd], ch_vert=g.integers(0, 16, (n, shape.W)) * (hd > 0),
                    ch_subvert=g.integers(0, 307, (n, shape.W)) * (hd > 0),
                    cd_title=tok[cd], cd_vert=g.integers(1, 16, (n, C)), cd_subvert=g.integers(1, 307, (n, C)))
    tr = block(n_train, 5)
    tr['cd_label'] = np.eye(5, dtype=np.float32)[np.zeros(n_train, dtype=int)]
    te = block(n_test, 1)
    # rows grouped by (user, impression) as the evaluation tail of `main.py cook` expects (main.py:250-286): users of
    # `per_user` consecutive impressions of `per_imp` rows, one click per impression, in-vocabulary flag per user
    per_imp, per_user = 3, 2
    imp = np.arange(n_test) // per_imp
    user = imp // per_user
    label = np.zeros(n_test, dtype=np.float32)
    for i in range(int(imp.max()) + 1):
        rows = np.where(imp == i)[0]
        label[rows[g.integers(0, len(rows))]] = 1.0
    iv = (g.random(int(user.max()) + 1) < 0.6).astype(np.float32)
    iv[:2] = [1.0, 0.0]
    te = dict(te, cd_title=te['cd_title'][:, 0], cd_vert=te['cd_vert'][:, 0], cd_subvert=te['cd_subvert'][:, 0],
              label=label, user=user, impr=imp, idx_mask=iv[user].reshape(n_test, 1), idx=(user % 50).reshape(n_test, 1))
    os.makedirs(dirname, exist_ok=True)
    np.savez(os.path.join(dirname, 'train_%ddays_%dwindow.npz' % (days, shape.W)), **tr)
    np.savez(os.path.join(dirname, 'test_%ddays_%dwindow.npz' % (days, shape.W)), **te)
    np.save(os.path.join(dirname, 'Vocab.tsv.npy'), make_vocab(shape.vocab, shape.E))


def write_cook_npz_shared(dirname, shape, n_train=23, n_impr=10, long_impr=40, seed=0, days=30):
    """Cook .npz files (write_cook_npz's layout) whose test file is laid out as the reference's data is: every candidate
    row of an impression repeats the impression's user, idx_mask and history.  Impressions have 2..8 candidates, one has
    `long_impr`; users have one or two impressions; about a third of the users are out of vocabulary (idx_mask 0, in the
    training file too); the title of document 0 (all zero) is a candidate in both files; titles recur across rows with
    other verticals: a slot carries its document's vertical and subvertical, one slot in ten other ones.  n_train is
    meant not to divide the batch size (a ragged last batch)."""
    import os
    g = np.random.default_rng(seed)
    tok, dvert, dsub = make_docs(shape.n_news, shape.L, shape.vocab)

    def verts(docs, lo):
        other = g.random(docs.shape) < 0.1
        v = np.where(other, g.integers(lo, 16, docs.shape), dvert[docs])
        s = np.where(other, g.integers(lo, 307, docs.shape), dsub[docs])
        return v * (docs > 0), s * (docs > 0)

    def hist(n):
        hd = g.integers(0, shape.n_news + 1, (n, shape.W))
        hd[:, :2] = 0
        return hd
    hd, cd = hist(n_train), g.integers(1, shape.n_news + 1, (n_train, 5))
    cd[0, 2] = 0
    (hv, hs), (cv, cs) = verts(hd, 0), verts(cd, 1)
    tr = dict(idx=g.integers(0, 50, (n_train, 1)), idx_mask=(g.random((n_train, 1)) < 0.7).astype(np.float32),
              ch_title=tok[hd], ch_vert=hv, ch_subvert=hs, cd_title=tok[cd], cd_vert=cv, cd_subvert=cs,
              cd_label=np.eye(5, dtype=np.float32)[np.zeros(n_train, dtype=int)])
    sizes = g.integers(2, 9, n_impr)
    sizes[n_impr // 2] = long_impr
    imp = np.repeat(np.arange(n_impr), sizes)
    h = n_impr // 2
    u_of = np.where(np.arange(n_impr) < h, np.arange(n_impr) // 2, np.arange(n_impr) - h + (h + 1) // 2)
    user = u_of[imp]                                      # users of two impressions, then users of one
    n = len(imp)
    iv = (g.random(int(user.max()) + 1) < 0.65).astype(np.float32)
    iv[:2] = [1.0, 0.0]
    hi = hist(n_impr)[imp]
    cdt = g.integers(1, shape.n_news + 1, n)
    cdt[np.cumsum(sizes)[:3] - 1] = 0                     # the all-zero title as a candidate
    label = np.zeros(n, dtype=np.float32)
    label[np.cumsum(sizes) - sizes + g.integers(0, sizes)] = 1.0
    hv, hs = (a[imp] for a in verts(hi[np.cumsum(sizes) - sizes], 0))
    cv, cs = verts(cdt, 1)
    te = dict(idx=(user % 50).reshape(n, 1), idx_mask=iv[user].reshape(n, 1), ch_title=tok[hi], ch_vert=hv, ch_subvert=hs,
              cd_title=tok[cdt], cd_vert=cv, cd_subvert=cs, label=label, user=user, impr=imp)
    os.makedirs(dirname, exist_ok=True)
    np.savez(os.path.join(dirname, 'train_%ddays_%dwindow.npz' % (days, shape.W)), **tr)
    np.savez(os.path.join(dirname, 'test_%ddays_%dwindow.npz' % (days, shape.W)), **te)
    np.save(os.path.join(dirname, 'Vocab.tsv.npy'), make_vocab(shape.vocab, shape.E))


# ---- a LEARNABLE synthetic click task (training-parity / AUC checks; BASELINE.json north_star: "AUC within 0.002 after
# a fixed step count").  make_batches() above draws positives at random, so nothing can be learnt from it; here every
# document carries a latent topic visible in its title tokens and every user prefers one topic, so a model that reads
# titles and user ids ranks the positive above random negatives after a few hundred steps. -----------------------------
def make_preference_task(shape, n_train, n_eval, seed=4321, n_topics=8, p_topic_token=0.8, p_pref=0.85):
    """-> tok (n_news+1, L), word_emb (V, E), train batches, eval batches (lists of dicts user / hist_doc / cand_doc,
    positive first).  The (frozen) word vectors of a topic's vocabulary slice share a centroid — as pre-trained
    vectors of related words do — so the topic is visible to the title encoder."""
    rng = np.random.default_rng(seed)
    n, L, V, W, K, B = shape.n_news + 1, shape.L, shape.vocab, shape.W, shape.K, shape.B
    topic = rng.integers(0, n_topics, n)
    length = np.clip(np.rint(rng.normal(0.6 * L, 0.2 * L, n)), min(3, L), L).astype(np.int64)
    span = (V - 1) // n_topics
    in_topic = rng.random((n, L)) < p_topic_token
    tok = np.where(in_topic, 1 + topic[:, None] * span + rng.integers(0, span, (n, L)), rng.integers(1, V, (n, L))).astype(np.int32)
    tok[np.arange(L)[None, :] >= length[:, None]] = 0
    tok[0] = 0
    by_topic = [np.where(topic[1:] == z)[0] + 1 for z in range(n_topics)]
    centroid = rng.standard_normal((n_topics, shape.E))
    word_topic = np.minimum((np.arange(V) - 1) // span, n_topics - 1)
    word_emb = (0.1 * (0.7 * centroid[word_topic] + 0.7 * rng.standard_normal((V, shape.E)))).astype(np.float32)
    word_emb[0] = 0.0
    pref = rng.integers(0, n_topics, shape.n_users)

    def draw(users, size):
        """documents for `users` (len m) -> (m, size): the preferred topic with probability p_pref, else any document"""
        m = len(users)
        out = rng.integers(1, n, (m, size))
        take = rng.random((m, size)) < p_pref
        for i, u in enumerate(users):
            pool = by_topic[pref[u]]
            k = int(take[i].sum())
            if k and len(pool):
                out[i, take[i]] = pool[rng.integers(0, len(pool), k)]
        return out

    def batch():
        user = rng.integers(0, shape.n_users, B).astype(np.int32)
        h = np.minimum(np.clip(rng.geometric(1.0 / (0.6 * W), B), 1, 3 * W), W)
        hist = draw(user, W).astype(np.int32)
        hist[np.arange(W)[None, :] < (W - h)[:, None]] = 0
        pos = draw(user, 1)
        neg = rng.integers(1, n, (B, K))
        return dict(user=user, hist_doc=hist, cand_doc=np.concatenate([pos, neg], 1).astype(np.int32))

    return tok, word_emb, [batch() for _ in range(n_train)], [batch() for _ in range(n_eval)]


def impression_auc(scores):
    """Mean per-impression AUC (task/paper.py:504-515 with sklearn's roc_auc_score): scores (n, 1+K), positive first;
    ties count one half."""
    s = np.asarray(scores, dtype=np.float64)
    pos, neg = s[:, :1], s[:, 1:]
    return float(((pos > neg) + 0.5 * (pos == neg)).mean(1).mean())
