"""Cook on its .npz rows interned on the GPU (mnexp_b200/intern.py, csrc/intern.cu): the interning contract against a
numpy statement of it, the sample gather against numpy indexing, the epoch draws against the host loop's (CPU),
device fit against host fit (bit for bit), device scoring and aggregation against the host path, and `main.cook` with
both device switches against the reference's logged records."""
import os
import sys
import tempfile
import types

import numpy as np
import pytest
import torch

from mnexp_b200 import evaluation, settings, synth, task
from mnexp_b200.engine import COOK_ARCH
from mnexp_b200.task import cook as mcook
from tolerances import elem_excess, rel

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, 'golden'))
import make_ref_golden as mk          # noqa: E402


# ---------------------------------------------------------------------------------------------- epoch draws (CPU)
@pytest.mark.parametrize('arch', ['ingru', 'inigru', 'inagru'])
def test_epoch_scales_match_the_host_loop_draws(arch):
    """epoch_scales draws what CookModel.fit's host loop draws batch by batch (the ragged tail padded with its first
    row), bit for bit, and leaves numpy's stream where the loop leaves it"""
    n, B, C, keep = 23, 10, 5, 0.8
    g = np.random.default_rng(3)
    mask = (g.random((n, 1)) < 0.7).astype(np.float32)
    owner = types.SimpleNamespace(config=types.SimpleNamespace(id_keep=keep, arch=arch), dv=0, ds=0)
    model = mcook.CookModel(owner, True)
    x = [np.arange(n).reshape(n, 1), mask, np.zeros((n, 2, 3)), np.zeros((n, 2)), np.zeros((n, 2)), np.zeros((n, C, 3)),
         np.zeros((n, C)), np.zeros((n, C))]
    two = arch in ('inigru', 'inagru')
    np.random.seed(77)
    ref = []
    for _ in range(2):
        order = np.random.permutation(n)
        for s in range(0, n, B):
            rows = order[s:s + B]
            if len(rows) < B:
                rows = np.concatenate([rows, np.full(B - len(rows), rows[0])])
            b = model._batch(x, rows, C, True)
            ref.append((b['user_scale'], b.get('user_scale2'), b['user']))
    after = np.random.random()
    np.random.seed(77)
    got = []
    for _ in range(2):
        order = np.random.permutation(n)
        s1, s2 = mcook.epoch_scales(mask, order, B, keep, two)
        assert s1.dtype == np.float32 and s1.shape == (30,)
        got += [(s1[i:i + B], None if s2 is None else s2[i:i + B]) for i in range(0, 30, B)]
    assert np.random.random() == after
    assert len(got) == len(ref)
    for (a1, a2, _), (b1, b2) in zip(ref, got):
        assert np.array_equal(a1.view(np.uint32), b1.view(np.uint32))
        assert (a2 is None) == (b2 is None) == (not two)
        if two:
            assert np.array_equal(a2.view(np.uint32), b2.view(np.uint32))
    assert any((a[0] == 0).any() and (a[0] > 1).any() for a in ref)       # draws did drop and rescale


def test_epoch_scales_without_id_dropout_draw_nothing():
    np.random.seed(5)
    mask = np.array([[1.0], [0.0], [1.0]], dtype=np.float32)
    s1, s2 = mcook.epoch_scales(mask, np.array([2, 0, 1]), 2, 1.0, True)
    assert s1.tolist() == [1.0, 1.0, 0.0, 0.0] and s2.tolist() == s1.tolist()
    after = np.random.random()
    np.random.seed(5)
    assert np.random.random() == after


# ---------------------------------------------------------------------------------------------- interning (GPU)
def ref_intern(tok, vert, subvert):
    """the contract in numpy: np.unique over the K columns, non-zero keys renumbered from 1 by first occurrence, the zero
    key 0; the table holds every key once, row 0 zero"""
    n, L = tok.shape
    keys = np.concatenate([tok.astype(np.int64), (np.zeros(n) if vert is None else vert).reshape(n, 1),
                           (np.zeros(n) if subvert is None else subvert).reshape(n, 1)], 1).astype(np.int64)
    if n == 0:
        return np.zeros(0, np.int64), np.zeros((1, L + 2), np.int64)
    u, first, inv = np.unique(keys, axis=0, return_index=True, return_inverse=True)
    nz = np.any(u != 0, axis=1)
    nzi = np.nonzero(nz)[0]
    by_first = nzi[np.argsort(first[nzi], kind='stable')]
    rank = np.zeros(len(u), np.int64)
    rank[by_first] = 1 + np.arange(len(by_first))
    table = np.zeros((1 + len(by_first), L + 2), np.int64)
    table[1:] = u[by_first]
    return rank[inv.reshape(-1)], table


def _cases():
    g = np.random.default_rng(11)
    L = 6
    out = {}
    base = g.integers(1, 50, (1, L))
    t = np.repeat(base, 40, 0)
    t[:, -1] = g.integers(0, 4, 40)
    out['last_token'] = (t, np.ones(40, np.int64), np.ones(40, np.int64))
    t = np.repeat(base, 40, 0)
    out['vertical'] = (t, g.integers(0, 5, 40), np.full(40, 3))
    out['subvertical'] = (t, np.full(40, 2), g.integers(0, 5, 40))
    pool = g.integers(0, 2 ** 31, (60, L + 2))
    pool[0] = 2 ** 31 - 1
    pool[1, :L] = 0
    pool[1, L:] = [1 << 30, 0]
    pool[2] = 0
    pick = g.integers(0, 60, 3000)
    out['values_to_2^31-1'] = (pool[pick, :L], pool[pick, L], pool[pick, L + 1])
    neg = pool.copy()
    neg[3:30:2] = -neg[3:30:2] - 1
    out['negative_values'] = (neg[pick, :L], neg[pick, L], neg[pick, L + 1])
    out['n=0'] = (np.zeros((0, L), np.int64), np.zeros(0, np.int64), np.zeros(0, np.int64))
    out['n=1'] = (base, np.array([4]), np.array([5]))
    out['n=1_zero'] = (np.zeros((1, L), np.int64), np.zeros(1, np.int64), np.zeros(1, np.int64))
    out['all_equal'] = (np.repeat(base, 5000, 0), np.full(5000, 7), np.full(5000, 8))
    d = np.arange(5000)
    out['all_distinct'] = (np.stack([d % 7, d // 7, d % 13, d, d * 3, 5 * np.ones_like(d)], 1), d % 3, d % 11)
    t = g.integers(0, 9, (20000, L))
    t[:, 2:] = 0                                            # many repeats, many zero rows
    out['repeats_and_zero_rows'] = (t, g.integers(0, 2, 20000) * (t[:, 0] > 0), None)
    out['tokens_only'] = (t[:500], None, None)
    return out


CASES = _cases()


def _intern_parts(parts, L):
    from mnexp_b200 import intern
    ids, table = intern.intern(parts, L)
    return np.concatenate([i.cpu().numpy().reshape(-1) for i in ids]) if ids else np.zeros(0), \
        {k: None if v is None else v.cpu().numpy() for k, v in table.items()}


@pytest.mark.gpu
@pytest.mark.parametrize('case', sorted(CASES))
def test_intern_matches_the_numpy_contract(lib, case):
    tok, v, s = CASES[case]
    n, L = tok.shape
    ref_ids, ref_table = ref_intern(tok, v, s)
    ids, table = _intern_parts([(tok, v, s)], L)
    assert np.array_equal(ids, ref_ids)
    assert np.array_equal(table['doc_tokens'], ref_table[:, :L])
    for k, col, a in (('doc_vert', L, v), ('doc_subvert', L + 1, s)):
        assert (table[k] is None) == (a is None)
        if a is not None:
            assert np.array_equal(table[k], ref_table[:, col])
    assert np.array_equal(table['doc_tokens'][ids], tok)          # every row reproduced, raw values kept
    # the same result from a second run and from another cut of the upload into parts
    ids2, table2 = _intern_parts([(tok, v, s)], L)
    cut = sorted({0, n // 3, n // 2 + 1, n})
    parts = [(tok[a:b], None if v is None else v[a:b], None if s is None else s[a:b]) for a, b in zip(cut[:-1], cut[1:])]
    ids3, table3 = _intern_parts(parts, L)
    for i, t in ((ids2, table2), (ids3, table3)):
        assert np.array_equal(i, ids)
        assert all((table[k] is None and t[k] is None) or np.array_equal(table[k], t[k]) for k in table)


# ---------------------------------------------------------------------------------------------- sample gather (GPU)
@pytest.mark.gpu
@pytest.mark.parametrize('m', [8, 5, 1])
def test_gather_samples_matches_numpy_indexing(lib, m):
    import ctypes
    g = np.random.default_rng(m)
    n, B, W, C = 17, 8, 4, 3
    tabs = dict(user=g.integers(0, 99, n).astype(np.int32), scale=g.random(n).astype(np.float32),
                hist=g.integers(0, 50, (n, W)).astype(np.int32), cand=g.integers(0, 50, (n, C)).astype(np.int32),
                label=g.random((n, C)).astype(np.float32))
    pos = g.permutation(n)[:B].astype(np.int32)
    dev = {k: torch.as_tensor(v).cuda() for k, v in tabs.items()}
    out = dict(user=torch.full((B,), -7, dtype=torch.int32), scale=torch.full((B,), -7.0), hist=torch.full((B, W), -7, dtype=torch.int32),
               cand=torch.full((B, C), -7, dtype=torch.int32), label=torch.full((B, C), -7.0))
    out = {k: v.cuda() for k, v in out.items()}
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    rc = lib.lstur_gather_samples(B, m, W, C, p(torch.as_tensor(pos).cuda()), p(dev['user']), p(dev['scale']), p(dev['hist']),
                                  p(dev['cand']), p(dev['label']), p(out['user']), p(out['scale']), p(out['hist']),
                                  p(out['cand']), p(out['label']), None)
    assert rc == 0
    torch.cuda.synchronize()
    rows = np.where(np.arange(B) < m, pos, pos[0])
    for k in ('user', 'scale', 'hist', 'cand'):
        assert np.array_equal(out[k].cpu().numpy(), tabs[k][rows]), k
    lab = tabs['label'][rows]
    lab[m:] = 0
    assert np.array_equal(out['label'].cpu().numpy(), lab)


# ---------------------------------------------------------------------------------------------- Cook handlers
def _handler(d, arch, score_model, precision, **kw):
    sh = mk.cook_shape(score_model, 'vs')
    c = dict(task='Cook', arch=arch, input_training_data_path=d, days=30, window_size=sh.W, batch_size=10,
             title_filter_shape=(sh.F, 3), user_embedding_dim=sh.U, dropout=0.0, score_model=score_model,
             use_vertical=True, use_vertical_type='vs', vertical_embedding_dim=mk.COOK_DV,
             subvertical_embedding_dim=mk.COOK_DS, precision=precision, validation_step=30, lrd_on_epochs=[0],
             learning_rate=0.001, id_keep=1.0)
    c.update(kw)
    return task.get(settings.Config(c))


_DATA = {}


def _dataset(kind, score_model):
    key = (kind, score_model)
    if key not in _DATA:
        d = tempfile.mkdtemp()
        (synth.write_cook_npz_shared if kind == 'shared' else synth.write_cook_npz)(d, mk.cook_shape(score_model, 'vs'))
        _DATA[key] = d
    return _DATA[key]


@pytest.mark.gpu
@pytest.mark.parametrize('precision', ['fp32', 'fp16_tc'])
@pytest.mark.parametrize('arch', ['ingru', 'inigru', 'ilstm'])
def test_device_fit_is_bit_identical_to_host_fit(lib, arch, precision, monkeypatch):
    """two epochs of fit from the same weights and numpy seed (id_keep 0.8, dropout, a ragged last batch of 3): the
    weights and the History values are identical, and the step loop never waits for the device"""
    d = _dataset('shared', 'ddot')

    def run(device):
        np.random.seed(2024)
        h = _handler(d, arch, 'ddot', precision, id_keep=0.8, dropout=0.2)
        model = h.build_model(0)
        x, y = h.device_train() if device else h.train()
        hist = model.fit(x, y, 10, epochs=2, initial_epoch=0, shuffle=True)
        torch.cuda.synchronize()
        return hist.history, h.current_params()

    orig = mcook.CookModel._device_steps
    calls = []

    def no_sync(*a):
        torch.cuda.set_sync_debug_mode('error')
        try:
            out = orig(*a)
        finally:
            torch.cuda.set_sync_debug_mode(0)
        calls.append(1)
        return out
    monkeypatch.setattr(mcook.CookModel, '_device_steps', staticmethod(no_sync))
    h_host, w_host = run(False)
    h_dev, w_dev = run(True)
    assert len(calls) == 2
    assert h_dev == h_host
    assert sorted(w_dev) == sorted(w_host)
    for k in w_host:
        assert np.array_equal(w_dev[k], w_host[k]), k


def _check_results(got, ref, tol=1e-6):
    for k in ('user', 'impr', 'iv_user', 'oov_user'):
        for f in ('auc', 'mrr', 'ndcgv', 'ndcgx', 'pos', 'size', 'idx'):
            a, b = getattr(got[k], f), getattr(ref[k], f)
            assert (np.isnan(a) and np.isnan(b)) or abs(a - b) <= tol, (k, f, a, b)


def _score_case(lib, arch, score_model, precision, kind):
    d = _dataset(kind, score_model)
    np.random.seed(7)
    h = _handler(d, arch, score_model, precision)
    h.build_model(0)
    h.predict_rows = 4          # plans of 4 rows: the long impression is split over several chunks
    tx, _ = h.test()
    host = h.test_model.predict(tx).reshape(-1)
    xd, _ = h.device_test()
    got = h.test_model.predict(xd).reshape(-1)
    tol = 2e-5 if precision == 'fp32' else 1e-3
    assert got.shape == host.shape
    assert rel(got, host) < tol and elem_excess(got, host, tol) <= 1.0, (rel(got, host), elem_excess(got, host, tol))
    return h, got


# 'dot' multiplies the user vector with the news vector (task/cook.py:200-201): only the archs whose user vector has the
# news vector's width build with it, in the reference as here
NO_DOT = ('igru', 'inigru', 'iavg', 'iatt', 'atgru', 'ilstm')
SCORED = [(a, s) for a in sorted(COOK_ARCH) for s in ('dot', 'dnn', 'ddot') if not (s == 'dot' and a in NO_DOT)]


@pytest.mark.gpu
@pytest.mark.parametrize('kind', ['shared', 'npz'])
@pytest.mark.parametrize('arch,score_model', SCORED)
def test_device_predict_matches_host_predict_fp32(lib, arch, score_model, kind):
    _score_case(lib, arch, score_model, 'fp32', kind)


@pytest.mark.gpu
@pytest.mark.parametrize('score_model', ['dnn', 'ddot'])
@pytest.mark.parametrize('arch', ['ingru', 'inigru', 'ilstm', 'iatt', 'vo'])
def test_device_predict_matches_host_predict_fp16_tc(lib, arch, score_model):
    _score_case(lib, arch, score_model, 'fp16_tc', 'shared')


@pytest.mark.gpu
@pytest.mark.parametrize('arch,score_model', [('ingru', 'ddot'), ('inigru', 'dnn'), ('avg', 'dot')])
def test_device_evaluation_tail_matches_host_formulas(lib, arch, score_model):
    """aggregate_test(device=True) = evaluation.aggregate on the same device scores; evaluate on device_valid = evaluate
    on valid up to the scores' rounding; null user scales are the unscaled path bit for bit"""
    h, scores = _score_case(lib, arch, score_model, 'fp32', 'shared')
    users, imprs, mask, y = [h.test_data[k] for k in ('user', 'impr', 'idx_mask', 'label')]
    lines = []
    res = h.aggregate_test(device=True, log=lines.append)
    assert len(lines) == 8
    _check_results(res, evaluation.aggregate(users, imprs, mask.reshape(-1), y, scores))
    ref = h.test_model.evaluate(*h.valid())
    got = h.test_model.evaluate(*h.device_valid())
    assert abs(got[0] - ref[0]) <= 1e-4 * max(1.0, abs(ref[0])) and abs(got[1] - ref[1]) <= 0.02, (got, ref)
    # user_scale = None against all-ones multipliers
    x, _ = h.device_test()
    eng = h.engine(h.predict_rows, 1, training=False)
    n = x.n
    off = np.arange(n + 1, dtype=np.int32)
    table = eng.eval_doc_table()
    a = eng.score_impressions(x.user, x.hist_doc, off, x.cand_doc.reshape(-1), table)
    ones = torch.ones(n, dtype=torch.float32, device=eng.device)
    b = eng.score_impressions(x.user, x.hist_doc, off, x.cand_doc.reshape(-1), table, user_scale=ones, user_scale2=ones)
    assert torch.equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize('precision', ['fp32', 'fp16_tc'])
def test_device_main_cook_loop_matches_reference(lib, precision):
    """`main.py cook` with device batches and device evaluation on the setup of test_ref_pinned's cook loop: every
    logged record within that test's tolerances"""
    from mnexp_b200 import main as mmain
    from test_ref_pinned import GOLD, _compare_records, _records
    sh = mk.cook_shape('ddot', 'vs')
    d = tempfile.mkdtemp()
    synth.write_cook_npz(d, sh)
    cfg = settings.Config(dict(task='Cook', arch='ingru', input_training_data_path=d, days=30, window_size=sh.W,
                               batch_size=mk.MAIN_COOK_BATCH,
                               title_filter_shape=(sh.F, 3), user_embedding_dim=sh.U, dropout=0.0, score_model='ddot',
                               use_vertical=True, use_vertical_type='vs', vertical_embedding_dim=mk.COOK_DV,
                               subvertical_embedding_dim=mk.COOK_DS, precision=precision, validation_step=6, epochs=2,
                               lrd_on_epochs=[0], learning_rate=0.001, learning_rate_decay=0.2, id_keep=1.0,
                               sparse_user_adam=False))

    def on_build(h):
        P = {}
        for k, v in h.params.items():
            ref = np.asarray(GOLD['main-cook/P/' + k], dtype=np.float32)
            if k in ('user_emb', 'user_emb2'):
                full = np.zeros(np.asarray(v).shape, dtype=np.float32)
                full[:len(ref)] = ref
                ref = full
            P[k] = ref.reshape(np.asarray(v).shape)
        h.params = P
        np.random.seed(4711)
    np.random.seed(4710)
    h, got = mmain.cook(cfg, on_build=on_build, device_batches=True, device_eval=True)
    assert h._device_data is not None
    _compare_records(got, _records('main-cook'), 1e-4 if precision == 'fp32' else 2e-3, 1e-6 if precision == 'fp32' else 0.35)
