"""The epoch-end ranking of the softmax-family task handlers on the device (handler.device_test / device_callback,
lstur_score_impressions).

CPU: the evaluation tables of build_tables, read by a numpy statement of the history rule, give impression by impression
the user, history, candidates and labels that test_gen gives through the handler's own window hooks.
GPU: device_test scores equal the scores handler.test yields on the same weights; device_callback logs what callback
logs; main.train(device_eval=True) runs the loop with it.

The dataset adds, to the synthetic one, a document whose title is all zero tokens (clicked in histories and shown as a
candidate), an impression of more than 32 candidates, and a user whose validation history has fully expired in the
Days handlers (and is masked everywhere: its only training click is the all-zero title)."""
import os
import tempfile

import numpy as np
import pytest
import torch

from mnexp_b200 import assemble, metrics, settings, synth, task, utils

from tolerances import assert_close

SH = synth.Shape('deval', 60, 80, 120, L=7, W=5, K=2, B=6, E=12, F=16, U=8)
ZERO_DOC = 3           # its DocMeta title is "0": all zero tokens
_DATA = {}


def _imp(pos, neg, day, hour=1):
    return '%s#TAB#%s#TAB#01/%02d/2019 %02d:00:00 PM' % (' '.join(map(str, pos)), ' '.join(map(str, neg)), day, hour)


def _dataset():
    if 'dir' in _DATA:
        return _DATA['dir']
    d = tempfile.mkdtemp()
    synth.write_dataset(d, SH)
    path = os.path.join(d, 'DocMeta.tsv')
    lines = open(path).read().splitlines()
    cols = lines[ZERO_DOC - 1].split('\t')
    assert cols[1] == str(ZERO_DOC)
    cols[4] = cols[5] = '0'
    lines[ZERO_DOC - 1] = '\t'.join(cols)
    open(path, 'w').write('\n'.join(lines) + '\n')
    big = list(range(10, 44))                                        # with the all-zero title: 35 distinct candidates
    extra = [
        # only training click: the all-zero title (a history with no unmasked slot); > 32 candidates, the all-zero title
        # among them
        ('ux0', _imp([ZERO_DOC], [50, 51], 3), _imp([big[0], ZERO_DOC], big[1:], 3, 2)),
        # clicks long before the validation impressions: every slot has expired under days = 1 and 2
        ('ux1', _imp([60, 61], [62, 63], 1) + '#N#' + _imp([64], [65, 66], 1, 3), _imp([70], [71, 72, ZERO_DOC], 25)),
        # the all-zero title in the middle of a history
        ('ux2', _imp([44, ZERO_DOC, 45], [46, 47], 4) + '#N#' + _imp([48], [49, 52], 4, 5),
         _imp([53], [54, 55, 56], 5) + '#N#' + _imp([57, 58], [59, 67], 5, 3)),
    ]
    with open(os.path.join(d, 'ClickData.tsv'), 'a') as f:
        for name, tr, va in extra:
            f.write('%s\tx\t%s\t%s\n' % (name, tr, va))
    _DATA['dir'] = d
    return d


def _handler(task_name, days=30, arch='igru', **kw):
    cfg = dict(task=task_name, arch=arch, input_training_data_path=_dataset(), title_shape=SH.L, window_size=SH.W,
               negative_samples=SH.K, batch_size=4, textual_embedding_dim=SH.E, title_filter_shape=(SH.F, 3),
               user_embedding_dim=SH.U, debug=True, dropout=0.0, days=days, validation_impression=1000,
               testing_impression=7, epochs=2, training_step=3, validation_step=2)
    cfg.update(kw)
    return task.get(settings.Config(cfg))


def _history(T, W, expire):
    """numpy statement of the history rule: the W stream entries before the impression's first click, left-padded with
    doc 0; with times, a slot older than the impression by more than `expire` seconds reads as doc 0."""
    first = T['eval_first_click'].astype(np.int64)
    user = T['click_user'][first]
    j = first[:, None] - W + np.arange(W)
    ok = j >= T['stream_off'][user][:, None]
    hist = np.where(ok, T['stream_docs'][np.maximum(j, 0)], 0)
    if 'click_time' in T:
        t = T['click_time'].astype(np.int64)
        hist = np.where(ok & (t[np.maximum(j, 0)] + expire >= t[first][:, None]), hist, 0)
    return user, hist


def _expire(h):
    w = h._w_device()
    return 0 if w is None else w[1]


HANDLERS = [('Seq2VecPaperSoftmax', 30, 'gru'), ('Seq2VecPaperSoftmaxId', 30, 'igru'), ('Seq2VecPaperSoftmaxDays', 1, 'gru'),
            ('Seq2VecPaperSoftmaxDays', 2, 'gru'), ('Seq2VecPaperSoftmaxDaysId', 1, 'igru'),
            ('Seq2VecPaperSoftmaxDaysId', 2, 'igru'), ('Seq2VecPaperSoftmaxDaysIdVert', 2, 'igru'),
            ('Seq2VecPaperSoftmaxDaysIdVertSup', 1, 'igru')]


@pytest.mark.parametrize('task_name,days,arch', HANDLERS)
def test_eval_tables_match_test_gen(task_name, days, arch):
    h = _handler(task_name, days, arch)
    T = assemble.build_tables(h.data, SH.W, h._w_device())
    user, hist = _history(T, SH.W, _expire(h))
    tok = h.doc_token_table()
    vert = isinstance(h, task.Seq2VecPaperSoftmaxDaysIdVert)
    dvert = h.device_doc_vert()
    off, docs, npos = T['eval_cand_off'], T['eval_cand_docs'], T['eval_npos']
    n = 0
    for i, rows in enumerate(h.test_gen()):
        cand = docs[off[i]:off[i + 1]]
        assert len(rows) == len(cand) and npos[i] >= 1, i
        for k, row in enumerate(rows):
            row = list(row)
            if h.HAS_USER:
                assert row.pop(0) == user[i], i
            assert np.array_equal(row[0], tok[hist[i]]), i              # the W history titles
            if vert:
                assert list(row[1]) == list(dvert[hist[i]]) and row[3] == dvert[cand[k]], i
                row = [row[0], row[2], row[4]]
            assert np.array_equal(row[1], tok[cand[k]]) and row[2] == int(k < npos[i]), (i, k)
        n += 1
    assert n == len(T['eval_first_click']) == len(off) - 1 > 10
    assert (np.diff(off) > 32).any()
    assert (docs == ZERO_DOC).any() and (hist == ZERO_DOC).any()
    assert (~tok[hist].any(-1)).all(-1).any()                         # some history has no unmasked slot
    if days == 1:                                                     # the time window really bites
        _, plain = _history(assemble.build_tables(h.data), SH.W, 0)
        assert ((plain != 0).sum(1) > (hist != 0).sum(1)).any()
        assert ((plain != 0).any(1) & (hist == 0).all(1)).any()       # a fully expired history


def test_handlers_without_device_evaluation_say_so():
    from mnexp_b200 import main
    for name, arch in (('Seq2VecPaperSoftmaxDaysIdVertAlt', 'igru'), ('Seq2VecPaper', 'gru')):
        h = _handler(name, 2, arch)
        with pytest.raises(NotImplementedError):
            h.device_callback(0)
        with pytest.raises(NotImplementedError):
            main.train(h.config, device_eval=True)


# ---- GPU ---------------------------------------------------------------------------------------------------------------
def _trained(task_name, days, arch, precision, seed=3, **kw):
    np.random.seed(seed)
    h = _handler(task_name, days, arch, precision=precision, **kw)
    model = h.build_model(0)
    model.fit_generator(h.device_train, 3)
    return h


def _host_scores(h):
    h.model, h.test_model = h.test_model, h.model
    try:
        out = [(np.asarray(p).reshape(-1), np.asarray(y).reshape(-1)) for p, y in h.test]
    finally:
        h.model, h.test_model = h.test_model, h.model
    return out


def _device_scores(h, n=10 ** 9):
    off, scores, labels = h.device_test(n)
    off, scores, labels = off.cpu().numpy(), scores.cpu().numpy(), labels.cpu().numpy()
    return [(scores[a:b], labels[a:b]) for a, b in zip(off[:-1], off[1:])]


TOL = {'fp32': 1e-5, 'fp16_tc': 1e-3}
SCORE_CASES = [('Seq2VecPaperSoftmaxId', 30, 'igru', 'dot'), ('Seq2VecPaperSoftmaxId', 30, 'igru', 'dnn'),
               ('Seq2VecPaperSoftmaxId', 30, 'igru', 'ddot'), ('Seq2VecPaperSoftmaxId', 30, 'gru', 'dnn'),
               ('Seq2VecPaperSoftmaxId', 30, 'dgru', 'dnn'), ('Seq2VecPaperSoftmax', 30, 'gru', 'dot'),
               ('Seq2VecPaperSoftmax', 30, 'att', 'dot'), ('Seq2VecPaperSoftmax', 30, 'avg', 'dot'),
               ('Seq2VecPaperSoftmaxDaysIdVert', 2, 'igru', 'dot'), ('Seq2VecPaperSoftmaxDaysId', 1, 'igru', 'ddot')]


@pytest.mark.gpu
@pytest.mark.parametrize('precision', ['fp32', 'fp16_tc'])
@pytest.mark.parametrize('task_name,days,arch,score_model', SCORE_CASES)
def test_device_scores_equal_host_scores(lib, task_name, days, arch, score_model, precision):
    h = _trained(task_name, days, arch, precision, score_model=score_model)
    host = _host_scores(h)
    dev = _device_scores(h)
    assert len(dev) == len(host) > 10
    assert max(len(s) for s, _ in dev) > 32
    eng = h._eval_engine()
    assert len(dev) > eng.B                                      # the evaluation spans several chunks
    for i, ((ds, dl), (hs, hl)) in enumerate(zip(dev, host)):
        assert np.array_equal(dl, hl), i
    assert_close(np.concatenate([s for s, _ in dev]), np.concatenate([s for s, _ in host]), tol=TOL[precision],
                 name='%s %s %s' % (task_name, arch, score_model))
    part = _device_scores(h, 5)                                  # the first n impressions only
    assert len(part) == 5 and all(np.array_equal(a[0], b[0]) for a, b in zip(part, dev))


def _logged(fn, *args):
    got = []
    orig = utils.logging_evaluation
    utils.logging_evaluation = lambda d: got.append(dict(d))
    try:
        fn(*args)
    finally:
        utils.logging_evaluation = orig
    return got


@pytest.mark.gpu
@pytest.mark.parametrize('precision', ['fp32', 'fp16_tc'])
def test_device_callback_logs_what_callback_logs(lib, precision):
    h = _trained('Seq2VecPaperSoftmaxId', 30, 'igru', precision, validation_impression=20)
    # after a few steps from the initial weights the scores crowd around 0.5; a larger Dense spreads them, so that no two
    # candidates of an impression are within reach of rounding (checked below in fp32)
    eng = h._core.train_engine
    for name in ('dense_w', 'dense_b'):
        off, cnt, _ = eng.layout[name]
        eng.dense[off:off + cnt] *= 6.0
    lr0 = h.model.optimizer.lr.value
    model, test_model = h.model, h.test_model
    runs = {}
    for name in ('callback', 'device_callback'):
        h.model.optimizer.lr.value = lr0
        h.is_training = True
        lines = _logged(getattr(h, name), 1)                          # the last epoch: the testing pass follows
        runs[name] = (lines, h.model.optimizer.lr.value, h.model is model and h.test_model is test_model,
                      h.is_training, dict(h.last_evaluation))
    (hl, hlr, hid, htr, hev), (dl, dlr, did, dtr, dev) = runs['callback'], runs['device_callback']
    assert len(hl) == len(dl) == 4 and [sorted(d) for d in hl] == [sorted(d) for d in dl]
    assert hlr == dlr and hid and did and htr is False and dtr is False
    assert [hl[1], hl[3]] == [dl[1], dl[3]]                           # pos / size / num
    assert hev.keys() == dev.keys()
    if precision == 'fp32':
        for s, _ in _host_scores(h)[:20]:                             # no rank can flip between the two paths
            s = np.sort(s)
            assert (np.diff(s) > 1e-5).all()
        for a, b in ((hl[0], dl[0]), (hl[2], dl[2])):
            for k in a:
                assert abs(a[k] - b[k]) <= 1e-6 or (np.isnan(a[k]) and np.isnan(b[k])), k
    else:
        dev_rows = _device_scores(h)
        got = h._device_rows(10 ** 9)[0]
        ref = metrics.ranking_metrics([s for s, _ in dev_rows], [y for _, y in dev_rows])
        assert np.array_equal(got, ref, equal_nan=True)
    again = _logged(h.device_callback, 0)                              # two passes on the same weights: the same values
    h.model.optimizer.lr.value = lr0
    assert repr(again) == repr(_logged(h.device_callback, 0)) and len(again) == 2


@pytest.mark.gpu
def test_impression_beyond_chunk_capacity_is_rejected(lib):
    from mnexp_b200._lib import LsturError
    h = _trained('Seq2VecPaperSoftmaxId', 30, 'igru', 'fp32')
    host, dev = h._uploaded_tables()
    eng = h._core.engine_infer(4, rows=8)                              # 32 pairs per chunk
    big = int(np.argmax(np.diff(host['eval_cand_off'])))
    a, b = host['eval_cand_off'][big:big + 2]
    assert b - a > 32
    zeros = lambda *s: torch.zeros(s, dtype=torch.int32, device=eng.device)
    with pytest.raises(LsturError, match='candidates'):
        eng.score_impressions(zeros(1), zeros(1, SH.W), np.array([0, b - a]), dev['eval_cand_docs'][a:b].contiguous(),
                              eng.eval_doc_table())


@pytest.mark.gpu
@pytest.mark.parametrize('device_batches', [False, True])
def test_main_train_device_eval(lib, device_batches):
    from mnexp_b200 import main
    runs = []
    for device_eval in (False, True):
        np.random.seed(2)
        h = _handler('Seq2VecPaperSoftmaxId', 30, 'igru', precision='fp32')
        _, records = main.train(h.config, device_batches=device_batches, device_eval=device_eval)
        runs.append(records)
    a, b = runs
    assert [(k, sorted(d)) for k, d in a] == [(k, sorted(d)) for k, d in b] and len(a) >= 8
    if not device_batches:
        for (ka, da), (kb, db) in zip(a, b):
            if ka == 'history':
                assert da == db
            else:
                for k in da:
                    assert abs(da[k] - db[k]) <= 1e-5 or (np.isnan(da[k]) and np.isnan(db[k])), (k, da[k], db[k])
