"""Batches assembled on the device (mnexp_b200/assemble.py, lstur_assemble_samples) for the softmax-family task handlers.

CPU: the host tables of build_tables, read by a numpy statement of the kernel's rule, give sample for sample the user,
history ids, positive and negatives that the handler's own Window / _w_push / _w_count / get_ids hooks give, for the
training and the validation split, with and without the Days time window.
GPU: the kernel equals that replay bit for bit; lstur_assemble_batch keeps its output; the training order, the
data-parallel sharding, training steps, evaluation and main.train through the Model protocol."""
import tempfile

import numpy as np
import pytest
import torch

from mnexp_b200 import assemble, rng, settings, synth, task, utils
from mnexp_b200.task.paper import _DaysWindowMixin

SH = synth.Shape('dev', 60, 80, 120, L=7, W=5, K=2, B=6, E=12, F=16, U=8)
_DATA = {}


def _handler(task_name, days=30, arch='igru', **kw):
    if 'dir' not in _DATA:
        _DATA['dir'] = tempfile.mkdtemp()
        synth.write_dataset(_DATA['dir'], SH)
    cfg = dict(task=task_name, arch=arch, input_training_data_path=_DATA['dir'], title_shape=SH.L, window_size=SH.W,
               negative_samples=SH.K, batch_size=8, textual_embedding_dim=SH.E, title_filter_shape=(SH.F, 3),
               user_embedding_dim=SH.U, debug=True, dropout=0.0, days=days, validation_impression=5,
               testing_impression=5, epochs=2, training_step=3, validation_step=2)
    cfg.update(kw)
    return task.get(settings.Config(cfg))


def _replay(h, split):
    """(user, W history ids, positive, impression negatives) per sample, in train_gen / valid_gen order, through the
    handler's own window hooks."""
    days = isinstance(h, _DaysWindowMixin)
    ids = lambda ch, imp: np.asarray(ch.get_ids(imp.time) if days else ch.get_ids(), dtype=np.int64)
    out = []
    for user, (ih, iv) in enumerate(h.data):
        if not ih or (split == 'valid' and not iv):
            continue
        ch = h._new_window()
        if split == 'train':
            for imp in ih:
                for pos in imp.pos:
                    if h._w_count(ch, imp):
                        out.append((user, ids(ch, imp), pos, list(imp.neg)))
                    h._w_push(ch, pos, imp)
            continue
        for imp in ih:
            for pos in imp.pos:
                h._w_push(ch, pos, imp)
        for imp in iv:
            for pos in imp.pos:
                out.append((user, ids(ch, imp), pos, list(imp.neg)))
            for pos in imp.pos:
                h._w_push(ch, pos, imp)
    return out


def _table_rows(T, split, W, expire):
    """numpy statement of lstur_assemble_samples over every sample of a split: user, history ids, positive, negatives."""
    click = T['sample_click'] if split == 'train' else T['valid_click']
    end = click if split == 'train' else T['valid_hist_end']
    user = T['click_user'][click]
    j = end[:, None].astype(np.int64) - W + np.arange(W)
    ok = j >= T['stream_off'][user][:, None]
    hist = np.where(ok, T['stream_docs'][np.maximum(j, 0)], 0)
    if 'click_time' in T:
        t = T['click_time'].astype(np.int64)
        hist = np.where(ok & (t[np.maximum(j, 0)] + expire >= t[click][:, None]), hist, 0)
    negs = [list(T['neg_docs'][T['neg_off'][c]:T['neg_off'][c + 1]]) for c in click]
    return user, hist, T['stream_docs'][click], negs


HANDLERS = [('Seq2VecPaperSoftmax', 30, 'gru'), ('Seq2VecPaperSoftmaxId', 30, 'igru'), ('Seq2VecPaperSoftmaxDays', 1, 'gru'),
            ('Seq2VecPaperSoftmaxDays', 2, 'gru'), ('Seq2VecPaperSoftmaxDaysId', 1, 'igru'),
            ('Seq2VecPaperSoftmaxDaysId', 2, 'igru')]


def _expire(h):
    w = h._w_device()
    return 0 if w is None else w[1]


@pytest.mark.parametrize('task_name,days,arch', HANDLERS)
def test_tables_match_window_replay(task_name, days, arch):
    h = _handler(task_name, days, arch)
    T = assemble.build_tables(h.data, SH.W, h._w_device())
    for split in ('train', 'valid'):
        want = _replay(h, split)
        user, hist, pos, negs = _table_rows(T, split, SH.W, _expire(h))
        assert len(want) == len(user) > 0, split
        for i, (u, w, p, n) in enumerate(want):
            assert user[i] == u and np.array_equal(hist[i], w) and pos[i] == p and negs[i] == n, (split, i)
    if days == 1:
        # the time window really bites: some training click has no live history, and some history slot has expired
        plain = assemble.build_tables(h.data)
        assert len(T['sample_click']) < len(plain['sample_click'])
        _, hp, _, _ = _table_rows(plain, 'train', SH.W, 0)
        _, hd, _, _ = _table_rows(T, 'train', SH.W, _expire(h))
        keep = np.isin(plain['sample_click'], T['sample_click'])
        assert ((hp[keep] != 0).sum(1) > (hd != 0).sum(1)).any()


@pytest.mark.parametrize('task_name,days,arch', [HANDLERS[1], HANDLERS[4]])
def test_validation_order_is_valid_gen_order(task_name, days, arch):
    h = _handler(task_name, days, arch)
    T = assemble.build_tables(h.data, SH.W, h._w_device())
    user, hist, pos, _ = _table_rows(T, 'valid', SH.W, _expire(h))
    gen = h.valid_gen()
    tok = h.doc_token_table()
    for i in range(len(user)):
        s = next(gen)
        if h.HAS_USER:
            assert s[0] == user[i]
            s = s[1:]
        assert np.array_equal(s[0], tok[hist[i]]) and np.array_equal(s[1], tok[pos[i]]), i
    s = next(gen)                                              # and then valid_gen starts over
    assert np.array_equal(s[2 if h.HAS_USER else 1], tok[pos[0]])


@pytest.mark.parametrize('task_name', ['Seq2VecPaperSoftmaxDaysIdVert', 'Seq2VecPaperSoftmaxDaysIdVertSup'])
def test_doc_vert_matches_handler_verticals(task_name):
    """The doc_vert table that device batches take their vertical ids from == the verticals the handler's own samples
    carry (_w_vert over the window, docs[·].vertical for the candidates) == the verticals the dataset was written with."""
    h = _handler(task_name, 2)
    dvert = h.device_doc_vert()
    written = synth.make_docs(SH.n_news, SH.L, SH.vocab, seed=7 + 1)[1]        # synth.write_dataset(d, SH) with seed 7
    assert dvert[0] == 0 and np.array_equal(dvert, written)
    n = 0
    for user, (ih, _) in enumerate(h.data):
        ch = h._new_window()
        for imp in ih:
            for pos in imp.pos:
                if h._w_count(ch, imp):
                    assert list(dvert[ch.get_ids(imp.time)]) == list(h._w_vert(ch, imp))
                    assert dvert[pos] == h.docs[pos].vertical and all(dvert[x] == h.docs[x].vertical for x in imp.neg)
                    n += 1
                h._w_push(ch, pos, imp)
    assert n > 0


def test_handlers_without_device_batches_say_so():
    from mnexp_b200 import main
    h = _handler('Seq2VecPaperSoftmaxDaysIdVertAlt', 2)
    with pytest.raises(NotImplementedError):
        h.device_train
    with pytest.raises(NotImplementedError):
        h.device_valid
    with pytest.raises(NotImplementedError):
        main.train(_handler('Seq2VecPaper', arch='gru').config, device_batches=True)


# ---- GPU ---------------------------------------------------------------------------------------------------------------
def _neg_replay(T, click, seed_step, row0, K, split_negs):
    B = len(click)
    r = rng.rng_u32(seed_step, (np.arange(B, dtype=np.uint64)[:, None] + row0) * K + np.arange(K, dtype=np.uint64))
    return np.array([[split_negs[b][int(r[b, k]) % len(split_negs[b])] for k in range(K)] for b in range(B)])


@pytest.mark.gpu
@pytest.mark.parametrize('task_name,days,arch', HANDLERS)
def test_device_batches_equal_replay(lib, task_name, days, arch):
    h = _handler(task_name, days, arch)
    for split in ('train', 'valid'):
        want = _replay(h, split)
        bt = assemble.DeviceBatcher(h.data, 16, SH.W, SH.K, seed=3, split=split, window=h._w_device())
        T = bt.host
        click = T['sample_click'] if split == 'train' else T['valid_click']
        for _ in range(4):
            idx, row0 = bt._next_indices()
            db = bt.assemble(idx, row0)
            seed_step = (bt.seed * 1000003 + bt.step) & 0xffffffff
            s = idx.cpu().numpy()
            user, hist, cand = (db[k].cpu().numpy() for k in ('user', 'hist_doc', 'cand_doc'))
            for b, si in enumerate(s):
                u, w, p, _ = want[si]
                assert user[b] == u and np.array_equal(hist[b], w) and cand[b, 0] == p, (split, b)
            negs = [list(T['neg_docs'][T['neg_off'][c]:T['neg_off'][c + 1]]) for c in click[s]]
            assert np.array_equal(cand[:, 1:], _neg_replay(T, click[s], seed_step, row0, SH.K, negs))
        if split == 'valid':     # valid batches walk the samples in order and wrap
            n = len(want)
            bt2 = assemble.DeviceBatcher(h.data, 16, SH.W, SH.K, split='valid', window=h._w_device(), tables=T)
            got = np.concatenate([bt2._next_indices()[0].cpu().numpy() for _ in range(3)])
            assert np.array_equal(got, np.arange(48) % n)


@pytest.mark.gpu
def test_assemble_batch_output_unchanged(lib):
    """lstur_assemble_batch, now a wrapper of lstur_assemble_samples, gives what it gave before: the W clicks before the
    sample (no time window even when the tables carry times), negatives from rng_u32(seed, b*K + k)."""
    import ctypes
    h = _handler('Seq2VecPaperSoftmaxDaysId', 1, 'igru')
    T = assemble.build_tables(h.data, SH.W, h._w_device())
    t = {k: torch.as_tensor(v).cuda() for k, v in T.items()}
    B, W, K, seed = 40, SH.W, SH.K, 12345
    s = np.random.default_rng(0).integers(0, len(T['sample_click']), B).astype(np.int32)
    idx = torch.as_tensor(s).cuda()
    out = [torch.full(shape, -1, dtype=torch.int32, device='cuda') for shape in ((B,), (B, W), (B, 1 + K))]
    p = lambda x: ctypes.c_void_p(x.data_ptr())
    assert lib.lstur_assemble_batch(B, W, K, p(t['sample_click']), p(idx), p(t['click_user']), p(t['stream_off']),
                                    p(t['stream_docs']), p(t['neg_off']), p(t['neg_docs']), seed, *[p(o) for o in out],
                                    ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)) == 0
    user, hist, cand = (o.cpu().numpy() for o in out)
    c = T['sample_click'][s]
    j = c[:, None].astype(np.int64) - W + np.arange(W)
    off = T['stream_off'][T['click_user'][c]]
    assert np.array_equal(user, T['click_user'][c])
    assert np.array_equal(hist, np.where(j >= off[:, None], T['stream_docs'][np.maximum(j, 0)], 0))
    assert np.array_equal(cand[:, 0], T['stream_docs'][c])
    negs = [list(T['neg_docs'][T['neg_off'][x]:T['neg_off'][x + 1]]) for x in c]
    assert np.array_equal(cand[:, 1:], _neg_replay(T, c, seed, 0, K, negs))


@pytest.mark.gpu
def test_training_epochs_visit_every_sample_once(lib):
    h = _handler('Seq2VecPaperSoftmaxId')
    bt = assemble.DeviceBatcher(h.data, 7, SH.W, SH.K, seed=9)
    n = bt.n_samples
    got = np.concatenate([bt._next_indices()[0].cpu().numpy() for _ in range(-(-2 * n // 7) + 1)])
    for e in range(2):
        assert np.array_equal(np.sort(got[e * n:(e + 1) * n]), np.arange(n)), e
    assert not np.array_equal(got[:n], got[n:2 * n])          # a new permutation per epoch


@pytest.mark.gpu
def test_two_ranks_see_the_rows_of_one(lib):
    h = _handler('Seq2VecPaperSoftmaxDaysId', 2, 'igru')
    B = 8
    one = assemble.DeviceBatcher(h.data, 2 * B, SH.W, SH.K, seed=4, window=h._w_device())
    ranks = [assemble.DeviceBatcher(h.data, B, SH.W, SH.K, seed=4, rank=r, world=2, window=h._w_device(), tables=one.host)
             for r in range(2)]
    for _ in range(2 * one.n_samples // (2 * B) + 2):       # past an epoch boundary
        full = one.next_batch()
        for r, bt in enumerate(ranks):
            part = bt.next_batch()
            for k in ('user', 'hist_doc', 'cand_doc'):
                assert torch.equal(part[k], full[k][r * B:(r + 1) * B]), (r, k)


def _host_inputs(h, db):
    """A device batch as the host token protocol: float64 token arrays (and per-slot vertical ids / one-hot targets)."""
    tok = h.doc_token_table().astype(np.float64)
    user, hist, cand = (db.as_dict()[k].cpu().numpy() for k in ('user', 'hist_doc', 'cand_doc'))
    C = cand.shape[1]
    x = ([user] if h.HAS_USER else []) + [tok[hist]]
    label = np.zeros((len(user), C), dtype=np.float32)
    label[:, 0] = 1
    dvert = h.device_doc_vert()
    if isinstance(h, task.Seq2VecPaperSoftmaxDaysIdVert):
        x = x + [dvert[hist]] + [tok[cand[:, k]] for k in range(C)] + [dvert[cand[:, k]] for k in range(C)]
    else:
        x = x + [tok[cand[:, k]] for k in range(C)]
    if isinstance(h, task.Seq2VecPaperSoftmaxDaysIdVertSup):
        verts = np.concatenate([dvert[hist], dvert[cand]], 1)
        y = [label, np.stack([np.eye(len(utils.verticals), dtype=np.float32)[v] for v in verts])]
    else:
        y = label
    return x, y


@pytest.mark.gpu
@pytest.mark.parametrize('precision', ['fp32', 'fp16_tc'])
@pytest.mark.parametrize('task_name,days,arch', [('Seq2VecPaperSoftmaxId', 30, 'igru'), ('Seq2VecPaperSoftmax', 30, 'gru'),
                                                 ('Seq2VecPaperSoftmaxDaysIdVert', 2, 'igru'),
                                                 ('Seq2VecPaperSoftmaxDaysIdVertSup', 2, 'igru')])
def test_same_batch_two_paths(lib, task_name, days, arch, precision):
    """Three training steps on device batches == the same steps on those batches as host arrays, bit for bit."""
    runs = []
    for path in ('device', 'host'):
        np.random.seed(11)
        h = _handler(task_name, days, arch, precision=precision, dropout=0.2)
        model = h.build_model(0)
        gen = h.device_train
        metrics = []
        for _ in range(3):
            db = next(gen)
            metrics.append(model.train_on_batch(db) if path == 'device' else model.train_on_batch(*_host_inputs(h, db)))
        runs.append((metrics, model.get_weights()))
    (m0, w0), (m1, w1) = runs
    assert m0 == m1
    assert len(w0) == len(w1) and all(np.array_equal(a, b) for a, b in zip(w0, w1))


@pytest.mark.gpu
@pytest.mark.parametrize('task_name,days,arch', [('Seq2VecPaperSoftmaxId', 30, 'igru'), ('Seq2VecPaperSoftmaxDaysIdVert', 2, 'igru'),
                                                 ('Seq2VecPaperSoftmaxDaysIdVertSup', 2, 'igru')])
def test_evaluate_generator_on_device_valid(lib, task_name, days, arch):
    h = _handler(task_name, days, arch)
    model = h.build_model(0)
    model.fit_generator(h.device_train, 2)
    got = model.evaluate_generator(h.device_valid, 3)
    dev = h._device_tables[1]
    gen = h.device_valid                       # a new generator starts from the first sample again
    assert h._device_tables[1] is dev          # ... on the tables the handler uploaded once
    tot = np.zeros(len(model.metrics_names))
    for _ in range(3):
        tot += model.evaluate(*_host_inputs(h, next(gen)))
    assert len(got) == len(model.metrics_names) and np.array_equal(np.asarray(got), tot / 3)


@pytest.mark.gpu
def test_fit_generator_on_device_batches_learns(lib):
    np.random.seed(5)
    h = _handler('Seq2VecPaperSoftmaxId', arch='dgru', score_model='dnn')
    model = h.build_model(0)
    hist = model.fit_generator(h.device_train, 12)
    assert set(hist.history) == {'loss', 'categorical_accuracy'} and np.isfinite(hist.history['loss'][0])
    fixed = next(h.device_valid)
    l0 = model.evaluate(fixed)[0]
    for _ in range(25):
        model.train_on_batch(fixed)
    assert model.evaluate(fixed)[0] < l0


@pytest.mark.gpu
@pytest.mark.parametrize('task_name,days,arch', [('Seq2VecPaperSoftmaxId', 30, 'igru'), ('Seq2VecPaperSoftmaxDays', 2, 'gru')])
def test_main_train_device_batches(lib, task_name, days, arch):
    from mnexp_b200 import main
    keys = []
    for device in (False, True):
        np.random.seed(2)
        h = _handler(task_name, days, arch)
        _, records = main.train(h.config, device_batches=device)
        keys.append([(kind, sorted(d)) for kind, d in records])
        if device:
            assert all(np.isfinite(v).all() for kind, d in records for v in d.values() if kind == 'history')
    assert keys[0] == keys[1] and len(keys[0]) >= 4
