"""`Cook` task handler of the reference (task/cook.py:4-285) on the CUDA engine.

Data: two .npz files (settings.Config.train_npz_input / test_npz_input) with `idx, idx_mask, ch_title (N,W,L), ch_vert,
ch_subvert (N,W), cd_title (N,5,L), cd_vert, cd_subvert (N,5), cd_label (N,5)`; the test file carries one candidate per
row (`cd_title (n,L), cd_vert, cd_subvert (n,), label, user, impr`).  `train()/valid()/test()` return the same
(features, labels) lists; `build_model(epoch)` returns `train_model` ((1+4)-way softmax CE + Adam) and sets `test_model`
(sigmoid score of one candidate), both with the Keras calls main.py's cook loop makes (fit / evaluate / predict /
predict_on_batch / metrics_names / optimizer.lr / summary).  News vector = [title CNN+attention ‖ Vemb[vert] ‖
Semb[subvert]] without the Dense (task/cook.py:99-113); the user id embedding is multiplied by
Dropout(1 - id_keep)(idx_mask) (:139-142).  Every branch of Cook.get_user_encoder is built (vo, avg, gru, igru, iavg,
iatt, ilstm, agru, ingru, inigru, inagru, atgru, algru, :146-193); unknown names raise the reference's NotImplementedError.
"""
import logging

import numpy as np

from .. import keras_like, metrics, settings, synth
from ..engine import COOK_ARCH

FEATURES = ['idx', 'idx_mask', 'ch_title', 'ch_vert', 'ch_subvert', 'cd_title', 'cd_vert', 'cd_subvert']
N_USER_ROWS = 25000                                       # keras.layers.Embedding(25000, ...), task/cook.py:137
TWO_ID_ARCHS = ('inigru', 'inagru')     # a second id embedding with its own Dropout layer (task/cook.py:169-183)


class CookDeviceData:
    """The rows of one Cook .npz file on the device, titles interned (mnexp_b200/intern.py): user (n,) int32 (`idx`),
    mask (n,) float32 (`idx_mask`), hist_doc (n, W) and cand_doc (n, C) int32 document ids, label (n, C) float32; plus
    host_mask, the host copy of `mask` the training draws read.  Cook.device_train / device_valid / device_test return
    it where train / valid / test return the feature lists."""
    __slots__ = ('user', 'mask', 'hist_doc', 'cand_doc', 'label', 'host_mask')

    def __init__(self, user, mask, hist_doc, cand_doc, label, host_mask):
        self.user, self.mask, self.hist_doc, self.cand_doc, self.label = user, mask, hist_doc, cand_doc, label
        self.host_mask = host_mask

    @property
    def n(self):
        return int(self.user.numel())

    def head(self, k):
        """the first k rows"""
        return CookDeviceData(self.user[:k], self.mask[:k], self.hist_doc[:k], self.cand_doc[:k], self.label[:k],
                              self.host_mask[:k])


def epoch_scales(mask, order, batch_size, keep, two):
    """The id-embedding multipliers of one epoch of CookModel.fit, drawn from numpy's global stream exactly as the host
    loop draws them batch by batch (CookModel._batch on the rows of each batch, the ragged last one padded with its first
    row): -> (scale, scale2) float32 arrays of ceil(n / B) * B entries, entry s*B + b for row b of batch s (scale2 None
    unless `two`, the archs with a second id table)."""
    n, B = len(order), batch_size
    nb = -(-n // B)
    slot = np.arange(nb * B)
    rows = np.asarray(order)[np.where(slot < n, slot, slot // B * B)]
    scale = np.asarray(mask, dtype=np.float32).reshape(-1)[rows]
    scale2 = scale.copy() if two else None
    if keep < 1.0:               # Dropout(1 - id_keep) on the mask (task/cook.py:141-142): random(B) per table per batch
        r = np.empty((nb, 2 if two else 1, B))
        for s in range(nb):
            for t in range(r.shape[1]):
                r[s, t] = np.random.random(B)
        scale = scale * (r[:, 0].reshape(-1) < keep).astype(np.float32) / keep
        if two:
            scale2 = scale2 * (r[:, 1].reshape(-1) < keep).astype(np.float32) / keep
    return scale, scale2


class CookModel:
    """train_model (train=True) or test_model of Cook._build_model, task/cook.py:214-277, over the engines, weights and
    optimizer of the handler's keras_like._Core."""

    def __init__(self, owner, train):
        self.owner, self.is_train = owner, train
        self.metrics_names = ['loss', 'categorical_accuracy'] if train else ['loss', 'auc_roc']

    @property
    def core(self):
        return self.owner._core

    @property
    def optimizer(self):
        return self.core.optimizer

    _current = get_weights_dict = keras_like.Model._current
    summary = keras_like.Model.summary

    def _batch(self, x, rows, C, training):
        idx, idx_mask, ch_title, ch_vert, ch_subvert, cd_title, cd_vert, cd_subvert = [np.asarray(a)[rows] for a in x]
        n = len(rows)
        scale = np.asarray(idx_mask, dtype=np.float32).reshape(n)
        keep = self.owner.config.id_keep
        scale2 = None
        two = self.owner.config.arch in TWO_ID_ARCHS
        if two:
            scale2 = scale.copy()
        if training and keep < 1.0:                       # Dropout(1 - id_keep) on the mask (task/cook.py:141-142)
            scale = scale * (np.random.random(n) < keep).astype(np.float32) / keep
            if two:
                scale2 = scale2 * (np.random.random(n) < keep).astype(np.float32) / keep
        b = dict(user=np.asarray(idx).reshape(n), user_scale=scale, hist_tok=ch_title,
                 cand_tok=np.asarray(cd_title).reshape(n, C, -1))
        if two:
            b['user_scale2'] = scale2
        if self.owner.dv:
            b['hist_vert'] = ch_vert
            b['cand_vert'] = np.asarray(cd_vert).reshape(n, C)
        if self.owner.ds:
            b['hist_subvert'] = ch_subvert
            b['cand_subvert'] = np.asarray(cd_subvert).reshape(n, C)
        return b

    def fit(self, x, y, batch_size=32, epochs=1, initial_epoch=0, shuffle=True, verbose=0, **_):
        assert self.is_train
        if isinstance(x, CookDeviceData):
            return self._fit_device(x, batch_size, epochs, initial_epoch, shuffle)
        y = np.asarray(y[0] if isinstance(y, (list, tuple)) else y, dtype=np.float32)
        n, C = y.shape
        h = keras_like.History()
        for epoch in range(initial_epoch, epochs):
            order = np.random.permutation(n) if shuffle else np.arange(n)
            tot, k = np.zeros(2), 0
            eng = self.core.engine_train(batch_size)
            eng.lr = self.optimizer.lr.value
            for s in range(0, n, batch_size):
                rows = order[s:s + batch_size]
                m = len(rows)
                lab = np.zeros((batch_size, C), dtype=np.float32)
                lab[:m] = y[rows]
                if m < batch_size:
                    # Keras trains the ragged last batch too (training.py fit_loop / make_batches).  The plan is per batch
                    # size, so the m samples run as batch_size rows: padding rows repeat the first sample under an all-zero
                    # target (zero loss, zero gradient) and the gradient scale is 1 / m
                    rows = np.concatenate([rows, np.full(batch_size - m, rows[0])])
                b = self._batch(x, rows, C, True)
                b['label'] = lab
                db = eng.to_device_batch(b)
                loss = eng.train_step(db, grad_scale=1.0 / m)
                probs = eng.view('probs').reshape(eng.B, eng.C)[:m]
                tot += [float(loss[0]) * batch_size, float((probs.argmax(1) == db['label'][:m].argmax(1)).float().sum())]
                k += m                              # Keras logs the sample-weighted mean over the batches
            h.epoch.append(epoch)
            for name, v in zip(self.metrics_names, tot / max(1, k)):
                h.history.setdefault(name, []).append(float(v))
        return h

    def _fit_device(self, x, batch_size, epochs, initial_epoch, shuffle):
        """fit on interned device rows (Cook.device_train): the host loop's permutation and id_keep draws, once per epoch
        (epoch_scales), batches gathered on the device (intern.gather_samples), and loss / accuracy summed on the device
        in step order and read once per epoch.  The kernels see the same token rows as in the host loop."""
        import torch
        n = x.n
        two = self.owner.config.arch in TWO_ID_ARCHS
        h = keras_like.History()
        for epoch in range(initial_epoch, epochs):
            order = np.random.permutation(n) if shuffle else np.arange(n)
            scale, scale2 = epoch_scales(x.host_mask, order, batch_size, self.owner.config.id_keep, two)
            eng = self.core.engine_train(batch_size)
            eng.lr = self.optimizer.lr.value
            up = lambda a: None if a is None else torch.as_tensor(a).to(eng.device)
            tot = self._device_steps(eng, x, up(order.astype(np.int32)), up(scale), up(scale2))
            h.epoch.append(epoch)
            for name, v in zip(self.metrics_names, tot.cpu().numpy() / max(1, n)):
                h.history.setdefault(name, []).append(float(v))
        return h

    @staticmethod
    def _device_steps(eng, x, order, scale, scale2):
        """One epoch of train steps over the rows `order` (device int32), batch s taking its id multipliers from entries
        s*B .. (s+1)*B of scale / scale2 (device float32; scale2 None for one id table).  Nothing waits for the device:
        -> (2,) float64 device tensor [sum of loss * B, count of correct argmaxes], summed in step order."""
        import torch
        from .. import intern
        n, B, C, W = int(order.numel()), eng.B, eng.C, x.hist_doc.shape[1]
        dev = eng.device
        src = dict(user=x.user, hist_doc=x.hist_doc, cand_doc=x.cand_doc, label=x.label)
        i32 = dict(dtype=torch.int32, device=dev)
        out = dict(user=torch.empty(B, **i32), hist_doc=torch.empty((B, W), **i32), cand_doc=torch.empty((B, C), **i32),
                   label=torch.empty((B, C), dtype=torch.float32, device=dev))
        tot = torch.zeros(2, dtype=torch.float64, device=dev)
        probs = eng.view('probs').reshape(B, C)
        for step, s in enumerate(range(0, n, B)):
            m = min(B, n - s)
            intern.gather_samples(order[s:], m, src, out)
            db = dict(out, user_scale=scale[step * B:(step + 1) * B])
            if scale2 is not None:
                db['user_scale2'] = scale2[step * B:(step + 1) * B]
            loss = eng.train_step(db, grad_scale=1.0 / m)
            tot[0] += loss[0].double() * B           # the host loop's float(loss) * batch_size, in float64
            tot[1] += (probs[:m].argmax(1) == out['label'][:m].argmax(1)).double().sum()
        return tot

    def _predict_device(self, x):
        """test_model scores of interned test rows (Cook.device_valid / device_test) -> (n,) float32 device tensor.
        Consecutive rows with the same user, mask and history form one impression of lstur_score_impressions (one user
        vector; split where it exceeds the plan's rows * candidates), every document is encoded once."""
        import torch
        from .. import intern
        assert not self.is_train and x.cand_doc.shape[1] == 1, 'device scoring is the one-candidate test model'
        n = x.n
        starts = intern.group_rows(x.user, x.mask, x.hist_doc)
        sizes = np.diff(np.append(starts, n))
        C = int(min(32, max(1, np.ceil(sizes.mean())))) if n else 1
        eng = self.core.engine_infer(C)
        cap = eng.B * eng.C
        pieces = np.concatenate([np.arange(a, a + k, cap) for a, k in zip(starts, sizes)]) if n else np.zeros(0, np.int64)
        off = np.append(pieces, n).astype(np.int32)
        P, W, dev = len(pieces), x.hist_doc.shape[1], eng.device
        out = torch.empty(n, dtype=torch.float32, device=dev)
        if n == 0:
            return out
        pos = torch.as_tensor(pieces.astype(np.int32)).to(dev)
        g = dict(user=torch.empty(P, dtype=torch.int32, device=dev), scale=torch.empty(P, dtype=torch.float32, device=dev),
                 hist_doc=torch.empty((P, W), dtype=torch.int32, device=dev))
        intern.gather_samples(pos, P, dict(user=x.user, scale=x.mask, hist_doc=x.hist_doc), g)
        two = self.owner.config.arch in TWO_ID_ARCHS        # the second table's Dropout sees the same mask
        return eng.score_impressions(g['user'], g['hist_doc'], off, x.cand_doc.reshape(-1), eng.eval_doc_table(), out=out,
                                     user_scale=g['scale'], user_scale2=g['scale'] if two else None)

    def predict(self, x, batch_size=None, verbose=0, **_):
        if isinstance(x, CookDeviceData):
            return self._predict_device(x).cpu().numpy().reshape(-1, 1)
        n = len(np.asarray(x[0]))
        C = np.asarray(x[5]).shape[1] if self.is_train else 1
        eng = self.core.engine_infer(C)
        R = eng.B
        out = np.zeros((n, C), dtype=np.float32)
        for s in range(0, n, R):
            rows = np.arange(s, min(n, s + R))
            pad = np.concatenate([rows, np.full(R - len(rows), rows[-1])])
            db = eng.to_device_batch(self._batch(x, pad, C, False))
            probs = eng.forward(db, training=False)
            res = probs if self.is_train else eng.score_sigmoid()
            out[rows] = res[:len(rows)].cpu().numpy()
        return out

    predict_on_batch = predict

    def evaluate(self, x, y, batch_size=None, verbose=0, **_):
        y = np.asarray(y[0] if isinstance(y, (list, tuple)) else y, dtype=np.float64)
        p = self.predict(x).astype(np.float64)          # interned rows: one read-back of the scores
        if self.is_train:
            return keras_like.categorical_loss_accuracy(p, y)
        q, yy = np.clip(p.reshape(-1), 1e-7, 1 - 1e-7), y.reshape(-1)     # binary_crossentropy + utils.auc_roc
        return [float(-(yy * np.log(q) + (1 - yy) * np.log(1 - q)).mean()), metrics.auc_roc(q, yy)]


def _core_attr(name):
    return property(lambda self: getattr(self._core, name), lambda self, v: setattr(self._core, name, v))


class Cook:
    def __init__(self, config: settings.Config):
        self.config = config
        logging.info('[+] loading training data')
        self.training_data = dict(np.load(self.config.train_npz_input))
        logging.info('[-] loaded training data')
        logging.info('[+] loading testing data')
        self.test_data = dict(np.load(self.config.test_npz_input))
        logging.info('[-] loaded testing data')
        self._device_data = None

    def train(self):
        return [self.training_data[x] for x in FEATURES], [self.training_data[x] for x in ['cd_label']]

    def valid(self):
        k = self.config.validation_step
        return [self.test_data[x][:k] for x in FEATURES], [self.test_data[x][:k] for x in ['label']]

    def test(self):
        return [self.test_data[x] for x in FEATURES], [self.test_data[x] for x in ['user', 'impr', 'idx_mask', 'label']]

    # ---- interned rows on the device: training batches gathered there, test rows scored per user group ---------------
    def _interned(self):
        """Intern the titles of both files into one document table (once; needs the built model, whose vertical
        embeddings decide whether the vertical / subvertical ids are part of the key) and keep each file's rows on the
        device as CookDeviceData.  The engines are rebuilt on the table (keras_like._Core.set_doc_table)."""
        import torch
        from .. import intern
        if self._device_data is None:
            assert hasattr(self, 'dv'), 'build_model(0) first'
            dev = torch.device('cuda', torch.cuda.current_device())
            parts = []
            for d in (self.training_data, self.test_data):
                for t in ('ch', 'cd'):
                    parts.append((d[t + '_title'], d[t + '_vert'] if self.dv else None, d[t + '_subvert'] if self.ds else None))
            ids, table = intern.intern(parts, self.L, dev)
            self._core.set_doc_table(**table)
            out = {}
            for i, (name, d) in enumerate((('train', self.training_data), ('test', self.test_data))):
                hist, cand = ids[2 * i], ids[2 * i + 1]
                n = hist.shape[0]
                lab = d['cd_label'] if name == 'train' else d['label']
                mask = np.asarray(d['idx_mask'], dtype=np.float32).reshape(n)
                out[name] = CookDeviceData(intern._upload(d['idx'], dev).reshape(n), torch.as_tensor(mask).to(dev),
                                           hist, cand.reshape(n, -1),
                                           torch.as_tensor(np.asarray(lab, dtype=np.float32).reshape(n, -1)).to(dev), mask)
            self._device_data = out
        return self._device_data

    def device_train(self):
        """train() with the features interned on the device: (CookDeviceData, [cd_label]) for CookModel.fit"""
        return self._interned()['train'], [self.training_data['cd_label']]

    def device_valid(self):
        """valid() interned: the first validation_step test rows, for test_model.evaluate"""
        k = self.config.validation_step
        return self._interned()['test'].head(k), [self.test_data['label'][:k]]

    def device_test(self):
        """test() interned: (CookDeviceData, [user, impr, idx_mask, label])"""
        return self._interned()['test'], [self.test_data[x] for x in ['user', 'impr', 'idx_mask', 'label']]

    def aggregate_test(self, batch_size=None, device=False, log=None):
        """The evaluation tail of `main.py cook` (main.py:216-297): score the test set with test_model and average the
        ranking metrics per impression, per user, and per in-vocabulary / out-of-vocabulary user.  Returns the four
        Result objects of mnexp_b200.evaluation.aggregate and logs them like the reference (through `log`, default
        utils.logging_evaluation).  device: score the interned rows (device_test) and compute every impression's
        metrics in one launch on the device scores."""
        from .. import evaluation, utils
        if not device:
            feature, (users, imprs, mask, y_true) = self.test()
            y_pred = self.test_model.predict(feature, batch_size=batch_size or self.config.batch_size).reshape(-1)
            res = evaluation.aggregate(users, imprs, np.asarray(mask).reshape(-1), y_true, y_pred)
        else:
            import torch
            x, (users, imprs, mask, y_true) = self.device_test()
            scores = self.test_model._predict_device(x)
            starts, ends = evaluation.impression_bounds(users, imprs)
            # the closed impressions are contiguous from row 0
            off = np.append(starts, ends[-1] if len(ends) else 0).astype(np.int32)
            m = metrics.device_ranking_metrics(torch.as_tensor(off).to(scores.device), scores, x.label)
            res = evaluation.aggregate_metrics(users, np.asarray(mask).reshape(-1), y_true, starts, ends, m.cpu().numpy())
        evaluation.log_aggregate(res, log or utils.logging_evaluation)
        return res

    def build_model(self, epoch):
        if epoch == 0:
            self._build_model()
        return self.train_model

    def get_score_model(self, u=None, d=None):
        if self.config.score_model not in ('dot', 'dnn', 'ddot'):
            raise NotImplementedError                      # task/cook.py:210-211
        return self.config.score_model

    def _build_model(self):
        c = self.config
        if c.arch not in COOK_ARCH:
            raise NotImplementedError()                    # task/cook.py:193-194
        if c.news_encoder != 'cnnatt':
            raise NotImplementedError()                    # task/cook.py:96-97
        self.get_score_model()
        word_emb = np.load(c.title_embedding_input + '.npy').astype(np.float32)
        self.W, self.L = self.training_data['ch_title'].shape[1:]
        F, k = c.title_filter_shape
        self.dv = c.vertical_embedding_dim if (c.use_vertical and c.use_vertical_type != 's') else 0
        self.ds = c.subvertical_embedding_dim if (c.use_vertical and c.use_vertical_type != 'v') else 0
        sh = synth.Shape('cook', n_users=N_USER_ROWS, n_news=1, vocab=word_emb.shape[0], L=self.L, W=self.W,
                         K=self.training_data['cd_title'].shape[1] - 1, B=c.batch_size, E=word_emb.shape[1], F=F, k=k,
                         U=c.user_embedding_dim, arch='igru')
        syn = {'vo': 'vo', 'avg': 'niavg', 'gru': 'nigru', 'igru': 'ngru', 'agru': 'pgru', 'ingru': 'igru',
               'inigru': 'iicat'}.get(c.arch, c.arch)      # iavg / iatt / ilstm / inagru / atgru / algru keep their names
        P = synth.make_weights(sh, arch=syn, seed=np.random.randint(1 << 30), word_emb=word_emb, keras_orthogonal=True,
                               score_model=c.score_model, cook=True, dv=self.dv, ds=self.ds)
        if not self.dv:
            P.pop('vert_emb', None)
        if not self.ds:
            P.pop('subvert_emb', None)
        self._core = keras_like._Core(P, c, None, True, c.arch, score_model=c.score_model, flavour='cook', W=self.W,
                                      L=self.L, n_cand=self.training_data['cd_title'].shape[1])
        self.optimizer = self._core.optimizer             # callback decays the learning rate the engines read
        self.train_model = CookModel(self, True)
        self.test_model = CookModel(self, False)
        self.title_encoder = None

    # the core's weights, plan rows and engines under the handler's names
    params = _core_attr('params')
    predict_rows = _core_attr('predict_rows')

    def current_params(self):
        return self.train_model.get_weights_dict()

    def engine(self, B, C, training):
        """the core's training engine of B rows, or its inference engine of B rows and C candidates"""
        if training:
            assert C == self._core.n_train_cand(), (C, self._core.n_train_cand())
            return self._core.engine_train(B)
        return self._core.engine_infer(C, rows=B)

    def callback(self, epoch):
        if epoch in self.config.lrd_on_epochs:             # task/cook.py:282-285
            self.optimizer.lr.value = self.optimizer.lr.value * self.config.learning_rate_decay
