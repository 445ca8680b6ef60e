"""The slice of the Keras Model protocol that the reference's drivers call on the LSTUR models
(SURVEY.md §8b "Model protocol used by callers"), implemented over LsturEngine.

  fit_generator / fit / train_on_batch          main.py:73-78, 172-178
  evaluate_generator / evaluate                 main.py:83-86, 189-192
  predict / predict_on_batch                    task/seq2vec.py:206, main.py:211
  metrics_names, optimizer.lr (+ backend.get_value/set_value)   main.py:87, task/paper.py:498-499
  get_layer(name), get_weights / set_weights, summary()         task/test_pipeline.py:28,87; utils.py:70,79

Inputs are host numpy arrays in the reference's order: [user(B,) , clicked(B,W,L), cand_0(B,L) .. cand_K(B,L)]
(user omitted for the classes without a user-ID embedding), target (B,1+K) one-hot.  train_on_batch / fit_generator /
evaluate / evaluate_generator of the softmax family also take batches assembled on the device (assemble.DeviceBatch,
the task handlers' device_train / device_valid): doc ids go to the engine as they are, the target is the positive in
column 0, and vertical ids come from the engine's doc_vert table.
"""
import numpy as np
import torch

from .assemble import DeviceBatch
from .engine import LsturEngine


class Variable:
    def __init__(self, value):
        self.value = float(value)


class backend:
    """keras.backend.get_value / set_value on optimizer.lr (task/paper.py:498-499)."""
    @staticmethod
    def get_value(v):
        return v.value

    @staticmethod
    def set_value(v, x):
        v.value = float(x)


class Adam:
    def __init__(self, lr=0.001):
        self.lr = Variable(lr)


class History:
    def __init__(self):
        self.history = {}
        self.epoch = []


class _Core:
    """Weights + engines shared by `model` (softmax/CE training graph) and `test_model` (sigmoid scoring graph)."""

    def __init__(self, params, cfg, doc_tokens, has_user, arch, predict_rows=256, score_model='dot', loss='softmax',
                 flavour='paper', has_vert=False):
        self.params, self.cfg, self.doc_tokens, self.has_user, self.arch = params, cfg, doc_tokens, has_user, arch
        self.score_model, self.loss, self.flavour = score_model, loss, flavour
        self.has_vert = has_vert        # inputs carry vertical ids next to the titles (task/paper.py:1205-1232)
        self.optimizer = Adam(cfg.learning_rate)
        self.train_engine = None
        self.infer_engines = {}
        self.predict_rows = predict_rows
        self.step_seed = 0
        self.freeze_encoder = False     # --enable-pretrain-encoder without --pretrain-encoder-trainable (task/paper.py:103-106)
        self.doc_vert = None            # (n_docs,) vertical of every document: vertical ids of device-assembled batches

    def precision(self):
        p = getattr(self.cfg, 'precision', 'auto')
        if p != 'auto':
            return p
        from . import _lib
        ks, E, F = self.params['conv_w'].shape
        ok = _lib.load().lstur_tc_supported(self.cfg.title_shape, E, F, ks)
        return 'fp16_tc' if ok else 'fp32'

    def engine_train(self, B):
        e = self.train_engine
        if e is None or e.B != B:
            old = e
            if e is not None:                      # batch size changed: carry the weights (and optimizer state, below) over
                self.params = e.get_weights_dict()
            c = self.cfg
            self.train_engine = LsturEngine(
                self.params, B, c.window_size, self.n_train_cand(), c.title_shape, arch=self.arch,
                dropout=c.dropout, lr=c.learning_rate, recurrent_activation=c.recurrent_activation,
                precision=self.precision(), doc_tokens=self.doc_tokens, training=True,
                sparse_user_adam=bool(c.sparse_user_adam), score_model=self.score_model,
                trainable_word_emb=bool(getattr(c, 'textual_embedding_trainable', False)), doc_vert=self.doc_vert,
                **self.head_kw())
            if old is not None:
                self.train_engine.adopt_state_from(old)
            self.train_engine.freeze_encoder = self.freeze_encoder
            self.infer_engines = {}
        return self.train_engine

    def engine_infer(self, C, rows=None):
        rows = rows or self.predict_rows
        key = C if rows == self.predict_rows else (C, rows)
        if key not in self.infer_engines:
            c = self.cfg
            # share the CURRENT training engine's device weights whatever its batch size (never rebuild it from here:
            # that would discard its optimizer state); create one only if training has not started
            base = self.train_engine if self.train_engine is not None else self.engine_train(c.batch_size)
            self.infer_engines[key] = LsturEngine(
                self.params, rows, c.window_size, C, c.title_shape, arch=self.arch, dropout=0.0,
                recurrent_activation=c.recurrent_activation, precision=self.precision(), training=False,
                share_weights_from=base, score_model=self.score_model, **self.head_kw())
        return self.infer_engines[key]

    def stage_tokens(self, name, arr, slot=0):
        """host token array (the reference feeds float64, document.py:39) -> int32 in a reusable PINNED buffer: the cast is
        one numpy pass (float64 -> int32, ids < 2^24 are exact) and the upload an asynchronous 4-byte-per-id copy instead
        of a pageable 8-byte-per-id copy followed by a cast on the device.  `slot` selects one of several buffer sets:
        fit_generator stages batch i+1 while the copy / kernels of batch i may still be in flight."""
        arr = np.asarray(arr)
        key = (name, arr.shape, slot)
        pin = self.__dict__.setdefault('_pinned', {})
        if key not in pin:
            pin[key] = torch.empty(arr.shape, dtype=torch.int32).pin_memory()
        np.copyto(pin[key].numpy(), arr, casting='unsafe')
        return pin[key]

    def dp(self, eng):
        """mnexp_b200.dist.DataParallel around the training engine when torch.distributed is initialised with more than one
        rank (one process per GPU, launched with torchrun): every process runs the same task / model code on its OWN batches
        of config.batch_size rows, the gradients are exchanged every step (dense arena all-reduce + user-row all-gather,
        dist.py) and the logged loss / accuracy are the means over the ranks.  None in a single process."""
        import torch.distributed as tdist
        if not (tdist.is_available() and tdist.is_initialized() and tdist.get_world_size() > 1):
            return None
        cached = self.__dict__.get('_dp')
        if cached is None or cached.eng is not eng:
            from .dist import DataParallel
            cached = self.__dict__['_dp'] = DataParallel(eng)
        return cached

    def n_train_cand(self):
        return 1 if self.loss == 'bce' else 1 + self.cfg.negative_samples

    def head_kw(self):
        kw = dict(flavour=self.flavour, loss=self.loss, gain=self.cfg.gain, bce_neg=self.cfg.negative_samples)
        if 'vs_w1' in self.params:      # ...VertSup: loss_weights=[1, config.gain] (task/paper.py:985)
            kw['aux_gain'] = self.cfg.gain
        return kw

    def split_inputs(self, x, n_cand):
        """[user?, clicked, clicked_vert?, cand_0..cand_{C-1}, cand_vert_0..?] -> user, clicked, cand (B,C,L), verts."""
        x = list(x)
        user = np.asarray(x.pop(0)).reshape(-1) if self.has_user else None
        clicked = np.asarray(x.pop(0))
        verts = None
        if self.has_vert:
            hist_vert = np.asarray(x.pop(0)).reshape(clicked.shape[0], -1)
            cand_vert = np.stack([np.asarray(v).reshape(-1) for v in x[n_cand:2 * n_cand]], axis=1)
            verts = (hist_vert, cand_vert)
        cand = np.stack([np.asarray(c) for c in x[:n_cand]], axis=1)     # (B, C, L)
        if user is None:
            user = np.zeros(clicked.shape[0], dtype=np.int32)
        return user, clicked, cand, verts

    def device_inputs(self, batch, n_cand, with_label=True):
        """assemble.DeviceBatch -> engine batch dict: the doc ids as they are (user zeroed for the classes without a
        user-ID embedding, as split_inputs does), the target = the positive in column 0."""
        if self.loss == 'bce':
            raise ValueError('device-assembled batches feed the softmax family only')
        B = batch.B
        assert batch.cand_doc.shape[1] == n_cand, 'the batch has %d candidates per row, the model %d' % (batch.cand_doc.shape[1], n_cand)
        dev = batch.hist_doc.device
        cache = self.__dict__.setdefault('_device_consts', {})
        user = batch.user
        if not self.has_user:
            if ('zeros', B) not in cache:
                cache[('zeros', B)] = torch.zeros(B, dtype=torch.int32, device=dev)
            user = cache[('zeros', B)]
        db = dict(user=user, hist_doc=batch.hist_doc, cand_doc=batch.cand_doc)
        if with_label:
            if ('label', B, n_cand) not in cache:
                lab = torch.zeros((B, n_cand), dtype=torch.float32, device=dev)
                lab[:, 0] = 1.0
                cache[('label', B, n_cand)] = lab
            db['label'] = cache[('label', B, n_cand)]
        return db

    def device_user_scale(self, B, device):
        """dgru's Dropout(0.5, noise_shape=(None, 1)) multipliers drawn on the device (0 or 2 per row), from a generator
        seeded once from numpy's global state."""
        g = self.__dict__.get('_scale_gen')
        if g is None:
            g = self.__dict__['_scale_gen'] = torch.Generator(device=device)
            g.manual_seed(int(np.random.randint(1 << 31)))
        return (torch.rand(B, device=device, generator=g) >= 0.5).to(torch.float32) * 2.0


class Model:
    """`model` (train=True: probabilities over the 1+K candidates) or `test_model` (sigmoid of one candidate)."""

    def __init__(self, core, train, name='model'):
        self.core, self.is_train, self.name = core, train, name
        self.metrics_names = ['loss', 'categorical_accuracy'] if train else ['loss']
        if core.loss == 'bce':                   # metrics=[utils.auc_roc], task/paper.py:250-255
            self.metrics_names = ['loss', 'auc_roc']
        self.layers = {}

    @property
    def optimizer(self):
        return self.core.optimizer

    # ---- training ---------------------------------------------------------------------------
    def _enqueue_train(self, x, y, slot=0, copy_stream=None, n_valid=None):
        """Stage one batch (pinned buffer set `slot`) and enqueue forward + backward + Adam plus an asynchronous copy of
        [loss, categorical_accuracy] into a pinned result; the host does not wait for the device.  -> handle for
        _finish_train.  (The weighted-BCE family reports a host-side AUC of the batch's scores, so its handle keeps the
        device tensors and has to be finished before the next step is enqueued.)"""
        assert self.is_train, 'test_model is not compiled for training'
        core = self.core
        C = core.n_train_cand()
        if isinstance(x, DeviceBatch):      # assembled on the device: nothing to stage or upload
            eng = core.engine_train(x.B)
            eng.lr = core.optimizer.lr.value
            db = core.device_inputs(x, C)
            if core.arch == 'dgru':
                db['user_scale'] = core.device_user_scale(x.B, eng.device)
        else:
            user, clicked, cand, verts = core.split_inputs(x, C)
            eng = core.engine_train(clicked.shape[0])
            eng.lr = core.optimizer.lr.value
            batch = dict(user=user, hist_tok=core.stage_tokens('hist', clicked, slot), cand_tok=core.stage_tokens('cand', cand, slot),
                         label=np.asarray(y, dtype=np.float32).reshape(len(clicked), C))
            if verts is not None:
                batch['hist_vert'], batch['cand_vert'] = verts
            if core.arch == 'dgru':     # Dropout(0.5, noise_shape=(None, 1)) on the user vector (task/paper.py:609)
                batch['user_scale'] = (np.random.random(clicked.shape[0]) >= 0.5).astype(np.float32) * 2.0
            if copy_stream is None:
                db = eng.to_device_batch(batch, non_blocking=True)
            else:       # upload on a side stream: it runs under the previous step's kernels; this step waits for it
                main = torch.cuda.current_stream()
                with torch.cuda.stream(copy_stream):
                    db = eng.to_device_batch(batch, non_blocking=True)
                    ready = torch.cuda.Event()
                    ready.record(copy_stream)
                main.wait_event(ready)
                for t in db.values():
                    t.record_stream(main)
        nv = eng.B if n_valid is None else int(n_valid)      # rows beyond nv are padding with an all-zero target (fit)
        dp = core.dp(eng)
        if dp is None:
            loss = eng.train_step(db, grad_scale=None if nv == eng.B else 1.0 / nv)
        else:
            assert nv == eng.B, 'data-parallel training needs full batches on every rank'
            loss = dp.train_step(db)
        probs = eng.view('probs').reshape(eng.B, eng.C)
        if core.loss == 'bce':
            return ('bce', loss, probs, y)
        acc = (probs[:nv].argmax(1) == db['label'][:nv].argmax(1)).float().mean()
        out = torch.stack([loss[0] * (eng.B / nv), acc])
        if dp is not None:                                   # what is logged: the mean over the ranks' equal-sized batches
            import torch.distributed as tdist
            tdist.all_reduce(out, group=dp.group)
            out = out / dp.world
        res = core.__dict__.setdefault('_results', {})
        if slot not in res:
            res[slot] = torch.empty(2, dtype=torch.float32).pin_memory()
        res[slot].copy_(out, non_blocking=True)
        done = torch.cuda.Event()
        done.record()
        return ('ce', res[slot], done)

    def _finish_train(self, handle):
        if handle[0] == 'bce':
            from . import metrics
            _, loss, probs, y = handle
            return [float(loss[0]), metrics.auc_roc(probs.reshape(-1).cpu().numpy(), np.asarray(y).reshape(-1))]
        _, res, done = handle
        done.synchronize()
        return [float(res[0]), float(res[1])]

    def train_on_batch(self, x, y=None):
        """x, y: host inputs and targets, or x = an assemble.DeviceBatch (no y)."""
        return self._finish_train(self._enqueue_train(x, y))

    def fit_generator(self, generator, steps_per_epoch, epochs=1, initial_epoch=0, verbose=0, **_):
        """main.py:73-78.  Software-pipelined by one step: while the device runs step i, the host pulls batch i+1 from the
        generator, casts it into the other pinned buffer set, uploads it on a side stream and enqueues step i+1; only then
        does it read step i's [loss, accuracy].  The sequence of updates and the logged averages are those of a plain train_on_batch loop."""
        h = History()
        pipelined = type(self).train_on_batch is Model.train_on_batch and self.core.loss != 'bce'
        copy_stream = None
        if pipelined:
            if '_copy_stream' not in self.core.__dict__:
                self.core.__dict__['_copy_stream'] = torch.cuda.Stream()
            copy_stream = self.core.__dict__['_copy_stream']
        for epoch in range(initial_epoch, epochs):
            tot = np.zeros(len(self.metrics_names))
            pending = None
            for step in range(steps_per_epoch):
                x, y = _unpack(next(generator))
                if not pipelined:
                    tot += self.train_on_batch(x, y)
                    continue
                handle = self._enqueue_train(x, y, slot=step & 1, copy_stream=copy_stream)
                if pending is not None:
                    tot += self._finish_train(pending)
                pending = handle
            if pending is not None:
                tot += self._finish_train(pending)
            h.epoch.append(epoch)
            for k, v in zip(self.metrics_names, tot / max(1, steps_per_epoch)):
                h.history.setdefault(k, []).append(float(v))
        return h

    def fit(self, x, y, batch_size=32, epochs=1, initial_epoch=0, shuffle=True, verbose=0, **_):
        y = y[0] if isinstance(y, (list, tuple)) else y
        n = len(y)
        h = History()
        for epoch in range(initial_epoch, epochs):
            order = np.random.permutation(n) if shuffle else np.arange(n)
            tot, k = np.zeros(2), 0
            pad_ok = self.core.loss != 'bce' and type(self).train_on_batch is Model.train_on_batch
            for s in range(0, n, batch_size):
                idx = order[s:s + batch_size]
                m = len(idx)
                if m < batch_size and not pad_ok:
                    break           # weighted BCE has no neutral target: the ragged tail of the sigmoid family is dropped
                yb = np.asarray(y)[idx]
                if m < batch_size:
                    # Keras trains the ragged last batch too; the plan is per batch size, so the m samples run as
                    # batch_size rows: padding rows repeat the first sample under an all-zero target (zero loss and
                    # gradient under categorical cross-entropy), gradient scale 1 / m
                    idx = np.concatenate([idx, np.full(batch_size - m, idx[0])])
                    yb = np.concatenate([yb, np.zeros((batch_size - m,) + yb.shape[1:], dtype=yb.dtype)])
                xb = [np.asarray(a)[idx] for a in x]
                r = self._finish_train(self._enqueue_train(xb, yb, n_valid=m)) if pad_ok else self.train_on_batch(xb, yb)
                tot += np.asarray(r) * m
                k += m                  # Keras logs the sample-weighted mean over the batches
            h.epoch.append(epoch)
            for name, v in zip(self.metrics_names, tot / max(1, k)):
                h.history.setdefault(name, []).append(float(v))
        return h

    # ---- inference --------------------------------------------------------------------------
    SHARED_C = 32          # candidates per row on the per-impression path (the plan's limit)

    def _score_one_impression(self, user, clicked, cand, verts):
        """Seq2Vec.test (task/seq2vec.py:202-206) feeds ONE impression per predict call: every row repeats the same user
        and click history next to a different candidate, so the reference encodes the history n times.  Here the history
        is encoded once per group of up to 32 candidates: rows = ceil(n / 32), candidates padded with the pad title."""
        core = self.core
        n, L = cand.shape[0], cand.shape[2]
        C = self.SHARED_C
        rows = (n + C - 1) // C
        eng = core.engine_infer(C, rows=8)
        out = np.zeros(n, dtype=np.float32)
        for r0 in range(0, rows, eng.B):
            m = min(eng.B, rows - r0)
            u = np.zeros(eng.B, dtype=np.int32); u[:m] = user[0]
            h = np.zeros((eng.B,) + clicked.shape[1:], dtype=np.int32); h[:m] = clicked[0]
            c = np.zeros((eng.B, C, L), dtype=np.int32)
            k0, k1 = r0 * C, min(n, (r0 + m) * C)
            c.reshape(-1, L)[:k1 - k0] = cand[k0:k1, 0]
            b = dict(user=u, hist_tok=h, cand_tok=c)
            if verts is not None:
                hv = np.zeros((eng.B, verts[0].shape[1]), dtype=np.int32); hv[:m] = verts[0][0]
                cv = np.zeros((eng.B, C), dtype=np.int32)
                cv.reshape(-1)[:k1 - k0] = verts[1][k0:k1, 0]
                b['hist_vert'], b['cand_vert'] = hv, cv
            probs = eng.forward(eng.to_device_batch(b), training=False)
            s = probs if core.loss == 'bce' else eng.score_sigmoid()
            out[k0:k1] = s.reshape(-1)[:k1 - k0].cpu().numpy()
        return out.reshape(n, 1)

    def _forward_chunks(self, x, n_cand):
        core = self.core
        user, clicked, cand, verts = core.split_inputs(x, n_cand)
        n = clicked.shape[0]
        if (n_cand == 1 and n > 1 and not self.is_train and core.loss != 'bce' and np.all(user == user[0])
                and np.array_equal(clicked, np.broadcast_to(clicked[:1], clicked.shape))
                and (verts is None or np.array_equal(verts[0], np.broadcast_to(verts[0][:1], verts[0].shape)))):
            return self._score_one_impression(user, clicked, cand, verts)
        eng = core.engine_infer(n_cand)
        R = eng.B
        outs = []
        for s in range(0, n, R):
            m = min(R, n - s)
            u = np.zeros(R, dtype=np.int32); u[:m] = user[s:s + m]
            h = np.zeros((R,) + clicked.shape[1:], dtype=np.int32); h[:m] = clicked[s:s + m]
            c = np.zeros((R,) + cand.shape[1:], dtype=np.int32); c[:m] = cand[s:s + m]
            b = dict(user=u, hist_tok=h, cand_tok=c)
            if verts is not None:
                hv = np.zeros((R, verts[0].shape[1]), dtype=np.int32); hv[:m] = verts[0][s:s + m]
                cv = np.zeros((R, n_cand), dtype=np.int32); cv[:m] = verts[1][s:s + m]
                b['hist_vert'], b['cand_vert'] = hv, cv
            db = eng.to_device_batch(b)
            probs = eng.forward(db, training=False)
            out = probs if (self.is_train or core.loss == 'bce') else eng.score_sigmoid()
            outs.append(out[:m].cpu().numpy().copy())
        return np.concatenate(outs) if outs else np.zeros((0, n_cand), dtype=np.float32)

    def predict(self, x, batch_size=None, **_):
        C = self.core.n_train_cand() if self.is_train else 1
        return self._forward_chunks(x, C)

    predict_on_batch = predict

    def _predict_device(self, batch):
        """probabilities (B, 1+K) of an assemble.DeviceBatch through the same inference engine and row chunks as predict
        on host arrays (pad rows = doc 0, the all-zero title)."""
        core = self.core
        if not self.is_train:
            raise ValueError('device-assembled batches carry 1+K candidates: evaluate them with `model`, not test_model')
        C = core.n_train_cand()
        src = core.device_inputs(batch, C, with_label=False)
        eng = core.engine_infer(C)
        R, n = eng.B, batch.B
        outs = []
        for s in range(0, n, R):
            m = min(R, n - s)
            db = {}
            for k, v in src.items():
                t = torch.zeros((R,) + tuple(v.shape[1:]), dtype=v.dtype, device=v.device)
                t[:m] = v[s:s + m]
                db[k] = t
            outs.append(eng.forward(db, training=False)[:m].cpu().numpy().copy())
        return np.concatenate(outs)

    def evaluate(self, x, y=None, batch_size=None, verbose=0, **_):
        if isinstance(x, DeviceBatch):
            p = self._predict_device(x).astype(np.float64)
            y = np.zeros(p.shape, dtype=np.float64)
            y[:, 0] = 1.0
        else:
            y = np.asarray(y[0] if isinstance(y, (list, tuple)) else y, dtype=np.float64)
            p = self.predict(x).astype(np.float64)
        if self.core.loss == 'bce':              # Seq2Vec.loss + utils.auc_roc
            from . import metrics
            K, yy, q = float(self.core.cfg.negative_samples), y.reshape(-1), p.reshape(-1)
            l = -0.5 * (1 + K) * np.mean(yy * np.log(q + 1e-8) * self.core.cfg.gain + (1 - yy) * np.log(1 - q + 1e-8) / K)
            return [float(l), metrics.auc_roc(q, yy)]
        if self.is_train:
            q = np.clip(p / p.sum(-1, keepdims=True), 1e-7, 1 - 1e-7)
            return [float((-(y * np.log(q)).sum(-1)).mean()), float((p.argmax(1) == y.argmax(1)).mean())]
        q = np.clip(p.reshape(-1), 1e-7, 1 - 1e-7)
        yy = y.reshape(-1)
        return [float(-(yy * np.log(q) + (1 - yy) * np.log(1 - q)).mean())]

    def evaluate_generator(self, generator, steps, verbose=0, **_):
        tot = np.zeros(len(self.metrics_names))
        for _ in range(steps):
            x, y = _unpack(next(generator))
            tot += self.evaluate(x, y)
        return list(tot / max(1, steps))

    # ---- weights / structure ------------------------------------------------------------------
    WEIGHT_ORDER = ('word_emb', 'conv_w', 'conv_b', 'att_w', 'att_b', 'dense_w', 'dense_b', 'vert_emb', 'subvert_emb', 'user_emb',
                    'user_emb2',
                    'gru_wx', 'gru_wh', 'gru_b', 'lstm_wx', 'lstm_wh', 'lstm_b', 'uatt_w', 'uatt_b', 'alpha', 'con_w', 'con_b', 'sh_w', 'sh_b', 'so_w', 'so_b', 'su_w', 'su_b', 'sd_w',
                    'sd_b', 'vs_w1', 'vs_b1', 'vs_w2', 'vs_b2', 'vcls_w', 'vcls_b')

    def _current(self):
        e = self.core.train_engine
        return e.get_weights_dict() if e is not None else self.core.params

    def get_weights(self):
        """List of numpy arrays in layer-creation order of the reference graph (embedding, conv, attention, dense,
        user embedding, GRU kernel/recurrent/bias, concat-Dense).  The Keras pickle order cannot be verified
        offline (SURVEY.md §7 risks); att_w is exported with Keras' (F,1) shape."""
        w = self._current()
        out = []
        for k in self.WEIGHT_ORDER:
            if k in w:
                a = np.asarray(w[k])
                out.append(a.reshape(-1, 1) if k == 'att_w' else a.reshape(1) if k == 'att_b' else a)
        return out

    def weight_specs(self):
        """[(name, shape)] in get_weights() order."""
        return [(k, tuple(int(d) for d in a.shape)) for k, a in
                zip([k for k in self.WEIGHT_ORDER if k in self._current()], self.get_weights())]

    def to_json(self):
        import json
        c = self.core
        specs = self.weight_specs()
        return json.dumps(dict(class_name='mnexp_b200.keras_like.Model', name=self.name, arch=c.arch, flavour=c.flavour,
                               score_model=c.score_model, loss=c.loss, weight_names=[n for n, _ in specs],
                               weight_shapes=[list(s) for _, s in specs]))

    def set_weights(self, weights):
        cur = self._current()
        names = [k for k in self.WEIGHT_ORDER if k in cur]
        assert len(names) == len(weights), 'expected %d arrays (%s)' % (len(names), names)
        new = {k: np.asarray(a, dtype=np.float32).reshape(np.asarray(cur[k]).shape) for k, a in zip(names, weights)}
        self.core.params = dict(cur, **new)
        if self.core.train_engine is not None:
            self.core.train_engine.set_weights_dict(self.core.params)

    def get_layer(self, name):
        return self.layers[name]

    def summary(self):
        w = self._current()
        lines = ['%-12s %-18s %d' % (k, tuple(np.asarray(v).shape), np.asarray(v).size) for k, v in w.items()]
        print('\n'.join(lines))
        print('Total params: %d' % sum(np.asarray(v).size for v in w.values()))


class VertSupModel(Model):
    """`model` of Seq2VecPaperSoftmaxDaysIdVertSup (task/paper.py:981-987): outputs [ranking (B,1+K), vert (B,W+1+K,n_vert)],
    losses [categorical CE, categorical CE], loss_weights [1, gain].  Targets arrive as [one-hot clicks, one-hot verticals of
    the W history slots followed by the 1+K candidates] (:897-902)."""

    def __init__(self, core, name='model'):
        Model.__init__(self, core, True, name)
        self.metrics_names = ['loss', 'ranking_loss', 'vert_loss', 'ranking_categorical_accuracy', 'vert_categorical_accuracy']

    def _vert_ids(self, y_vert, W):
        ids = np.asarray(y_vert).argmax(-1).astype(np.int32)          # to_categorical inverse
        return ids[:, :W], ids[:, W:]

    def _metrics(self, eng, db):
        probs = eng.view('probs').reshape(eng.B, eng.C)
        acc = float((probs.argmax(1) == db['label'].argmax(1)).float().mean())
        n = eng.B * (eng.W + eng.C)
        vp = eng.view('vs_probs').reshape(n, eng.aux_nv)
        if 'hist_vert' in db:
            lab = torch.cat([db['hist_vert'].reshape(-1), db['cand_vert'].reshape(-1)])
        else:                       # device batch: the verticals of its documents
            lab = eng.doc_vert[torch.cat([db['hist_doc'].reshape(-1), db['cand_doc'].reshape(-1)]).long()]
        vacc = float((vp.argmax(1) == lab).float().mean())
        main, aux = eng.loss(), eng.aux_loss()
        return [main + eng.aux_gain * aux, main, aux, acc, vacc]

    def train_on_batch(self, x, y=None):
        core = self.core
        C = core.n_train_cand()
        if isinstance(x, DeviceBatch):
            eng = core.engine_train(x.B)
            eng.lr = core.optimizer.lr.value
            db = core.device_inputs(x, C)
            eng.train_step(db)
            return self._metrics(eng, db)
        user, clicked, cand, _ = core.split_inputs(x, C)
        eng = core.engine_train(clicked.shape[0])
        eng.lr = core.optimizer.lr.value
        hv, cv = self._vert_ids(y[1], clicked.shape[1])
        batch = dict(user=user, hist_tok=clicked, cand_tok=cand, hist_vert=hv, cand_vert=cv,
                     label=np.asarray(y[0], dtype=np.float32).reshape(len(clicked), C))
        db = eng.to_device_batch(batch)
        eng.train_step(db)
        return self._metrics(eng, db)

    def evaluate(self, x, y=None, batch_size=None, verbose=0, **_):
        core = self.core
        C = core.n_train_cand()
        if isinstance(x, DeviceBatch):
            eng = core.engine_train(x.B)
            db = core.device_inputs(x, C)
            eng.forward(db, training=False)
            return self._metrics(eng, db)
        user, clicked, cand, _ = core.split_inputs(x, C)
        eng = core.engine_train(clicked.shape[0])
        hv, cv = self._vert_ids(y[1], clicked.shape[1])
        db = eng.to_device_batch(dict(user=user, hist_tok=clicked, cand_tok=cand, hist_vert=hv, cand_vert=cv,
                                      label=np.asarray(y[0], dtype=np.float32).reshape(len(clicked), C)))
        eng.forward(db, training=False)
        return self._metrics(eng, db)

    def predict(self, x, batch_size=None, **_):
        """[ranking probabilities (n, 1+K), vertical probabilities (n, W+1+K, n_vert)] like the two-output Keras model."""
        core = self.core
        C = core.n_train_cand()
        user, clicked, cand, _ = core.split_inputs(x, C)
        eng = core.engine_train(clicked.shape[0])
        z = np.zeros((clicked.shape[0], clicked.shape[1]), dtype=np.int32)
        db = eng.to_device_batch(dict(user=user, hist_tok=clicked, cand_tok=cand, hist_vert=z,
                                      cand_vert=np.zeros((clicked.shape[0], C), dtype=np.int32)))
        probs = eng.forward(db, training=False).cpu().numpy().copy()
        B, W = eng.B, eng.W
        vp = eng.view('vs_probs').reshape(B * (W + C), eng.aux_nv).cpu().numpy()
        return [probs, np.concatenate([vp[:B * W].reshape(B, W, -1), vp[B * W:].reshape(B, C, -1)], 1)]

    predict_on_batch = predict


class VertModel:
    """`vert_model` of Seq2VecPaperSoftmaxDaysIdVertAlt (task/paper.py:1128-1136): title (n,L) -> softmax over the
    verticals, categorical cross-entropy, its own Adam; shares the doc_encoder weights with the click model."""

    def __init__(self, core, name='vert_model'):
        self.core, self.name = core, name
        self.metrics_names = ['loss', 'categorical_accuracy']
        self.optimizer = Adam(core.cfg.learning_rate)
        self.layers = {}

    def _engine(self):
        c = self.core.cfg
        return self.core.train_engine if self.core.train_engine is not None else self.core.engine_train(c.batch_size)

    def _chunks(self, eng, n):
        cap = eng.B * (eng.W + eng.C)
        return [(s, min(cap, n - s)) for s in range(0, n, cap)]

    def train_on_batch(self, x, y):
        eng = self._engine()
        x = np.asarray(x[0] if isinstance(x, (list, tuple)) else x)
        lab = np.asarray(y[0] if isinstance(y, (list, tuple)) else y).argmax(-1)
        assert len(x) <= eng.B * (eng.W + eng.C), 'vertical batch exceeds the plan\'s title capacity'
        loss, acc = eng.title_cls_train_step(x, lab, lr=self.optimizer.lr.value)
        return [float(loss[0]), float(acc)]

    def fit_generator(self, generator, steps_per_epoch, epochs=1, initial_epoch=0, verbose=0, **_):
        h = History()
        for epoch in range(initial_epoch, epochs):
            tot = np.zeros(2)
            for _ in range(steps_per_epoch):
                x, y = next(generator)
                tot += self.train_on_batch(x, y)
            h.epoch.append(epoch)
            for k, v in zip(self.metrics_names, tot / max(1, steps_per_epoch)):
                h.history.setdefault(k, []).append(float(v))
        return h

    def predict(self, x, batch_size=None, **_):
        eng = self._engine()
        x = np.asarray(x[0] if isinstance(x, (list, tuple)) else x)
        out = []
        for s, m in self._chunks(eng, len(x)):
            out.append(eng.title_cls_forward(x[s:s + m], np.zeros(m, dtype=np.int32)).cpu().numpy().copy())
        return np.concatenate(out) if out else np.zeros((0, eng.cls_nv), dtype=np.float32)

    predict_on_batch = predict

    def evaluate(self, x, y, batch_size=None, verbose=0, **_):
        y = np.asarray(y[0] if isinstance(y, (list, tuple)) else y, dtype=np.float64)
        p = self.predict(x).astype(np.float64)
        q = np.clip(p / p.sum(-1, keepdims=True), 1e-7, 1 - 1e-7)
        return [float((-(y * np.log(q)).sum(-1)).mean()), float((p.argmax(1) == y.argmax(1)).mean())]

    def evaluate_generator(self, generator, steps, verbose=0, **_):
        tot = np.zeros(2)
        for _ in range(steps):
            x, y = next(generator)
            tot += self.evaluate(x, y)
        return list(tot / max(1, steps))


def _unpack(item):
    """a generator's item -> (x, y): an assemble.DeviceBatch carries its own target"""
    return (item, None) if isinstance(item, DeviceBatch) else item


class _InputLayer:
    """The slice of keras.layers.InputLayer the reference reads: `.input_shape` (task/test_pipeline.py:29, 88)."""

    def __init__(self, name, shape):
        self.name, self.input_shape, self.output_shape = name, shape, shape


class DocEncoderModel:
    """`doc_encoder` layer: (n, L) token ids -> (n, U) news vectors (task/paper.py:160)."""
    name = 'doc_encoder'

    def __init__(self, core):
        self.core = core
        self.layers = [_InputLayer('doc_encoder_input', (None, core.cfg.title_shape))]

    ENC_ORDER = ('word_emb', 'conv_w', 'conv_b', 'att_w', 'att_b', 'dense_w', 'dense_b')   # keras get_weights() order of the
                                                                                           # encoder graph, task/paper.py:132-160
    trainable = True       # `encoder.trainable = False` (task/paper.py:105-106) freezes the title encoder's weights

    def __setattr__(self, k, v):
        object.__setattr__(self, k, v)
        if k == 'trainable' and 'core' in self.__dict__:
            self.core.freeze_encoder = not v
            if self.core.train_engine is not None:
                self.core.train_engine.freeze_encoder = not v

    def _current(self):
        e = self.core.train_engine
        return e.get_weights_dict() if e is not None else self.core.params

    def get_weights(self):
        w = self._current()
        return [np.asarray(w[k]).reshape(-1, 1) if k == 'att_w' else np.asarray(w[k]).reshape(1) if k == 'att_b' else np.asarray(w[k])
                for k in self.ENC_ORDER if k in w]

    def weight_specs(self):
        return [(k, tuple(int(d) for d in a.shape)) for k, a in zip([k for k in self.ENC_ORDER if k in self._current()], self.get_weights())]

    def to_json(self):
        import json
        specs = self.weight_specs()
        return json.dumps(dict(class_name='mnexp_b200.keras_like.DocEncoderModel', name=self.name, arch='doc_encoder',
                               weight_names=[n for n, _ in specs], weight_shapes=[list(s) for _, s in specs]))

    def set_weights(self, weights):
        cur = self._current()
        names = [k for k in self.ENC_ORDER if k in cur]
        assert len(names) == len(weights), 'expected %d arrays (%s)' % (len(names), names)
        new = {k: np.asarray(a, dtype=np.float32).reshape(np.asarray(cur[k]).shape) for k, a in zip(names, weights)}
        self.core.params = dict(cur, **new)
        if self.core.train_engine is not None:
            self.core.train_engine.set_weights_dict(self.core.params)

    def predict(self, titles, batch_size=None, **_):
        """title tokens straight through the news-encoder kernels (lstur_encode_titles): no history, no scorer"""
        core = self.core
        titles = np.asarray(titles)
        eng = core.engine_infer(1)
        dv = eng.encode_titles(titles)
        return dv[:, :eng.cfg.Dd].cpu().numpy().copy()      # the doc_encoder layer is the title encoder alone (no vertical columns)


class UserEncoderModel:
    """`user_encoder` layer (task/paper.py:584-633): inputs [user (n,1)] + `user_clicked_vec` (n, W, D) -> (n, U); the
    reference's decomposed pipeline fetches it with get_layer('user_encoder') and reads the shape of its
    'user_clicked_vec' input (task/test_pipeline.py:87-88)."""
    name = 'user_encoder'

    def __init__(self, core, doc_dim):
        self.core = core
        self._inputs = {'user_clicked_vec': _InputLayer('user_clicked_vec', (None, core.cfg.window_size, doc_dim))}
        if core.has_user:
            self._inputs['user'] = _InputLayer('user', (None, 1))
        self.layers = list(self._inputs.values())

    def get_layer(self, name):
        return self._inputs[name]

    def predict(self, x, batch_size=None, **_):
        core = self.core
        if isinstance(x, (list, tuple)):
            user, vecs = (x[0], x[1]) if len(x) == 2 else (None, x[0])
        else:
            user, vecs = None, x
        vecs = np.asarray(vecs, dtype=np.float32)
        if user is None:
            user = np.zeros(vecs.shape[0], dtype=np.int32)
        eng = core.engine_infer(1)
        return eng.encode_users(np.asarray(user).reshape(-1), vecs).cpu().numpy().copy()
