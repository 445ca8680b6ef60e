"""Model-builder surface of the reference's task/paper.py for the LSTUR path, backed by the CUDA engine.

Same class names, hyper-parameters (settings.Config), arch names, builder hooks and forward / loss / score semantics:

  Seq2VecPaper            data side: Impression (pos/neg/time), _load_data (task/paper.py:6-35)
  Seq2VecPaperSoftmax     (1+K)-way softmax CE, news encoder cnnatt, user encoder arch 'gru' (task/paper.py:386-524)
  Seq2VecPaperSoftmaxId   = LSTUR: user-ID embedding; arch igru (ini), gru / hgru / ngru / dgru (con), pgru, nigru,
                            vo (task/paper.py:527-665)

`get_doc_encoder / get_user_encoder / score_encoder / _score_model / _build_model / build_model / callback` keep the
reference's names and effects; the Keras graph they used to assemble is the fixed-function plan of
csrc/engine.cu.  Unsupported options raise the reference's own exceptions.
"""
import logging
import random
from datetime import datetime, timedelta

import numpy as np
from .. import keras_like, metrics, synth, utils
from .seq2vec import Seq2Vec


class Seq2VecPaper(Seq2Vec):
    class Impression:
        __slots__ = ['pos', 'neg', 'time']

        def __init__(self, d):
            d = d.split('#TAB#')
            self.pos = [int(k) for k in d[0].split(' ')]
            self.neg = [int(k) for k in d[1].split(' ')]
            if len(d) >= 3:
                self.time = datetime.strptime(d[2], '%m/%d/%Y %I:%M:%S %p')

        def negative_samples(self, n):
            return np.random.choice(self.neg, n)            # task/paper.py:17-18

    def _extract_impressions(self, x):
        return [self.Impression(d) for d in x.split('#N#') if not d.startswith('#TAB#')]

    def _load_data(self):
        """ClickData.tsv: column 2 = training impressions, column 3 = validation impressions (task/paper.py:24-35)."""
        logging.info('[+] loading data')
        self.data = []
        with open(self.config.training_data_input) as file:
            for line in file:
                line = line.strip('\n').split('\t')
                self.data.append((self._extract_impressions(line[2]) if line[2] else [],
                                  self._extract_impressions(line[3]) if line[3] else []))
        super(Seq2VecPaper, self)._load_data()
        logging.info('[-] loaded data')

    def save_model(self):
        pass                                                 # task/paper.py:254-255

    DEVICE_EVAL = False     # handlers whose epoch-end ranking can run on the GPU (device_callback)

    def device_callback(self, epoch):
        raise NotImplementedError('%s has no device evaluation (the softmax-family handlers have): use handler.callback'
                                  % type(self).__name__)

    # ---- sigmoid family: one (history, candidate, label) sample per row, weighted BCE (task/paper.py:36-256) ----
    HAS_USER = False
    SCORE = 'dnn'                                            # score_encoder: Dense(relu)([u ‖ d]) -> Dense(1, sigmoid), :222-226
    # config.arch -> (engine arch, oracle/synth arch); 'att' = SimpleAttentionMaskSupport over the click window (:206-208)
    USER_ARCHS = {'gru': ('nigru', 'nigru'), 'avg': ('niavg', 'niavg'), 'att': ('att', 'att')}

    def _row(self, user, clicked, title, label):
        return ((user,) if self.HAS_USER else ()) + (clicked, title, label)

    def train_gen(self):
        while True:
            for user, (ih, _) in enumerate(self.data):
                if ih:
                    ch = self.Window(self.docs, self.config.window_size)
                    if len(ih) > self.config.max_impression:
                        chosen = set(random.sample(range(len(ih)), self.config.max_impression))
                    else:
                        chosen = None
                    for i, impression in enumerate(ih):
                        trainable = chosen is None or i in chosen
                        for pos in impression.pos:
                            if ch.count and trainable:
                                clicked = ch.get_title()
                                yield self._row(user, clicked, self.docs[pos].title, 1)
                                for neg in impression.negative_samples(self.config.negative_samples):
                                    yield self._row(user, clicked, self.docs[neg].title, 0)
                            ch.push(pos)

    def valid_gen(self):
        while True:
            for user, (ih1, ih2) in enumerate(self.data):
                if ih1 and ih2:
                    ch = self.Window(self.docs, self.config.window_size)
                    for impression in ih1:
                        for pos in impression.pos:
                            ch.push(pos)
                    for impression in ih2:
                        for pos in impression.pos:
                            clicked = ch.get_title()
                            yield self._row(user, clicked, self.docs[pos].title, 1)
                            for neg in impression.negative_samples(self.config.negative_samples):
                                yield self._row(user, clicked, self.docs[neg].title, 0)
                        for pos in impression.pos:
                            ch.push(pos)

    def test_gen(self):
        for user, (ih1, ih2) in enumerate(self.data):
            if ih1 and ih2:
                ch = self.Window(self.docs, self.config.window_size)
                for impression in ih1:
                    for pos in impression.pos:
                        ch.push(pos)
                for impression in ih2:
                    clicked = ch.get_title()
                    yield [self._row(user, clicked, self.docs[p].title, 1) for p in impression.pos] + \
                          [self._row(user, clicked, self.docs[n].title, 0) for n in impression.neg]
                    for pos in impression.pos:
                        ch.push(pos)

    def _title_embedding(self):
        if self.config.debug:                                # task/paper.py:109-110
            return np.load(self.config.title_embedding_input + '.npy')
        return utils.load_textual_embedding(self.config.title_embedding_input, self.config.textual_embedding_dim)

    def _pretrained_encoder(self):
        """--enable-pretrain-encoder (task/paper.py:103-107): the title encoder's weights come from a json + pkl pair
        (utils.load_model: written by save_model here, or by the reference for a Keras doc encoder) and stay frozen
        unless --pretrain-encoder-trainable."""
        loaded = utils.load_model(self.config.encoder_input)
        enc = keras_like.DocEncoderModel(self._core)
        P = loaded.params()
        missing = [k for k in enc.ENC_ORDER if k in self._core.params and k not in P]
        if missing:
            raise ValueError('pre-trained encoder file lacks %s' % missing)
        for k in enc.ENC_ORDER:
            if k in self._core.params:
                if tuple(P[k].shape) != tuple(np.asarray(self._core.params[k]).shape):
                    raise ValueError('pre-trained encoder: %s has shape %s, the configured model needs %s'
                                     % (k, P[k].shape, np.asarray(self._core.params[k]).shape))
                self._core.params[k] = P[k]
        if not self.config.pretrain_encoder_trainable:
            enc.trainable = False
        return enc

    def get_doc_encoder(self):
        if self.config.news_encoder != 'cnnatt':
            raise Exception('Unsupport doc model')           # task/paper.py:130,195
        if self.config.enable_pretrain_encoder:
            return self._pretrained_encoder()
        return keras_like.DocEncoderModel(self._core)

    def _archs(self):
        if self.config.arch not in self.USER_ARCHS:
            raise Exception('Unsupport user model')          # task/paper.py:216-217, 355-356
        return self.USER_ARCHS[self.config.arch]

    def get_user_encoder(self, window_size=None):
        self._archs()
        return keras_like.UserEncoderModel(self._core, self._doc_dim())

    def _doc_dim(self):
        P = self._core.params
        return int(P['dense_w'].shape[1]) + (int(P['vert_emb'].shape[1]) if 'vert_emb' in P else 0)

    def _build_model(self):
        """task/paper.py:228-256 / 360-383: `model` = sigmoid score, loss = Seq2Vec.loss (weighted BCE), Adam."""
        c = self.config
        eng_arch, syn_arch = self._archs()
        F, k = c.title_filter_shape
        word_emb = self._title_embedding().astype(np.float32)
        sh = synth.Shape('cfg', n_users=len(self.data), n_news=self.doc_count - 1, vocab=word_emb.shape[0],
                         L=c.title_shape, W=c.window_size, K=c.negative_samples, B=c.batch_size, E=word_emb.shape[1],
                         F=F, k=k, U=c.user_embedding_dim, arch=syn_arch)
        params = synth.make_weights(sh, arch=syn_arch, seed=np.random.randint(1 << 30), word_emb=word_emb, keras_orthogonal=True,
                                    score_model=self.SCORE)
        self._core = keras_like._Core(params, c, self.doc_token_table(), self.HAS_USER, eng_arch, score_model=self.SCORE,
                                      loss='bce', flavour='sigmoid')
        self.doc_encoder = self.get_doc_encoder()
        self.user_encoder = self.get_user_encoder()
        self.model = keras_like.Model(self._core, train=True, name='model')
        self.model.layers['doc_encoder'] = self.doc_encoder
        self.model.layers['user_encoder'] = self.user_encoder


class Seq2VecPaperDot(Seq2VecPaper):
    SCORE = 'dot'                                            # sigmoid(Dot([1, 1])), task/paper.py:258-262


class Seq2VecPaperId(Seq2VecPaper):
    """User-ID variants of the sigmoid family (task/paper.py:265-383)."""
    HAS_USER = True
    USER_ARCHS = {'gru': ('gru', 'ngru'), 'igru': ('igru', 'igru'), 'iigru': ('iigru', 'iicat'), 'vo': ('vo', 'vo')}


class Seq2VecPaperSoftmax(Seq2VecPaper):
    HAS_USER = False
    USER_ARCHS = ('gru', 'avg', 'att')                       # Seq2VecPaper.get_user_encoder (inherited), task/paper.py:199-221
    NO_USER_ARCH = {'gru': 'nigru', 'avg': 'niavg', 'att': 'att'}

    # ---- sample generators (task/paper.py:387-441); the window calls go through four hooks so that the time-window
    # variants (Seq2VecPaperSoftmaxDays*, task/paper.py:668-792) only replace the Window -----------------------------
    def _new_window(self):
        return self.Window(self.docs, self.config.window_size)

    def _w_count(self, ch, impression):
        return ch.count

    def _w_title(self, ch, impression):
        return ch.get_title()

    def _w_push(self, ch, pos, impression):
        ch.push(pos)

    def _sample(self, user, ch, pos, impression, label):
        row = [self._w_title(ch, impression), self.docs[pos].title] + \
              [self.docs[neg].title for neg in impression.negative_samples(self.config.negative_samples)] + [label]
        return ([user] + row) if self.HAS_USER else row

    def train_gen(self):
        label = [1] + [0 for _ in range(self.config.negative_samples)]
        while True:
            for user, (ih, _) in enumerate(self.data):
                if ih:
                    ch = self._new_window()
                    for impression in ih:
                        for pos in impression.pos:
                            if self._w_count(ch, impression):
                                yield self._sample(user, ch, pos, impression, label)
                            self._w_push(ch, pos, impression)

    def valid_gen(self):
        label = [1] + [0 for _ in range(self.config.negative_samples)]
        while True:
            for user, (ih1, ih2) in enumerate(self.data):
                if ih1 and ih2:
                    ch = self._new_window()
                    for impression in ih1:
                        for pos in impression.pos:
                            self._w_push(ch, pos, impression)
                    for impression in ih2:
                        for pos in impression.pos:
                            yield self._sample(user, ch, pos, impression, label)
                        for pos in impression.pos:
                            self._w_push(ch, pos, impression)

    # ---- device-assembled batches (mnexp_b200/assemble.py): an opt-in alternative to `train` / `valid` with its own
    # sampling — a device permutation per epoch instead of the 100·B shuffle pool, counter-based negatives instead of
    # np.random.choice — over the same samples, windows and candidates ------------------------------------------------
    DEVICE_SEED = 0         # the same on every data-parallel rank: the ranks draw one permutation and take disjoint rows

    def _w_device(self):
        """The time window of `_new_window` as build_tables wants it: None (no expiry) here, (time_of, seconds) for Days."""
        return None

    def _host_tables(self):
        from .. import assemble
        if getattr(self, '_device_tables', None) is None:       # (host tables, their device copies): built once
            self._device_tables = (assemble.build_tables(self.data, self.config.window_size, self._w_device()), None)
        return self._device_tables[0]

    def _uploaded_tables(self):
        import torch
        host = self._host_tables()
        dev = self._device_tables[1]
        if dev is None:
            device = torch.device('cuda', torch.cuda.current_device())
            dev = {k: torch.as_tensor(v).to(device) for k, v in host.items()}
            self._device_tables = (host, dev)
        return host, dev

    def _device_batcher(self, split):
        from .. import assemble
        import torch.distributed as tdist
        self._host_tables()
        rank, world = 0, 1
        if split == 'train' and tdist.is_available() and tdist.is_initialized():
            rank, world = tdist.get_rank(), tdist.get_world_size()
        c = self.config
        host, dev = self._device_tables
        bt = assemble.DeviceBatcher(self.data, c.batch_size, c.window_size, c.negative_samples, seed=self.DEVICE_SEED,
                                    split=split, rank=rank, world=world, window=self._w_device(), tables=host,
                                    device_tables=dev)
        self._device_tables = (host, bt.t)
        return bt

    @property
    def device_train(self):
        """Endless generator of assembled training batches (assemble.DeviceBatch) for model.fit_generator; under
        torch.distributed every rank yields its own disjoint share of each global batch."""
        return self._device_batcher('train').batches()

    @property
    def device_valid(self):
        """Endless generator of assembled validation batches for model.evaluate_generator, in valid_gen order from the
        first sample on."""
        return self._device_batcher('valid').batches()

    # ---- device evaluation: the impressions of test_gen ranked on the GPU from news vectors encoded once per pass -----
    DEVICE_EVAL = True

    def _eval_engine(self):
        """Inference engine of the device evaluation (shares the live weights): C = the mean impression size (at most the
        plan's 32), and enough rows that the largest impression fits one chunk of rows * C pairs."""
        sizes = np.diff(self._host_tables()['eval_cand_off'])
        C = int(min(32, max(1, np.ceil(sizes.mean())))) if len(sizes) else 1
        rows = max(int(self.config.batch_size), -(-int(sizes.max(initial=1)) // C))
        return self._core.engine_infer(C, rows=rows)

    def device_test(self, n):
        """The first n impressions of test_gen (all of them if there are fewer, as zip(range(n), self.test)) scored on the
        GPU by test_model's head -> (offsets (m + 1,), scores (offsets[-1],), labels (offsets[-1],)) device tensors; the
        candidates of impression i are entries offsets[i] .. offsets[i+1] in test_gen order, positives (label 1) first.
        Every document is encoded once, the user encoder runs once per impression (LsturEngine.score_impressions)."""
        import torch
        from .. import assemble
        host, dev = self._uploaded_tables()
        m = min(int(n), len(host['eval_first_click']))
        off = host['eval_cand_off'][:m + 1]
        if getattr(self, '_eval_label', None) is None:
            sizes = np.diff(host['eval_cand_off'])
            rank = np.arange(int(host['eval_cand_off'][-1])) - np.repeat(host['eval_cand_off'][:-1], sizes)
            self._eval_label = torch.as_tensor((rank < np.repeat(host['eval_npos'], sizes)).astype(np.float32)).to(
                dev['eval_cand_off'].device)
        eng = self._eval_engine()
        idx = torch.arange(m, dtype=torch.int32, device=eng.device)
        w = self._w_device()
        # the history of impression i: the W stream entries before its first click (K = 0: no negatives are drawn)
        b = assemble.assemble_samples(dev, dev['eval_first_click'], dev['eval_first_click'], idx, self.config.window_size,
                                      0, 0 if w is None else int(w[1]))
        table = eng.eval_doc_table()
        scores = eng.score_impressions(b['user'], b['hist_doc'], off, dev['eval_cand_docs'], table)
        P = int(off[-1])
        return dev['eval_cand_off'][:m + 1], scores[:P], self._eval_label[:P]

    def _device_rows(self, x):
        off, scores, labels = self.device_test(x)
        out = metrics.device_ranking_metrics(off, scores, labels)
        n = int(out.shape[0])
        host = self._host_tables()
        return out.cpu().numpy(), host['eval_npos'][:n].tolist(), np.diff(host['eval_cand_off'][:n + 1]).tolist()

    def device_callback(self, epoch):
        """callback with the impressions ranked on the GPU (device_test + the device metrics): the same learning-rate
        decay, model swap, last_evaluation and logged lines; the metrics differ from callback's by rounding only."""
        self._ranking_callback(epoch, self._device_rows)

    def device_doc_vert(self):
        """(doc_count,) int32 vertical of every document (doc 0 and ids absent from DocMeta -> 0): the engine's doc_vert
        table, from which device batches take their vertical ids."""
        tab = np.zeros(self.doc_count, dtype=np.int32)
        for i, d in self.docs.items():
            if i:
                tab[i] = getattr(d, 'vertical', 0)
        return tab

    def test_gen(self):
        def __gen__(_user, _clicked, _impression):
            for p in _impression.pos:
                yield ((_user,) if self.HAS_USER else ()) + (_clicked, self.docs[p].title, 1)
            for n in _impression.neg:
                yield ((_user,) if self.HAS_USER else ()) + (_clicked, self.docs[n].title, 0)

        for user, (ih1, ih2) in enumerate(self.data):
            if ih1 and ih2:
                ch = self._new_window()
                for impression in ih1:
                    for pos in impression.pos:
                        self._w_push(ch, pos, impression)
                for impression in ih2:
                    clicked = self._w_title(ch, impression)
                    yield list(__gen__(user, clicked, impression))
                    for pos in impression.pos:
                        self._w_push(ch, pos, impression)

    # ---- builder hooks ----------------------------------------------------------------------------
    def _title_embedding(self):
        if self.config.debug:                                # task/paper.py:109-110
            return np.load(self.config.title_embedding_input + '.npy')
        return utils.load_textual_embedding(self.config.title_embedding_input, self.config.textual_embedding_dim)

    def get_doc_encoder(self):
        return self._get_doc_encoder(self.config.title_shape)

    def _get_doc_encoder(self, input_shape=None):
        if self.config.news_encoder != 'cnnatt':
            raise Exception('Unsupport doc model')           # task/paper.py:130,195 (non-LSTUR encoders are out of scope)
        if self.config.enable_pretrain_encoder:
            return self._pretrained_encoder()
        return keras_like.DocEncoderModel(self._core)

    def _engine_arch(self):
        arch = self.config.arch
        if arch not in self.USER_ARCHS:
            raise Exception('Unsupport user model')          # task/paper.py:216-217, 629-630
        if arch in ('ngru', 'dgru') and self.config.score_model == 'dot':
            # the reference graph fails to build here too: keras.layers.dot rejects (2U) . (U) (task/paper.py:447)
            raise ValueError("arch '%s' yields a 2U user vector: use score_model 'dnn' or 'ddot'" % arch)
        return self.NO_USER_ARCH[arch] if not self.HAS_USER else arch

    def get_user_encoder(self, window_size=None):
        """Model named 'user_encoder' with the input 'user_clicked_vec' (task/paper.py:590, 632): the user-encoder part of
        the fused plan, callable on cached history vectors (lstur_forward_docvecs)."""
        self._engine_arch()
        return keras_like.UserEncoderModel(self._core, self._doc_dim())

    def _score_model(self, u=None, d=None):
        if self.config.score_model not in ('dot', 'dnn', 'ddot'):
            raise NotImplementedError                          # task/paper.py:456-457
        self.score_model = self.config.score_model

    def score_encoder(self, user_vec=None, candidate_vecs=None):
        self._score_model()
        return self.score_model

    def _init_params(self):
        c = self.config
        F, k = c.title_filter_shape
        word_emb = self._title_embedding().astype(np.float32)
        sh = synth.Shape('cfg', n_users=len(self.data), n_news=self.doc_count - 1, vocab=word_emb.shape[0],
                         L=c.title_shape, W=c.window_size, K=c.negative_samples, B=c.batch_size, E=word_emb.shape[1],
                         F=F, k=k, U=c.user_embedding_dim, arch=self._engine_arch())
        return synth.make_weights(sh, arch=self._engine_arch(), seed=np.random.randint(1 << 30), word_emb=word_emb, keras_orthogonal=True,
                                  score_model=c.score_model)

    def _build_model(self):
        """task/paper.py:466-495 / 635-665: `model` = softmax CE + Adam, `test_model` = sigmoid score, shared weights."""
        arch = self._engine_arch()
        params = self._init_params()
        self._core = keras_like._Core(params, self.config, self.doc_token_table(), self.HAS_USER, arch,
                                      score_model=self.config.score_model)
        self.doc_encoder = self.get_doc_encoder()
        self.user_encoder = self.get_user_encoder()
        self.score_encoder()
        self.model = keras_like.Model(self._core, train=True, name='model')
        self.test_model = keras_like.Model(self._core, train=False, name='test_model')
        for m in (self.model, self.test_model):
            m.layers['doc_encoder'] = self.doc_encoder
            m.layers['user_encoder'] = self.user_encoder

    def _host_rows(self, x):
        # the reference scores one impression at a time on the host (roc_auc_score, utils.ndcg_score / mrr_score);
        # here the x impressions are ranked in ONE launch of the device kernel (mnexp_b200/metrics.py)
        preds, trues = [], []
        for _, (y_pred, y_true) in zip(range(x), self.test):
            preds.append(np.asarray(y_pred).reshape(-1)); trues.append(np.asarray(y_true).reshape(-1))
        return metrics.ranking_metrics(preds, trues), [np.sum(y) for y in trues], [len(y) for y in trues]

    def _ranking_callback(self, epoch, rows_of):
        """LR decay, the model swap, and the two evaluation lines of the first validation_impression impressions (two more
        of the first testing_impression after the last epoch); rows_of(x) -> ((x, 4) metrics, positives, sizes)."""
        keras_like.backend.set_value(self.model.optimizer.lr,
                                     keras_like.backend.get_value(self.model.optimizer.lr) * self.config.learning_rate_decay)
        self.model, self.test_model = self.test_model, self.model

        def __gen__(x):
            m, pos, size = rows_of(x)
            for i, (row, p, n) in enumerate(zip(m, pos, size)):
                yield float(row[0]), float(row[1]), float(row[2]), float(row[3]), p, n, i

        values = [np.mean(x) for x in zip(*__gen__(self.config.validation_impression))]
        self.last_evaluation = dict(auc=values[0], ndcgx=values[1], ndcgv=values[2], mrr=values[3])
        utils.logging_evaluation(self.last_evaluation)
        utils.logging_evaluation(dict(pos=values[4], size=values[5], num=values[6] * 2 + 1))
        if epoch == self.config.epochs - 1:
            self.is_training = False
            values = [np.mean(x) for x in zip(*__gen__(self.config.testing_impression))]
            utils.logging_evaluation(dict(auc=values[0], ndcgx=values[1], ndcgv=values[2], mrr=values[3]))
            utils.logging_evaluation(dict(pos=values[4], size=values[5], num=values[6] * 2 + 1))
        self.model, self.test_model = self.test_model, self.model

    def callback(self, epoch):
        """LR decay + per-impression AUC / nDCG@10 / nDCG@5 / MRR on the validation split (task/paper.py:497-524)."""
        self._ranking_callback(epoch, self._host_rows)


class Seq2VecPaperSoftmaxId(Seq2VecPaperSoftmax):
    """LSTUR (task/paper.py:527-665): igru = LSTUR-ini; gru / hgru / ngru / dgru = LSTUR-con."""
    HAS_USER = True
    USER_ARCHS = ('igru', 'gru', 'ngru', 'hgru', 'dgru', 'iigru', 'nigru', 'pgru', 'vo', 'niavg')   # task/paper.py:596-628


class _DaysWindowMixin:
    """Time-window click history (task/paper.py:669-694, 763-792): a click expires `config.days` after it was made;
    expired slots read as the pad document, and a sample needs at least one live click."""

    class Window:
        __slots__ = ['docs', 'click_history', 'click_history_time', 'delta']
        zero = datetime.strptime('01/01/2000', '%m/%d/%Y')

        def __init__(self, docs, window_size, delta):
            self.docs = docs
            self.delta = timedelta(days=delta)
            self.click_history = [0 for _ in range(window_size)]
            self.click_history_time = [self.zero for _ in range(window_size)]

        def get_ids(self, time):
            return [i if t >= time else 0 for i, t in zip(self.click_history, self.click_history_time)]

        def get_title(self, time):
            return np.stack([self.docs[i].title for i in self.get_ids(time)])

        def push(self, doc, time):
            self.click_history.append(doc)
            self.click_history.pop(0)
            self.click_history_time.append(time + self.delta)
            self.click_history_time.pop(0)

        @property
        def window_size(self):
            return len(self.click_history)

        def count(self, time):
            return sum(1 for t in self.click_history_time if t >= time)

    def _new_window(self):
        return self.Window(self.docs, self.config.window_size, self.config.days)

    def _w_count(self, ch, impression):
        return ch.count(impression.time)

    def _w_title(self, ch, impression):
        return ch.get_title(impression.time)

    def _w_push(self, ch, pos, impression):
        ch.push(pos, impression.time)

    def _w_device(self):
        zero = self.Window.zero
        return (lambda imp: (imp.time - zero) // timedelta(seconds=1)), timedelta(days=self.config.days) // timedelta(seconds=1)


class Seq2VecPaperSoftmaxDays(_DaysWindowMixin, Seq2VecPaperSoftmax):
    """task/paper.py:668-750."""


class Seq2VecPaperSoftmaxDaysId(_DaysWindowMixin, Seq2VecPaperSoftmaxId):
    """task/paper.py:753-881: time windows + the vertical column of DocMeta on every document (:793-822)."""

    class News:
        __slots__ = ['title', 'body', 'vertical']

        def __init__(self, title, body, vertical=0):
            self.title, self.body, self.vertical = title, body, vertical

    def _load_docs(self):
        super(Seq2VecPaperSoftmaxDaysId, self)._load_docs()
        with open(self.config.doc_meta_input) as file:
            for line in file:
                line = line.strip('\n').split('\t')
                self.docs[int(line[1])].vertical = utils.get_vertical(line[2])


class Seq2VecPaperSoftmaxDaysIdVert(Seq2VecPaperSoftmaxDaysId):
    """task/paper.py:1138-1255: news vector = [Dense(U)(title) ‖ Vemb[vertical]] for history and candidates; the user
    encoder is built with user_embedding_dim + vertical_embedding_dim.  Inputs:
    [user, clicked, clicked_vert, cand_0..K, cand_vert_0..K]; test model [user, clicked, clicked_vert, cand, cand_vert]."""

    def _w_vert(self, ch, impression):
        return [self.docs[i].vertical for i in ch.get_ids(impression.time)]

    def _sample(self, user, ch, pos, impression, label):
        negs = impression.negative_samples(self.config.negative_samples)
        return [user, self._w_title(ch, impression), self._w_vert(ch, impression), self.docs[pos].title] + \
               [self.docs[neg].title for neg in negs] + [self.docs[pos].vertical] + \
               [self.docs[neg].vertical for neg in negs] + [label]

    def test_gen(self):
        for user, (ih1, ih2) in enumerate(self.data):
            if ih1 and ih2:
                ch = self._new_window()
                for impression in ih1:
                    for pos in impression.pos:
                        self._w_push(ch, pos, impression)
                for impression in ih2:
                    clicked, cv = self._w_title(ch, impression), self._w_vert(ch, impression)
                    yield [(user, clicked, cv, self.docs[p].title, self.docs[p].vertical, 1) for p in impression.pos] + \
                          [(user, clicked, cv, self.docs[n].title, self.docs[n].vertical, 0) for n in impression.neg]
                    for pos in impression.pos:
                        self._w_push(ch, pos, impression)

    def _init_params(self):
        c = self.config
        F, k = c.title_filter_shape
        word_emb = self._title_embedding().astype(np.float32)
        sh = synth.Shape('cfg', n_users=len(self.data), n_news=self.doc_count - 1, vocab=word_emb.shape[0],
                         L=c.title_shape, W=c.window_size, K=c.negative_samples, B=c.batch_size, E=word_emb.shape[1],
                         F=F, k=k, U=c.user_embedding_dim, arch=self._engine_arch())
        return synth.make_weights(sh, arch=self._engine_arch(), seed=np.random.randint(1 << 30), word_emb=word_emb, keras_orthogonal=True,
                                  score_model=c.score_model, paper_vert=c.vertical_embedding_dim)

    def _build_model(self):
        super(Seq2VecPaperSoftmaxDaysIdVert, self)._build_model()
        self._core.has_vert = True
        # vertical ids of device batches (host batches carry their own)
        self._core.set_doc_table(self._core.doc_tokens, self.device_doc_vert())


def _to_categorical(ids, num_classes):
    out = np.zeros((len(ids), num_classes), dtype=np.float32)
    out[np.arange(len(ids)), np.asarray(ids, dtype=np.int64)] = 1.0
    return out


class Seq2VecPaperSoftmaxDaysIdVertSup(Seq2VecPaperSoftmaxDaysId):
    """task/paper.py:884-1000: LSTUR with an auxiliary vertical classifier.  Samples carry a second target, the one-hot
    verticals of the W history slots and the 1+K candidates (:897-902); the model has two outputs ('ranking', 'vert') and
    the loss 1 * CE_ranking + config.gain * CE_vert (:981-987); test_model is the plain sigmoid scorer (:989-997)."""

    def _w_vert(self, ch, impression):
        return [self.docs[i].vertical for i in ch.get_ids(impression.time)]

    def _sample(self, user, ch, pos, impression, label):
        negs = impression.negative_samples(self.config.negative_samples)
        verts = self._w_vert(ch, impression) + [self.docs[pos].vertical] + [self.docs[neg].vertical for neg in negs]
        return [user, self._w_title(ch, impression), self.docs[pos].title] + [self.docs[neg].title for neg in negs] + \
               [label, _to_categorical(verts, len(utils.verticals))]

    @property
    def train(self):
        """Same shuffle pool as Seq2Vec.train, two targets per batch (task/paper.py:928-939)."""
        from .seq2vec import _stack_columns
        bs = self.config.batch_size
        pool, samples = [], self.train_gen()
        while True:
            pool.append(next(samples))
            if len(pool) < 100 * bs:
                continue
            np.random.shuffle(pool)
            batch = _stack_columns(pool[:bs])
            del pool[:bs]
            yield batch[:-2], batch[-2:]

    @property
    def valid(self):
        from .seq2vec import _stack_columns
        samples = self.valid_gen()
        while True:
            batch = _stack_columns([next(samples) for _ in range(self.config.batch_size)])
            yield batch[:-2], batch[-2:]

    def get_vertical_classifier(self, input_shape=None):
        """Dense(hidden_dim, relu) -> Dense(len(utils.verticals), softmax) (task/paper.py:948-952): (n_vert, hidden_dim)."""
        return len(utils.verticals), self.config.hidden_dim

    def _init_params(self):
        c = self.config
        F, k = c.title_filter_shape
        word_emb = self._title_embedding().astype(np.float32)
        sh = synth.Shape('cfg', n_users=len(self.data), n_news=self.doc_count - 1, vocab=word_emb.shape[0],
                         L=c.title_shape, W=c.window_size, K=c.negative_samples, B=c.batch_size, E=word_emb.shape[1],
                         F=F, k=k, U=c.user_embedding_dim, arch=self._engine_arch())
        return synth.make_weights(sh, arch=self._engine_arch(), seed=np.random.randint(1 << 30), word_emb=word_emb, keras_orthogonal=True,
                                  score_model=c.score_model, vertsup=self.get_vertical_classifier())

    def _build_model(self):
        super(Seq2VecPaperSoftmaxDaysIdVertSup, self)._build_model()
        # vertical labels of device batches (host batches carry their own)
        self._core.set_doc_table(self._core.doc_tokens, self.device_doc_vert())
        layers = self.model.layers
        self.model = keras_like.VertSupModel(self._core, name='model')
        self.model.layers.update(layers)


class Seq2VecPaperSoftmaxDaysIdVertAlt(Seq2VecPaperSoftmaxDaysId):
    """task/paper.py:1003-1136: the click model and a vertical classifier on the shared doc_encoder are trained in
    alternation — `round - 1` epochs of the vertical model (on 10 % of the documents, validated on the rest), then one
    epoch of the click model; `callback_valid` switches `self.model` between `seq_model` and `vert_model`."""

    def __init__(self, config):
        super(Seq2VecPaperSoftmaxDaysIdVertAlt, self).__init__(config)
        self.round = self.config.round
        self.config.epochs *= self.round

    def _device_batcher(self, split):
        # the vertical epochs train VertModel on title batches, which device-assembled click batches cannot feed
        raise NotImplementedError('device-assembled batches do not cover the alternating vertical model of '
                                  'Seq2VecPaperSoftmaxDaysIdVertAlt: train it from handler.train / handler.valid')

    DEVICE_EVAL = False

    def device_test(self, n):
        raise NotImplementedError('the device evaluation does not cover Seq2VecPaperSoftmaxDaysIdVertAlt, whose epochs '
                                  'alternate with the vertical model: evaluate it with handler.callback')

    def device_callback(self, epoch):
        return self.device_test(self.config.validation_impression)

    def _load_docs(self):
        super(Seq2VecPaperSoftmaxDaysIdVertAlt, self)._load_docs()
        names = {}
        with open(self.config.doc_meta_input) as file:
            for line in file:
                cols = line.rstrip('\n').split('\t')
                names[int(cols[1])] = cols[2]
        # the reference indexes list(set(names)) (arbitrary order, :1025-1028); sorted here so that runs are reproducible
        self.verticals = sorted(set(names.values()))
        ids = [i for i in self.docs if i != 0]
        self.data_verticals = _to_categorical([self.verticals.index(names[i]) for i in ids], len(self.verticals))
        self.data_titles = np.stack([self.docs[i].title for i in ids])
        data = np.arange(len(ids))
        np.random.shuffle(data)
        self.train_index = data[:len(ids) // 10]
        self.valid_index = data[len(ids) // 10:]

    @property
    def training_step(self):
        return self.config.training_step if self.train_seq else len(self.train_index) // self.config.batch_size

    @training_step.setter
    def training_step(self, value):
        pass

    @property
    def validation_step(self):
        return self.config.validation_step if self.train_seq else len(self.valid_index) // self.config.batch_size

    @validation_step.setter
    def validation_step(self, value):
        pass

    train_seq = False

    def _vert_batches(self, index, shuffle):
        bs = self.config.batch_size
        if len(index) <= bs:       # the reference's loop (task/paper.py:1069-1075) would spin forever without yielding
            raise ValueError('vertical split of %d documents yields no batch of %d' % (len(index), bs))
        while True:
            if shuffle:
                np.random.shuffle(index)
            titles, verts = self.data_titles[index], self.data_verticals[index]
            for end in range(bs, len(index), bs):              # task/paper.py:1073-1075
                yield titles[end - bs:end], verts[end - bs:end]

    @property
    def train_vert(self):
        return self._vert_batches(self.train_index, True)

    @property
    def valid_vert(self):
        return self._vert_batches(self.valid_index, False)

    @property
    def train(self):
        train_vert = self.train_vert
        train = super(Seq2VecPaperSoftmaxDaysIdVertAlt, self).train
        while True:
            yield next(train) if self.train_seq else next(train_vert)

    @property
    def valid(self):
        return super(Seq2VecPaperSoftmaxDaysIdVertAlt, self).valid if self.train_seq else self.valid_vert

    def callback(self, epoch):
        if self.train_seq:
            super(Seq2VecPaperSoftmaxDaysIdVertAlt, self).callback(epoch)
        elif epoch % self.round == self.round - 2:
            keras_like.backend.set_value(self.model.optimizer.lr,
                                         keras_like.backend.get_value(self.model.optimizer.lr) * self.config.learning_rate_decay)

    def callback_valid(self, epoch):
        self.train_seq = epoch % self.round == self.round - 2
        self.model = self.seq_model if self.train_seq else self.vert_model

    def _init_params(self):
        c = self.config
        F, k = c.title_filter_shape
        word_emb = self._title_embedding().astype(np.float32)
        sh = synth.Shape('cfg', n_users=len(self.data), n_news=self.doc_count - 1, vocab=word_emb.shape[0],
                         L=c.title_shape, W=c.window_size, K=c.negative_samples, B=c.batch_size, E=word_emb.shape[1],
                         F=F, k=k, U=c.user_embedding_dim, arch=self._engine_arch())
        return synth.make_weights(sh, arch=self._engine_arch(), seed=np.random.randint(1 << 30), word_emb=word_emb, keras_orthogonal=True,
                                  score_model=c.score_model, vertalt=len(self.verticals))

    def _build_model(self):
        self.train_seq = False
        super(Seq2VecPaperSoftmaxDaysIdVertAlt, self)._build_model()
        self.seq_model = self.model
        self.model = self.vert_model = keras_like.VertModel(self._core)
        self.vert_model.layers['doc_encoder'] = self.doc_encoder
