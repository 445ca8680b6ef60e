"""Host-side engine: owns device buffers (via torch) and drives the C-ABI plan.

torch is plumbing only — allocation, streams, torch.distributed.  Every FLOP of
the LSTUR path runs in liblstur_b200.so (mnexp_b200/csrc).  Construction raises
if CUDA or the shared library is unavailable: there is no CPU fallback.
"""
import ctypes
import math

import numpy as np
import torch

from . import _lib
from ._lib import lstur_batch, lstur_config, lstur_weights

ARCH = {  # reference arch names -> engine arch (SURVEY.md §9.9); paper.py names
    'igru': 0, 'gru': 1, 'ngru': 2, 'hgru': 2, 'dgru': 2, 'nigru': 3, 'pgru': 4, 'vo': 5, 'niavg': 6, 'iigru': 7,
    'att': 10,                                    # Seq2VecPaper.get_user_encoder (task/paper.py:206-208)
}
SCORE = {'dot': 0, 'dnn': 1, 'ddot': 2}          # task/paper.py:443-458; cook's 'ddot' is linear (task/cook.py:206-209)
# sigmoid family (Seq2VecPaperId.get_user_encoder, task/paper.py:328-358): 'gru' is the plain concat, 'iigru' has no Dense
SIGMOID_ARCH = {'gru': 2, 'igru': 0, 'iigru': 8, 'vo': 5, 'nigru': 3, 'niavg': 6, 'att': 10}
# task/cook.py:146-193 — every branch of Cook.get_user_encoder
COOK_ARCH = {'ingru': 0, 'igru': 2, 'gru': 3, 'agru': 4, 'vo': 5, 'avg': 6, 'inigru': 8, 'iavg': 9, 'iatt': 11,
             'inagru': 12, 'atgru': 13, 'algru': 14, 'ilstm': 15}
TWO_TABLE_ARCHS = (7, 8, 12)      # [user_emb | user_emb2] as the column halves of one device table
DENSE_NAMES = ('conv_w', 'conv_b', 'att_w', 'att_b', 'dense_w', 'dense_b', 'vert_emb', 'subvert_emb',
               'gru_wx', 'gru_wh', 'gru_b', 'lstm_wx', 'lstm_wh', 'lstm_b', 'uatt_w', 'uatt_b', 'alpha', 'con_w', 'con_b',
               'sh_w', 'sh_b', 'so_w', 'so_b', 'su_w', 'su_b', 'sd_w', 'sd_b', 'vs_w1', 'vs_b1', 'vs_w2', 'vs_b2',
               'vcls_w', 'vcls_b')
PREC = {'fp32': 0, 'bf16_tc': 1, 'fp16_tc': 2}


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


class LsturEngine:
    """One replica of the LSTUR model on one GPU.

    params: dict of numpy arrays (names: oracle/lstur_numpy.py docstring).
    """

    def __init__(self, params, B, W, C, L, arch='igru', flavour='paper', dropout=0.0, lr=1e-3,
                 recurrent_activation='hard_sigmoid', precision='fp32', doc_tokens=None, device=None,
                 training=True, sparse_user_adam=True, trainable_word_emb=False, share_weights_from=None,
                 doc_vert=None, doc_subvert=None, score_model='dot', loss='softmax', gain=1.0, bce_neg=4, aux_gain=1.0):
        if not torch.cuda.is_available():
            raise _lib.LsturError('LsturEngine needs a CUDA device (no CPU fallback)')
        self.lib = _lib.load()
        self.device = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
        self.trainable_word_emb = bool(trainable_word_emb) and bool(training)
        amap = {'paper': ARCH, 'sigmoid': SIGMOID_ARCH}.get(flavour, COOK_ARCH)
        if loss not in ('softmax', 'bce'):
            raise ValueError(loss)
        self.loss_model = loss
        if arch not in amap:
            raise Exception('Unsupport user model')                      # task/paper.py:630
        self.arch_name, self.arch = arch, amap[arch]
        if self.arch in TWO_TABLE_ARCHS:
            # 'iigru' has two user tables (task/paper.py:614-619): one (n_users, 2U) device table [user_emb | user_emb2]
            # — the first U columns seed the GRU, the rest join the concat; row-wise Adam is the same arithmetic
            params = dict(params)
            params['user_emb'] = np.concatenate([params['user_emb'], params['user_emb2']], 1)
        if score_model not in SCORE:
            raise NotImplementedError                                    # task/paper.py:456-457
        self.score_model = score_model
        sm = SCORE[score_model] + (1 if (score_model == 'ddot' and flavour == 'cook') else 0)
        Hs = {'dot': 0, 'dnn': params['sh_w'].shape[1] if 'sh_w' in params else 0,
              'ddot': params['su_w'].shape[1] if 'su_w' in params else 0}[score_model]
        ks, E, F = params['conv_w'].shape
        use_dense = 'dense_w' in params
        Dd = params['dense_w'].shape[1] if use_dense else F
        G = params['gru_wh'].shape[0] if 'gru_wh' in params else 0
        if self.arch == 15:
            G = params['lstm_wh'].shape[0]
        Ue = params['user_emb'].shape[1] if 'user_emb' in params and self.arch not in (3, 6, 10) else 0
        if self.arch in (5, 6, 9, 10, 11):
            G = 0
        # Cook.get_doc_encoder concat (task/cook.py:99-113): [title | Vemb[vert] | Semb[subvert]]
        dv = params['vert_emb'].shape[1] if 'vert_emb' in params else 0
        ds = params['subvert_emb'].shape[1] if 'subvert_emb' in params else 0
        U = {0: G, 1: params['con_w'].shape[1] if 'con_w' in params else 0, 2: G + Ue, 3: G, 4: G, 5: Ue,
             6: Dd + dv + ds, 7: params['con_w'].shape[1] if 'con_w' in params else 0, 8: Ue,
             9: Dd + dv + ds + Ue, 10: Dd + dv + ds, 11: Dd + dv + ds + Ue, 12: G, 13: 1, 14: G, 15: G + Ue}[self.arch]
        # 13 = cook 'atgru': the 2G entries of [GRU ; id] pooled to ONE scalar per user (task/cook.py:184-190 as written)
        _sd = share_weights_from.doc_tokens if share_weights_from is not None else None
        n_docs = doc_tokens.shape[0] if doc_tokens is not None else (0 if _sd is None else _sd.shape[0])
        self.cfg = lstur_config(
            B=B, W=W, C=C, L=L, E=E, F=F, KS=ks, use_dense=int(use_dense), Dd=Dd, dv=dv, ds=ds, G=G, Ue=Ue, U=U,
            arch=self.arch, score_model=sm, rec_act=0 if recurrent_activation == 'hard_sigmoid' else 1,
            precision=PREC[precision], V=params['word_emb'].shape[0],
            n_users=params['user_emb'].shape[0] if Ue else 0,
            n_docs=n_docs, dropout=float(dropout),
            save_for_backward=int(training),
            n_vert=params['vert_emb'].shape[0] if dv else 0, n_subvert=params['subvert_emb'].shape[0] if ds else 0,
            Hs=Hs, loss_model=1 if loss == 'bce' else 0, bce_neg=int(bce_neg), gain=float(gain),
            trainable_word_emb=int(self.trainable_word_emb),
            # auxiliary vertical classifier (...VertSup, task/paper.py:948-990) / vertical model (...VertAlt, :1128-1136):
            # present iff their weights are
            aux_nv=params['vs_w2'].shape[1] if 'vs_w2' in params else 0,
            aux_hidden=params['vs_w1'].shape[1] if 'vs_w1' in params else 0, aux_gain=float(aux_gain),
            cls_nv=params['vcls_w'].shape[1] if 'vcls_w' in params else 0)
        self.aux_nv, self.cls_nv, self.aux_gain = self.cfg.aux_nv, self.cfg.cls_nv, float(aux_gain)
        self.B, self.W, self.C, self.L, self.D, self.U, self.Ue, self.G = B, W, C, L, Dd + dv + ds, U, Ue, G
        plan = ctypes.c_void_p()
        _lib.check(self.lib.lstur_plan_create(ctypes.byref(self.cfg), ctypes.byref(plan)))
        self.plan = plan
        dev = self.device
        self.n_dense = int(self.lib.lstur_plan_dense_count(plan))
        src = share_weights_from
        self.dense = torch.zeros(self.n_dense, dtype=torch.float32, device=dev) if src is None else src.dense
        assert self.dense.numel() == self.n_dense
        self.layout = {}
        for name in DENSE_NAMES:
            off, cnt = ctypes.c_longlong(), ctypes.c_longlong()
            if self.lib.lstur_plan_dense_offset(plan, name.encode(), ctypes.byref(off), ctypes.byref(cnt)) == 0:
                self.layout[name] = (off.value, cnt.value, tuple(np.asarray(params[name]).shape))
        if src is None:
            self.word_emb = torch.as_tensor(np.ascontiguousarray(params['word_emb'], dtype=np.float32)).to(dev)
            self.user_emb = torch.as_tensor(np.ascontiguousarray(params['user_emb'], dtype=np.float32)).to(dev) if Ue else None
        else:                                   # inference replica sharing the training engine's device weights
            self.word_emb, self.user_emb = src.word_emb, src.user_emb
        # version of the word table shared by every engine that aliases it: the plan keeps a 16-bit operand copy that
        # is re-packed only when the table was written (lstur_plan_invalidate_tables)
        self._emb_version = [0] if src is None else src._emb_version
        self._emb_seen = -1
        def i32dev(a):              # host arrays are uploaded; device tensors (e.g. an interned table) are used in place
            if a is None:
                return None
            if torch.is_tensor(a):
                return a.to(dev, dtype=torch.int32).contiguous()
            return torch.as_tensor(np.ascontiguousarray(a, dtype=np.int32)).to(dev)
        if doc_tokens is None and src is not None:
            self.doc_tokens = src.doc_tokens
        else:
            self.doc_tokens = i32dev(doc_tokens)
        self.doc_vert = i32dev(doc_vert) if src is None or doc_vert is not None else src.doc_vert
        self.doc_subvert = i32dev(doc_subvert) if src is None or doc_subvert is not None else src.doc_subvert
        if src is None:
            self.set_weights_dict(params)
        ws_bytes = int(self.lib.lstur_plan_workspace_bytes(plan))
        self.ws_bytes = ws_bytes
        self.ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        self.training_plan = bool(training)
        if training:
            self.dense_grad = torch.zeros_like(self.dense)
            self.adam_m = torch.zeros_like(self.dense)
            self.adam_v = torch.zeros_like(self.dense)
            if Ue:
                self.user_m = torch.zeros_like(self.user_emb)
                self.user_v = torch.zeros_like(self.user_emb)
                self.user_grad_dense = None if sparse_user_adam else torch.zeros_like(self.user_emb)
            if self.trainable_word_emb:
                # keras Embedding(trainable=True) (task/paper.py:136): dense gradient (rows of absent tokens are zero, as
                # tf.IndexedSlices densify to) and dense Keras-Adam moments — reference semantics, SURVEY.md §9.7
                self.word_grad = torch.zeros_like(self.word_emb)
                self.word_m = torch.zeros_like(self.word_emb)
                self.word_v = torch.zeros_like(self.word_emb)
        self.sparse_user_adam = sparse_user_adam
        # `encoder.trainable = False` of a pre-trained title encoder (task/paper.py:103-106): its gradients — the word
        # table and the conv / attention / Dense tensors, which lead the arena — are zeroed before every update (Adam
        # moments that never see a gradient never move the weights)
        self.freeze_encoder = False
        self.lr = float(lr)
        self.t = 0
        self.step_seed = 0
        self.gpu_launches = 0
        self._w = lstur_weights(dense=self.dense.data_ptr(), word_emb=self.word_emb.data_ptr(),
                                user_emb=self.user_emb.data_ptr() if Ue else None,
                                doc_tokens=self.doc_tokens.data_ptr() if self.doc_tokens is not None else None,
                                doc_vert=self.doc_vert.data_ptr() if self.doc_vert is not None else None,
                                doc_subvert=self.doc_subvert.data_ptr() if self.doc_subvert is not None else None)

    def __del__(self):
        try:
            if getattr(self, 'plan', None):
                self.lib.lstur_plan_destroy(self.plan)
                self.plan = None
        except Exception:
            pass

    def adopt_state_from(self, old):
        """A training engine rebuilt for another batch shape takes over the old one's device weights AND its optimizer
        state (Adam moments, step count, dropout seed counter), so that changing the batch size mid-training does not
        reset the optimizer or replay dropout masks."""
        assert self.training_plan and old.training_plan and self.n_dense == old.n_dense
        for name in ('dense', 'adam_m', 'adam_v', 'word_emb', 'user_emb', 'user_m', 'user_v', 'word_m', 'word_v'):
            a, b = getattr(self, name, None), getattr(old, name, None)
            if a is not None and b is not None:
                a.copy_(b)
        self.t, self.step_seed, self.lr = old.t, old.step_seed, old.lr
        self._emb_version[0] += 1

    # ---- weights ------------------------------------------------------------------------
    def set_weights_dict(self, params):
        host = np.zeros(self.n_dense, dtype=np.float32)
        for name, (off, cnt, shape) in self.layout.items():
            host[off:off + cnt] = np.asarray(params[name], dtype=np.float32).reshape(-1)
        self.dense.copy_(torch.from_numpy(host))
        if 'word_emb' in params:
            self.word_emb.copy_(torch.as_tensor(np.ascontiguousarray(params['word_emb'], dtype=np.float32)))
            self._emb_version[0] += 1
        if self.user_emb is not None and 'user_emb' in params:
            ue = params['user_emb']
            if self.arch in TWO_TABLE_ARCHS and ue.shape[1] != self.Ue:
                ue = np.concatenate([ue, params['user_emb2']], 1)
            self.user_emb.copy_(torch.as_tensor(np.ascontiguousarray(ue, dtype=np.float32)))

    def _unflatten(self, flat):
        host = flat.detach().cpu().numpy()
        return {name: host[off:off + cnt].reshape(shape).copy() for name, (off, cnt, shape) in self.layout.items()}

    def get_weights_dict(self):
        out = self._unflatten(self.dense)
        out['word_emb'] = self.word_emb.cpu().numpy()
        if self.user_emb is not None:
            out['user_emb'] = self.user_emb.cpu().numpy()
            if self.arch in TWO_TABLE_ARCHS:
                out['user_emb'], out['user_emb2'] = out['user_emb'][:, :self.G].copy(), out['user_emb'][:, self.G:].copy()
        return out

    def get_dense_grads_dict(self):
        """Dense gradients of the last backward (lstur_backward or lstur_title_cls_backward)."""
        out = self._unflatten(self.dense_grad)
        if self.trainable_word_emb:
            out['word_emb'] = self.word_grad.cpu().numpy()
        return out

    def get_grads_dict(self):
        """Dense gradients plus the (densified) user-embedding gradient of the last backward."""
        out = self._unflatten(self.dense_grad)
        if self.trainable_word_emb:
            out['word_emb'] = self.word_grad.cpu().numpy()
        if self.user_emb is not None:
            g = np.zeros(tuple(self.user_emb.shape), dtype=np.float32)
            n = int(self.view('n_user_rows', torch.int32)[0])
            rows = self.view('user_rows', torch.int32)[:n].cpu().numpy()
            g[rows] = self.view('d_user_rows').reshape(-1, self.Ue)[:n].cpu().numpy()
            out['user_emb'] = g
            if self.arch in TWO_TABLE_ARCHS:
                out['user_emb'], out['user_emb2'] = g[:, :self.G].copy(), g[:, self.G:].copy()
        return out

    # ---- workspace views ------------------------------------------------------------------
    def view(self, name, dtype=torch.float32):
        key = (name, dtype)
        cache = self.__dict__.setdefault('_views', {})
        if key in cache:
            return cache[key]
        ptr, cnt = ctypes.c_void_p(), ctypes.c_longlong()
        _lib.check(self.lib.lstur_plan_view(self.plan, _ptr(self.ws), name.encode(), ctypes.byref(ptr), ctypes.byref(cnt)))
        off = ptr.value - self.ws.data_ptr()
        cache[key] = self.ws[off:off + 4 * cnt.value].view(dtype)
        return cache[key]

    # ---- batches --------------------------------------------------------------------------
    def to_device_batch(self, batch, non_blocking=False):
        """dict of host arrays/tensors -> dict of int32/float32 device tensors."""
        out = {}
        for k, v in batch.items():
            if v is None:
                continue
            t = v if torch.is_tensor(v) else torch.from_numpy(np.ascontiguousarray(v))
            if k in ('label', 'user_scale', 'user_scale2'):
                t = t.to(self.device, dtype=torch.float32, non_blocking=non_blocking)
            else:
                t = t.to(self.device, non_blocking=non_blocking)
                if t.dtype != torch.int32:
                    t = t.to(torch.int32)          # reference feeds float64 token ids (document.py:39); ids < 2^24
            out[k] = t.contiguous()
        return out

    def _cbatch(self, db):
        g = lambda k: db[k].data_ptr() if k in db else None
        return lstur_batch(user=g('user'), hist_doc=g('hist_doc'), cand_doc=g('cand_doc'), hist_tok=g('hist_tok'),
                           cand_tok=g('cand_tok'), label=g('label'), user_scale=g('user_scale'),
                           hist_vert=g('hist_vert'), hist_subvert=g('hist_subvert'), cand_vert=g('cand_vert'),
                           cand_subvert=g('cand_subvert'), user_scale2=g('user_scale2'))

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ---- the hot path ---------------------------------------------------------------------
    def forward(self, db, training=False, seed=0):
        cb = self._cbatch(db)
        if self._emb_seen != self._emb_version[0]:
            _lib.check(self.lib.lstur_plan_invalidate_tables(self.plan))
            self._emb_seen = self._emb_version[0]
        _lib.check(self.lib.lstur_forward(self.plan, ctypes.byref(self._w), ctypes.byref(cb), _ptr(self.ws),
                                          int(training), ctypes.c_uint(seed), self._stream()))
        return self.view('probs').reshape(self.B, self.C)

    # ---- decomposed inference (task/test_pipeline.py:37-211; BASELINE config 4) ---------------------------------
    def encode_docs(self, doc_ids):
        """doc_encoder.predict over documents given by id (TestPipeline.test_doc_vec): -> (n, D) device tensor.
        Processed in chunks of B*(W+C) titles, the title capacity of this engine's plan."""
        ids = doc_ids if torch.is_tensor(doc_ids) else torch.as_tensor(np.ascontiguousarray(doc_ids))
        ids = ids.to(self.device, dtype=torch.int32).contiguous()
        n = int(ids.numel())
        out = torch.empty((n, self.D), dtype=torch.float32, device=self.device)
        if self._emb_seen != self._emb_version[0]:
            _lib.check(self.lib.lstur_plan_invalidate_tables(self.plan))
            self._emb_seen = self._emb_version[0]
        cap = self.B * (self.W + self.C)
        for i in range(0, n, cap):
            m = min(cap, n - i)
            _lib.check(self.lib.lstur_encode_docs(self.plan, ctypes.byref(self._w), _ptr(self.ws), m,
                                                  ctypes.c_void_p(ids.data_ptr() + 4 * i),
                                                  ctypes.c_void_p(out.data_ptr() + 4 * i * self.D), self.D, self._stream()))
        return out

    def encode_titles(self, titles):
        """doc_encoder.predict on explicit token rows: (n, L) ids (host or device) -> (n, D) device tensor, in chunks of
        the plan's title capacity B*(W+C)."""
        t = titles if torch.is_tensor(titles) else torch.as_tensor(np.ascontiguousarray(titles))
        t = t.to(self.device)
        if t.dtype != torch.int32:
            t = t.to(torch.int32)          # the reference feeds float64 ids (document.py:39)
        t = t.contiguous()
        n = int(t.shape[0])
        assert t.dim() == 2 and t.shape[1] == self.L
        out = torch.empty((n, self.D), dtype=torch.float32, device=self.device)
        if self._emb_seen != self._emb_version[0]:
            _lib.check(self.lib.lstur_plan_invalidate_tables(self.plan))
            self._emb_seen = self._emb_version[0]
        cap = self.B * (self.W + self.C)
        for i in range(0, n, cap):
            m = min(cap, n - i)
            _lib.check(self.lib.lstur_encode_titles(self.plan, ctypes.byref(self._w), _ptr(self.ws), m,
                                                    ctypes.c_void_p(t.data_ptr() + 4 * i * self.L),
                                                    ctypes.c_void_p(out.data_ptr() + 4 * i * self.D), self.D, self._stream()))
        return out

    def encode_users(self, users, clicked_vecs):
        """user_encoder.predict: users (n,) ids (ignored by the archs without a user table), clicked_vecs (n, W, D)
        history vectors -> (n, U) user vectors.  An all-zero history vector is a masked slot (keras Masking())."""
        cv = clicked_vecs if torch.is_tensor(clicked_vecs) else torch.as_tensor(np.ascontiguousarray(clicked_vecs, dtype=np.float32))
        cv = cv.to(self.device, dtype=torch.float32).contiguous()
        n = int(cv.shape[0])
        assert cv.shape[1] == self.W and cv.shape[2] == self.D
        us = torch.as_tensor(np.ascontiguousarray(users)).to(self.device).to(torch.int32).reshape(-1)
        out = torch.empty((n, self.U), dtype=torch.float32, device=self.device)
        R = self.B
        hist = torch.arange(R * self.W, dtype=torch.int32, device=self.device).reshape(R, self.W) + 1    # row 0 = zero vector
        cand = torch.zeros((R, self.C), dtype=torch.int32, device=self.device)
        table = torch.zeros((R * self.W + 1, self.D), dtype=torch.float32, device=self.device)
        for s in range(0, n, R):
            m = min(R, n - s)
            table[1:1 + m * self.W] = cv[s:s + m].reshape(m * self.W, self.D)
            if m < R:
                table[1 + m * self.W:].zero_()
            u = torch.zeros(R, dtype=torch.int32, device=self.device)
            u[:m] = us[s:s + m]
            self.forward_docvecs(dict(user=u, hist_doc=hist, cand_doc=cand), table)
            out[s:s + m] = self.view('user_vec').reshape(R, self.U)[:m]
        return out

    def build_doc_table(self):
        """Vectors of every document of the token table, row 0 (the pad / unknown document) zeroed: the reference's
        pipeline leaves history slots without a known document at zero (task/test_pipeline.py:100-108)."""
        n_docs = int(self.doc_tokens.shape[0])
        table = self.encode_docs(torch.arange(n_docs, dtype=torch.int32, device=self.device))
        table[0].zero_()
        return table

    def eval_doc_table(self):
        """Vectors of every document of the token table, as the news encoder gives them (row 0, the pad document, is
        Dense(0) = the bias), with the vertical columns of the doc_vert / doc_subvert tables in plans that have them:
        the candidate rows of score_impressions."""
        n_docs = int(self.doc_tokens.shape[0])
        ids = torch.arange(n_docs, dtype=torch.int32, device=self.device)
        table = self.encode_docs(ids)
        if self.cfg.dv + self.cfg.ds:
            assert (self.cfg.dv == 0 or self.doc_vert is not None) and (self.cfg.ds == 0 or self.doc_subvert is not None), \
                'the vertical columns need the doc_vert / doc_subvert tables'
            _lib.check(self.lib.lstur_vert_concat(
                n_docs, self.D, self.D - self.cfg.dv - self.cfg.ds, self.cfg.dv, self.cfg.ds, n_docs, self.cfg.n_vert,
                self.cfg.n_subvert, _ptr(ids), _ptr(self.doc_vert), _ptr(self.doc_subvert),
                ctypes.c_void_p(self.dense.data_ptr() + 4 * self.layout['vert_emb'][0]) if self.cfg.dv else None,
                ctypes.c_void_p(self.dense.data_ptr() + 4 * self.layout['subvert_emb'][0]) if self.cfg.ds else None,
                _ptr(table), None, None, self._stream()))
        return table

    def score_impressions(self, user, hist_doc, cand_off, cand_doc, table, out=None, user_scale=None, user_scale2=None):
        """Test-head scores of whole impressions (lstur_score_impressions): user (n,), hist_doc (n, W), cand_doc (pairs,)
        int32 device tensors, cand_off (n + 1,) host int32 offsets into cand_doc, table = eval_doc_table().  The user
        encoder runs once per impression.  user_scale / user_scale2: optional (n,) float32 device multipliers of the
        impression's user embedding, as the batch entries of the same names in forward().  -> (cand_off[-1],) float32
        device tensor of sigmoid scores (entries before cand_off[0] are left as they were in `out`)."""
        off = np.ascontiguousarray(cand_off, dtype=np.int32)
        n = len(off) - 1
        assert table.dtype == torch.float32 and table.is_contiguous() and table.shape[1] == self.D
        if out is None:
            out = torch.empty(int(off[-1]) if n >= 0 else 0, dtype=torch.float32, device=self.device)
        for t in (user, hist_doc, cand_doc):
            assert t.dtype == torch.int32 and t.is_contiguous() and t.device == self.device
        for t in (user_scale, user_scale2):
            assert t is None or (t.dtype == torch.float32 and t.is_contiguous() and t.device == self.device and t.numel() >= n)
        _lib.check(self.lib.lstur_score_impressions(self.plan, ctypes.byref(self._w), _ptr(self.ws), n, _ptr(user),
                                                    _ptr(user_scale), _ptr(user_scale2), _ptr(hist_doc),
                                                    off.ctypes.data_as(ctypes.c_void_p), _ptr(cand_doc),
                                                    _ptr(table), int(table.shape[0]), _ptr(out), self._stream()))
        return out

    def forward_docvecs(self, db, table):
        """User encoder + scorer over cached document vectors (TestPipeline.test_user_vec / test_user_doc_score);
        db carries user, hist_doc (B,W), cand_doc (B,C).  Returns the (B, C) softmax probabilities; score_sigmoid()
        gives the test head as after forward()."""
        cb = self._cbatch(db)
        assert table.dtype == torch.float32 and table.is_contiguous() and table.shape[1] == self.D
        _lib.check(self.lib.lstur_forward_docvecs(self.plan, ctypes.byref(self._w), ctypes.byref(cb), _ptr(self.ws),
                                                  _ptr(table), self.D, int(table.shape[0]), self._stream()))
        return self.view('probs').reshape(self.B, self.C)

    def backward(self, db, grad_scale=None):
        cb = self._cbatch(db)
        gs = 1.0 / self.B if grad_scale is None else grad_scale
        _lib.check(self.lib.lstur_backward_w(self.plan, ctypes.byref(self._w), ctypes.byref(cb), _ptr(self.ws),
                                             _ptr(self.dense_grad), _ptr(self.word_grad) if self.trainable_word_emb else None,
                                             ctypes.c_float(gs), self._stream()))

    def apply_adam(self, b1=0.9, b2=0.999, eps=1e-7, user_rows=None):
        """Keras Adam on the dense arena and the user table.  user_rows = (max_rows, rows, n_rows, g_rows)
        device tensors overrides the local unique rows (data-parallel: globally exchanged rows)."""
        self.t += 1
        st = self._stream()
        if self.freeze_encoder:
            last = 'dense_b' if 'dense_b' in self.layout else 'att_b'
            end = self.layout[last][0] + self.layout[last][1]
            self.dense_grad[:end].zero_()
            if self.trainable_word_emb:
                self.word_grad.zero_()
        _lib.check(self.lib.lstur_adam_dense(self.n_dense, _ptr(self.dense), _ptr(self.dense_grad), _ptr(self.adam_m),
                                             _ptr(self.adam_v), self.lr, self.t, b1, b2, eps, 1.0, st))
        if 'alpha' in self.layout:     # AlphaAdd's constraint MinMaxNorm(0, 1) runs after the update (models.py:545)
            off = self.layout['alpha'][0]
            _lib.check(self.lib.lstur_minmaxnorm(1, 0.0, 1.0, ctypes.c_void_p(self.dense.data_ptr() + 4 * off), st))
        if self.trainable_word_emb:
            _lib.check(self.lib.lstur_adam_dense(self.word_emb.numel(), _ptr(self.word_emb), _ptr(self.word_grad),
                                                 _ptr(self.word_m), _ptr(self.word_v), self.lr, self.t, b1, b2, eps, 1.0, st))
            self._emb_version[0] += 1          # the plans re-pack their 16-bit operand copy of the table
        if self.user_emb is not None:
            if user_rows is None:
                user_rows = (self.B, self.view('user_rows', torch.int32), self.view('n_user_rows', torch.int32),
                             self.view('d_user_rows'))
            mx, rows, nrows, grows = user_rows
            if self.sparse_user_adam:
                _lib.check(self.lib.lstur_adam_rows(mx, _ptr(nrows), self.Ue, _ptr(rows), _ptr(grows),
                                                    _ptr(self.user_emb), _ptr(self.user_m), _ptr(self.user_v),
                                                    self.lr, self.t, b1, b2, eps, 1.0, st))
            else:   # reference semantics: dense Adam over the whole table (SURVEY §9.7)
                self.user_grad_dense.zero_()
                _lib.check(self.lib.lstur_rows_add(mx, _ptr(nrows), self.Ue, _ptr(rows), _ptr(grows),
                                                   _ptr(self.user_grad_dense), st))
                _lib.check(self.lib.lstur_adam_dense(self.user_emb.numel(), _ptr(self.user_emb), _ptr(self.user_grad_dense),
                                                     _ptr(self.user_m), _ptr(self.user_v), self.lr, self.t, b1, b2, eps, 1.0, st))

    def new_event(self):
        ev = ctypes.c_void_p()
        _lib.check(self.lib.lstur_event_create(ctypes.byref(ev)))
        return ev

    def elapsed_ms(self, a, b):
        ms = ctypes.c_float()
        _lib.check(self.lib.lstur_event_elapsed_ms(a, b, ctypes.byref(ms)))
        return ms.value

    def set_probe(self, probe_id, ev_start=None, ev_stop=None):
        """Record two CUDA events (new_event()) around one kernel of the step (bench.py roofline)."""
        _lib.check(self.lib.lstur_plan_set_probe(self.plan, probe_id, ev_start, ev_stop))

    def train_step(self, db, seed=None, grad_scale=None):
        """forward + backward + Adam on a device batch; returns the loss (mean over the B rows) as a 1-element device
        tensor.  grad_scale overrides 1 / B: a ragged last batch of n < B samples is run as B rows whose padding rows carry
        an all-zero target (no loss, no gradient) with grad_scale = 1 / n."""
        self.step_seed += 1
        self.forward(db, training=True, seed=self.step_seed if seed is None else seed)
        self.backward(db, grad_scale=grad_scale)
        self.apply_adam()
        return self.view('loss')

    def loss(self):
        return float(self.view('loss')[0])

    def aux_loss(self):
        """mean categorical cross-entropy of the auxiliary vertical classifier in the last forward (...VertSup); the
        compiled Keras loss is loss() + aux_gain * aux_loss() (loss_weights=[1, gain], task/paper.py:985)."""
        return float(self.view('vs_loss')[0])

    # ---- vertical model of ...VertAlt (task/paper.py:1128-1136): its own Adam (a second optimizer over the shared weights)
    def title_cls_forward(self, tokens, labels, training=False, seed=0):
        t = tokens if torch.is_tensor(tokens) else torch.as_tensor(np.ascontiguousarray(tokens))
        t = t.to(self.device).to(torch.int32).contiguous()
        y = labels if torch.is_tensor(labels) else torch.as_tensor(np.ascontiguousarray(labels))
        y = y.to(self.device).to(torch.int32).contiguous().reshape(-1)
        n = int(t.shape[0])
        assert t.shape[1] == self.L and y.numel() == n
        if self._emb_seen != self._emb_version[0]:
            _lib.check(self.lib.lstur_plan_invalidate_tables(self.plan))
            self._emb_seen = self._emb_version[0]
        _lib.check(self.lib.lstur_title_cls_forward(self.plan, ctypes.byref(self._w), _ptr(self.ws), n, _ptr(t), _ptr(y),
                                                    int(training), ctypes.c_uint(seed), self._stream()))
        self._cls_n = n
        return self.view('vc_probs')[:n * self.cls_nv].reshape(n, self.cls_nv)

    def title_cls_backward(self, grad_scale=None):
        gs = 1.0 / self._cls_n if grad_scale is None else grad_scale
        _lib.check(self.lib.lstur_title_cls_backward(self.plan, ctypes.byref(self._w), _ptr(self.ws), _ptr(self.dense_grad),
                                                     _ptr(self.word_grad) if self.trainable_word_emb else None,
                                                     ctypes.c_float(gs), self._stream()))

    def title_cls_train_step(self, tokens, labels, lr=None, b1=0.9, b2=0.999, eps=1e-7):
        """one step of vert_model.fit: forward, backward, Keras-Adam with the vertical model's OWN moments and step count
        (keras compiles vert_model with a second Adam, task/paper.py:1132-1136).  Returns (loss, accuracy) device scalars."""
        if getattr(self, 'cls_m', None) is None:
            self.cls_m, self.cls_v, self.cls_t = torch.zeros_like(self.dense), torch.zeros_like(self.dense), 0
            if self.trainable_word_emb:
                self.cls_word_m, self.cls_word_v = torch.zeros_like(self.word_emb), torch.zeros_like(self.word_emb)
        self.step_seed += 1
        probs = self.title_cls_forward(tokens, labels, training=True, seed=self.step_seed)
        self.title_cls_backward()
        self.cls_t += 1
        st = self._stream()
        lr = self.lr if lr is None else float(lr)
        if self.freeze_encoder:
            last = 'dense_b' if 'dense_b' in self.layout else 'att_b'
            self.dense_grad[:self.layout[last][0] + self.layout[last][1]].zero_()
        _lib.check(self.lib.lstur_adam_dense(self.n_dense, _ptr(self.dense), _ptr(self.dense_grad), _ptr(self.cls_m),
                                             _ptr(self.cls_v), lr, self.cls_t, b1, b2, eps, 1.0, st))
        if self.trainable_word_emb and not self.freeze_encoder:
            _lib.check(self.lib.lstur_adam_dense(self.word_emb.numel(), _ptr(self.word_emb), _ptr(self.word_grad),
                                                 _ptr(self.cls_word_m), _ptr(self.cls_word_v), lr, self.cls_t, b1, b2, eps, 1.0, st))
            self._emb_version[0] += 1
        lab = self.view('vc_label', torch.int32)[:self._cls_n]
        acc = (probs.argmax(1) == lab).float().mean()
        return self.view('vc_loss'), acc

    def score_sigmoid(self):
        """sigmoid(user_vec . cand_vec) for every (row, candidate) of the last forward — the reference's test head
        (task/paper.py:661-665).  Returns a (B, C) device tensor."""
        out = torch.empty((self.B, self.C), dtype=torch.float32, device=self.device)
        if self.score_model != 'dot':     # sigmoid of the raw scores the scorer left in the workspace
            if getattr(self, '_ones', None) is None:
                self._ones = torch.ones(self.B, dtype=torch.float32, device=self.device)
            _lib.check(self.lib.lstur_score_sigmoid(self.B * self.C, self.C, 1, _ptr(self._ones), 1,
                                                    _ptr(self.view('logits')), 1, _ptr(out), 1, self._stream()))
            return out
        nh = self.B * self.W
        dv = self.view('doc_vec')
        cand = dv[nh * self.D:]
        _lib.check(self.lib.lstur_score_sigmoid(self.B * self.C, self.C, self.D, _ptr(self.view('user_vec')), self.U,
                                                _ptr(cand), self.D, _ptr(out), 1, self._stream()))
        return out
