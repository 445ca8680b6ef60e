"""Device-side batch assembly for the generator-fed LSTUR path (SURVEY §8f rank 1).

The reference builds every sample in Python (`train_gen` / `valid_gen` → `Window.get_title` → `np.stack`,
task/paper.py:387-441, task/seq2vec.py:17-53, 182-200), which caps its throughput far below the kernels.  Here the click
streams and the negatives of every impression live on the GPU as CSR tables, and one kernel (lstur_assemble_samples)
emits the compact doc-id batch `user (B) / hist_doc (B,W) / cand_doc (B,1+K)` that LsturEngine consumes:
  * history windows are bit-exact with `Window` (last W clicks before the sample, left-padded with doc 0), including the
    Days variants' expiry (a click older than `days` reads as doc 0) and the validation rule (the history of a
    validation click ends before the first click of its impression);
  * the positive is the click itself, negatives are K draws with replacement from the impression's negatives
    (`Impression.negative_samples`), from the counter-based RNG instead of numpy's (distribution, not stream, parity);
  * training order: one device permutation per epoch instead of the reference's 100·B shuffle pool; validation walks
    the samples in `valid_gen` order.
"""
import ctypes

import numpy as np
import torch

from . import _lib


def build_tables(data, W=None, window=None):
    """handler.data = [(train_impressions, valid_impressions)] per user -> host CSR tables of both splits.

    window: None, or (time_of, expire_seconds) for the Days handlers: time_of(impression) = int seconds since the Days
    Window's zero, expire_seconds = the Window's `days` in whole seconds (floored: the times are whole seconds).
    W (the window size) is needed with a window only: a training click is a sample iff its window has a live slot.

    Every user's stream holds the training clicks, then the validation clicks, in file order; each click carries its
    impression's negatives (neg_off / neg_docs, per click) and, with a window, its impression's time (click_time).
    sample_click: training samples in train_gen order.  valid_click / valid_hist_end: validation samples in valid_gen
    order (every positive of every validation impression of a user with both splits) and the stream index of the first
    click of their impression (valid_gen pushes an impression's clicks only after yielding all of them).
    eval_*: one entry per validation impression of a user with both splits, in test_gen order — eval_first_click (the
    stream index of its first click: its history is the W stream entries before it, its user and time those of that
    click), eval_npos (its positives), eval_cand_off (n + 1) / eval_cand_docs (CSR: its positives in file order, then all
    its negatives in file order, as test_gen yields them)."""
    imps = [(u, s, imp) for u, (ih, iv) in enumerate(data) for s, part in ((0, ih), (1, iv)) for imp in part]
    i64 = lambda a: np.asarray(a, dtype=np.int64)
    imp_user = i64([u for u, _, _ in imps])
    imp_split = i64([s for _, s, _ in imps])
    imp_npos = i64([len(imp.pos) for _, _, imp in imps])
    imp_nneg = i64([len(imp.neg) for _, _, imp in imps])
    stream_docs = i64([p for _, _, imp in imps for p in imp.pos])
    neg_flat = i64([n for _, _, imp in imps for n in imp.neg])
    n_users = len(data)

    click_imp = np.repeat(np.arange(len(imps)), imp_npos)
    click_user = imp_user[click_imp]
    click_split = imp_split[click_imp]
    stream_off = np.concatenate([[0], np.cumsum(np.bincount(click_user, minlength=n_users))])
    imp_first = np.concatenate([[0], np.cumsum(imp_npos)])[:-1]          # stream index of every impression's first click
    # the impression's negatives, repeated for each of its clicks
    click_nneg = imp_nneg[click_imp]
    neg_off = np.concatenate([[0], np.cumsum(click_nneg)])
    imp_neg0 = np.concatenate([[0], np.cumsum(imp_nneg)])[:-1]
    neg_docs = neg_flat[np.repeat(imp_neg0[click_imp] - neg_off[:-1], click_nneg) + np.arange(int(neg_off[-1]))]

    c = np.arange(len(stream_docs))
    pos_in_stream = c - stream_off[click_user]            # training clicks lead the stream: = pushes before a training click
    click_time = None
    if window is None:
        live = pos_in_stream > 0                          # `if ch.count:`
    else:
        time_of, expire = window
        assert W is not None and W > 0, 'the time window needs the window size'
        click_time = i64([time_of(imp) for _, _, imp in imps])[click_imp]
        # count(time): slots of the last W pushes with push time + days >= the impression's time; the Window's unfilled
        # slots carry the zero time itself (no `days` added) and count when the impression is not after it
        live = np.maximum(0, W - pos_in_stream) * (click_time <= 0)
        for w in range(1, W + 1):
            j = c - w
            ok = pos_in_stream >= w
            live = live + (ok & (click_time[np.maximum(j, 0)] + expire >= click_time))
        live = live > 0
    sample_click = c[(click_split == 0) & live]

    has_both = np.zeros(n_users, dtype=bool)
    has_both[imp_user[imp_split == 0]] = True
    has_v = np.zeros(n_users, dtype=bool)
    has_v[imp_user[imp_split == 1]] = True
    has_both &= has_v
    valid = (click_split == 1) & has_both[click_user]
    valid_click = c[valid]
    valid_hist_end = imp_first[click_imp[valid]]

    # evaluation impressions (test_gen order): every validation impression of a user with both splits; its candidates
    # are its positives in file order, then all its negatives in file order
    ev = np.nonzero((imp_split == 1) & has_both[imp_user])[0]
    eval_first_click, eval_npos, ev_nneg = imp_first[ev], imp_npos[ev], imp_nneg[ev]
    eval_cand_off = np.concatenate([[0], np.cumsum(eval_npos + ev_nneg)])
    eval_cand_docs = np.zeros(int(eval_cand_off[-1]), dtype=np.int64)
    dst0 = eval_cand_off[:-1]
    for n, src, src0, dst in ((eval_npos, stream_docs, eval_first_click, dst0), (ev_nneg, neg_flat, imp_neg0[ev], dst0 + eval_npos)):
        k = np.repeat(np.arange(len(ev)), n)                       # the impression of every entry
        j = np.arange(len(k)) - np.repeat(np.cumsum(n) - n, n)     # its index within the impression's positives / negatives
        eval_cand_docs[dst[k] + j] = src[src0[k] + j]

    i32 = lambda a: np.ascontiguousarray(a, dtype=np.int32)
    out = dict(stream_off=i32(stream_off), stream_docs=i32(stream_docs if len(stream_docs) else [0]), click_user=i32(click_user),
               neg_off=i32(neg_off), neg_docs=i32(neg_docs if len(neg_docs) else [0]), sample_click=i32(sample_click),
               valid_click=i32(valid_click), valid_hist_end=i32(valid_hist_end), eval_first_click=i32(eval_first_click),
               eval_npos=i32(eval_npos), eval_cand_off=i32(eval_cand_off),
               eval_cand_docs=i32(eval_cand_docs if len(eval_cand_docs) else [0]))
    if click_time is not None:
        assert click_time.size == 0 or (click_time.min() >= -2 ** 31 and click_time.max() < 2 ** 31), 'times beyond int32 seconds'
        out['click_time'] = i32(click_time)
    return out


class DeviceBatch:
    """One assembled batch on the device: user (B), hist_doc (B,W), cand_doc (B,1+K) int32; the positive is column 0 of
    cand_doc.  keras_like.Model accepts it wherever it accepts a host (inputs, targets) pair."""
    __slots__ = ('user', 'hist_doc', 'cand_doc')

    def __init__(self, user, hist_doc, cand_doc):
        self.user, self.hist_doc, self.cand_doc = user, hist_doc, cand_doc

    @property
    def B(self):
        return int(self.hist_doc.shape[0])

    def as_dict(self):
        return dict(user=self.user, hist_doc=self.hist_doc, cand_doc=self.cand_doc)


class DeviceBatcher:
    """Batches of B rows assembled on the device from build_tables(data, W, window).

    split='train': every rank draws the same seeded device permutations, one per epoch, laid end to end; global batch i is
    rows [i·world·B, (i+1)·world·B) of that sequence and rank r assembles its B rows [r·B, (r+1)·B) with the negatives of
    global rows r·B + b — so `world` ranks together see exactly the rows of one batcher of world·B rows, and each epoch
    visits every sample once.
    split='valid': batches walk the validation samples in valid_gen order from sample 0 and wrap at the end (rank and
    world do not apply: every rank evaluates the same batches).
    tables / device_tables: the host tables (build_tables) and their device copies (another batcher's `t`) to share
    instead of building or uploading them again."""

    def __init__(self, data, B, W, K, device=None, seed=0, split='train', rank=0, world=1, window=None, tables=None,
                 device_tables=None):
        if not torch.cuda.is_available():
            raise _lib.LsturError('DeviceBatcher needs a CUDA device (no CPU fallback)')
        if split not in ('train', 'valid'):
            raise ValueError(split)
        assert 0 <= rank < world
        self.lib = _lib.load()
        self.device = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
        self.B, self.W, self.K, self.seed = B, W, K, seed
        self.split, self.rank, self.world = split, rank, world
        self.host = build_tables(data, W, window) if tables is None else tables
        if device_tables is None:
            device_tables = {k: torch.as_tensor(v).to(self.device) for k, v in self.host.items()}
        self.t = device_tables
        self.expire = 0 if window is None else int(window[1])
        key = 'sample_click' if split == 'train' else 'valid_click'
        self.n_samples = int(self.host[key].shape[0])
        self._click = self.t[key]
        self._hist_end = self.t['valid_hist_end'] if split == 'valid' else None
        self.gen = torch.Generator(device=self.device)
        self.gen.manual_seed(seed)
        self.order, self.cursor, self.step = None, 0, 0

    def _next_indices(self):
        """(B) int32 device sample numbers of this rank's rows of the next global batch, and the global row of its first."""
        n, B = self.n_samples, self.B
        if self.split == 'valid':
            idx = ((torch.arange(B, dtype=torch.int64, device=self.device) + self.cursor) % n).to(torch.int32)
            self.cursor = (self.cursor + B) % n
            return idx, 0
        need = self.world * B
        while self.order is None or self.cursor + need > self.order.numel():
            rest = self.order[self.cursor:] if self.order is not None else self.order
            perm = torch.randperm(n, device=self.device, generator=self.gen, dtype=torch.int32)
            self.order = perm if rest is None else torch.cat([rest, perm])
            self.cursor = 0
        r0 = self.rank * B
        idx = self.order[self.cursor + r0:self.cursor + r0 + B].contiguous()
        self.cursor += need
        return idx, r0

    def assemble(self, idx, row0=0):
        """idx: (B) int32 device tensor of sample numbers -> device batch dict for LsturEngine."""
        B, W, K = int(idx.numel()), self.W, self.K
        user = torch.empty(B, dtype=torch.int32, device=self.device)
        hist = torch.empty((B, W), dtype=torch.int32, device=self.device)
        cand = torch.empty((B, 1 + K), dtype=torch.int32, device=self.device)
        p = lambda x: ctypes.c_void_p(None if x is None else x.data_ptr())
        t = self.t
        self.step += 1
        _lib.check(self.lib.lstur_assemble_samples(
            B, W, K, p(self._click), p(self._hist_end), p(idx), p(t['click_user']), p(t.get('click_time')), self.expire,
            p(t['stream_off']), p(t['stream_docs']), p(t['neg_off']), p(t['neg_docs']),
            ctypes.c_uint((self.seed * 1000003 + self.step) & 0xffffffff), row0, p(user), p(hist), p(cand),
            ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))
        return dict(user=user, hist_doc=hist, cand_doc=cand)

    def next_batch(self):
        assert self.n_samples > 0, 'no %s samples' % self.split
        idx, row0 = self._next_indices()
        return self.assemble(idx, row0)

    def batches(self):
        """Endless generator of DeviceBatch objects (the device counterpart of handler.train / handler.valid)."""
        while True:
            yield DeviceBatch(**self.next_batch())
