"""GPU ranking metrics of the evaluation loop (task/paper.py:497-524): AUC, nDCG@10, nDCG@5, MRR per impression.

Host counterparts: mnexp_b200/utils.py (ndcg_score, mrr_score — reference utils.py:106-124) and sklearn's
roc_auc_score; the device kernel (csrc/score.cu: ranking_metrics_kernel) computes all four for every impression of a
ragged batch in one launch."""
import ctypes

import numpy as np
import torch

from . import _lib


def ranking_metrics(scores, labels, device=None):
    """scores / labels: lists of 1-D arrays (one per impression).  -> (n_impr, 4) float32 numpy array with columns
    auc, ndcg@10, ndcg@5, mrr (NaN where the host formulas divide by zero)."""
    if not torch.cuda.is_available():
        raise _lib.LsturError('ranking_metrics needs a CUDA device (no CPU fallback; use mnexp_b200.utils on the host)')
    dev = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
    lens = np.array([len(s) for s in scores], dtype=np.int64)
    assert all(len(a) == len(b) for a, b in zip(scores, labels))
    off = np.zeros(len(lens) + 1, dtype=np.int32)
    off[1:] = np.cumsum(lens)
    if len(lens) == 0:
        return np.zeros((0, 4), dtype=np.float32)
    s = torch.as_tensor(np.concatenate([np.asarray(x, dtype=np.float32).reshape(-1) for x in scores])).to(dev)
    y = torch.as_tensor(np.concatenate([np.asarray(x, dtype=np.float32).reshape(-1) for x in labels])).to(dev)
    return device_ranking_metrics(torch.as_tensor(off).to(dev), s, y).cpu().numpy()


def device_ranking_metrics(offsets, scores, labels):
    """ranking_metrics of impressions already on the device: offsets (n_impr + 1,) int32, scores / labels float32
    device tensors, impression i = entries offsets[i] .. offsets[i+1].  -> (n_impr, 4) float32 device tensor; nothing
    waits for the device."""
    n = int(offsets.numel()) - 1
    out = torch.empty((n, 4), dtype=torch.float32, device=offsets.device)
    if n:
        p = lambda t: ctypes.c_void_p(t.data_ptr())
        _lib.check(_lib.load().lstur_ranking_metrics(n, p(offsets), p(scores), p(labels), p(out),
                                                     ctypes.c_void_p(torch.cuda.current_stream(offsets.device).cuda_stream)))
    return out


def auc_roc(scores, labels):
    """Batch ROC-AUC reported as the training metric of the sigmoid family (utils.auc_roc wraps tf.metrics.auc,
    utils.py:84-96; here the exact rank statistic of the batch, ties counted half).  0.5 when one class is absent."""
    s = np.asarray(scores, dtype=np.float64).reshape(-1)
    y = np.asarray(labels).reshape(-1) > 0.5
    pos, neg = s[y], s[~y]
    if len(pos) == 0 or len(neg) == 0:
        return 0.5
    d = pos[:, None] - neg[None, :]
    return float(((d > 0).sum() + 0.5 * (d == 0).sum()) / d.size)
