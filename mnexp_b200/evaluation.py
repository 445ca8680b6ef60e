"""Per-impression / per-user / in-vocabulary / out-of-vocabulary aggregation of the scored test set — the tail of the
reference's `cook` command (main.py:224-297) — with the per-impression ranking metrics computed on the GPU in one launch
(mnexp_b200/metrics.py) instead of one sklearn / numpy call per impression.

Input: flat arrays over the candidate rows of the test set, as Cook.test() yields them (task/cook.py:25-28):
users, imprs (ids; a new impression starts where either changes), mask (1 = the user id is in the training vocabulary,
0 = out of vocabulary), y_true, y_pred.

The reference's grouping loop is mirrored exactly, including its two edge effects: an impression is closed when the NEXT
row belongs to another one — so the last impression of the file is never closed or counted — and a user is closed on the
first row of the next user, reading `mask` at that row's index (which is the first row of the user's own last
impression at that moment, because `index` has just been advanced only if the impression was closed).
"""
import numpy as np

from . import metrics


class Result:
    __slots__ = ('auc', 'mrr', 'ndcgv', 'ndcgx', 'pos', 'size', 'idx')

    def __init__(self, auc, mrr, ndcgv, ndcgx, pos, size, idx):
        self.auc, self.mrr, self.ndcgv, self.ndcgx, self.pos, self.size, self.idx = auc, mrr, ndcgv, ndcgx, pos, size, idx

    @property
    def result(self):
        return dict(auc=self.auc, ndcgx=self.ndcgx, ndcgv=self.ndcgv, mrr=self.mrr)

    @property
    def info(self):
        return dict(pos=self.pos, size=self.size, num=self.idx * 2 + 1)


def average(results):
    f = lambda name: float(np.mean([getattr(r, name) for r in results])) if results else float('nan')
    return Result(f('auc'), f('mrr'), f('ndcgv'), f('ndcgx'), f('pos'), f('size'), f('idx'))


def impression_bounds(users, imprs):
    """[start, end) of every impression the reference closes (all but the last one of the file)."""
    users, imprs = np.asarray(users), np.asarray(imprs)
    n = len(users)
    if n == 0:
        return np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.int64)
    change = np.where((users[1:] != users[:-1]) | (imprs[1:] != imprs[:-1]))[0] + 1     # first row of a new impression
    starts = np.concatenate([[0], change[:-1]]) if len(change) else np.zeros(0, dtype=np.int64)
    return starts.astype(np.int64), change.astype(np.int64)


def aggregate(users, imprs, mask, y_true, y_pred, metric_fn=None):
    """-> dict(user=Result, impr=Result, iv_user=Result, oov_user=Result) (main.py:250-297).
    metric_fn(scores_list, labels_list) -> (n, 4) [auc, ndcg@10, ndcg@5, mrr]; default: the device kernel."""
    users, imprs, mask = np.asarray(users), np.asarray(imprs), np.asarray(mask)
    y_true, y_pred = np.asarray(y_true, dtype=np.float32).reshape(-1), np.asarray(y_pred, dtype=np.float32).reshape(-1)
    starts, ends = impression_bounds(users, imprs)
    metric_fn = metric_fn or metrics.ranking_metrics
    m = metric_fn([y_pred[a:b] for a, b in zip(starts, ends)], [y_true[a:b] for a, b in zip(starts, ends)]) if len(starts) else np.zeros((0, 4))
    return aggregate_metrics(users, mask, y_true, starts, ends, m)


def aggregate_metrics(users, mask, y_true, starts, ends, m):
    """The averaging of aggregate() over precomputed per-impression metrics: starts / ends = impression_bounds(users,
    imprs), m (len(starts), 4) = [auc, ndcg@10, ndcg@5, mrr] of each of those impressions."""
    users, mask = np.asarray(users), np.asarray(mask)
    y_true = np.asarray(y_true, dtype=np.float32).reshape(-1)
    impr_results = [Result(float(m[i, 0]), float(m[i, 3]), float(m[i, 2]), float(m[i, 1]), float(y_true[a:b].sum()), int(b - a), i)
                    for i, (a, b) in enumerate(zip(starts, ends))]           # ndcgv = nDCG@5, ndcgx = nDCG@10 (main.py:262-263)
    user_results, iv, oov = [], [], []
    impr_index = 0
    for i, (a, b) in enumerate(zip(starts, ends)):
        # the row that closes impression i is row b; if it also starts a new user, the user's impressions so far are
        # averaged and filed by mask[b] — `index` equals b in the reference at that point
        if users[b] != users[b - 1]:
            avg = average(impr_results[impr_index:i + 1])
            user_results.append(avg)
            if mask[b] == 1:
                iv.append(avg)
            elif mask[b] == 0:
                oov.append(avg)
            impr_index = i + 1
    return dict(user=average(user_results), impr=average(impr_results), iv_user=average(iv), oov_user=average(oov))


def log_aggregate(res, log):
    """the eight logging_evaluation lines of main.py:288-296"""
    for k in ('user', 'impr', 'iv_user', 'oov_user'):
        log(res[k].result)
        log(res[k].info)
