"""Time of the epoch-end ranking pass (handler.callback) on the host path and on the device path (handler.device_callback),
at the C3 widths (W 50, L 30, E 300, F 400, U 200; 130 k news; Seq2VecPaperSoftmaxId 'igru', 'dot', fp16_tc), on a
synthetic on-disk dataset:

  host     handler.callback(0)          test_gen in Python, one forward per impression (Model.predict), metrics on the GPU
  device   handler.device_callback(0)   every document encoded once, the user encoder once per impression, scores and
                                        metrics on the GPU (lstur_score_impressions + lstur_ranking_metrics)

The two arms alternate, `--reps` times each, at validation_impression = 1000 and at the number of impressions the
dataset holds; each call is timed with a host clock that ends in a device synchronise.  The device arm's parts are timed
the same way: the document table (LsturEngine.eval_doc_table), the user pass (lstur_score_impressions with every
impression's candidate list emptied: history gather + user encoder, chunks of B impressions), the full scoring pass, and
the metrics, each on every impression of the dataset.  Prints the GPU's name and power limit, read in the same run, and one JSON line."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from mnexp_b200 import _lib, settings, synth, task, utils  # noqa: E402


def gpu_info():
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i',
                          str(torch.cuda.current_device())], capture_output=True, text=True)
    return out.stdout.strip() if out.returncode == 0 else 'unknown (nvidia-smi: %s)' % out.stderr.strip()


def timed(fn, *args):
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn(*args)
    torch.cuda.synchronize()
    return time.perf_counter() - t, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--users', type=int, default=4000)
    ap.add_argument('--news', type=int, default=130000)
    ap.add_argument('--vocab', type=int, default=30000)
    ap.add_argument('--batch', type=int, default=1024, help='config.batch_size: the rows of one evaluation chunk')
    ap.add_argument('--reps', type=int, default=3, help='calls per arm and count, alternating')
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'this measurement needs a GPU'
    with tempfile.TemporaryDirectory(prefix='perf_device_eval_') as d:         # the dataset is removed afterwards
        run(args, d)


def run(args, d):
    sh = synth.Shape('perf', args.users, args.news, args.vocab, B=args.batch)     # C3 widths
    t0 = time.time()
    synth.write_dataset(d, sh)
    cfg = settings.Config(dict(task='Seq2VecPaperSoftmaxId', arch='igru', input_training_data_path=d, title_shape=sh.L,
                               window_size=sh.W, negative_samples=sh.K, batch_size=sh.B, textual_embedding_dim=sh.E,
                               title_filter_shape=(sh.F, sh.k), user_embedding_dim=sh.U, debug=True, dropout=0.2,
                               precision='fp16_tc', epochs=2))
    np.random.seed(0)
    h = task.get(cfg)
    h.build_model(0).fit_generator(h.device_train, 3)
    host, dev = h._uploaded_tables()
    n_all = len(host['eval_first_click'])
    print('dataset: %d users, %d evaluation impressions, %d candidates (written and loaded in %.1f s)'
          % (len(h.data), n_all, int(host['eval_cand_off'][-1]), time.time() - t0))
    utils.logging_evaluation = lambda d: None                      # the arms' log lines are not part of the measurement
    lr = h.model.optimizer.lr

    def arm(name, n):
        h.config.validation_impression = n
        lr.value = cfg.learning_rate
        return timed(getattr(h, name), 0)[0]

    counts = sorted({min(1000, n_all), n_all})
    for n in counts:                                                # warm-up: plans, every shape
        arm('device_callback', n)
    arm('callback', min(10, n_all))
    res = {}
    for n in counts:
        t = {'callback': [], 'device_callback': []}
        for _ in range(args.reps):
            for name in t:
                t[name].append(arm(name, n))
        res[n] = t

    # the device path's parts, at every impression of the dataset
    eng = h._eval_engine()
    W = cfg.window_size
    parts = {'doc_table': [], 'user_pass': [], 'scoring': [], 'metrics': []}
    off = host['eval_cand_off']
    p = lambda x: ctypes.c_void_p(x.data_ptr())
    idx = torch.arange(n_all, dtype=torch.int32, device=eng.device)
    user = torch.empty(n_all, dtype=torch.int32, device=eng.device)
    hist = torch.empty((n_all, W), dtype=torch.int32, device=eng.device)
    pos = torch.empty((n_all, 1), dtype=torch.int32, device=eng.device)
    _lib.check(eng.lib.lstur_assemble_samples(n_all, W, 0, p(dev['eval_first_click']), p(dev['eval_first_click']), p(idx),
                                              p(dev['click_user']), None, 0, p(dev['stream_off']), p(dev['stream_docs']),
                                              p(dev['neg_off']), p(dev['neg_docs']), 0, 0, p(user), p(hist), p(pos),
                                              eng._stream()))
    _, labels = h.device_test(n_all)[1:]
    out = torch.empty((n_all, 4), dtype=torch.float32, device=eng.device)
    dummy = torch.empty(1, dtype=torch.float32, device=eng.device)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    for _ in range(args.reps):
        ta, table = timed(eng.eval_doc_table)
        tu, _ = timed(eng.score_impressions, user, hist, np.zeros_like(off), dev['eval_cand_docs'], table, dummy)
        ts, scores = timed(eng.score_impressions, user, hist, off, dev['eval_cand_docs'], table)
        tm, _ = timed(lambda: _lib.check(eng.lib.lstur_ranking_metrics(n_all, p(dev['eval_cand_off']), p(scores), p(labels),
                                                                        p(out), stream)))
        for k, v in zip(parts, (ta, tu, ts, tm)):
            parts[k].append(v)
    gpu = gpu_info()
    print('GPU: %s' % gpu)
    for n, t in res.items():
        hm, dm = np.median(t['callback']), np.median(t['device_callback'])
        print('%6d impressions: callback %8.1f ms (min %.1f, max %.1f), device_callback %7.1f ms (min %.1f, max %.1f), '
              'ratio %.1f' % (n, 1e3 * hm, 1e3 * min(t['callback']), 1e3 * max(t['callback']), 1e3 * dm,
                              1e3 * min(t['device_callback']), 1e3 * max(t['device_callback']), hm / dm))
    print('device parts at %d impressions (median ms): %s' % (n_all, ', '.join(
        '%s %.2f' % (k, 1e3 * np.median(v)) for k, v in parts.items())))
    print(json.dumps(dict(gpu=gpu, batch=sh.B, users=len(h.data), impressions=n_all, reps=args.reps,
                          seconds={str(n): t for n, t in res.items()}, parts_seconds=parts)))


if __name__ == '__main__':
    main()
