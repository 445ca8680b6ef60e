"""Cook's training loop and evaluation tail on the host path and on the interned device path, at the reference's launch
configuration (run.sh: batch 400, window 20) and the C3 widths (L 30, E 300, F 400, U 200), Cook 'ingru' / 'ddot' /
use_vertical_type 'vs', fp16_tc, dropout 0.2, id_keep 0.8, on a synthetic on-disk dataset (synth.write_cook_npz_shared:
the candidates of a test impression share its history):

  interning   Cook._interned on the first call (upload + lstur_intern_rows / lstur_intern_table of both files), then
              intern.intern of the same four parts again, --reps times
  fit         one epoch of CookModel.fit on train() (host batches) and on device_train() (batches gathered on the GPU),
              alternating, --reps times each: steps/s and samples/s
  tail        aggregate_test (test_model.predict + the per-impression metrics + the averaging) on test() and with
              device=True, alternating, --reps times each

Every call is timed with a host clock that ends in a device synchronise.  Prints the GPU's name and power limit, read in
the same run, and one JSON line."""
import argparse
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

from mnexp_b200 import intern, settings, synth, task, utils  # noqa: E402


def gpu_info():
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i',
                          str(torch.cuda.current_device())], capture_output=True, text=True)
    return out.stdout.strip() if out.returncode == 0 else 'unknown (nvidia-smi: %s)' % out.stderr.strip()


def timed(fn, *args, **kw):
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn(*args, **kw)
    torch.cuda.synchronize()
    return time.perf_counter() - t, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--train', type=int, default=100000, help='training samples')
    ap.add_argument('--impressions', type=int, default=10000, help='test impressions (2..8 candidates each)')
    ap.add_argument('--news', type=int, default=130000)
    ap.add_argument('--vocab', type=int, default=30000)
    ap.add_argument('--reps', type=int, default=2, help='calls per arm, alternating')
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'this measurement needs a GPU'
    with tempfile.TemporaryDirectory(prefix='perf_cook_') as d:         # the dataset is removed afterwards
        run(args, d)


def run(args, d):
    sh = synth.Shape('perf', 25000, args.news, args.vocab, L=30, W=20, B=400, E=300, F=400, U=200)
    t0 = time.time()
    synth.write_cook_npz_shared(d, sh, n_train=args.train, n_impr=args.impressions, long_impr=300)
    cfg = settings.Config(dict(task='Cook', arch='ingru', input_training_data_path=d, days=30, window_size=sh.W,
                               batch_size=sh.B, title_filter_shape=(sh.F, 3), user_embedding_dim=sh.U, dropout=0.2,
                               score_model='ddot', use_vertical=True, use_vertical_type='vs', vertical_embedding_dim=100,
                               subvertical_embedding_dim=100, precision='fp16_tc', id_keep=0.8, epochs=1))
    np.random.seed(0)
    h = task.get(cfg)
    model = h.build_model(0)
    n_train, n_test = len(h.training_data['idx']), len(h.test_data['idx'])
    print('dataset: %d training samples, %d test rows in %d impressions (written and loaded in %.1f s)'
          % (n_train, n_test, args.impressions, time.time() - t0))
    t_first, _ = timed(h._interned)
    parts = [(dd[t + '_title'], dd[t + '_vert'], dd[t + '_subvert']) for dd in (h.training_data, h.test_data) for t in ('ch', 'cd')]
    t_intern = [timed(intern.intern, parts, h.L)[0] for _ in range(args.reps)]
    n_docs = int(h._core.doc_tokens.shape[0])
    print('interning: first call %.1f ms (with the upload), again %s ms; %d documents from %d rows'
          % (1e3 * t_first, ', '.join('%.1f' % (1e3 * t) for t in t_intern), n_docs,
             sum(int(np.prod(np.shape(p[0])[:-1])) for p in parts)))
    utils.logging_evaluation = lambda r: None
    arms = {'host': h.train, 'device': h.device_train}
    model.fit(*h.device_train(), sh.B, epochs=1)                       # warm-up: plans, every shape
    fit = {k: [] for k in arms}
    for _ in range(args.reps):
        for k, data in arms.items():
            fit[k].append(timed(model.fit, *data(), sh.B, epochs=1)[0])
    h.aggregate_test(device=True)                                       # warm-up
    h.aggregate_test(device=False)
    tail = {'host': [], 'device': []}
    for _ in range(args.reps):
        for k in tail:
            tail[k].append(timed(h.aggregate_test, device=(k == 'device'))[0])
    gpu = gpu_info()
    steps = -(-n_train // sh.B)
    print('GPU: %s' % gpu)
    for k, t in fit.items():
        m = np.median(t)
        print('fit %-6s epoch %7.2f s (min %.2f, max %.2f): %7.1f steps/s, %9.0f samples/s'
              % (k, m, min(t), max(t), steps / m, n_train / m))
    for k, t in tail.items():
        m = np.median(t)
        print('tail %-6s %8.1f ms (min %.1f, max %.1f): %9.0f impressions/s'
              % (k, 1e3 * m, 1e3 * min(t), 1e3 * max(t), args.impressions / m))
    print(json.dumps(dict(gpu=gpu, batch=sh.B, train=n_train, test_rows=n_test, impressions=args.impressions,
                          documents=n_docs, reps=args.reps, intern_first_s=t_first, intern_s=t_intern, fit_s=fit,
                          tail_s=tail, steps_per_epoch=steps)))


if __name__ == '__main__':
    main()
