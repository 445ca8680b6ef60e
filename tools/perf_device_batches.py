"""Training throughput of a softmax-family task handler fed three ways, at the C3 widths (B 1024, W 50, L 30, K 4, E 300,
F 400, U 200; Seq2VecPaperSoftmaxId 'igru', fp16_tc, dropout 0.2), on a synthetic on-disk dataset:

  host     model.fit_generator(handler.train, n)          samples built in Python (Window, np.random.choice, shuffle pool)
  device   model.fit_generator(handler.device_train, n)   batches assembled on the GPU (mnexp_b200/assemble.py)
  engine   LsturEngine.train_step on pre-assembled device batches (the kernels alone: no assembly, no Model protocol)

The arms alternate within one process; each is timed with a host clock around n steps that end in a device
synchronise, after a warm-up (the host arm's warm-up includes filling its 100·B shuffle pool).  Prints impressions/s
per arm (median and spread over the repetitions) with the GPU's name and power limit, and one JSON line."""
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

from mnexp_b200 import settings, synth, task  # noqa: E402
from mnexp_b200.assemble import DeviceBatch  # noqa: E402


def gpu_info():
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i',
                          str(torch.cuda.current_device())], capture_output=True, text=True)
    return out.stdout.strip() if out.returncode == 0 else 'unknown (nvidia-smi: %s)' % out.stderr.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--users', type=int, default=30000)
    ap.add_argument('--news', type=int, default=130000)
    ap.add_argument('--vocab', type=int, default=30000)
    ap.add_argument('--steps', type=int, default=40, help='training steps per timed window')
    ap.add_argument('--reps', type=int, default=3, help='timed windows per arm, alternating')
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'this measurement needs a GPU'
    with tempfile.TemporaryDirectory(prefix='perf_device_batches_') as d:       # the dataset is removed afterwards
        run(args, d)


def run(args, d):
    sh = synth.Shape('perf', args.users, args.news, args.vocab, B=1024)          # C3 widths
    t0 = time.time()
    synth.write_dataset(d, sh)
    cfg = settings.Config(dict(task='Seq2VecPaperSoftmaxId', arch='igru', input_training_data_path=d, title_shape=sh.L,
                               window_size=sh.W, negative_samples=sh.K, batch_size=sh.B, textual_embedding_dim=sh.E,
                               title_filter_shape=(sh.F, sh.k), user_embedding_dim=sh.U, debug=True, dropout=0.2,
                               precision='fp16_tc'))
    np.random.seed(0)
    h = task.get(cfg)
    model = h.build_model(0)
    pre = h._device_batcher('train')
    print('dataset: %d users, %d training samples, %d validation samples (written and loaded in %.1f s)'
          % (len(h.data), len(pre.host['sample_click']), len(pre.host['valid_click']), time.time() - t0))

    host_gen, dev_gen = h.train, h.device_train
    eng = h._core.engine_train(sh.B)
    C = h._core.n_train_cand()
    batches = [h._core.device_inputs(DeviceBatch(**pre.next_batch()), C) for _ in range(args.steps)]

    def engine_arm(n):
        for db in batches[:n]:
            eng.train_step(db)

    arms = {'host': lambda n: model.fit_generator(host_gen, n),
            'device': lambda n: model.fit_generator(dev_gen, n),
            'engine': engine_arm}
    t0 = time.time()
    for fn in arms.values():                                        # warm-up: pool fill, plan, every shape
        fn(3)
    torch.cuda.synchronize()
    print('warm-up %.1f s' % (time.time() - t0))
    rates = {k: [] for k in arms}
    for _ in range(args.reps):
        for name, fn in arms.items():
            torch.cuda.synchronize()
            t = time.perf_counter()
            fn(args.steps)
            torch.cuda.synchronize()
            rates[name].append(args.steps * sh.B / (time.perf_counter() - t))
    gpu = gpu_info()
    print('GPU: %s' % gpu)
    for name, r in rates.items():
        r = np.asarray(r)
        print('%-7s %10.0f impressions/s  (%.2f ms/step; min %.0f, max %.0f over %d windows of %d steps)'
              % (name, np.median(r), 1e3 * sh.B / np.median(r), r.min(), r.max(), len(r), args.steps))
    med = {k: float(np.median(v)) for k, v in rates.items()}
    print('device / engine = %.3f, device / host = %.1f' % (med['device'] / med['engine'], med['device'] / med['host']))
    print(json.dumps(dict(gpu=gpu, batch=sh.B, steps=args.steps, reps=args.reps, users=len(h.data),
                          impressions_per_s=med, all=rates)))


if __name__ == '__main__':
    main()
