#!/usr/bin/env python
"""LSTUR training throughput on B200 (BASELINE.json metric) — contract in the task statement.

  python bench.py --gpus N --steps K --warmup W            our arm (CUDA through the C-ABI)
  python bench.py --impl reference --gpus N ...            reference arm: the CPU restatement of the
                                                           reference's Keras graph on the host cores
  --workload C1|C2|C3|C5        BASELINE.json configs (default C3, the config the metric is quoted on)
  --trainable-emb               textual_embedding_trainable (conv input gradient + word-table scatter; F_train = 3 x fwd)
  --scaling weak|strong         weak: B rows per rank (default); strong: the workload's B split over the ranks
  --no-extras                   skip the sub-records (drop-in protocol timing, per-kernel probes, C2, C4)
  --dump-outputs DIR            write what the last timed step computed as DIR/<name>.npy (rank 0; see dump_outputs)

A "step" is one LSTUR training step (forward + backward + Keras-Adam) over one batch of B
impressions per rank; value = impressions/s over all ranks.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
import types

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'lstur_train_impressions_per_sec'
UNIT = 'impressions/s'


def flops_per_impression(sh, trainable_emb=False):
    """SURVEY.md §8d / BASELINE.md §3: algorithmic FLOPs (no dedup)."""
    T = sh.W + 1 + sh.K
    tok = T * sh.L
    conv = tok * 2 * sh.k * sh.E * sh.F
    rest = tok * 4 * sh.F + T * 2 * sh.F * sh.U + sh.W * 2 * (sh.U * 3 * sh.U + sh.U * 3 * sh.U) + (1 + sh.K) * 2 * sh.U
    fwd = conv + rest
    return dict(conv_fwd=conv, fwd=fwd, gru_fwd=sh.W * 2 * (sh.U * 3 * sh.U + sh.U * 3 * sh.U),
                train=3 * fwd if trainable_emb else fwd + conv + 2 * rest)


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return d, 'measured'
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0), 'fallback'


def ncu_traffic(kernel_substr):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the newest committed
    `ncu --set full` summary of this same command (profiles/r*_ncu_full_summary.json); None if absent."""
    import glob
    for p in sorted(glob.glob(os.path.join(ROOT, 'profiles', 'r*_ncu_full_summary.json')), reverse=True):
        try:
            for row in json.load(open(p)):
                if kernel_substr in row['kernel']:
                    return (row['dram_read_GB'] + row['dram_write_GB']) * 1e9, os.path.basename(p)
        except Exception:
            pass
    return None, None


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(',')])

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[5:9]):
                    if v.lower().startswith('active'):
                        reasons.add(name)
            except Exception:
                pass
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


def build_workload(sh, n_batches, rank, B, full_history=False):
    from mnexp_b200 import synth
    tok, _, _ = synth.make_docs(sh.n_news, sh.L, sh.vocab)
    P = synth.make_weights(sh, arch=sh.arch)
    batches, pad_frac = synth.make_batches(sh, n_batches, seed=1236 + 1000 * rank, B=B, full_history=full_history)
    return tok, P, batches, pad_frac


def cpu_reference_run(sh, steps, warmup, sample_B, threads=None, trainable_emb=False):
    """The reference's Keras graph restated in torch-CPU fp32 (oracle/lstur_torch.py), all host threads,
    on a bounded sample of the workload: `sample_B` rows per step, same tables, dropout on, dense Keras Adam."""
    import torch
    from oracle import lstur_torch as ot
    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    tok, P, batches, _ = build_workload(sh, warmup + steps, 0, sample_B)
    ora = ot.LsturOracle(P, arch=sh.arch, dtype=torch.float32, lr=1e-3, dropout=0.2, trainable_word_emb=trainable_emb)
    times = []
    for i, b in enumerate(batches):
        t0 = time.perf_counter()
        ora.train_step(b['user'], tok[b['hist_doc']], tok[b['cand_doc']], training=True)
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    t = float(np.sum(times))
    return dict(value=sample_B * len(times) / t, unit=UNIT, cores=threads, kind='port', batch=sample_B,
                sample='%d steps of %d impressions (NOT the GPU arm\'s batch) of workload %s: same tables / shapes, dropout 0.2, '
                       'dense Keras-Adam on every tensor incl. the %d x %d user table (reference semantics); torch-CPU fp32 '
                       'restatement of the Keras graph (reproduces the reference\'s own code, run over oracle/keras_shim, to 1e-9: '
                       'tests/test_ref_pinned.py)' % (len(times), sample_B, sh.name, sh.n_users, sh.U),
                ms_per_step=1e3 * t / len(times))


def timed_ms(torch, fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    r = fn()
    e1.record()
    torch.cuda.synchronize()
    return r, e0.elapsed_time(e1)


DUMP_LIMIT_BYTES = 64 << 20
DUMP_WORD_ROWS = 8192


def last_step_outputs(torch, eng, batch):
    """What a caller of the timed train step holds after its last step, copied to the host: the loss it returned, the
    probabilities of its forward, every dense weight after the Adam update, and the rows of the embedding tables the step
    updated (the batch's users; with a trainable word table, a seeded sample of the batch's tokens).  The tables themselves
    (up to 1M x 200 floats) are too large to write whole."""
    rows = lambda table, ids: table[torch.as_tensor(ids, dtype=torch.int64, device=eng.device)].cpu().numpy()
    out = dict(loss=eng.view('loss').cpu().numpy().copy(), probs=eng.view('probs').reshape(eng.B, eng.C).cpu().numpy().copy())
    out.update(('weight_' + k, v) for k, v in eng._unflatten(eng.dense).items())
    if eng.user_emb is not None:
        users = np.unique(batch['user'])
        out['user_emb_row_ids'] = users.astype(np.float64)
        out['user_emb_rows'] = rows(eng.user_emb, users)
    if eng.trainable_word_emb:
        tokens = np.unique(rows(eng.doc_tokens, np.concatenate([batch['hist_doc'].ravel(), batch['cand_doc'].ravel()])))
        if tokens.size > DUMP_WORD_ROWS:
            tokens = np.sort(np.random.default_rng(0).choice(tokens, DUMP_WORD_ROWS, replace=False))
        out['word_emb_row_ids'] = tokens.astype(np.float64)
        out['word_emb_rows'] = rows(eng.word_emb, tokens)
    return out


def dump_outputs(dirname, arrays):
    """DIR/<name>.npy for every array, float32 or float64, at most DUMP_LIMIT_BYTES in all."""
    arrays = {k: v if v.dtype in (np.float32, np.float64) else v.astype(np.float64) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError('--dump-outputs: %d bytes exceed the %d byte limit' % (total, DUMP_LIMIT_BYTES))
    os.makedirs(dirname, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(dirname, k + '.npy'), v)


def extra_records(torch, lib, sh, eng, dbs, batches, tok, P, precision, pk, args, B, live_frac=1.0):
    """Sub-records of the N=1 line (each bounded to a few seconds; failures are recorded, never fatal)."""
    from mnexp_b200 import synth
    from mnexp_b200.engine import LsturEngine
    out = {}
    fl = flops_per_impression(sh, args.trainable_emb)
    tensor_peak, hbm = pk['bf16_tflops_sustained'], pk['hbm_gbs']

    # ---- per-kernel probes inside the training step (CUDA events recorded by the plan around one launch)
    try:
        kern = {}
        probes = [('conv_wgrad', 2, fl['conv_fwd']), ('attn_bwd', 7, None), ('gru_fwd', 4, fl['gru_fwd']), ('gru_bwd', 8, None)]
        if args.trainable_emb:
            probes += [('conv_dgrad', 5, fl['conv_fwd']), ('word_scatter', 6, None)]
        for name, pid, flops in probes:
            evs = [(eng.new_event(), eng.new_event()) for _ in range(3)]
            for i, (a, b) in enumerate(evs):
                eng.set_probe(pid, a, b)
                eng.train_step(dbs[i % len(dbs)])
            torch.cuda.synchronize()
            eng.set_probe(0)
            ms = float(np.median([eng.elapsed_ms(a, b) for a, b in evs]))
            rec = dict(ms=ms)
            if flops:
                lf = live_frac if name.startswith('conv') else 1.0
                rec['tflops'] = flops * B * lf / (ms / 1e3) / 1e12          # executed (live titles) FLOPs
                rec['frac_of_sustained_tensor_peak'] = rec['tflops'] / tensor_peak
            kern[name] = rec
        if args.trainable_emb:
            T = sh.W + 1 + sh.K
            n_unique = int((eng.word_grad.abs().amax(1) > 0).sum())
            nbytes = B * T * sh.L * (sh.E * 2 + 4) + n_unique * sh.E * 4
            kern['word_scatter'].update(algorithmic_bytes=nbytes, gbs=nbytes / (kern['word_scatter']['ms'] / 1e3) / 1e9,
                                        frac_of_hbm=nbytes / (kern['word_scatter']['ms'] / 1e3) / 1e9 / hbm, unique_rows=n_unique,
                                        note='16-bit dX rows + ids read, unique fp32 rows written; includes the radix sort')
        out['kernels'] = kern
    except Exception as ex:          # noqa: BLE001
        out['kernels'] = dict(error=repr(ex))

    # ---- the reference's data protocol, timed once (SURVEY §8d): keras-like Model.train_on_batch fed float64 (B,W,L)
    # token arrays + one-hot target from host memory, as main.py:73-78 / task/paper.py:538-541 feed it
    try:
        from mnexp_b200 import keras_like
        cfg = types.SimpleNamespace(learning_rate=1e-3, window_size=sh.W, title_shape=sh.L, negative_samples=sh.K, dropout=0.2,
                                    recurrent_activation='hard_sigmoid', batch_size=B, sparse_user_adam=True, gain=1.0,
                                    precision=precision, textual_embedding_trainable=args.trainable_emb)
        core = keras_like._Core(P, cfg, tok, True, sh.arch)
        model = keras_like.Model(core, train=True)
        xs = []
        for b in batches[:3]:
            clicked = tok[b['hist_doc']].astype(np.float64)
            cands = [tok[b['cand_doc'][:, j]].astype(np.float64) for j in range(1 + sh.K)]
            y = np.zeros((B, 1 + sh.K)); y[:, 0] = 1
            xs.append(([b['user']] + [clicked] + cands, y))
        import itertools
        gen = itertools.cycle(xs)
        model.fit_generator(gen, 2, epochs=1)
        n = 6
        _, ms = timed_ms(torch, lambda: model.fit_generator(gen, n, epochs=1))
        _, ms_tob = timed_ms(torch, lambda: [model.train_on_batch(*xs[i % 3]) for i in range(4)])
        h2d = sum(int(np.asarray(a).nbytes) for a in xs[0][0]) + int(xs[0][1].nbytes)
        out['dropin_protocol'] = dict(value=B * n / (ms / 1e3), unit=UNIT, ms_per_step=ms / n, host_bytes_per_step=h2d,
                                      train_on_batch_ms_per_step=ms_tob / 4,
                                      api='keras_like.Model.fit_generator(generator of ([user, clicked(B,W,L) float64, cand_0..K (B,L) '
                                          'float64], one-hot (B,1+K)), steps) as main.py:73-78 calls it: float64 host arrays in, '
                                          '[loss, categorical_accuracy] out every step; staging of batch i+1 overlaps the device '
                                          'step i (train_on_batch alone, unpipelined, beside it)')
        del model, core
    except Exception as ex:          # noqa: BLE001
        out['dropin_protocol'] = dict(error=repr(ex))
    torch.cuda.empty_cache()

    # ---- C2: LSTUR-con at MIND-small-scale shape (BASELINE.json configs[1]), B = 1024
    if sh.name != 'C2':
        try:
            s2 = synth.SHAPES['C2']
            tok2, P2, b2, _ = build_workload(s2, 3, 0, s2.B)
            e2 = LsturEngine(P2, s2.B, s2.W, 1 + s2.K, s2.L, arch=s2.arch, doc_tokens=tok2, dropout=0.2, lr=1e-3,
                             precision=precision, sparse_user_adam=True)
            d2 = [e2.to_device_batch(b) for b in b2]
            for i in range(3):
                e2.train_step(d2[i])
            n = 10
            _, ms = timed_ms(torch, lambda: [e2.train_step(d2[i % 3]) for i in range(n)])
            f2 = flops_per_impression(s2)
            v = s2.B * n / (ms / 1e3)
            out['C2'] = dict(workload='C2: LSTUR-con (gru: Dense([GRU | user])), %d users / %d news / %d vocab, B=%d'
                                      % (s2.n_users, s2.n_news, s2.vocab, s2.B), value=v, unit=UNIT, ms_per_step=ms / n,
                             step_frac_of_train_roofline=v * f2['train'] / (tensor_peak * 1e12), loss=e2.loss())
            del e2, d2
        except Exception as ex:      # noqa: BLE001
            out['C2'] = dict(error=repr(ex))
        torch.cuda.empty_cache()

    # ---- C4: decomposed inference (BASELINE.json configs[3]): encode all news once, then users x 20 candidates
    try:
        s4 = synth.SHAPES['C4']
        if sh.name in ('C3', 'C4'):
            tok4, P4 = tok, P
        else:
            tok4, _, _ = synth.make_docs(s4.n_news, s4.L, s4.vocab)
            P4 = synth.make_weights(s4, arch='igru')
        B4, C4 = 2048, 20
        e4 = LsturEngine(P4, B4, s4.W, C4, s4.L, arch='igru', doc_tokens=tok4, precision=precision, training=False)
        e4.build_doc_table()
        table, ms_docs = timed_ms(torch, e4.build_doc_table)
        g = np.random.default_rng(0)
        d4 = []
        for i in range(4):
            lens = np.clip(g.geometric(1 / 30.0, B4), 1, s4.W)
            hist = g.integers(1, s4.n_news + 1, (B4, s4.W)).astype(np.int32)
            hist[np.arange(s4.W)[None, :] < (s4.W - lens)[:, None]] = 0
            d4.append(e4.to_device_batch(dict(user=g.integers(0, s4.n_users, B4).astype(np.int32), hist_doc=hist,
                                              cand_doc=g.integers(1, s4.n_news + 1, (B4, C4)).astype(np.int32))))
        nb = 64                        # 131 072 users: a bounded sample of the 1M-user pass

        def users():
            for i in range(nb):
                e4.forward_docvecs(d4[i % 4], table)
                s = e4.score_sigmoid()
            return s
        users()
        _, ms_users = timed_ms(torch, users)
        ups = nb * B4 / (ms_users / 1e3)
        gru_flops = s4.W * 2 * (s4.U * 3 * s4.U + s4.U * 3 * s4.U)
        out['C4'] = dict(workload='C4: %d news encoded once, then %d users x %d candidates through the GRU user encoder (sample of the 1M-user pass)'
                                  % (s4.n_news + 1, nb * B4, C4),
                         news_docs_per_s=table.shape[0] / (ms_docs / 1e3), news_pass_ms=ms_docs,
                         users_per_s=ups, pairs_per_s=ups * C4, user_pass_ms_per_1M_users=1e6 / ups * 1e3,
                         user_pass_frac_of_tensor_bound=ups * gru_flops / (tensor_peak * 1e12),
                         note='bound = GRU FLOPs at the sustained tensor peak (SURVEY §8d: 17.4 ms per 1M users)')
        del e4, d4, table
    except Exception as ex:          # noqa: BLE001
        out['C4'] = dict(error=repr(ex))
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='C3')
    ap.add_argument('--precision', default=os.environ.get('LSTUR_PRECISION', 'auto'))
    ap.add_argument('--batch', type=int, default=0, help='rows per rank (default: the workload batch size)')
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'])
    ap.add_argument('--trainable-emb', action='store_true')
    ap.add_argument('--full-history', action='store_true',
                    help='every user has W clicks (no left padding): nothing for the live-title compaction to skip')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-extras', action='store_true')
    ap.add_argument('--cpu-sample', type=int, default=64)
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the loss, probabilities, updated weights and updated table rows of the last timed step '
                         'as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes what the CUDA path computed (--impl ours)')
    args.warmup = max(args.warmup, 3) if args.impl == 'ours' else args.warmup

    from mnexp_b200 import synth
    sh = synth.SHAPES[args.workload]
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    B = args.batch or sh.B
    if args.scaling == 'strong':
        assert B % world == 0, 'strong scaling: the global batch must divide by the number of ranks'
        B //= world
    config = dict(workload='%s: LSTUR-%s train step, %d users / %d news / %d vocab, L%d W%d K%d E%d F%d U%d, B=%d per rank'
                           % (sh.name, 'ini' if sh.arch == 'igru' else 'con', sh.n_users, sh.n_news, sh.vocab, sh.L, sh.W,
                              sh.K, sh.E, sh.F, sh.U, B),
                  global_batch=B * world, parallelism='dp%d' % world, dropout=0.2, optimizer='Keras-Adam',
                  word_emb_trainable=bool(args.trainable_emb))

    if args.impl == 'reference':
        if rank != 0:
            return 0
        r = cpu_reference_run(sh, max(1, args.steps), min(args.warmup, 1), args.cpu_sample, trainable_emb=args.trainable_emb)
        # this arm's real per-step batch and optimizer (the workload string names the GPU arm's shape)
        config.update(reference_arm_batch=args.cpu_sample, global_batch=args.cpu_sample, parallelism='cpu',
                      optimizer='dense Keras-Adam on every tensor (user table included)',
                      workload=config['workload'].rsplit(',', 1)[0] + ', B=%d per step on the CPU arm' % args.cpu_sample)
        line = dict(metric=METRIC, value=r['value'], unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                    ms_per_step=r['ms_per_step'], higher_is_better=True, scaling=args.scaling, vs_baseline=None, dtype='f32',
                    data='synthetic', impl='reference', config=config,
                    cpu_baseline=dict(value=r['value'], unit=UNIT, cores=r['cores'], kind=r['kind'], sample=r['sample']),
                    e2e=dict(value=r['value'], unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist
    from mnexp_b200 import _lib
    from mnexp_b200.dist import DataParallel, init_process_group
    from mnexp_b200.engine import LsturEngine
    torch.cuda.set_device(local_rank)
    if world > 1:
        init_process_group(local_rank)
    lib = _lib.load()
    precision = args.precision
    if precision == 'auto':
        precision = 'fp16_tc' if lib.lstur_tc_supported(sh.L, sh.E, sh.F, sh.k) else 'fp32'
    n_batches = 6 if sh.name != 'C5' else 3
    tok, P, batches, pad_frac = build_workload(sh, n_batches, rank, B, full_history=args.full_history)
    eng = LsturEngine(P, B, sh.W, 1 + sh.K, sh.L, arch=sh.arch, doc_tokens=tok, dropout=0.2, lr=1e-3,
                      precision=precision, sparse_user_adam=True, trainable_word_emb=args.trainable_emb)
    dp = DataParallel(eng)
    dbs = [eng.to_device_batch(b) for b in batches]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up
    for i in range(args.warmup):
        dp.train_step(dbs[i % n_batches])
    barrier()
    # ---- timed region: device-resident inputs, CUDA events, probe events around the dominant kernel
    probe_id = 1
    probes = [(eng.new_event(), eng.new_event()) for _ in range(args.steps)]
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    barrier()
    l0 = lib.lstur_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    t_host = time.perf_counter()
    for i in range(args.steps):
        eng.set_probe(probe_id, *probes[i])
        dp.train_step(dbs[i % n_batches])
    host_enqueue_ms = 1e3 * (time.perf_counter() - t_host) / args.steps      # CPU time to enqueue a step (no sync inside)
    ev1.record()
    barrier()
    launches = int(lib.lstur_launch_count() - l0)
    eng.set_probe(0)
    clocks = sampler.stop() if rank == 0 else None
    ms = torch.tensor([ev0.elapsed_time(ev1)], device='cuda')
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms[0])
    value = B * world * args.steps / (ms_total / 1e3)
    probe_ms = float(np.mean([eng.elapsed_ms(a, b) for a, b in probes]))
    loss_last = eng.loss()
    # taken before the e2e and extra passes below train the engine further
    outputs = last_step_outputs(torch, eng, batches[(args.steps - 1) % n_batches]) if args.dump_outputs and rank == 0 else None

    # ---- e2e: host (pinned) batches in, loss out, every step
    e2e = None
    if not args.no_e2e:
        hb = [{k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for k, v in b.items()} for b in batches]
        h2d = sum(int(t.numel() * t.element_size()) for t in hb[0].values())
        for i in range(2):
            float(dp.train_step(eng.to_device_batch(hb[i], non_blocking=True))[0])
        barrier()
        ev0.record()
        for i in range(args.steps):
            db = eng.to_device_batch(hb[i % n_batches], non_blocking=True)
            loss_host = float(dp.train_step(db)[0].item())
        ev1.record()
        barrier()
        ms2 = torch.tensor([ev0.elapsed_time(ev1)], device='cuda')
        if world > 1:
            dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
        e2e = dict(value=B * world * args.steps / (float(ms2[0]) / 1e3), unit=UNIT, h2d_bytes_per_step=h2d,
                   d2h_bytes_per_step=4, api='LsturEngine.train_step(doc-id batch from pinned host memory) -> loss.item()')

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return 0
    pk, pk_kind = peaks()
    fl = flops_per_impression(sh, args.trainable_emb)
    tensor_peak = pk['bf16_tflops_sustained']
    # the tensor-core kernels run over the live titles only (an all-pad title is exactly zero in value and gradient): the
    # kernel's own utilisation is quoted on the FLOPs it executes, the algorithmic rate (what the reference graph computes,
    # pad titles included) beside it
    T_ = sh.W + 1 + sh.K
    live_frac = 1.0
    if precision != 'fp32':
        live_frac = float(np.mean([((b['hist_doc'] != 0).sum() + b['cand_doc'].size) / float(B * T_) for b in batches]))
    conv_tflops_alg = fl['conv_fwd'] * B / (probe_ms / 1e3) / 1e12
    conv_tflops = conv_tflops_alg * live_frac
    traffic, traffic_src = ncu_traffic('news_conv_tc') if (B == sh.B and sh.name == 'C3') else (None, None)
    T = sh.W + 1 + sh.K
    gather_bytes = B * T * sh.L * (4 + sh.E * 2)          # SURVEY §8d: tok * (4 + E * s), 16-bit table
    roofline = dict(bound='tensor', kernel='title Conv1D forward (implicit GEMM, fused gather + attention pooling), precision=%s' % precision,
                    achieved=conv_tflops, peak=tensor_peak, unit='TFLOP/s', frac=conv_tflops / tensor_peak,
                    achieved_note='executed FLOPs (live titles only) / kernel time', live_title_frac=live_frac,
                    algorithmic_tflops=conv_tflops_alg, traffic=traffic,
                    traffic_unit='bytes of DRAM traffic per launch (ncu --set full, profiles/%s)' % traffic_src,
                    peak_kind='%s bf16_tflops_sustained' % pk_kind, kernel_ms=probe_ms,
                    fused_gather_gbs=gather_bytes / (probe_ms / 1e3) / 1e9,
                    fused_gather_note='algorithmic gather bytes (ids + 16-bit rows) over the fused kernel\'s time; the rows come from L2 '
                                      '(profiles/r02_ncu_l2_traffic.txt: lts__t_sectors of the kernel, 79.9 % L2 hit rate, 0.04 GB of DRAM reads), so this is '
                                      'not an HBM roofline',
                    step_frac_of_train_roofline=(value / world) * fl['train'] / (tensor_peak * 1e12),
                    flops_per_impression_train=fl['train'])
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_reference_run(sh, 6, 1, args.cpu_sample, trainable_emb=args.trainable_emb)
        cpu.pop('ms_per_step', None)
    extra = None
    if world == 1 and not args.no_extras:
        extra = extra_records(torch, lib, sh, eng, dbs, batches, tok, P, precision, pk, args, B, live_frac)
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
                ms_per_step=ms_total / args.steps, higher_is_better=True, scaling=args.scaling, vs_baseline=None,
                dtype={'bf16_tc': 'bf16', 'fp16_tc': 'f16'}.get(precision, 'f32'), data='synthetic',
                config=dict(config, precision=precision, l2='inputs larger than L2: %d distinct batches, >%d MB activations per step'
                                                          % (n_batches, eng.ws_bytes >> 20),
                            user_adam='row-sparse (documented deviation from dense Keras-Adam)', hist_pad_frac=round(pad_frac, 3)),
                roofline=roofline, cpu_baseline=cpu, e2e=e2e, gpu_launches=launches, clocks=clocks, loss=loss_last,
                host_enqueue_ms_per_step=host_enqueue_ms, extra=extra)
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == '__main__':
    sys.exit(main())
