#!/usr/bin/env python
"""bench.py -- articles/sec of the DAE-with-triplet-loss training hot path (BASELINE.json metric).

    python bench.py [--config C1|C2|C3|C4|C5] [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A "step" is one training step (corrupt -> encode -> decode -> loss -> triplet mining -> backward -> optimizer) on one batch of
B = 800 articles.  Default workload = BASELINE.json configs[1] (C2): 100 000 synthetic articles per rank, 10 000-dim sparse TF-IDF
(1 % nnz), 500 hidden units, batch_all triplet loss, sigmoid/sigmoid, cross-entropy, SGD.  The other configs of BASELINE.json are
selectable (`--config`); their lines are committed under profiles/.
N > 1: one process per GPU under torchrun (weak scaling: every rank trains B rows per step on its own shard, ONE exchange of the
flat gradient per step).

`--impl reference` times the reference algorithm restated on PyTorch-CPU (oracle/dae_oracle.py; TensorFlow 1.12 cannot be installed
offline) on the host cores, same config.

`--dump-outputs DIR` writes what the K-th step of the (first) timed window left to its caller -- the parameters enc_w, enc_b, dec_b
and the step's scalars -- as DIR/<name>.npy.  Data, corruption and the epoch permutations are seeded, so the same arguments feed the
same inputs and two runs agree to rounding (the kernels accumulate with float atomics).
"""
import argparse
import gc
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

_COMMON = dict(F=10000, H=500, B=800, mean_nnz=100, n_classes=4, loss='cross_entropy', enc='sigmoid', dec='sigmoid',
               opt='gradient_descent', lr=0.1, corr_frac=0.3, alpha=1.0, rows=100000)
CONFIGS = {
    # BASELINE.json configs[0]: the reference's own CPU-runnable case, real data (fixture written by tools/make_uci_fixture.py)
    'C1': dict(_COMMON, name='C1: UCI news 8000 x 10000 binary, H=500, triplet_strategy none, SGD, B=800', kind='uci', strategy='none',
               rows=8000),
    'C2': dict(_COMMON, name='C2: synthetic tf-idf 10000-dim 1% nnz, H=500, batch_all, B=800', kind='tfidf', strategy='batch_all'),
    # 1M articles over 8 ranks = 125 000 rows per rank (what one rank of the 8-GPU job holds)
    'C3': dict(_COMMON, name='C3: synthetic binary 10000-dim 1% nnz, masking 0.3, H=500, batch_hard, B=800 per rank', kind='binary',
               strategy='batch_hard', rows=125000),
    'C4': dict(_COMMON, name='C4: synthetic tf-idf 50000-dim 0.2% nnz, H=1000, batch_all, B=800 (CSR-SpMM stress)', kind='tfidf',
               strategy='batch_all', F=50000, H=1000),
    # 200k (anchor, pos, neg) triples over 4 ranks = 50 000 per rank; a step encodes/decodes 3 x 800 rows
    'C5': dict(_COMMON, name='C5: explicit (anchor,pos,neg) triplets, binary 10000-dim 1% nnz, H=500, alpha=1, B=800 triples per rank',
               kind='binary', strategy='explicit', rows=50000),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--config', default='C2', choices=sorted(CONFIGS))
    ap.add_argument('--rows', type=int, default=0, help='articles per rank (default: the config\'s count)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-fit-api', action='store_true', help='skip the DenoisingAutoencoder.fit measurement')
    ap.add_argument('--no-graph', action='store_true', help='launch the step eagerly instead of replaying the captured CUDA graph')
    ap.add_argument('--cpu-steps', type=int, default=3)
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the parameters and scalars of the last timed step as DIR/<name>.npy (same arguments, same inputs)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    return args


def make_data(w, n_rows, seed):
    """-> (x, labels) or, for the explicit-triplet config, ({'org','pos','neg'}, None)."""
    from dae_rnn_news_recommendation_b200.synth import make_sparse, make_labels, perturb_rows
    if w['kind'] == 'uci':
        z = np.load(os.path.join(ROOT, 'tests', 'golden', 'uci_c1.npz'))
        import scipy.sparse as sp
        shape = tuple(int(v) for v in z['train_shape'])
        ind, ptr = z['train_indices'].astype(np.int32), z['train_indptr'].astype(np.int64)
        x = sp.csr_matrix((np.ones(len(ind), dtype=np.float32), ind, ptr), shape=shape)
        reps = -(-n_rows // shape[0])
        if reps > 1:
            x = sp.vstack([x] * reps).tocsr()
        return x[:n_rows], np.zeros(n_rows, np.float32)
    if w['strategy'] == 'explicit':
        org = make_sparse(n_rows, w['F'], w['mean_nnz'], 'binary', seed=seed)
        pos = perturb_rows(org, 0.3, seed=seed + 1)
        neg = make_sparse(n_rows, w['F'], w['mean_nnz'], 'binary', seed=seed + 2)
        return {'org': org, 'pos': pos, 'neg': neg}, None
    x = make_sparse(n_rows, w['F'], w['mean_nnz'], w['kind'], seed=seed)
    return x, make_labels(n_rows, w['n_classes'], seed=seed)


def xavier(F, H, seed=0):
    b = np.sqrt(6.0 / (F + H))
    return np.random.default_rng(seed).uniform(-b, b, (F, H)).astype(np.float32)


# ----------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port (reference algorithm on PyTorch-CPU), used for cpu_baseline and --impl reference
# ----------------------------------------------------------------------------------------------------------------------
def cpu_steps(w, x, labels, n_steps, n_warm, seed=0, threads=None):
    import torch
    from oracle.dae_oracle import OracleDAE, masking_noise
    torch.set_num_threads(threads or os.cpu_count())
    B = w['B']
    explicit = w['strategy'] == 'explicit'
    model = OracleDAE(xavier(w['F'], w['H'], seed), enc_act_func=w['enc'], dec_act_func=w['dec'], loss_func=w['loss'],
                      opt=w['opt'], learning_rate=w['lr'], alpha=w['alpha'],
                      triplet_strategy='none' if explicit else w['strategy'])
    rng = np.random.RandomState(seed)
    times = []
    for s in range(n_steps + n_warm):
        t0 = time.perf_counter()
        sl = slice(s * B, (s + 1) * B)
        if explicit:
            xs = [x[k][sl] for k in ('org', 'pos', 'neg')]
            model.step_explicit(xs, [masking_noise(m, w['corr_frac'], rng) for m in xs])
        else:
            xb = x[sl]
            xc = masking_noise(xb, w['corr_frac'], rng)       # host corruption + batching are inside the reference's window
            model.step(xb, xc, labels[sl])
        if s >= n_warm:
            times.append(time.perf_counter() - t0)
    return times


def best_cpu_threads(w, x, labels):
    """The reference arm gets the thread count it is FASTEST with: the B x B x B elementwise chain is memory-bound and slows down
    when a 128-core host runs it on every core.  One probe step per candidate; returns (threads, seconds of the best probe)."""
    n = os.cpu_count() or 1
    best = None
    for t in sorted({n, min(n, 32), min(n, 64)}, reverse=True):
        dt = cpu_steps(w, x, labels, 1, 1, threads=t)[0]
        if best is None or dt < best[1]:
            best = (t, dt)
    return best


def cpu_info():
    model = ''
    try:
        for line in open('/proc/cpuinfo'):
            if line.startswith('model name'):
                model = line.split(':', 1)[1].strip()
                break
    except OSError:
        pass
    return model


def run_reference(args):
    """Reference arm: rank 0 only; bounded so the run ends within a few minutes."""
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    w = CONFIGS[args.config]
    B = w['B']
    warm = 1
    x, labels = make_data(w, (warm + 1) * B, seed=0)
    threads, t_probe = best_cpu_threads(w, x, labels)
    budget = 120.0
    k = int(max(1, min(args.steps, budget // max(t_probe, 1e-3))))
    x, labels = make_data(w, (k + 1) * B, seed=1)
    times = cpu_steps(w, x, labels, k, 1, threads=threads)
    t = float(np.sum(times))
    val = k * B / t
    out = {'impl': 'reference', 'metric': 'articles/sec', 'value': val, 'unit': 'articles/s', 'n_gpus': args.gpus, 'steps': k,
           'steps_requested': args.steps, 'warmup': 1, 'ms_per_step': 1e3 * t / k, 'higher_is_better': True,
           'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'real (UCI news fixture)' if w['kind'] == 'uci' else 'synthetic',
           'config': {'workload': w['name'], 'global_batch': B, 'note': 'reference algorithm restated on PyTorch-CPU '
                      '(TF 1.12 unavailable offline); steps capped to fit ~120 s after the thread-count probes'},
           'cpu_baseline': {'value': val, 'unit': 'articles/s', 'cores': threads, 'kind': 'port',
                            'sample': '%d steps of B=%d on %d of %d host threads (the fastest of the probed counts; %s)'
                                      % (k, B, threads, os.cpu_count(), cpu_info())},
           'e2e': {'value': val, 'unit': 'articles/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(out))


# ----------------------------------------------------------------------------------------------------------------------
# clocks sampler: NVML polled from a thread (nvidia-smi's loop mode block-buffers its pipe and starts too slowly for a
# timed region of a few milliseconds)
# ----------------------------------------------------------------------------------------------------------------------
class Clocks:
    REASONS = {0x8: 'hw_slowdown', 0x40: 'hw_thermal_slowdown', 0x20: 'sw_thermal_slowdown', 0x4: 'sw_power_cap'}

    def __init__(self, index, period_s=0.0005):
        self.index, self.samples, self.stop_flag, self.thr, self.h, self.err = index, [], False, None, None, None
        self.period_s = period_s

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get('CUDA_VISIBLE_DEVICES')
            idx = int(vis.split(',')[self.index]) if vis and vis.split(',')[self.index].isdigit() else self.index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nv = pynvml
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:   # noqa: BLE001
            self.err = repr(e)
            return
        self.thr = threading.Thread(target=self._poll, daemon=True)
        self.thr.start()

    def _poll(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:   # noqa: BLE001
                    rs = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.samples.append((time.time(), sm, rs))
            except Exception as e:   # noqa: BLE001
                self.err = repr(e)
                return
            time.sleep(self.period_s)

    def stop(self, t0, t1):
        self.stop_flag = True
        if self.thr is not None:
            self.thr.join(timeout=2.0)
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples: %s' % self.err], 'samples': 0}
        sel = [s for s in self.samples if t0 <= s[0] <= t1]
        inside = len(sel)
        if not sel:   # the timed region was shorter than one NVML poll: take the samples around it
            sel = [s for s in self.samples if t0 - 0.05 <= s[0] <= t1 + 0.05] or self.samples
        reasons = set()
        for _, _, rs in sel:
            for bit, name in self.REASONS.items():
                if rs & bit:
                    reasons.add(name)
        return {'sm_mhz': float(np.median([s[1] for s in sel])), 'sm_max_mhz': self.max_sm, 'reasons': sorted(reasons),
                'samples': len(sel), 'samples_inside_timed_region': inside, 'source': 'NVML polled every ~%g ms' % (self.period_s * 1e3)}


# ----------------------------------------------------------------------------------------------------------------------
# roofline bookkeeping: ALGORITHMIC work per launch of each kernel tag (DESIGN.md section 4)
# ----------------------------------------------------------------------------------------------------------------------
def kernel_work(tag, w, s):
    """-> (bound, work per launch).  s: measured batch statistics (nnz per batch, kept nnz, distinct columns, valid triplets)."""
    F, H = w['F'], w['H']
    B = w['B'] * (3 if w['strategy'] == 'explicit' else 1)      # rows through the encode / decode kernels per step
    Hp = (H + 1 + 63) // 64 * 64
    if tag in ('gemm_decode_fwd', 'gemm_decode_dW', 'gemm_decode_dE'):
        return 'tensor', 2.0 * B * F * H
    if tag in ('gemm_gram', 'gemm_dE_tri'):
        return 'tensor', 2.0 * B * B * H
    if tag == 'dae_encode_csr_fwd':     # CSR stream (all stored entries are read), touched W rows once, E + its bf16 hi/lo copy out
        return 'hbm', s['nnz'] * 8.0 + (B + 1) * 8.0 + s['cols'] * H * 4.0 + H * 4.0 + B * H * 4.0 + B * Hp * 4.0
    if tag == 'dae_encode_csr_bwd':     # CSR stream, dE in / dA out once, bucketed entries out + in, touched dW rows read-modify-write
        return 'hbm', s['nnz'] * 8.0 + 2.0 * B * H * 4.0 + s['nnz_c'] * 24.0 + s['cols_c'] * H * 8.0
    if tag == 'dae_optimizer_step':     # theta, grad in; theta + bf16 hi/lo of W out
        return 'hbm', 3.0 * (F * H + F + H) * 4.0 + F * Hp * 4.0
    if tag == 'dae_triplet_batch_all':
        return 'issue', s['triplets']
    if tag == 'dae_triplet_batch_hard':
        return 'hbm', 3.0 * B * B * 4.0
    return None, 0.0


DUMP_W_BYTES = 60_000_000     # the encoder weights' share of the 64 MB that --dump-outputs may write


def dump_outputs(dirname, F, H, theta, stats):
    """What a caller of the training step holds after it: the updated parameters (float32) and the step's scalars (float64, the
    slots of _cabi.STAT).  A weight matrix above DUMP_W_BYTES is written as a fixed, seeded sample of its rows (sorted)."""
    os.makedirs(dirname, exist_ok=True)
    theta = theta.cpu().numpy()
    W = theta[:F * H].reshape(F, H)
    out = {'enc_b': theta[F * H:F * H + H], 'dec_b': theta[F * H + H:], 'step_stats': stats.cpu().numpy()}
    if W.nbytes <= DUMP_W_BYTES:
        out['enc_w'] = W
    else:
        rows = np.sort(np.random.default_rng(0).choice(F, DUMP_W_BYTES // W[0].nbytes, replace=False))
        out['enc_w_row_sample'] = W[rows]
    for name, a in out.items():
        np.save(os.path.join(dirname, name + '.npy'), a)


def batch_stats(w, x, labels, rng):
    """Per-batch figures of the algorithmic-work model, measured on one host-side sample batch."""
    B = w['B']
    if w['strategy'] == 'explicit':
        xb = [x[k][:B] for k in ('org', 'pos', 'neg')]
        nnz = sum(m.nnz for m in xb)
        idx = np.concatenate([m.indices for m in xb])
    else:
        xb = x[:B]
        nnz, idx = xb.nnz, xb.indices
    keep = rng.random(len(idx)) >= w['corr_frac']
    s = {'nnz': float(nnz), 'nnz_c': float(keep.sum()), 'cols': float(len(np.unique(idx))), 'cols_c': float(len(np.unique(idx[keep]))),
         'triplets': 0.0}
    if w['strategy'] == 'batch_all':
        _, cnt = np.unique(labels[:B], return_counts=True)
        s['triplets'] = float(np.sum(cnt * (cnt - 1.0) * (B - cnt)))
    return s


def main():
    args = parse()
    if args.impl == 'reference':
        run_reference(args)
        return
    import torch
    import torch.distributed as dist
    from dae_rnn_news_recommendation_b200.engine import TrainEngine, DeviceCSR, HostFeed
    import scipy.sparse as sp
    w = CONFIGS[args.config]
    world = int(os.environ.get('WORLD_SIZE', 1))
    rank = int(os.environ.get('RANK', 0))
    local = int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    B, F, H, K, W = w['B'], w['F'], w['H'], args.steps, max(args.warmup, 3)
    explicit = w['strategy'] == 'explicit'
    n_rows = args.rows or w['rows']
    x, labels = make_data(w, n_rows, seed=1000 + rank)
    stats = batch_stats(w, x, labels, np.random.default_rng(5))

    eng = TrainEngine(F, H, enc_act_func=w['enc'], dec_act_func=w['dec'], loss_func=w['loss'], opt=w['opt'],
                      learning_rate=w['lr'], alpha=w['alpha'], triplet_strategy=w['strategy'], device=dev)
    eng.set_parameters(xavier(F, H, 0))
    if explicit:
        csr = DeviceCSR(sp.vstack([x['org'], x['pos'], x['neg']]).tocsr(), dev)
        eng.set_data(csr, None, None)
    else:
        csr = DeviceCSR(x, dev)
        eng.set_data(csr, None, torch.from_numpy(labels).to(dev))
    steps_per_epoch = n_rows // B
    perm_buf = torch.zeros(n_rows, dtype=torch.int32, device=dev)
    use_graph = not args.no_graph
    perm_gen = torch.Generator(device=dev)
    perm_gen.manual_seed(4321 + rank)        # the default CUDA generator is seeded differently in every process

    def epoch_start(epoch):
        eng.corrupt_masking(w['corr_frac'], seed=1234 + rank, epoch=epoch)           # utils.masking_noise, on device
        perm_buf.copy_(torch.randperm(n_rows, device=dev, dtype=torch.int32, generator=perm_gen))   # utils.gen_batches shuffle

    def eager_step(offset, log_row):
        if explicit:
            eng.step_explicit(perm_buf, offset, B, n_rows, log_row)
        else:
            eng.step(perm_buf, offset, B, log_row)

    state = {'epoch': -1}

    def run(n, first_step, log=None, graph=False):
        """n steps starting at global step `first_step`; epoch boundaries re-corrupt + re-shuffle inside the window."""
        for i in range(n):
            ep, in_epoch = divmod(first_step + i, steps_per_epoch)
            if ep != state['epoch']:
                epoch_start(ep)
                state['epoch'] = ep
            if graph and (i == 0 or in_epoch == 0):
                eng.set_step_cursor(in_epoch * B, i)
            if graph:
                eng.replay_step()
            else:
                eager_step(in_epoch * B, None if log is None else log[i])

    run(W, 0)  # warm-up (also allocates the workspaces)
    torch.cuda.synchronize()

    # -- per-kernel pass: every kernel bracketed by CUDA events, the step serialised on ONE stream (no branch overlap), and the
    #    stream PRE-LOADED behind a spin kernel so that the host's launch latency (tensor-map encodes, 8 ranks sharing the cores)
    #    cannot sit between an event pair: the durations are device time only and do not depend on the rank count.
    tags = ['gemm_decode_fwd', 'gemm_decode_dW', 'gemm_decode_dE', 'gemm_gram', 'gemm_dE_tri', 'dae_encode_csr_fwd',
            'dae_encode_csr_bwd', 'dae_triplet_batch_all', 'dae_triplet_batch_hard', 'dae_triplet_explicit',
            'dae_batch_prepare', 'dae_batch_prepare_explicit', 'dae_step_finalize', 'dae_optimizer_step']

    def profile(first_step, n=3):
        fork = eng.fork_branches
        eng.fork_branches = False
        eng.time_kernels(tags)
        torch.cuda.synchronize()
        torch.cuda._sleep(60_000_000)          # ~30 ms of device spin: the n steps below are fully enqueued before they start
        run(n, first_step)
        out = {k: float(np.sum(v)) / n for k, v in eng.kernel_times_ms().items() if v}
        eng.time_kernels(None)
        eng.fork_branches = fork
        return out

    # -- timed region: EXACTLY K steps, barrier + synchronize on both sides, CUDA events, max over ranks.  The window starts at an
    #    epoch boundary, so ONE corruption pass over the rank's whole set and ONE permutation are inside it.
    first = -(-(W) // steps_per_epoch) * steps_per_epoch
    log = torch.zeros(K, 16, dtype=torch.float64, device=dev)
    if use_graph:
        eng.capture_step_graph(perm_buf, B, log, explicit_n=n_rows if explicit else None)   # one CUDA graph of the whole step
    def timed_window(first):
        launches0 = eng.launches
        # multi-GPU: NVML calls from a process whose kernels talk to peer / multicast memory stall those kernels (measured at 2 GPUs with a
        # 0.5 ms poll: 0.31 -> 0.47 ms per step with NCCL, 0.33 -> 1.4 ms with the in-switch exchange; at 8 GPUs a 5 ms poll still cost NCCL
        # 0.38 -> 0.99 ms), so the poll is 20x coarser there: the samples fall into the spin kernel that precedes the steps and into the steps
        clocks = Clocks(local, period_s=0.0005 if world == 1 else 0.01)
        if rank == 0:
            clocks.start()
            time.sleep(0.05)
        # a generation-2 collection of the interpreter (torch + scipy keep ~1 M tracked objects alive: tens of ms) must not fall between
        # two graph launches of a 5 ms timed region: collect now, then keep the collector off inside the timed regions
        gc.collect()
        gc.freeze()
        gc.disable()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        # device time, not host hiccups: the K steps (and the epoch-start work) are enqueued BEHIND a ~15 ms spin kernel, so the events
        # bracket back-to-back device execution even if a host thread (NVML poll, another rank's process) delays a launch call
        torch.cuda._sleep(30_000_000)
        t_wall0 = time.time()
        e0.record()
        run(K, first, log=log, graph=use_graph)
        e1.record()
        torch.cuda.synchronize()
        t_wall1 = time.time()
        if world > 1:
            dist.barrier()
        ms = e0.elapsed_time(e1)
        gpu_launches = eng.launches - launches0
        clk = clocks.stop(t_wall0, t_wall1) if rank == 0 else None
        tms = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        ms = float(tms.item())
        return ms, gpu_launches, clk

    ms, gpu_launches, clk = timed_window(first)
    losses = log.cpu().numpy()
    # the first window's K-th step: its inputs do not depend on whether a host-stalled window is re-measured below
    last_step = (eng.theta.clone(), log[K - 1].clone()) if args.dump_outputs else None
    prof = profile(first + K)
    # validity guard: the overlapped step cannot take longer than its kernels run one after another on ONE stream (`prof`, device time)
    # plus the gradient exchange.  A window above 1.25x that bound had the GPU idle waiting for the host (a stalled launch call: seen
    # about once in a dozen runs on shared boxes, 1.3 ms per step instead of 0.22) and is re-measured, at most twice, every attempt
    # again EXACTLY K steps from an epoch boundary; all attempts are reported in config.timed_windows_ms_per_step.
    lim = torch.tensor([1.25 * sum(prof.values()) + (0.3 if world > 1 else 0.0)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(lim, op=dist.ReduceOp.MAX)
    attempts = [ms / K]
    while use_graph and attempts[-1] > float(lim.item()) and len(attempts) < 3:
        first = -(-(first + K + 8) // steps_per_epoch) * steps_per_epoch
        ms, gpu_launches, clk = timed_window(first)
        losses = log.cpu().numpy()
        attempts.append(ms / K)
    value = K * B * world / (ms * 1e-3)

    # -- e2e: per-step HOST feed (pinned) -> H2D -> step -> D2H of the step's scalars, through TrainEngine.run_feed
    Ke = min(K, 20)
    rng = np.random.RandomState(7 + rank)
    batches = []
    for i in range(Ke + 2):
        idx = rng.randint(0, n_rows, B)
        xb = sp.vstack([x[k][idx] for k in ('org', 'pos', 'neg')]).tocsr() if explicit else x[idx]
        keep = rng.rand(xb.nnz) >= w['corr_frac']
        batches.append((xb, xb.data * keep, None if explicit else labels[idx]))
    cap = max(b[0].nnz for b in batches)   # one device layout for every feed -> the step is captured once and replayed
    feeds = [HostFeed(xb, xc, lb, cap_nnz=None if args.no_graph else cap) for xb, xc, lb in batches]
    for f in feeds[:2]:
        eng.run_feed(f)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for f in feeds[2:]:
        eng.run_feed(f)                      # synchronous: H2D -> step -> D2H -> host sync, every step (session.run semantics)
    f1.record()
    torch.cuda.synchronize()
    tme = torch.tensor([f0.elapsed_time(f1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tme, op=dist.ReduceOp.MAX)
    e2e_sync = Ke * B * world / (float(tme.item()) * 1e-3)
    e2e_val, e2e_api = e2e_sync, 'TrainEngine.run_feed(HostFeed) per step: pinned host batch -> H2D -> step -> D2H scalars, synchronised'
    if not args.no_graph:                    # streamed: the same copies every step, the next feed's H2D overlapping the current step
        eng.run_feeds(feeds[:2])
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        f0.record()
        eng.run_feeds(feeds[2:])             # Ke feeds, every one copied H2D inside the window (pipeline fill and drain included)
        f1.record()
        torch.cuda.synchronize()
        tme = torch.tensor([f0.elapsed_time(f1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tme, op=dist.ReduceOp.MAX)
        e2e_val = Ke * B * world / (float(tme.item()) * 1e-3)
        e2e_api = ('TrainEngine.run_feeds(HostFeeds): per step a pinned host batch -> H2D (copy stream, overlapping the previous step) -> '
                   'step (the next batch\'s label sort staged on a side branch) -> async D2H of the scalars; one host sync after the last step')
    h2d = int(np.mean([f.nbytes for f in feeds[2:]]))

    # -- roofline table (every kernel of the step) and the longest kernel's entry
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except (OSError, ValueError):
        pass
    src = 'MEASURED_PEAKS.json' if peaks else 'fallback (B200_PROFILING.md)'
    sm_clk = peaks.get('sm_max_mhz', 1965.0) * 1e6
    PEAK = {'tensor': (peaks.get('bf16_tflops_sustained', 1400.0), 'TFLOP/s', 1e12, src + ' bf16_tflops_sustained'),
            'hbm': (peaks.get('hbm_gbs', 6650.0), 'GB/s', 1e9, src + ' hbm_gbs'),
            # fp32 issue slots: 148 SMs x 128 lanes x clock, at the formulation's minimum of 8 instructions per triplet
            'issue': (148 * 128 * sm_clk / 8.0 / 1e9, 'Gtriplet/s', 1e9, '148 SMs x 128 fp32 lanes x %.0f MHz / 8 instr per triplet' % (sm_clk / 1e6))}
    traffic_tab = {}
    try:  # DRAM bytes per launch from the committed `ncu --set full` capture (profiles/traffic.json)
        traffic_tab = json.load(open(os.path.join(ROOT, 'profiles', 'traffic.json')))
    except (OSError, ValueError):
        pass
    table = {}
    for tag, t_ms in prof.items():
        bound, work = kernel_work(tag, w, stats)
        row = {'ms': t_ms, 'share_of_serialised_step': t_ms / sum(prof.values())}
        if bound:
            peak, unit, scale, psrc = PEAK[bound]
            ach = work / (t_ms * 1e-3) / scale
            row.update(bound=bound, work=work, achieved=ach, peak=peak, unit=unit, frac=ach / peak)
        table[tag] = row
    dominant = max(prof, key=prof.get)
    d = table[dominant]
    tj = traffic_tab.get(dominant, {}) if args.config == 'C2' else {}
    roofline = {'kernel': dominant, 'bound': d.get('bound', 'latency'), 'achieved': d.get('achieved'), 'peak': d.get('peak'),
                'unit': d.get('unit'), 'frac': d.get('frac'), 'traffic': tj.get('traffic_bytes'), 'algorithmic_work': d.get('work'),
                'ncu': {k: v for k, v in tj.items() if k != 'traffic_bytes'},
                'peak_source': PEAK[d['bound']][3] if 'bound' in d else None,
                'note': ('algorithmic FLOPs = 2*M*N*K; the kernel executes 3x that as bf16 MMAs (hi/lo split) for fp32 parity'
                         if d.get('bound') == 'tensor' else
                         'valid triplets per launch; neither HBM- nor tensor-bound: the B^3 sweep runs out of registers' if d.get('bound') == 'issue' else ''),
                'avg_launch_ms': d['ms'], 'share_of_step': d['ms'] / (ms / K),
                'timing': 'CUDA events around each launch, step serialised on one stream, stream pre-loaded (device time only)'}

    # -- the public estimator API: DenoisingAutoencoder(.Triplet).fit on the same data, articles/s in the reference's own
    #    train_time window (corruption + permutation + every step of an epoch, autoencoder.py:193-197), last of 3 epochs
    fit_api = None
    set_mb, exchange = csr.h2d_bytes / 1e6 + csr.nnz * 4 / 1e6, eng.allreduce_mode
    if not args.no_fit_api and world == 1:   # (single process: the estimator's data-parallel path is covered by tests/test_gpu_multi.py)
        import tempfile
        from dae_rnn_news_recommendation_b200.autoencoder import DenoisingAutoencoder, DenoisingAutoencoderTriplet
        torch.cuda.empty_cache()
        cwd = os.getcwd()
        with tempfile.TemporaryDirectory() as td:
            os.chdir(td)
            try:
                kw = dict(model_name='bench', main_dir='bench', compress_factor=F // H, enc_act_func=w['enc'], dec_act_func=w['dec'],
                          loss_func=w['loss'], num_epochs=3, batch_size=B, opt=w['opt'], learning_rate=w['lr'], corr_type='masking',
                          corr_frac=w['corr_frac'], verbose=0, verbose_step=100, seed=0, alpha=w['alpha'], device=str(dev))
                if explicit:
                    m = DenoisingAutoencoderTriplet(**kw)
                    m.fit(x)
                else:
                    m = DenoisingAutoencoder(triplet_strategy=w['strategy'], **kw)
                    m.fit(x, train_set_label=labels)
                t = torch.tensor([m.train_time], dtype=torch.float64, device=dev)
                if world > 1:
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                rows_epoch = (n_rows // (B * world)) * B * world if world > 1 else n_rows
                fit_api = {'value': rows_epoch / float(t.item()), 'unit': 'articles/s', 'epoch_s': float(t.item()), 'rows_per_epoch': rows_epoch,
                           'api': '%s.fit, rng_mode=device, train_time of the 3rd epoch' % type(m).__name__}
                del m
            finally:
                os.chdir(cwd)

    gc.enable()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, F, H, *last_step)

    cpu_baseline = None
    if not args.no_cpu_baseline:
        n = max(1, args.cpu_steps)
        xs, ls = make_data(w, (n + 1) * B, seed=1)
        threads, _ = best_cpu_threads(w, xs, ls)
        ts = cpu_steps(w, xs, ls, n, 1, threads=threads)
        cpu_baseline = {'value': n * B / float(np.sum(ts)), 'unit': 'articles/s', 'cores': threads, 'kind': 'port',
                        'sample': '%d steps of B=%d after 1 warm-up step on %d of %d host threads (the fastest of the probed counts), '
                                  'reference algorithm restated on PyTorch-CPU (%s)' % (n, B, threads, os.cpu_count(), cpu_info())}

    state_mb = (3 * (F * H + F + H) * 4 + 2 * F * ((H + 64) // 64 * 64) * 2 + 2 * B * ((F + 31) // 32 * 32) * 2) / 1e6
    out = {
        'metric': 'articles/sec', 'value': value, 'unit': 'articles/s', 'n_gpus': world, 'steps': K, 'warmup': W,
        'ms_per_step': ms / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
        'data': 'real (UCI news fixture tests/golden/uci_c1.npz)' if w['kind'] == 'uci' else 'synthetic',
        'config': {'workload': w['name'], 'global_batch': B * world, 'rows_per_rank': n_rows, 'parallelism': 'dp%d' % world,
                   'l2': 'inputs larger than L2: every step gathers %d fresh rows of the %.0f MB device-resident set (CSR + corrupted values) '
                         'and streams %.0f MB of parameter / gradient / operand state; L2 is 126 MB'
                         % (B * (3 if explicit else 1), set_mb, state_mb),
                   'window': 'K steps from an epoch boundary: one corruption pass over the set and one permutation inside; CUDA events '
                             'around the K steps, which are enqueued behind a 15 ms spin kernel (device time without host launch hiccups)',
                   'loss_first_last': [float(losses[0, 0]), float(losses[-1, 0])],
                   'timed_windows_ms_per_step': attempts,     # more than one entry: a host-stalled window was re-measured (see bench.py)
                   'launch': 'cuda graph replay' if use_graph else 'eager', 'grad_exchange': exchange},
        'clocks': clk,
        'e2e': {'value': e2e_val, 'unit': 'articles/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': 128, 'steps': Ke, 'api': e2e_api,
                'synchronous_per_step': {'value': e2e_sync, 'api': 'TrainEngine.run_feed(HostFeed): host sync after every step'}},
        'fit_api': fit_api,
        'gpu_launches': gpu_launches,
        'roofline': roofline,
        'kernels': table,
        'batch_stats': stats,
        'cpu_baseline': cpu_baseline,
    }
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
