#!/usr/bin/env python
"""bench.py -- samples/sec of the DeepFM Criteo-shape training step (BASELINE.json config 2) on the fused sm_100a
sparse path, driven through the product surface: EasyRecEstimator(pipeline_config) built from a protobuf-text config.

Contract: `python bench.py --gpus N --steps K --warmup W` (torchrun for N>1) prints ONE JSON line on rank 0.
A step = K1 hash/bucketize -> K2 gather+pool -> FM + MLPs -> sigmoid CE -> backward -> K7 dedup + fused row update
-> dense optimizer, on one batch of the config-2 shape (26 sparse + 13 dense, V rows x 16 fp32, batch 8192 per GPU;
V = 10M, and 100M - the north-star size - when N = 8).

  value        samples/s with the batches already resident in HBM (CUDA events, max over ranks), CUDA-graph replay
  e2e          EasyRecEstimator.train(input_fn) over pinned HOST batches: a parsing thread, pinned double-buffered
               H2D (readers.DeviceFeeder), the step, and a D2H read of the loss after every step, all inside the
               timed region.  e2e.from_csv / e2e.from_parquet: the same through the CSV / Parquet readers over files
               written by workloads.write_c2_files (host parsing included)
  optimizers   the same device-resident step with lazy_adam_optimizer and adam_optimizer (tf.train.AdamOptimizer:
               dense decay sweep over the whole table) - every optimizer runs CUDA-graph captured
  lines        a second workload: C3 = DIN (batch 4096, two length-50 histories, 1M-row item table)
  roofline     the dominant own HBM-bound kernel (K7 = er_embedding_bwd, else K2 = er_embedding_fwd): algorithmic
               bytes (SURVEY.md 8d) / CUDA-event time, L2 flushed between launches, vs MEASURED_PEAKS.json hbm_gbs
  cpu_baseline the CPU oracle port of the same step on a bounded sample (rank 0, N = 1)

`--dump-outputs DIR` writes what the last timed train_step returned (loss, predictions) as DIR/<name>.npy on rank 0;
the batches and the initial weights are seeded, so the same arguments give the same inputs on every run.

`--impl reference` times the CPU oracle port (TensorFlow, hence the real reference, cannot be installed in this
image: DESIGN.md) with the host threads it runs fastest with, for exactly --steps / --warmup steps (capped at 64).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)

METRIC = 'samples_per_sec'
BATCH = 8192
N_SPARSE, N_DENSE, DIM = 26, 13, 16


def parse():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=2000)
  ap.add_argument('--warmup', type=int, default=50)
  ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
  ap.add_argument('--vocab', type=int, default=0, help='table rows; 0 = 10M, 100M at 8 GPUs')
  ap.add_argument('--batch', type=int, default=BATCH)
  ap.add_argument('--optimizer', default='adagrad_optimizer',
                  choices=['adagrad_optimizer', 'lazy_adam_optimizer', 'adam_optimizer'])
  ap.add_argument('--workload', default='deepfm_c2', choices=['deepfm_c2', 'dssm_c4', 'mmoe_c5'],
                  help='deepfm_c2 = the headline metric; dssm_c4 = BASELINE.json configs[3] (row-sharded item table)')
  ap.add_argument('--parallelism', default='', choices=['', 'dp', 'ep'],
                  help='N > 1: ep = row-sharded tables + all-to-all (EmbeddingParallelStrategy; the default), dp = replicated '
                       'tables + row all-gather')
  ap.add_argument('--uniform-ids', action='store_true')
  ap.add_argument('--no-graph', action='store_true')
  ap.add_argument('--no-cpu-baseline', action='store_true')
  ap.add_argument('--no-extras', action='store_true', help='skip the optimizer / file / C3 lines (quick runs)')
  ap.add_argument('--kernel-iters', type=int, default=30)
  ap.add_argument('--dump-outputs', default='', metavar='DIR',
                  help='after the timed steps, write what the last timed train_step returned (loss, predictions) '
                       'as DIR/<name>.npy, so that two builds can be compared output for output')
  return ap.parse_args()


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, outputs):
  """outputs: name -> tensor, array, or a list / dict of them.  Each leaf is written as DIR/<name>.npy in float32
  (float64 stays float64).  If the leaves exceed DUMP_BYTES in all, each is replaced by a fixed, seeded sample of
  its flattened elements (sorted indices), the same sample on every run."""
  import torch
  leaves = {}

  def walk(name, x):
    if isinstance(x, dict):
      for k in sorted(x):
        walk('%s_%s' % (name, k), x[k])
    elif isinstance(x, (list, tuple)):
      for i, v in enumerate(x):
        walk('%s_%d' % (name, i), v)
    elif x is not None:
      t = torch.as_tensor(x).detach()
      leaves[name] = (t.double() if t.dtype == torch.float64 else t.float()).cpu().numpy()

  for name, x in outputs.items():
    walk(name, x)
  total = sum(a.nbytes for a in leaves.values())
  os.makedirs(out_dir, exist_ok=True)
  for name, a in leaves.items():
    if total > DUMP_BYTES:
      keep = max(1, int(a.size * DUMP_BYTES // total))
      idx = np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))
      a = a.reshape(-1)[idx]
    np.save(os.path.join(out_dir, name + '.npy'), a)


def peaks():
  p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(p):
    d = json.load(open(p))
    return float(d['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)', float(d.get('bf16_tflops', 2250.0))
  return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)', 2250.0


class ClockSampler(threading.Thread):
  """nvidia-smi clocks + throttle reasons during the timed regions (B200_PROFILING.md)."""

  def __init__(self, index=0):
    super().__init__(daemon=True)
    self.index = index
    self.rows = []
    self.stop_flag = False
    self.proc = None
    self.t_mark = 0.0

  def run(self):
    q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')
    try:
      self.proc = subprocess.Popen(
          ['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q, '--format=csv,noheader,nounits',
           '-lms', '20'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      for line in self.proc.stdout:
        self.rows.append((time.time(), [x.strip() for x in line.split(',')]))
        if self.stop_flag:
          break
    except Exception:
      pass

  def mark(self):
    """start of the timed regions: samples taken before it (warm-up) only count if none falls inside"""
    self.t_mark = time.time()

  def finish(self):
    t_end = time.time() + 0.06
    while time.time() < t_end and not any(t >= self.t_mark for t, _ in self.rows):
      time.sleep(0.01)
    self.stop_flag = True
    if self.proc is not None:
      try:
        self.proc.terminate()
      except Exception:
        pass
    sm, mx, reasons = [], 0.0, set()
    names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
    inside = [r for t, r in self.rows if t >= self.t_mark]
    for r in (inside or [r for _, r in self.rows]):
      try:
        sm.append(float(r[0]))
        mx = max(mx, float(r[1]))
        for n, v in zip(names, r[2:6]):
          if v.lower().startswith('active'):
            reasons.add(n)
      except Exception:
        continue
    return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': mx or None,
            'reasons': sorted(reasons), 'samples': len(sm)}


def algorithmic_bytes(L, S, U, D, k):
  """SURVEY.md section 8d: fwd = L*(8+R) + S*R ; bwd+update = S*R + 8*L + U*(8 + k*R)."""
  R = 4 * D
  return L * (8 + R) + S * R, S * R + 8 * L + U * (8 + k * R)


# --------------------------------------------------------------------------------------
def cpu_step_oracle(state, ids, dense, labels, V, B, lr=0.01):
  """One training step of the same DeepFM on the CPU oracle (numpy + oracle/er_oracle.c)."""
  from easyrec_b200 import workloads
  from oracle import oracle as O
  rows_id, _ = O.bucketize(ids, 0, V, N_DENSE)
  rows = np.concatenate([np.repeat(np.arange(N_DENSE, dtype=np.int64), B), rows_id])
  mn = np.array(workloads.CRITEO_MIN, np.float32)
  mx = np.array(workloads.CRITEO_MAX, np.float32)
  dn = ((dense - mn) / (mx - mn)).astype(np.float32)
  w = np.concatenate([dn.T.reshape(-1), np.ones(N_SPARSE * B, np.float32)])
  F = N_SPARSE + N_DENSE
  rp = np.arange(F * B + 1, dtype=np.int32)
  deep_seg, _ = O.embedding_fwd(state['t16'], rows, rp, 0, weights=w)
  wide_seg, _ = O.embedding_fwd(state['t1'], rows, rp, 0, weights=w)
  deep = np.ascontiguousarray(deep_seg.reshape(F, B, DIM).transpose(1, 0, 2).reshape(B, F * DIM))
  wide = np.ascontiguousarray(wide_seg.reshape(F, B).T)
  logits, cache = O.deepfm_forward(wide, deep, F, DIM, state['params'])
  loss, _, g_logits = O.sigmoid_ce(logits, labels)
  g_wide, g_deep, grads = O.deepfm_backward(g_logits, wide, deep, F, DIM, state['params'], cache)
  g_deep = g_deep + np.float32(state['emb_reg']) * deep
  g_wide = g_wide + np.float32(state['emb_reg']) * wide
  gd = np.ascontiguousarray(g_deep.reshape(B, F, DIM).transpose(1, 0, 2).reshape(F * B, DIM))
  gw = np.ascontiguousarray(g_wide.T.reshape(F * B, 1))
  O.embedding_bwd(state['t16'], state['a16'], None, rows, None, gd, O.OPT_ADAGRAD, lr, weights=w)
  O.embedding_bwd(state['t1'], state['a1'], None, rows, None, gw, O.OPT_ADAGRAD, lr, weights=w)
  # dense adagrad (tf.train.AdagradOptimizer), incl. l2 on kernels
  for tag in ('dnn', 'final'):
    for L_, G_ in zip(state['params'][tag], grads[tag]):
      for k in ('W', 'b', 'gamma', 'beta'):
        g = G_[k] + (np.float32(state['l2']) * L_[k] if k == 'W' else 0)
        acc = state['acc'].setdefault((tag, id(L_), k), np.full_like(L_[k], 0.1))
        acc += g * g
        L_[k] -= (lr * g / np.sqrt(acc)).astype(np.float32)
  return loss


def make_cpu_state(V, seed=0):
  rng = np.random.default_rng(seed)
  F = N_SPARSE + N_DENSE

  def mk(i, o):
    lim = np.sqrt(6.0 / (i + o))
    return {'W': rng.uniform(-lim, lim, (i, o)).astype(np.float32), 'b': np.zeros(o, np.float32),
            'gamma': np.ones(o, np.float32), 'beta': np.zeros(o, np.float32)}

  params = {'dnn': [mk(F * DIM, 256), mk(256, 128), mk(128, 64)],
            'final': [mk(1 + DIM + 64, 256), mk(256, 128), mk(128, 64)],
            'out_W': rng.uniform(-0.3, 0.3, (64, 1)).astype(np.float32), 'out_b': np.zeros(1, np.float32)}
  n16 = V + N_DENSE
  return {'t16': (rng.standard_normal((n16, DIM), dtype=np.float32) * 0.0025),
          'a16': np.full((n16, DIM), 0.1, np.float32),
          't1': (rng.standard_normal((n16, 1), dtype=np.float32) * 0.01),
          'a1': np.full((n16, 1), 0.1, np.float32), 'params': params, 'acc': {}, 'l2': 1e-5,
          'emb_reg': 1e-5}


def cpu_threads():
  """threads for the oracle port: a quarter of the host's hardware threads, at least 8, at most 32 - where the
  small per-step matrices stop scaling (more threads only add fork/join cost); the same rule on every box"""
  n = os.cpu_count() or 1
  return int(max(1, min(32, max(8, n // 4), n)))


def run_cpu(args, steps, warmup, vocab):
  """CPU oracle port of the step; returns (samples/s, threads, seconds)."""
  from easyrec_b200 import workloads
  from oracle import oracle as O
  B = args.batch
  state = make_cpu_state(vocab)
  batches = [workloads.criteo_batch(B, 1000 + i, uniform=args.uniform_ids) for i in range(4)]
  n = cpu_threads()
  O.set_num_threads(n)
  ctx = None
  try:
    from threadpoolctl import threadpool_limits
    ctx = threadpool_limits(limits=n)
  except Exception:
    pass
  cpu_step_oracle(state, *batches[0], vocab, B)   # first touch of the tables
  for i in range(warmup):
    cpu_step_oracle(state, *batches[i % 4], vocab, B)
  t0 = time.perf_counter()
  for i in range(steps):
    cpu_step_oracle(state, *batches[i % 4], vocab, B)
  dt = time.perf_counter() - t0
  del ctx
  return B * steps / dt, n, dt


def ncu_traffic(kernel_key):
  """dram bytes per launch of a kernel from the committed ncu summary (profiles/r02_ncu_traffic.json), or None."""
  p = os.path.join(ROOT, 'profiles', 'r02_ncu_traffic.json')
  if not os.path.exists(p):
    return None, None
  d = json.load(open(p))
  v = d.get(kernel_key)
  return (float(v['dram_bytes']), 'profiles/' + v.get('source', 'r02_ncu_traffic.json')) if v else (None, None)


def main():
  args = parse()
  if os.environ.get('ER_BENCH_WATCHDOG'):   # dump every thread's Python stack if the run is still going after N seconds
    import faulthandler
    faulthandler.dump_traceback_later(int(os.environ['ER_BENCH_WATCHDOG']), exit=True)
  rank = int(os.environ.get('RANK', 0))
  world = int(os.environ.get('WORLD_SIZE', 1))
  local_rank = int(os.environ.get('LOCAL_RANK', 0))
  B = args.batch
  vocab = args.vocab or (100_000_000 if world >= 8 else 10_000_000)
  par = args.parallelism or 'ep'   # N > 1: row-sharded tables scale (constant per-rank work); dp is kept as an option
  ep = world > 1 and par == 'ep'
  opt_name = {'adagrad_optimizer': 'adagrad', 'lazy_adam_optimizer': 'lazy_adam', 'adam_optimizer': 'adam'}
  workload = 'deepfm_criteo_c2(26 sparse+13 dense, shared table V=%d x emb16 fp32, batch %d/GPU, %s ids)' % (
      vocab, B, 'uniform' if args.uniform_ids else 'zipf1.05')
  config = {'workload': workload,
            'optimizer': '%s(sparse rows fused in backward)+%s(dense)' % (opt_name[args.optimizer], opt_name[args.optimizer]),
            'built_from': 'EasyRecEstimator(protobuf-text pipeline config: workloads.c2_config_text)',
            'l2_flush': 'none in the step loop: table+optimizer state %.1f GB >> 126 MB L2, ids rotate over 16 distinct '
                        'batches; the per-kernel roofline timings flush L2 (256 MB write) before every launch'
            % ((vocab + 13) * 17 * 4 * 2 / 1e9), 'parallelism': '%s%d' % ('ep' if ep else 'dp', world)}

  if args.impl == 'reference':
    if rank != 0:
      return 0
    steps = max(1, min(args.steps, 64))
    warm = max(0, min(args.warmup, 16))
    v, threads, dt = run_cpu(args, steps, warm, min(vocab, 10_000_000))
    line = {'metric': METRIC, 'value': v, 'unit': 'samples/s', 'n_gpus': args.gpus, 'steps': steps,
            'warmup': warm, 'ms_per_step': 1000.0 * dt / steps, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'impl': 'reference', 'config': config,
            'cpu_baseline': {'value': v, 'unit': 'samples/s', 'cores': threads, 'kind': 'port',
                             'sample': '%d full steps of batch %d after %d warm-up steps (CPU oracle: C sparse path with '
                                       'OpenMP + numpy/BLAS dense, %d of %d host threads); TensorFlow is not installable '
                                       'here so the TF graph itself is not what runs'
                                       % (steps, B, warm, threads, os.cpu_count() or 1)},
            'e2e': {'value': v, 'unit': 'samples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line))
    return 0

  import torch
  import torch.distributed as dist
  from easyrec_b200 import _lib, workloads
  from easyrec_b200.estimator import EasyRecEstimator
  torch.backends.cuda.matmul.allow_tf32 = False
  torch.backends.cudnn.allow_tf32 = False
  torch.cuda.set_device(local_rank)
  dev = 'cuda:%d' % local_rank
  if world > 1:
    dist.init_process_group('nccl', device_id=torch.device(dev))
  lib = _lib.load()
  graph = not args.no_graph

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  def max_over_ranks(ms):
    if world > 1:
      tms = torch.tensor([ms], device=dev)
      dist.all_reduce(tms, op=dist.ReduceOp.MAX)
      return float(tms.item())
    return ms

  def build(optimizer, v=vocab, input_type='CSVInput'):
    text = workloads.c2_config_text(v, B, optimizer=optimizer, lr=0.01, input_type=input_type)
    return EasyRecEstimator(text, device=dev, seed=20240, use_cuda_graph=graph, world_size=world, rank=rank,
                            embedding_parallel=ep)

  if args.workload in ('dssm_c4', 'mmoe_c5'):
    return run_c4(args, rank, world, dev, ep, graph, barrier, max_over_ranks)

  n_rot = 16
  host = [workloads.criteo_batch(B, 20240 + rank * 1000 + i, uniform=args.uniform_ids) for i in range(n_rot)]
  pinned = [({'sparse_fea': torch.from_numpy(a).pin_memory(), 'dense_fea': torch.from_numpy(b).pin_memory()},
             torch.from_numpy(c).pin_memory()) for a, b, c in host]
  devb = [({k: v.to(dev) for k, v in f.items()}, l.to(dev)) for f, l in pinned]
  W = max(args.warmup, 3)

  def nxt(i, n):
    """row-sharded runs name the next batch (its id exchange runs beside the current step); None on the last step"""
    return devb[(i + 1) % n_rot][0] if (ep and i + 1 < n) else None

  def timed_resident(est, steps, warm):
    """device-resident throughput: CUDA events around `steps` train_step calls; also returns what the last of them
    returned (under CUDA-graph replay these are the graph's output buffers, rewritten by the next step)"""
    for i in range(warm):
      est.trainer.train_step(*devb[i % n_rot], next_features=nxt(i, warm))
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(steps):
      loss, probs = est.trainer.train_step(*devb[i % n_rot], next_features=nxt(i, steps))
    ev1.record()
    barrier()
    return max_over_ranks(ev0.elapsed_time(ev1)), loss, probs

  def timed_train(est, input_fn, steps, warm):
    """EasyRecEstimator.train end to end: reader thread -> pinned staging -> H2D -> step -> loss D2H, per step"""
    est.train(input_fn, steps=warm, fetch_loss_every_step=True)
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    est.train(input_fn, steps=steps, fetch_loss_every_step=True)
    ev1.record()
    barrier()
    return max_over_ranks(ev0.elapsed_time(ev1))

  # ---- headline: device-resident, then end to end through EasyRecEstimator.train ----------------------------
  sampler = ClockSampler(local_rank)   # started before the warm-up so nvidia-smi is already sampling
  if rank == 0:
    sampler.start()
  est = build(args.optimizer)
  il = est.input_layer
  for i in range(W):
    est.trainer.train_step(*devb[i % n_rot], next_features=nxt(i, W))
  barrier()
  sampler.mark()
  ms, last_loss, last_probs = timed_resident(est, args.steps, 0)
  final_loss = float(last_loss)
  if args.dump_outputs and rank == 0:
    dump_outputs(args.dump_outputs, {'loss': last_loss, 'probs': last_probs})
  value = world * B * args.steps / (ms / 1000.0)
  per_step_launches = getattr(est.trainer, 'launches_per_step', None)
  if per_step_launches is None:   # eager run: count the launches of one step
    n0 = lib.er_launch_count()
    est.trainer.train_step(*devb[0])
    per_step_launches = int(lib.er_launch_count() - n0)

  def mem_input_fn():
    def gen():
      i = 0
      while True:
        yield pinned[i % n_rot]
        i += 1
    return gen()

  e2e_ms = timed_train(est, mem_input_fn, args.steps, 3)
  clocks = sampler.finish() if rank == 0 else None
  e2e_value = world * B * args.steps / (e2e_ms / 1000.0)
  h2d = pinned[0][0]['sparse_fea'].numel() * 8 + pinned[0][0]['dense_fea'].numel() * 4 + pinned[0][1].numel() * 4
  e2e = {'value': e2e_value, 'unit': 'samples/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': 4,
         'ms_per_step': e2e_ms / args.steps,
         'through': 'EasyRecEstimator.train(input_fn) - Prefetcher thread + pinned double-buffered DeviceFeeder; the loss '
                    'of every step is read back through pinned slots one step behind the device (the last one before '
                    'train() returns)'}

  def leave():
    """multi-GPU exit: no destroy_process_group - it blocks while captured graphs still hold NCCL work"""
    if world > 1:
      barrier()
      sys.stdout.flush()
      os._exit(0)
    return 0

  il.check_exchange()   # row-sharded runs: no per-peer block of the exchange overflowed during the timed steps
  replicas_identical = None
  if world > 1:
    # every replica must hold the same dense parameters (and, under dp, the same tables) after the timed steps
    chk = [est.trainer.dense_opt.flat_p.double().sum()]
    if not ep:
      chk += [a.weight.double().sum() for a in il.arenas.values()]
    chk = torch.stack(chk)
    lo, hi = chk.clone(), chk.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    replicas_identical = bool(torch.equal(lo, hi))
  if rank != 0:
    return leave()

  extras = world == 1 and not args.no_extras
  opt_lines, lines = [], []
  roofline = None
  if extras:
    # ---- e2e from files: the CSV (native er_csv_parse) and Parquet (pyarrow) readers feed the same estimator -----
    n_file = 16
    tmp = tempfile.mkdtemp(prefix='er_bench_')
    tsv, pq_path = workloads.write_c2_files(os.path.join(tmp, 'c2'), n_file, B, seed=20240, uniform=args.uniform_ids)
    from easyrec_b200.input import readers
    file_steps = min(args.steps, 200)
    cfg = est._pipeline_config
    ms_csv = timed_train(est, lambda: readers.make_input(cfg, il, tsv), file_steps, 3)
    e2e['from_csv'] = {'value': B * file_steps / (ms_csv / 1000.0), 'unit': 'samples/s', 'steps': file_steps,
                       'file_mb': os.path.getsize(tsv) / 1e6,
                       'reader': 'CSVInput: native er_csv_parse, %d parser threads' % max(1, min(16, (os.cpu_count() or 1) // 2))}
    # (the per-kernel roofline needs this estimator's arena: measured before the other estimators are built)
    roofline = measure_roofline(args, est, devb, B, dev)
    del est
    torch.cuda.empty_cache()
    est_pq = build(args.optimizer, input_type='ParquetInput')
    for i in range(3):
      est_pq.trainer.train_step(*devb[i % n_rot])
    cfg_pq = est_pq._pipeline_config
    ms_pq = timed_train(est_pq, lambda: readers.make_input(cfg_pq, est_pq.input_layer, pq_path), file_steps, 3)
    e2e['from_parquet'] = {'value': B * file_steps / (ms_pq / 1000.0), 'unit': 'samples/s', 'steps': file_steps,
                           'file_mb': os.path.getsize(pq_path) / 1e6, 'reader': 'ParquetInput: pyarrow row groups'}
    del est_pq
    torch.cuda.empty_cache()
    # ---- the other optimizers of BASELINE.md C2, all CUDA-graph captured -----------------------------------------
    o_steps, o_warm = min(args.steps, 200), min(W, 10)
    for o in ('adagrad_optimizer', 'lazy_adam_optimizer', 'adam_optimizer'):
      if o == args.optimizer:
        opt_lines.append({'optimizer': o, 'value': value, 'ms_per_step': ms / args.steps, 'cuda_graph': graph,
                          'gpu_launches_per_step': int(per_step_launches)})
        continue
      e = build(o)
      m, _, _ = timed_resident(e, o_steps, o_warm + 3)
      row = {'optimizer': o, 'value': B * o_steps / (m / 1000.0), 'ms_per_step': m / o_steps,
             'cuda_graph': graph and e.trainer._graph is not None,
             'gpu_launches_per_step': int(getattr(e.trainer, 'launches_per_step', 0) or 0)}
      if o == 'adam_optimizer':
        row['note'] = ('tf.train.AdamOptimizer semantics: every row of the table decays each step '
                       '(er_adam_dense_sweep streams the %.1f GB of [w|m|v] rows)' % ((vocab + 13) * 17 * 12 / 1e9))
      opt_lines.append(row)
      del e
      torch.cuda.empty_cache()
    # ---- C3: DIN ----------------------------------------------------------------------------------------------
    B3, T3 = 4096, 50
    est3 = EasyRecEstimator(workloads.c3_config_text(B3, 1_000_000, T3), device=dev, seed=20240, use_cuda_graph=graph,
                            default_seq_len=T3)
    b3 = []
    for i in range(8):
      f, l = workloads.c3_batch(B3, T3, 777 + i, 1_000_000)
      b3.append(({'sparse_fea': f['sparse_fea'].to(dev), 'dense_fea': f['dense_fea'].to(dev),
                  'seq_fea': {k: (a.to(dev), b.to(dev)) for k, (a, b) in f['seq_fea'].items()}}, l.to(dev)))
    for i in range(o_warm + 3):
      est3.trainer.train_step(*b3[i % 8])
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(o_steps):
      est3.trainer.train_step(*b3[i % 8])
    ev1.record()
    torch.cuda.synchronize()
    m3 = ev0.elapsed_time(ev1)
    lines.append({'workload': 'din_c3(MultiTowerDIN, batch %d, 2 histories x %d, item table 1M x 16, attention MLP '
                              '[128,64,32,1])' % (B3, T3), 'value': B3 * o_steps / (m3 / 1000.0), 'unit': 'samples/s',
                  'ms_per_step': m3 / o_steps, 'steps': o_steps, 'cuda_graph': graph and est3.trainer._graph is not None,
                  'gpu_launches_per_step': int(getattr(est3.trainer, 'launches_per_step', 0) or 0)})
    del est3
    torch.cuda.empty_cache()
  elif world == 1:
    roofline = measure_roofline(args, est, devb, B, dev)

  # ---- CPU baseline (oracle port) on a bounded sample ---------------------------------
  cpu = None
  if world == 1 and not args.no_cpu_baseline:
    v, threads, dt = run_cpu(args, 8, 2, min(vocab, 10_000_000))
    cpu = {'value': v, 'unit': 'samples/s', 'cores': threads, 'kind': 'port',
           'sample': '8 full training steps of batch %d after 2 warm-up steps on the CPU oracle (C sparse path + numpy '
                     'dense, %d of %d host threads), %.1f s' % (B, threads, os.cpu_count() or 1, dt)}

  line = {'metric': METRIC, 'value': value, 'unit': 'samples/s', 'n_gpus': world, 'steps': args.steps,
          'warmup': W, 'ms_per_step': ms / args.steps, 'higher_is_better': True,
          'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'config': config,
          'clocks': clocks, 'e2e': e2e,
          'gpu_launches': int(per_step_launches * args.steps), 'gpu_launches_per_step': int(per_step_launches),
          'cuda_graph': graph, 'replicas_identical': replicas_identical, 'roofline': roofline, 'cpu_baseline': cpu, 'optimizers': opt_lines, 'lines': lines,
          'final_loss': final_loss}
  print(json.dumps(line))
  return leave()


def run_c4(args, rank, world, dev, ep, graph, barrier, max_over_ranks):
  """BASELINE.json configs[3]: DSSM two towers, in-batch negatives, the item table row-sharded over the ranks
  (EmbeddingParallelStrategy: ids bucketed per owner, three all-to-alls per step, owner-side fused row update)."""
  import torch
  from easyrec_b200 import _lib, workloads
  from easyrec_b200.estimator import EasyRecEstimator
  c5 = args.workload == 'mmoe_c5'
  if c5:
    # BASELINE.json configs[4]: 3-task MMoE over a DCN-style backbone, 40 id slots on one 100M x 32 table (12.5M rows per
    # rank at 8 GPUs; smaller worlds take the same rows per rank), batch 16384 per GPU
    B = args.batch if args.batch != BATCH else 16384
    item_vocab = args.vocab or 12_500_000 * world
    text = workloads.c5_config_text(B, item_vocab, embedding_parallel=ep)
    make_batch = lambda seed: workloads.c5_batch(B, seed)   # noqa: E731
    metric = 'samples/sec MMoE-3task over a DCN backbone (BASELINE.json configs[4])'
    wl = ('mmoe_c5(40 id slots on one shared table %d rows x emb32, deep MLP [256,128] + 3 Cross layers, 4 experts '
          '[128,64], 3 towers [64]; batch %d/GPU, zipf1.05 ids)' % (item_vocab, B))
  else:
    B = args.batch if args.batch != BATCH else 4096
    item_vocab = args.vocab or {1: 25_000_000, 2: 50_000_000, 4: 100_000_000}.get(world, 200_000_000)
    text = workloads.c4_config_text(B, item_vocab, embedding_parallel=ep)
    make_batch = lambda seed: workloads.c4_batch(B, seed)   # noqa: E731
    metric = 'samples/sec DSSM two-tower in-batch negatives (BASELINE.json configs[3])'
    wl = ('dssm_c4(user tower 5 ids, item tower 3 ids + price, towers [256,128,64,32], cosine, in-batch '
          'softmax; item table %d rows x emb16, batch %d/GPU, zipf1.05 ids)' % (item_vocab, B))
  est = EasyRecEstimator(text, device=dev, seed=20240, use_cuda_graph=graph, world_size=world, rank=rank,
                         embedding_parallel=ep)
  n_rot = 16
  pinned = []
  for i in range(n_rot):
    f, l = make_batch(4040 + rank * 1000 + i)
    pinned.append(({k: v.pin_memory() for k, v in f.items()}, l.pin_memory()))
  devb = [({k: v.to(dev) for k, v in f.items()}, l.to(dev)) for f, l in pinned]
  W = max(args.warmup, 3)
  steps = args.steps
  sampler = ClockSampler(int(os.environ.get('LOCAL_RANK', 0)))
  if rank == 0:
    sampler.start()
  def nxt(i, n):
    return devb[(i + 1) % n_rot][0] if (ep and i + 1 < n) else None
  for i in range(W):
    est.trainer.train_step(*devb[i % n_rot], next_features=nxt(i, W))
  barrier()
  sampler.mark()
  lib = _lib.load()
  n0 = lib.er_launch_count()
  ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  ev0.record()
  for i in range(steps):
    loss, probs = est.trainer.train_step(*devb[i % n_rot], next_features=nxt(i, steps))
  ev1.record()
  barrier()
  ms = max_over_ranks(ev0.elapsed_time(ev1))
  if args.dump_outputs and rank == 0:
    dump_outputs(args.dump_outputs, {'loss': loss, 'probs': probs})
  launches = int(lib.er_launch_count() - n0)
  if getattr(est.trainer, 'launches_per_step', None):
    launches = int(est.trainer.launches_per_step) * steps

  def input_fn():
    def gen():
      i = 0
      while True:
        yield pinned[i % n_rot]
        i += 1
    return gen()
  est.train(input_fn, steps=3, fetch_loss_every_step=True)
  barrier()
  ev0.record()
  est.train(input_fn, steps=steps, fetch_loss_every_step=True)
  ev1.record()
  barrier()
  e2e_ms = max_over_ranks(ev0.elapsed_time(ev1))
  est.input_layer.check_exchange()
  clocks = sampler.finish() if rank == 0 else None
  if rank == 0:
    h2d = sum(v.numel() * v.element_size() for v in pinned[0][0].values()) + pinned[0][1].numel() * 4
    print(json.dumps({
        'metric': metric,
        'value': world * B * steps / (ms / 1000.0), 'unit': 'samples/s', 'n_gpus': world, 'steps': steps, 'warmup': W,
        'ms_per_step': ms / steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic',
        'config': {'workload': wl,
                   'built_from': 'EasyRecEstimator(protobuf-text pipeline config: workloads.%s_config_text)' % ('c5' if c5 else 'c4'),
                   'parallelism': '%s%d' % ('ep' if ep else 'dp', world),
                   'l2_flush': 'none: tables >> L2 and ids rotate over 16 distinct batches'},
        'clocks': clocks,
        'e2e': {'value': world * B * steps / (e2e_ms / 1000.0), 'unit': 'samples/s', 'h2d_bytes_per_step': h2d,
                'd2h_bytes_per_step': 4, 'ms_per_step': e2e_ms / steps,
                'through': 'EasyRecEstimator.train(input_fn), the loss of every step read back (pinned slots, one step behind)'},
        'gpu_launches': launches, 'gpu_launches_per_step': launches // steps, 'cuda_graph': bool(graph),
        'roofline': None, 'cpu_baseline': None, 'final_loss': float(loss)}))
  if world > 1:
    barrier()
    sys.stdout.flush()
    os._exit(0)
  return 0


def measure_roofline(args, est, devb, B, dev):
  """per-kernel roofline of the estimator's own kernels: CUDA events on the launching stream, L2 flushed"""
  import torch
  from easyrec_b200 import _lib, kernels as K
  peak, peak_src, bf16_peak = peaks()
  il = est.input_layer
  call = il.calls[DIM]
  arena = il.arenas[DIM]
  kind = arena.opt_kind
  k_rw = {_lib.OPT_SGD: 2, _lib.OPT_ADAGRAD: 4}.get(kind, 6)
  F = N_SPARSE + N_DENSE
  L = S = F * B
  flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
  gout = torch.randn(B, call.out_strides[0], device=dev) * 1e-3
  outs = call.alloc_outputs()
  rows_list, w_list, uniq = [], [], []
  for i in range(4):
    feats, _ = devb[i]
    dn = il.normalize_dense(feats['dense_fea'])
    cids, w = il._gather_inputs(DIM, feats['sparse_fea'], dn)
    rows = K.bucketize(cids, call.slots_dev, call.n_slots, call.n_seg)
    rows_list.append(rows.clone())
    w_list.append(w.clone())
    uniq.append(int(torch.unique(rows).numel()))
  opt = K.make_opt(kind, 0.01)
  st = torch.cuda.current_stream()

  def time_kernel(fn, iters, pre=None):
    tot = 0.0
    for it in range(iters):
      if pre:
        pre(it)
      flush.fill_(float(it))  # evict L2 between timed launches
      e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      e0.record(st)
      fn(it)
      e1.record(st)
      e1.synchronize()
      tot += e0.elapsed_time(e1)
    return tot / iters

  def run_fwd(it):
    K.embedding_fwd(arena.weight, DIM, rows_list[it % 4], call.slots_dev, call.n_slots, call.n_seg, outs,
                    weights=w_list[it % 4])

  def run_bwd(it):
    K.embedding_bwd(arena.weight, arena.state0, arena.state1, DIM, rows_list[it % 4], call.slots_dev, call.n_slots,
                    call.n_seg, [gout], opt, call.ws, weights=w_list[it % 4])

  def run_place(it):
    K.embedding_bwd_presort(rows_list[it % 4], arena.n_rows, DIM, call.ws, call.slots_dev, call.n_slots)

  def run_after_place(it):
    K.embedding_bwd(arena.weight, arena.state0, arena.state1, DIM, rows_list[it % 4], call.slots_dev, call.n_slots,
                    call.n_seg, [gout], opt, call.ws, weights=w_list[it % 4], sorted_from=(call.ws, DIM))

  for it in range(3):
    run_fwd(it)
    run_bwd(it)
  torch.cuda.synchronize()
  fwd_ms = time_kernel(run_fwd, args.kernel_iters)
  bwd_ms = time_kernel(run_bwd, args.kernel_iters)
  place_ms = time_kernel(run_place, args.kernel_iters)
  upd_ms = time_kernel(run_after_place, args.kernel_iters, pre=run_place)
  U = float(np.mean(uniq))
  fwd_bytes, bwd_bytes = algorithmic_bytes(L, S, U, DIM, k_rw)
  fwd_bytes += 4 * L  # per-lookup weights (13 raw slots carry values)
  bwd_bytes += 4 * L
  # dense-tower GEMM on the tensor cores: the largest layer of the step (forward 624 -> 256), timed alone
  gx_ = torch.randn(B, F * DIM, device=dev)
  gw_ = torch.randn(F * DIM, 256, device=dev) * 0.05
  gout_ = torch.empty(B, 256, device=dev)
  for it in range(3):
    K.gemm(gx_, gw_, out=gout_)
  gemm_ms = time_kernel(lambda it: K.gemm(gx_, gw_, out=gout_), args.kernel_iters)
  gemm_flop = 2.0 * B * F * DIM * 256
  k_gemm = {'kernel': 'er_gemm (gemm_tf32x3_kernel, [8192 x 624] x [624 x 256])', 'bound': 'tensor',
            'achieved': gemm_flop / (gemm_ms * 1e-3) / 1e12, 'peak': bf16_peak, 'unit': 'TFLOP/s', 'ms': gemm_ms,
            'algorithmic_flop': gemm_flop,
            'note': 'fp32-accurate product = 3 TF32 MMAs per k-step at half the bf16 rate: tensor-pipe '
                    'work is 6x the algorithmic flop count against this bf16 peak'}
  k_gemm['frac'] = k_gemm['achieved'] / bf16_peak
  k_gemm['tensor_pipe_frac'] = 6.0 * k_gemm['frac']
  if os.environ.get('ER_K7') == 'radix':
    bwd_name = 'er_embedding_bwd (init_hist + 3 x scatter radix sort + bwd_scan_vec_kernel<4> + bwd_long_vec_kernel<4,1>)'
  else:
    bwd_name = ('er_embedding_bwd (memset + bk_count_kernel + bk_place_kernel + bk_fused_kernel<4> [warp-per-bucket sort, '
                'staged sums, fused row update, one-row column sums] + bk_reduce_big_kernel<4> + bwd_long_vec_kernel<4,1>)')
  k_fwd = {'kernel': 'er_embedding_fwd (fwd_single_kernel<4,4>)', 'bound': 'hbm',
           'achieved': fwd_bytes / (fwd_ms * 1e-3) / 1e9, 'peak': peak, 'unit': 'GB/s',
           'ms': fwd_ms, 'algorithmic_bytes': fwd_bytes}
  k_bwd = {'kernel': bwd_name, 'bound': 'hbm', 'achieved': bwd_bytes / (bwd_ms * 1e-3) / 1e9, 'peak': peak, 'unit': 'GB/s',
           'ms': bwd_ms, 'algorithmic_bytes': bwd_bytes, 'unique_rows': U}
  k_upd = {'kernel': 'er_embedding_bwd after the row-only placement (the part that needs the gradient: per-bucket sort, '
                     'segment sums, fused row update)', 'bound': 'hbm',
           'achieved': (bwd_bytes - 8 * L) / (upd_ms * 1e-3) / 1e9, 'peak': peak, 'unit': 'GB/s', 'ms': upd_ms,
           'algorithmic_bytes': bwd_bytes - 8 * L, 'placement_ms': place_ms,
           'note': 'the placement (placement_ms) depends only on the rows and runs on a side stream under the dense '
                   'forward/backward inside the step'}
  for k in (k_fwd, k_bwd, k_upd):
    k['frac'] = k['achieved'] / peak
  dom = k_bwd if bwd_ms >= fwd_ms else k_fwd
  traffic, traffic_src = ncu_traffic('er_embedding_bwd' if dom is k_bwd else 'er_embedding_fwd')
  return {'bound': 'hbm', 'achieved': dom['achieved'], 'peak': peak, 'unit': 'GB/s', 'frac': dom['frac'],
          'traffic': traffic, 'traffic_source': traffic_src,
          'kernel': dom['kernel'], 'peak_source': peak_src,
          'kernels': [k_fwd, k_bwd, k_upd, k_gemm],
          'random_64B_row_ceiling_gbs': 1000.0,
          'ceiling_note': 'tools/microbench_gather.cu: independent random 64 B row reads reach 15.6 Grows/s '
                          '(1.0 TB/s of rows) at 320K lookups on this B200, not the 6.57 TB/s copy peak'}


if __name__ == '__main__':
  sys.exit(main())
