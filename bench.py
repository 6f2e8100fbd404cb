#!/usr/bin/env python
"""bench.py — lists/sec of the LTR training hot path on B200 (BASELINE.json metric).

Workloads (`--config`, BASELINE.json `configs[k - 1]`; the driver default is 2, the
configuration the metric is quoted on):
  2  ApproxNDCG + 3-layer MLP (256-128-64 relu), B=1024 N=200 D=136, fp32 (3xTF32)
  3  LambdaLoss (pairwise logistic + NDCGLambdaWeight), bf16 scorer, N=512 D=256,
     512 lists per GPU (B=4096 over 8 GPUs)
  4  groupwise scoring group_size=2 + softmax loss, B=2048 N=128 D=512, tensor-core path
  5  list-size sweep N in {32..1024} of the fused pairwise-logistic kernel (loss only)
All are weak scaling: every rank steps its own batch; the flat scorer gradient is summed
once per step by the fused all-reduce + optimizer kernel over NVLink (`--collective nccl`
selects one ncclAllReduce + optimizer kernel instead).

One "step" = scorer fwd -> loss fwd+bwd -> scorer bwd -> gradient sum -> Adagrad, on
synthetic data.  Prints ONE JSON line:
  value        whole-job lists/s with inputs resident in HBM (CUDA events, max over ranks,
               barrier + synchronize on both sides)
  e2e          same metric through the public API from pinned HOST batches (H2D of every
               batch + D2H of every loss inside the timed region)
  roofline     the dominant kernel group: algorithmic FLOPs or bytes / its measured time
  cpu_baseline the reference algorithm's CPU step (oracle port) on the host cores
`--impl reference` times the reference algorithm's CPU path on all host cores (oracle
port: the reference needs TensorFlow, which cannot be installed here).

`--dump-outputs DIR` writes what the last timed step computed to DIR/<name>.npy (float32,
or float64 for float64 arrays): for configs 2-4 the loss, per-list losses, scores, d loss /
d scores, the flat scorer gradient and the updated parameters; for config 5 the loss,
per-list losses and d loss / d scores of every sweep row.  Inputs and initial parameters
are seeded, so two builds run with the same arguments can be compared file by file.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True   # the benchmark leaves the tree it runs from unchanged

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)

import torch  # noqa: E402

HIDDEN = [256, 128, 64]          # examples/tf_ranking_libsvm.py:87-88
LEARNING_RATE = 0.05
N_RESIDENT = 4                   # distinct resident batches cycled so X never sits in L2

WORKLOADS = {
    2: dict(name='BASELINE.json configs[1]: approx_ndcg_loss + 3-layer MLP scorer '
                 '(256-128-64 relu), fp32',
            B=1024, N=200, D=136, loss='approx_ndcg_loss', lam=None, precision='tf32x3',
            group_size=1, cpu_sample=1024),
    3: dict(name='BASELINE.json configs[2]: LambdaLoss (pairwise_logistic_loss + '
                 'NDCGLambdaWeight) + 3-layer MLP scorer (256-128-64 relu), bf16; '
                 'B=4096 over 8 GPUs = 512 lists per GPU',
            B=512, N=512, D=256, loss='pairwise_logistic_loss', lam='ndcg', precision='bf16',
            group_size=1, cpu_sample=128),
    4: dict(name='BASELINE.json configs[3]: groupwise scoring group_size=2 + softmax_loss, '
                 '3-layer MLP group score function (256-128-64 relu), tensor-core path',
            B=2048, N=128, D=512, loss='softmax_loss', lam=None, precision='tf32x3',
            group_size=2, cpu_sample=256),
}
SWEEP_NS = (32, 64, 128, 256, 512, 1024)
DTYPE_NAME = {'fp32': 'fp32', 'tf32x3': 'fp32 (3xTF32 on tcgen05)', 'tf32': 'tf32',
              'bf16': 'bf16 (fp32 accumulate, fp32 master weights)'}


def make_batch(seed, b, n, d, x_dtype=torch.float32):
  """Synthetic ELWC-shaped batch (SURVEY.md §8d): X ~ N(0,1); graded labels 0-4
  with MSLR-like frequencies; list lengths U[ceil(N/2), N], tail padded with -1."""
  g = torch.Generator().manual_seed(seed)
  x = torch.randn(b, n, d, generator=g).to(x_dtype)
  probs = torch.tensor([.55, .25, .12, .06, .02])
  y = torch.multinomial(probs, b * n, replacement=True, generator=g).reshape(
      b, n).float()
  lens = torch.randint((n + 1) // 2, n + 1, (b,), generator=g)
  y = torch.where(torch.arange(n).unsqueeze(0) < lens.unsqueeze(1), y,
                  torch.full_like(y, -1.))
  return x, y


def mlp_flops_per_list(n, d, hidden, group_size=1):
  """Algorithmic FLOPs of one training step of the scorer per list (DESIGN.md):
  forward 2 * rows * sum(in * out); backward dW for every layer + dH for all but the
  first layer.  Groupwise: N groups per list, tower over group_size * D inputs."""
  dims = [d * group_size] + list(hidden) + [group_size]
  fwd = sum(2 * n * dims[i] * dims[i + 1] for i in range(len(dims) - 1))
  dw = fwd
  dh = sum(2 * n * dims[i] * dims[i + 1] for i in range(1, len(dims) - 1))
  return fwd, fwd + dw + dh


def load_peaks():
  path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(path):
    p = json.load(open(path))
    return {'hbm_gbs': p['hbm_gbs'], 'bf16_tflops': p['bf16_tflops'],
            'bf16_tflops_sustained': p.get('bf16_tflops_sustained',
                                           p['bf16_tflops']),
            'source': 'measured'}
  return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0,
          'bf16_tflops_sustained': 1400.0, 'source': 'fallback'}


DUMP_MAX_ELEMS = 1 << 18   # keeps a config-5 dump (12 sweep rows) near 15 MB


def dump_outputs(out_dir, arrays):
  """Writes every tensor of `arrays` (name -> tensor) to out_dir/<name>.npy, float64 tensors
  as float64 and all others as float32.  A tensor of more than DUMP_MAX_ELEMS elements is
  written as its flattened elements at DUMP_MAX_ELEMS sorted indices drawn with a fixed
  seed, the same indices for every run of the same shape."""
  import numpy as np
  os.makedirs(out_dir, exist_ok=True)
  for name, t in arrays.items():
    t = t.detach()
    t = t.double() if t.dtype == torch.float64 else t.float()
    if t.numel() > DUMP_MAX_ELEMS:
      idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))
      t = t.reshape(-1)[idx[:DUMP_MAX_ELEMS].sort().values.to(t.device)]
    np.save(os.path.join(out_dir, name + '.npy'), t.cpu().numpy())


class ClockSampler(threading.Thread):
  """Streams `nvidia-smi -lms` clocks / throttle reasons for the whole run and
  keeps the samples that fall inside marked (timed) windows."""

  Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,'
       'clocks_event_reasons.hw_thermal_slowdown,'
       'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
  NAMES = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']

  def __init__(self, index):
    super().__init__(daemon=True)
    self.index = index
    self.samples = []     # (t, sm_mhz, reasons)
    self.max_mhz = None
    self.windows = []
    self.proc = None

  def run(self):
    try:
      self.proc = subprocess.Popen(
          ['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
           '--format=csv,noheader,nounits', '-lms', '20'], stdout=subprocess.PIPE,
          stderr=subprocess.DEVNULL, text=True)
      for line in self.proc.stdout:
        out = line.strip().split(',')
        try:
          mhz = float(out[0])
          self.max_mhz = float(out[1])
        except (ValueError, IndexError):
          continue
        reasons = {nm for nm, v in zip(self.NAMES, out[2:])
                   if v.strip().lower().startswith('active')}
        self.samples.append((time.perf_counter(), mhz, reasons))
    except Exception:   # nvidia-smi missing: report nothing
      pass

  def stop(self):
    if self.proc is not None:
      self.proc.terminate()

  def mark(self, t0, t1):
    self.windows.append((t0, t1))

  def summary(self):
    inside = [s for s in self.samples
              if any(t0 - 0.02 <= s[0] <= t1 + 0.02 for t0, t1 in self.windows)]
    use = inside if inside else self.samples
    mhz = sorted(s[1] for s in use)
    reasons = set()
    for s in use:
      reasons |= s[2]
    return {'sm_mhz': mhz[len(mhz) // 2] if mhz else None, 'sm_max_mhz': self.max_mhz,
            'reasons': sorted(reasons), 'samples_in_timed_regions': len(inside),
            'samples_total': len(self.samples)}


# ------------------------------------------------------------------------------
# CPU arm: the reference algorithm (oracle port) on ALL host cores
# ------------------------------------------------------------------------------
def _cpu_worker(cfg_id, lists, threads, steps, warmup, seed, barrier, out_q):
  """One worker process: its share of the batch, `threads` intra-op threads."""
  import torch as _t
  _t.set_num_threads(threads)
  from oracle.train_step import OracleTrainer
  from oracle import keras_losses as KO
  w = WORKLOADS[cfg_id]
  kw = {}
  if w['lam'] == 'ndcg':
    kw['lambda_weight'] = KO.NDCGLambdaWeight()
  tr = OracleTrainer(w['D'], HIDDEN, w['loss'], activation='relu',
                     learning_rate=LEARNING_RATE, loss_kwargs=kw,
                     group_size=w['group_size'])
  batches = [make_batch(seed + i, lists, w['N'], w['D']) for i in range(2)]
  for i in range(warmup):
    tr.train_step(*batches[i % 2])
  barrier.wait()
  t0 = time.perf_counter()
  for i in range(steps):
    tr.train_step(*batches[i % 2])
  out_q.put(time.perf_counter() - t0)


def cpu_reference_run(cfg_id, total_lists, procs, threads, steps, warmup):
  """`procs` worker processes x `threads` threads step `total_lists` lists per step
  between them (lists are independent: the per-shard gradients of the shared scorer would
  be summed once per step, 76 K floats, which is not timed).  Returns seconds per step
  (slowest worker) and the lists actually stepped."""
  import multiprocessing as mp
  ctx = mp.get_context('spawn')
  per = max(1, total_lists // procs)
  barrier = ctx.Barrier(procs)
  q = ctx.Queue()
  ps = [ctx.Process(target=_cpu_worker,
                    args=(cfg_id, per, threads, steps, warmup, 1234 + 31 * r, barrier, q))
        for r in range(procs)]
  for p in ps:
    p.start()
  times = [q.get() for _ in ps]
  for p in ps:
    p.join()
  return max(times) / steps, per * procs


def pick_cpu_layout(cfg_id, sample_lists):
  """(processes, threads per process) that uses every host core the oracle can keep busy:
  one quick step per candidate, best lists/s wins."""
  ncpu = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (
      os.cpu_count() or 1)
  cands = []
  for threads in (4, 8, 16):
    procs = max(1, ncpu // threads)
    procs = min(procs, sample_lists)
    if (procs, threads) not in cands:
      cands.append((procs, threads))
  best, best_rate = cands[0], 0.0
  for procs, threads in cands:
    try:
      sec, lists = cpu_reference_run(cfg_id, sample_lists, procs, threads, 1, 1)
    except Exception:   # noqa: BLE001
      continue
    rate = lists / sec
    if rate > best_rate:
      best, best_rate = (procs, threads), rate
  return best, ncpu


def cpu_baseline_block(cfg_id, sample_lists, steps):
  (procs, threads), ncpu = pick_cpu_layout(cfg_id, sample_lists)
  sec, lists = cpu_reference_run(cfg_id, sample_lists, procs, threads, steps, 1)
  return {
      'value': lists / sec, 'unit': 'lists/s', 'cores': procs * threads,
      'kind': 'port', 'host_cores': ncpu,
      'layout': '%d processes x %d threads' % (procs, threads),
      'sample': '%d lists/step x %d steps of the same workload (oracle: torch-CPU '
                'restatement of the reference algorithm, [B,N,N] formulation; lists are '
                'independent, so worker processes step disjoint shards)' % (lists, steps)}, sec


def workload_config(cfg_id, n_gpus, precision, extra=None):
  w = WORKLOADS[cfg_id]
  xbytes = 2 if precision == 'bf16' else 4
  cfg = {
      'workload': w['name'],
      'batch_lists_per_gpu': w['B'], 'list_size': w['N'], 'feature_dim': w['D'],
      'global_batch_lists': w['B'] * n_gpus, 'hidden_layer_dims': HIDDEN,
      'loss': w['loss'], 'lambda_weight': w['lam'], 'group_size': w['group_size'],
      'scorer_precision': precision,
      'optimizer': 'adagrad', 'parallelism': 'dp%d' % n_gpus,
      'padding': 'list lengths U[N/2, N], label -1',
      'l2_policy': 'inputs rotate over %d resident batches (%d MB > 126 MB L2)'
                   % (N_RESIDENT, N_RESIDENT * w['B'] * w['N'] * w['D'] * xbytes // 2**20),
  }
  if extra:
    cfg.update(extra)
  return cfg


def run_reference(args):
  rank = int(os.environ.get('RANK', '0'))
  if rank != 0:
    return
  cfg_id = args.config
  if cfg_id == 5:
    return run_reference_sweep(args)
  w = WORKLOADS[cfg_id]
  sample = args.cpu_sample_lists or w['cpu_sample']
  block, sec = cpu_baseline_block(cfg_id, sample, args.steps)
  value = block['value']
  line = {
      'impl': 'reference', 'metric': 'lists_per_sec', 'value': value,
      'unit': 'lists/s', 'n_gpus': args.gpus, 'steps': args.steps,
      'warmup': args.warmup, 'ms_per_step': sec * 1e3, 'higher_is_better': True,
      'scaling': 'weak', 'vs_baseline': None, 'dtype': 'fp32',
      'data': 'synthetic',
      'config': workload_config(cfg_id, args.gpus, args.precision or w['precision']),
      'reference_arm': 'oracle port of the tensorflow_ranking CPU path (TensorFlow is not '
                       'installable offline), torch CPU fp32, [B,N,N] formulation; ~ the '
                       'TF-CPU step, not TF itself',
      'cpu_baseline': block,
      'e2e': {'value': value, 'unit': 'lists/s', 'h2d_bytes_per_step': 0,
              'd2h_bytes_per_step': 0},
      'gpu_launches': 0,
  }
  emit(line)


def run_reference_sweep(args):
  """Config 5 on the CPU: pairwise-logistic loss + gradient (oracle) per list size."""
  from oracle import keras_losses as KO
  ncpu = len(os.sched_getaffinity(0))
  torch.set_num_threads(min(ncpu, 32))
  rows = []
  for n in SWEEP_NS:
    b = max(8, (1 << 15) // n)
    _, y = make_batch(5, b, n, 1)
    s = (torch.randn(b, n, generator=torch.Generator().manual_seed(n)) * 2).requires_grad_()
    loss = KO.PairwiseLogisticLoss()
    for _ in range(2):
      loss(y, s).backward()
    t0 = time.perf_counter()
    for _ in range(args.steps):
      s.grad = None
      loss(y, s).backward()
    sec = (time.perf_counter() - t0) / args.steps
    rows.append({'N': n, 'B': b, 'ms': sec * 1e3, 'lists_per_s': b / sec,
                 'pair_evals_per_s': float(n) * n * b / sec})
  ref = [r for r in rows if r['N'] == 256][0]
  emit({'impl': 'reference', 'metric': 'lists_per_sec', 'value': ref['lists_per_s'],
        'unit': 'lists/s', 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': ref['ms'], 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'fp32', 'data': 'synthetic',
        'config': sweep_config(args.gpus), 'sweep': rows,
        'cpu_baseline': {'value': ref['lists_per_s'], 'unit': 'lists/s',
                         'cores': min(ncpu, 32), 'kind': 'port', 'host_cores': ncpu,
                         'sample': 'pairwise logistic loss + autograd on %d lists of N=256'
                                   % ref['B']},
        'e2e': {'value': ref['lists_per_s'], 'unit': 'lists/s', 'h2d_bytes_per_step': 0,
                'd2h_bytes_per_step': 0}, 'gpu_launches': 0})


def sweep_config(n_gpus):
  return {'workload': 'BASELINE.json configs[4]: list-size sweep N in %s of '
                      'pairwise_logistic_loss (fused forward + backward loss kernel, scores '
                      'resident); headline value = N=256 row' % (list(SWEEP_NS),),
          'parallelism': 'dp%d (independent shards, no collective: the loss has no '
                         'parameters)' % n_gpus,
          'l2_policy': 'inputs rotate over 8 resident batches'}


# ------------------------------------------------------------------------------
def init_dist():
  import torch.distributed as dist
  world = int(os.environ.get('WORLD_SIZE', '1'))
  rank = int(os.environ.get('RANK', '0'))
  local_rank = int(os.environ.get('LOCAL_RANK', '0'))
  torch.cuda.set_device(local_rank)
  dev = torch.device('cuda', local_rank)
  if world > 1:
    dist.init_process_group('nccl', device_id=dev)
  import __graft_entry__ as entry
  if rank == 0:
    entry.build()
  if world > 1:
    dist.barrier()
  return world, rank, local_rank, dev, dist


def run_gpu(args):
  world, rank, local_rank, dev, dist = init_dist()
  import ranking_b200 as tfr
  from ranking_b200 import _C
  from ranking_b200 import dp as tfr_dp
  cfg_id = args.config
  w = WORKLOADS[cfg_id]
  B, N, D, gs = w['B'], w['N'], w['D'], w['group_size']
  precision = args.precision or w['precision']
  full_affinity = os.sched_getaffinity(0)
  numa = tfr_dp.bind_to_gpu_numa_node(local_rank)   # before any pinned allocation

  tower = tfr.keras.layers.create_tower(HIDDEN, gs, activation='relu',
                                        use_batch_norm=False, dropout=0,
                                        input_dim=D * gs, seed=1238,
                                        precision=precision)
  if world > 1:   # identical replicas
    dist.broadcast(tower.flat.data, src=0)
  lam = tfr.keras.losses.NDCGLambdaWeight() if w['lam'] == 'ndcg' else None
  loss_obj = tfr.keras.losses.get(w['loss'], lambda_weight=lam)
  kw = dict(optimizer='adagrad', learning_rate=LEARNING_RATE, collective=args.collective)
  if gs > 1:
    trainer = tfr.train.GroupwiseRankingTrainer(tower, loss_obj, gs, **kw)
  else:
    trainer = tfr.train.RankingTrainer(tower, loss_obj, **kw)
  xdt = tower.input_dtype
  host = [make_batch(1234 + 17 * rank + i, B, N, D, xdt) for i in range(N_RESIDENT)]
  resident = [(x.to(dev), y.to(dev)) for x, y in host]
  stream = torch.cuda.current_stream()

  def sync_all():
    torch.cuda.synchronize()
    if world > 1:
      dist.barrier()
      torch.cuda.synchronize()

  # ---- value: inputs resident, device-timed ----------------------------------
  for i in range(args.warmup):
    trainer.train_step(*resident[i % N_RESIDENT])
  sampler = ClockSampler(local_rank)
  if rank == 0:
    sampler.start()
    time.sleep(0.3)      # let the sampling stream start (before the barrier!)
  sync_all()
  launches0 = _C.lib.tfr_launch_count()
  t_val0 = time.perf_counter()
  ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  ev0.record(stream)
  for i in range(args.steps):
    loss = trainer.train_step(*resident[i % N_RESIDENT])
  ev1.record(stream)
  sync_all()
  launches = _C.lib.tfr_launch_count() - launches0
  ms_total = ev0.elapsed_time(ev1)
  sampler.mark(t_val0, time.perf_counter())
  if args.dump_outputs and rank == 0:   # before the phase and e2e runs step the trainer on
    dump_outputs(args.dump_outputs, {
        'loss': loss, 'per_list_loss': trainer.per_list[0], 'scores': trainer.scores,
        'dscores': trainer.dscores, 'grads': trainer.grads, 'params': tower.flat})
  t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
  if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
  ms_step = float(t) / args.steps
  value = B * world / (ms_step * 1e-3)
  final_loss = float(loss)

  # ---- per-phase device time (same process, CUDA events on the launch stream) --
  phase = phase_times(trainer, resident, args.steps, stream)

  # ---- e2e: pinned host batches through the public API --------------------------
  pinned = [(x.pin_memory(), y.pin_memory()) for x, y in host]
  pipe = tfr.train.HostBatchPipeline(trainer, B, N, D)
  pipe.run([pinned[i % N_RESIDENT] for i in range(max(args.warmup, 3))])
  sync_all()
  t0 = time.perf_counter()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record(stream)
  losses = pipe.run([pinned[i % N_RESIDENT] for i in range(args.steps)])
  e1.record(stream)
  sync_all()
  wall = time.perf_counter() - t0
  sampler.mark(t0, time.perf_counter())
  if rank == 0:
    sampler.stop()
  e2e_ms = max(e0.elapsed_time(e1), wall * 1e3)
  t = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
  if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
  e2e_value = B * world * args.steps / (float(t) * 1e-3)

  parity = ndcg10_parity(tfr, trainer, host[0], dev) if rank == 0 else None

  if rank == 0:
    peaks = load_peaks()
    fwd_fl, step_fl = mlp_flops_per_list(N, D, HIDDEN, gs)
    gemm_ms = phase['mlp_fwd_ms'] + phase['mlp_bwd_ms']
    achieved = step_fl * B / (gemm_ms * 1e-3) / 1e12
    peak = peaks['bf16_tflops_sustained']
    # SURVEY.md §8(d): the algorithmic bytes of the scorer are X read twice (forward and
    # dW_1); activations are recomputable on chip, so what the layer-by-layer plan moves
    # beyond that is re-read traffic, reported as `traffic` / `traffic_ratio`.
    xbytes = 2 if precision == 'bf16' else 4
    alg_bytes = 2 * D * xbytes * N * B
    traffic = load_traffic(cfg_id, precision)
    loss_bytes = (12 * N + 16) * B
    pair_evals = float(N) * N * B
    tf32_peak = measure_tf32_peak(dev) if precision in ('tf32x3', 'tf32') else None
    roof_gemm = {
        'kernel': 'scorer tower GEMMs (tfr_mlp_fwd + tfr_mlp_bwd)',
        'bound': 'tensor', 'achieved': achieved, 'peak': peak,
        'unit': 'TFLOP/s', 'frac': achieved / peak,
        'peak_source': peaks['source'] + ' bf16 sustained',
        'traffic': traffic['scorer_gemm_dram_bytes_per_step'] if traffic else None,
        'traffic_source': traffic['source'] if traffic else None,
        'algorithmic_flops_per_step': step_fl * B,
        'algorithmic_bytes_per_step': alg_bytes,
        'traffic_ratio': (traffic['scorer_gemm_dram_bytes_per_step'] / alg_bytes
                          if traffic else None),
        'kernel_ms_per_step': gemm_ms,
    }
    if tf32_peak:
      roof_gemm.update({
          'note': '3xTF32 issues 3 TF32 MMAs per algorithmic product, so the ceiling of '
                  'this fraction is 1/6 of the nominal bf16 peak; the measured ceiling is '
                  'tf32_cublas_tflops / 3',
          'tf32_cublas_tflops': tf32_peak,
          'frac_of_3xtf32_ceiling': achieved / (tf32_peak / 3.0)})
    roof_hbm = {
        'kernel': 'scorer tower GEMMs (tfr_mlp_fwd + tfr_mlp_bwd)',
        'bound': 'hbm', 'achieved': alg_bytes / (gemm_ms * 1e-3) / 1e9,
        'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
        'frac': alg_bytes / (gemm_ms * 1e-3) / 1e9 / peaks['hbm_gbs'],
        'algorithmic_bytes_per_step': alg_bytes,
        'note': 'SURVEY.md §8(d) bytes: X read twice',
        'traffic': roof_gemm['traffic'], 'traffic_ratio': roof_gemm['traffic_ratio'],
    }
    roof_loss = {
        'kernel': {'approx_ndcg_loss': 'approx_loss_kernel',
                   'pairwise_logistic_loss': 'pairwise_tri_kernel',
                   'softmax_loss': 'softmax_loss_kernel'}[w['loss']],
        'bound': 'hbm', 'achieved': loss_bytes / (phase['loss_ms'] * 1e-3) / 1e9,
        'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
        'frac': loss_bytes / (phase['loss_ms'] * 1e-3) / 1e9 / peaks['hbm_gbs'],
        'algorithmic_bytes_per_step': loss_bytes,
        'pair_evals_per_s': (pair_evals / (phase['loss_ms'] * 1e-3)
                             if w['loss'] != 'softmax_loss' else None),
        'kernel_ms_per_step': phase['loss_ms'],
        'note': 'O(N^2) pair work on O(N) bytes: MUFU / issue bound, the HBM fraction is '
                'small by construction (SURVEY.md §7)',
    }
    dominant = roof_gemm if gemm_ms >= phase['loss_ms'] else roof_loss
    line = {
        'metric': 'lists_per_sec', 'value': value, 'unit': 'lists/s',
        'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None,
        'dtype': DTYPE_NAME[precision],
        'data': 'synthetic',
        'config': workload_config(cfg_id, world, precision),
        'final_loss': final_loss,
        'roofline': dominant,
        'roofline_gemm': roof_gemm,
        'roofline_hbm': roof_hbm,
        'roofline_loss': roof_loss,
        'phases_ms': phase,
        'collective': {
            'kind': args.collective if world > 1 else 'none',
            'exposed_us_per_step': (phase['opt_ms'] - phase.get('opt_local_ms', 0.0)) * 1e3
            if world > 1 else 0.0,
            'note': 'device time of the gradient-sum + optimizer phase minus the local '
                    'optimizer kernel: flag round (waits for the slowest rank) + peer reads'},
        'e2e': {'value': e2e_value, 'unit': 'lists/s',
                'h2d_bytes_per_step': pipe.h2d_bytes,
                'd2h_bytes_per_step': pipe.d2h_bytes,
                'ms_per_step': float(t) / args.steps,
                'last_loss': losses[-1], 'numa_binding': numa},
        'ndcg10_parity': parity,
        'gpu_launches': int(launches),
        'clocks': sampler.summary(),
    }
    if world == 1 and not args.no_cpu_baseline:
      sample = args.cpu_sample_lists or min(w['cpu_sample'], 256)
      os.sched_setaffinity(0, full_affinity)   # the CPU arm gets every host core again
      block, _ = cpu_baseline_block(cfg_id, sample, args.cpu_steps)
      line['cpu_baseline'] = block
    emit(line)
  if trainer.reducer is not None:
    trainer.reducer.close()
  if world > 1:
    dist.barrier()
    dist.destroy_process_group()


def load_traffic(cfg_id, precision):
  """dram__bytes_read + write of the scorer GEMM kernels per step, from the committed ncu
  capture of this round (profiles/r02_traffic.json), if one exists for this workload."""
  tpath = os.path.join(ROOT, 'profiles', 'r02_traffic.json')
  if not os.path.exists(tpath):
    return None
  t = json.load(open(tpath))
  return t.get('config%d_%s' % (cfg_id, precision))


def ndcg10_parity(tfr, trainer, host_batch, dev, lists=64):
  """NDCG@10 of the scores the GPU scorer produces, computed by the CUDA metric kernel and
  by the oracle metric on the SAME scores (first `lists` lists of a batch): per-list max
  abs difference, and equality of the integer rank arrays."""
  try:
    from oracle import metrics_impl as OM
    from oracle import losses_impl as OL
    x, y = host_batch
    x, y = x[:lists], y[:lists]
    scores = trainer.predict(x.to(dev), mask=None, y_true=y.to(dev)).clone()
    if trainer.__class__.__name__ == 'RankingTrainer':
      # the univariate scorer leaves padded slots unmasked here; metrics ignore them
      pass
    yd = y.to(dev)
    m = tfr.metrics_impl.NDCGMetric(name=None, topn=10)
    got, got_w = m.compute(yd, scores, None)
    ref, ref_w = OM.NDCGMetric(name=None, topn=10).compute(y.double(), scores.double().cpu(),
                                                          None)
    ranks = tfr.utils.sorted_ranks(scores, yd).cpu().long()
    ref_ranks = OL._compute_ranks(scores.double().cpu(), y >= 0)
    diff = float((got.double().cpu() - ref).abs().max())
    return {'lists': int(lists), 'topn': 10,
            'ndcg10_gpu_mean': float(got.mean()), 'ndcg10_oracle_mean': float(ref.mean()),
            'max_abs_diff_per_list': diff, 'fp32_ulps': diff / 1.1920929e-07,
            'rank_arrays_equal': bool(torch.equal(ranks, ref_ranks)),
            'note': 'same GPU scores fed to the CUDA metric kernel and to the oracle '
                    '(fp64) metric; ties broken by index on both sides'}
  except Exception as e:   # noqa: BLE001  (a diagnostic block must not kill the bench line)
    return {'error': repr(e)[:300]}


def measure_tf32_peak(dev, n=8192, reps=5):
  """Dense TF32 throughput of this GPU as cuBLAS reaches it (torch.matmul, 8192^3, best
  of `reps`): the measured roof of `kind::tf32` MMAs — MEASURED_PEAKS.json only carries
  the bf16 number.  Measurement aid outside every timed region; never on the product path."""
  try:
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    a = torch.randn(n, n, device=dev)
    b = torch.randn(n, n, device=dev)
    for _ in range(2):
      a @ b
    torch.cuda.synchronize(dev)
    best = float('inf')
    for _ in range(reps):
      e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      e0.record()
      a @ b
      e1.record()
      torch.cuda.synchronize(dev)
      best = min(best, e0.elapsed_time(e1))
    torch.backends.cuda.matmul.allow_tf32 = prev
    del a, b
    return 2.0 * n ** 3 / (best * 1e-3) / 1e12
  except Exception:   # noqa: BLE001  (reference number only)
    return None


def phase_times(trainer, resident, steps, stream):
  """Average device time of each phase of the step, by CUDA events recorded on the
  launching stream around every phase (same process as the timed run; all ranks run it,
  so the collective phase sees its peers)."""
  import ctypes
  names = ['mlp_fwd_ms', 'loss_ms', 'mlp_bwd_ms', 'opt_ms']
  acc = dict.fromkeys(names, 0.0)
  steps = max(3, min(steps, 20))
  t = trainer.tower
  for i in range(steps):
    x, y = resident[i % len(resident)]
    b, n, d = x.shape
    trainer._ensure(b, n)
    x = trainer._prep_x(x)
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    run_cfg = t._run_cfg(training=True)
    cfg = ctypes.byref(run_cfg)
    grads = trainer.reducer.grads() if trainer.reducer is not None else trainer.grads
    evs[0].record(stream)
    trainer._forward(x, y, None, cfg, True)
    evs[1].record(stream)
    trainer.loss.fused_fwd_bwd(y, trainer.scores, None, trainer.dscores,
                               trainer.per_list, trainer.total2)
    evs[2].record(stream)
    trainer._backward(x, None, cfg, grads)
    evs[3].record(stream)
    trainer._apply(grads)
    evs[4].record(stream)
    torch.cuda.synchronize()
    for k, nm in enumerate(names):
      acc[nm] += evs[k].elapsed_time(evs[k + 1])
  out = {k: v / steps for k, v in acc.items()}
  # the local optimizer kernel alone (what the last phase costs without a collective)
  from ranking_b200 import _C
  scratch_p = t.flat.data.clone()
  scratch_a = trainer.accum.clone()
  g = torch.zeros_like(scratch_p)
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record(stream)
  for _ in range(10):
    _C.check(_C.lib.tfr_optimizer_step(_C.ptr(scratch_p), _C.ptr(g), _C.ptr(scratch_a),
                                       g.numel(), trainer.opt_kind, trainer.lr, trainer.eps,
                                       1.0, _C.stream()))
  e1.record(stream)
  torch.cuda.synchronize()
  out['opt_local_ms'] = e0.elapsed_time(e1) / 10
  return out


# ------------------------------------------------------------------------------
# config 5: list-size sweep of the pairwise-logistic kernel
# ------------------------------------------------------------------------------
def run_sweep(args):
  world, rank, local_rank, dev, dist = init_dist()
  import ranking_b200 as tfr
  from ranking_b200 import _C
  peaks = load_peaks()
  stream = torch.cuda.current_stream()
  sampler = ClockSampler(local_rank)
  if rank == 0:
    sampler.start()
    time.sleep(0.3)
  rows = []
  launches = 0
  for lam_name in ('none', 'ndcg'):
    lam = tfr.keras.losses.NDCGLambdaWeight() if lam_name == 'ndcg' else None
    loss = tfr.keras.losses.PairwiseLogisticLoss(lambda_weight=lam)
    for n in SWEEP_NS:
      b = max(64, (1 << 21) // n)
      nbuf = 8
      bufs = []
      for i in range(nbuf):
        _, y = make_batch(100 + 13 * rank + i, b, n, 1)
        s = torch.randn(b, n, generator=torch.Generator().manual_seed(7 * rank + i)).mul(2)
        bufs.append((s.to(dev), y.to(dev)))
      grad = torch.empty(b, n, device=dev)
      per_list = torch.empty(2, b, device=dev)
      total2 = torch.zeros(2, device=dev)
      for i in range(max(args.warmup, 3)):
        loss.fused_fwd_bwd(bufs[i % nbuf][1], bufs[i % nbuf][0], None, grad, per_list, total2)
      torch.cuda.synchronize()
      if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
      l0 = _C.lib.tfr_launch_count()
      t0 = time.perf_counter()
      e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      e0.record(stream)
      for i in range(args.steps):
        loss.fused_fwd_bwd(bufs[i % nbuf][1], bufs[i % nbuf][0], None, grad, per_list, total2)
      e1.record(stream)
      torch.cuda.synchronize()
      if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
      sampler.mark(t0, time.perf_counter())
      launches += _C.lib.tfr_launch_count() - l0
      if args.dump_outputs and rank == 0:
        tag = '%s_N%d_' % (lam_name, n)
        dump_outputs(args.dump_outputs, {tag + 'loss': total2[0],
                                         tag + 'per_list_loss': per_list[0],
                                         tag + 'dscores': grad})
      t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
      if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
      ms = float(t) / args.steps
      bytes_ = (12 * n + 16) * b * world
      rows.append({'lambda_weight': lam_name, 'N': n, 'lists_per_step': b * world, 'ms': ms,
                   'lists_per_s': b * world / (ms * 1e-3),
                   'hbm_gbs_algorithmic': bytes_ / (ms * 1e-3) / 1e9,
                   'hbm_frac_per_gpu': bytes_ / world / (ms * 1e-3) / 1e9 / peaks['hbm_gbs'],
                   'pair_evals_per_s': float(n) * n * b * world / (ms * 1e-3)})
      del bufs
  if rank == 0:
    sampler.stop()
    head = [r for r in rows if r['N'] == 256 and r['lambda_weight'] == 'none'][0]
    emit({'metric': 'lists_per_sec', 'value': head['lists_per_s'], 'unit': 'lists/s',
          'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
          'ms_per_step': head['ms'], 'higher_is_better': True, 'scaling': 'weak',
          'vs_baseline': None, 'dtype': 'fp32', 'data': 'synthetic',
          'config': sweep_config(world), 'sweep': rows,
          'roofline': {'kernel': 'pairwise_tri_kernel (N=256 row)', 'bound': 'hbm',
                       'achieved': head['hbm_gbs_algorithmic'] / world,
                       'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
                       'frac': head['hbm_frac_per_gpu'], 'traffic': None,
                       'peak_source': peaks['source'],
                       'note': '(12 N + 16) algorithmic bytes per list; the kernel does N^2 '
                               'pair evaluations per list on them: MUFU / issue bound, see '
                               'sweep[].pair_evals_per_s'},
          'e2e': None, 'gpu_launches': int(launches), 'clocks': sampler.summary()})
  if world > 1:
    dist.barrier()
    dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line):
  """Writes the JSON line to the process's real stdout (see main)."""
  data = (json.dumps(line) + '\n').encode()
  if _REAL_STDOUT is None:
    sys.stdout.write(data.decode())
    sys.stdout.flush()
  else:
    os.write(_REAL_STDOUT, data)


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=20)
  ap.add_argument('--warmup', type=int, default=5)
  ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
  ap.add_argument('--config', type=int, default=2, choices=[2, 3, 4, 5],
                  help='BASELINE.json workload (configs[k - 1]); default 2 = the '
                       'configuration the metric is quoted on')
  ap.add_argument('--precision', default=None,
                  choices=['fp32', 'tf32x3', 'tf32', 'bf16'],
                  help='scorer GEMM arithmetic (default: the workload\'s: tf32x3 = '
                       'fp32-faithful 3xTF32 on tcgen05 for configs 2 / 4, bf16 for 3)')
  ap.add_argument('--collective', default='fused', choices=['fused', 'nccl'])
  ap.add_argument('--cpu-sample-lists', type=int, default=0)
  ap.add_argument('--cpu-steps', type=int, default=3)
  ap.add_argument('--no-cpu-baseline', action='store_true')
  ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                  help='write the outputs of the last timed step to DIR/<name>.npy')
  args = ap.parse_args()
  if args.steps < 1:
    ap.error('--steps must be at least 1')
  if args.dump_outputs and args.impl == 'reference':
    ap.error('--dump-outputs dumps the CUDA path: use it with --impl b200')
  args.warmup = max(args.warmup, 3)
  # The contract is ONE JSON line on stdout.  Libraries print banners there (e.g.
  # "NCCL version ..." at communicator creation), so everything but the final line is
  # routed to stderr: fd 1 is parked and only `emit` writes to it.
  global _REAL_STDOUT
  sys.stdout.flush()
  _REAL_STDOUT = os.dup(1)
  os.dup2(2, 1)
  if args.impl == 'reference':
    run_reference(args)
  elif args.config == 5:
    run_sweep(args)
  else:
    run_gpu(args)


if __name__ == '__main__':
  main()
