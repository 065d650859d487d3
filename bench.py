#!/usr/bin/env python
"""bench.py -- learner env-frames/sec of the V-trace hot path on B200.

  python bench.py --gpus N --steps K --warmup W            (this framework, CUDA)
  python bench.py --impl reference --gpus N --steps K ...  (the reference's algorithm on
                                                            the host CPU cores: oracle port)
  python bench.py ... --dump-outputs DIR                    (also write the last timed step's outputs
                                                            as DIR/<name>.npy)
Under torchrun (N > 1) every rank runs one learner replica on its own GPU (batch-axis
sharding, B=64 unrolls per GPU) with ONE NCCL all-reduce(SUM) of the flat gradient arena
per step; the timed region is bracketed by barrier + synchronize, timed with CUDA events,
MAX over ranks; rank 0 prints one JSON line.

A "step" = one `minimize` (reference agents/vtrace/learner.py:255-280) on one synthetic
unroll batch already resident in HBM: ImpalaDeep unroll forward -> fused V-trace loss ->
backward -> [all-reduce] -> Adam.  metric = B_global * T * num_action_repeats / step_time
(== the reference's speed/steps_per_sec, common/utils.py:659-661).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'env-frames/sec (learner, device-timed) on synthetic 84x84x4 T=20 unrolls @1/2/4/8 B200'
UNIT = 'env-frames/s'
A = 18
OBS = (84, 84, 4)


def parse_args():
  p = argparse.ArgumentParser()
  p.add_argument('--gpus', type=int, default=1)
  p.add_argument('--steps', type=int, default=50)
  p.add_argument('--warmup', type=int, default=10)
  p.add_argument('--impl', default='b200', choices=['b200', 'reference'])
  p.add_argument('--net', default='deep', choices=['deep', 'shallow'])
  p.add_argument('--agent', default='vtrace', choices=['vtrace', 'r2d2'],
                 help='vtrace = the headline IMPALA learner (BASELINE configs[1..3]); r2d2 = configs[4]: '
                      'DuelingLSTMDQNNet learner step on synthetic prioritized replay')
  p.add_argument('--batch', type=int, default=64, help='unrolls per GPU')
  p.add_argument('--unroll', type=int, default=20)
  p.add_argument('--cpu-batch', type=int, default=0,
                 help='unrolls per CPU-baseline step (0 = the same batch as the GPU arm)')
  p.add_argument('--conv', default='tc3p', choices=['simt', 'tc', 'tc3', 'tc3p'],
                 help="contraction path of the convs and dense layers: fp32 SIMT, tcgen05 bf16, "
                      "tcgen05 bf16x3 (fp32-faithful split operands), or tc3p = bf16x3 on HBM-resident "
                      "operand planes with TMA-fed warp-specialised kernels (deep net; the default)")
  p.add_argument('--no-extras', action='store_true',
                 help='skip the profiling pass, the loss-kernel sweep and the CPU baseline')
  p.add_argument('--dump-outputs', metavar='DIR',
                 help='after the timed steps, write what the last timed step computed (loss terms, updated '
                      'parameters, gradients; R2D2 also priorities and sampled indices) as DIR/<name>.npy')
  a = p.parse_args()
  if a.steps < 1:
    p.error('--steps must be at least 1')
  if a.dump_outputs and a.impl == 'reference':
    p.error('--dump-outputs writes the outputs of the CUDA path (--impl b200)')
  if a.net == 'shallow' and a.conv == 'tc3p':
    a.conv = 'tc3'
  if a.cpu_batch <= 0:
    a.cpu_batch = a.batch
  return a


# ----------------------------------------------------------------------------------------
def cpu_learner_throughput(net, T, B, steps, warmup, threads=None):
  """The reference's algorithm (oracle port, torch-CPU fp32) on the host cores."""
  import torch
  from oracle import learner_oracle, loss_oracle
  cfg = loss_oracle.default_config()
  lr = learner_oracle.CpuLearner(net, A, OBS, cfg, lr=4.8e-4, beta1=0.0, eps=3.125e-7,
                                 decay_steps=10**6)
  batch = learner_oracle.synthetic_batch(T, B, A, OBS, seed=1234)
  if threads:
    torch.set_num_threads(threads)
  else:
    # give the CPU arm its best thread count: small convolutions over-subscribe badly on
    # many-core hosts, so try a few pool sizes (1 step each) and keep the fastest.
    ncpu = os.cpu_count() or 1
    best = None
    for n in sorted({min(ncpu, c) for c in (8, 16, 32, ncpu)}):
      torch.set_num_threads(n)
      lr.step(batch)
      t0 = time.perf_counter(); lr.step(batch); dt = time.perf_counter() - t0
      if best is None or dt < best[0]:
        best = (dt, n)
    torch.set_num_threads(best[1])
  cores = torch.get_num_threads()
  for _ in range(warmup):
    lr.step(batch)
  t0 = time.perf_counter()
  for _ in range(steps):
    lr.step(batch)
  dt = (time.perf_counter() - t0) / max(steps, 1)
  return dict(value=B * T / dt, ms_per_step=dt * 1e3, cores=cores,
              sample='%d steps of B=%d unrolls x T=%d (%s net) after %d warm-up; torch-CPU fp32 '
                     'oracle port, %d threads' % (steps, B, T, net, warmup, cores))


def run_reference(args):
  rank = int(os.environ.get('RANK', '0'))
  if rank != 0:
    return
  r = cpu_learner_throughput(args.net, args.unroll, args.cpu_batch, args.steps, args.warmup)
  line = {
      'impl': 'reference', 'metric': METRIC, 'value': r['value'], 'unit': UNIT,
      'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
      'ms_per_step': r['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak',
      'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
      'config': workload_config(args, max(args.gpus, 1)),
      'cpu_baseline': {'value': r['value'], 'unit': UNIT, 'cores': r['cores'], 'kind': 'port',
                       'sample': r['sample']},
      'e2e': {'value': r['value'], 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
      'gpu_launches': 0,
      'cpu_batch_per_step': args.cpu_batch,
      'note': 'TensorFlow 2.4.1 is not installable here (no network): this arm times the CPU '
              'oracle, a line-by-line torch-CPU restatement of the reference learner step.'}
  emit(line)


def workload_config(args, n):
  """Identical for both arms (the reference arm runs the same batch per step on the host)."""
  return {
      'workload': 'Impala%s learner step, T=%d, B=%d unrolls/GPU, synthetic 84x84x4 uint8 '
                  '(BASELINE configs[3]; per-GPU slice is the configs[1]/[2] shape)' %
                  ('Deep' if args.net == 'deep' else 'Shallow', args.unroll, args.batch),
      'net': 'ImpalaDeep (dmlab/networks.py:63-171)' if args.net == 'deep' else 'IMPALA shallow (paper)',
      'unroll_length': args.unroll, 'batch_per_gpu': args.batch,
      'global_batch': args.batch * n, 'num_actions': A,
      'num_action_repeats': 1,
      'optimizer': 'Adam lr=4.8e-4 beta1=0 eps=3.125e-7 (dmlab/vtrace_main.py:46-51)',
      'loss': 'gamma=0.99 lambda=1 baseline_cost=0.5 entropy_cost=2.5e-4 kl_cost=0',
      'grad_reduce': 'sum', 'parallelism': 'dp%d' % n,
      'l2': 'per-step inputs (37.9 MB uint8 frames) + activations (>2 GB) exceed the 126 MB L2; '
            'no explicit flush'}


# ----------------------------------------------------------------------------------------
class ClockSampler(object):
  """`nvidia-smi -lms 20` beside the benchmark.  Started BEFORE the warm-up steps: the tool's own
  start-up (NVML initialisation) can stall the GPU for tens of milliseconds, its 20 ms polls do not --
  `ready()` waits for the first sample, `begin()` marks the start of the timed region, and `stop()`
  keeps the samples taken between `begin()` and `stop()` (the timed region)."""
  Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
       'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
       'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,timestamp')

  def __init__(self, gpu_index):
    self.gpu = gpu_index
    self.t0 = None
    self.f = tempfile.NamedTemporaryFile('w+', suffix='.csv', delete=False)
    try:
      self.p = subprocess.Popen(['nvidia-smi', '--query-gpu=' + self.Q, '--format=csv,noheader,nounits',
                                 '-lms', '20', '-i', str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
    except Exception:
      self.p = None

  def ready(self, timeout=5.0):
    t_end = time.time() + timeout
    while self.p is not None and time.time() < t_end:
      try:
        if os.path.getsize(self.f.name) > 0:
          return True
      except OSError:
        pass
      time.sleep(0.01)
    return False

  def begin(self):
    self.t0 = time.time()

  @staticmethod
  def _stamp(text):
    import datetime
    try:
      return datetime.datetime.strptime(text.strip(), '%Y/%m/%d %H:%M:%S.%f').timestamp()
    except Exception:
      return None

  def stop(self):
    out = {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
    if self.p is None:
      return out
    t1 = time.time()
    self.p.terminate()
    try:
      self.p.wait(5)
    except Exception:
      self.p.kill()
    self.f.flush()
    rows = [l.strip().split(', ') for l in open(self.f.name) if l.strip()]
    os.unlink(self.f.name)
    if self.t0 is not None:
      inside = [r for r in rows if len(r) > 9 and self._stamp(r[9]) is not None and
                self.t0 - 0.02 <= self._stamp(r[9]) <= t1 + 0.02]
      if inside:
        rows = inside
    sm, reasons, mx = [], set(), None
    for r in rows:
      try:
        sm.append(float(r[1])); mx = float(r[2])
        for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[5:9]):
          if v.strip() == 'Active':
            reasons.add(name)
      except Exception:
        pass
    if sm:
      sm.sort()
      out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))
    return out


def conv_bytes_per_step(N, cat):
  """Algorithmic HBM bytes of one learner step for the conv categories (ImpalaDeep,
  fp32 activations, uint8 frames): every operand read once, every result written once."""
  stacks = [(84, 84, 4, 16), (42, 42, 16, 32), (21, 21, 32, 32)]
  tot, launches = 0, 0
  for si, (h, w, cin, c) in enumerate(stacks):
    ho, wo = (h + 1) // 2, (w + 1) // 2
    full_in = N * h * w * cin * (1 if si == 0 else 4)
    full_out = N * h * w * c * 4
    pooled = N * ho * wo * c * 4
    if cat == 'conv3x3_fwd':
      tot += full_in + full_out          # stack conv
      tot += 4 * (2 * pooled) + 2 * pooled   # 4 res convs (in+out) + 2 residual reads
      launches += 5
    elif cat == 'conv3x3_dgrad':
      tot += 4 * (2 * pooled) + 4 * pooled + 2 * pooled   # dy in, dx out, mask reads, 2 residual reads
      launches += 4
      if si > 0:
        tot += full_out + N * h * w * cin * 4
        launches += 1
    elif cat == 'conv3x3_wgrad':
      tot += full_in + full_out + 4 * (2 * pooled)        # x and dy read once per conv
      launches += 10                                      # kernel + reduce per conv
  return tot, launches


def conv_bytes_per_step_planes(N, cat):
  """Same accounting for conv_mode 'tc3p' (DESIGN 4.2): plane tensors hold hi+lo bf16 = 4 bytes per
  element (padding positions not counted); which tensors each kernel reads / writes differs from
  the fp32 layout: conv01 / conv11 write a raw and (conv01) a ReLU'd copy, the ReLU mask of a data
  gradient is the hi plane only (2 bytes per element)."""
  stacks = [(84, 84, 4, 16), (42, 42, 16, 32), (21, 21, 32, 32)]
  tot, launches = 0, 0
  for si, (h, w, cin, c) in enumerate(stacks):
    ho, wo = (h + 1) // 2, (w + 1) // 2
    full_in = N * h * w * cin * (1 if si == 0 else 4)
    full_out = N * h * w * c * 4
    pooled = N * ho * wo * c * 4
    taps = N * ho * wo * c                    # arg-max taps, 1 byte per pooled element
    if cat == 'conv3x3_fwd':
      if si == 0:
        tot += full_in + 2 * pooled + taps    # fused conv + pool: frames in, raw + ReLU'd pooled planes + taps out
      else:
        tot += full_in + full_out             # stack conv: plane tensor in, fp32 NHWC out (pooled by poolp_fwd)
      tot += 2 * pooled                       # conv00: relu(p) in, relu(c0) out
      tot += 4 * pooled                       # conv01: relu(c0) + p in, o0 and relu(o0) out
      tot += 2 * pooled                       # conv10
      tot += 3 * pooled                       # conv11: relu(c1) + o0 in, o1 out
      launches += 5
    elif cat == 'conv3x3_dgrad':
      tot += 4 * (2 * pooled) + 4 * (pooled // 2) + 2 * pooled   # dy in, dx out, hi-plane masks, 2 residuals
      launches += 4
      if si > 0:
        tot += full_out + N * h * w * cin * 4
        launches += 1
    elif cat == 'conv3x3_wgrad':
      if si == 0:
        tot += full_in + pooled + taps        # first layer: frames + POOLED gradient + taps (no full-resolution tensor)
      else:
        tot += full_in + full_out
      tot += 4 * (2 * pooled)
      launches += 5
  if cat == 'conv3x3_wgrad':
    launches += 1                             # one deferred reduce of all partials
  return tot, launches


def inference_path_bench(agent, iters=200, warmup=30, N=64, num_envs=256, T=20, batch=64, cuda_graph=None):
  """Hot path (1) of the north star: the batched central-inference step (reference
  agents/vtrace/learner.py:349-407) -- host batch -> H2D -> gather of the previous action / LSTM
  state -> T=1 ImpalaDeep forward -> in-kernel sampling -> write-back + unroll-store append ->
  actions back on the host -- through the public `InferenceHost.inference` call (no RPC
  transport), with a consumer draining the zero-copy training batches as a learner would.
  Wall clock (the call returns host actions, i.e. it is synchronous per batch)."""
  import threading
  import numpy as np
  import torch
  from seed_rl_b200 import _lib
  from seed_rl_b200.agents.vtrace import learner_loop
  from seed_rl_b200.common import utils
  host = learner_loop.InferenceHost(agent, num_envs, T, N, OBS, training_batch_size=batch, cuda_graph=cuda_graph)
  stop = []

  def drain():
    try:
      while True:
        slot, _ = learner_loop.assembled_batch(host.assembler)
        host.assembler.release(slot)
        stop.append(1)
    except utils.QueueClosedError:
      return
  th = threading.Thread(target=drain, daemon=True); th.start()
  rng = np.random.default_rng(7)
  run_ids = rng.integers(1, 2**40, num_envs)
  groups = [np.arange(g * N, (g + 1) * N, dtype=np.int32) for g in range(num_envs // N)]
  obs = [torch.from_numpy(rng.integers(0, 256, (N,) + OBS, dtype=np.uint8)).pin_memory().numpy() for _ in groups]
  zeros = np.zeros(N, np.float32)

  def one(i):
    g = i % len(groups)
    ids = groups[g]
    env = utils.EnvOutput(rng.normal(size=N).astype(np.float32), rng.random(N) < 0.01, obs[g],
                          np.zeros(N, bool), np.full(N, i, np.int32))
    return host.inference(ids, run_ids[ids], env, zeros)
  for i in range(warmup):
    one(i)
  torch.cuda.synchronize()
  n0 = _lib.launch_count()
  lat = []
  t0 = time.perf_counter()
  for i in range(iters):
    t1 = time.perf_counter()
    one(warmup + i)
    lat.append(time.perf_counter() - t1)
  dt = time.perf_counter() - t0
  launches = (_lib.launch_count() - n0) / iters
  host.assembler.close()
  lat.sort()
  h2d = N * (28224 + 4 + 1 + 1 + 4) + N * 4 + N * 8
  return {
      'what': 'central inference step (agents/vtrace/learner.py:349-407): host batch -> pinned staging -> H2D -> '
              '[gather prev action/state -> T=1 ImpalaDeep forward (conv_mode %s) -> sample -> scatter + '
              'unroll-store append]%s -> actions D2H; public API InferenceHost.inference, no RPC transport' %
              (agent.conv_mode, ' replayed as ONE CUDA graph' if host.use_graph else ''),
      'cuda_graph': bool(host.use_graph),
      'inference_batch_size': N, 'num_envs': num_envs, 'iters': iters,
      'inferences_per_sec': N * iters / dt, 'us_per_batch_mean': dt / iters * 1e6,
      'us_per_batch_p50': lat[len(lat) // 2] * 1e6, 'us_per_batch_p99': lat[int(len(lat) * 0.99)] * 1e6,
      'library_launches_per_batch': launches, 'h2d_bytes_per_batch': h2d, 'd2h_bytes_per_batch': N * 8,
      'training_batches_assembled': len(stop),
      'bound': 'latency: 64 frames x 0.11 GFLOP = 7 GFLOP and 1.8 MB of frames per batch are ~10 us of '
               'tensor / HBM time; the step is a chain of ~40 dependent small kernels (each pays its launch + '
               'setup: TMEM allocation, weights into shared memory) + 1.8 MB H2D + host bookkeeping; replaying it '
               'as a CUDA graph removes the CPU issue cost but not the dependent-kernel chain (measured: same '
               'p50), so throughput scales with the inference batch size instead',
  }


def inference_lanes_bench(agent, lanes=2, iters=150, warmup=30, N=64, num_envs=256, T=20, batch=64):
  """Aggregate central-inference throughput of `lanes` independent InferenceHosts on ONE GPU, each
  with its own environment shard, unroll store, CUDA graph and stream, driven by its own host thread
  (the reference builds one such host per core group, agents/vtrace/learner.py:314-416): the host
  side of one lane's call overlaps the other lane's graph replay.  Wall clock over all lanes."""
  import threading
  import numpy as np
  import torch
  from seed_rl_b200.agents.vtrace import learner_loop
  from seed_rl_b200.common import utils
  dev = torch.cuda.current_device()
  capture_lock = threading.Lock()
  gate = threading.Barrier(lanes + 1)
  errors, lat = [], [[] for _ in range(lanes)]

  def lane(k):
    host = None
    try:
      torch.cuda.set_device(dev)
      host = learner_loop.InferenceHost(agent, num_envs, T, N, OBS, training_batch_size=batch, cuda_graph=True)

      def drain():
        try:
          while True:
            slot, _ = learner_loop.assembled_batch(host.assembler)
            host.assembler.release(slot)
        except utils.QueueClosedError:
          return
      threading.Thread(target=drain, daemon=True).start()
      rng = np.random.default_rng(100 + k)
      run_ids = rng.integers(1, 2**40, num_envs)
      groups = [np.arange(g * N, (g + 1) * N, dtype=np.int32) for g in range(num_envs // N)]
      obs = [torch.from_numpy(rng.integers(0, 256, (N,) + OBS, dtype=np.uint8)).pin_memory().numpy() for _ in groups]
      zeros = np.zeros(N, np.float32)

      def one(i):
        ids = groups[i % len(groups)]
        env = utils.EnvOutput(rng.normal(size=N).astype(np.float32), rng.random(N) < 0.01, obs[i % len(groups)],
                              np.zeros(N, bool), np.full(N, i, np.int32))
        return host.inference(ids, run_ids[ids], env, zeros)
      with capture_lock:                       # one lane captures its graph at a time
        for i in range(warmup):
          one(i)
      gate.wait(120)
      for i in range(iters):
        t1 = time.perf_counter()
        one(warmup + i)
        lat[k].append(time.perf_counter() - t1)
      gate.wait(120)
    except Exception as exc:                   # pylint: disable=broad-except
      errors.append(repr(exc)[:200])
      gate.abort()
    finally:
      if host is not None and host.assembler is not None:
        host.assembler.close()
  threads = [threading.Thread(target=lane, args=(k,), daemon=True) for k in range(lanes)]
  for th in threads:
    th.start()
  try:
    gate.wait(180)
    t0 = time.perf_counter()
    gate.wait(180)
    wall = time.perf_counter() - t0
  except threading.BrokenBarrierError:
    return {'unavailable': '; '.join(errors) or 'barrier broken'}
  for th in threads:
    th.join(10)
  allat = sorted(x for l in lat for x in l)
  return {'lanes': lanes, 'inference_batch_size': N, 'envs_per_lane': num_envs, 'iters_per_lane': iters,
          'inferences_per_sec': lanes * N * iters / wall, 'us_per_batch_p50': allat[len(allat) // 2] * 1e6,
          'what': '%d independent InferenceHosts (own env shard / store / CUDA graph / stream / host thread) on one '
                  'GPU sharing the agent; aggregate wall-clock throughput' % lanes}


def r2d2_cpu_throughput(B, steps, warmup, burn_in=40, unroll=100):
  """The reference's R2D2 learner step (oracle port, torch-CPU fp32) on a bounded sample."""
  import torch
  from oracle import r2d2_learner_oracle as RL
  torch.set_num_threads(min(32, os.cpu_count() or 1))
  T = burn_in + unroll + 1
  lr = RL.CpuR2D2Learner(A, (84, 84, 1), 4, burn_in=burn_in, lr=0.00048, eps=1e-3)
  b = RL.synthetic_replay_batch(T, B, A, (84, 84, 1), seed=1234)
  for _ in range(warmup):
    lr.step(b)
  t0 = time.perf_counter()
  for _ in range(steps):
    lr.step(b)
  dt = (time.perf_counter() - t0) / max(steps, 1)
  return dict(value=B * unroll / dt, ms_per_step=dt * 1e3, cores=torch.get_num_threads(),
              sample='%d steps of B=%d sampled unrolls x (burn-in %d + %d + 1) after %d warm-up; torch-CPU fp32 '
                     'oracle port of agents/r2d2/learner.py:333-386,581-634, %d threads' %
                     (steps, B, burn_in, unroll, warmup, torch.get_num_threads()))


def run_r2d2(args):
  """BASELINE configs[4]: R2D2 LSTM agent, synthetic replay, n-step targets, 1 x B200.  A step =
  insert `batch/replay_ratio` new unrolls into the prioritized replay -> sample `batch` unrolls by
  priority (+ importance weights) -> burn-in + suffix unrolls of the online and target networks ->
  n-step double-DQN loss -> backward -> global-norm clip -> Adam -> priority write-back
  (reference agents/r2d2/learner.py:389-467,581-634,856-885)."""
  import numpy as np
  import torch
  from seed_rl_b200 import _lib
  from seed_rl_b200.agents.r2d2 import learner
  from seed_rl_b200.atari import networks
  from seed_rl_b200.common import optimizers, utils
  if args.impl == 'reference':
    if int(os.environ.get('RANK', '0')) != 0:
      return
    r = r2d2_cpu_throughput(4, max(1, min(args.steps, 3)), 1)
    return emit({'impl': 'reference', 'metric': R2D2_METRIC, 'value': r['value'], 'unit': UNIT, 'n_gpus': args.gpus,
                 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': r['ms_per_step'],
                 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
                 'data': 'synthetic', 'config': r2d2_config(args), 'gpu_launches': 0,
                 'cpu_baseline': {'value': r['value'], 'unit': UNIT, 'cores': r['cores'], 'kind': 'port',
                                  'sample': r['sample']},
                 'e2e': {'value': r['value'], 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}})
  torch.cuda.set_device(int(os.environ.get('LOCAL_RANK', '0')))
  st = learner.default_settings(batch_size=args.batch)
  obs, S = (84, 84, 1), 4
  T = st.burn_in + st.unroll_length + 1
  B, n_ins = st.batch_size, learner.get_replay_insertion_batch_size(st)
  agent = networks.DuelingLSTMDQNNet(A, obs, S, seed=0)
  target = networks.DuelingLSTMDQNNet(A, obs, S, seed=0)
  step = learner.R2D2LearnerStep(agent, target, optimizers.Adam(0.00048, epsilon=1e-3), settings=st)
  TS = utils.TensorSpec
  agent_state_specs = networks.AgentState((TS([512], 'float32', 'h'), TS([512], 'float32', 'c')),
                                          TS([84 * 84], 'int32', 'frames'))
  env_specs = utils.EnvOutput(TS([T], 'float32', 'reward'), TS([T], 'bool', 'done'),
                              TS([T, 84, 84, 1], 'uint8', 'observation'), TS([T], 'bool', 'abandoned'),
                              TS([T], 'int32', 'episode_step'))
  unroll_specs = learner.Unroll(agent_state_specs, TS([], 'float32', 'priority'), TS([T], 'int32', 'prev_actions'),
                                env_specs, learner.AgentOutput(TS([T], 'int32', 'action'), TS([T, A], 'float32', 'q')))
  replay = utils.PrioritizedReplay(st.replay_buffer_size, unroll_specs, st.importance_sampling_exponent)
  feeder = learner.ReplayFeeder(replay, st, generator=torch.Generator(device='cuda').manual_seed(1))
  rng = np.random.default_rng(1234)

  def host_unrolls(n):       # what the inference side would enqueue: env-major [n, T, ...], pinned
    pin = lambda a: torch.from_numpy(a).pin_memory()
    return learner.Unroll(
        networks.AgentState((pin(np.zeros((n, 512), np.float32)), pin(np.zeros((n, 512), np.float32))),
                            pin(np.zeros((n, 84 * 84), np.int32))),
        pin((rng.random(n) + 0.1).astype(np.float32)), pin(rng.integers(0, A, (n, T)).astype(np.int32)),
        utils.EnvOutput(pin(rng.normal(size=(n, T)).astype(np.float32)), pin(rng.random((n, T)) < 0.01),
                        pin(rng.integers(0, 256, (n, T) + obs, dtype=np.uint8)), pin(np.zeros((n, T), bool)),
                        pin(np.zeros((n, T), np.int32))),
        learner.AgentOutput(pin(rng.integers(0, A, (n, T)).astype(np.int32)),
                            pin(rng.normal(size=(n, T, A)).astype(np.float32))))
  host_new = host_unrolls(n_ins)
  h2d = sum(t.numel() * t.element_size() for t in utils.flatten(host_new))
  dev_new = utils.map_structure(lambda t: t.cuda(), host_new)
  while not feeder.ready() or replay.num_inserted < st.replay_buffer_size:
    feeder.insert(dev_new)

  last_step = [None]

  def one_step(from_host):
    new = utils.map_structure(lambda t: t.cuda(non_blocking=True), host_new) if from_host else dev_new
    feeder.insert(new)
    sampled = feeder.sample()
    loss, priorities, indices, norm = step.minimize(sampled)
    feeder.update_priorities(indices, priorities)
    last_step[0] = (loss, priorities, indices, norm)
    return loss

  def timed(fn, k):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(k):
      fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / k
  sampler = ClockSampler(torch.cuda.current_device())
  for _ in range(max(args.warmup, 16)):     # the caching allocator settles after a dozen sample/gather shapes
    one_step(False)
  sampler.ready()
  sampler.begin()
  n0 = _lib.launch_count()
  ms = timed(lambda: one_step(False), args.steps)
  launches = (_lib.launch_count() - n0) // args.steps
  agent.check_errors()
  clocks = sampler.stop()
  if args.dump_outputs:
    loss, priorities, indices, norm = last_step[0]
    outputs = {'loss': loss, 'priorities': priorities, 'indices': indices, 'gradient_norm': norm}
    outputs.update(('param/' + k, v) for k, v in agent.named_parameters().items())
    outputs.update(('grad/' + k, v) for k, v in agent.named_gradients().items())
    dump_outputs(args.dump_outputs, outputs)
  ms_e2e = timed(lambda: float(one_step(True)), args.steps)
  frames = B * st.unroll_length
  line = {'metric': R2D2_METRIC, 'value': frames / (ms * 1e-3), 'unit': UNIT, 'n_gpus': 1, 'steps': args.steps,
          'warmup': max(args.warmup, 16), 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak',
          'vs_baseline': None, 'dtype': 'bf16x3 (fp32-faithful tensor-core contraction), f32 elsewhere',
          'data': 'synthetic', 'config': r2d2_config(args), 'clocks': clocks,
          'e2e': {'value': frames / (ms_e2e * 1e-3), 'unit': UNIT, 'ms_per_step': ms_e2e,
                  'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': 4,
                  'api': 'ReplayFeeder.insert/sample/update_priorities + R2D2LearnerStep.minimize; the %d new '
                         'unrolls of every step come from pinned host memory' % n_ins},
          'gpu_launches': int(launches * args.steps), 'gpu_launches_per_step': int(launches), 'impl': 'b200'}
  if not args.no_extras:
    import ctypes
    L = _lib.lib()
    ncat = L.seedrl_profile_num_categories()
    ms_c = (ctypes.c_double * ncat)(); n_c = (ctypes.c_uint64 * ncat)()
    _lib.check(L.seedrl_profile_begin(_lib.stream_ptr()))
    one_step(False)
    _lib.check(L.seedrl_profile_end(ms_c, n_c))
    line['kernel_time_ms_per_step'] = {L.seedrl_profile_category_name(i).decode(): round(ms_c[i], 4) for i in range(ncat)}
    line['kernel_time_note'] = ('conv3x3_fwd = im2col, conv3x3_dgrad = col2im, sgemm = every GEMM incl. the three '
                                'convolutions (tcgen05 bf16x3), lstm_pointwise = the persistent LSTM(512) recurrences')
    # roofline of the dominant family: the tcgen05 GEMMs, against the dense bf16 peak x 1/3 (bf16x3)
    peaks = {}
    try:
      peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
      pass
    fl = r2d2_gemm_flops(T, B, st.burn_in)
    tf = fl * 3 / (ms_c[[L.seedrl_profile_category_name(i).decode() for i in range(ncat)].index('sgemm')] * 1e-3) / 1e12
    peak = float(peaks.get('bf16_tflops_sustained', 1465.2))
    line['roofline'] = {'kernel': 'gemm_tc_kernel (all contractions of the step, bf16x3: 3 MMAs per fp32 product)',
                        'bound': 'tensor', 'achieved': tf, 'peak': peak, 'unit': 'TFLOP/s', 'frac': tf / peak,
                        'traffic': None, 'fp32_equivalent_flops_per_step': fl}
    r = r2d2_cpu_throughput(4, 2, 1)
    line['cpu_baseline'] = {'value': r['value'], 'unit': UNIT, 'cores': r['cores'], 'kind': 'port',
                            'sample': r['sample'], 'ms_per_step': r['ms_per_step']}
  emit(line)


R2D2_METRIC = ('learner env-frames/sec (R2D2 learner step, device-timed; frames = batch_size x unroll_length) on '
               'synthetic prioritized replay @1 B200')


def r2d2_config(args):
  return {'workload': 'R2D2 learner step (BASELINE configs[4]): DuelingLSTMDQNNet 84x84x1 frames, stack 4, batch %d '
                      'sampled unrolls x (burn-in 40 + unroll 100 + 1), replay 100 unrolls, priority exponent 0.9, '
                      'n_steps 5, gamma 0.997, clip_norm 40, Adam lr 4.8e-4 eps 1e-3 (agents/r2d2/learner.py:43-92, '
                      'atari/r2d2_main.py:36-51)' % args.batch,
          'batch_size': args.batch, 'unroll_length': 100, 'burn_in': 40, 'num_actions': A, 'parallelism': 'dp1',
          'l2': 'per-step activations (>10 GB) exceed the 126 MB L2; no explicit flush'}


def r2d2_gemm_flops(T, B, burn_in):
  """2*MAC of every contraction of one step: online + target forward over all T rows, backward
  (2x) of the online suffix."""
  per_frame = (20 * 20 * 256 * 32 + 9 * 9 * 512 * 64 + 7 * 7 * 576 * 64 + 3136 * 512 + (512 + 1 + A) * 2048 +
               512 * 2048 + 2 * 512 * 512 + 512 * (1 + A))
  fwd = 2 * T * B * per_frame
  bwd = 2 * (T - burn_in) * B * per_frame
  return 2 * (fwd + bwd)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, arrays):
  """Writes every tensor of `arrays` as path/<name>.npy ('/' in a name becomes '.'): floating point as
  float32 (float64 stays float64), integers as float64 (exact below 2**53), so that two builds can be
  compared file by file."""
  import numpy as np
  out = {}
  for name, t in arrays.items():
    a = t.detach().cpu().numpy()
    out[name.replace('/', '.')] = a.astype(np.float32 if a.dtype.kind == 'f' and a.itemsize <= 4 else np.float64)
  total = sum(a.nbytes for a in out.values())
  if total > DUMP_LIMIT_BYTES:
    raise SystemExit('bench.py: --dump-outputs would write %d bytes, more than %d' % (total, DUMP_LIMIT_BYTES))
  os.makedirs(path, exist_ok=True)
  for name, a in out.items():
    np.save(os.path.join(path, name + '.npy'), a)


_JSON_FD = None


def emit(line):
  """The ONE JSON line goes to the real stdout; everything libraries print (e.g. NCCL's
  version banner) was redirected to stderr by main()."""
  data = (json.dumps(line) + '\n').encode()
  if _JSON_FD is None:
    sys.stdout.write(data.decode()); sys.stdout.flush()
  else:
    os.write(_JSON_FD, data)


def main():
  global _JSON_FD
  args = parse_args()
  sys.stdout.flush()
  _JSON_FD = os.dup(1)
  os.dup2(2, 1)
  if args.agent == 'r2d2':
    return run_r2d2(args)
  if args.impl == 'reference':
    return run_reference(args)

  import numpy as np
  import torch
  import torch.distributed as dist
  from seed_rl_b200 import _lib
  from seed_rl_b200.agents.vtrace import learner
  from seed_rl_b200.common import optimizers, utils
  from seed_rl_b200.dmlab import networks

  if not torch.cuda.is_available():
    raise SystemExit('bench.py: no CUDA device. The product path has no CPU fallback; use '
                     '--impl reference for the CPU oracle arm.')
  world = int(os.environ.get('WORLD_SIZE', '1'))
  rank = int(os.environ.get('RANK', '0'))
  local = int(os.environ.get('LOCAL_RANK', '0'))
  torch.cuda.set_device(local)
  if world > 1:
    dist.init_process_group('nccl', device_id=torch.device('cuda', local))
  T, B = args.unroll, args.batch
  T1 = T + 1

  # ---- synthetic batch (SURVEY 8d), seeded per rank, pinned on the host ----------------
  rng = np.random.default_rng(1234 + rank)
  host = dict(
      observation=rng.integers(0, 256, (T1, B) + OBS, dtype=np.uint8),
      reward=rng.normal(size=(T1, B)).astype(np.float32),
      done=rng.random((T1, B)) < 0.02,
      prev_actions=rng.integers(0, A, (T1, B), dtype=np.int64),
      action=rng.integers(0, A, (T1, B), dtype=np.int64),
      behaviour_logits=rng.normal(size=(T1, B, A)).astype(np.float32),
      behaviour_baseline=rng.normal(size=(T1, B)).astype(np.float32),
      h0=np.zeros((B, 256), np.float32), c0=np.zeros((B, 256), np.float32))
  pinned = {k: torch.from_numpy(v).pin_memory() for k, v in host.items()}
  h2d_bytes = sum(v.numel() * v.element_size() for v in pinned.values())
  dev = {k: torch.empty_like(v, device='cuda') for k, v in pinned.items()}

  def upload():
    for k in pinned:
      dev[k].copy_(pinned[k], non_blocking=True)

  def make_unroll():
    env = utils.EnvOutput(dev['reward'], dev['done'], dev['observation'],
                          torch.zeros(T1, B, dtype=torch.bool, device='cuda'),
                          torch.zeros(T1, B, dtype=torch.int32, device='cuda'))
    ao = networks.AgentOutput(dev['action'], dev['behaviour_logits'], dev['behaviour_baseline'])
    return learner.Unroll((dev['h0'], dev['c0']), dev['prev_actions'], env, ao)

  upload()
  unroll = make_unroll()
  cls = networks.ImpalaDeep if args.net == 'deep' else networks.ImpalaShallow
  agent = cls(A, OBS, seed=0, conv_mode=args.conv)   # same seed on every rank: replicas start identical
  opt = optimizers.Adam(optimizers.PolynomialDecay(4.8e-4, 10**6, 0.0), beta_1=0.0, epsilon=3.125e-7)
  step = learner.LearnerStep(agent, opt, settings=learner.default_loss_settings(), grad_reduce='sum',
                             overlap_reduce=os.environ.get('SEEDRL_OVERLAP_REDUCE', '1') != '0')

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  last_median = [None]

  def timed(fn, k):
    """EXACTLY k calls between one pair of CUDA events (barrier + synchronize on both sides,
    MAX over ranks); an event after every call also gives the per-step median (reported beside
    the mean, never instead of it)."""
    barrier()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(k + 1)]
    evs[0].record()
    for i in range(k):
      fn()
      evs[i + 1].record()
    barrier()
    ms = torch.tensor([evs[0].elapsed_time(evs[k])], device='cuda')
    if world > 1:
      dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    per = sorted(evs[i].elapsed_time(evs[i + 1]) for i in range(k))
    last_median[0] = per[len(per) // 2]
    return float(ms) / k

  # ---- kernel-only (inputs resident in HBM) --------------------------------------------
  sampler = ClockSampler(local) if rank == 0 else None       # its start-up overlaps the warm-up, not the timed steps
  for _ in range(max(args.warmup, 3)):
    step.minimize(unroll)
  if sampler:
    sampler.ready()
    sampler.begin()
  n0 = _lib.launch_count()
  ms_step = timed(lambda: step.minimize(unroll), args.steps)
  launches = (_lib.launch_count() - n0) // args.steps
  ms_step_median = last_median[0]
  agent.check_errors()      # raises if any kernel of the timed steps timed out on a barrier
  clocks = sampler.stop() if sampler else None
  if args.dump_outputs and rank == 0:
    # the last timed step's loss terms (the loss `minimize` returned is 'total') and the state it left
    outputs = {'loss/' + k: step.last_loss_terms[i] for k, i in _lib.LT.items()}
    outputs.update(('param/' + k, v) for k, v in agent.named_parameters().items())
    outputs['param/entropy_cost_param'] = agent.entropy_cost_param
    outputs.update(('grad/' + k, v) for k, v in agent.named_gradients().items())
    dump_outputs(args.dump_outputs, outputs)
  value = world * B * T / (ms_step * 1e-3)

  # ---- end to end: pinned host batch -> H2D -> step -> loss to host ---------------------
  d2h_bytes = 4

  # The public feed API (learner.DeviceFeeder): every step uploads ONE full batch from pinned
  # host memory (38 MB) and reads the loss back; the upload of batch i+1 runs on a copy stream
  # while step i trains (double buffering), as the reference's prefetching input pipeline does.
  feeder = learner.DeviceFeeder(pinned)

  def unroll_of(d):
    env = utils.EnvOutput(d['reward'], d['done'], d['observation'],
                          torch.zeros(T1, B, dtype=torch.bool, device='cuda'),
                          torch.zeros(T1, B, dtype=torch.int32, device='cuda'))
    ao = networks.AgentOutput(d['action'], d['behaviour_logits'], d['behaviour_baseline'])
    return learner.Unroll((d['h0'], d['c0']), d['prev_actions'], env, ao)
  slot_unrolls = [unroll_of(d) for d in feeder.slots]
  feeder.put(pinned)                      # batch 0 (before the timed region; K more follow inside)

  def e2e_step():
    slot, _ = feeder.get()
    feeder.put(pinned)                    # this step's upload: the NEXT batch, overlapped with the step
    loss, _ = step.minimize(slot_unrolls[slot])
    feeder.done_with(slot)
    float(loss)          # device -> host read of the step's result
  for _ in range(2):
    e2e_step()
  ms_e2e = timed(e2e_step, args.steps)
  e2e_value = world * B * T / (ms_e2e * 1e-3)

  def e2e_serial_step():                  # same, without overlap: copy, then step (for reference)
    upload()
    loss, _ = step.minimize(unroll)
    float(loss)
  ms_e2e_serial = timed(e2e_serial_step, max(3, args.steps // 2))

  line = {
      'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
      'warmup': max(args.warmup, 3), 'ms_per_step': ms_step, 'ms_per_step_median': ms_step_median,
      'higher_is_better': True,
      'scaling': 'weak', 'vs_baseline': None,
      'dtype': {'tc': 'bf16', 'tc3': 'bf16x3 (fp32-faithful tensor-core contraction), f32 elsewhere',
                'tc3p': 'bf16x3 (fp32-faithful tensor-core contraction; activations stored as bf16 hi+lo '
                        'pairs), f32 elsewhere',
                'simt': 'f32'}[args.conv], 'data': 'synthetic',
      'config': workload_config(args, world), 'conv_path': args.conv, 'clocks': clocks,
      'e2e': {'value': e2e_value, 'unit': UNIT, 'ms_per_step': ms_e2e,
              'h2d_bytes_per_step': h2d_bytes, 'd2h_bytes_per_step': d2h_bytes,
              'api': 'seed_rl_b200.agents.vtrace.learner.DeviceFeeder.put/get + LearnerStep.minimize(Unroll)',
              'overlap': 'H2D of batch i+1 on a copy stream during step i (double-buffered device slots)',
              'ms_per_step_serial_copy_then_step': ms_e2e_serial},
      'gpu_launches': int(launches * args.steps), 'gpu_launches_per_step': int(launches),
      'impl': 'b200'}

  if world > 1:
    # data-parallel replicas must stay bit-identical (deterministic kernels + the same reduced
    # gradient everywhere): compare a checksum of the parameter arena across ranks
    cs = agent.params.double().sum().reshape(1)
    lo, hi = cs.clone(), cs.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    line['replicas_in_sync'] = bool((lo == hi).item())
    line['grad_exchange'] = (('ncclAllReduce(SUM) in two buckets: heads+Dense+LSTM (94 %% of the %.2f MB arena) on a '
                              'side stream during the conv backward, conv stacks after it' if step.overlap_reduce else
                              'one ncclAllReduce(SUM) of the %.2f MB arena after the backward') %
                             (agent.params.numel() * 4 / 1e6))
  peaks = {}
  try:
    peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
  except Exception:
    pass
  hbm_peak = float(peaks.get('hbm_gbs', 6650.0))
  peak_src = 'measured (MEASURED_PEAKS.json hbm_gbs)' if 'hbm_gbs' in peaks else 'fallback 6.65 TB/s'

  if not args.no_extras:
    # ---- profiling pass (separate from the timed regions) --------------------------------
    L = _lib.lib()
    ncat = L.seedrl_profile_num_categories()
    ms_c = (ctypes.c_double * ncat)(); n_c = (ctypes.c_uint64 * ncat)()
    PSTEPS = 3
    barrier()
    _lib.check(L.seedrl_profile_begin(_lib.stream_ptr()))
    for _ in range(PSTEPS):
      step.minimize(unroll)
    _lib.check(L.seedrl_profile_end(ms_c, n_c))
    barrier()
    cats = {L.seedrl_profile_category_name(i).decode(): (ms_c[i] / PSTEPS, int(n_c[i]) // PSTEPS)
            for i in range(ncat)}
    tot = sum(v[0] for v in cats.values())
    line['kernel_time_ms_per_step'] = {k: round(v[0], 4) for k, v in cats.items()}
    line['kernel_launches_per_step'] = {k: v[1] for k, v in cats.items()}
    if args.net == 'deep':
      conv_cats = [k for k in ('conv3x3_fwd', 'conv3x3_dgrad', 'conv3x3_wgrad')]
      dom = max(conv_cats, key=lambda k: cats[k][0])
      nbytes, nl = (conv_bytes_per_step_planes if args.conv == 'tc3p' else conv_bytes_per_step)(T1 * B, dom)
      ms_dom = cats[dom][0]
      ach = nbytes / (ms_dom * 1e-3) / 1e9
      line['roofline'] = {
          'kernel': dom, 'bound': 'hbm', 'achieved': ach, 'peak': hbm_peak, 'unit': 'GB/s',
          'frac': ach / hbm_peak, 'traffic': None,
          'algorithmic_bytes_per_launch': nbytes / max(cats[dom][1], 1),
          'avg_launch_ms': ms_dom / max(cats[dom][1], 1), 'launches_per_step': cats[dom][1],
          'share_of_step': ms_dom / tot if tot else None, 'peak_source': peak_src,
          'per_category': {
              k: {'ms': cats[k][0], 'algorithmic_bytes': (conv_bytes_per_step_planes if args.conv == 'tc3p'
                                                          else conv_bytes_per_step)(T1 * B, k)[0]}
              for k in conv_cats},
          'note': 'category time from CUDA events around every launch of 3 profiled steps; algorithmic bytes = '
                  'every operand read once + every result written once in the layout of this conv path '
                  '(bench.py conv_bytes_per_step*); the convs are HBM-bound (AI ~ 36-70 FLOP/B), tensor FLOPs '
                  'are not the limit'}
      for k, v in line['roofline']['per_category'].items():
        v['GBps'] = v['algorithmic_bytes'] / (v['ms'] * 1e-3) / 1e9 if v['ms'] else None
        v['frac'] = v['GBps'] / hbm_peak if v['ms'] else None

    if rank == 0 and world == 1:
      # ---- the fused V-trace loss kernel: B sweep (north star: >= 60% HBM at streaming size)
      sweep = []
      st = learner.default_loss_settings()
      ecp = agent.entropy_cost_param
      for Bs in (64, 4096, 65536):
        g = torch.Generator(device='cuda').manual_seed(0)
        ll = torch.randn(T1, Bs, A, device='cuda', generator=g); lb = torch.randn(T1, Bs, device='cuda', generator=g)
        bl = torch.randn(T1, Bs, A, device='cuda', generator=g)
        act = torch.randint(0, A, (T1, Bs), device='cuda', generator=g)
        rew = torch.randn(T1, Bs, device='cuda', generator=g); dn = torch.rand(T1, Bs, device='cuda', generator=g) < 0.02
        flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
        for _ in range(3):
          learner.vtrace_loss_fwd_bwd(st, ll, lb, bl, act, rew, dn, ecp)
        times = []
        for _ in range(10):
          flush.zero_()          # evict L2 (256 MB > 126 MB)
          e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
          e0.record()
          learner.vtrace_loss_fwd_bwd(st, ll, lb, bl, act, rew, dn, ecp)
          e1.record(); torch.cuda.synchronize()
          times.append(e0.elapsed_time(e1))
        times.sort()
        ms = times[len(times) // 2]
        nb = (161 + 76) * T * Bs + 4 * Bs + 32          # SURVEY 8(d) algorithmic bytes
        # kernel alone: 20 launches back to back between one pair of events (the Python
        # wrapper costs ~30 us of host time per call, which a single-launch bracket includes)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record()
        for _ in range(20):
          learner.vtrace_loss_fwd_bwd(st, ll, lb, bl, act, rew, dn, ecp)
        e1.record(); torch.cuda.synchronize()
        msk = e0.elapsed_time(e1) / 20
        ws = 3 * T1 * Bs * A * 4
        sweep.append({'B': Bs, 'ms_single_launch_l2_flushed': ms, 'ms_back_to_back': msk,
                      'working_set_bytes': ws, 'exceeds_l2': ws > (126 << 20),
                      'algorithmic_bytes': nb, 'GBps': nb / (msk * 1e-3) / 1e9,
                      'frac_of_hbm_peak': nb / (msk * 1e-3) / 1e9 / hbm_peak,
                      'GBps_single_launch': nb / (ms * 1e-3) / 1e9})
        del ll, lb, bl, act, rew, dn, flush
      line['roofline_vtrace_loss'] = {
          'bound': 'hbm', 'peak': hbm_peak, 'unit': 'GB/s', 'peak_source': peak_src,
          'kernel': 'vtrace_loss_stream_kernel (B >= 148 tiles) / vtrace_loss_kernel (small B)',
          'timing': 'GBps = algorithmic bytes / mean of 20 back-to-back launches (inputs + outputs of the '
                    'B=65536 case are 297 MB > 126 MB L2; the smaller cases are L2-resident and '
                    'host-launch-bound, reported for latency only); ms_single_launch_l2_flushed = median of '
                    '10 single launches after an L2 flush, including the Python wrapper',
          'sweep': sweep}
      # ---- the other contraction paths, same workload (5 steps each) ----------------------
      others = {}
      for mode in ('simt', 'tc', 'tc3', 'tc3p'):
        if mode == args.conv or (mode == 'tc3p' and args.net != 'deep'):
          continue
        ag = cls(A, OBS, seed=0, conv_mode=mode)
        stp = learner.LearnerStep(ag, optimizers.Adam(4.8e-4, beta_1=0.0, epsilon=3.125e-7),
                                  settings=learner.default_loss_settings())
        for _ in range(3):
          stp.minimize(unroll)
        ms = timed(lambda: stp.minimize(unroll), 5)
        others[mode] = {'ms_per_step': ms, 'value': B * T / (ms * 1e-3)}
        del ag, stp
      line['other_conv_paths'] = others
      # ---- CPU baseline beside it (bounded sample) ----------------------------------------
      r = cpu_learner_throughput(args.net, T, args.cpu_batch, 5, 2)
      line['cpu_baseline'] = {'value': r['value'], 'unit': UNIT, 'cores': r['cores'], 'kind': 'port',
                              'sample': r['sample'], 'ms_per_step': r['ms_per_step']}

    if rank == 0 and world == 1 and args.net == 'deep':
      try:
        line['inference_path'] = inference_path_bench(agent)
        eager = inference_path_bench(agent, cuda_graph=False)
        line['inference_path']['without_cuda_graph'] = {k: eager[k] for k in (
            'inferences_per_sec', 'us_per_batch_mean', 'us_per_batch_p50', 'library_launches_per_batch')}
        big = inference_path_bench(agent, N=256, num_envs=1024, iters=100, warmup=20)
        line['inference_path']['at_inference_batch_256'] = {k: big[k] for k in (
            'inference_batch_size', 'num_envs', 'inferences_per_sec', 'us_per_batch_mean', 'us_per_batch_p50',
            'h2d_bytes_per_batch')}
      except Exception as exc:        # pylint: disable=broad-except
        line['inference_path'] = {'unavailable': repr(exc)[:300]}
      try:
        if isinstance(line.get('inference_path'), dict) and 'unavailable' not in line['inference_path']:
          line['inference_path']['two_lanes'] = inference_lanes_bench(agent, lanes=2)
      except Exception as exc:        # pylint: disable=broad-except
        line['inference_path']['two_lanes'] = {'unavailable': repr(exc)[:300]}

    if rank == 0 and world == 1 and args.net == 'deep' and args.conv != 'simt':
      # ---- the most time-consuming single kernel instance of the step, alone: the 16->16 conv
      # @42x42 on all T1*B frames (8 launches/step as forward + data gradient).  Launch time
      # measured live with CUDA events (10 back-to-back launches, working set ~300 MB >> L2).
      # Runs LAST and guarded: a failure here must never cost the bench line.
      try:
        Nf, Hh, Cc = T1 * B, 42, 16
        xk = torch.randn(Nf, Hh, Hh, Cc, device='cuda'); wk = torch.randn(3, 3, Cc, Cc, device='cuda') * 0.1
        bk = torch.zeros(Cc, device='cuda')
        wqk = torch.empty(2 * 9 * 16 * Cc * 2, dtype=torch.uint8, device='cuda')
        errk = torch.zeros(1, dtype=torch.int32, device='cuda')
        if args.conv == 'tc3p':
          nb = int(L.seedrl_debug_planes_bytes(Nf, Hh, Hh, Cc))
          xin = torch.empty(nb, dtype=torch.uint8, device='cuda'); ok = torch.empty(nb, dtype=torch.uint8, device='cuda')
          _lib.check(L.seedrl_debug_to_planes(Nf, Hh, Hh, Cc, 1, _lib.ptr(xk), _lib.ptr(xin), _lib.stream_ptr()))
          kname = 'convp_kernel<16,16,4> (TMA + tcgen05 bf16x3, plane tensors in/out) N=%d 42x42' % Nf

          def conv_once():
            _lib.check(L.seedrl_debug_convp(Cc, Cc, Nf, Hh, Hh, _lib.ptr(xin), _lib.ptr(wk), _lib.ptr(bk), None, None,
                                            0, None, _lib.ptr(ok), None, _lib.ptr(wqk), _lib.ptr(errk),
                                            _lib.stream_ptr()))
        else:
          ok = torch.empty(Nf, Hh, Hh, Cc, device='cuda')
          splitk = 1 if args.conv == 'tc3' else 0
          kname = 'conv3x3_tc_kernel<16,16,relu-in,%s,512> N=%d 42x42' % ('bf16x3' if splitk else 'bf16', Nf)

          def conv_once():
            _lib.check(L.seedrl_debug_conv3x3_tc(Cc, Cc, 1, splitk, Nf, Hh, Hh, _lib.ptr(xk), _lib.ptr(wk),
                                                 _lib.ptr(bk), None, None, _lib.ptr(ok), 0, 0, _lib.ptr(wqk),
                                                 _lib.ptr(errk), _lib.stream_ptr()))
        for _ in range(3):
          conv_once()
        ms_k = timed(conv_once, 10)
        alg = 2.0 * Nf * Hh * Hh * Cc * 4
        # DRAM traffic of this kernel from the committed `ncu --set full` capture of the same source
        # (profiles/r02_ncu_traffic.json, tools/ncu_traffic.py), scaled by the frame count
        traffic, tc_busy, tsrc = None, None, None
        try:
          tj = json.load(open(os.path.join(ROOT, 'profiles', 'r02_ncu_traffic.json')))
          for kn, rec in tj.items():
            if 'convp_kernel<16, 16, 4>' in kn and args.conv == 'tc3p':
              traffic = (rec['dram_read_bytes'] + rec['dram_write_bytes']) * Nf / rec['frames']
              tc_busy, tsrc = rec['tensor_pipe_active_pct'], 'profiles/' + rec['report'].replace('.ncu-rep', '.txt')
        except Exception:
          pass
        line['roofline_dominant_kernel'] = {
            'kernel': kname + ' (+ its 3 us weight-pack launch)',
            'bound': 'hbm', 'algorithmic_bytes_per_launch': alg, 'avg_launch_ms': ms_k,
            'achieved': alg / (ms_k * 1e-3) / 1e9, 'peak': hbm_peak, 'unit': 'GB/s',
            'frac': alg / (ms_k * 1e-3) / 1e9 / hbm_peak, 'traffic': traffic,
            'traffic_source': tsrc, 'tensor_pipe_busy_pct_ncu': tc_busy,
            'second_bound': 'tensor pipe: small-N tcgen05.mma is limited by its 4 KB A-tile read from shared '
                            'memory (~39 clk per 128xNx16 whatever N); ncu shows the pipe ~80 % busy at ~50 % of '
                            'HBM peak, i.e. the kernel sits at the instruction-rate limit of bf16x3 at N = 16..64',
            'launches_per_step': 8, 'ok': int(errk.item()) == 0}
        if traffic and 'roofline' in line:
          line['roofline']['traffic'] = traffic * line['roofline']['algorithmic_bytes_per_launch'] / alg
          line['roofline']['traffic_note'] = ('DRAM bytes of the dominant conv instance (ncu) scaled by the '
                                              "family's algorithmic bytes per launch")
        del xk, ok
      except Exception as exc:        # pylint: disable=broad-except
        line['roofline_dominant_kernel'] = {'unavailable': repr(exc)[:200]}

  if rank == 0:
    emit(line)
  if world > 1:
    dist.destroy_process_group()


if __name__ == '__main__':
  main()
