#!/usr/bin/env python
"""bench.py - QT-Opt replay transitions/sec on B200 (BASELINE.json metric), one JSON line.

  python bench.py --gpus 1 --steps K --warmup W                   # config C2 (default), this engine
  python bench.py --config c3|c4|c5 ...                           # the other BASELINE.json configs
  python bench.py --impl reference --steps K --warmup W           # the reference path's CPU restatement
  torchrun ... bench.py --gpus N ...                              # data parallel, one rank per GPU

Configs (BASELINE.json `configs`, SURVEY.md 8d):
  c2  QT-Opt ResNet-50 Q-critic (or --model grasping44) train step, synthetic 472x472 replay, batch 512 per GPU:
      crop/convert of the uint8 512x640 frames -> critic forward -> log loss -> backward -> bucketed NCCL all-reduce
      -> fused optimizer + EMA.
  c3  c2 with the CEM-maximised Bellman target computed inside the step: next-state tower of the lagged target
      network once, 2 x (Philox sampling, one [B*64] post-merge pass, elite refit), y = r + gamma (1-done) max Q,
      then the c2 step on y.  Also reports CEM Q-evals/s.
  c4  BC-Z FiLM-ResNet-18 behaviour cloning (language conditioned, 200x200, 10 waypoints) train step.
  c5  Grasp2Vec (two truncated ResNet-50 towers, n-pairs loss) train step on 224x224 triples.

`value` times the step with the batch resident in HBM (CUDA events, max over ranks); `e2e` times the same step through
the public API with the batch in HOST memory - for c2 / c4 / c5 through train_eval_model + the T2R model (the
reference's own entry point, utils/train_eval.py:424-438: pinned staging, H2D on a copy stream, preprocessor,
train_step) with the loss read back every step, for c3 through BellmanCriticTrainStep.step with pinned buffers.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np
import torch

METRIC = 'qtopt_replay_transitions_per_sec'
# Algorithmic work per unit (SURVEY.md 8d / BASELINE.md 2; 2*MACs, train = 3x forward).
TRAIN_GFLOP = {'resnet50': 110.9, 'grasping44': 26.4}
CEM_GFLOP_PER_QEVAL = {'resnet50': 7.4, 'grasping44': 0.346}
STATE_TOWER_GFLOP = {'resnet50': 29.5, 'grasping44': 8.44}
CONFIG_NAMES = {
    'c2': 'C2: QT-Opt {critic} Q-critic train step, synthetic 512x640 uint8 replay frames -> 472x472 crop',
    'c3': 'C3: QT-Opt {critic} Q-critic train step WITH the CEM-maximised Bellman target (64 samples x 2 iterations, '
          'lagged target network) inside the step, synthetic 512x640 uint8 replay (state + next-state frames)',
    'c4': 'C4: BC-Z FiLM-ResNet-18 behaviour cloning train step (language conditioning, 512x640 uint8 -> crop 450 -> '
          '200x200, 10 waypoints, xyz + quaternion + gripper heads)',
    'c5': 'C5: Grasp2Vec train step (scene + goal truncated ResNet-50 towers, n-pairs loss) on 224x224 triples',
}
# --dump-outputs: at most 4 Mi float32 elements per array, 64 MB over the three arrays a step writes
DUMP_MAX_ELEMENTS = 1 << 22


def parse_args():
  p = argparse.ArgumentParser()
  p.add_argument('--gpus', type=int, default=1)
  p.add_argument('--steps', type=int, default=8)
  p.add_argument('--warmup', type=int, default=3)
  p.add_argument('--impl', default='b200', choices=['b200', 'reference'])
  p.add_argument('--config', default='c2', choices=['c2', 'c3', 'c4', 'c5'])
  p.add_argument('--model', default='resnet50', choices=['resnet50', 'grasping44'])
  p.add_argument('--batch', type=int, default=None, help='units per GPU per step (default: 512 for c2/c3, 256 for c4/c5)')
  p.add_argument('--cpu-batch', type=int, default=8, help='batch of the bounded CPU sample')
  p.add_argument('--cem-chunk', type=int, default=32, help='transitions per post-merge pass of the ResNet-50 CEM')
  p.add_argument('--data', default='synthetic', choices=['synthetic', 'records'],
                 help="e2e input: host numpy batches, or TFRecord shards of JPEG-encoded transitions (c2 only): read, CRC, "
                      "tf.Example parse, split JPEG decode (Huffman on host threads, IDCT/colour on the GPU), step")
  p.add_argument('--records', type=int, default=2048, help='synthetic transitions written per rank for --data records')
  p.add_argument('--no-cpu-baseline', action='store_true')
  p.add_argument('--no-e2e', action='store_true')
  p.add_argument('--no-extras', action='store_true', help='skip the Grasping44 / CEM side measurements of c2')
  p.add_argument('--dump-outputs', metavar='DIR', default=None,
                 help='after the timed steps, write what the last timed step computed (its loss, the trainable variables '
                      'and the moving statistics it updated) as DIR/<name>.npy in float32; an array of more than %d '
                      'elements is replaced by the elements at a fixed, seeded sample of its indices' % DUMP_MAX_ELEMENTS)
  args = p.parse_args()
  if args.dump_outputs and args.impl != 'b200':
    p.error('--dump-outputs writes the outputs of the b200 engine')
  if args.batch is None:
    args.batch = 512 if args.config in ('c2', 'c3') else 256
  return args


# ---------------------------------------------------------------------------------------------
# clocks (B200_PROFILING.md recipe), sampled DURING the timed region
# ---------------------------------------------------------------------------------------------
class ClockSampler(object):
  QUERY = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
           'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
           'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

  def __init__(self, index):
    self.index, self.proc, self.lines = index, None, []

  def start(self):
    try:
      self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.QUERY,
                                    '--format=csv,noheader,nounits', '-lms', '200'],
                                   stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      self.thread = threading.Thread(target=self._read, daemon=True)
      self.thread.start()
    except OSError:
      self.proc = None

  def _read(self):
    for line in self.proc.stdout:
      self.lines.append(line.strip())

  def stop(self):
    if self.proc is None:
      return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
    self.proc.terminate()
    try:
      self.proc.wait(timeout=5)
    except subprocess.TimeoutExpired:
      self.proc.kill()
    sm, smax, reasons = [], [], set()
    names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
    for line in self.lines:
      f = [x.strip() for x in line.split(',')]
      if len(f) < 9:
        continue
      try:
        sm.append(float(f[1]))
        smax.append(float(f[2]))
      except ValueError:
        continue
      for name, v in zip(names, f[5:9]):
        if v.lower().startswith('active'):
          reasons.add(name)
    return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(smax) if smax else None,
            'reasons': sorted(reasons), 'samples': len(sm)}


def measured_peaks():
  path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(path):
    with open(path) as f:
      d = json.load(f)
    return {'tflops': d.get('bf16_tflops_sustained', 1400.0), 'tflops_burst': d.get('bf16_tflops', 1590.0),
            'hbm_gbs': d.get('hbm_gbs', 6650.0), 'source': 'measured'}
  return {'tflops': 1400.0, 'tflops_burst': 1590.0, 'hbm_gbs': 6650.0, 'source': 'fallback'}


def dominant_kernel_traffic():
  """dram read + write bytes of ONE launch of the dominant kernel from the committed ncu --set full capture
  (profiles/r02_dominant_kernel_traffic.json, written from the .ncu-rep by scripts/ncu_traffic.py); None without it."""
  path = os.path.join(ROOT, 'profiles', 'r02_dominant_kernel_traffic.json')
  if os.path.exists(path):
    with open(path) as f:
      return json.load(f)
  return None


def workload_config(args, world):
  critic = {'resnet50': 'ResNet-50', 'grasping44': 'Grasping44'}[args.model]
  cfg = {'workload': CONFIG_NAMES[args.config].format(critic=critic), 'baseline_config': args.config,
         'per_gpu_batch': args.batch, 'global_batch': args.batch * world, 'parallelism': 'dp%d' % world,
         'l2_flush': 'inputs and activations of every step exceed the 126 MB L2 (two alternating input sets)'}
  if args.config in ('c2', 'c3'):
    cfg.update(critic=args.model, image='472x472x3', optimizer='momentum+EMA')
  if args.config == 'c3':
    cfg.update(cem_samples=64, cem_iterations=2, cem_elites=10, gamma=0.9, target_network='lagged copy, refresh every 100 steps')
  if args.config == 'c4':
    cfg.update(tower='FiLM-ResNet-18 v2', image='200x200x3', optimizer='adam')
  if args.config == 'c5':
    cfg.update(tower='2 x ResNet-50 v2 truncated after block layer 3', image='224x224x3 (3 per sample)', optimizer='adam')
  return cfg


# ---------------------------------------------------------------------------------------------
# CPU baseline: the oracle restatement of the reference step (bench `cpu_baseline` / --impl reference)
# ---------------------------------------------------------------------------------------------
def usable_host_threads():
  """Host threads this process can really run: the affinity mask capped by the cgroup CPU quota (a
  128-core box with a 16-CPU quota runs a 128-thread torch step 70x slower than a 16-thread one)."""
  n = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
  try:
    quota, period = open('/sys/fs/cgroup/cpu.max').read().split()
    if quota != 'max':
      n = min(n, max(1, int(int(quota) / int(period))))
  except (OSError, ValueError):
    try:
      quota = int(open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us').read())
      period = int(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
      if quota > 0:
        n = min(n, max(1, quota // period))
    except (OSError, ValueError):
      pass
  return n


def cpu_reference_rate(args, steps, warmup):
  """Units/s of the torch-CPU fp32 restatement of the reference step on all usable host cores, on a bounded sample
  (batch args.cpu_batch) of the same workload.  Executes oracle/ - allowed only here.  Returns (rate, threads,
  seconds per step, description of what ran)."""
  from oracle import qtopt_networks, resnet as oracle_resnet, tf_ops
  threads = usable_host_threads()
  torch.set_num_threads(threads)
  rng = np.random.RandomState(0)
  batch = args.cpu_batch
  if args.config in ('c2', 'c3'):
    size = 472
    img = torch.from_numpy(rng.uniform(0, 1, (batch, size, size, 3)).astype(np.float32))
    grasp = torch.from_numpy(rng.uniform(-1, 1, (batch, 10)).astype(np.float32))
    reward = torch.from_numpy((rng.uniform(size=(batch, 1)) < 0.3).astype(np.float32))
    if args.model == 'grasping44':
      variables = qtopt_networks.to_torch(qtopt_networks.init_variables(0))
      fwd = lambda im, gr, train: qtopt_networks.model(variables, im, gr, train)
      predict = lambda im, gr: (lambda ep: (qtopt_networks.model(variables, im, gr, False, end_points=ep), ep)[1])({})['predictions']
    else:
      variables = {}
      with torch.no_grad():
        oracle_resnet.critic(variables, img[:1], grasp[:1], False, rng=np.random.RandomState(0))
      for k, v in variables.items():
        v.requires_grad_(not (k.endswith('moving_mean') or k.endswith('moving_variance')))
      fwd = lambda im, gr, train: oracle_resnet.critic(variables, im, gr, train)
      predict = lambda im, gr: (lambda ep: (oracle_resnet.critic(variables, im, gr, False, end_points=ep), ep)[1])({})['predictions']
    params = [v for v in variables.values() if v.requires_grad]
    momentum = [torch.zeros_like(p) for p in params]
    what = 'torch-CPU fp32 restatement of the reference train step (forward, log loss + l2, backward, momentum)'

    def cem_target(next_img):
      """policies/policies.py:133-169 on the host: numpy CEM (64 x 2, 10 elites) over the oracle's Q."""
      from oracle import cem as oracle_cem
      targets = []
      for i in range(next_img.shape[0]):
        rs = np.random.RandomState(i)

        def objective(samples):
          actions = torch.from_numpy(np.asarray(samples, np.float32))[None]
          with torch.no_grad():
            q = predict(next_img[i:i + 1], actions)
          return list(q.numpy().reshape(-1))

        _, values, _ = oracle_cem.cross_entropy_method(
            lambda mean, stddev: list(mean + stddev * rs.standard_normal((64, 10))), objective,
            oracle_cem.normal_update_fn, {'mean': np.zeros(10), 'stddev': np.ones(10)}, 10, 2)
        targets.append(float(max(values)))
      return torch.tensor(targets, dtype=torch.float32).reshape(-1, 1)

    def step():
      label = reward
      if args.config == 'c3':
        label = reward + 0.9 * cem_target(img)     # the same frames stand in for the next states
      logits = fwd(img, grasp, True)
      loss = tf_ops.log_loss(label.clamp(0, 1), torch.sigmoid(logits))
      loss = loss + sum(tf_ops.l2_regularizer(7e-5, v) for k, v in variables.items()
                        if k.endswith('/weights') or k.endswith('/kernel'))
      grads = torch.autograd.grad(loss, params)
      with torch.no_grad():
        for p_, g_, m_ in zip(params, grads, momentum):
          m_.mul_(0.9).add_(g_)
          p_.sub_(1e-4 * m_)
      return float(loss.detach())
    if args.config == 'c3':
      what += ' preceded by numpy CEM (64 samples x 2 iterations) over the oracle Q for every transition'
  else:
    # c4 / c5: the vision towers dominate; the CPU sample runs the oracle tower forward + backward with a stand-in loss
    size, n_img, rs = (200, 1, 18) if args.config == 'c4' else (224, 3, 50)
    img = torch.from_numpy(rng.uniform(0, 1, (batch * n_img, size, size, 3)).astype(np.float32))
    variables = {}

    def tower(im, train, rng_=None):
      builder = oracle_resnet._Builder(variables, train, 'resnet_model/', None, rng_)
      x = oracle_resnet.stem(builder, im)
      return oracle_resnet.block_layers(builder, x, rs, 0, 3 if args.config == 'c5' else 4)

    with torch.no_grad():
      tower(img[:1], False, np.random.RandomState(0))
    for k, v in variables.items():
      v.requires_grad_(not (k.endswith('moving_mean') or k.endswith('moving_variance')))
    params = [v for v in variables.values() if v.requires_grad]
    what = ('torch-CPU fp32 restatement of the ResNet-%d v2 tower(s) of the step (forward + backward, stand-in mean '
            'loss; heads / FiLM / losses omitted)' % rs)

    def step():
      out = tower(img, True)
      loss = out.mean()
      torch.autograd.grad(loss, params)
      return float(loss.detach())

  for _ in range(warmup):
    step()
  t0 = time.perf_counter()
  for _ in range(steps):
    step()
  dt = time.perf_counter() - t0
  return batch * steps / dt, threads, dt / steps, what


def metric_and_unit(config):
  if config == 'c4':
    return 'bcz_train_samples_per_sec', 'samples/s'
  if config == 'c5':
    return 'grasp2vec_train_triplets_per_sec', 'samples/s'
  return METRIC, 'transitions/s'


def run_reference(args):
  rank = int(os.environ.get('RANK', '0'))
  if rank != 0:
    return
  metric, unit = metric_and_unit(args.config)
  rate, threads, sec, what = cpu_reference_rate(args, args.steps, args.warmup)
  sample = '%d timed steps (+%d warm-up) of batch %d (a bounded sample of the per-GPU batch %d): %s; %.2f s/step' % (
      args.steps, args.warmup, args.cpu_batch, args.batch, what, sec)
  cfg = workload_config(args, args.gpus)
  cfg['reference_sample_batch'] = args.cpu_batch
  line = {
      'impl': 'reference', 'metric': metric, 'value': rate, 'unit': unit, 'n_gpus': args.gpus,
      'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': sec * 1e3, 'higher_is_better': True, 'scaling': 'weak',
      'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'config': cfg,
      'cpu_baseline': {'value': rate, 'unit': unit, 'cores': threads, 'kind': 'port', 'sample': sample},
      'e2e': {'value': rate, 'unit': unit, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
  }
  print(json.dumps(line))


# ---------------------------------------------------------------------------------------------
# the engine
# ---------------------------------------------------------------------------------------------
class Runtime(object):
  """Process-group / device bookkeeping shared by the config runners."""

  def __init__(self, args):
    import torch.distributed as dist
    self.dist = dist
    self.world = int(os.environ.get('WORLD_SIZE', '1'))
    self.rank = int(os.environ.get('RANK', '0'))
    self.local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if self.world != args.gpus and self.world == 1 and args.gpus > 1:
      raise SystemExit('launch with torchrun --nproc-per-node %d for --gpus %d' % (args.gpus, args.gpus))
    torch.cuda.set_device(self.local_rank)
    self.dev = torch.device('cuda', self.local_rank)
    if self.world > 1:
      dist.init_process_group('nccl', device_id=self.dev)

  def barrier(self):
    if self.world > 1:
      self.dist.barrier()
    torch.cuda.synchronize()

  def max_over_ranks(self, value):
    if self.world > 1:
      t = torch.tensor([value], device=self.dev, dtype=torch.float64)
      self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
      return float(t.item())
    return float(value)

  def close(self):
    if self.world > 1:
      self.dist.destroy_process_group()


def timed_steps(rt, fn, steps, warmup, profile=True, sample_clocks=False):
  """W untimed + K timed calls of fn(i), bracketed by barrier + synchronize; CUDA events on the launching stream,
  max over ranks.  Returns (ms per step, last result, conv profile entries, kernel launches, clocks)."""
  from tensor2robot_b200 import _lib, nn
  out = None
  for i in range(warmup):
    out = fn(i)
  rt.barrier()
  sampler = ClockSampler(rt.local_rank) if (sample_clocks and rt.rank == 0) else None
  if sampler:
    sampler.start()
  nn.PROFILE = [] if profile else None
  launches0 = _lib.launch_count()
  ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  ev0.record()
  for i in range(steps):
    out = fn(warmup + i)
  ev1.record()
  rt.barrier()
  launches = _lib.launch_count() - launches0
  prof, nn.PROFILE = (nn.PROFILE or []), None
  clocks = sampler.stop() if sampler else None
  return rt.max_over_ranks(ev0.elapsed_time(ev1)) / steps, out, prof, int(launches), clocks


def dump_outputs(args, rt, loss, vs):
  """--dump-outputs: the loss the last timed step returned and the variables it left behind (trainable, then moving
  statistics), as float32 .npy files.  Equal arguments give equal inputs, so two builds can be compared file by file.
  Larger arrays keep the elements at the same RandomState(0) sample of indices in every run."""
  if not args.dump_outputs or rt.rank != 0:
    return
  os.makedirs(args.dump_outputs, exist_ok=True)
  for name, t in (('loss', loss), ('trainable_variables', vs.flat), ('moving_statistics', vs.state_flat)):
    a = t.detach().float().cpu().numpy()
    if a.size > DUMP_MAX_ELEMENTS:
      a = a.reshape(-1)[np.sort(np.random.RandomState(0).choice(a.size, DUMP_MAX_ELEMENTS, replace=False))]
    np.save(os.path.join(args.dump_outputs, name + '.npy'), a)


def conv_roofline(prof, elapsed_ms_total, steps, rank):
  by_kind, by_shape = {}, {}
  peaks = measured_peaks()
  bound_ms = {'tensor': 0.0, 'hbm': 0.0}     # per-launch roofline time, split by which roof binds that launch
  spent_ms = {'tensor': 0.0, 'hbm': 0.0}
  for tag, flops, e0, e1, nbytes in prof:
    ms = e0.elapsed_time(e1)
    t_tensor, t_hbm = flops / (peaks['tflops'] * 1e9), nbytes / (peaks['hbm_gbs'] * 1e6)
    roof = 'hbm' if t_hbm > t_tensor else 'tensor'
    bound_ms[roof] += max(t_tensor, t_hbm)
    spent_ms[roof] += ms
    for table, key in ((by_kind, tag.split('|')[0]), (by_shape, tag)):
      d = table.setdefault(key, [0.0, 0.0, 0])
      d[0] += flops
      d[1] += ms
      d[2] += 1
  if os.environ.get('T2R_BENCH_DETAIL') and rank == 0:
    for key, v in sorted(by_shape.items(), key=lambda kv: -kv[1][1]):
      sys.stderr.write('%-48s n=%3d  %8.3f ms/step  %7.1f TFLOP/s\n' % (
          key, v[2] // steps, v[1] / steps, v[0] / max(v[1], 1e-9) / 1e9))
  conv_ms = sum(v[1] for v in by_kind.values())
  conv_flops = sum(v[0] for v in by_kind.values())
  dominant = max(by_kind.items(), key=lambda kv: kv[1][1])[0] if by_kind else None
  kinds = {k: {'launches': v[2], 'ms': v[1], 'tflops': v[0] / max(v[1], 1e-9) / 1e9} for k, v in by_kind.items()}
  achieved = conv_flops / max(conv_ms, 1e-9) / 1e9
  traffic = dominant_kernel_traffic()
  return {
      'bound': 'tensor',
      'kernel': 'conv_igemm_kernel / conv_igemm_tma_kernel / conv_halo_kernel / conv_wgrad_kernel (tcgen05 implicit GEMM)',
      'achieved': achieved, 'peak': peaks['tflops'], 'unit': 'TFLOP/s', 'frac': achieved / peaks['tflops'],
      'peak_source': peaks['source'] + ' sustained cuBLAS bf16 (kernels timed inside a long step)',
      'traffic': traffic['dram_bytes_per_launch'] if traffic else None,
      'traffic_kernel': (traffic or {}).get('kernel'), 'traffic_algorithmic_bytes': (traffic or {}).get('algorithmic_bytes'),
      'dominant': dominant, 'by_kind': kinds,
      # every launch against ITS OWN roof (max of flops / sustained tensor peak and in + out bytes / copy peak): the
      # layer-1 / layer-2 1x1 convolutions are HBM-bound, so 'frac' above (all flops / tensor peak) understates them
      'per_launch_roofline': {
          'frac': (bound_ms['tensor'] + bound_ms['hbm']) / max(conv_ms, 1e-9),
          'tensor_bound': {'ms_per_step': spent_ms['tensor'] / max(steps, 1),
                           'frac': bound_ms['tensor'] / max(spent_ms['tensor'], 1e-9)},
          'hbm_bound': {'ms_per_step': spent_ms['hbm'] / max(steps, 1), 'frac': bound_ms['hbm'] / max(spent_ms['hbm'], 1e-9),
                        'bytes': 'input + output once (bf16); residual / weight reads not counted', 'peak_gbs': peaks['hbm_gbs']}},
      'share_of_step': conv_ms / max(elapsed_ms_total, 1e-9),
      'algorithmic_tflop_per_step': conv_flops / max(steps, 1) / 1e12,
  }


def make_critic(model):
  from tensor2robot_b200.research.qtopt import networks, resnet_critic
  return resnet_critic.ResNet50QCritic() if model == 'resnet50' else \
      networks.Grasping44E2EOpenCloseTerminateGripperStatusHeightToBottom()


def make_engine_step(args, rt, model, bellman):
  from tensor2robot_b200 import engine
  from tensor2robot_b200.models import optimizers
  # research/qtopt/optimizer_builder.py defaults: momentum 0.9, staircase decay, EMA 0.9999
  lr = optimizers.create_exp_decaying_learning_rate(1e-4, int(3e6 / 32 * 2), 0.999, True)
  opt = optimizers.MovingAverageOptimizer(optimizers.MomentumOptimizer(lr, 0.9), 0.9999)
  kwargs = dict(device=rt.dev, seed=0, world_size=rt.world, rank=rt.rank)
  if bellman:
    return engine.BellmanCriticTrainStep(make_critic(model), opt, gamma=0.9, cem_samples=64, cem_iters=2, num_elites=10,
                                         target_update_every=100,
                                         cem_chunk=args.cem_chunk if model == 'resnet50' else None, **kwargs)
  return engine.CriticTrainStep(make_critic(model), opt, **kwargs)


def device_replay(rt, b, n_sets, with_next):
  g = torch.Generator(device=rt.dev)
  g.manual_seed(1234 + rt.rank)
  sets = []
  for _ in range(n_sets):
    s = [torch.randint(0, 256, (b, 512, 640, 3), dtype=torch.uint8, device=rt.dev, generator=g),
         torch.rand((b, 10), device=rt.dev, generator=g) * 2 - 1,
         (torch.rand((b, 1), device=rt.dev, generator=g) < 0.3).float()]
    if with_next:
      s += [torch.randint(0, 256, (b, 512, 640, 3), dtype=torch.uint8, device=rt.dev, generator=g),
            (torch.rand((b, 1), device=rt.dev, generator=g) < 0.1).float()]
    sets.append(tuple(s))
  return sets


def allreduce_probe(rt, vs):
  """Isolated all-reduce of the flat gradient buffer (what the step overlaps with its backward pass)."""
  if rt.world <= 1:
    return None
  buf = torch.zeros_like(vs.flat_grad)
  for _ in range(2):
    rt.dist.all_reduce(buf)
  rt.barrier()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for _ in range(5):
    rt.dist.all_reduce(buf)
  e1.record()
  rt.barrier()
  ms = rt.max_over_ranks(e0.elapsed_time(e1)) / 5
  nbytes = buf.numel() * 4
  return {'isolated_ms': ms, 'bytes': nbytes, 'dtype': 'f32',
          'bus_gbs': 2.0 * (rt.world - 1) / rt.world * nbytes / max(ms, 1e-9) / 1e6,
          'in_step': 'bucketed (engine.GradientReducer), launched as each bucket completes during the backward pass'}


def write_replay_shards(directory, n_records, shards=8, seed=1234):
  """SURVEY 8(d) transition records: image_1 = JPEG (quality 90, 4:2:0) of a 512x640 box-filtered noise frame, the
  QT-Opt action floats and grasp_success, as tf.Examples in uncompressed TFRecord shards.  Returns the file pattern."""
  import concurrent.futures
  import io
  from PIL import Image
  from tensor2robot_b200.utils import example_proto as ep
  from tensor2robot_b200.utils import writer

  def make(i):
    rng = np.random.default_rng(seed=seed + i)
    noise = rng.integers(0, 256, (512 + 8, 640 + 8, 3)).astype(np.float32)
    c = np.cumsum(np.cumsum(noise, 0), 1)                       # 8x8 box filter through an integral image
    box = (c[8:, 8:] - c[:-8, 8:] - c[8:, :-8] + c[:-8, :-8]) / 64.0
    img = np.clip((box - 127.5) * 2.0 + 127.5, 0, 255).astype(np.uint8)
    buf = io.BytesIO()
    Image.fromarray(img).save(buf, format='JPEG', quality=90, subsampling=2)
    f = {'image_1': ep.bytes_feature([buf.getvalue()]), 'world_vector': ep.float_feature(rng.uniform(-1, 1, 3)),
         'vertical_rotation': ep.float_feature(rng.uniform(-1, 1, 2)),
         'grasp_success': ep.float_feature([float(rng.random() < 0.3)]),
         'height_to_bottom': ep.float_feature([rng.random()])}
    for k in ('close_gripper', 'open_gripper', 'terminate_episode', 'gripper_closed'):
      f[k] = ep.float_feature([float(rng.random() < 0.5)])
    return ep.Example(f)

  with concurrent.futures.ThreadPoolExecutor(max_workers=usable_host_threads()) as pool:
    examples = list(pool.map(make, range(n_records)))
  per = (n_records + shards - 1) // shards
  total_bytes = 0
  for s in range(shards):
    w = writer.TFRecordReplayWriter()
    w.open(os.path.join(directory, 'replay-%05d' % s))
    w.write(examples[s * per:(s + 1) * per])
    w.close()
    total_bytes += os.path.getsize(os.path.join(directory, 'replay-%05d.tfrecord' % s))
  return os.path.join(directory, 'replay-*.tfrecord'), total_bytes / max(n_records, 1)


# ---- end to end through train_eval_model (the B-1 boundary) ------------------------------------
def e2e_train_eval(rt, t2r_model, batch, steps, warmup, records=0):
  """The same metric through the reference's own entry point: host numpy batches -> input generator ->
  train_eval_model (pinned staging + H2D on a copy stream, preprocessor, T2RModel.train_step), the loss read back to
  the host after every step.  Returns (units/s over all ranks, H2D bytes per step, D2H bytes per step, ms/step)."""
  from tensor2robot_b200.hooks import hook_builder
  from tensor2robot_b200.input_generators import default_input_generator as gens
  from tensor2robot_b200.utils import tensorspec_utils, train_eval

  class CyclingGenerator(gens.GeneratorInputGenerator):
    """Two fixed host batches in turn (drawing 0.5 GB of fresh random numbers per step would time numpy)."""

    def _generator_fn(self, batch_size):
      def pinned(struct):
        """The batches live in page-locked host memory, as the contract's e2e leg asks (and as a reader that parses into
        pinned buffers provides): every step still pays the H2D copy of its 0.25-0.75 GB of frames."""
        flat = tensorspec_utils.flatten_spec_structure(struct)
        for k in list(flat.keys()):
          a = np.ascontiguousarray(flat[k])
          flat[k] = torch.from_numpy(a).pin_memory().numpy() if torch.cuda.is_available() and a.nbytes >= (1 << 20) else a
        return flat

      sets = [(pinned(tensorspec_utils.make_random_numpy(self._feature_spec, batch_size, self._sequence_length)),
               pinned(tensorspec_utils.make_random_numpy(self._label_spec, batch_size, self._sequence_length)))
              for _ in range(2)]
      self.h2d_bytes = sum(int(np.asarray(v).nbytes) for part in sets[0]
                           for v in tensorspec_utils.flatten_spec_structure(part).values())
      i = 0
      while True:
        yield sets[i % 2]
        i += 1

  class Timer(hook_builder.TrainHook):
    """Reads every step's loss back to the host inside the timed region.  The read is pipelined one step behind (the
    D2H copy of step n into pinned memory is enqueued after step n and resolved while step n + 1 is being launched), as a
    trainer that logs every step would do it; the last step's value is resolved before the clock stops."""

    def __init__(self):
      self.t0 = self.t1 = None
      self.losses = []
      self._slots = [torch.empty((), dtype=torch.float32).pin_memory() for _ in range(2)]
      self._pending = None

    def before_step(self, step):
      if step == warmup:
        rt.barrier()
        self.t0 = time.perf_counter()

    def _resolve(self):
      if self._pending is not None:
        buf, event = self._pending
        event.synchronize()
        self.losses.append(float(buf))
        self._pending = None

    def after_step(self, step, loss):
      buf = self._slots[step % 2]
      buf.copy_(loss.detach().reshape(()).float(), non_blocking=True)      # device -> host read of the step result
      event = torch.cuda.Event()
      event.record()
      self._resolve()                                                      # the previous step's value
      self._pending = (buf, event)
      if step == warmup + steps:
        self._resolve()
        rt.barrier()
        self.t1 = time.perf_counter()

  class Builder(hook_builder.HookBuilder):

    def __init__(self, hook):
      self.hook = hook

    def create_hooks(self, t2r_model, model_dir):
      return [self.hook]

  timer = Timer()
  with tempfile.TemporaryDirectory() as model_dir:
    if records:
      # the reference's record path (utils/tfdata.py:629-689 + default_input_generator.py:77-101): every rank reads its
      # own shards; the JPEG bytes are what crosses PCIe (as Huffman-decoded coefficients)
      from tensor2robot_b200.utils import tfdata
      tfdata.set_image_decoder('device')
      pattern, record_bytes = write_replay_shards(model_dir, records, seed=1234 + 100000 * rt.rank)
      gen = gens.DefaultRecordInputGenerator(file_patterns=pattern, batch_size=batch)
      gen.h2d_bytes = int(batch * (512 * 640 * 1.5 * 2 + 44))      # int16 coefficients of 4:2:0 frames + the floats
      gen.record_bytes = record_bytes
    else:
      gen = CyclingGenerator(batch_size=batch)
    train_eval.train_eval_model(t2r_model=t2r_model, input_generator_train=gen, max_train_steps=warmup + steps,
                                model_dir=os.path.join(model_dir, 'model'), train_hook_builders=[Builder(timer)],
                                device=rt.dev, log_every_n_steps=10**9)
  seconds = rt.max_over_ranks(timer.t1 - timer.t0)
  return batch * rt.world * steps / seconds, gen.h2d_bytes, 4, seconds / steps * 1e3


# ---- C2 / C3 -----------------------------------------------------------------------------------
def run_critic(args, rt):
  from tensor2robot_b200.research.qtopt import t2r_models
  b, bellman = args.batch, args.config == 'c3'
  step = make_engine_step(args, rt, args.model, bellman)
  sets = device_replay(rt, b, 2, bellman)
  step.build(*sets[0][:2])
  ms, loss, prof, launches, clocks = timed_steps(rt, lambda i: step.step(*sets[i % 2]), args.steps, args.warmup,
                                                 sample_clocks=True)
  dump_outputs(args, rt, loss, step.vs)
  loss_value = float(loss)
  roofline = conv_roofline(prof, ms * args.steps, args.steps, rt.rank)
  value = b * rt.world * 1000.0 / ms
  extra = {'loss': loss_value, 'peak_mem_gb': torch.cuda.max_memory_allocated(rt.dev) / 1e9,
           'allreduce': allreduce_probe(rt, step.vs)}
  unit_gflop = TRAIN_GFLOP[args.model]

  if bellman:
    # the target computation alone (BASELINE metric "CEM Q-evals/sec"): tower once + 2 x [B*64] post-merge passes
    def target_only(i):
      s = sets[i % 2]
      x_next = step.preprocess(s[3], training=False)
      _, max_q, _ = step.cem.maximize(x_next)
      return step.cem.bellman_target(s[2].reshape(-1), s[4].reshape(-1), max_q, 0.9)
    cem_ms, target, cem_prof, _, _ = timed_steps(rt, target_only, max(2, min(args.steps, 4)), 1)
    cem_roof = conv_roofline(cem_prof, 1.0, 1, -1)
    unit_gflop += STATE_TOWER_GFLOP[args.model] + 128 * CEM_GFLOP_PER_QEVAL[args.model]
    extra['cem'] = {'q_evals_per_sec': b * rt.world * 128 * 1000.0 / cem_ms, 'ms': cem_ms, 'samples': 64, 'iterations': 2,
                    'elites': 10, 'per_gpu_batch': b, 'chunk': args.cem_chunk if args.model == 'resnet50' else b,
                    'conv_tflops': cem_roof['achieved'], 'conv_frac_of_peak': cem_roof['frac'],
                    'target_mean': float(target.mean())}

  # ---- end to end ----
  e2e = None
  if not args.no_e2e:
    if bellman:
      host = [tuple(t.cpu().pin_memory() for t in s) for s in sets]
      h2d = sum(t.numel() * t.element_size() for t in host[0])
      slots = [tuple(torch.empty_like(t, device=rt.dev) for t in host[0]) for _ in range(2)]
      copy_stream = torch.cuda.Stream(device=rt.dev)

      def stage(i):   # H2D of batch i on the copy stream, overlapping the previous step's compute
        with torch.cuda.stream(copy_stream):
          for dst, src in zip(slots[i % 2], host[i % 2]):
            dst.copy_(src, non_blocking=True)
          done = torch.cuda.Event()
          done.record(copy_stream)
        return done

      def loop(n):
        ready = stage(0)
        for i in range(n):
          torch.cuda.current_stream().wait_event(ready)
          if i + 1 < n:
            ready = stage(i + 1)
          step.step(*slots[i % 2]).to('cpu')          # device -> host read of the step result

      loop(max(2, args.warmup))
      rt.barrier()
      t0 = time.perf_counter()
      loop(args.steps)
      rt.barrier()
      sec = rt.max_over_ranks(time.perf_counter() - t0)
      e2e = {'value': b * rt.world * args.steps / sec, 'unit': 'transitions/s', 'h2d_bytes_per_step': h2d,
             'd2h_bytes_per_step': 4, 'ms_per_step': sec / args.steps * 1e3,
             'api': 'engine.BellmanCriticTrainStep.step on pinned host batches (state + next-state frames)'}
    else:
      del step, sets   # free the engine-level replica before the T2R model builds its own
      torch.cuda.empty_cache()
      cls = t2r_models.ResNet50QCriticModel if args.model == 'resnet50' else \
          t2r_models.Grasping44E2EOpenCloseTerminateGripperStatusHeightToBottom
      records = args.records if args.data == 'records' else 0
      rate, h2d, d2h, e_ms = e2e_train_eval(rt, cls(device=rt.dev), b, args.steps, max(2, args.warmup), records)
      e2e = {'value': rate, 'unit': 'transitions/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
             'ms_per_step': e_ms, 'api': 'utils.train_eval.train_eval_model + research.qtopt.t2r_models.%s' % cls.__name__,
             'input': ('TFRecord shards of JPEG transitions: read + CRC-32C + tf.Example parse + split JPEG decode '
                       '(Huffman on %d host threads, IDCT / upsampling / colour on the GPU)' % usable_host_threads())
                      if records else 'host numpy batches in pinned memory (decoded uint8 frames)',
             'host_threads': usable_host_threads()}

  # ---- side measurements of the default run: the reference's own critic and CEM on it ----
  if args.config == 'c2' and args.model == 'resnet50' and not args.no_extras:
    torch.cuda.empty_cache()
    g44 = make_engine_step(args, rt, 'grasping44', True)
    gsets = device_replay(rt, b, 2, True)
    g44.build(*gsets[0][:2])
    g_ms, _, g_prof, _, _ = timed_steps(rt, lambda i: g44.step(*gsets[i % 2][:3]), max(3, min(args.steps, 8)), 3)
    g_roof = conv_roofline(g_prof, g_ms, 1, -1)
    c_ms, _, _, _, _ = timed_steps(rt, lambda i: g44.step(*gsets[i % 2]), max(2, min(args.steps, 4)), 2, profile=False)
    extra['grasping44'] = {
        'note': 'the reference QT-Opt critic (research/qtopt/networks.py:343-615), same batch / frames / optimizer',
        'c2_transitions_per_sec': b * rt.world * 1000.0 / g_ms, 'c2_ms_per_step': g_ms,
        'c2_conv_tflops': g_roof['achieved'], 'c2_conv_frac_of_peak': g_roof['frac'],
        'c2_model_tflops': b * rt.world * 1000.0 / g_ms * TRAIN_GFLOP['grasping44'] / 1e3,
        'c3_transitions_per_sec': b * rt.world * 1000.0 / c_ms, 'c3_ms_per_step': c_ms,
        'c3_q_evals_per_sec_in_step': b * rt.world * 128 * 1000.0 / max(c_ms - g_ms, 1e-6)}
    del g44, gsets
  extra['model_tflops'] = value * unit_gflop / 1e3
  return ms, value, roofline, launches, clocks, e2e, extra


# ---- C4 / C5 -----------------------------------------------------------------------------------
def make_t2r_model(args, rt):
  if args.config == 'c4':
    from tensor2robot_b200.research.bcz import model as bcz
    # run_train_bc_langcond_trajectory.gin: ResNet-18 + FiLM on a 512-d sentence embedding, crop 450 -> 200, 10 waypoints
    pre = lambda **kw: bcz.BCZPreprocessor(image_size=(200, 200), crop_size=(450, 450), input_size=(512, 640), **kw)
    return bcz.BCZModel(image_size=(200, 200), input_size=(512, 640), resnet_size=18, num_waypoints=10,
                        cond_modality=bcz.ConditionMode.LANGUAGE_EMBEDDING, preprocessor_cls=pre, device=rt.dev)
  from tensor2robot_b200.research.grasp2vec import grasp2vec_model
  # BASELINE C5 geometry: 224x224 crops of the 512x640 frames (the reference crops 472x472)
  crop = (0, 288, 224, 0, 416, 224)
  pre = lambda **kw: grasp2vec_model.Grasp2VecPreprocessor(scene_crop=crop, goal_crop=crop, **kw)
  return grasp2vec_model.Grasp2VecModel(scene_size=(224, 224), goal_size=(224, 224), preprocessor_cls=pre, device=rt.dev)


def run_t2r(args, rt):
  from tensor2robot_b200.utils import tensorspec_utils
  model = make_t2r_model(args, rt)
  pre = model.preprocessor
  def device_batch():
    def to_dev(spec):
      host = tensorspec_utils.make_random_numpy(spec, args.batch)
      flat = tensorspec_utils.flatten_spec_structure(host)
      return tensorspec_utils.TensorSpecStruct([(k, torch.from_numpy(np.ascontiguousarray(v)).to(rt.dev)) for k, v in flat.items()])
    return to_dev(pre.get_in_feature_specification('train')), to_dev(pre.get_in_label_specification('train'))

  sets = [device_batch() for _ in range(2)]

  def clone(struct):
    return tensorspec_utils.TensorSpecStruct([(k, v) for k, v in tensorspec_utils.flatten_spec_structure(struct).items()])

  def one(i):
    f, l = sets[i % 2]
    features, labels = pre.preprocess(clone(f), clone(l) if len(l) else None, 'train')
    return model.train_step(features, labels)

  ms, loss, prof, launches, clocks = timed_steps(rt, one, args.steps, args.warmup, sample_clocks=True)
  dump_outputs(args, rt, loss, model.variable_store)
  roofline = conv_roofline(prof, ms * args.steps, args.steps, rt.rank)
  value = args.batch * rt.world * 1000.0 / ms
  extra = {'loss': float(loss), 'peak_mem_gb': torch.cuda.max_memory_allocated(rt.dev) / 1e9,
           'model_tflops': roofline['algorithmic_tflop_per_step'] * 1000.0 / ms,
           'allreduce': allreduce_probe(rt, model.variable_store)}
  e2e = None
  if not args.no_e2e:
    del sets
    torch.cuda.empty_cache()
    fresh = make_t2r_model(args, rt)
    rate, h2d, d2h, e_ms = e2e_train_eval(rt, fresh, args.batch, args.steps, max(2, args.warmup))
    e2e = {'value': rate, 'unit': 'samples/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h, 'ms_per_step': e_ms,
           'api': 'utils.train_eval.train_eval_model + %s' % type(fresh).__name__}
  return ms, value, roofline, launches, clocks, e2e, extra


def run_b200(args):
  from tensor2robot_b200.preprocessors import image_transformations
  # the c4 / c5 batches and the e2e host batches come from make_random_numpy (global NumPy RNG), the training crops
  # and photometric draws from image_transformations: seeded (per rank) so that equal arguments give equal inputs in
  # every run
  rank = int(os.environ.get('RANK', '0'))
  np.random.seed(rank)
  image_transformations.seed(rank)
  rt = Runtime(args)
  if args.config in ('c2', 'c3'):
    ms, value, roofline, launches, clocks, e2e, extra = run_critic(args, rt)
  else:
    ms, value, roofline, launches, clocks, e2e, extra = run_t2r(args, rt)
  (metric, unit), dtype = metric_and_unit(args.config), 'bf16'
  if rt.rank != 0:
    rt.close()
    return
  cpu = None
  if rt.world == 1 and not args.no_cpu_baseline:
    rate, threads, sec, what = cpu_reference_rate(args, 2, 1)
    cpu = {'value': rate, 'unit': unit, 'cores': threads, 'kind': 'port',
           'sample': '2 timed steps (+1 warm-up) of batch %d: %s; %.1f s/step' % (args.cpu_batch, what, sec)}
  line = {
      'metric': metric, 'value': value, 'unit': unit, 'n_gpus': rt.world, 'steps': args.steps,
      'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak',
      'vs_baseline': None, 'dtype': dtype, 'data': 'synthetic',
      'config': workload_config(args, rt.world), 'clocks': clocks, 'gpu_launches': launches,
      'roofline': roofline, 'cpu_baseline': cpu, 'e2e': e2e,
  }
  line.update(extra)
  print(json.dumps(line))
  rt.close()


def main():
  args = parse_args()
  if args.impl == 'reference':
    run_reference(args)
  else:
    run_b200(args)


if __name__ == '__main__':
  main()
