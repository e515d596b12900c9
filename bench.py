#!/usr/bin/env python
"""Benchmark of the TwinGAN G+D step (BASELINE.json metric: images/sec at 256x256, batch 16 per GPU).

  python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K --warmup W   # CPU restatement of the reference (oracle port)

One "step" = everything a reference session.run(train_tensor) computes (16 network passes + 2 DRAGAN passes,
generator-set and discriminator-set gradients) plus BOTH Adam applies (SURVEY 8d, "mode B").
`value` = (source,target) pairs per second over all ranks with inputs resident in HBM; `e2e` = the same through
the public API (GanModel.train_step) with pinned-host inputs copied H2D and the losses read back D2H every step.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)

import torch  # noqa: E402

HW = 256
BATCH = 16
MAXC = 256
NORM = 'instance_norm'     # north_star: "per-domain AdaIN"
METRIC = 'images/sec G+D step @256x256 bs=16'
UNIT = 'pairs/s'           # one (source,target) image pair per unit; 2 real images touched per pair


def _peaks():
  p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(p):
    try:
      d = json.load(open(p))
      return {'hbm_gbs': float(d['hbm_gbs']), 'tf': float(d.get('bf16_tflops_sustained') or d['bf16_tflops']),
              'which': 'measured'}
    except (OSError, ValueError, KeyError, TypeError):
      pass
  return {'hbm_gbs': 6650.0, 'tf': 1400.0, 'which': 'fallback'}


class ClockSampler(threading.Thread):
  """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

  def __init__(self, index=0):
    super().__init__(daemon=True)
    self.index = index
    self.samples = []
    self.stop_flag = False

  def run(self):
    q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')
    while not self.stop_flag:
      try:
        out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q, '--format=csv,noheader,nounits'],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        if out:
          self.samples.append([s.strip() for s in out.split(',')])
      except Exception:
        pass
      time.sleep(0.2)

  def summary(self):
    sm = sorted(float(s[0]) for s in self.samples if s and s[0].replace('.', '').isdigit())
    if not sm:
      return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': []}
    names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
    reasons = [n for i, n in enumerate(names) if any(len(s) > 3 + i and s[3 + i].lower().startswith('active') for s in self.samples)]
    return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': float(self.samples[0][1]), 'reasons': reasons,
            'samples': len(sm)}


def model_state(model):
  """Everything a training step reads and updates: parameters, Adam slots, normaliser state, step counters."""
  v = model.variables
  return ([t.clone() for t in (v.flat, v.adam_m, v.adam_v, v.state, v.state_snapshot, model._counters)],
          (v.adam_t, model.flags.global_step, model._counters_mirror))


def restore_model_state(model, saved):
  v = model.variables
  with torch.no_grad():
    for dst, src in zip((v.flat, v.adam_m, v.adam_v, v.state, v.state_snapshot, model._counters), saved[0]):
      dst.copy_(src)
  v.adam_t, model.flags.global_step, model._counters_mirror = saved[1]
  if v.weight_table is not None:
    v.weight_table.dirty = True      # the step rebuilds the weight planes from the restored parameters


def step_outputs(model, losses):
  """What one training step hands its caller, as float32 host arrays: the two returned losses and the step's named
  losses (GanModel.last_losses)."""
  out = {'generator_loss': losses[0], 'discriminator_loss': losses[1]}
  out.update({'loss_' + k: t for k, t in model.last_losses.items() if k not in out})
  return {k: t.detach().to('cpu', torch.float32).reshape(-1).numpy() for k, t in out.items()}


def bench_cuda(args):
  import torch.distributed as dist
  from twingan_b200 import ops, twingan, flops
  from twingan_b200._lib import lib
  world = int(os.environ.get('WORLD_SIZE', '1'))
  rank = int(os.environ.get('RANK', '0'))
  local = int(os.environ.get('LOCAL_RANK', '0'))
  torch.cuda.set_device(local)
  dev = torch.device('cuda', local)
  pg = None
  if world > 1:
    dist.init_process_group('nccl', device_id=dev)
    pg = dist.group.WORLD
  hw, batch = args.hw, args.batch
  flags = twingan.Flags(train_image_size=hw, pggan_max_num_channels=args.max_channels, generator_norm_type=args.norm,
                        num_clones=world, batch_passes=not args.pass_by_pass)
  model = twingan.GanModel(flags, device=dev, seed=1234, process_group=pg)
  gen = torch.Generator(device=dev).manual_seed(100 + rank)
  n_sets = 2
  dev_inputs = []
  host_inputs = []
  for i in range(n_sets):
    s = torch.rand((batch, hw, hw, 3), device=dev, generator=gen)
    t = torch.rand((batch, hw, hw, 3), device=dev, generator=gen)
    r = twingan.make_dragan_rand(batch, hw, dev, gen)
    dev_inputs.append((s, t, r))
    host_inputs.append((s.cpu().pin_memory(), t.cpu().pin_memory(), {k: v.cpu().pin_memory() for k, v in r.items()}))
  h2d_bytes = sum(x.numel() * 4 for x in (host_inputs[0][0], host_inputs[0][1])) + \
      sum(v.numel() * 4 for v in host_inputs[0][2].values())

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  for kv in args.set_option:
    from twingan_b200._lib import lib as _twg_lib
    key, value = kv.split('=')
    _twg_lib().call('twg_set_option', int(key), int(value))
  ddp_check = None
  if world > 1 and not args.no_ddp_check:
    # pre-flight: N NCCL ranks == N sequential micro-batches through the product, parameters identical across ranks
    from twingan_b200 import ddp
    ddp_check = ddp.selfcheck(dev, pg)
  # --dump-outputs: the last timed step starts again from the seeded initial state.  Steps are reproducible only to fp32
  # rounding (atomics order in split-K / wgrad reductions) and training amplifies that from step to step, so without the
  # reset what the last step computes would differ from run to run.  The reset is one copy inside the timed window.
  initial_state = model_state(model) if args.dump_outputs else None
  use_graph = not args.no_graph
  if use_graph:
    model.capture(*dev_inputs[0])
  train_step = model.train_step_graphed if use_graph else model.train_step

  def step_resident(i):
    s, t, r = dev_inputs[i % n_sets]
    return train_step(s, t, r)

  # End to end through the public feeding path (twingan_b200.prefetch.DevicePrefetcher, the runner's loader): every step's
  # batch is copied from pinned host memory inside the timed region -- on a side stream, one batch ahead, so the copy of
  # batch k+1 overlaps step k -- and every step's losses are read back to the host before the next step is issued.
  from twingan_b200.prefetch import DevicePrefetcher

  def host_batches():
    i = 0
    while True:
      yield host_inputs[i % n_sets]
      i += 1
  feed = DevicePrefetcher(host_batches(), dev)

  def step_e2e(i):
    s, t, r = next(feed)
    gl, dl = train_step(s, t, r)
    feed.release()
    return torch.stack([gl.reshape(()), dl.reshape(())]).cpu()     # D2H read of the step's result

  for i in range(args.warmup):
    step_resident(i)
  barrier()
  sampler = ClockSampler(local) if rank == 0 else None
  if sampler:
    sampler.start()
  L = lib()
  launches0 = L.launch_count()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for i in range(args.steps):
    if initial_state is not None and i == args.steps - 1:
      restore_model_state(model, initial_state)
    last = step_resident(i)
  e1.record()
  barrier()
  # copied now: the legs below run further steps on the same model
  dumped = step_outputs(model, last) if args.dump_outputs and rank == 0 else None
  launches = (L.launch_count() - launches0) if not use_graph else model.launches_per_step * args.steps
  ms = e0.elapsed_time(e1)
  # e2e leg
  step_e2e(0)
  barrier()
  e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  t_wall0 = time.perf_counter()
  e2.record()
  for i in range(args.steps):
    step_e2e(i)
  e3.record()
  barrier()
  wall_e2e = (time.perf_counter() - t_wall0) * 1e3
  ms_e2e = max(e2.elapsed_time(e3), wall_e2e)
  if sampler:
    sampler.stop_flag = True
  # roofline pass: one more step with per-launch CUDA events around every conv-family kernel
  ops.enable_conv_timing(True)
  model.train_step(*dev_inputs[0])     # eager (per-launch events cannot be recorded inside a graph replay)
  torch.cuda.synchronize()
  conv_stats = ops.collect_conv_timing()
  ops.enable_conv_timing(False)
  t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
  if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
  ms, ms_e2e = t.tolist()
  if rank == 0:
    peaks = _peaks()
    per_step = ms / args.steps
    value = batch * world / (per_step * 1e-3)
    e2e_value = batch * world / (ms_e2e / args.steps * 1e-3)
    fl = flops.step_flops_per_pair(hw, False, args.max_channels)
    step_flop = fl['total'] * batch
    mixed = flops.mixed_roofline_seconds(hw, batch, peaks['tf'] * 1e12, peaks['hbm_gbs'] * 1e9,
                                         max_num_channels=args.max_channels)
    # Per-family detail comes from one eager pass with CUDA events around every conv launch; events serialise the launches
    # and add their own latency, so the family times sum to MORE than the graph-replayed step -- use them as shares.
    KERNELS = {'tc_tap': 'k_conv_htap_tc<BN> (persistent wide-layer halo kernel) + k_conv_fwd_tc<CC,BN> (tap-per-TMA, hw < 16): '
                         'fwd+dgrad of the wide layers',
               'tc_halo': 'k_conv_halo_tc<CIN,BN,SUB> (halo-tile persistent implicit GEMM, fwd+dgrad of the 16-64-channel layers)',
               'tc_wgrad': 'k_conv_wgrad_rows<CN,BNW> (row-shift, narrow layers) + k_conv_wgrad_halo<CN,BNW> (W >= 16) + '
                           'k_conv_wgrad_tc2<CN,BNW> (4x4 / 8x8): weight gradients',
               'fp32_cuda_core': 'k_conv_*_simt (exact fp32 CUDA-core convs: 4x4 VALID head, FC, non-tensor-core shapes)',
               'tc_ws': 'k_pw_* (fromRGB / toRGB 1x1 convs, exact fp32)'}
    families = {}
    for k in ('tc_tap', 'tc_wgrad', 'tc_halo', 'tc_ws', 'fp32_cuda_core'):
      v = conv_stats.get(k)
      if v:
        families[k] = {'kernel': KERNELS[k], 'launches_per_step': v['launches'], 'ms_eager_events': v['ms'],
                       'algorithmic_tflops': v['tflops'], 'frac_of_bf16_peak': round(v['tflops'] / peaks['tf'], 5),
                       'algorithmic_gbs': v.get('algorithmic_gbs'),
                       'frac_of_measured_hbm': round(v.get('algorithmic_gbs', 0.0) / peaks['hbm_gbs'], 4)}
    conv_ms = sum(v['ms'] for v in conv_stats.values())
    conv_fl = sum(v['flops'] for v in conv_stats.values())
    step_tf = step_flop / (per_step * 1e-3) / 1e12
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, 'profiles', 'r02_ncu_traffic.json')
    if os.path.exists(tpath):
      try:
        tj = json.load(open(tpath))
        traffic, traffic_src = tj.get('dominant_kernel_dram_bytes_per_launch'), tj
      except (OSError, ValueError):
        pass
    out = {
        'metric': METRIC, 'value': round(value, 3), 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': round(per_step, 3), 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32 (conv MACs as split-bf16 x3 on tcgen05, fp32 accumulate)',
        'data': 'synthetic',
        'config': {'workload': 'configs[3]: %dx%d full TwinGAN G+D step (mode B: 16 passes + 2 DRAGAN, both gradient '
                               'sets, both Adam applies), batch %d/GPU, %s, pixel-norm, UNet, DRAGAN' % (hw, hw, batch, args.norm),
                   'global_batch': batch * world, 'parallelism': 'dp%d' % world,
                   'l2': 'activation working set >> L2 (GBs per step); two alternating input sets',
                   'conv_precision': 'tcgen05 split-bf16' if ops.get_precision() else 'fp32 CUDA cores',
                   'pass_structure': 'pass-by-pass (16 separate passes)' if args.pass_by_pass else
                                     'weight-sharing passes batched: E 2x16, G 4x16, E 2x16, D 3x16 per domain, DRAGAN 16+16',
                   'images_per_pair': 2, 'cuda_graph': use_graph},
        'e2e': {'value': round(e2e_value, 3), 'unit': UNIT, 'h2d_bytes_per_step': h2d_bytes, 'd2h_bytes_per_step': 8},
        'gpu_launches': int(launches),
        'clocks': sampler.summary() if sampler else None,
        # Step-level roofline (stable from run to run; the per-family table below is detail): algorithmic conv FLOPs of the
        # whole G+D step over the step time, against the measured dense bf16 peak.
        'roofline': {
            'bound': 'tensor', 'achieved': round(step_tf, 3), 'peak': peaks['tf'], 'unit': 'TFLOP/s',
            'frac': round(step_tf / peaks['tf'], 5), 'traffic': traffic,
            'kernel': 'whole G+D step: %.3f TFLOP of algorithmic conv MACs (12 F_E + 12 F_G + 34 F_D per pair) in %.2f ms, %d '
                      'launches' % (step_flop / 1e12, per_step, int(launches) // max(args.steps, 1)),
            'ceiling': 'split-bf16 forms 3 partial products per MAC, so a tensor-bound layer caps at 0.333 of the bf16 peak; '
                       'every hw >= 64 layer is HBM-bound (SURVEY 8a.1), hence step_mixed_frac',
            'peak_source': peaks['which'] + ' bf16 sustained (MEASURED_PEAKS.json)',
            'step_tc_frac': round(step_tf / peaks['tf'], 5),
            'step_mixed_frac': round(mixed['step'] / (per_step * 1e-3), 5),
            'step_mixed_bound_ms': round(mixed['step'] * 1e3, 3),
            'step_algorithmic_tflop': round(step_flop / 1e12, 4),
            'conv_family_tflops': round(conv_fl / max(conv_ms, 1e-9) / 1e9, 3), 'conv_family_ms_eager_events': round(conv_ms, 3),
            'families': families,
            'traffic_source': traffic_src,
        },
    }
    if ddp_check is not None:
      out['ddp_check'] = ddp_check
    if world == 1 and not args.no_secondary:
      try:
        out['secondary'] = {'infer': infer_measure(args, dev)}
      except Exception as e:   # noqa: BLE001 -- the headline line must survive a failure of the secondary workload
        out['secondary'] = {'infer': {'error': repr(e)}}
    if not args.no_cpu_baseline and world == 1:
      out['cpu_baseline'] = cpu_baseline_subprocess(args)
    if dumped is not None:
      import numpy as np
      os.makedirs(args.dump_outputs, exist_ok=True)
      for k, a in dumped.items():
        np.save(os.path.join(args.dump_outputs, k + '.npy'), a)
      out['dumped_outputs'] = {'dir': args.dump_outputs, 'arrays': len(dumped),
                               'bytes': sum(a.nbytes for a in dumped.values())}
    print(json.dumps(out), flush=True)
  if world > 1:
    dist.destroy_process_group()


def infer_measure(args, dev, steps=None):
  """BASELINE configs[4]: the inference wrapper (inference/image_translation_infer.py:46-99), E(x; '_s', eval) ->
  G(.; '_t', eval, UNet skips), 64 images at 256x256, eval-mode batch-renorm with moving statistics."""
  from twingan_b200 import flops, twingan
  from twingan_b200._lib import lib
  steps = steps or args.steps
  batch = 64
  model = twingan.GanModel(twingan.Flags(train_image_size=args.hw, pggan_max_num_channels=args.max_channels,
                                         generator_norm_type='batch_renorm'), device=dev)
  gen = torch.Generator(device=dev).manual_seed(7)
  v = model.variables
  with torch.no_grad():
    for key, (o, C) in v.state_offsets.items():
      v.state[o:o + C] = 0.1 * torch.randn(C, device=dev, generator=gen)
      v.state[o + C:o + 2 * C] = 0.5 + torch.rand(C, device=dev, generator=gen)
  xs = [torch.rand((batch, args.hw, args.hw, 3), device=dev, generator=gen) for _ in range(2)]
  hx = [x.cpu().pin_memory() for x in xs]
  hout = torch.empty((batch, args.hw, args.hw, 3), dtype=torch.float32).pin_memory()
  for i in range(max(args.warmup, 3)):
    model.infer(xs[i % 2])
  torch.cuda.synchronize()
  L = lib()
  n0 = L.launch_count()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for i in range(steps):
    model.infer(xs[i % 2])
  e1.record()
  torch.cuda.synchronize()
  launches = L.launch_count() - n0
  ms = e0.elapsed_time(e1) / steps
  # end to end through the public pipelined call (twingan.infer_batches): every batch comes from pinned host memory and every
  # result goes back to pinned host memory inside the timed region; the copies of neighbouring batches overlap the compute
  import time

  def host_batches(n):
    for i in range(n):
      yield hx[i % 2]
  pipe = twingan.InferencePipeline(model, use_graph=not getattr(args, 'no_graph', False))
  for _, ev in pipe.run(host_batches(3)):
    pass
  torch.cuda.synchronize()
  t0 = time.perf_counter()
  last = None
  for last, ev in pipe.run(host_batches(steps)):
    pass
  torch.cuda.synchronize()
  ms_e2e = (time.perf_counter() - t0) * 1e3 / steps
  hout = last
  ms_eager = ms
  if pipe.use_graph:
    # resident latency of the same public path: the batch as one CUDA-graph replay (input already in HBM)
    for i in range(3):
      pipe._infer(xs[i % 2])
    torch.cuda.synchronize()
    e4, e5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e4.record()
    for i in range(steps):
      pipe._infer(xs[i % 2])
    e5.record()
    torch.cuda.synchronize()
    ms = e4.elapsed_time(e5) / steps
  fl = flops.step_flops_per_pair(args.hw, False, args.max_channels)
  gflop = (fl['F_E'] + fl['F_G']) / 1e9
  nbytes = batch * args.hw * args.hw * 3 * 4
  peaks = _peaks()
  # algorithmic HBM bytes of the pass: every conv layer reads its input and writes its output once (fp32 activations),
  # SURVEY 8a.1 layer table -> flops.mixed_roofline_seconds' byte model
  mixed = flops.mixed_roofline_seconds(args.hw, batch, peaks['tf'] * 1e12, peaks['hbm_gbs'] * 1e9, max_num_channels=args.max_channels)
  alg_bytes = mixed.get('fwd_bytes_E', 0.0) + mixed.get('fwd_bytes_G', 0.0)
  out = {'metric': 'images/sec inference @%dx%d bs=%d' % (args.hw, args.hw, batch), 'value': round(batch / (ms * 1e-3), 2),
         'unit': 'images/s', 'latency_ms': round(ms, 3), 'latency_ms_eager_launches': round(ms_eager, 3),
         'cuda_graph': bool(pipe.use_graph), 'steps': steps,
         'config': {'workload': 'configs[4]: %dx%d inference, batch %d, E(x;_s)->G(.;_t) eval mode, moving statistics' % (
             args.hw, args.hw, batch), 'gflop_per_image': round(gflop, 2)},
         'e2e': {'value': round(batch / (ms_e2e * 1e-3), 2), 'unit': 'images/s', 'h2d_bytes_per_step': nbytes,
                 'd2h_bytes_per_step': nbytes},
         'gpu_launches': int(launches), 'achieved_tflops': round(gflop * 1e9 * batch / (ms * 1e-3) / 1e12, 2),
         'frac_of_bf16_peak': round(gflop * 1e9 * batch / (ms * 1e-3) / 1e12 / peaks['tf'], 5)}
  if alg_bytes:
    out['algorithmic_gbs'] = round(alg_bytes / (ms * 1e-3) / 1e9, 1)
    out['frac_of_measured_hbm'] = round(alg_bytes / (ms * 1e-3) / 1e9 / peaks['hbm_gbs'], 4)
    out['algorithmic_bytes'] = alg_bytes
  return out


def bench_infer(args):
  """Secondary line on its own (`--workload infer`); the default run embeds the same measurement as `secondary.infer`."""
  dev = torch.device('cuda', int(os.environ.get('LOCAL_RANK', '0')))
  torch.cuda.set_device(dev)
  sampler = ClockSampler(dev.index or 0)
  sampler.start()
  m = infer_measure(args, dev)
  sampler.stop_flag = True
  m.update({'n_gpus': 1, 'warmup': args.warmup, 'ms_per_step': m['latency_ms'], 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32 (conv MACs as split-bf16 x3 on tcgen05, fp32 accumulate)', 'data': 'synthetic',
            'clocks': sampler.summary()})
  print(json.dumps(m), flush=True)


def profile_one_step(args):
  from twingan_b200 import twingan
  dev = torch.device('cuda', 0)
  model = twingan.GanModel(twingan.Flags(train_image_size=args.hw, pggan_max_num_channels=args.max_channels,
                                         generator_norm_type=args.norm, batch_passes=not args.pass_by_pass), device=dev)
  gen = torch.Generator(device=dev).manual_seed(100)
  s = torch.rand((args.batch, args.hw, args.hw, 3), device=dev, generator=gen)
  t = torch.rand((args.batch, args.hw, args.hw, 3), device=dev, generator=gen)
  r = twingan.make_dragan_rand(args.batch, args.hw, dev, gen)
  for _ in range(2):
    model.train_step(s, t, r)
  torch.cuda.synchronize()


def host_threads(cap=64):
  """Threads the CPU arm may really use: the affinity mask and the cgroup CPU quota, not the machine's core count
  (a container that sees 200+ cores but owns a few would oversubscribe and crawl)."""
  n = os.cpu_count() or 1
  try:
    n = min(n, len(os.sched_getaffinity(0)))
  except (AttributeError, OSError):
    pass
  try:   # cgroup v2
    quota, period = open('/sys/fs/cgroup/cpu.max').read().split()[:2]
    if quota != 'max':
      n = min(n, max(1, int(float(quota) / float(period))))
  except (OSError, ValueError):
    try:   # cgroup v1
      q = int(open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us').read())
      per = int(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
      if q > 0 and per > 0:
        n = min(n, max(1, q // per))
    except (OSError, ValueError):
      pass
  return max(1, min(n, cap))


def cpu_baseline(hw, sample_batch, max_channels, norm, steps=1, warmup=0, budget_s=120.0):
  """The oracle port (fp32, all usable host threads) timed on a bounded sample: the same G+D step at a smaller batch.
  The sample is cut (fewer timed steps, never fewer than one) when the box is too slow for `budget_s`."""
  from oracle import twingan_oracle as O
  cores = host_threads()
  torch.set_num_threads(cores)
  cfg = O.Config(hw=hw, max_num_channels=max_channels, generator_norm_type=norm)
  params = O.init_params(cfg, dtype=torch.float32)
  state = O.init_norm_state(cfg, dtype=torch.float32)
  m = {k: torch.zeros_like(v) for k, v in params.items()}
  v = {k: torch.zeros_like(p) for k, p in params.items()}
  src, tgt, rand = O.make_inputs(cfg, sample_batch, dtype=torch.float32)
  t_adam = 0
  times = []
  t_begin = time.perf_counter()
  for i in range(warmup + steps):
    t0 = time.perf_counter()
    _, _, _, _, t_adam = O.train_step(cfg, params, m, v, state, src, tgt, rand, t_adam)
    dt = time.perf_counter() - t0
    if i >= warmup:
      times.append(dt)
    if times and (time.perf_counter() - t_begin) + dt > budget_s:
      break
  sec = sum(times) / len(times)
  return {'value': round(sample_batch / sec, 5), 'unit': UNIT, 'cores': cores, 'kind': 'port',
          'threads': torch.get_num_threads(), 'machine_cores': os.cpu_count(), 'seconds_per_step': round(sec, 3),
          'timed_steps': len(times),
          'sample': 'oracle/twingan_oracle.py (PyTorch-CPU fp32 restatement, NOT twingan.py under TF): the same '
                    '%dx%d G+D step at batch %d pairs, %d step(s)' % (hw, hw, sample_batch, len(times))}


def cpu_baseline_subprocess(args, timeout_s=200.0):
  """Run the CPU arm in its own process with a hard time limit, so a slow or oversubscribed host can never take
  the GPU line down with it."""
  import subprocess
  cmd = [sys.executable, os.path.abspath(__file__), '--impl', 'reference', '--steps', '1', '--warmup', '1',
         '--hw', str(args.hw), '--max-channels', str(args.max_channels), '--norm', args.norm,
         '--cpu-sample-batch', str(args.cpu_sample_batch)]
  env = {k: v for k, v in os.environ.items() if k not in ('RANK', 'LOCAL_RANK', 'WORLD_SIZE')}
  try:
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout_s, env=env)
    line = [l for l in r.stdout.splitlines() if l.startswith('{')][-1]
    return json.loads(line)['cpu_baseline']
  except subprocess.TimeoutExpired:
    return {'value': None, 'unit': UNIT, 'cores': host_threads(), 'kind': 'port',
            'sample': 'oracle port, one %dx%d G+D step at batch %d pairs: did not finish within %.0f s on this host'
                      % (args.hw, args.hw, args.cpu_sample_batch, timeout_s)}
  except Exception as e:   # noqa: BLE001 -- the GPU line must survive any failure of the CPU arm
    return {'value': None, 'unit': UNIT, 'cores': host_threads(), 'kind': 'port', 'sample': 'CPU arm failed: %r' % (e,)}


def bench_reference(args):
  rank = int(os.environ.get('RANK', '0'))
  if rank != 0:
    return
  world = int(os.environ.get('WORLD_SIZE', '1'))
  cb = cpu_baseline(args.hw, args.cpu_sample_batch, args.max_channels, args.norm, steps=args.steps, warmup=min(args.warmup, 1),
                    budget_s=150.0)
  out = {'impl': 'reference', 'metric': METRIC, 'value': cb['value'], 'unit': UNIT, 'n_gpus': world, 'steps': cb['timed_steps'],
         'steps_requested': args.steps,
         'warmup': min(args.warmup, 1), 'ms_per_step': round(cb['seconds_per_step'] * 1e3, 1), 'higher_is_better': True,
         'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
         'config': {'workload': 'configs[3]: %dx%d full TwinGAN G+D step (mode B), CPU restatement, bounded sample of '
                                'batch %d pairs per step' % (args.hw, args.hw, args.cpu_sample_batch),
                    'cpu_sample_batch': args.cpu_sample_batch, 'global_batch': args.cpu_sample_batch,
                    'note': 'values are per pair, so the GPU arm (16 pairs/step/GPU) and this bounded sample divide fairly'},
         'cpu_baseline': cb,
         'e2e': {'value': cb['value'], 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
         'gpu_launches': 0}
  print(json.dumps(out), flush=True)


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=5)
  ap.add_argument('--warmup', type=int, default=3)
  ap.add_argument('--impl', default='cuda', choices=['cuda', 'reference'])
  ap.add_argument('--workload', default='train', choices=['train', 'infer'],
                  help="'infer': secondary line for BASELINE configs[4] (64-image inference); the headline metric is 'train'")
  ap.add_argument('--hw', type=int, default=HW)
  ap.add_argument('--batch', type=int, default=BATCH)
  ap.add_argument('--max-channels', type=int, default=MAXC)
  ap.add_argument('--norm', default=NORM)
  ap.add_argument('--prec', type=int, default=1)
  ap.add_argument('--cpu-sample-batch', type=int, default=2)
  ap.add_argument('--no-cpu-baseline', action='store_true')
  ap.add_argument('--no-graph', action='store_true', help='eager launches instead of CUDA-graph replay')
  ap.add_argument('--pass-by-pass', action='store_true',
                  help="A/B: run the reference's 16 separate network passes instead of batching the weight-sharing ones")
  ap.add_argument('--set-option', action='append', default=[], metavar='KEY=VALUE',
                  help='twg_set_option A/B switch applied before the run (e.g. 2=1: one sub-tile per halo tile)')
  ap.add_argument('--profile-one-step', action='store_true', help='1 warm-up + 1 step only (for ncu launch lists)')
  ap.add_argument('--no-secondary', action='store_true', help='skip the configs[4] inference measurement (secondary.infer)')
  ap.add_argument('--no-ddp-check', action='store_true', help='skip the data-parallel pre-flight at N > 1')
  ap.add_argument('--dump-outputs', metavar='DIR',
                  help='write the losses the last timed training step returned as DIR/<name>.npy; that step starts from '
                       'the seeded initial model state and its inputs are seeded, so two builds compare output for output')
  args = ap.parse_args()
  if args.dump_outputs and (args.impl != 'cuda' or args.workload != 'train' or args.profile_one_step):
    ap.error('--dump-outputs writes the outputs of the timed training step: --impl cuda --workload train only')
  if args.steps < 1:
    ap.error('--steps must be at least 1')
  if args.impl == 'reference':
    bench_reference(args)
    return
  if not torch.cuda.is_available():
    raise SystemExit('bench.py needs a CUDA device for --impl cuda (there is no CPU fallback)')
  from twingan_b200 import ops
  ops.set_precision(args.prec)
  if args.profile_one_step:
    profile_one_step(args)
    return
  if args.warmup < 3:
    args.warmup = 3
  if args.workload == 'infer':
    bench_infer(args)
    return
  bench_cuda(args)


if __name__ == '__main__':
  main()
