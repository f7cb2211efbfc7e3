#!/usr/bin/env python
"""Benchmark of the hot path.

  python bench.py --gpus N --steps K --warmup W            our arm (one rank per GPU, NCCL)
  python bench.py --impl reference --gpus N --steps K ...  CPU arm: the oracle restatement of
                                                           the reference (JAX is not installable here)
  --workload train360 (default)  BASELINE config 2: 360.gin train step, 16384 rays x (64+64+32) samples
             refnerf             BASELINE config 3: blender_refnerf.gin train step, 4096 rays x (128+128)
             raw                 BASELINE config 4: llff_raw.gin train step, 8192 rays x (128+128)
             render              BASELINE config 5: 1560x1040 image, 360.gin, chunks of 16384 rays sharded
                                 over the ranks, pixels all-gathered (one step = one image)
Prints ONE JSON line (see README/DESIGN.md for the field contract).  A train "step" is one full
train step (forward, losses, backward, grad all-reduce, clip+Adam, weight repack) on one synthetic
batch of `batch_size` rays (global; sharded B/N per GPU, as train.py:52-53).
  --dump-outputs DIR   after the timed steps, write what the last timed step returned to its caller as
                       DIR/<name>.npy (see dump_outputs): the inputs are seeded, so two builds run with the
                       same arguments can be compared output for output.
Timing: CUDA events on the launching stream, barrier + synchronize on both sides, max over
ranks; the activations written per step (>10 GB) exceed the 126 MB L2, so no flush is needed.
"""
import argparse
import datetime
import json
import math
import os
import subprocess
import sys
import tempfile
import time

# The CPU arm must own the host's threads.  torchrun exports OMP_NUM_THREADS=1 to every rank, which
# (set before the OpenMP / MKL runtimes start) would throttle the reference arm by two orders of
# magnitude, so that arm resets the variables before numpy / torch are imported.
# CPU_THREADS: pinned from the thread sweep of tools/cpu_sweep.py on the GPU box's host
# (profiles/r02_cpu_sweep.txt): the torch-CPU graph of many small ops stops scaling past this count.
CPU_THREADS_DEFAULT = 16
if '--impl' in sys.argv and sys.argv[sys.argv.index('--impl') + 1:sys.argv.index('--impl') + 2] == ['reference'] \
    or '--impl=reference' in sys.argv:
  _t = str(min(os.cpu_count() or 1, int(os.environ.get('MNRF_CPU_THREADS', str(CPU_THREADS_DEFAULT)))))
  for _k in ('OMP_NUM_THREADS', 'MKL_NUM_THREADS', 'OPENBLAS_NUM_THREADS'):
    os.environ[_k] = _t

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FWD_FLOP_PER_RAY = 638435328           # SURVEY.md section 8(d): 2 * MACs of Prop x128 + Nerf x32
TRAIN_FLOP_PER_RAY = 1815994368        # 3 x fwd - unneeded dgrad (canonical, never overstated)

WORKLOADS = {
    'train360': dict(kind='train', bundle='bundle_360', batch=16384, cpu_rays=1024,
                     metric='train-step rays/sec @16384 rays x (64+64+32) samples',
                     name='mip-NeRF 360 (360.gin) train step: %d rays x (64+64+32) samples, PropMLP 4x256, NerfMLP 8x1024'),
    'refnerf': dict(kind='train', bundle='bundle_blender_refnerf', batch=4096, cpu_rays=128,
                    metric='train-step rays/sec @4096 rays x (128+128) samples (blender_refnerf.gin)',
                    name='Ref-NeRF (blender_refnerf.gin) train step: %d rays x (128+128) samples, NerfMLP 8x256 + IDE view MLP 8x128'),
    'raw': dict(kind='train', bundle='bundle_llff_raw', batch=8192, cpu_rays=256,
                metric='train-step rays/sec @8192 rays x (128+128) samples (llff_raw.gin)',
                name='RawNeRF (llff_raw.gin) train step: %d rays x (128+128) samples, NerfMLP 8x256, rawnerf loss'),
    'render': dict(kind='render', bundle='bundle_360', H=1040, W=1560, cpu_rays=1024,
                   metric='render rays/sec, 1560x1040 image, 360.gin, (64+64+32) samples/ray',
                   name='render.py full image 1560x1040 (360.gin, 160 MLP queries per ray), %d-ray chunks sharded over '
                        'the ranks, pixels all-gathered'),
}


def plan_flops(bundle):
  """Canonical FLOPs per ray from the layer tables (logical flax shapes, 2 x MACs), as SURVEY.md 8(d) counts
  them: forward = every Dense of every level; train = 3 x forward minus the input-gradient GEMMs autodiff
  never needs (layer 0, the feature slice of skip layers, the view-direction slice of the view MLP).
  Ref-NeRF density normals are counted as the reference computes them (reverse mode: one extra trunk pass
  in the forward, trained through), not as the three forward-mode tangent streams this implementation runs."""
  from multinerf_b200.models import MLPPlan
  m = bundle.model
  plans = {'nerf': MLPPlan(bundle.nerf_mlp, m.use_viewdirs, glo_features=m.num_glo_features)}
  plans['prop'] = plans['nerf'] if m.single_mlp else MLPPlan(bundle.prop_mlp, m.use_viewdirs)
  fwd_ray = train_ray = 0
  for i in range(m.num_levels):
    last = i == m.num_levels - 1
    plan = plans['nerf'] if last else plans['prop']
    S = m.num_nerf_samples if last else m.num_prop_samples
    fwd = sum(2 * sp.in_dim * sp.out_dim for sp in plan.specs)
    trunk = plan.by_role('trunk')
    W, F = plan.cfg.net_width, plan.F
    if plan.density_normals:
      fwd += sum(2 * sp.in_dim * sp.out_dim for sp in trunk) + 2 * W
    unneeded = 0
    for j, sp in enumerate(trunk):
      if j == 0:
        unneeded += 2 * sp.in_dim * sp.out_dim
      elif sp.row_map is not None:
        unneeded += 2 * F * sp.out_dim
    for sp in plan.specs:
      if sp.role not in ('trunk', 'view', 'rgb') and sp.row_map is not None:
        unneeded += 2 * F * sp.out_dim
    if plan.has_rgb and not plan.ref_stage:
      views = plan.by_role('view')
      dirw = plan.vin_dim - plan.cfg.bottleneck_width - plan.glo_features
      unneeded += 2 * dirw * views[0].out_dim * (1 + len(plan.view_concat_after))
    if plan.density_normals:
      unneeded = 0          # positions are differentiated through: nothing is skipped
    fwd_ray += S * fwd
    train_ray += S * (3 * fwd - unneeded)
  return fwd_ray, train_ray


def synth_batch(seed, B, workload='train360'):
  """SURVEY.md 8(d) recipe: unit-cube origins, normalised directions x U(.8,1.2) (360); cameras on a
  sphere looking inward (Ref-NeRF, blender bounds 2..6); forward-facing NDC-style rays with per-ray
  exposures and a Bayer loss mask (RawNeRF)."""
  rng = np.random.default_rng(seed)
  f = np.float32
  extra = {}
  if workload == 'raw':
    o = np.concatenate([rng.uniform(-1, 1, (B, 2)), -np.ones((B, 1))], -1).astype(f)
    d = np.concatenate([rng.uniform(-.5, .5, (B, 2)), 2 * np.ones((B, 1))], -1)
    v = (d / np.linalg.norm(d, axis=-1, keepdims=True)).astype(f)
    d = d.astype(f)
    eidx = rng.integers(0, 4, (B, 1)).astype(np.int32)
    extra = dict(exposure_idx=eidx, exposure_values=(2.0 ** -eidx).astype(f))
    lossmult = np.eye(3, dtype=f)[rng.integers(0, 3, B)]
    near, far, radii = 0.0, 1.0, rng.uniform(1e-3, 2e-3, (B, 1)).astype(f)
  elif workload == 'refnerf':
    o = rng.normal(size=(B, 3))
    o = o / np.linalg.norm(o, axis=-1, keepdims=True) * 4.0
    d = -o / 4.0 + rng.normal(size=(B, 3)) * 0.1
    d /= np.linalg.norm(d, axis=-1, keepdims=True)
    o, v, d = o.astype(f), d.astype(f), d.astype(f)
    lossmult = np.ones((B, 1), f)
    near, far, radii = 2.0, 6.0, rng.uniform(5e-4, 1e-3, (B, 1)).astype(f)
  else:
    o = rng.uniform(-1, 1, (B, 3)).astype(f)
    d = rng.normal(size=(B, 3))
    d /= np.linalg.norm(d, axis=-1, keepdims=True)
    v = d.astype(f)
    d = (d * rng.uniform(0.8, 1.2, (B, 1))).astype(f)
    lossmult = np.ones((B, 1), f)
    near, far, radii = 0.2, 1e6, rng.uniform(5e-4, 1e-3, (B, 1)).astype(f)
  rays = dict(origins=o, directions=d, viewdirs=v, radii=radii,
              imageplane=np.zeros((B, 2), f), lossmult=lossmult,
              near=np.full((B, 1), near, f), far=np.full((B, 1), far, f),
              cam_idx=np.zeros((B, 1), np.int32), **extra)
  rgb = rng.uniform(0, 1, (B, 3)).astype(f)
  return rays, rgb


def image_rays(H, W):
  """A 1560x1040 perspective camera inside the unit cube (BASELINE config 5), rays as [H, W, n]."""
  f = np.float32
  ys, xs = np.meshgrid(np.arange(H, dtype=np.float64), np.arange(W, dtype=np.float64), indexing='ij')
  cam = np.array([0.5, 0.5, 0.3])
  fwd = -cam / np.linalg.norm(cam)
  right = np.cross(fwd, [0, 0, 1.0])
  right /= np.linalg.norm(right)
  up = np.cross(right, fwd)
  d = ((xs - W / 2)[..., None] * right + (H / 2 - ys)[..., None] * up) / 1200.0 + fwd
  v = d / np.linalg.norm(d, axis=-1, keepdims=True)
  return dict(origins=np.broadcast_to(cam, d.shape).astype(f).copy(), directions=d.astype(f), viewdirs=v.astype(f),
              radii=np.full((H, W, 1), 2 / (1200 * np.sqrt(12)), f), imageplane=np.zeros((H, W, 2), f),
              lossmult=np.ones((H, W, 1), f), near=np.full((H, W, 1), 0.2, f), far=np.full((H, W, 1), 1e6, f),
              cam_idx=np.zeros((H, W, 1), np.int32))


def peaks():
  """(burst bf16 TFLOP/s, sustained bf16 TFLOP/s, HBM GB/s, source)."""
  path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(path):
    with open(path) as fh:
      p = json.load(fh)
    return p.get('bf16_tflops'), p.get('bf16_tflops_sustained', p.get('bf16_tflops')), p.get('hbm_gbs'), 'measured'
  return 1650.0, 1400.0, 6650.0, 'fallback'      # B200_PROFILING.md fallback figures


class ClockSampler:
  """nvidia-smi clocks / throttle reasons sampled DURING the timed region.  The sampler is started early
  (nvidia-smi takes about a second to produce its first line) and polls every 25 ms; `window()` marks the
  host-time interval of the timed region and only samples inside it are reported, so even a 0.1 s region
  (8 GPUs) carries clock evidence."""
  Q = ('timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
       'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
       'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

  def __init__(self, gpu_index):
    self.idx = gpu_index
    self.proc = None
    self.path = None
    self.t0 = self.t1 = None

  def start(self):
    try:
      fd, self.path = tempfile.mkstemp(suffix='.csv')
      os.close(fd)
      self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                    '-lms', '25', '-i', str(self.idx)],
                                   stdout=open(self.path, 'w'), stderr=subprocess.DEVNULL)
    except Exception:  # pylint: disable=broad-except
      self.proc = None

  def window(self, t0, t1):
    self.t0, self.t1 = t0, t1

  def stop(self):
    out = {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': []}
    if self.proc is None:
      return out
    time.sleep(0.05)
    self.proc.terminate()
    try:
      self.proc.wait(timeout=5)
    except Exception:  # pylint: disable=broad-except
      self.proc.kill()
    rows = []
    try:
      for line in open(self.path):
        p = [x.strip() for x in line.split(',')]
        if len(p) < 10:
          continue
        try:
          ts = datetime.datetime.strptime(p[0], '%Y/%m/%d %H:%M:%S.%f').timestamp()
        except ValueError:
          continue
        rows.append((ts, float(p[2]), float(p[3]), float(p[4]), p[6:10]))
      os.unlink(self.path)
    except Exception:  # pylint: disable=broad-except
      pass
    if not rows:
      return out
    inside = [r for r in rows if self.t0 is not None and self.t0 <= r[0] <= self.t1]
    where = 'timed region'
    if not inside and self.t0 is not None:      # region shorter than the polling period: nearest samples
      mid = 0.5 * (self.t0 + self.t1)
      inside = sorted(rows, key=lambda r: abs(r[0] - mid))[:2]
      where = 'nearest to the timed region'
    if not inside:
      inside, where = rows, 'whole run'
    reasons = set()
    for r in inside:
      for name, val in zip(['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'], r[4]):
        if val.lower().startswith('active'):
          reasons.add(name)
    return {'sm_mhz': float(np.median([r[1] for r in inside])), 'sm_max_mhz': float(max(r[2] for r in inside)),
            'power_w': float(np.median([r[3] for r in inside])), 'reasons': sorted(reasons),
            'samples': len(inside), 'sampled': where}


def roofline_block(canon_flops, gemm_ms, gemm_flops, n_gemm, step_ms, clocks, traffic, kernel):
  burst, sustained, _, kind = peaks()
  capped = 'sw_power_cap' in (clocks.get('reasons') or [])
  # the denominator follows the observed cap state: a power-capped step is held against the sustained
  # cuBLAS figure, an uncapped one against the burst figure; both fractions are printed
  peak = sustained if capped else burst
  achieved = canon_flops / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
  whole = canon_flops / (step_ms / 1e3) / 1e12
  return {'bound': 'tensor', 'achieved': achieved, 'peak': peak, 'unit': 'TFLOP/s',
          'frac': achieved / peak if peak else None, 'traffic': traffic,
          'traffic_unit': 'DRAM bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum)',
          'peak_kind': f'{kind} {"sustained (step ran under sw_power_cap)" if capped else "burst (no cap active)"} bf16',
          'frac_vs_burst': achieved / burst if burst else None,
          'frac_vs_sustained': achieved / sustained if sustained else None,
          'launches_per_step': n_gemm, 'avg_launch_ms': gemm_ms / max(1, n_gemm),
          'algorithmic_flop_per_launch': canon_flops / max(1, n_gemm), 'kernel': kernel,
          'gemm_ms_per_step': gemm_ms, 'gemm_share_of_step': gemm_ms / step_ms,
          'executed_tflops': gemm_flops / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0,
          'whole_step_tflops': whole, 'whole_step_frac': whole / peak if peak else None}


DUMP_BYTES = 64 * 10**6


def sample_positions(size, kept):
  """Flat (C-order) indices, ascending, of the `kept` elements that dump_outputs writes of an array of `size`."""
  return np.sort(np.random.default_rng(0).choice(size, kept, replace=False))


def dump_outputs(out_dir, arrays):
  """Writes `arrays` (name -> tensor or ndarray) as <out_dir>/<name>.npy, float64 kept, everything else as
  float32, DUMP_BYTES in all at most.  The budget is split evenly over the arrays, smallest first; an array
  larger than its share is written flattened, only its elements at sample_positions(size, kept): the same
  positions on every run.  <out_dir>/dump.json gives each array's original shape and, when sampled, `kept`."""
  import torch
  host = {}
  for name, v in arrays.items():
    if isinstance(v, torch.Tensor):
      v = v.detach().cpu()
      v = (v if v.dtype == torch.float64 else v.float()).numpy()
    v = np.asarray(v)
    host[name] = v if v.dtype == np.float64 else v.astype(np.float32)
  names = sorted(host, key=lambda k: (host[k].nbytes, k))
  left = DUMP_BYTES - 256 * len(names) - 65536    # room for the .npy headers and dump.json
  share = None                                    # set by the first array over its share: all later ones are too
  index = {}
  os.makedirs(out_dir, exist_ok=True)
  for i, name in enumerate(names):
    v = host[name]
    index[name] = {'shape': list(v.shape), 'kept': None}
    if share is None and v.nbytes > left // (len(names) - i):
      share = left // (len(names) - i)
    if share is not None:
      index[name]['kept'] = share // v.itemsize
      v = v.reshape(-1)[sample_positions(v.size, share // v.itemsize)]
    left -= v.nbytes
    np.save(os.path.join(out_dir, name + '.npy'), v)
  with open(os.path.join(out_dir, 'dump.json'), 'w') as f:
    json.dump({'arrays': dict(sorted(index.items())),
               'sampled': 'an array with `kept` set holds only the flattened elements at '
                          'bench.sample_positions(prod(shape), kept)'}, f, indent=1)


def train_outputs(params, stats):
  """What a train step hands back: the updated state (flat fp32 parameters and Adam moments) and the
  step's loss statistics."""
  stats.materialize()
  out = {'params': params.flat, 'adam_mu': params.mu, 'adam_nu': params.nu, 'mses': stats['mses'],
         'psnrs': stats['psnrs'], 'loss': np.float64(stats['loss'])}
  out.update({'loss_' + k: np.float64(v) for k, v in stats['losses'].items()})
  return out


def render_outputs(rendering):
  """What render_image hands back: the [H, W, ...] image buffers and the per-level ray_* bundles."""
  out = {}
  for k, v in rendering.items():
    if k.startswith('ray_'):
      out.update({f'{k}_{i}': lv for i, lv in enumerate(v)})
    else:
      out[k] = v
  return out


def run_ours(args):
  import torch
  import torch.distributed as dist
  from multinerf_b200 import configs, models, ops, train_utils, utils

  wl = WORKLOADS[args.workload]
  world = int(os.environ.get('WORLD_SIZE', '1'))
  rank = int(os.environ.get('RANK', '0'))
  local = int(os.environ.get('LOCAL_RANK', '0'))
  sampler = ClockSampler(local)
  if rank == 0:
    sampler.start()                     # long before the timed region
  torch.cuda.set_device(local)
  if world > 1:
    os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
    dist.init_process_group('nccl', device_id=torch.device('cuda', local))
  dev = torch.device('cuda', local)
  bundle = getattr(configs, wl['bundle'])()
  fwd_flop_ray, train_flop_ray = plan_flops(bundle)
  if args.workload == 'train360':
    assert (fwd_flop_ray, train_flop_ray) == (FWD_FLOP_PER_RAY, TRAIN_FLOP_PER_RAY), (fwd_flop_ray, train_flop_ray)

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  def max_over_ranks(ms):
    if world > 1:
      t = torch.tensor([ms], device=dev)
      dist.all_reduce(t, op=dist.ReduceOp.MAX)
      ms = float(t)
    return ms

  if wl['kind'] == 'render':
    return run_render(args, wl, bundle, fwd_flop_ray, world, rank, dev, sampler, barrier, max_over_ranks)

  B_global = args.batch_size or wl['batch']
  if args.scaling == 'weak':
    B_global *= world
  assert B_global % world == 0
  B = B_global // world
  model, variables = models.construct_model(2, None, bundle, device=dev)
  step_fn = train_utils.create_train_step(model, bundle.config, use_graph=not args.no_graph)
  state = train_utils.TrainState(variables)
  gen = torch.Generator(device=dev)
  gen.manual_seed(1234 + rank)

  # host batches in pinned memory; every step copies its batch H2D inside the timed region (e2e)
  nbuf = 4
  host = []
  for i in range(nbuf):
    rays_np, rgb_np = synth_batch(100 + i, B_global, args.workload)
    sl = slice(rank * B, (rank + 1) * B)
    hr = {k: torch.from_numpy(np.ascontiguousarray(v[sl])).pin_memory() for k, v in rays_np.items()}
    host.append((hr, torch.from_numpy(np.ascontiguousarray(rgb_np[sl])).pin_memory()))
  h2d_bytes = sum(t.numel() * t.element_size() for t in host[0][0].values()) + host[0][1].numel() * 4

  def device_batch(i):
    hr, hrgb = host[i % nbuf]
    rays = utils.Rays(**{k: v.to(dev, non_blocking=True) for k, v in hr.items()})
    return utils.Batch(rays=model._prep_rays(rays), rgb=hrgb.to(dev, non_blocking=True))

  resident = [device_batch(i) for i in range(nbuf)]
  torch.cuda.synchronize()

  def timed(n, e2e):
    nonlocal state
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    loss_host = stats = None
    t0 = time.time()
    e0.record()
    for i in range(n):
      batch = device_batch(i) if e2e else resident[i % nbuf]
      state, stats, _ = step_fn(gen, state, batch, None, 0.5)
      if e2e:
        loss_host = stats._buf.to('cpu', non_blocking=False)     # D2H read of the step's losses
    e1.record()
    barrier()
    t1 = time.time()
    return max_over_ranks(e0.elapsed_time(e1)), loss_host, (t0, t1), stats

  timed(args.warmup, False)
  ops.LAUNCHES = 0
  ms, _, win, stats = timed(args.steps, False)
  sampler.window(*win)
  if args.dump_outputs and rank == 0:
    # before the end-to-end loop below: it keeps training the same state in place
    dump_outputs(args.dump_outputs, train_outputs(state.params, stats))
  launches_total = ops.LAUNCHES                 # our kernels launched inside the timed region (all K steps)
  launches = launches_total // max(1, args.steps)
  # stop the poller before the end-to-end loop: nvidia-smi queries contend with the driver calls of a loop
  # that synchronises every step (D2H read of the losses)
  clocks = sampler.stop() if rank == 0 else {}
  ms_e2e, loss_host, _, _ = timed(args.steps, True)

  # dominant kernel (tcgen05 GEMM, all three modes): CUDA events around every launch of one
  # extra step; achieved = canonical train FLOPs of the step / time spent inside the GEMMs
  eager_fn = train_utils.create_train_step(model, bundle.config, use_graph=False)
  ops.GEMM_EVENTS = []
  barrier()
  state, _, _ = eager_fn(gen, state, resident[0], None, 0.5)
  barrier()
  evs = ops.GEMM_EVENTS
  ops.GEMM_EVENTS = None
  torch.cuda.synchronize()
  gemm_ms = sum(a.elapsed_time(b) for a, b, _ in evs)
  gemm_flops = sum(f for _, _, f in evs)

  if rank != 0:
    if world > 1:
      dist.destroy_process_group()
    return
  rays_per_s = B_global * args.steps / (ms / 1e3)
  rays_per_s_e2e = B_global * args.steps / (ms_e2e / 1e3)
  # DRAM bytes per GEMM launch from the committed ncu capture (tools/summarize_profile.py); only valid for
  # the configuration it was captured on (1 GPU, 16384 rays)
  traffic = None
  tpath = os.path.join(ROOT, 'profiles', 'gemm_tc_traffic.json')
  if os.path.exists(tpath) and B == 16384 and args.workload == 'train360':
    with open(tpath) as f:
      traffic = json.load(f).get('dram_bytes_per_launch')
  out = {
      'metric': wl['metric'],
      'value': rays_per_s, 'unit': 'rays/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
      'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': args.scaling,
      'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
      'config': {'workload': wl['name'] % B_global,
                 'global_batch': B_global, 'rays_per_gpu': B, 'parallelism': f'dp{world}',
                 'cuda_graphs': not args.no_graph,
                 'l2_flush': 'not needed: >10 GB of activations streamed per step (L2 = 126 MB)'},
      'e2e': {'value': rays_per_s_e2e, 'unit': 'rays/s', 'h2d_bytes_per_step': int(h2d_bytes * world),
              'd2h_bytes_per_step': int(loss_host.numel() * 4 * world) if loss_host is not None else 0,
              'ms_per_step': ms_e2e / args.steps},
      'gpu_launches': int(launches_total), 'gpu_launches_per_step': int(launches),
      'roofline': roofline_block(train_flop_ray * B, gemm_ms, gemm_flops, len(evs), ms / args.steps, clocks, traffic,
                                 'gemm_tc_kernel (tcgen05 fwd+dgrad+wgrad)'),
      'clocks': clocks,
  }
  if world == 1 and not args.no_cpu_baseline:
    out['cpu_baseline'] = cpu_baseline(args.workload, args.cpu_rays or wl['cpu_rays'], 1, 1)
  print(json.dumps(out), flush=True)
  if world > 1:
    dist.destroy_process_group()


def run_render(args, wl, bundle, fwd_flop_ray, world, rank, dev, sampler, barrier, max_over_ranks):
  """BASELINE config 5.  One step = one 1560x1040 image through models.render_image: 16384-ray chunks,
  each sharded over the ranks, one packed all-gather of the last level's pixels per chunk."""
  import torch
  import torch.distributed as dist
  from multinerf_b200 import models, ops, train_utils, utils
  H, W = wl['H'], wl['W']
  rays_np = image_rays(H, W)
  model, state, _, _, _ = train_utils.setup_model(bundle, 0, device=dev)
  render_eval = train_utils.create_render_fn(model, use_graph=not args.no_graph)
  render_fn = lambda rng, r: render_eval(state.params, 1.0, None, r)
  dev_rays = utils.Rays(**{k: torch.as_tensor(v).to(dev) for k, v in rays_np.items()})
  host_rays = utils.Rays(**{k: torch.from_numpy(v).pin_memory() for k, v in rays_np.items()})
  chunk = bundle.config.render_chunk_size
  n_chunks = (H * W + chunk - 1) // chunk

  def timed(n, e2e):
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    img = None
    t0 = time.time()
    e0.record()
    for _ in range(n):
      out = models.render_image(render_fn, host_rays if e2e else dev_rays, None, bundle, verbose=False,
                                world_size=world, rank=rank)
      if e2e:
        img = out['rgb'].to('cpu', non_blocking=False)          # D2H of the finished image
    e1.record()
    barrier()
    t1 = time.time()
    return max_over_ranks(e0.elapsed_time(e1)), img, out, (t0, t1)

  timed(max(1, args.warmup), False)
  ops.LAUNCHES = 0
  ms, _, out, win = timed(args.steps, False)
  sampler.window(*win)
  if args.dump_outputs and rank == 0:
    dump_outputs(args.dump_outputs, render_outputs(out))
  launches_total = ops.LAUNCHES
  clocks = sampler.stop() if rank == 0 else {}
  ms_e2e, img, _, _ = timed(args.steps, True)
  # GEMM time of one eager chunk (this rank's shard)
  per = chunk // world
  one = dev_rays.map(lambda a: a.reshape(H * W, -1)[:per])
  ops.GEMM_EVENTS = []
  barrier()
  model.apply(state.params, None, one, 1.0, True)
  barrier()
  evs = ops.GEMM_EVENTS
  ops.GEMM_EVENTS = None
  gemm_ms = sum(a.elapsed_time(b) for a, b, _ in evs)
  gemm_flops = sum(f for _, _, f in evs)
  if rank != 0:
    if world > 1:
      dist.destroy_process_group()
    return
  n = H * W
  s_img = ms / 1e3 / args.steps
  h2d = sum(v.numel() * v.element_size() for v in [getattr(host_rays, k) for k in rays_np])
  keys = [k for k in out if not k.startswith('ray_')]
  gathered_floats = sum(int(np.prod(out[k].shape[2:])) if out[k].dim() > 2 else 1 for k in keys)
  res = {
      'metric': wl['metric'], 'value': n / s_img, 'unit': 'rays/s', 'n_gpus': world, 'steps': args.steps,
      'warmup': max(1, args.warmup), 'ms_per_step': ms / args.steps, 's_per_image': s_img,
      'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
      'config': {'workload': wl['name'] % chunk, 'image': [W, H], 'render_chunk_size': chunk, 'chunks_per_image': n_chunks,
                 'rays_per_gpu_per_chunk': per, 'parallelism': f'dp{world}', 'compute_extras': True,
                 'cuda_graphs': not args.no_graph,
                 'l2_flush': 'not needed: each chunk streams >1 GB of activations (L2 = 126 MB)'},
      'e2e': {'value': n / (ms_e2e / 1e3 / args.steps), 'unit': 'rays/s', 'h2d_bytes_per_step': int(h2d),
              'd2h_bytes_per_step': int(img.numel() * 4) if img is not None else 0,
              'ms_per_step': ms_e2e / args.steps},
      'gpu_launches': int(launches_total), 'gpu_launches_per_step': int(launches_total // max(1, args.steps)),
      'all_gather': {'collectives_per_image': n_chunks if world > 1 else 0,
                     'bytes_per_image_per_rank_out': int(n * gathered_floats * 4) if world > 1 else 0,
                     'keys': keys},
      'roofline': roofline_block(fwd_flop_ray * per, gemm_ms, gemm_flops, len(evs), ms / args.steps / n_chunks,
                                 clocks, None, 'gemm_tc_kernel (tcgen05 forward), one chunk'),
      'clocks': clocks,
  }
  if world == 1 and not args.no_cpu_baseline:
    res['cpu_baseline'] = cpu_baseline('render', args.cpu_rays or wl['cpu_rays'], 1, 1)
  print(json.dumps(res), flush=True)
  if world > 1:
    dist.destroy_process_group()


def cpu_baseline(workload, n_rays, steps, warmup):
  """The oracle (CPU restatement of the reference), fp32 torch-CPU, on a bounded ray sample of the workload:
  the train step (forward, losses, autograd backward, clip, Adam) or, for `render`, the deterministic
  Model.__call__ with compute_extras."""
  import torch
  from multinerf_b200 import configs
  from multinerf_b200.models import MLPPlan, _init_kernel
  from oracle import o_models, o_train
  cores = os.cpu_count() or 1
  threads = min(cores, int(os.environ.get('MNRF_CPU_THREADS', str(CPU_THREADS_DEFAULT))))
  torch.set_num_threads(threads)
  wl = WORKLOADS[workload]
  bundle = getattr(configs, wl['bundle'])()
  rng = np.random.default_rng(2)
  m = bundle.model
  plans = {'NerfMLP_0': MLPPlan(bundle.nerf_mlp, m.use_viewdirs, glo_features=m.num_glo_features)}
  if not m.single_mlp:
    plans['PropMLP_0'] = MLPPlan(bundle.prop_mlp, m.use_viewdirs)
  params = {name: {sp.name: {'kernel': torch.tensor(_init_kernel(rng, pl.cfg.weight_init, sp.in_dim, sp.out_dim)),
                             'bias': torch.zeros(sp.out_dim)} for sp in pl.specs}
            for name, pl in plans.items()}
  if m.learned_exposure_scaling:
    params['exposure_scaling_offsets'] = {'embedding': torch.zeros(m.num_glo_embeddings, 3)}
  bases = {'nerf': plans['NerfMLP_0'].basis, 'prop': plans.get('PropMLP_0', plans['NerfMLP_0']).basis}
  rays_np, rgb_np = synth_batch(7, n_rays, 'train360' if workload == 'render' else workload)

  class R:
    pass
  rays = R()
  rays.exposure_idx = rays.exposure_values = None
  for k2, v in rays_np.items():
    setattr(rays, k2, torch.tensor(v))
  target = torch.tensor(rgb_np)
  S = [m.num_prop_samples] * (m.num_levels - 1) + [m.num_nerf_samples]
  rand = {'jitter': [torch.rand(n_rays, 1) if m.single_jitter else torch.rand(n_rays, s) for s in S],
          'density_noise': [torch.randn(n_rays, s) for s in S]}
  opt = {'count': 0, 'mu': {}, 'nu': {}}
  times = []
  for i in range(warmup + steps):
    t0 = time.perf_counter()
    if wl['kind'] == 'render':
      with torch.no_grad():
        o_models.model_apply(params, bundle, bases, rays, 1.0, True, rand=None)
    else:
      params, opt, _, _ = o_train.train_step(params, opt, bundle, bases, rays, target, 0.5, rand=rand)
    times.append(time.perf_counter() - t0)
  t = float(np.mean(times[warmup:]))
  what = 'deterministic render (Model.__call__, compute_extras)' if wl['kind'] == 'render' else 'train step'
  return {'value': n_rays / t, 'unit': 'rays/s', 'cores': threads, 'host_cores': cores, 'kind': 'port',
          'sample': f'{n_rays} rays of the same {wl["bundle"][7:]} {what}, fp32 torch-CPU, '
                    f'{steps} timed step(s) after {warmup} warm-up, {threads} threads (the best point of the thread sweep in '
                    'profiles/r02_cpu_sweep.txt: 16 > 32 > 64 >> 128 on the 128-core host); CPU restatement of the reference '
                    '(JAX/Flax are not installable in this image)',
          's_per_step': t}


def run_reference(args):
  rank = int(os.environ.get('RANK', '0'))
  if rank != 0:
    return
  wl = WORKLOADS[args.workload]
  n_rays = args.cpu_rays or wl['cpu_rays']
  base = cpu_baseline(args.workload, n_rays, max(1, args.steps), max(0, min(args.warmup, 3)))
  out = {
      'impl': 'reference', 'metric': wl['metric'],
      'value': base['value'], 'unit': 'rays/s', 'n_gpus': int(os.environ.get('WORLD_SIZE', '1')),
      'steps': max(1, args.steps), 'warmup': max(0, min(args.warmup, 3)),
      'ms_per_step': base['s_per_step'] * 1e3, 'higher_is_better': True, 'scaling': args.scaling,
      'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
      'config': {'workload': (wl['name'] % (wl.get('batch') or 16384)) +
                             ' -- bounded sample of %d rays per step on the host CPU (reference arm = oracle port; '
                             'JAX unavailable)' % n_rays},
      'cpu_baseline': base,
      'e2e': {'value': base['value'], 'unit': 'rays/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
  }
  print(json.dumps(out), flush=True)


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=10)
  ap.add_argument('--warmup', type=int, default=3)
  ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
  ap.add_argument('--workload', default='train360', choices=sorted(WORKLOADS))
  ap.add_argument('--batch_size', type=int, default=0, help='global rays per train step (default: the workload\'s)')
  ap.add_argument('--scaling', default='strong', choices=['strong', 'weak'])
  ap.add_argument('--cpu_rays', type=int, default=0, help='rays per CPU-arm step (default: the workload\'s)')
  ap.add_argument('--no_cpu_baseline', action='store_true')
  ap.add_argument('--no_graph', action='store_true', help='launch every kernel from Python (no CUDA graphs)')
  ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                  help='write what the last timed step returned as DIR/<name>.npy (float32/float64, <= 64 MB in all)')
  args = ap.parse_args()
  if args.dump_outputs and args.impl != 'ours':
    ap.error('--dump-outputs applies to --impl ours')
  if args.impl == 'reference':
    # exactly K timed steps; each step is a bounded ray sample of the workload, shrunk for large K so
    # that the whole run stays within a few minutes of CPU time (1024 rays of 360.gin ~ 3 s per step)
    if not args.cpu_rays:
      args.cpu_rays = WORKLOADS[args.workload]['cpu_rays']
    if args.steps > 40:
      args.cpu_rays = max(32, int(args.cpu_rays * 40 / args.steps) // 32 * 32)
    run_reference(args)
    return
  world = int(os.environ.get('WORLD_SIZE', '1'))
  if args.gpus > 1 and world == 1:
    # convenience: re-launch under torchrun when called directly with --gpus N
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', f'--nproc-per-node={args.gpus}',
           '--master-addr', '127.0.0.1', '--master-port', '29517', os.path.abspath(__file__)] + sys.argv[1:]
    sys.exit(subprocess.call(cmd))
  run_ours(args)


if __name__ == '__main__':
  main()
