"""Model-level parity on the GPU: Model.__call__ and the train step vs the CPU oracle on
identical synthetic rays and weights (SURVEY.md section 8d).  Needs a B200.

The Dense layers run in bf16 on tensor cores, so the oracle is evaluated with the same
bf16-rounded weights and bf16-rounded layer inputs (fp32 accumulation) -- see
oracle/o_models.py `bf16=True`.  Achieved errors are asserted with explicit tolerances.
"""
import copy
import math
import os

import numpy as np
import pytest
import torch

from oracle import o_models, o_train
from util import close

pytestmark = pytest.mark.gpu


def synth_rays(seed, B, near, far, unit_cube=True, radius=4.0):
  from multinerf_b200 import utils
  rng = np.random.default_rng(seed)
  if unit_cube:
    o = rng.uniform(-1, 1, (B, 3))
    d = rng.normal(size=(B, 3))
    d /= np.linalg.norm(d, axis=-1, keepdims=True)
  else:   # cameras on a sphere looking at the origin (tests/render_test.py:137-143 style)
    o = rng.normal(size=(B, 3))
    o = o / np.linalg.norm(o, axis=-1, keepdims=True) * radius
    d = -o / radius + rng.normal(size=(B, 3)) * 0.1
    d /= np.linalg.norm(d, axis=-1, keepdims=True)
  v = d.copy()
  d = d * rng.uniform(0.8, 1.2, (B, 1))
  f = np.float32
  return utils.Rays(origins=o.astype(f), directions=d.astype(f), viewdirs=v.astype(f),
                    radii=rng.uniform(5e-4, 1e-3, (B, 1)).astype(f),
                    imageplane=np.zeros((B, 2), f), lossmult=np.ones((B, 1), f),
                    near=np.full((B, 1), near, f), far=np.full((B, 1), far, f),
                    cam_idx=np.zeros((B, 1), np.int32)), rng


def mini360():
  from multinerf_b200 import configs
  b = configs.bundle_360()
  b.model.num_prop_samples = 32
  b.model.num_nerf_samples = 16
  b.prop_mlp.net_depth, b.prop_mlp.net_width = 2, 64
  b.nerf_mlp.net_depth, b.nerf_mlp.net_width = 6, 128
  b.nerf_mlp.bottleneck_width, b.nerf_mlp.net_width_viewdirs = 64, 64
  return b


def plumbing_blender():
  from multinerf_b200 import configs
  b = configs.bundle_blender_256()
  b.model.num_levels = 1
  b.model.num_nerf_samples = 32
  return b


def torch_tree(tree):
  return {k: (torch_tree(v) if isinstance(v, dict) else torch.tensor(v)) for k, v in tree.items()}


class TRays:
  pass


def oracle_rays(rays):
  r = TRays()
  for k, v in rays.__dict__.items():
    setattr(r, k, None if v is None else torch.tensor(np.asarray(v)))
  return r


@pytest.fixture(scope='module')
def mods():
  from multinerf_b200 import lib, models, train_utils
  lib.require_device()
  return models, train_utils


def test_param_counts_known_answers(mods):
  # scripts/generate_tables.ipynb:145 and sibling rows (SURVEY.md fact 3)
  from multinerf_b200 import configs
  models, _ = mods
  assert models.Model(configs.bundle_360()).num_params() == 9007493
  assert models.Model(configs.bundle_blender_256()).num_params() == 835205
  raw = models.Model(configs.bundle_llff_raw())
  assert raw.num_params() + sum(raw.extra_params.values()) == 615740      # generate_tables.ipynb (llff_raw)


@pytest.mark.parametrize('which', ['plumbing', 'mini360'])
def test_model_forward_vs_oracle(mods, which):
  models, _ = mods
  bundle = plumbing_blender() if which == 'plumbing' else mini360()
  B = 64 if which == 'plumbing' else 160
  near, far = (2.0, 6.0) if which == 'plumbing' else (0.2, 1e6)
  rays, rng = synth_rays(0 if which == 'plumbing' else 1, B, near, far, unit_cube=which != 'plumbing')
  model, variables = models.construct_model(2, rays, bundle)
  params = torch_tree(model.export_flax())
  bases = {'nerf': model.plans['NerfMLP_0'].basis,
           'prop': model.plans.get('PropMLP_0', model.plans['NerfMLP_0']).basis}
  orays = oracle_rays(rays)
  sched = model.level_schedule(0.5)[2]
  for randomized in [False, True]:
    rand = None
    if randomized:
      rand = {'jitter': [torch.tensor(rng.uniform(0, 1, (B, 1)).astype(np.float32)) for _ in sched]}
    with torch.no_grad():
      rend_o, hist_o, dbg_o = o_models.model_apply(params, bundle, bases, orays, 0.5, True, rand=rand,
                                                   bf16=True, return_debug=True)
    rend, hist = model(rand, rays, 0.5, True)
    torch.cuda.synchronize()
    # level 0 resamples the trivial [0,1] histogram: identical inputs on both sides
    close(hist[0]['sdist'], hist_o[0]['sdist'], atol=1e-6, rtol=1e-6, msg='level-0 sdist')
    # per-level check with the sample positions pinned to the oracle's
    B_, lv_states = B, model.forward_levels(rand, model._prep_rays(rays), 0.5, True, True)
    r = model._prep_rays(rays)
    from multinerf_b200 import ops
    for i, st in enumerate(lv_states):
      st.sdist.copy_(hist_o[i]['sdist'].cuda())
      model._mlp_forward(st, model.mlps[st.mname], r)
      comp = ops.composite_fwd(st.raw_density, st.raw_rgb, st.sdist, r.directions, r.near_flat, r.far_flat,
                               cfg=st.comp_cfg, want_samples=True, want_extras=True)
      torch.cuda.synchronize()
      dens_o, dens = hist_o[i]['density'], comp['density'].cpu()
      # bf16 tensor-core MLP vs bf16-emulating oracle: state the achieved error
      err = (dens - dens_o).abs() / (1.0 + dens_o.abs())
      assert float(err.max()) < 0.08 and float(err.mean()) < 4e-3, (i, float(err.max()), float(err.mean()))
      close(comp['weights'], hist_o[i]['weights'], atol=2e-2, rtol=0, msg=f'weights level {i}')
      close(comp['rgb'], rend_o[i]['rgb'], atol=1e-2, rtol=0, msg=f'pixel level {i}')
      if st.raw_rgb is not None:
        close(comp['rgb_samples'], hist_o[i]['rgb'], atol=3e-2, rtol=0, msg=f'rgb samples level {i}')
      close(comp['acc'], rend_o[i]['acc'], atol=1e-2, rtol=0, msg=f'acc level {i}')
    # end to end (sample positions drift with the bf16-level differences of earlier levels)
    close(rend[-1]['rgb'], rend_o[-1]['rgb'], atol=2e-2, rtol=0, msg='final pixel end-to-end')
    assert rend[-1]['rgb'].shape == (B, 3) and hist[-1]['weights'].shape == (B, sched[-1]['S'])
    for k in ['acc', 'distance_mean', 'distance_median', 'distance_percentile_5', 'distance_percentile_95',
              'ray_sdist', 'ray_weights', 'ray_rgbs']:
      assert k in rend[-1]


@pytest.mark.parametrize('which,impl', [('mini360', 1), ('mini360', 0), ('plumbing', 0)])
def test_train_step_vs_oracle(mods, which, impl):
  models, train_utils = mods
  from multinerf_b200 import utils
  bundle = plumbing_blender() if which == 'plumbing' else mini360()
  bundle.config.grad_max_norm = 0.0      # compare raw Adam first; clipping is covered below
  B = 64 if which == 'plumbing' else 160
  near, far = (2.0, 6.0) if which == 'plumbing' else (0.2, 1e6)
  rays, rng = synth_rays(3, B, near, far, unit_cube=which != 'plumbing')
  target = rng.uniform(0, 1, (B, 3)).astype(np.float32)
  model, variables = models.construct_model(4, rays, bundle)
  params0 = torch_tree(model.export_flax())
  bases = {'nerf': model.plans['NerfMLP_0'].basis,
           'prop': model.plans.get('PropMLP_0', model.plans['NerfMLP_0']).basis}
  sched = model.level_schedule(0.5)[2]
  rand = {'jitter': [torch.tensor(rng.uniform(0, 1, (B, 1)).astype(np.float32)) for _ in sched]}
  # oracle step (bf16-emulated forward, fp32 autograd)
  opt0 = {'count': 0, 'mu': {}, 'nu': {}}
  new_o, opt_o, stats_o, grads_o = o_train.train_step(params0, opt0, bundle, bases, oracle_rays(rays),
                                                      torch.tensor(target), 0.5, rand=rand, bf16=True)
  step_fn = train_utils.create_train_step(model, bundle.config, impl=impl)
  state = train_utils.TrainState(variables)
  batch = utils.Batch(rays=rays, rgb=target)
  state, stats, _ = step_fn(rand, state, batch, None, 0.5)
  torch.cuda.synchronize()
  stats.materialize()
  close(stats['mses'], stats_o['mses'].detach(), atol=2e-3, rtol=2e-2, msg='mses')
  assert abs(stats['loss'] - float(stats_o['loss'].detach())) < 2e-2 * max(1.0, abs(float(stats_o['loss'].detach())))
  g = model.export_grads_flax()
  worst = 0.0
  for mname in g:
    for lname in g[mname]:
      for leaf in ['kernel', 'bias']:
        a = torch.tensor(g[mname][lname][leaf]).double().flatten()
        b = grads_o[(mname, lname, leaf)].double().flatten()
        if float(b.norm()) == 0.0:            # module unused by this config (e.g. PropMLP at 1 level)
          assert float(a.norm()) == 0.0, (mname, lname, leaf)
          continue
        denom = b.norm().clamp(min=1e-12)
        rel = float((a - b).norm() / denom)
        cos = float((a @ b) / (a.norm() * b.norm()).clamp(min=1e-30))
        worst = max(worst, rel)
        # dY travels between layers in bf16 on both sides (different rounding points): the deepest
        # backward path (Dense_0) accumulates the most; measured 0.09 rel / 0.996 cos on B200
        assert rel < 0.12 and cos > 0.993, (mname, lname, leaf, rel, cos)
  # parameters after one Adam step (first step moves every weight by ~lr regardless of scale)
  newp = model.export_flax()
  lr = o_train.lr_at(0, bundle.config)
  for mname in newp:
    for lname in newp[mname]:
      a = torch.tensor(newp[mname][lname]['kernel'])
      b = new_o[mname][lname]['kernel']
      assert float((a - b).abs().max()) <= 2.1 * lr, (mname, lname)
      agree = ((a - params0[mname][lname]['kernel']).sign() == (b - params0[mname][lname]['kernel']).sign())
      assert float(agree.float().mean()) > 0.95, (mname, lname, float(agree.float().mean()))


def test_cuda_graph_train_step_matches_eager(mods):
  """The captured one-graph step (forward + backward + clip/Adam/repack) must track the eager step
  while train_frac, the learning rate, the Adam bias corrections and the jitter change per step."""
  models, train_utils = mods
  from multinerf_b200 import utils
  bundle = mini360()
  B = 256
  rays, rng = synth_rays(5, B, 0.2, 1e6)
  sched_n = 3
  steps = 5
  batches = [(synth_rays(10 + i, B, 0.2, 1e6)[0], rng.uniform(0, 1, (B, 3)).astype(np.float32)) for i in range(steps)]
  rands = [{'jitter': [torch.tensor(rng.uniform(0, 1, (B,)).astype(np.float32)) for _ in range(sched_n)]}
           for _ in range(steps)]
  results = []
  for use_graph in [False, True]:
    model, variables = models.construct_model(6, rays, bundle)
    step_fn = train_utils.create_train_step(model, bundle.config, use_graph=use_graph)
    state = train_utils.TrainState(variables)
    losses = []
    for i in range(steps):
      r, tgt = batches[i]
      state, stats, _ = step_fn(rands[i], state, utils.Batch(rays=r, rgb=tgt), None, i / 10.0)
      losses.append(stats.materialize()['loss'])
    torch.cuda.synchronize()
    results.append((losses, variables.flat.clone(), variables.step))
    if use_graph:
      assert step_fn.graph_info['state'] == 2 and step_fn.graph_info['launches'] > 20
  (l0, p0, s0), (l1, p1, s1) = results
  assert s0 == s1 == steps
  for a, b in zip(l0, l1):
    assert abs(a - b) < 2e-3 * max(1.0, abs(a)), (l0, l1)
  # fp32 atomics make the two runs differ in the last bits only
  rel = float((p0 - p1).norm() / p0.norm())
  assert rel < 2e-3, rel


def _data_parallel_worker(rank, world, port, q):
  """One rank of the world-2 graph-vs-eager check: its own half of the rays, both ranks on cuda:0."""
  import traceback
  import torch.distributed as dist
  try:
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    from multinerf_b200 import lib, models, train_utils, utils
    lib.require_device()
    torch.cuda.set_device(0)
    bundle = mini360()
    # The global-norm clip sums the gradient norm with fp32 atomics, whose order differs between processes; without
    # it the update is elementwise, so replicas that apply the same all-reduced gradient stay bit-identical.
    bundle.config.grad_max_norm = 0.0
    B, steps = 256, 4
    rays, rng = synth_rays(5, B, 0.2, 1e6)
    shard = lambda x: x[rank * B:(rank + 1) * B]
    batches = [(synth_rays(10 + i, world * B, 0.2, 1e6)[0].map(shard),
                shard(rng.uniform(0, 1, (world * B, 3)).astype(np.float32))) for i in range(steps)]
    rands = [{'jitter': [torch.tensor(shard(rng.uniform(0, 1, (world * B,)).astype(np.float32))) for _ in range(3)]}
             for _ in range(steps)]
    out = {}
    for use_graph in (False, True):
      model, variables = models.construct_model(6, rays, bundle)
      step_fn = train_utils.create_train_step(model, bundle.config, use_graph=use_graph)
      state = train_utils.TrainState(variables)
      losses = []
      for i in range(steps):
        state, stats, _ = step_fn(rands[i], state, utils.Batch(rays=batches[i][0], rgb=batches[i][1]), None, i / 10.0)
        losses.append(stats.materialize()['loss'])
      torch.cuda.synchronize()
      g = step_fn.graph_info
      out[use_graph] = (losses, variables.flat.cpu().numpy(), g['state'], g['opt'] is not None)
    q.put((rank, out, None))
    dist.destroy_process_group()
  except Exception:  # pylint: disable=broad-except
    q.put((rank, None, traceback.format_exc()))


def test_cuda_graph_train_step_world_size_2_matches_eager():
  """Data-parallel step at world size 2 (two processes on one device, gloo all-reduce): the two captured graphs
  (forward + backward | clip + Adam + repack) with the all-reduce between the replays must track the eager step,
  and both ranks must end with the same parameters."""
  import torch.multiprocessing as mp
  ctx = mp.get_context('spawn')
  q = ctx.Queue()
  port = 29900 + os.getpid() % 90
  procs = [ctx.Process(target=_data_parallel_worker, args=(r, 2, port, q)) for r in range(2)]
  for p in procs:
    p.start()
  res = {}
  try:
    for _ in range(2):
      rank, out, err = q.get(timeout=300)
      assert err is None, f'rank {rank}:\n{err}'
      res[rank] = out
  finally:
    for p in procs:
      p.join(60)
      if p.is_alive():             # a rank that failed leaves its peer waiting in a collective
        p.terminate()
  for out in res.values():
    (l0, p0, _, _), (l1, p1, state, two_graphs) = out[False], out[True]
    assert state == 2 and two_graphs
    for a, b in zip(l0, l1):
      assert abs(a - b) < 2e-3 * max(1.0, abs(a)), (l0, l1)
    rel = float(np.linalg.norm(p0 - p1) / np.linalg.norm(p0))
    assert rel < 2e-3, rel
  for use_graph in (False, True):
    np.testing.assert_array_equal(res[0][use_graph][1], res[1][use_graph][1])


def test_cuda_graph_gradients_track_eager_with_moving_weights(mods):
  """Graph replays must read the CURRENT weights everywhere, including the fp32 density-head row the
  NerfMLP dgrad folds in as a rank-1 term (`colv_density`).  A dozen replays at a large learning rate move
  the weights by tens of percent; then ONE more step is taken twice from the same state -- by graph replay
  and by a fresh eager step function -- and the gradients must agree to fp32-atomics noise.  A pointer
  captured to a stale copy of any weight would show up as a gradient error of the size of the drift."""
  models, train_utils = mods
  from multinerf_b200 import utils
  bundle = mini360()
  bundle.config.lr_init = bundle.config.lr_final = 5e-3
  bundle.config.lr_delay_steps = 0
  B, steps = 256, 12
  rays, rng = synth_rays(55, B, 0.2, 1e6)
  batches = [(synth_rays(60 + i, B, 0.2, 1e6)[0], rng.uniform(0, 1, (B, 3)).astype(np.float32))
             for i in range(steps + 1)]
  rands = [{'jitter': [torch.tensor(rng.uniform(0, 1, (B,)).astype(np.float32)) for _ in range(3)]}
           for _ in range(steps + 1)]
  model, variables = models.construct_model(56, rays, bundle)
  d = model.plans['NerfMLP_0'].one('density')
  w0 = model.mlps['NerfMLP_0'].W(d).clone()
  step_fn = train_utils.create_train_step(model, bundle.config, use_graph=True)
  state = train_utils.TrainState(variables)
  for i in range(steps):
    r, tgt = batches[i]
    state, stats, _ = step_fn(rands[i], state, utils.Batch(rays=r, rgb=tgt), None, i / 20.0)
  torch.cuda.synchronize()
  assert step_fn.graph_info['state'] == 2
  w1 = model.mlps['NerfMLP_0'].W(d)
  assert float((w1 - w0).norm() / w0.norm()) > 0.05            # the head really moved
  # the fp32 row handed to the dgrad epilogue is the bf16 rounding of the current master weights
  assert torch.equal(model.mlps['NerfMLP_0'].colv_density[:w1.shape[0]], w1[:, 0].to(torch.bfloat16).float())
  p = variables
  snap = (p.flat.clone(), p.mu.clone(), p.nu.clone(), p.step)
  r, tgt = batches[steps]
  state, _, _ = step_fn(rands[steps], state, utils.Batch(rays=r, rgb=tgt), None, 0.6)      # replay
  torch.cuda.synchronize()
  g_graph = model.export_grads_flax()
  p.flat.copy_(snap[0]); p.mu.copy_(snap[1]); p.nu.copy_(snap[2]); p.step = snap[3]
  for mlp in model.mlps.values():
    mlp.repack()
  eager_fn = train_utils.create_train_step(model, bundle.config, use_graph=False)
  state, _, _ = eager_fn(rands[steps], state, utils.Batch(rays=r, rgb=tgt), None, 0.6)
  torch.cuda.synchronize()
  g_eager = model.export_grads_flax()
  for mname in g_graph:
    for lname in g_graph[mname]:
      a = torch.tensor(g_graph[mname][lname]['kernel']).double().flatten()
      b = torch.tensor(g_eager[mname][lname]['kernel']).double().flatten()
      rel = float((a - b).norm() / b.norm().clamp(min=1e-30))
      assert rel < 5e-3, (mname, lname, rel)


def test_rawnerf_train_step_vs_oracle(mods):
  """BASELINE config 4 (llff_raw.gin) at reduced size: single MLP for both levels, cylinder rays,
  safe_exp colours, per-sample jitter, density noise, exposure scaling with learned offsets, Bayer
  lossmult, rawnerf loss, coarse data loss, value + norm clipping."""
  models, train_utils = mods
  from multinerf_b200 import configs, utils
  bundle = configs.bundle_llff_raw()
  bundle.model.num_prop_samples = bundle.model.num_nerf_samples = 32
  bundle.nerf_mlp.net_width, bundle.nerf_mlp.bottleneck_width, bundle.nerf_mlp.net_width_viewdirs = 128, 64, 64
  bundle.config.grad_max_norm = 0.0
  bundle.config.grad_max_val = 0.0
  B, S = 192, 32
  rng = np.random.default_rng(21)
  f = np.float32
  o = np.concatenate([rng.uniform(-1, 1, (B, 2)), -np.ones((B, 1))], -1)
  d = np.concatenate([rng.uniform(-.5, .5, (B, 2)), 2 * np.ones((B, 1))], -1)
  v = d / np.linalg.norm(d, axis=-1, keepdims=True)
  eidx = rng.integers(0, 4, (B, 1)).astype(np.int32)
  lossmult = np.eye(3, dtype=f)[rng.integers(0, 3, B)]           # Bayer mask: one channel per ray
  rays = utils.Rays(origins=o.astype(f), directions=d.astype(f), viewdirs=v.astype(f),
                    radii=rng.uniform(1e-3, 2e-3, (B, 1)).astype(f), imageplane=np.zeros((B, 2), f),
                    lossmult=lossmult, near=np.zeros((B, 1), f), far=np.ones((B, 1), f),
                    cam_idx=np.zeros((B, 1), np.int32), exposure_idx=eidx,
                    exposure_values=(2.0 ** -eidx).astype(f))
  target = (rng.uniform(0, 1, (B, 3)) ** 2).astype(f)
  model, variables = models.construct_model(8, rays, bundle)
  tree = model.export_flax()
  tree['exposure_scaling_offsets']['embedding'] = rng.normal(size=(1000, 3)).astype(f) * 0.1
  variables = model.init(flax_params=tree)
  params0 = torch_tree(model.export_flax())
  bases = {'nerf': model.plans['NerfMLP_0'].basis, 'prop': model.plans['NerfMLP_0'].basis}
  rand = {'jitter': [torch.tensor(rng.uniform(0, 1, (B, S)).astype(f)) for _ in range(2)],
          'density_noise': [torch.tensor(rng.normal(size=(B, S)).astype(f)) for _ in range(2)]}
  opt0 = {'count': 0, 'mu': {}, 'nu': {}}
  new_o, opt_o, stats_o, grads_o = o_train.train_step(params0, opt0, bundle, bases, oracle_rays(rays),
                                                      torch.tensor(target), 0.3, rand=rand, bf16=True)
  step_fn = train_utils.create_train_step(model, bundle.config)
  state = train_utils.TrainState(variables)
  state, stats, _ = step_fn(rand, state, utils.Batch(rays=rays, rgb=target), None, 0.3)
  torch.cuda.synchronize()
  stats.materialize()
  close(stats['mses'], stats_o['mses'].detach(), atol=2e-3, rtol=3e-2, msg='mses')
  lo = float(stats_o['loss'].detach())
  assert abs(stats['loss'] - lo) < 3e-2 * max(1.0, abs(lo)), (stats['loss'], lo)
  g = model.export_grads_flax()
  a = torch.tensor(g['exposure_scaling_offsets']['embedding']).double().flatten()
  b = grads_o[('exposure_scaling_offsets', 'embedding')].double().flatten()
  assert float((a - b).norm() / b.norm()) < 0.05 and float(b.norm()) > 0, float((a - b).norm() / b.norm())
  assert float(a.reshape(-1, 3)[0].abs().max()) == 0.0      # index 0 is pinned (mask = idx > 0)
  for lname in g['NerfMLP_0']:
    a = torch.tensor(g['NerfMLP_0'][lname]['kernel']).double().flatten()
    b = grads_o[('NerfMLP_0', lname, 'kernel')].double().flatten()
    rel = float((a - b).norm() / b.norm().clamp(min=1e-12))
    cos = float((a @ b) / (a.norm() * b.norm()).clamp(min=1e-30))
    assert rel < 0.15 and cos > 0.99, (lname, rel, cos)


def mini_refnerf():
  from multinerf_b200 import configs
  b = configs.Bundle()
  c, m, n = b.config, b.model, b.nerf_mlp
  c.data_loss_type, c.distortion_loss_mult, c.interlevel_loss_mult, c.data_coarse_loss_mult = 'mse', 0.0, 0.0, 0.1
  c.orientation_loss_mult, c.orientation_coarse_loss_mult = 0.1, 0.01
  c.predicted_normal_loss_mult, c.predicted_normal_coarse_loss_mult = 3e-4, 3e-5
  c.adam_eps, c.near, c.far = 1e-8, 2.0, 6.0
  m.num_levels, m.single_mlp, m.num_prop_samples, m.num_nerf_samples = 2, True, 16, 16
  m.anneal_slope, m.dilation_multiplier, m.dilation_bias, m.single_jitter, m.resample_padding = 0., 0., 0., False, 0.01
  n.net_depth, n.net_width, n.net_depth_viewdirs, n.net_width_viewdirs = 6, 128, 6, 64
  n.basis_shape, n.basis_subdivisions, n.disable_density_normals, n.enable_pred_normals = 'octahedron', 1, False, True
  n.use_directional_enc = n.use_reflections = n.enable_pred_roughness = True
  n.use_diffuse_color = n.use_specular_tint = n.use_n_dot_v = True
  n.deg_view, n.bottleneck_width, n.density_bias, n.max_deg_point = 5, 64, 0.5, 16
  return b


def test_refnerf_forward_and_train_step_vs_oracle(mods):
  """BASELINE config 3 (blender_refnerf.gin) at reduced size: IDE of reflected directions, predicted
  and density-gradient normals (forward-mode tangent chain), diffuse + tinted specular colour,
  n.v, 6-layer view MLP with a skip connection, orientation + predicted-normal losses."""
  models, train_utils = mods
  from multinerf_b200 import utils
  bundle = mini_refnerf()
  bundle.config.grad_max_norm = 0.0
  B, S = 96, 16
  rays, rng = synth_rays(7, B, 2.0, 6.0, unit_cube=False)
  target = rng.uniform(0, 1, (B, 3)).astype(np.float32)
  model, variables = models.construct_model(9, rays, bundle)
  params0 = torch_tree(model.export_flax())
  bases = {'nerf': model.plans['NerfMLP_0'].basis, 'prop': model.plans['NerfMLP_0'].basis}
  rand = {'jitter': [torch.tensor(rng.uniform(0, 1, (B, S)).astype(np.float32)) for _ in range(2)]}
  orays = oracle_rays(rays)
  # ---- forward (sample positions pinned to the oracle's per level)
  rend_o, hist_o = o_models.model_apply(params0, bundle, bases, orays, 0.5, True, rand=rand, bf16=True)
  rend_o = [{k: v.detach() for k, v in r.items()} for r in rend_o]
  hist_o = [{k: (v.detach() if v is not None else None) for k, v in h.items()} for h in hist_o]
  r = model._prep_rays(rays)
  from multinerf_b200 import ops
  states = model.forward_levels(rand, r, 0.5, True, True)
  for i, st in enumerate(states):
    st.sdist.copy_(hist_o[i]['sdist'].cuda())
    model._mlp_forward(st, model.mlps[st.mname], r)
    comp = ops.composite_fwd(st.raw_density, st.raw_rgb, st.sdist, r.directions, r.near_flat, r.far_flat,
                             cfg=st.comp_cfg, raw_diffuse=st.heads.get('diffuse'), raw_tint=st.heads.get('tint'),
                             want_samples=True, want_extras=True)
    torch.cuda.synchronize()
    err = (comp['density'].cpu() - hist_o[i]['density']).abs() / (1.0 + hist_o[i]['density'].abs())
    assert float(err.max()) < 0.08 and float(err.mean()) < 4e-3, (i, float(err.max()), float(err.mean()))
    close(st.normals_pred.cpu().view(B, S, 3), hist_o[i]['normals_pred'], atol=3e-2, rtol=0, msg='normals_pred')
    # density normals: bf16 tangent chain vs fp32 autograd of the bf16-emulated forward
    cosn = (st.normals.cpu().view(B, S, 3) * hist_o[i]['normals']).sum(-1)
    assert float((cosn > 0.98).float().mean()) > 0.97, float((cosn > 0.98).float().mean())
    close(st.roughness.cpu().view(B, S, 1), hist_o[i]['roughness'], atol=2e-2, rtol=0, msg='roughness')
    close(comp['rgb_samples'], hist_o[i]['rgb'], atol=4e-2, rtol=0, msg=f'rgb samples level {i}')
    close(comp['rgb'], rend_o[i]['rgb'], atol=1.5e-2, rtol=0, msg=f'pixel level {i}')
  rend, hist = model(rand, rays, 0.5, True)
  for k in ['normals', 'normals_pred', 'roughness']:
    assert k in rend[-1] and hist[-1][k] is not None
  close(rend[-1]['rgb'], rend_o[-1]['rgb'], atol=3e-2, rtol=0, msg='final pixel end-to-end')
  # ---- one train step
  opt0 = {'count': 0, 'mu': {}, 'nu': {}}
  new_o, opt_o, stats_o, grads_o = o_train.train_step(params0, opt0, bundle, bases, orays, torch.tensor(target), 0.5,
                                                      rand=rand, bf16=True)
  step_fn = train_utils.create_train_step(model, bundle.config)
  state = train_utils.TrainState(variables)
  state, stats, _ = step_fn(rand, state, utils.Batch(rays=rays, rgb=target), None, 0.5)
  torch.cuda.synchronize()
  stats.materialize()
  close(stats['mses'], stats_o['mses'].detach(), atol=2e-3, rtol=3e-2, msg='mses')
  for k in ['orientation', 'predicted_normals']:
    lo = float(stats_o['losses'][k].detach())
    assert abs(stats['losses'][k] - lo) < 0.05 * abs(lo) + 1e-7, (k, stats['losses'][k], lo)
  g = model.export_grads_flax()
  report = {}
  for lname in g['NerfMLP_0']:
    a = torch.tensor(g['NerfMLP_0'][lname]['kernel']).double().flatten()
    b = grads_o[('NerfMLP_0', lname, 'kernel')].double().flatten()
    rel = float((a - b).norm() / b.norm().clamp(min=1e-12))
    cos = float((a @ b) / (a.norm() * b.norm()).clamp(min=1e-30))
    report[lname] = (round(rel, 3), round(cos, 4))
  bad = {k: v for k, v in report.items() if not (v[0] < 0.2 and v[1] > 0.98)}
  assert not bad, (bad, report)


def test_weight_decay_random_background_and_bottleneck_noise(mods):
  """Smaller switches of the path: weight_decay_mults (train_utils.py:304-309), random background
  colours (models.py:240-254) and bottleneck noise (models.py:529-533) against the oracle."""
  models, train_utils = mods
  from multinerf_b200 import utils
  bundle = mini360()
  bundle.config.grad_max_norm = 0.0
  bundle.config.weight_decay_mults = {'NerfMLP_0': 1e-3, 'PropMLP_0/Dense_0': 1e-2}
  bundle.model.bg_intensity_range = (0.2, 0.9)
  bundle.nerf_mlp.bottleneck_noise = 0.3
  B = 128
  rays, rng = synth_rays(13, B, 0.2, 1e6)
  target = rng.uniform(0, 1, (B, 3)).astype(np.float32)
  model, variables = models.construct_model(14, rays, bundle)
  params0 = torch_tree(model.export_flax())
  bases = {'nerf': model.plans['NerfMLP_0'].basis, 'prop': model.plans['PropMLP_0'].basis}
  S = [32, 32, 16]
  rand = {'jitter': [torch.tensor(rng.uniform(0, 1, (B, 1)).astype(np.float32)) for _ in S],
          'bg': [torch.tensor(rng.uniform(0, 1, (B, 3)).astype(np.float32)) for _ in S],
          'bottleneck_noise': [torch.tensor(rng.normal(size=(B, s, 64)).astype(np.float32)) for s in S]}
  # deterministic render: midpoint background
  rend_o, _ = o_models.model_apply(params0, bundle, bases, oracle_rays(rays), 0.5, False, rand=None, bf16=True)
  rend, _ = model(None, rays, 0.5, False)
  close(rend[0]['rgb'], rend_o[0]['rgb'].detach(), atol=1e-2, rtol=0, msg='midpoint background')
  opt0 = {'count': 0, 'mu': {}, 'nu': {}}
  new_o, opt_o, stats_o, grads_o = o_train.train_step(params0, opt0, bundle, bases, oracle_rays(rays),
                                                      torch.tensor(target), 0.5, rand=rand, bf16=True)
  step_fn = train_utils.create_train_step(model, bundle.config, use_graph=True)   # falls back to eager
  state = train_utils.TrainState(variables)
  state, stats, _ = step_fn(rand, state, utils.Batch(rays=rays, rgb=target), None, 0.5)
  torch.cuda.synchronize()
  stats.materialize()
  close(stats['mses'], stats_o['mses'].detach(), atol=3e-3, rtol=3e-2, msg='mses (random bg)')
  g = model.export_grads_flax()
  for mname, lname in [('NerfMLP_0', 'Dense_3'), ('PropMLP_0', 'Dense_0'), ('PropMLP_0', 'Dense_1')]:
    a = torch.tensor(g[mname][lname]['kernel']).double().flatten()
    b = grads_o[(mname, lname, 'kernel')].double().flatten()
    assert float((a - b).norm() / b.norm()) < 0.15, (mname, lname, float((a - b).norm() / b.norm()))


def test_glo_embeddings_vs_oracle(mods):
  """configs/360_glo4.gin at reduced size: per-camera GLO vectors appended to the view-MLP input
  (models.py:101-110,565-569), their gradient scattered back into the embedding table."""
  models, train_utils = mods
  from multinerf_b200 import utils
  bundle = mini360()
  bundle.config.grad_max_norm = 0.0
  bundle.model.num_glo_features = 4
  bundle.model.num_glo_embeddings = 16
  B = 128
  rays, rng = synth_rays(17, B, 0.2, 1e6)
  rays.cam_idx = rng.integers(0, 16, (B, 1)).astype(np.int32)
  target = rng.uniform(0, 1, (B, 3)).astype(np.float32)
  model, variables = models.construct_model(18, rays, bundle)
  params0 = torch_tree(model.export_flax())
  assert params0['Embed_0']['embedding'].shape == (16, 4)
  assert params0['NerfMLP_0']['Dense_8']['kernel'].shape[0] == 64 + 27 + 4
  bases = {'nerf': model.plans['NerfMLP_0'].basis, 'prop': model.plans['PropMLP_0'].basis}
  rand = {'jitter': [torch.tensor(rng.uniform(0, 1, (B, 1)).astype(np.float32)) for _ in range(3)]}
  orays = oracle_rays(rays)
  orays.cam_idx = torch.tensor(rays.cam_idx)
  # zero_glo=True (construct/eval default) vs False
  for zero_glo in [True, False]:
    rend_o, _ = o_models.model_apply(params0, bundle, bases, orays, 0.5, False, rand=rand, zero_glo=zero_glo, bf16=True)
    rend, _ = model(rand, rays, 0.5, False, zero_glo=zero_glo)
    close(rend[-1]['rgb'], rend_o[-1]['rgb'].detach(), atol=2e-2, rtol=0, msg=f'pixel zero_glo={zero_glo}')
  opt0 = {'count': 0, 'mu': {}, 'nu': {}}
  new_o, opt_o, stats_o, grads_o = o_train.train_step(params0, opt0, bundle, bases, orays, torch.tensor(target), 0.5,
                                                      rand=rand, bf16=True)
  step_fn = train_utils.create_train_step(model, bundle.config)
  state = train_utils.TrainState(variables)
  state, stats, _ = step_fn(rand, state, utils.Batch(rays=rays, rgb=target), None, 0.5)
  torch.cuda.synchronize()
  g = model.export_grads_flax()
  a = torch.tensor(g['Embed_0']['embedding']).double().flatten()
  b = grads_o[('Embed_0', 'embedding')].double().flatten()
  rel = float((a - b).norm() / b.norm())
  assert float(b.norm()) > 0 and rel < 0.15, rel


def test_full_size_properties(mods):
  """BASELINE size (360.gin: 16384 rays x (64+64+32) samples, PropMLP 4x256, NerfMLP 8x1024), where the
  oracle is too slow: size-independent properties of the path.
    * every level: sdist sorted inside [0,1], weights >= 0 with sum <= 1, colours inside the padded
      sigmoid range, percentiles ordered, everything finite;
    * rays are independent: rendering the batch == rendering its two halves, bit for bit;
    * the loss is a mean over rays: grad(batch) == (grad(half 1) + grad(half 2)) / 2 up to bf16 noise."""
  models, train_utils = mods
  from multinerf_b200 import configs, utils
  bundle = configs.bundle_360()
  B = 16384
  rays, rng = synth_rays(21, B, 0.2, 1e6)
  model, variables = models.construct_model(3, rays, bundle)
  assert model.num_params() == 9007493
  rend, hist = model(None, rays, 1.0, True)
  torch.cuda.synchronize()
  S = [64, 64, 32]
  pad = bundle.nerf_mlp.rgb_padding
  for lvl, (r, h) in enumerate(zip(rend, hist)):
    sd, w = h['sdist'], h['weights']
    assert sd.shape == (B, S[lvl] + 1) and w.shape == (B, S[lvl])
    assert bool((sd[:, 1:] >= sd[:, :-1]).all()) and float(sd.min()) >= 0.0 and float(sd.max()) <= 1.0
    assert float(w.min()) >= 0.0 and float(w.sum(-1).max()) <= 1.0 + 1e-5
    assert bool(torch.isfinite(r['rgb']).all()) and float(r['rgb'].min()) >= -pad - 1e-6 and float(r['rgb'].max()) <= 1 + pad + 1e-6
    assert float(r['acc'].min()) >= 0.0 and float(r['acc'].max()) <= 1.0 + 1e-5
    assert bool((r['distance_percentile_5'] <= r['distance_median'] + 1e-6).all())
    assert bool((r['distance_median'] <= r['distance_percentile_95'] + 1e-6).all())
    assert bool(torch.isfinite(r['distance_mean']).all()) and bool(torch.isfinite(h['density']).all())
  full_rgb = rend[-1]['rgb'].clone()
  full_w = hist[-1]['weights'].clone()
  import dataclasses
  halves = []
  for sl in (slice(0, B // 2), slice(B // 2, B)):
    sub = utils.Rays(**{f.name: (None if getattr(rays, f.name) is None else getattr(rays, f.name)[sl])
                        for f in dataclasses.fields(rays)})
    r2, h2 = model(None, sub, 1.0, True)
    halves.append((r2[-1]['rgb'].clone(), h2[-1]['weights'].clone(), sub))
  assert torch.equal(torch.cat([halves[0][0], halves[1][0]]), full_rgb)
  assert torch.equal(torch.cat([halves[0][1], halves[1][1]]), full_w)

  # gradient of the mean loss = mean of the halves' gradients (same parameters, no optimizer step applied)
  target = rng.uniform(0, 1, (B, 3)).astype(np.float32)
  cfg = copy.deepcopy(bundle.config)
  cfg.lr_init = cfg.lr_final = 1e-30            # keep the parameters (and their bf16 copies) fixed
  jit = [torch.tensor(rng.uniform(0, 1, (B, 1)).astype(np.float32)) for _ in range(3)]
  step_fn = train_utils.create_train_step(model, cfg)
  state = train_utils.TrainState(variables)

  def grad_of(sl):
    sub = utils.Rays(**{f.name: (None if getattr(rays, f.name) is None else getattr(rays, f.name)[sl])
                        for f in dataclasses.fields(rays)})
    nonlocal state
    state, stats, _ = step_fn({'jitter': [j[sl] for j in jit]}, state, utils.Batch(rays=sub, rgb=target[sl]), None, 0.5)
    torch.cuda.synchronize()
    return model.params.grads.clone().double(), stats.materialize()['loss']

  g_full, l_full = grad_of(slice(0, B))
  g1, l1 = grad_of(slice(0, B // 2))
  g2, l2 = grad_of(slice(B // 2, B))
  g_sum = 0.5 * (g1 + g2)
  rel = float((g_full - g_sum).norm() / g_full.norm())
  assert rel < 2e-2, rel
  assert abs(l_full - 0.5 * (l1 + l2)) < 1e-4 * abs(l_full), (l_full, l1, l2)


@pytest.mark.parametrize('B', [1, 37, 130])
def test_ragged_batches_match_their_rows_in_a_full_batch(mods, B):
  """Ragged ray counts (sample rows not a multiple of any tile: TMA zero-fill / store clipping, the
  single-CTA GEMM variant, partial warps): the first B rays rendered alone == the same rays inside a
  256-ray batch, bit for bit; a train step on them stays finite."""
  models, train_utils = mods
  import dataclasses
  from multinerf_b200 import utils
  bundle = mini360()
  rays, rng = synth_rays(8, 256, 0.2, 1e6)
  model, variables = models.construct_model(2, rays, bundle)
  rend, _ = model(None, rays, 1.0, True)
  want = {k: rend[-1][k][:B].clone() for k in ('rgb', 'acc', 'distance_median')}
  sub = utils.Rays(**{f.name: (None if getattr(rays, f.name) is None else getattr(rays, f.name)[:B])
                      for f in dataclasses.fields(rays)})
  r2, h2 = model(None, sub, 1.0, True)
  for k, v in want.items():
    assert torch.equal(r2[-1][k], v), k
  assert h2[-1]['weights'].shape == (B, bundle.model.num_nerf_samples)
  step_fn = train_utils.create_train_step(model, bundle.config)
  state = train_utils.TrainState(variables)
  state, stats, _ = step_fn(None, state, utils.Batch(rays=sub, rgb=rng.uniform(0, 1, (B, 3)).astype(np.float32)), None, 0.3)
  torch.cuda.synchronize()
  assert np.isfinite(stats.materialize()['loss']) and bool(torch.isfinite(model.params.flat).all())


def test_empty_batch(mods):
  """Zero rays: every entry point returns without launching; outputs are empty with the right shapes."""
  models, _ = mods
  import dataclasses
  from multinerf_b200 import utils
  bundle = mini360()
  rays, _ = synth_rays(8, 4, 0.2, 1e6)
  model, _ = models.construct_model(2, rays, bundle)
  empty = utils.Rays(**{f.name: (None if getattr(rays, f.name) is None else getattr(rays, f.name)[:0])
                        for f in dataclasses.fields(rays)})
  rend, hist = model(None, empty, 1.0, True)
  assert rend[-1]['rgb'].shape == (0, 3) and hist[-1]['sdist'].shape == (0, bundle.model.num_nerf_samples + 1)


def _variant(name):
  b = mini360()
  m = b.model
  if name == 'samples_128_128_64':
    m.num_prop_samples, m.num_nerf_samples = 128, 64
  elif name == 'four_levels':
    m.num_levels = 4
  elif name == 'per_sample_jitter':
    m.single_jitter = False
  elif name == 'cylinder':
    m.ray_shape = 'cylinder'
  elif name == 'no_integration':
    # plain PE: without the Gaussian attenuation a random-init MLP of 2^11-frequency features is not a
    # smooth function of the sample positions, so the end-to-end comparison is only well conditioned at
    # low degrees
    m.disable_integration = True
    b.prop_mlp.max_deg_point = b.nerf_mlp.max_deg_point = 5
  elif name == 'no_dilation_padded':
    m.dilation_multiplier, m.dilation_bias, m.resample_padding = 0.0, 0.0, 0.01
  elif name == 'gpu_resampling_flag':
    m.use_gpu_resampling = True
  elif name == 'piecewise_raydist':
    m.raydist_fn = 'piecewise'
  elif name == 'translucent_white_bg':
    m.opaque_background, m.bg_intensity_range = False, (1.0, 1.0)
  elif name == 'coarse_data_loss_mse':
    b.config.data_coarse_loss_mult, b.config.data_loss_type = 0.1, 'mse'
  # ---- MLP switches
  elif name == 'trunk_skip_every_2':            # several skip concatenations in both trunks
    b.nerf_mlp.skip_layer, b.prop_mlp.skip_layer, b.prop_mlp.net_depth = 2, 2, 4
  elif name == 'deep_view_mlp':                 # view MLP with its own skip (models.py:575-580)
    b.nerf_mlp.net_depth_viewdirs, b.nerf_mlp.skip_layer_dir = 4, 2
  elif name == 'degrees_2_to_9_view_deg_2':
    for c in (b.nerf_mlp, b.prop_mlp):
      c.min_deg_point, c.max_deg_point = 2, 9
    b.nerf_mlp.deg_view = 2
  elif name == 'octahedron_basis':
    for c in (b.nerf_mlp, b.prop_mlp):
      c.basis_shape, c.basis_subdivisions = 'octahedron', 1
  elif name == 'icosahedron_1_basis':
    for c in (b.nerf_mlp, b.prop_mlp):
      c.basis_subdivisions = 1
  elif name == 'rgb_head_settings':
    b.nerf_mlp.rgb_premultiplier, b.nerf_mlp.rgb_bias, b.nerf_mlp.rgb_padding = 2.0, -0.5, 0.0
    b.nerf_mlp.density_bias, b.prop_mlp.density_bias = 0.5, 0.5
  elif name == 'glorot_uniform_init':
    b.nerf_mlp.weight_init = b.prop_mlp.weight_init = 'glorot_uniform'
  elif name == 'single_mlp':
    m.single_mlp = True
  else:
    raise KeyError(name)
  return b


@pytest.mark.parametrize('name', ['samples_128_128_64', 'four_levels', 'per_sample_jitter', 'cylinder',
                                  'no_integration', 'no_dilation_padded', 'gpu_resampling_flag',
                                  'piecewise_raydist', 'translucent_white_bg', 'coarse_data_loss_mse',
                                  'trunk_skip_every_2', 'deep_view_mlp', 'degrees_2_to_9_view_deg_2',
                                  'octahedron_basis', 'icosahedron_1_basis', 'rgb_head_settings',
                                  'glorot_uniform_init', 'single_mlp'])
def test_config_variants_vs_oracle(mods, name):
  """Model / Config switches away from the shipped 360.gin values, each against the oracle: rendered
  pixels and level-0 sample positions of a randomized forward pass, then loss, per-level MSEs and the
  direction of every layer's gradient for one train step."""
  models, train_utils = mods
  from multinerf_b200 import utils
  bundle = _variant(name)
  bundle.config.grad_max_norm = 0.0
  B = 96
  near, far = (0.5, 30.0) if name == 'piecewise_raydist' else (0.2, 1e6)
  rays, rng = synth_rays(31, B, near, far)
  target = rng.uniform(0, 1, (B, 3)).astype(np.float32)
  model, variables = models.construct_model(6, rays, bundle)
  params0 = torch_tree(model.export_flax())
  bases = {'nerf': model.plans['NerfMLP_0'].basis,
           'prop': model.plans.get('PropMLP_0', model.plans['NerfMLP_0']).basis}
  sched = model.level_schedule(0.5)[2]
  width = lambda lv: 1 if bundle.model.single_jitter else lv['S']
  rand = {'jitter': [torch.tensor(rng.uniform(0, 1, (B, width(lv))).astype(np.float32)) for lv in sched]}
  with torch.no_grad():
    rend_o, hist_o = o_models.model_apply(params0, bundle, bases, oracle_rays(rays), 0.5, True, rand=rand, bf16=True)
  rend, hist = model(rand, rays, 0.5, True)
  torch.cuda.synchronize()
  assert len(rend) == bundle.model.num_levels
  close(hist[0]['sdist'], hist_o[0]['sdist'], atol=1e-6, rtol=1e-6, msg='level-0 sdist')
  close(rend[-1]['rgb'], rend_o[-1]['rgb'], atol=2e-2, rtol=0, msg='final pixel')
  close(rend[-1]['acc'], rend_o[-1]['acc'], atol=2e-2, rtol=0, msg='final acc')
  opt0 = {'count': 0, 'mu': {}, 'nu': {}}
  _, _, stats_o, grads_o = o_train.train_step(params0, opt0, bundle, bases, oracle_rays(rays), torch.tensor(target),
                                              0.5, rand=rand, bf16=True)
  step_fn = train_utils.create_train_step(model, bundle.config)
  state = train_utils.TrainState(variables)
  state, stats, _ = step_fn(rand, state, utils.Batch(rays=rays, rgb=target), None, 0.5)
  torch.cuda.synchronize()
  stats.materialize()
  close(stats['mses'], stats_o['mses'].detach(), atol=2e-3, rtol=3e-2, msg='mses')
  lo = float(stats_o['loss'].detach())
  assert abs(stats['loss'] - lo) < 3e-2 * max(1.0, abs(lo)), (stats['loss'], lo)
  g = model.export_grads_flax()
  for mname in g:
    for lname in g[mname]:
      a = torch.tensor(g[mname][lname]['kernel']).double().flatten()
      b = grads_o[(mname, lname, 'kernel')].double().flatten()
      if float(b.norm()) == 0.0:
        assert float(a.norm()) == 0.0, (mname, lname)
        continue
      cos = float((a @ b) / (a.norm() * b.norm()).clamp(min=1e-30))
      rel = float((a - b).norm() / b.norm())
      assert cos > 0.98 and rel < 0.25, (name, mname, lname, cos, rel)


def _refnerf_variant(name):
  b = mini_refnerf()
  c, n = b.config, b.nerf_mlp
  if name == 'pred_normals_only':
    n.disable_density_normals = True
    c.predicted_normal_loss_mult = c.predicted_normal_coarse_loss_mult = 0.0
  elif name == 'density_normals_only':
    n.enable_pred_normals = False
    c.orientation_loss_target = 'normals'
    c.predicted_normal_loss_mult = c.predicted_normal_coarse_loss_mult = 0.0
  elif name == 'reflections_with_plain_pe':
    n.use_directional_enc, n.deg_view = False, 4
  elif name == 'no_diffuse_no_tint_no_ndotv':
    n.use_diffuse_color = n.use_specular_tint = n.use_n_dot_v = False
  else:
    raise KeyError(name)
  return b


@pytest.mark.parametrize('name', ['pred_normals_only', 'density_normals_only', 'reflections_with_plain_pe',
                                  'no_diffuse_no_tint_no_ndotv'])
def test_refnerf_variants_vs_oracle(mods, name):
  """Ref-NeRF switches one at a time (models.py:473-604): which normals feed the reflection and the
  orientation loss, IDE vs plain PE of the (reflected) direction, the colour-composition terms."""
  models, train_utils = mods
  from multinerf_b200 import utils
  bundle = _refnerf_variant(name)
  bundle.config.grad_max_norm = 0.0
  B, S = 96, 16
  rays, rng = synth_rays(17, B, 2.0, 6.0, unit_cube=False)
  target = rng.uniform(0, 1, (B, 3)).astype(np.float32)
  model, variables = models.construct_model(5, rays, bundle)
  params0 = torch_tree(model.export_flax())
  bases = {'nerf': model.plans['NerfMLP_0'].basis, 'prop': model.plans['NerfMLP_0'].basis}
  rand = {'jitter': [torch.tensor(rng.uniform(0, 1, (B, S)).astype(np.float32)) for _ in range(2)]}
  orays = oracle_rays(rays)
  rend_o, hist_o = o_models.model_apply(params0, bundle, bases, orays, 0.5, True, rand=rand, bf16=True)
  rend, hist = model(rand, rays, 0.5, True)
  torch.cuda.synchronize()
  close(rend[-1]['rgb'], rend_o[-1]['rgb'].detach(), atol=3e-2, rtol=0, msg='final pixel')
  opt0 = {'count': 0, 'mu': {}, 'nu': {}}
  _, _, stats_o, grads_o = o_train.train_step(params0, opt0, bundle, bases, orays, torch.tensor(target), 0.5,
                                              rand=rand, bf16=True)
  step_fn = train_utils.create_train_step(model, bundle.config)
  state = train_utils.TrainState(variables)
  state, stats, _ = step_fn(rand, state, utils.Batch(rays=rays, rgb=target), None, 0.5)
  torch.cuda.synchronize()
  stats.materialize()
  close(stats['mses'], stats_o['mses'].detach(), atol=2e-3, rtol=3e-2, msg='mses')
  lo = float(stats_o['losses']['orientation'].detach())
  assert abs(stats['losses']['orientation'] - lo) < 0.05 * abs(lo) + 1e-7, (stats['losses']['orientation'], lo)
  g = model.export_grads_flax()
  bad = {}
  for lname in g['NerfMLP_0']:
    a = torch.tensor(g['NerfMLP_0'][lname]['kernel']).double().flatten()
    b = grads_o[('NerfMLP_0', lname, 'kernel')].double().flatten()
    if float(b.norm()) == 0.0:
      assert float(a.norm()) == 0.0, lname
      continue
    rel = float((a - b).norm() / b.norm())
    cos = float((a @ b) / (a.norm() * b.norm()).clamp(min=1e-30))
    # with density-gradient normals alone, every colour gradient reaches the first layers through the
    # bf16 forward-mode tangent streams as well: measured 0.24 / 0.971 on Dense_0
    lim_rel, lim_cos = (0.3, 0.96) if name == 'density_normals_only' else (0.25, 0.98)
    if not (rel < lim_rel and cos > lim_cos):
      bad[lname] = (round(rel, 3), round(cos, 4))
  assert not bad, bad
  if name == 'reflections_with_plain_pe':
    broken = _refnerf_variant(name)
    broken.nerf_mlp.use_directional_enc, broken.nerf_mlp.use_reflections = True, False
    with pytest.raises(ValueError):
      models.Model(broken)


def _family(name, rng, B):
  """(bundle, rays, per-level jitter width) of a reduced-size model family with per-step varying inputs."""
  from multinerf_b200 import configs, utils
  f = np.float32
  if name == 'rawnerf':
    bundle = configs.bundle_llff_raw()
    bundle.model.num_prop_samples = bundle.model.num_nerf_samples = 32
    bundle.nerf_mlp.net_width, bundle.nerf_mlp.bottleneck_width, bundle.nerf_mlp.net_width_viewdirs = 128, 64, 64
    bundle.nerf_mlp.density_noise = 0.0           # the graph path refreshes jitter only from a generator or dict
    o = np.concatenate([rng.uniform(-1, 1, (B, 2)), -np.ones((B, 1))], -1)
    d = np.concatenate([rng.uniform(-.5, .5, (B, 2)), 2 * np.ones((B, 1))], -1)
    eidx = rng.integers(0, 4, (B, 1)).astype(np.int32)
    rays = utils.Rays(origins=o.astype(f), directions=d.astype(f),
                      viewdirs=(d / np.linalg.norm(d, axis=-1, keepdims=True)).astype(f),
                      radii=rng.uniform(1e-3, 2e-3, (B, 1)).astype(f), imageplane=np.zeros((B, 2), f),
                      lossmult=np.eye(3, dtype=f)[rng.integers(0, 3, B)], near=np.zeros((B, 1), f),
                      far=np.ones((B, 1), f), cam_idx=np.zeros((B, 1), np.int32), exposure_idx=eidx,
                      exposure_values=(2.0 ** -eidx).astype(f))
    return bundle, rays, [32, 32]
  if name == 'refnerf':
    bundle = mini_refnerf()
    rays, _ = synth_rays(int(rng.integers(1 << 30)), B, 2.0, 6.0, unit_cube=False)
    return bundle, rays, [16, 16]
  if name == 'glo':
    bundle = mini360()
    bundle.model.num_glo_features, bundle.model.num_glo_embeddings = 4, 16
    rays, _ = synth_rays(int(rng.integers(1 << 30)), B, 0.2, 1e6)
    rays.cam_idx = rng.integers(0, 16, (B, 1)).astype(np.int32)
    return bundle, rays, [1, 1, 1]
  raise KeyError(name)


@pytest.mark.parametrize('family', ['rawnerf', 'refnerf', 'glo'])
def test_cuda_graph_matches_eager_other_families(mods, family):
  """Graph capture of the step for the other model families (exposure-offset and GLO scatter-adds, the
  Ref-NeRF tangent chain and reflection stage): five steps with changing rays, targets, jitter,
  train_frac and learning rate track the eager run."""
  models, train_utils = mods
  from multinerf_b200 import utils
  B, steps = 192, 5
  rng = np.random.default_rng(77)
  batches = []
  for _ in range(steps):
    bundle, rays, widths = _family(family, rng, B)
    rand = {'jitter': [torch.tensor(rng.uniform(0, 1, (B, w)).astype(np.float32)) for w in widths]}
    batches.append((rays, rng.uniform(0, 1, (B, 3)).astype(np.float32), rand))
  results = []
  for use_graph in [False, True]:
    model, variables = models.construct_model(6, batches[0][0], bundle)
    step_fn = train_utils.create_train_step(model, bundle.config, use_graph=use_graph)
    state = train_utils.TrainState(variables)
    losses = []
    for i, (rays, tgt, rand) in enumerate(batches):
      state, stats, _ = step_fn(rand, state, utils.Batch(rays=rays, rgb=tgt), None, i / 10.0)
      losses.append(stats.materialize()['loss'])
    torch.cuda.synchronize()
    results.append((losses, variables.flat.clone()))
    if use_graph:
      assert step_fn.graph_info['state'] == 2, step_fn.graph_info['state']
  (l0, p0), (l1, p1) = results
  for a, b in zip(l0, l1):
    assert abs(a - b) < 2e-3 * max(1.0, abs(a)), (l0, l1)
  assert float((p0 - p1).norm() / p0.norm()) < 2e-3
