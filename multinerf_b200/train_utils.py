"""Train-step closure and render function over the CUDA hot path.

Keeps the reference's surface (internal/train_utils.py):
  setup_model(config, rng, dataset=None) -> (model, state, render_eval_pfn, train_pstep, lr_fn)
                                                                train_utils.py:399-419
  train_pstep(rngs, state, batch, cameras, train_frac, loss_threshold) -> (state, stats, rngs)
                                                                train_utils.py:239-346
  render_eval_pfn(variables, train_frac, _, rays)               train_utils.py:377-396
The reference runs one process with `jax.pmap`; here it is one process per GPU
(`torchrun`), rays pre-sharded per rank, and the two collectives of the path are
NCCL: all-reduce(mean) of the flat gradient (pmean, train_utils.py:319-321) and
all-gather of the rendered pixels (train_utils.py:380-388).
"""
import math

import torch
import torch.distributed as dist

from . import camera_utils
from . import configs
from . import models
from . import ops
from . import utils


def learning_rate_decay(step, lr_init, lr_final, max_steps, lr_delay_steps=0, lr_delay_mult=1):
  """internal/math.py:66-98 (host scalar)."""
  if lr_init <= 0 or lr_final <= 0:
    raise ValueError(f'Interpolants {lr_init} and {lr_final} must be positive.')
  if lr_delay_steps > 0:
    delay_rate = lr_delay_mult + (1 - lr_delay_mult) * math.sin(
        0.5 * math.pi * min(max(step / lr_delay_steps, 0.0), 1.0))
  else:
    delay_rate = 1.0
  t = min(max(step / max_steps, 0.0), 1.0)
  return delay_rate * math.exp(t * (math.log(lr_final) - math.log(lr_init)) + math.log(lr_init))


def _world():
  if dist.is_available() and dist.is_initialized():
    return dist.get_world_size(), dist.get_rank()
  return 1, 0


class TrainState:
  """Counterpart of flax TrainState: step counter + params + Adam moments (all in `params`)."""

  def __init__(self, params):
    self.params = params

  @property
  def step(self):
    return self.params.step


STAT_NAMES = ('data', 'mse', 'distortion', 'interlevel')


def _anneal(mcfg, train_frac):
  if mcfg.anneal_slope > 0:
    sl = mcfg.anneal_slope
    return (sl * train_frac) / ((sl - 1) * train_frac + 1)
  return 1.0


def create_train_step(model: models.Model, config: configs.Config, impl=0, use_graph=False, dataset=None):
  """Returns train_pstep (train_utils.py:221-346) for this rank's shard of the batch.

  With `config.cast_rays_in_train_step`, `batch.rays` is a utils.Pixels and the rays are generated
  on the device from `cameras` first (train_utils.py:266-268; camera type from `dataset.camtype`
  as train_utils.py:234-237).

  use_graph=True captures the step after one eager warm-up step: into ONE CUDA graph on a single GPU
  (forward + backward + clip/Adam/repack), into TWO when data-parallel (forward + backward | clip +
  Adam + repack, with the NCCL all-reduce between the replays); per-step scalars
  (annealing exponent, learning rate, Adam bias corrections) and the jitter draws live in device
  buffers that are refreshed before each replay, so train_frac and the step count may advance.
  """
  mcfg = model.mcfg
  camtype = getattr(dataset, 'camtype', camera_utils.ProjectionType.PERSPECTIVE)
  if config.data_loss_type not in ('mse', 'charb', 'rawnerf'):
    raise NotImplementedError(f'data_loss_type {config.data_loss_type!r}')
  if use_graph and (mcfg.near_anneal_rate is not None or
                    mcfg.bg_intensity_range[0] != mcfg.bg_intensity_range[1] or
                    any(p.cfg.bottleneck_noise > 0 for p in model.plans.values())):
    use_graph = False          # init_s_near by value / extra random draws: stay eager
  # weight decay (train_utils.py:304-309): 'Module' or 'Module/Dense_k' -> multiplier on ||.||^2
  decay_views = []
  for key, mult in dict(config.weight_decay_mults).items():
    parts = key.split('/')
    if parts[0] not in model.plans or len(parts) > 2:
      raise ValueError(f'weight_decay_mults: unknown parameter subtree {key!r}')
    decay_views.append((parts[0], parts[1] if len(parts) == 2 else None, float(mult)))
  dev = model.device
  if mcfg.num_levels * 8 > models.Params.STATS_TAIL:
    raise ValueError(f'num_levels {mcfg.num_levels} > {models.Params.STATS_TAIL // 8}')

  def stats_view(params):
    # the loss accumulators ride in the tail of the flat gradient buffer: one collective per step
    return params.stats_tail[:mcfg.num_levels * 8].view(mcfg.num_levels, 8)
  scratch = torch.zeros(4, device=dev)
  dyn = torch.zeros(4, device=dev)               # lr, 1-b1^t, 1-b2^t, annealing exponent: ONE H2D copy per step
  # Pinned staging ring for the per-step scalars: the host may run several graph replays ahead of the
  # device, so a slot is rewritten only after the H2D copy that last read it has completed (event).
  DYN_SLOTS = 8
  dyn_host = [torch.zeros(4).pin_memory() for _ in range(DYN_SLOTS)]
  dyn_events = [None] * DYN_SLOTS
  anneal_dev = dyn[3:4]
  G = {'state': 0, 'fb': None, 'opt': None, 'rays': None, 'target': None, 'jitter': None,
       'noise': None, 'launches': 0}
  def fb_begin(rng, rays, target, train_frac, anneal_ptr):
    """Zero the gradients, run the forward pass of every level; returns the context of the backward pass."""
    params = model.params
    lossmult = rays.lossmult
    if config.disable_multiscale_loss:
      lossmult = torch.ones_like(lossmult)
    lm_ch = lossmult.shape[-1]
    inv_denom = (1.0 / (lossmult.sum() * (3 if lm_ch == 1 else 1))).reshape(1)
    params.grads_ext.zero_()
    states = model.forward_levels(rng if config.randomized else None, rays, train_frac,
                                  compute_extras=False, want_samples=False, impl=impl,
                                  anneal_dev=anneal_ptr, loss_config=config, zero_glo=False)
    return dict(params=params, states=states, rays=rays, target=target, lossmult=lossmult, inv_denom=inv_denom,
                stats=stats_view(params))

  def fb_level(ctx, i):
    """Losses + backward of level i (accumulates parameter gradients)."""
    params, states, rays = ctx['params'], ctx['states'], ctx['rays']
    st, fine, n = states[i], states[-1], len(states)
    is_fine = i == n - 1
    ops.composite_bwd(
        st.raw_density, st.raw_rgb, st.sdist, rays.directions, rays.near_flat, rays.far_flat,
        ctx['target'], ctx['lossmult'], ctx['inv_denom'], ctx['stats'][i], cfg=st.comp_cfg,
        loss_type=config.data_loss_type, charb_padding=config.charb_padding,
        data_mult=config.data_loss_mult if is_fine else config.data_coarse_loss_mult,
        distortion_mult=config.distortion_loss_mult if is_fine else 0.0,
        interlevel_mult=0.0 if is_fine else config.interlevel_loss_mult,
        sdist_fine=None if is_fine else fine.sdist,
        weights_fine=None if is_fine else fine.comp['weights'],
        density_noise=st.noise, bg_rgb=st.bg_rgb, rgb_scale=st.rgb_scale, d_raw_density=st.d_raw_density,
        d_raw_rgb=st.d_raw_rgb, d_rgb_scale=_d_scale_buf(st),
        raw_diffuse=st.heads.get('diffuse'), raw_tint=st.heads.get('tint'),
        extra_dw=st.extra_dw if st.loss_mults is not None else None,
        d_raw_diffuse=st.d_heads.get('diffuse'), d_raw_tint=st.d_heads.get('tint'))
    if st.rgb_scale is not None and mcfg.learned_exposure_scaling:
      # d offsets[idx] += [idx > 0] * exposure_values * d_scale   (adjoint of models.py:262-267)
      eidx = rays.exposure_idx[:, 0].long()
      g = (eidx > 0).to(torch.float32)[:, None] * rays.exposure_values * st.d_rgb_scale
      params.seg('exposure_scaling_offsets', params.grads).view(-1, 3).index_add_(0, eidx, g)
    model._mlp_backward(st, model.mlps[st.mname], rays=rays, impl=impl, loss_mults=st.loss_mults,
                        stats=ctx['stats'][i])

  def fwd_bwd(rng, rays, target, train_frac, anneal_ptr):
    """Forward, backward last level to first, weight decay: the parameter gradients of this rank's shard."""
    ctx = fb_begin(rng, rays, target, train_frac, anneal_ptr)
    for i in range(len(ctx['states']) - 1, -1, -1):
      fb_level(ctx, i)
    if decay_views:
      weight_decay()

  def weight_decay():
    # loss += mult * sum(w^2)  ->  grad += 2 mult w ; the loss value goes to stats row 0, slot 6
    params = model.params
    for mname, lname, mult in decay_views:
      mlp = model.mlps[mname]
      for sp in mlp.plan.specs:
        if lname is None or sp.name == lname:
          for view_p, view_g in ((mlp.W(sp), mlp.W(sp, mlp.grads)), (mlp.b(sp), mlp.b(sp, mlp.grads))):
            view_g.add_(view_p, alpha=2.0 * mult)
            stats_view(params)[0, 6] += mult * (view_p * view_p).sum()

  def _d_scale_buf(st):
    if st.rgb_scale is None:
      return None
    if getattr(st, 'd_rgb_scale', None) is None or st.d_rgb_scale.shape[0] != st.B:
      st.d_rgb_scale = torch.empty(st.B, 3, device=dev)
    return st.d_rgb_scale

  def optim(grad_scale, step, lr, dyn_ptr):
    params = model.params
    for name in list(model.plans) + list(model.extra_params):
      ops.clip_adam(params.seg(name), params.seg(name, params.grads), params.seg(name, params.mu),
                    params.seg(name, params.nu), scratch, step=step, lr=lr,
                    beta1=config.adam_beta1, beta2=config.adam_beta2, eps=config.adam_eps,
                    grad_max_val=config.grad_max_val, grad_max_norm=config.grad_max_norm,
                    grad_scale=grad_scale, dyn=dyn_ptr)
    for mlp in model.mlps.values():
      mlp.repack()

  def set_dyn(step, lr, anneal=1.0):
    slot = G['dyn_slot'] = (G.get('dyn_slot', -1) + 1) % DYN_SLOTS
    if dyn_events[slot] is not None:
      dyn_events[slot].synchronize()
    h = dyn_host[slot]
    h[0] = lr
    h[1] = 1.0 - config.adam_beta1 ** step
    h[2] = 1.0 - config.adam_beta2 ** step
    h[3] = anneal
    dyn.copy_(h, non_blocking=True)
    if dyn_events[slot] is None:
      dyn_events[slot] = torch.cuda.Event()
    dyn_events[slot].record()

  def draw_randomness(rng, B, sched):
    """Explicit draws for this step (the reference splits a threefry key per level)."""
    if rng is None or not config.randomized:
      return None
    jit = G['jitter']
    if jit is None:
      # all levels' draws live in one flat buffer each: one RNG launch per step instead of one per level
      def views(shapes):
        sizes = [int(torch.Size(sh).numel()) for sh in shapes]
        flat = torch.empty(sum(sizes), device=dev)
        out, o = [], 0
        for sh, n_ in zip(shapes, sizes):
          out.append(flat[o:o + n_].view(sh))
          o += n_
        return flat, out
      G['jitter_flat'], jit = views([(B,) if mcfg.single_jitter else (B, lv['S']) for lv in sched])
      G['jitter'] = jit
      G['noise_flat'], G['noise'] = views([(B, lv['S']) for lv in sched])
    out = {'jitter': jit}
    need_noise = any(p.cfg.density_noise > 0 for p in model.plans.values())
    if isinstance(rng, dict):        # explicit draws: stage them in the static buffers
      for t, src in zip(jit, rng['jitter']):
        t.copy_(torch.as_tensor(src).to(dev).reshape(t.shape), non_blocking=True)
      if need_noise:
        for t, src in zip(G['noise'], rng['density_noise']):
          t.copy_(torch.as_tensor(src).to(dev).reshape(t.shape), non_blocking=True)
    else:
      G['jitter_flat'].uniform_(0.0, 1.0, generator=rng)
      if need_noise:
        G['noise_flat'].normal_(0.0, 1.0, generator=rng)
    if need_noise:
      out['density_noise'] = G['noise']
    return out

  def train_step(rng, state, batch, cameras, train_frac, loss_threshold=1.0):
    world, _ = _world()
    params = state.params
    if model.params is not params:
      model.bind(params)
      G['state'] = 0
    rays = batch.rays
    if config.cast_rays_in_train_step:
      if not isinstance(rays, utils.Pixels):
        raise ValueError('cast_rays_in_train_step: batch.rays must be a utils.Pixels')
      if cameras is None:
        raise ValueError('cast_rays_in_train_step: cameras = (pixtocams, camtoworlds, distortion_params, '
                         'pixtocam_ndc) is required')
      rays = camera_utils.cast_ray_batch(cameras, rays, camtype, device=dev)
    rays = rays if hasattr(rays, 'radii_flat') else model._prep_rays(rays)
    B = rays.origins.shape[0]
    target = torch.as_tensor(batch.rgb).to(dev, torch.float32).reshape(B, -1)[:, :3].contiguous()
    sched = model.level_schedule(train_frac)[2]
    n = len(sched)
    grad_scale = 1.0 / world
    params.step += 1
    lr = learning_rate_decay(params.step - 1, config.lr_init, config.lr_final, config.max_steps,
                             config.lr_delay_steps, config.lr_delay_mult)
    if not use_graph or G['state'] == 0:
      # eager step (also the warm-up that allocates every buffer before a capture)
      fwd_bwd(draw_randomness(rng, B, sched) if use_graph else rng, rays, target, train_frac, None)
      allreduce_flat_(params, world)
      optim(grad_scale, params.step, lr, None)
      G['state'] = 1 if use_graph else 0
      G['B'] = B
      return state, LazyStats(stats_view(params).clone(), n, grad_scale), rng
    if G['B'] != B:
      raise ValueError(f'graph mode needs a fixed batch size ({G["B"]} rays per rank), got {B}')
    rand = draw_randomness(rng, B, sched)
    set_dyn(params.step, lr, _anneal(mcfg, train_frac))
    if G['state'] == 1:
      # capture: inputs live in static buffers from now on
      import dataclasses
      G['rays'] = rays
      G['rays'] = type(rays)(**{f.name: (None if getattr(rays, f.name) is None else getattr(rays, f.name).clone())
                                for f in dataclasses.fields(rays)})
      for extra in ('radii_flat', 'near_flat', 'far_flat'):
        setattr(G['rays'], extra, getattr(rays, extra).clone())
      G['target'] = target.clone()
      torch.cuda.synchronize()
      before = ops.LAUNCHES
      G['fb'] = torch.cuda.CUDAGraph()
      with torch.cuda.graph(G['fb']):
        fwd_bwd(rand, G['rays'], G['target'], train_frac, anneal_dev)
        if world == 1:
          optim(grad_scale, params.step, lr, dyn)
      G['opt'] = None
      if world > 1:
        # NCCL stays outside the graphs (capturing the all-reduce hung on torch 2.11 / NCCL 2.28, 2 x B200):
        # the all-reduce runs between the replays of the two graphs
        G['opt'] = torch.cuda.CUDAGraph()
        with torch.cuda.graph(G['opt']):
          optim(grad_scale, params.step, lr, dyn)
      G['launches'] = ops.LAUNCHES - before
      G['state'] = 2
    else:
      import dataclasses
      # one fused multi-tensor copy of the step's inputs into the graph's static buffers
      dsts, srcs = [G['target']], [target]
      for name in [f.name for f in dataclasses.fields(rays)] + ['radii_flat', 'near_flat', 'far_flat']:
        v = getattr(rays, name)
        if v is not None:
          dsts.append(getattr(G['rays'], name))
          srcs.append(v)
      by_dtype = {}
      for d_, s_ in zip(dsts, srcs):
        by_dtype.setdefault((d_.dtype, s_.dtype), ([], []))
        by_dtype[(d_.dtype, s_.dtype)][0].append(d_)
        by_dtype[(d_.dtype, s_.dtype)][1].append(s_)
      for (dd, ss) in by_dtype.values():
        torch._foreach_copy_(dd, ss, non_blocking=True)
    G['fb'].replay()
    if G['opt'] is not None:
      allreduce_flat_(params, world)
      G['opt'].replay()
    ops.LAUNCHES += G['launches']
    return state, LazyStats(stats_view(params).clone(), n, grad_scale), rng

  train_step.graph_info = G
  return train_step


class LazyStats(dict):
  """Reads the step's loss accumulators only when asked (no sync in the step).  `buf` is this step's own
  snapshot of the shared accumulator, so stats kept across steps stay distinct (train.py averages the
  print window)."""

  def __init__(self, buf, n, scale=1.0):
    super().__init__()
    self._buf, self._n, self._scale = buf, n, scale

  def materialize(self):
    b = self._buf.detach().cpu() * self._scale       # pmean of the per-rank stats: SUM all-reduce x 1/world
    mses = b[:, 1].clone()
    losses = {'data': float(b[:, 0].sum()), 'interlevel': float(b[:, 3].sum()),
              'distortion': float(b[:, 2].sum()), 'orientation': float(b[:, 4].sum()),
              'predicted_normals': float(b[:, 5].sum())}
    if float(b[:, 6].abs().sum()) > 0:
      losses['weight'] = float(b[:, 6].sum())
    self.update(mses=mses, psnrs=-10.0 / math.log(10.0) * torch.log(mses), losses=losses,
                loss=sum(losses.values()))
    self['psnr'] = float(self['psnrs'][-1])
    return self


def gather_renderings(renderings, world, all_levels=False):
  """all_gather of the per-pixel buffers (lax.all_gather, train_utils.py:380-388) as ONE collective per
  chunk: the per-pixel outputs of a level are packed into one [rays, C] fp32 buffer, gathered with a
  single all_gather_into_tensor and unpacked (rank r's rows land at [r*n, (r+1)*n)).  `ray_*`
  visualisation bundles stay local.  The reference gathers every level and render_image then keeps
  only the last one (models.py:689-694); here only the last level travels unless `all_levels`."""
  if world <= 1:
    return renderings
  out = []
  for i, r in enumerate(renderings):
    if not all_levels and i != len(renderings) - 1:
      out.append({k: v for k, v in r.items() if k.startswith('ray_')})
      continue
    keys = [k for k in r if not k.startswith('ray_')]
    g = {k: v for k, v in r.items() if k.startswith('ray_')}
    if keys:
      n = r[keys[0]].shape[0]
      cols = [r[k].reshape(n, -1).to(torch.float32) for k in keys]
      widths = [c.shape[1] for c in cols]
      packed = torch.cat(cols, 1).contiguous()
      buf = torch.empty(world * n, packed.shape[1], device=packed.device, dtype=packed.dtype)
      dist.all_gather_into_tensor(buf, packed)
      c0 = 0
      for k, w in zip(keys, widths):
        g[k] = buf[:, c0:c0 + w].reshape((world * n,) + tuple(r[k].shape[1:])).to(r[k].dtype)
        c0 += w
    out.append(g)
  return out


def allreduce_flat_(params, world):
  """pmean of gradients and stats as ONE collective over the flat buffer (gradients + stats tail); the
  1/world factor is applied downstream (clip_adam grad_scale, LazyStats scale)."""
  if world > 1:
    dist.all_reduce(params.grads_ext, op=dist.ReduceOp.SUM)
  return 1.0 / world


def create_render_fn(model: models.Model, use_graph=False):
  """render_eval_pfn(variables, train_frac, _, rays): deterministic render of this rank's rays,
  with the per-rank pixel buffers all-gathered (train_utils.py:377-396).

  use_graph=True replays one captured CUDA graph per (chunk size, train_frac): a full image is ~100 chunks
  of the same shape, and at 8 GPUs a 16384-ray chunk leaves 2048 rays per rank, where the ~45 launches of
  a forward pass cost more host time than device time.  Ragged chunks (the last one) run eagerly."""
  import dataclasses
  G = {}

  def render_eval_fn(variables, train_frac, _, rays):
    world, rank = _world()
    if variables is not model.params:
      model.bind(variables)
      G.clear()
    if not use_graph:
      renderings, ray_history = model.apply(variables, None, rays, train_frac=train_frac, compute_extras=True)
      return gather_renderings(renderings, world), ray_history
    r = model._prep_rays(rays)
    B = r.origins.shape[0]
    lead = tuple(rays.origins.shape[:-1])
    key = (B, float(train_frac), lead)
    ent = G.get(key)
    if ent is None:
      # first sight of this shape: eager (allocates the level buffers); capture on the second
      G[key] = {'graph': None}
      renderings, ray_history = model.call_prepped(None, r, lead, train_frac, True)
      return gather_renderings(renderings, world), ray_history
    fields = [f.name for f in dataclasses.fields(r) if getattr(r, f.name) is not None] + \
        ['radii_flat', 'near_flat', 'far_flat']
    if ent['graph'] is None:
      ent['rays'] = type(r)(**{f.name: (None if getattr(r, f.name) is None else getattr(r, f.name).clone())
                               for f in dataclasses.fields(r)})
      for extra in ('radii_flat', 'near_flat', 'far_flat'):
        setattr(ent['rays'], extra, getattr(r, extra).clone())
      torch.cuda.synchronize()
      before = ops.LAUNCHES
      ent['graph'] = torch.cuda.CUDAGraph()
      with torch.cuda.graph(ent['graph']):
        ent['out'] = model.call_prepped(None, ent['rays'], lead, train_frac, True)
      ent['launches'] = ops.LAUNCHES - before
    else:
      for name in fields:
        getattr(ent['rays'], name).copy_(getattr(r, name), non_blocking=True)
    ent['graph'].replay()
    ops.LAUNCHES += ent['launches']
    renderings, ray_history = ent['out']
    # static output buffers are overwritten by the next replay: hand out copies of what render_image keeps
    # (the last level's pixels -- for world > 1 the gather itself copies them -- and the ray_* bundles)
    last = len(renderings) - 1
    renderings = [{k: (v.clone() if (world == 1 or k.startswith('ray_')) else v) for k, v in rr.items()
                   if i == last or k.startswith('ray_')} for i, rr in enumerate(renderings)]
    return gather_renderings(renderings, world), ray_history

  return render_eval_fn


def create_optimizer(config, variables):
  lr_fn = lambda step: learning_rate_decay(step, config.lr_init, config.lr_final, config.max_steps,
                                           config.lr_delay_steps, config.lr_delay_mult)
  return TrainState(variables), lr_fn


def setup_model(config, rng, dataset=None, device=None):
  """train_utils.py:399-419.  `config` is a configs.Bundle (Config + Model + MLP bindings)."""
  bundle = config if isinstance(config, configs.Bundle) else configs.Bundle(config=config)
  dummy = utils.dummy_rays(include_exposure_idx=bundle.config.rawnerf_mode,
                           include_exposure_values=True)
  model, variables = models.construct_model(rng, dummy, bundle, device=device)
  state, lr_fn = create_optimizer(bundle.config, variables)
  render_eval_pfn = create_render_fn(model)
  train_pstep = create_train_step(model, bundle.config, dataset=dataset)
  return model, state, render_eval_pfn, train_pstep, lr_fn
