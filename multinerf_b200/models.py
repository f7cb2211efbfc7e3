"""Host side of the hot path: `Model.__call__` / `render_image` over the sm_100a kernels.

Keeps the reference's surface (internal/models.py):
  Model.__call__(rng, rays, train_frac, compute_extras, zero_glo) -> (renderings, ray_history)
                                                      models.py:75-312
  construct_model(rng, rays, config) -> (model, variables)    models.py:315-338
  render_image(render_fn, rays, rng, config)                  models.py:625-706
Python only orchestrates: per level it launches resample -> cast+IPE -> Dense chain (tcgen05)
-> heads -> compositing; the backward chain mirrors it (train_utils.py:239-339 closure lives
in multinerf_b200/train_utils.py).  PyTorch provides device buffers, streams and RNG draws.
There is no CPU path: constructing a Model without a B200 raises.
"""
import dataclasses
import math
from typing import Any, Dict, List, Optional

import numpy as np
import torch

from . import configs
from . import geopoly
from . import lib as L
from . import ops
from . import utils


def _pad64(n):
  return (n + 63) // 64 * 64


@dataclasses.dataclass
class DenseSpec:
  """One nn.Dense of the reference MLP (creation order = flax auto-name Dense_k)."""
  name: str
  role: str            # trunk | density | bottleneck | view | rgb
  in_dim: int          # logical inputs (flax kernel rows)
  in_pad: int          # rows of the padded master / K of the GEMM
  out_dim: int
  head: bool           # True: narrow head kernel, False: tcgen05 GEMM
  act: int = L.ACT_NONE
  # row map: logical flax row -> padded master row (skip-concat / view-input padding)
  row_map: Optional[np.ndarray] = None
  w_off: int = 0       # offsets (floats) into the module's flat master buffer
  b_off: int = 0


class MLPPlan:
  """Static layout of one MLP: layer table (flax creation order), buffer widths, flat offsets."""

  HEAD_SLOTS = {'density': (0, 1), 'grad_pred': (1, 3), 'diffuse': (4, 3), 'tint': (7, 3),
                'roughness': (10, 1)}     # column slots of the head-gradient slab (csrc/refnerf.cu)

  def __init__(self, cfg: configs.MLPConfig, use_viewdirs=True, glo_features=0):
    cfg.validate()
    self.glo_features = glo_features
    if cfg.net_activation != 'relu' or cfg.density_activation != 'softplus' or \
       cfg.roughness_activation != 'softplus':
      raise NotImplementedError('CUDA path supports relu trunk / softplus density and roughness')
    if cfg.num_rgb_channels != 3:
      raise NotImplementedError('num_rgb_channels != 3')
    self.cfg = cfg
    self.density_normals = not cfg.disable_density_normals
    self.pred_normals = cfg.enable_pred_normals
    if self.density_normals and cfg.warp_fn is not None:
      raise NotImplementedError('density normals through a contraction warp')
    self.basis = np.ascontiguousarray(
        geopoly.generate_basis(cfg.basis_shape, cfg.basis_subdivisions), dtype=np.float32)
    self.K = self.basis.shape[0]
    self.L = cfg.max_deg_point - cfg.min_deg_point
    self.F = 2 * self.K * self.L
    self.Fpad = _pad64(self.F)
    W = cfg.net_width
    # tensor-core tiling constraints are checked by Model (the table itself is layout-agnostic)
    self.device_constraints = [('net_width', W)]
    specs: List[DenseSpec] = []
    k = 0

    def add(role, in_dim, in_pad, out_dim, head, act=L.ACT_NONE, rm=None):
      nonlocal k
      specs.append(DenseSpec(f'Dense_{k}', role, in_dim, in_pad, out_dim, head, act, rm))
      k += 1
    x_dim, x_pad, x_has_feat = self.F, self.Fpad, False
    self.concat_after = []    # trunk layers whose output is concatenated with the features
    for i in range(cfg.net_depth):
      rm = np.concatenate([np.arange(W), W + np.arange(self.F)]) if x_has_feat else None
      add('trunk', x_dim, x_pad, W, False, L.ACT_RELU, rm)
      if i % cfg.skip_layer == 0 and i > 0:
        self.concat_after.append(i)
        x_dim, x_pad, x_has_feat = W + self.F, W + self.Fpad, True
      else:
        x_dim, x_pad, x_has_feat = W, W, False
    self.last_has_feat = x_has_feat
    self.x_dim, self.x_pad = x_dim, x_pad
    rmx = np.concatenate([np.arange(W), W + np.arange(self.F)]) if x_has_feat else None
    add('density', x_dim, x_pad, 1, True, rm=rmx)
    if self.pred_normals:
      add('grad_pred', x_dim, x_pad, 3, True, rm=rmx)
    self.has_rgb = not cfg.disable_rgb
    self.use_viewdirs = use_viewdirs
    self.ref_stage = False
    if (self.pred_normals or self.density_normals) and not self.has_rgb:
      raise NotImplementedError('normals on an MLP with disable_rgb (no consumer on the CUDA path)')
    if self.has_rgb:
      if not use_viewdirs:
        raise NotImplementedError('use_viewdirs=False with rgb is not wired into the CUDA path')
      if cfg.bottleneck_width <= 0:
        raise NotImplementedError('bottleneck_width == 0 is not supported (models.py:536-554)')
      if cfg.use_diffuse_color:
        add('diffuse', x_dim, x_pad, 3, True, rm=rmx)
      if cfg.use_specular_tint:
        add('tint', x_dim, x_pad, 3, True, rm=rmx)
      if cfg.enable_pred_roughness:
        add('roughness', x_dim, x_pad, 1, True, rm=rmx)
      if cfg.use_directional_enc and not cfg.enable_pred_roughness:
        raise NotImplementedError('IDE without a predicted roughness (kappa_inv would be None)')
      if cfg.use_directional_enc and not cfg.use_reflections:
        # models.py:548-554: dir_enc_fn(viewdirs [..., 3], roughness [..., S, 1]) does not broadcast in the
        # reference either (ref_utils.py:141-148); every shipped config pairs IDE with reflections
        raise ValueError('use_directional_enc needs use_reflections (per-sample roughness cannot attenuate '
                         'the encoding of a per-ray view direction)')
      bw = cfg.bottleneck_width
      self.device_constraints.append(('bottleneck_width', bw))
      add('bottleneck', x_dim, x_pad, bw, False, L.ACT_NONE, rmx)
      self.ref_stage = (self.pred_normals or self.density_normals or cfg.use_reflections or
                        cfg.use_directional_enc or cfg.use_n_dot_v)
      if cfg.use_directional_enc:
        from . import ref_utils
        self.dir_dim = ref_utils.ide_dim(cfg.deg_view)
      else:
        self.dir_dim = 3 + 6 * cfg.deg_view
      self.glo_col0 = bw + self.dir_dim + (1 if cfg.use_n_dot_v else 0)
      vin = self.glo_col0 + glo_features            # [bottleneck | dir enc | n.v | GLO] (models.py:556-572)
      vin_pad = _pad64(vin)
      if self.ref_stage and vin_pad - bw < 11:
        vin_pad += 64
      self.vin_dim, self.vin_pad = vin, vin_pad
      Wv = cfg.net_width_viewdirs
      self.device_constraints.append(('net_width_viewdirs', Wv))
      v_dim, v_pad, v_has_in = vin, vin_pad, False
      self.view_concat_after = []
      for i in range(cfg.net_depth_viewdirs):
        rmv = np.concatenate([np.arange(Wv), Wv + np.arange(vin)]) if v_has_in else None
        add('view', v_dim, v_pad, Wv, False, L.ACT_RELU, rmv)
        if i % cfg.skip_layer_dir == 0 and i > 0:
          self.view_concat_after.append(i)
          v_dim, v_pad, v_has_in = Wv + vin, Wv + vin_pad, True
        else:
          v_dim, v_pad, v_has_in = Wv, Wv, False
      if len(self.view_concat_after) > 1:
        raise NotImplementedError('more than one skip connection inside the view MLP')
      rmv = np.concatenate([np.arange(Wv), Wv + np.arange(vin)]) if v_has_in else None
      if cfg.net_depth_viewdirs == 0:
        raise NotImplementedError('net_depth_viewdirs == 0')
      add('rgb', v_dim, v_pad, cfg.num_rgb_channels, True, rm=rmv)
    off = 0
    for sp in specs:
      sp.w_off = off
      off += sp.in_pad * sp.out_dim
      off = (off + 3) // 4 * 4
      sp.b_off = off
      off += sp.out_dim
      off = (off + 3) // 4 * 4
    self.specs = specs
    self.flat_size = off
    self.num_params = sum(sp.in_dim * sp.out_dim + sp.out_dim for sp in specs)

  def by_role(self, role):
    return [sp for sp in self.specs if sp.role == role]

  def one(self, role):
    r = self.by_role(role)
    return r[0] if r else None


class MLPDevice:
  """Device state of one MLP: fp32 master slice, bf16 shadows, gradient views."""

  def __init__(self, plan: MLPPlan, master, grads, device):
    self.plan = plan
    self.master, self.grads = master, grads           # views into the global flat buffers
    self.device = device
    self.basis = torch.tensor(plan.basis, device=device)
    self.w_nk, self.w_kn, self.colv = {}, {}, {}
    for sp in plan.specs:
      self.w_nk[sp.name] = torch.zeros(sp.out_dim, sp.in_pad, device=device, dtype=torch.bfloat16)
      if not sp.head:
        self.w_kn[sp.name] = torch.zeros(sp.in_pad, sp.out_dim, device=device, dtype=torch.bfloat16)
    self.repack()

  def W(self, s, buf=None):
    buf = self.master if buf is None else buf
    return buf[s.w_off:s.w_off + s.in_pad * s.out_dim].view(s.in_pad, s.out_dim)

  def b(self, s, buf=None):
    buf = self.master if buf is None else buf
    return buf[s.b_off:s.b_off + s.out_dim]

  def repack(self):
    """fp32 master -> bf16 operand layouts (after init and after every optimizer step)."""
    plan = self.plan
    if getattr(self, '_pack_table', None) is None:      # buffers never move: build the device table once
      self._pack_table = ops.pack_table([(self.W(sp), self.w_nk[sp.name], self.w_kn.get(sp.name))
                                         for sp in plan.specs], self.device)
    ops.pack_weights_batched(self._pack_table)
    d = plan.one('density')
    # bf16-rounded, as the fwd used.  Updated IN PLACE: captured CUDA graphs hold this pointer
    # (DGRAD colv / outer_mask), so the tensor must never be re-allocated.
    if getattr(self, 'colv_density', None) is None:
      self.colv_density = torch.zeros(d.in_pad, device=self.device)
    self.colv_density.copy_(self.w_nk[d.name][0])
    if plan.ref_stage:
      # [x_pad, vin_pad] K-major B operand of the trunk-entry dgrad:  [ W_bottleneck | head weights ]
      bt = plan.one('bottleneck')
      bw = bt.out_dim
      if not hasattr(self, 'wcat_kn'):
        self.wcat_kn = torch.zeros(plan.x_pad, plan.vin_pad, device=self.device, dtype=torch.bfloat16)
      self.wcat_kn[:, :bw] = self.w_kn[bt.name]
      for role, (c0, n) in plan.HEAD_SLOTS.items():
        sp = plan.one(role)
        if sp is not None:
          self.wcat_kn[:, bw + c0:bw + c0 + n] = self.w_nk[sp.name].t()

  def ide_tables(self):
    if not hasattr(self, '_ide'):
      from . import ref_utils
      m, l, mat = ref_utils.ide_tables(self.plan.cfg.deg_view)
      self._ide = (torch.tensor(mat, dtype=torch.float32, device=self.device).contiguous(),
                   torch.tensor(np.stack([m, l]), dtype=torch.int32, device=self.device).contiguous(), len(m))
    return self._ide


class LevelState:
  """Per-level device buffers kept from forward for the backward pass."""
  pass


class Params:
  """`variables`: flat fp32 parameter/gradient/Adam buffers + per-module views."""

  STATS_TAIL = 64      # floats: [num_levels, 8] loss accumulators (num_levels <= 8)

  def __init__(self, plans: Dict[str, MLPPlan], device, extra: Dict[str, int]):
    self.plans = plans
    self.offsets = {}
    off = 0
    for name, plan in plans.items():
      self.offsets[name] = (off, plan.flat_size)
      off += plan.flat_size
    for name, n in extra.items():
      self.offsets[name] = (off, n)
      off += (n + 3) // 4 * 4
    self.total = off
    self.flat = torch.zeros(off, device=device)
    # gradient buffer + a small tail that carries the step's loss statistics, so the data-parallel
    # exchange of a train step is ONE all-reduce over one flat buffer (pmean of grad and stats,
    # train_utils.py:319-321)
    self.grads_ext = torch.zeros(off + self.STATS_TAIL, device=device)
    self.grads = self.grads_ext[:off]
    self.stats_tail = self.grads_ext[off:]
    self.mu = torch.zeros(off, device=device)
    self.nu = torch.zeros(off, device=device)
    self.step = 0

  def seg(self, name, buf=None):
    o, n = self.offsets[name]
    return (self.flat if buf is None else buf)[o:o + n]


def _init_kernel(rng, name, fan_in, fan_out):
  """flax initialisers (he_uniform / glorot_uniform ...) restated; host numpy.  PARITY UNPINNED:
  threefry streams cannot be reproduced, only the distribution (SURVEY.md section 8c)."""
  if name == 'he_uniform':
    lim = math.sqrt(6.0 / fan_in)
    return rng.uniform(-lim, lim, (fan_in, fan_out)).astype(np.float32)
  if name == 'glorot_uniform':
    lim = math.sqrt(6.0 / (fan_in + fan_out))
    return rng.uniform(-lim, lim, (fan_in, fan_out)).astype(np.float32)
  if name == 'he_normal':
    return (rng.standard_normal((fan_in, fan_out)) * math.sqrt(2.0 / fan_in) / .87962566103423978
            ).clip(-2 * math.sqrt(2.0 / fan_in) / .87962566103423978,
                   2 * math.sqrt(2.0 / fan_in) / .87962566103423978).astype(np.float32)
  if name == 'glorot_normal':
    return (rng.standard_normal((fan_in, fan_out)) * math.sqrt(2.0 / (fan_in + fan_out))
            ).astype(np.float32)
  raise ValueError(f'unknown weight_init {name!r}')


class Model:
  """The mip-NeRF 360 model (reference class `Model`, internal/models.py:47-312)."""

  def __init__(self, bundle: configs.Bundle, device=None):
    L.require_device()
    self.bundle = bundle
    self.config = bundle.config
    self.mcfg = bundle.model
    m = self.mcfg
    self.device = torch.device(device if device is not None else torch.device('cuda', torch.cuda.current_device()))
    for f in dataclasses.fields(m):            # expose Model.<field> like the reference
      setattr(self, f.name, getattr(m, f.name))
    if m.num_glo_features > 0 and m.single_mlp:
      raise ValueError('GLO with single_mlp feeds two input widths to the same view MLP (flax would reject it)')
    if m.ray_shape not in L.RAY_SHAPE:
      raise ValueError("ray_shape must be 'cone' or 'cylinder'")
    if m.raydist_fn not in L.RAYDIST:
      raise ValueError(f'raydist_fn {m.raydist_fn!r} not supported')
    if not m.stop_level_grad:
      raise NotImplementedError('stop_level_grad=False (gradients through resampling)')
    self.plans = {'NerfMLP_0': MLPPlan(bundle.nerf_mlp, m.use_viewdirs, glo_features=m.num_glo_features)}
    if not m.single_mlp:
      self.plans['PropMLP_0'] = MLPPlan(bundle.prop_mlp, m.use_viewdirs)
    for pname, plan in self.plans.items():
      for field, val in plan.device_constraints:
        if val % 64 != 0:
          raise ValueError(f'{pname}.{field} = {val}: the tcgen05 path tiles layer widths in multiples of 64')
    # non-MLP top-level parameter modules (flax names), each clipped/updated on its own
    self.extra_params = {}
    if m.learned_exposure_scaling:
      self.extra_params['exposure_scaling_offsets'] = m.num_glo_embeddings * 3   # Embed [N,3], zeros
    if m.num_glo_features > 0:
      self.extra_params['Embed_0'] = m.num_glo_embeddings * m.num_glo_features    # GLO vectors
    self.params: Optional[Params] = None
    self.mlps: Dict[str, MLPDevice] = {}
    self._levels: Dict[Any, LevelState] = {}
    self._u_cache = {}
    self._init_hist = {}

  # ------------------------------------------------------------------ parameters
  def num_params(self):
    return sum(p.num_params for p in self.plans.values())

  def init(self, seed=0, flax_params=None):
    """Creates `variables` (random init like flax, or from a flax-style tree of arrays)."""
    params = Params(self.plans, self.device, self.extra_params)
    rng = np.random.default_rng(seed)
    host = np.zeros(params.total, np.float32)
    for mname, plan in self.plans.items():
      o, _ = params.offsets[mname]
      for s in plan.specs:
        if flax_params is not None:
          kern = np.asarray(flax_params[mname][s.name]['kernel'], np.float32)
          bias = np.asarray(flax_params[mname][s.name]['bias'], np.float32)
          if kern.shape != (s.in_dim, s.out_dim):
            raise ValueError(f'{mname}/{s.name}: kernel {kern.shape} != {(s.in_dim, s.out_dim)}')
        else:
          kern = _init_kernel(rng, plan.cfg.weight_init, s.in_dim, s.out_dim)
          bias = np.zeros(s.out_dim, np.float32)
        Wp = np.zeros((s.in_pad, s.out_dim), np.float32)
        rows = s.row_map if s.row_map is not None else np.arange(s.in_dim)
        Wp[rows] = kern
        host[o + s.w_off:o + s.w_off + Wp.size] = Wp.reshape(-1)
        host[o + s.b_off:o + s.b_off + s.out_dim] = bias
    if flax_params is not None:
      for name in self.extra_params:
        if name in flax_params:
          o, n = params.offsets[name]
          host[o:o + n] = np.asarray(flax_params[name]['embedding'], np.float32).reshape(-1)
    elif 'Embed_0' in self.extra_params:
      # flax nn.Embed default init: variance_scaling(1.0, 'fan_in', 'normal', out_axis=0)
      o, n = params.offsets['Embed_0']
      host[o:o + n] = rng.standard_normal(n).astype(np.float32) / math.sqrt(self.mcfg.num_glo_features)
    params.flat.copy_(torch.from_numpy(host))
    self.bind(params)
    return params

  def bind(self, params: Params):
    self.params = params
    self.mlps = {n: MLPDevice(p, params.seg(n), params.seg(n, params.grads), self.device)
                 for n, p in self.plans.items()}
    for st in self._levels.values():        # cached chain descriptors point into the previous buffers
      st.__dict__.pop('_chain', None)

  def export_flax(self):
    """Parameters as the reference's flax tree (numpy), dropping the padding rows."""
    out = {}
    for mname, plan in self.plans.items():
      mlp = self.mlps[mname]
      out[mname] = {}
      for s in plan.specs:
        Wp = mlp.W(s).detach().cpu().numpy()
        rows = s.row_map if s.row_map is not None else np.arange(s.in_dim)
        out[mname][s.name] = {'kernel': Wp[rows].copy(), 'bias': mlp.b(s).detach().cpu().numpy().copy()}
    for name in self.extra_params:
      out[name] = {'embedding': self.params.seg(name).detach().cpu().numpy().reshape(
          self.mcfg.num_glo_embeddings, -1).copy()}
    return out

  def export_grads_flax(self):
    out = {}
    for mname, plan in self.plans.items():
      mlp = self.mlps[mname]
      out[mname] = {}
      for s in plan.specs:
        Wp = mlp.W(s, mlp.grads).detach().cpu().numpy()
        rows = s.row_map if s.row_map is not None else np.arange(s.in_dim)
        out[mname][s.name] = {'kernel': Wp[rows].copy(),
                              'bias': mlp.b(s, mlp.grads).detach().cpu().numpy().copy()}
    for name in self.extra_params:
      out[name] = {'embedding': self.params.seg(name, self.params.grads).detach().cpu().numpy().reshape(
          self.mcfg.num_glo_embeddings, -1).copy()}
    return out

  # ------------------------------------------------------------------ schedule
  def level_schedule(self, train_frac):
    m = self.mcfg
    init_s_near = 0.0
    if m.near_anneal_rate is not None:
      init_s_near = min(max(1 - train_frac / m.near_anneal_rate, 0.0), m.near_anneal_init)
    init_s_far = 1.0
    prod = 1
    out = []
    for i in range(m.num_levels):
      is_prop = i < m.num_levels - 1
      ns = m.num_prop_samples if is_prop else m.num_nerf_samples
      dilation = m.dilation_bias + m.dilation_multiplier * (init_s_far - init_s_near) / prod
      prod *= ns
      use_dil = (m.dilation_bias > 0 or m.dilation_multiplier > 0) and i > 0
      if m.anneal_slope > 0:
        s = m.anneal_slope
        anneal = (s * train_frac) / ((s - 1) * train_frac + 1)
      else:
        anneal = 1.0
      out.append(dict(is_prop=is_prop, S=ns, dilation=dilation, use_dilation=use_dil, anneal=anneal))
    return init_s_near, init_s_far, out

  def _u(self, S, randomized):
    key = (S, randomized)
    if key not in self._u_cache:
      ub, mj = ops.u_grid(S, randomized)
      self._u_cache[key] = (ub.to(self.device), mj)
    return self._u_cache[key]

  def _comp_cfg(self, cfg):
    return dict(raydist_fn=self.mcfg.raydist_fn, opaque_background=self.mcfg.opaque_background,
                density_bias=cfg.density_bias, density_noise=cfg.density_noise,
                rgb_activation=cfg.rgb_activation, rgb_premultiplier=cfg.rgb_premultiplier,
                rgb_bias=cfg.rgb_bias, rgb_padding=cfg.rgb_padding,
                bg_const=self.mcfg.bg_intensity_range[0],
                rgb_mode=1 if (cfg.use_diffuse_color and not cfg.disable_rgb) else 0)

  # ------------------------------------------------------------------ buffers
  def _level_state(self, key, mname, B, S):
    # one buffer set per (level, module, shape), never replaced: captured CUDA graphs (train step, render
    # chunks) hold raw pointers into these buffers, so a differently shaped call (the ragged last chunk of
    # an image) must not free them
    key = (key, mname, B, S)
    st = self._levels.get(key)
    plan = self.plans[mname]
    if st is not None:
      return st
    st = LevelState()
    st.B, st.S, st.mname = B, S, mname
    M = B * S
    dev = self.device
    cfg = plan.cfg
    W = cfg.net_width
    bf = torch.bfloat16
    st.sdist = torch.empty(B, S + 1, device=dev)

    def trunk_buffers(rows):
      # the layer whose output is concatenated with the features owns the feature columns
      # (encode writes there), otherwise features get their own buffer
      acts = [torch.empty(rows, W + plan.Fpad if i in plan.concat_after else W, device=dev, dtype=bf)
              for i in range(cfg.net_depth)]
      if plan.concat_after:
        feat = acts[plan.concat_after[0]][:, W:]
        copies = [acts[i][:, W:] for i in plan.concat_after[1:]]
      else:
        feat, copies = torch.empty(rows, plan.Fpad, device=dev, dtype=bf), []
      return acts, feat, copies
    st.acts, st.feat, st.feat_copies = trunk_buffers(M)
    st.bits = [torch.empty(M, W // 32, device=dev, dtype=torch.int32) for _ in range(cfg.net_depth)]
    st.raw_density = torch.empty(B, S, device=dev)
    st.d_raw_density = torch.empty(B, S, device=dev)
    st.raw_rgb = st.d_raw_rgb = None
    st.heads, st.d_heads = {}, {}
    st.extra_dw = None
    st.normals = st.normals_pred = st.roughness = None
    if plan.density_normals:
      # forward-mode tangents d(.)/d(mean_x|y|z), three stacked streams of M rows
      st.tacts, st.tfeat, st.tfeat_copies = trunk_buffers(3 * M)
      st.rgd = torch.empty(3, M, device=dev)
      st.d_rgd = torch.empty(3, M, device=dev)
      st.normals = torch.empty(M, 3, device=dev)
    if plan.has_rgb:
      Wv = cfg.net_width_viewdirs
      nv = cfg.net_depth_viewdirs
      st.vacts = [torch.empty(M, Wv + plan.vin_pad if i in plan.view_concat_after else Wv, device=dev, dtype=bf)
                  for i in range(nv)]
      st.vbits = [torch.empty(M, Wv // 32, device=dev, dtype=torch.int32) for _ in range(nv)]
      if plan.view_concat_after:
        st.vin = st.vacts[plan.view_concat_after[0]][:, Wv:]
      else:
        st.vin = torch.empty(M, plan.vin_pad, device=dev, dtype=bf)
      st.raw_rgb = torch.empty(B, S, 3, device=dev)
      st.d_raw_rgb = torch.empty(B, S, 3, device=dev)
      for role in ('grad_pred', 'diffuse', 'tint', 'roughness'):
        sp = plan.one(role)
        if sp is not None:
          st.heads[role] = torch.empty(M, sp.out_dim, device=dev)
          st.d_heads[role] = torch.empty(M, sp.out_dim, device=dev)
      if plan.ref_stage:
        if plan.pred_normals:
          st.normals_pred = torch.empty(M, 3, device=dev)
        if cfg.enable_pred_roughness:
          st.roughness = torch.empty(M, device=dev)
        st.extra_dw = torch.empty(B, S, device=dev)
    st.bwd = None   # backward scratch, allocated on first backward
    st.keep_acts = True     # False: render-only pass, the chained trunk skips activation / mask stores
    self._levels[key] = st
    return st

  def _refdir_desc(self, st, plan):
    cfg = plan.cfg
    bw = cfg.bottleneck_width
    ide_n = self.mlps[st.mname].ide_tables()[2] if cfg.use_directional_enc else 0
    return ops.refdir_desc(
        st.B * st.S, st.S, use_pred_normals=plan.pred_normals, use_density_normals=plan.density_normals,
        use_reflections=cfg.use_reflections, use_ide=cfg.use_directional_enc, use_n_dot_v=cfg.use_n_dot_v,
        use_roughness=cfg.enable_pred_roughness, deg_view=cfg.deg_view, ide_n=ide_n,
        roughness_bias=cfg.roughness_bias, ld=0, col0=bw, col_end=plan.vin_pad)

  # NB: with GLO the slab's zero-fill would also clear the GLO columns; they are written after it.

  # ------------------------------------------------------------------ forward
  def _mlp_forward(self, st: LevelState, mlp: MLPDevice, rays, impl=0, loss_mults=None):
    """loss_mults = (orientation, predicted-normal) multipliers of this level divided by the number
    of rays, + orientation target flag: when given, the Ref-NeRF stage also emits d(loss)/d(weights)."""
    plan = mlp.plan
    cfg = plan.cfg
    B, S = st.B, st.S
    M = B * S
    W = cfg.net_width
    m = self.mcfg
    ops.encode(st.sdist, rays.origins, rays.directions, rays.radii_flat, rays.near_flat,
               rays.far_flat, mlp.basis, min_deg=cfg.min_deg_point, max_deg=cfg.max_deg_point,
               raydist_fn=m.raydist_fn, ray_shape=m.ray_shape, warp_contract=cfg.warp_fn == 'contract',
               disable_integration=m.disable_integration, feat=st.feat, feat_cols=plan.Fpad,
               tfeat=st.tfeat if plan.density_normals else None)
    for c in st.feat_copies:
      c.copy_(st.feat)
    x = st.feat
    trunk = plan.by_role('trunk')
    d = plan.one('density')
    chained = self._use_chain(plan, M, impl)
    if chained:
      # the whole trunk (+ the Dense(1) density head when it reads the plain 256-wide output) in ONE launch
      ops.mlp_chain(self._chain_fwd_desc(st, mlp))
      x = st.acts[-1]
      if plan.last_has_feat:
        ops.head_fwd(x, mlp.w_nk[d.name], mlp.b(d), 1, d.in_pad, raw=st.raw_density.view(M, 1))
    else:
      for i, sp in enumerate(trunk):
        ops.gemm(L.GEMM_FWD, x, mlp.w_nk[sp.name], st.acts[i][:, :W], m=M, n=W, k=sp.in_pad, act=L.ACT_RELU,
                 bias=mlp.b(sp), maskbits=st.bits[i], impl=impl)
        x = st.acts[i]          # full width (incl. concatenated features) feeds the next layer
      ops.head_fwd(x, mlp.w_nk[d.name], mlp.b(d), 1, d.in_pad, raw=st.raw_density.view(M, 1))
    st.x_last = x
    if plan.density_normals:
      # raw_grad_density = d raw_density / d mean by forward mode (replaces vmap(value_and_grad),
      # models.py:473-492): tangents see the same weights, no bias, and the primal's ReLU masks
      for c in st.tfeat_copies:
        c.copy_(st.tfeat)
      t = st.tfeat
      for i, sp in enumerate(trunk):
        ops.gemm(L.GEMM_DGRAD, t, mlp.w_nk[sp.name], st.tacts[i][:, :W], m=3 * M, n=W, k=sp.in_pad,
                 maskbits=st.bits[i], mask_mod=M, impl=impl)
        t = st.tacts[i]
      st.t_last = t
      ops.head_fwd(t, mlp.w_nk[d.name], None, 1, d.in_pad, raw=st.rgd.view(3 * M, 1))
    if not plan.has_rgb:
      return
    for role in ('grad_pred', 'diffuse', 'tint', 'roughness'):
      sp = plan.one(role)
      if sp is not None:
        ops.head_fwd(x, mlp.w_nk[sp.name], mlp.b(sp), sp.out_dim, sp.in_pad, raw=st.heads[role])
    bt = plan.one('bottleneck')
    ops.gemm(L.GEMM_FWD, x, mlp.w_nk[bt.name], st.vin[:, :bt.out_dim], m=M, n=bt.out_dim,
             k=bt.in_pad, act=L.ACT_NONE, bias=mlp.b(bt), impl=impl)
    if cfg.bottleneck_noise > 0 and getattr(st, 'bneck_noise', None) is not None:
      # models.py:529-533 (regulariser, unused by the shipped configs): plain elementwise add
      st.vin[:, :bt.out_dim].add_((cfg.bottleneck_noise * st.bneck_noise).to(torch.bfloat16))
    if plan.ref_stage:
      desc = self._refdir_desc(st, plan)
      desc.ld = st.vin.stride(0)
      mat, ml, _ = mlp.ide_tables() if cfg.use_directional_enc else (None, None, 0)
      om, pm, on_pred = loss_mults if loss_mults is not None else (0.0, 0.0, True)
      ops.refdir_fwd(desc, mat, ml, st.heads.get('grad_pred'), st.heads.get('roughness'),
                     st.rgd if plan.density_normals else None, rays.viewdirs, st.normals_pred, st.normals,
                     st.roughness, st.vin, om, pm, on_pred,
                     st.extra_dw if loss_mults is not None else None)
    else:
      ops.viewdir_enc(rays.viewdirs, S, cfg.deg_view, st.vin, bt.out_dim, plan.vin_pad)
    if plan.glo_features > 0:
      # GLO vector of the ray's camera, broadcast over the samples (models.py:565-569)
      g0 = plan.glo_col0
      st.vin.view(B, S, st.vin.stride(0))[:, :, g0:g0 + plan.glo_features] = \
          (st.glo_vec if st.glo_vec is not None else torch.zeros(B, plan.glo_features, device=st.vin.device)
           )[:, None, :].to(torch.bfloat16)
    v = st.vin
    for i, sp in enumerate(plan.by_role('view')):
      Wv = sp.out_dim
      ops.gemm(L.GEMM_FWD, v, mlp.w_nk[sp.name], st.vacts[i][:, :Wv], m=M, n=Wv, k=sp.in_pad,
               act=L.ACT_RELU, bias=mlp.b(sp), maskbits=st.vbits[i], impl=impl)
      v = st.vacts[i]
    st.v_last = v
    r = plan.one('rgb')
    ops.head_fwd(v, mlp.w_nk[r.name], mlp.b(r), r.out_dim, r.in_pad, raw=st.raw_rgb.view(M, 3))

  # ------------------------------------------------------------------ layer-chained 256-wide trunks
  def _use_chain(self, plan, M, impl=0):
    """One persistent launch per trunk (csrc/chain.cu) when every trunk layer is 256 wide."""
    if impl != 0:
      return False
    cfg = plan.cfg
    return (cfg.net_width == 256 and cfg.net_depth <= L.CHAIN_MAX_LAYERS and M >= 512 and
            plan.Fpad % 64 == 0)

  def _chain_fwd_desc(self, st, mlp):
    key = ('fwd', st.keep_acts)
    cache = st.__dict__.setdefault('_chain', {})
    if key in cache:
      return cache[key]
    plan = mlp.plan
    W = plan.cfg.net_width
    M = st.B * st.S
    nf = plan.Fpad // 64
    trunk = plan.by_role('trunk')
    layers = []
    for i, sp in enumerate(trunk):
      ly = dict(w=mlp.w_nk[sp.name], bias=mlp.b(sp))
      if i == 0:
        ly.update(n_stream=nf, stream_col0=0, stream_kb0=0)
      else:
        ly.update(n_res=W // 64, res_kb0=0)
        if sp.in_pad == W + plan.Fpad:          # skip layer: [hidden | features] against [W | Fpad] weight columns
          ly.update(n_stream=nf, stream_col0=0, stream_kb0=W // 64)
      last = i == len(trunk) - 1
      if st.keep_acts or (last and (plan.has_rgb or plan.last_has_feat)):
        ly['out'] = st.acts[i][:, :W]
      if st.keep_acts:
        ly['maskbits'] = st.bits[i]
      layers.append(ly)
    head = {}
    if not plan.last_has_feat:
      dsp = plan.one('density')
      head = dict(head_w=mlp.colv_density, head_b=mlp.b(dsp), head_out=st.raw_density.view(M))
    cache[key] = ops.chain_desc(L.CHAIN_FWD, M, layers, stream=st.feat, stream_cols=plan.Fpad, **head)
    return cache[key]

  def _chain_bwd_desc(self, st, mlp, dyl):
    """dyl[i] = gradient w.r.t. the (pre-activation-masked) output of trunk layer i; dyl[-1] is the input."""
    cache = st.__dict__.setdefault('_chain', {})
    if 'bwd' in cache:
      return cache['bwd']
    plan = mlp.plan
    W = plan.cfg.net_width
    M = st.B * st.S
    trunk = plan.by_role('trunk')
    g = mlp.grads
    layers = []
    for j, i in enumerate(range(len(trunk) - 1, 0, -1)):
      sp = trunk[i]
      ly = dict(w=mlp.w_kn[sp.name], maskbits=st.bits[i - 1], out=dyl[i - 1])
      if j == 0:
        ly.update(n_stream=W // 64, stream_col0=0, stream_kb0=0)
      else:
        ly.update(n_res=W // 64, res_kb0=0)
      layers.append(ly)
    cache['bwd'] = ops.chain_desc(L.CHAIN_BWD, M, layers, stream=dyl[-1], stream_cols=W)
    return cache['bwd']

  def _prep_rays(self, rays):
    r = utils.to_device_flat(rays, self.device)
    r.radii_flat = r.radii[:, 0].contiguous()
    r.near_flat = r.near[:, 0].contiguous()
    r.far_flat = r.far[:, 0].contiguous()
    return r

  def level_loss_mults(self, config, i_level, B):
    """(orientation, predicted-normal) multipliers of level i divided by the ray count, target flag
    (train_utils.py:162-197)."""
    fine = i_level == self.mcfg.num_levels - 1
    om = config.orientation_loss_mult if fine else config.orientation_coarse_loss_mult
    pm = config.predicted_normal_loss_mult if fine else config.predicted_normal_coarse_loss_mult
    if config.orientation_loss_target not in ('normals', 'normals_pred'):
      raise ValueError(f'orientation_loss_target {config.orientation_loss_target!r}')
    return om / B, pm / B, config.orientation_loss_target == 'normals_pred'

  def forward_levels(self, rng, rays, train_frac, compute_extras, want_samples, impl=0, anneal_dev=None,
                     loss_config=None, zero_glo=True):
    """Runs all levels; returns the list of LevelState (buffers stay valid until the next call)."""
    if self.params is None:
      raise RuntimeError('Model has no parameters: call construct_model()/init() first')
    m = self.mcfg
    B = rays.origins.shape[0]
    s_near, s_far, sched = self.level_schedule(train_frac)
    dev = self.device
    # RawNeRF exposure logic (models.py:257-267): one per-ray colour scale for every level
    rgb_scale = None
    if getattr(rays, 'exposure_idx', None) is not None:
      rgb_scale = rays.exposure_values.expand(B, 3)
      if m.learned_exposure_scaling:
        eidx = rays.exposure_idx[:, 0].long()
        mask = (eidx > 0).to(torch.float32)[:, None]
        off = self.params.seg('exposure_scaling_offsets').view(-1, 3)[eidx]
        rgb_scale = rgb_scale * (1 + mask * off)
      rgb_scale = rgb_scale.contiguous()
    # the initial one-interval histogram [s_near, s_far] with weight 1 is a constant of (B, s_near, s_far): built
    # once, so a captured step does not replay three fill kernels for it
    ck = (B, float(s_near), float(s_far))
    init = self._init_hist.get(ck)
    if init is None:
      sd0 = torch.empty(B, 2, device=dev)
      sd0[:, 0] = s_near
      sd0[:, 1] = s_far
      init = (sd0, torch.ones(B, 1, device=dev))
      # entries are never evicted (a captured graph may hold their addresses); with near-plane annealing s_near
      # changes every step, so the table simply stops growing
      if len(self._init_hist) < 8 and not torch.cuda.is_current_stream_capturing():
        self._init_hist[ck] = init
    sdist_prev, w_prev = init
    states = []
    for i, lv in enumerate(sched):
      mname = 'NerfMLP_0' if (m.single_mlp or not lv['is_prop']) else 'PropMLP_0'
      mlp = self.mlps[mname]
      st = self._level_state(i, mname, B, lv['S'])
      st.lv = lv
      st.is_prop = lv['is_prop']
      # activations and ReLU masks are kept for a backward pass (and for the Ref-NeRF tangent chain)
      st.keep_acts = loss_config is not None or mlp.plan.density_normals
      jit = None
      if rng is not None:
        if isinstance(rng, dict):
          jit = rng['jitter'][i].to(dev).contiguous()
          jit = jit.reshape(B) if m.single_jitter else jit.reshape(B, lv['S'])
        else:
          shape = (B,) if m.single_jitter else (B, lv['S'])
          jit = torch.rand(shape, device=dev, generator=rng)
      u_base, max_jitter = self._u(lv['S'], jit is not None)
      ops.sample_level(sdist_prev, w_prev, lv['S'], dilation=lv['dilation'],
                       use_dilation=lv['use_dilation'], domain=(s_near, s_far), anneal=lv['anneal'],
                       resample_padding=m.resample_padding, jitter=jit, single_jitter=m.single_jitter,
                       u_base=u_base, max_jitter=max_jitter, out=st.sdist, anneal_dev=anneal_dev)
      st.glo_vec = None
      if m.num_glo_features > 0 and not lv['is_prop'] and not zero_glo:
        st.glo_vec = self.params.seg('Embed_0').view(m.num_glo_embeddings, -1)[rays.cam_idx[:, 0].long()]
      st.bneck_noise = None
      if mlp.plan.cfg.bottleneck_noise > 0 and rng is not None and mlp.plan.has_rgb:
        bwid = mlp.plan.cfg.bottleneck_width
        if isinstance(rng, dict):
          st.bneck_noise = rng['bottleneck_noise'][i].to(dev).reshape(B * lv['S'], bwid)
        else:
          st.bneck_noise = torch.randn(B * lv['S'], bwid, device=dev, generator=rng)
      st.loss_mults = self.level_loss_mults(loss_config, i, B) if (loss_config is not None and
                                                                   mlp.plan.ref_stage) else None
      if st.loss_mults is not None:
        om, pm, on_pred = st.loss_mults
        if (om > 0 and ((on_pred and not mlp.plan.pred_normals) or (not on_pred and not mlp.plan.density_normals))):
          raise ValueError('Normals cannot be None if orientation loss is on.')
        if pm > 0 and not (mlp.plan.pred_normals and mlp.plan.density_normals):
          raise ValueError('Predicted normals and gradient normals cannot be None if '
                           'predicted normal loss is on.')
      self._mlp_forward(st, mlp, rays, impl=impl, loss_mults=st.loss_mults)
      st.noise = None
      if mlp.plan.cfg.density_noise > 0 and rng is not None:
        if isinstance(rng, dict):
          st.noise = rng['density_noise'][i].to(dev).reshape(B, lv['S']).contiguous()
        else:
          st.noise = torch.randn(B, lv['S'], device=dev, generator=rng)
      st.comp_cfg = self._comp_cfg(mlp.plan.cfg)
      # background colour (models.py:240-254): constant, midpoint (rng=None) or per-ray uniform draws
      lo, hi = m.bg_intensity_range
      st.bg_rgb = None
      if lo != hi:
        if rng is None:
          st.comp_cfg['bg_const'] = (lo + hi) / 2
        else:
          if isinstance(rng, dict):
            ub = rng['bg'][i].to(dev).reshape(B, 3)
          else:
            ub = torch.rand(B, 3, device=dev, generator=rng)
          st.bg_rgb = (lo + (hi - lo) * ub).contiguous()
      st.comp = ops.composite_fwd(st.raw_density, st.raw_rgb, st.sdist, rays.directions,
                                  rays.near_flat, rays.far_flat, cfg=st.comp_cfg,
                                  density_noise=st.noise, bg_rgb=st.bg_rgb,
                                  rgb_scale=rgb_scale if st.raw_rgb is not None else None,
                                  raw_diffuse=st.heads.get('diffuse'), raw_tint=st.heads.get('tint'),
                                  want_samples=want_samples, want_extras=compute_extras)
      st.rgb_scale = rgb_scale if st.raw_rgb is not None else None
      sdist_prev, w_prev = st.sdist, st.comp['weights']
      states.append(st)
    return states

  def __call__(self, rng, rays, train_frac, compute_extras, zero_glo=True):
    """models.py:75-312.  rng: None (deterministic), a torch.Generator on the device, or a
    dict of explicit draws {'jitter': [per level], 'density_noise': [per level]}."""
    r = self._prep_rays(rays)
    lead = tuple(np.asarray(rays.origins).shape[:-1]) if not isinstance(rays.origins, torch.Tensor) \
        else tuple(rays.origins.shape[:-1])
    return self.call_prepped(rng, r, lead, train_frac, compute_extras, zero_glo)

  def call_prepped(self, rng, r, lead, train_frac, compute_extras, zero_glo=True):
    """`__call__` on rays already flattened on the device (`_prep_rays`): device work only, so a render
    chunk can be captured in a CUDA graph (train_utils.create_render_fn)."""
    states = self.forward_levels(rng, r, train_frac, compute_extras, want_samples=True, zero_glo=zero_glo)
    renderings, ray_history = [], []
    n_vis = self.config.vis_num_rays
    for st in states:
      c = st.comp
      rend = {'rgb': c['rgb'].view(lead + (3,))}
      if compute_extras:
        rend['acc'] = c['acc'].view(lead)
        for j, k in enumerate(['distance_mean', 'distance_percentile_5', 'distance_median',
                               'distance_percentile_95']):
          rend[k] = c['dist'][:, j].contiguous().view(lead)
        w3 = c['weights'][..., None]
        for k, v in (('normals', st.normals), ('normals_pred', st.normals_pred), ('roughness', st.roughness)):
          if v is not None:     # volumetric_rendering extras (render.py:186-189)
            rend[k] = (w3 * v.view(st.B, st.S, -1)).sum(-2).view(lead + (-1,))
        rend['ray_sdist'] = st.sdist[:n_vis].clone()
        rend['ray_weights'] = c['weights'][:n_vis].clone()
        rend['ray_rgbs'] = c['rgb_samples'][:n_vis].clone()
      renderings.append(rend)
      S = st.S
      ray_history.append(dict(
          density=c['density'].view(lead + (S,)), rgb=c['rgb_samples'].view(lead + (S, 3)),
          raw_grad_density=None if st.normals is None else st.rgd.t().reshape(lead + (S, 3)),
          grad_pred=None if 'grad_pred' not in st.heads else st.heads['grad_pred'].view(lead + (S, 3)),
          normals=None if st.normals is None else st.normals.view(lead + (S, 3)),
          normals_pred=None if st.normals_pred is None else st.normals_pred.view(lead + (S, 3)),
          roughness=None if st.roughness is None else st.roughness.view(lead + (S, 1)),
          sdist=st.sdist.clone().view(lead + (S + 1,)), weights=c['weights'].view(lead + (S,))))
    if compute_extras:
      final_rgb = (renderings[-1]['ray_rgbs'] * renderings[-1]['ray_weights'][..., None]).sum(-2)
      for rr in renderings[:-1]:
        rr['ray_rgbs'] = final_rgb[:, None, :].expand(rr['ray_rgbs'].shape).contiguous()
    return renderings, ray_history

  def apply(self, variables, rng, rays, train_frac, compute_extras, zero_glo=True):
    """flax-style entry: model.apply(variables, rng, rays, train_frac=..., compute_extras=...)."""
    if variables is not self.params:
      self.bind(variables)
    return self(rng, rays, train_frac, compute_extras, zero_glo)

  # ------------------------------------------------------------------ backward
  def _mlp_backward(self, st: LevelState, mlp: MLPDevice, rays=None, impl=0, loss_mults=None, stats=None):
    """Accumulates parameter gradients of one level into mlp.grads (fp32).

    Bias gradients are column sums of the dY buffers, never a separate pass over HBM.  Where they come from is
    chosen by what is measured to be free: for the 1024-wide layers the dgrad epilogue that PRODUCES the dY
    (`colsum`, hidden under a K = 1024 main loop); for chained 256-wide trunks the weight-gradient GEMM, whose
    idle epilogue warps read the dY tiles of its main loop (`mnrf_gemm_wgrad` `bsum`; those GEMMs are HBM-bound,
    while the same trick costs a 1024-wide weight gradient +48 %).  The bottleneck's weight gradient also carries
    the Dense(1) density head's weight gradient (`side_aw`), which used to re-read the activation.
    """
    plan = mlp.plan
    cfg = plan.cfg
    M = st.B * st.S
    W = cfg.net_width
    dev = self.device
    bf = torch.bfloat16
    if st.bwd is None:
      bw_ = LevelState()
      # per-layer gradient buffers when the dgrad chain runs as one launch (its wgrads come after)
      n_dy = cfg.net_depth if self._use_chain(plan, M, impl) else 2
      bw_.dy = [torch.empty(M, W, device=dev, dtype=bf) for _ in range(n_dy)]
      if plan.has_rgb:
        Wv = cfg.net_width_viewdirs
        bw_.dv = [torch.empty(M, Wv, device=dev, dtype=bf) for _ in range(2)]
        bw_.d_vin = torch.empty(M, plan.vin_pad, device=dev, dtype=bf)
        bw_.d_vin_skip = torch.empty(M, plan.vin_pad, device=dev, dtype=bf) if plan.view_concat_after else None
      if plan.density_normals:
        bw_.h = [torch.empty(3 * M, W, device=dev, dtype=bf) for _ in range(2)]
      st.bwd = bw_
    sc = st.bwd
    g = mlp.grads
    # bias gradients of the trunk come from its weight-gradient GEMMs when its dgrad chain is one launch
    side = self._use_chain(plan, M, impl) and len(plan.by_role('trunk')) > 1
    d = plan.one('density')
    trunk = plan.by_role('trunk')
    x_last = st.x_last
    dy = sc.dy[0]
    d_raw_density = st.d_raw_density.view(M, 1)
    if plan.has_rgb:
      r = plan.one('rgb')
      views = plan.by_role('view')
      Wv = cfg.net_width_viewdirs
      bt = plan.one('bottleneck')
      bw = bt.out_dim
      dcur = sc.dv[0]
      ops.head_bwd(st.v_last, mlp.w_nk[r.name], st.d_raw_rgb.view(M, 3), r.out_dim, r.in_pad, dx=dcur,
                   relu_mask=True, dw=mlp.W(r, g), db=mlp.b(r, g), dxsum=mlp.b(views[-1], g))
      have_skip_grad = False
      for i in range(len(views) - 1, -1, -1):
        sp = views[i]
        xin = st.vin if i == 0 else st.vacts[i - 1]
        ops.gemm(L.GEMM_WGRAD, xin, dcur, mlp.W(sp, g), m=sp.in_pad, n=Wv, k=M, impl=impl)
        if i > 0:
          if (i - 1) in plan.view_concat_after:
            # this layer also consumed vin (skip concat): its second gradient contribution
            ops.gemm(L.GEMM_DGRAD, dcur, mlp.w_kn[sp.name][Wv:], sc.d_vin_skip, m=M, n=plan.vin_pad, k=Wv,
                     impl=impl)
            have_skip_grad = True
          nxt = sc.dv[1] if dcur is sc.dv[0] else sc.dv[0]
          ops.gemm(L.GEMM_DGRAD, dcur, mlp.w_kn[sp.name], nxt, m=M, n=Wv, k=Wv,
                   maskbits=st.vbits[i - 1], colsum=mlp.b(views[i - 1], g), impl=impl)
          dcur = nxt
      s0 = views[0]
      if plan.ref_stage:
        # full d vin: [ d bottleneck | d direction encoding (| d n.v) ]
        ops.gemm(L.GEMM_DGRAD, dcur, mlp.w_kn[s0.name], sc.d_vin, m=M, n=plan.vin_pad, k=Wv,
                 addend=sc.d_vin_skip if have_skip_grad else None, impl=impl)
        d_glo_ref = None
        if plan.glo_features > 0 and st.glo_vec is not None:     # before the slab columns are re-used
          g0 = plan.glo_col0
          d_glo_ref = sc.d_vin.view(st.B, st.S, plan.vin_pad)[:, :, g0:g0 + plan.glo_features].float().sum(1)
        desc = self._refdir_desc(st, plan)
        desc.ld = st.vin.stride(0)
        mat, ml, _ = mlp.ide_tables() if cfg.use_directional_enc else (None, None, 0)
        om, pm, on_pred = loss_mults if loss_mults is not None else (0.0, 0.0, True)
        ops.refdir_bwd(desc, mat, ml, st.heads.get('grad_pred'), st.heads.get('roughness'),
                       st.rgd if plan.density_normals else None, rays.viewdirs, st.comp['weights'], sc.d_vin,
                       om, pm, on_pred, st.d_raw_density, st.d_heads.get('diffuse'), st.d_heads.get('tint'),
                       st.d_heads.get('grad_pred'), st.d_heads.get('roughness').view(M) if 'roughness' in st.d_heads else None,
                       st.d_rgd if plan.density_normals else None, stats)
        # parameter gradients of the narrow heads (x^T d_raw)
        for role in ('grad_pred', 'diffuse', 'tint', 'roughness'):
          sp = plan.one(role)
          if sp is not None:
            ops.head_bwd(x_last, mlp.w_nk[sp.name], st.d_heads[role], sp.out_dim, sp.in_pad, dx=None,
                         dw=mlp.W(sp, g), db=mlp.b(sp, g))
        # bottleneck dW + db, and the Dense(1) density head's dW from the same x_last tiles
        ops.gemm_wgrad(x_last, sc.d_vin[:, :bw], mlp.W(bt, g), m=bt.in_pad, n=bw, k=M, bsum=mlp.b(bt, g),
                       side_w=st.d_raw_density.view(M), side_aw=mlp.W(d, g).view(-1), impl=impl)
        # d x_last = relu'(x_last) * ([d bottleneck | head gradients] @ [W_b | w_heads]^T)
        ops.gemm(L.GEMM_DGRAD, sc.d_vin, mlp.wcat_kn, dy, m=M, n=W, k=plan.vin_pad,
                 maskbits=st.bits[-1], colsum=None if side else mlp.b(trunk[-1], g), impl=impl)
      else:
        dbott = sc.d_vin[:, :bw]
        # d vin[:, :bw] = dcur * Wv0[:bw, :]^T  (no activation on the bottleneck)
        if plan.glo_features > 0:
          # the GLO columns of vin carry gradient too: full-width dgrad, then sum over the samples
          ops.gemm(L.GEMM_DGRAD, dcur, mlp.w_kn[s0.name], sc.d_vin, m=M, n=plan.vin_pad, k=Wv,
                   addend=sc.d_vin_skip if have_skip_grad else None, impl=impl)
        else:
          ops.gemm(L.GEMM_DGRAD, dcur, mlp.w_kn[s0.name], dbott, m=M, n=bw, k=Wv,
                   addend=sc.d_vin_skip[:, :bw] if have_skip_grad else None, impl=impl)
        # bottleneck dW + db, and the Dense(1) density head's dW from the same x_last tiles (models.py:460,527)
        ops.gemm_wgrad(x_last, dbott, mlp.W(bt, g), m=bt.in_pad, n=bw, k=M, bsum=mlp.b(bt, g),
                       side_w=st.d_raw_density.view(M), side_aw=mlp.W(d, g).view(-1), impl=impl)
        # d x_last = (dbott * Wb^T + d_raw_density (x) w_density) * relu'(x_last)
        ops.gemm(L.GEMM_DGRAD, dbott, mlp.w_kn[bt.name], dy, m=M, n=W, k=bw,
                 rowv=st.d_raw_density.view(M), colv=mlp.colv_density, maskbits=st.bits[-1],
                 colsum=None if side else mlp.b(trunk[-1], g), impl=impl)
      # bias gradient of the density head: a plain sum of d_raw_density
      mlp.b(d, g).add_(st.d_raw_density.sum())
      if plan.glo_features > 0 and st.glo_vec is not None:
        g0 = plan.glo_col0
        d_glo = d_glo_ref if plan.ref_stage else \
            sc.d_vin.view(st.B, st.S, plan.vin_pad)[:, :, g0:g0 + plan.glo_features].float().sum(1)
        self.params.seg('Embed_0', self.params.grads).view(self.mcfg.num_glo_embeddings, -1).index_add_(
            0, rays.cam_idx[:, 0].long(), d_glo)
    else:
      ops.head_bwd(x_last, mlp.w_nk[d.name], d_raw_density, 1, d.in_pad, dx=dy, relu_mask=True,
                   dw=mlp.W(d, g), db=mlp.b(d, g), dxsum=None if side else mlp.b(trunk[-1], g))
    if plan.density_normals:
      # adjoint of the tangent chain: H_last = relu'(x_last) * (d_rgd (x) w_density), three streams
      hcur, hoth = sc.h[0], sc.h[1]
      ops.outer_mask(st.d_rgd.view(3 * M), mlp.colv_density, st.bits[-1], hcur, rows=3 * M, n=W, mask_mod=M)
      ops.head_bwd(st.t_last, mlp.w_nk[d.name], st.d_rgd.view(3 * M, 1), 1, d.in_pad, dx=None,
                   dw=mlp.W(d, g), db=None)
      for i in range(len(trunk) - 1, -1, -1):
        sp = trunk[i]
        tin = st.tfeat if i == 0 else st.tacts[i - 1]
        ops.gemm(L.GEMM_WGRAD, tin, hcur, mlp.W(sp, g), m=sp.in_pad, n=W, k=3 * M, impl=impl)
        if i > 0:
          ops.gemm(L.GEMM_DGRAD, hcur, mlp.w_kn[sp.name], hoth, m=3 * M, n=W, k=W,
                   maskbits=st.bits[i - 1], mask_mod=M, impl=impl)
          hcur, hoth = hoth, hcur
    if self._use_chain(plan, M, impl) and len(trunk) > 1:
      # dyl[i] = d loss / d (output of trunk layer i); dyl[-1] was produced above (sc.dy[0])
      nl = len(trunk)
      dyl = [sc.dy[nl - 1 - i] for i in range(nl)]        # dyl[nl-1] is sc.dy[0]
      ops.mlp_chain(self._chain_bwd_desc(st, mlp, dyl))
      for i in range(nl - 1, -1, -1):
        sp = trunk[i]
        xin = st.feat if i == 0 else st.acts[i - 1]
        ops.gemm_wgrad(xin, dyl[i], mlp.W(sp, g), m=sp.in_pad, n=W, k=M, bsum=mlp.b(sp, g), impl=impl)
      return
    cur, other = sc.dy[0], sc.dy[1]
    for i in range(len(trunk) - 1, -1, -1):
      sp = trunk[i]
      xin = st.feat if i == 0 else st.acts[i - 1]
      ops.gemm(L.GEMM_WGRAD, xin, cur, mlp.W(sp, g), m=sp.in_pad, n=W, k=M, impl=impl)
      if i > 0:
        # only the hidden part of the input carries gradient (features are constants:
        # stop_gradient(sdist), models.py:200-201)
        ops.gemm(L.GEMM_DGRAD, cur, mlp.w_kn[sp.name], other, m=M, n=W, k=W,
                 maskbits=st.bits[i - 1], colsum=mlp.b(trunk[i - 1], g), impl=impl)
        cur, other = other, cur


def construct_model(rng, rays, config, device=None):
  """models.py:315-338.  `config` is a configs.Bundle; `rng` an int seed (or None -> 0)."""
  bundle = config if isinstance(config, configs.Bundle) else configs.Bundle(config=config)
  model = Model(bundle, device=device)
  seed = 0 if rng is None else (rng if isinstance(rng, int) else int(torch.as_tensor(rng).sum()))
  variables = model.init(seed)
  return model, variables


def render_image(render_fn, rays, rng, config, verbose=True, world_size=1, rank=0):
  """Render all pixels of an image in chunks (models.py:625-706).

  render_fn(rng, chunk_rays) -> (renderings, ray_history) with every rank's rays gathered
  (multinerf_b200.train_utils.create_render_fn).  `rays` leaves are [H, W, n].
  """
  cfg = config.config if isinstance(config, configs.Bundle) else config
  height, width = np.asarray(rays.origins).shape[:2] if not isinstance(rays.origins, torch.Tensor) \
      else rays.origins.shape[:2]
  num_rays = height * width
  flat = rays.map(lambda r: r.reshape((num_rays, -1)))
  chunks = []
  idx0s = range(0, num_rays, cfg.render_chunk_size)
  for i_chunk, idx0 in enumerate(idx0s):
    if verbose and i_chunk % max(1, len(idx0s) // 10) == 0:
      print(f'Rendering chunk {i_chunk}/{len(idx0s)-1}')
    chunk = flat.map(lambda r: r[idx0:idx0 + cfg.render_chunk_size])
    actual = chunk.origins.shape[0]
    rem = actual % world_size
    padding = 0
    if rem != 0:
      padding = world_size - rem
      def pad(r):
        if isinstance(r, torch.Tensor):
          return torch.cat([r, r[-1:].expand(padding, *r.shape[1:])], 0)
        return np.concatenate([r, np.repeat(r[-1:], padding, 0)], 0)
      chunk = chunk.map(pad)
    per = chunk.origins.shape[0] // world_size
    mine = chunk.map(lambda r: r[rank * per:(rank + 1) * per])
    chunk_renderings, _ = render_fn(rng, mine)
    if padding > 0:
      chunk_renderings = [{k: (v[:-padding] if not k.startswith('ray_') else v) for k, v in r.items()}
                          for r in chunk_renderings]
    out = dict(chunk_renderings[-1])
    for k in chunk_renderings[0]:
      if k.startswith('ray_'):
        out[k] = [r[k] for r in chunk_renderings]
    chunks.append(out)
  rendering = {}
  for k in chunks[0]:
    if k.startswith('ray_'):
      rendering[k] = [torch.cat([c[k][i] for c in chunks]) for i in range(len(chunks[0][k]))]
    else:
      z = torch.cat([c[k] for c in chunks])
      rendering[k] = z.reshape((height, width) + tuple(z.shape[1:]))
  keys = [k for k in rendering if k.startswith('ray_')]
  if keys:
    n = rendering[keys[0]][0].shape[0]
    # the reference takes jax.random.permutation(PRNGKey(0)) (threefry, not reproducible here):
    # a fixed numpy permutation plays the same role
    ray_idx = torch.as_tensor(np.random.default_rng(0).permutation(n)[:cfg.vis_num_rays])
    for k in keys:
      rendering[k] = [r[ray_idx.to(r.device)] for r in rendering[k]]
  return rendering
