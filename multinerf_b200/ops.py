"""Thin tensor-level wrappers over the C ABI (one Python function per entry point).

These mirror the reference's free functions where one exists (stepfun.sample_intervals,
render.cast_rays + coord.integrated_pos_enc, render.compute_alpha_weights +
volumetric_rendering, ...) but operate on flat [B, ...] CUDA tensors.
"""
import ctypes as C
import math

import torch

from . import lib as L

EPS = float(torch.finfo(torch.float32).eps)

# Instrumentation used by bench.py: number of kernels launched (counted per ABI call), and --
# when set to a list -- CUDA event pairs around every tensor-core GEMM launch.
LAUNCHES = 0
GEMM_EVENTS = None


def _count(n=1):
  global LAUNCHES
  LAUNCHES += n


def _f32(t):
  assert t is None or (t.dtype == torch.float32 and t.is_contiguous()), 'need contiguous fp32'
  return t


def u_grid(num_samples, randomized):
  """Host-side u grid of stepfun.sample (stepfun.py:190-209): (u_base[S] fp32, max_jitter)."""
  eps = EPS
  if not randomized:
    pad = 1 / (2 * num_samples)
    return torch.linspace(pad, 1.0 - pad - eps, num_samples, dtype=torch.float32), 0.0
  u_max = eps + (1 - eps) / num_samples
  max_jitter = (1 - u_max) / (num_samples - 1) - eps
  return torch.linspace(0, 1 - u_max, num_samples, dtype=torch.float32), max_jitter


def sample_level(sdist_prev, w_prev, num_samples, *, dilation=0.0, use_dilation=False,
                 domain=(0.0, 1.0), anneal=1.0, resample_padding=0.0, jitter=None,
                 single_jitter=True, u_base=None, max_jitter=None, cw_in=None, want_index=False,
                 want_debug=False, out=None, anneal_dev=None):
  """One level of hierarchical resampling -> sdist [B, S+1] (+ int32 idx, debug arrays)."""
  lib = L.load()
  if num_samples <= 1:
    raise ValueError(f'num_samples must be > 1, is {num_samples}.')
  B, P = w_prev.shape
  assert sdist_prev.shape == (B, P + 1)
  dev = sdist_prev.device
  if u_base is None:
    ub, mj = u_grid(num_samples, jitter is not None)
    u_base = ub.to(dev)
    max_jitter = mj if max_jitter is None else max_jitter
  d = L.SampleDesc(B, P, num_samples, int(use_dilation), float(dilation), float(domain[0]),
                   float(domain[1]), float(anneal), float(resample_padding),
                   0 if jitter is None else (1 if single_jitter else 2), float(max_jitter or 0.0))
  nb = 3 * P - 2 if use_dilation else P
  sdist = out if out is not None else torch.empty(B, num_samples + 1, device=dev)
  idx = torch.empty(B, num_samples, device=dev, dtype=torch.int32) if want_index else None
  cw = torch.empty(B, nb + 1, device=dev) if want_debug else None
  tdil = torch.empty(B, nb + 1, device=dev) if want_debug else None
  wdil = torch.empty(B, nb, device=dev) if want_debug else None
  _count()
  if anneal_dev is not None:
    assert cw_in is None and not want_index and not want_debug
    L.check(lib.mnrf_sample_level_dyn(C.byref(d), L.ptr(_f32(sdist_prev)), L.ptr(_f32(w_prev)),
                                      L.ptr(_f32(u_base)), L.ptr(_f32(jitter)), L.ptr(anneal_dev),
                                      L.ptr(sdist), L.stream_ptr()))
    return sdist
  L.check(lib.mnrf_sample_level(C.byref(d), L.ptr(_f32(sdist_prev)), L.ptr(_f32(w_prev)),
                                L.ptr(_f32(u_base)), L.ptr(_f32(jitter)), L.ptr(_f32(cw_in)),
                                L.ptr(sdist), L.ptr(idx), L.ptr(cw), L.ptr(tdil), L.ptr(wdil),
                                L.stream_ptr()))
  if want_index or want_debug:
    return sdist, dict(idx=idx, cw=cw, tdil=tdil, wdil=wdil)
  return sdist


def encode(sdist, origins, directions, radii, near, far, basis, *, min_deg, max_deg,
           raydist_fn=None, ray_shape='cone', warp_contract=False, disable_integration=False,
           feat=None, feat_cols=None, want_f32=False, want_tdist=False, tfeat=None):
  """cast_rays + (contract) + lift + IPE -> bf16 features [B*S, ld] (row stride from `feat`)."""
  lib = L.load()
  if ray_shape not in L.RAY_SHAPE:
    raise ValueError("ray_shape must be 'cone' or 'cylinder'")
  B, S1 = sdist.shape
  S = S1 - 1
  K = basis.shape[0]
  F = 2 * K * (max_deg - min_deg)
  if feat_cols is None:
    feat_cols = (F + 63) // 64 * 64
  if feat is None:
    feat = torch.empty(B * S, feat_cols, device=sdist.device, dtype=torch.bfloat16)
  assert feat.dtype == torch.bfloat16 and feat.stride(1) == 1
  ld = feat.stride(0)
  d = L.EncodeDesc(B, S, L.RAYDIST[raydist_fn], L.RAY_SHAPE[ray_shape], int(warp_contract),
                   int(disable_integration), K, min_deg, max_deg, ld, feat_cols)
  f32 = torch.empty(B * S, F, device=sdist.device) if want_f32 else None
  tdist = torch.empty(B, S + 1, device=sdist.device) if want_tdist else None
  _count()
  if tfeat is not None:
    assert tfeat.dtype == torch.bfloat16 and tfeat.stride(1) == 1 and not want_f32 and not want_tdist
    L.check(lib.mnrf_encode_tangent(C.byref(d), L.ptr(_f32(sdist)), L.ptr(_f32(origins)),
                                    L.ptr(_f32(directions)), L.ptr(_f32(radii)), L.ptr(_f32(near)),
                                    L.ptr(_f32(far)), L.ptr(_f32(basis)), L.ptr(feat), L.ptr(tfeat),
                                    tfeat.stride(0), L.stream_ptr()))
    return feat, None, None
  L.check(lib.mnrf_encode(C.byref(d), L.ptr(_f32(sdist)), L.ptr(_f32(origins)),
                          L.ptr(_f32(directions)), L.ptr(_f32(radii)), L.ptr(_f32(near)),
                          L.ptr(_f32(far)), L.ptr(_f32(basis)), L.ptr(feat), L.ptr(f32),
                          L.ptr(tdist), L.stream_ptr()))
  return feat, f32, tdist


def viewdir_enc(viewdirs, num_samples, deg, out, col0, col_end):
  lib = L.load()
  B = viewdirs.shape[0]
  _count()
  L.check(lib.mnrf_viewdir_enc(B, num_samples, deg, L.ptr(_f32(viewdirs)), L.ptr(out),
                               out.stride(0), col0, col_end, L.stream_ptr()))


def gemm(mode, a, b, out, *, m, n, k, act=L.ACT_NONE, bias=None, rowv=None, colv=None, mask=None,
         maskbits=None, colsum=None, mask_mod=0, addend=None, impl=0):
  """Dense-layer GEMM (see include/mnrf.h).  a/b/out/mask are 2-D views with unit inner stride."""
  lib = L.load()
  for t in (a, b, out) + ((mask,) if mask is not None else ()):
    assert t.stride(-1) == 1
  if maskbits is not None:
    assert maskbits.dtype == torch.int32 and maskbits.stride(-1) == 1
  d = L.GemmDesc(mode, act, m, n, k, a.stride(0), b.stride(0), out.stride(0),
                 mask.stride(0) if mask is not None else 0,
                 maskbits.stride(0) if maskbits is not None else 0,
                 addend.stride(0) if addend is not None else 0, mask_mod, impl)
  _count()
  ev = None
  if GEMM_EVENTS is not None:
    ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    ev[0].record()
  L.check(lib.mnrf_gemm(C.byref(d), L.ptr(a), L.ptr(b), L.ptr(bias), L.ptr(rowv), L.ptr(colv),
                        L.ptr(mask), L.ptr(maskbits), L.ptr(colsum), L.ptr(addend), L.ptr(out), L.stream_ptr()))
  if ev is not None:
    ev[1].record()
    GEMM_EVENTS.append((ev[0], ev[1], 2.0 * m * n * k))
  return out


def gemm_wgrad(x, dy, out, *, m, n, k, bsum=None, side_w=None, side_aw=None, impl=0):
  """dW[m, n] += x[k, m]^T dy[k, n], plus (optional) bsum[n] += column sums of dy (the layer's bias gradient) and
  side_aw[m] += sum_r side_w[r] x[r, m] (weight gradient of a Dense(1) head on x) -- include/mnrf.h."""
  lib = L.load()
  assert x.stride(-1) == 1 and dy.stride(-1) == 1 and out.stride(-1) == 1
  d = L.GemmDesc(L.GEMM_WGRAD, L.ACT_NONE, m, n, k, x.stride(0), dy.stride(0), out.stride(0), 0, 0, 0, 0, impl)
  _count()
  ev = None
  if GEMM_EVENTS is not None:
    ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    ev[0].record()
  L.check(lib.mnrf_gemm_wgrad(C.byref(d), L.ptr(x), L.ptr(dy), L.ptr(bsum), L.ptr(_f32(side_w)), L.ptr(side_aw),
                              L.ptr(out), L.stream_ptr()))
  if ev is not None:
    ev[1].record()
    GEMM_EVENTS.append((ev[0], ev[1], 2.0 * m * n * k))
  return out




def chain_desc(mode, m, layers, *, stream=None, stream_cols=0, head_w=None, head_b=None, head_out=None):
  """Descriptor of one layer-chained launch (include/mnrf.h mnrf_chain_desc).  layers: list of dicts with
  w [256, ldw] bf16, optional bias / maskbits / colsum / out, n_stream, stream_col0, stream_kb0, n_res, res_kb0.
  The tensors must outlive the descriptor (the caller keeps them: level-state / weight buffers)."""
  d = L.ChainDesc()
  d.mode, d.num_layers, d.width, d.stream_cols, d.m = mode, len(layers), 256, stream_cols, m
  if stream is not None:
    assert stream.dtype == torch.bfloat16 and stream.stride(1) == 1
    d.stream, d.ldstream = stream.data_ptr(), stream.stride(0)
  if head_w is not None:
    d.head_w, d.head_out = head_w.data_ptr(), head_out.data_ptr()
    d.head_b = head_b.data_ptr() if head_b is not None else None
  flops = 0.0
  for j, ly in enumerate(layers):
    c = d.layer[j]
    w = ly['w']
    assert w.dtype == torch.bfloat16 and w.stride(1) == 1
    c.w, c.ldw = w.data_ptr(), w.stride(0)
    for name in ('bias', 'colsum'):
      t = ly.get(name)
      setattr(c, name, t.data_ptr() if t is not None else None)
    mb = ly.get('maskbits')
    if mb is not None:
      assert mb.dtype == torch.int32 and mb.stride(1) == 1
      c.maskbits, c.ldmaskbits = mb.data_ptr(), mb.stride(0)
    out = ly.get('out')
    if out is not None:
      assert out.dtype == torch.bfloat16 and out.stride(1) == 1
      c.out, c.ldo = out.data_ptr(), out.stride(0)
    c.n_stream, c.stream_col0, c.stream_kb0 = ly.get('n_stream', 0), ly.get('stream_col0', 0), ly.get('stream_kb0', 0)
    c.n_res, c.res_kb0 = ly.get('n_res', 0), ly.get('res_kb0', 0)
    flops += 2.0 * m * 256 * 64 * (c.n_stream + c.n_res)
  return d, flops


def mlp_chain(desc):
  """One launch for a whole 256-wide trunk (forward) or its input-gradient chain (backward)."""
  lib = L.load()
  d, flops = desc
  _count()
  ev = None
  if GEMM_EVENTS is not None:
    ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    ev[0].record()
  L.check(lib.mnrf_mlp_chain(C.byref(d), L.stream_ptr()))
  if ev is not None:
    ev[1].record()
    GEMM_EVENTS.append((ev[0], ev[1], flops))


def head_fwd(x, w_nk, bias, n_out, k, raw=None):
  lib = L.load()
  M = x.shape[0]
  if raw is None:
    raw = torch.empty(M, n_out, device=x.device)
  _count()
  L.check(lib.mnrf_head_fwd(M, k, n_out, L.ptr(x), x.stride(0), L.ptr(w_nk), L.ptr(bias),
                            L.ptr(raw), L.stream_ptr()))
  return raw


def head_bwd(x, w_nk, draw, n_out, k, dx=None, relu_mask=False, dw=None, db=None, dxsum=None):
  lib = L.load()
  M = x.shape[0]
  _count()
  L.check(lib.mnrf_head_bwd(M, k, n_out, L.ptr(x), x.stride(0), L.ptr(w_nk), L.ptr(_f32(draw)),
                            L.ptr(dx), dx.stride(0) if dx is not None else 0, int(relu_mask),
                            L.ptr(dw), L.ptr(db), L.ptr(dxsum), L.stream_ptr()))


def colsum(x, n, out):
  lib = L.load()
  _count()
  L.check(lib.mnrf_colsum(x.shape[0], n, L.ptr(x), x.stride(0), L.ptr(out), L.stream_ptr()))


def _cdesc(B, S, *, raydist_fn, opaque_background, density_bias, density_noise, rgb_activation,
           rgb_premultiplier, rgb_bias, rgb_padding, bg_const, rgb_mode=0):
  if rgb_activation not in L.RGB_ACT:
    raise ValueError(f'rgb_activation {rgb_activation!r} not supported by the CUDA path')
  return L.CompositeDesc(B, S, L.RAYDIST[raydist_fn], int(opaque_background), float(density_bias),
                         float(density_noise), L.RGB_ACT[rgb_activation], float(rgb_premultiplier),
                         float(rgb_bias), float(rgb_padding), float(bg_const), int(rgb_mode))


def composite_fwd(raw_density, raw_rgb, sdist, directions, near, far, *, cfg, density_noise=None,
                  bg_rgb=None, rgb_scale=None, raw_diffuse=None, raw_tint=None, want_samples=False,
                  want_extras=False):
  """compute_alpha_weights + volumetric_rendering.  cfg: kwargs of _cdesc."""
  lib = L.load()
  B, S = raw_density.shape
  dev = raw_density.device
  d = _cdesc(B, S, **cfg)
  weights = torch.empty(B, S, device=dev)
  rgb = torch.empty(B, 3, device=dev)
  dens = torch.empty(B, S, device=dev) if want_samples else None
  rgbs = torch.empty(B, S, 3, device=dev) if want_samples else None
  acc = torch.empty(B, device=dev) if want_extras else None
  dist = torch.empty(B, 4, device=dev) if want_extras else None
  _count()
  L.check(lib.mnrf_composite_fwd(C.byref(d), L.ptr(_f32(raw_density)), L.ptr(_f32(raw_rgb)),
                                 L.ptr(_f32(density_noise)), L.ptr(_f32(sdist)),
                                 L.ptr(_f32(directions)), L.ptr(_f32(near)), L.ptr(_f32(far)),
                                 L.ptr(_f32(bg_rgb)), L.ptr(_f32(rgb_scale)), L.ptr(_f32(raw_diffuse)),
                                 L.ptr(_f32(raw_tint)), L.ptr(weights), L.ptr(rgb),
                                 L.ptr(dens), L.ptr(rgbs), L.ptr(acc), L.ptr(dist), L.stream_ptr()))
  return dict(weights=weights, rgb=rgb, density=dens, rgb_samples=rgbs, acc=acc, dist=dist)


def composite_bwd(raw_density, raw_rgb, sdist, directions, near, far, target_rgb, lossmult,
                  inv_denom, stats, *, cfg, loss_type, charb_padding, data_mult, distortion_mult,
                  interlevel_mult, sdist_fine=None, weights_fine=None, density_noise=None,
                  bg_rgb=None, rgb_scale=None, d_raw_density=None, d_raw_rgb=None, d_rgb_scale=None,
                  raw_diffuse=None, raw_tint=None, extra_dw=None, d_raw_diffuse=None, d_raw_tint=None):
  lib = L.load()
  B, S = raw_density.shape
  dev = raw_density.device
  Sf = sdist_fine.shape[1] - 1 if sdist_fine is not None else 0
  d = L.LossDesc(_cdesc(B, S, **cfg), L.LOSS_TYPE[loss_type], float(charb_padding), float(data_mult),
                 float(distortion_mult), float(interlevel_mult), Sf,
                 lossmult.shape[-1] if lossmult.dim() > 1 else 1)
  if d_raw_density is None:
    d_raw_density = torch.empty(B, S, device=dev)
  if raw_rgb is not None and d_raw_rgb is None:
    d_raw_rgb = torch.empty(B, S, 3, device=dev)
  _count()
  L.check(lib.mnrf_composite_bwd(C.byref(d), L.ptr(_f32(raw_density)), L.ptr(_f32(raw_rgb)),
                                 L.ptr(_f32(density_noise)), L.ptr(_f32(sdist)),
                                 L.ptr(_f32(directions)), L.ptr(_f32(near)), L.ptr(_f32(far)),
                                 L.ptr(_f32(bg_rgb)), L.ptr(_f32(rgb_scale)), L.ptr(_f32(raw_diffuse)),
                                 L.ptr(_f32(raw_tint)), L.ptr(_f32(extra_dw)), L.ptr(_f32(target_rgb)),
                                 L.ptr(_f32(lossmult)), L.ptr(_f32(inv_denom)),
                                 L.ptr(_f32(sdist_fine)), L.ptr(_f32(weights_fine)),
                                 L.ptr(d_raw_density), L.ptr(d_raw_rgb), L.ptr(d_rgb_scale),
                                 L.ptr(d_raw_diffuse), L.ptr(d_raw_tint), L.ptr(stats), L.stream_ptr()))
  return d_raw_density, d_raw_rgb


def clip_adam(params, grads, mu, nu, scratch, *, step, lr, beta1, beta2, eps, grad_max_val,
              grad_max_norm, grad_scale=1.0, dyn=None):
  lib = L.load()
  d = L.AdamDesc(params.numel(), float(grad_max_val), float(grad_max_norm), float(lr), float(beta1),
                 float(beta2), float(eps), int(step), float(grad_scale))
  _count(2 if grad_max_norm > 0 else 1)
  if dyn is not None:
    L.check(lib.mnrf_clip_adam_dyn(C.byref(d), L.ptr(params), L.ptr(grads), L.ptr(mu), L.ptr(nu),
                                   L.ptr(scratch), L.ptr(dyn), L.stream_ptr()))
    return
  L.check(lib.mnrf_clip_adam(C.byref(d), L.ptr(params), L.ptr(grads), L.ptr(mu), L.ptr(nu),
                             L.ptr(scratch), L.stream_ptr()))


def pack_weights(master, w_nk, w_kn):
  lib = L.load()
  in_pad, out = master.shape
  _count()
  L.check(lib.mnrf_pack_weights(in_pad, out, L.ptr(master), L.ptr(w_nk), L.ptr(w_kn),
                                L.stream_ptr()))


def pack_table(layers, device):
  """Device table for pack_weights_batched: layers = [(master[in_pad,out], w_nk or None, w_kn or None)]."""
  import ctypes
  import numpy as np
  items = (L.PackItem * len(layers))()
  tile = 0
  for i, (master, w_nk, w_kn) in enumerate(layers):
    in_pad, out = master.shape
    items[i] = L.PackItem(master.data_ptr(), w_nk.data_ptr() if w_nk is not None else None,
                          w_kn.data_ptr() if w_kn is not None else None, in_pad, out, tile, 0)
    tile += ((out + 31) // 32) * ((in_pad + 31) // 32)
  raw = np.frombuffer(ctypes.string_at(ctypes.addressof(items), ctypes.sizeof(items)), dtype=np.uint8).copy()
  return torch.from_numpy(raw).to(device), len(layers), tile


def pack_weights_batched(table):
  lib = L.load()
  dev_items, count, tiles = table
  _count()
  L.check(lib.mnrf_pack_weights_batched(count, L.ptr(dev_items), tiles, L.stream_ptr()))


def refdir_desc(M, S, *, use_pred_normals, use_density_normals, use_reflections, use_ide, use_n_dot_v,
                use_roughness, deg_view, ide_n, roughness_bias, ld, col0, col_end):
  return L.RefdirDesc(M, S, int(use_pred_normals), int(use_density_normals), int(use_reflections),
                      int(use_ide), int(use_n_dot_v), int(use_roughness), deg_view, ide_n,
                      float(roughness_bias), ld, col0, col_end)


def refdir_fwd(desc, ide_mat, ide_ml, grad_pred, raw_rough, raw_grad_density, viewdirs, normals_pred,
               normals, roughness, slab, orient_mult=0.0, prednorm_mult=0.0, orient_on_pred=True,
               extra_dw=None):
  lib = L.load()
  _count()
  L.check(lib.mnrf_refdir_fwd(C.byref(desc), L.ptr(ide_mat), L.ptr(ide_ml), L.ptr(_f32(grad_pred)),
                              L.ptr(_f32(raw_rough)), L.ptr(_f32(raw_grad_density)), L.ptr(_f32(viewdirs)),
                              L.ptr(normals_pred), L.ptr(normals), L.ptr(roughness), L.ptr(slab),
                              float(orient_mult), float(prednorm_mult), int(orient_on_pred),
                              L.ptr(extra_dw), L.stream_ptr()))


def refdir_bwd(desc, ide_mat, ide_ml, grad_pred, raw_rough, raw_grad_density, viewdirs, weights, d_slab,
               orient_mult, prednorm_mult, orient_on_pred, d_raw_density, d_raw_diffuse, d_raw_tint,
               d_grad_pred, d_raw_rough, d_raw_grad_density, stats):
  lib = L.load()
  _count()
  L.check(lib.mnrf_refdir_bwd(C.byref(desc), L.ptr(ide_mat), L.ptr(ide_ml), L.ptr(_f32(grad_pred)),
                              L.ptr(_f32(raw_rough)), L.ptr(_f32(raw_grad_density)), L.ptr(_f32(viewdirs)),
                              L.ptr(_f32(weights)), L.ptr(d_slab), d_slab.stride(0), float(orient_mult),
                              float(prednorm_mult), int(orient_on_pred), L.ptr(_f32(d_raw_density)),
                              L.ptr(_f32(d_raw_diffuse)), L.ptr(_f32(d_raw_tint)), L.ptr(d_grad_pred),
                              L.ptr(d_raw_rough), L.ptr(d_raw_grad_density), L.ptr(stats), L.stream_ptr()))


def outer_mask(rowv, colv, maskbits, out, *, rows, n, mask_mod=0):
  lib = L.load()
  _count()
  L.check(lib.mnrf_outer_mask(rows, n, mask_mod, L.ptr(_f32(rowv)), L.ptr(_f32(colv)), L.ptr(maskbits),
                              maskbits.stride(0) if maskbits is not None else 0, L.ptr(out), out.stride(0),
                              L.stream_ptr()))
