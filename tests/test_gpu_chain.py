"""The layer-chained 256-wide trunk kernel (csrc/chain.cu, mnrf_mlp_chain) against the per-layer
tcgen05 GEMMs (mnrf_gemm) and a plain fp32 torch product of the same bf16 operands.  Needs a B200.

Reference being replaced: the Dense + ReLU loop of internal/models.py:441-465 (forward, skip concat at
:458-459) and its reverse-mode input-gradient chain."""
import math

import numpy as np
import pytest
import torch

from util import close

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def ops():
  from multinerf_b200 import lib, ops as _ops
  lib.require_device()
  return _ops


def _bf(x):
  return torch.tensor(x).to(torch.bfloat16).cuda()


def _unpack_bits(bits, n):
  return ((bits.cpu().long()[:, :, None] >> torch.arange(32)) & 1).reshape(bits.shape[0], n).bool()


@pytest.mark.parametrize('M,depth,Fpad,skip', [
    (512, 4, 512, 0),          # one unit; PropMLP of 360.gin (icosahedron features, 8 streamed k-blocks)
    (16384, 4, 512, 0),        # 256 rays x 64 samples: 32 units
    (100352, 4, 512, 0),       # 196 units > 74 CTA pairs: several units per pair, ring wrap-around across units
    (1000, 4, 128, 0),         # ragged last unit (rows past M zero-filled / clipped)
    (8320, 8, 128, 4),         # NerfMLP 8 x 256 of the blender / llff configs: skip concat after layer 4
    (4096, 2, 64, 0), (777, 1, 192, 0),
])
def test_chain_forward_vs_per_layer(ops, M, depth, Fpad, skip):
  from multinerf_b200 import lib as L
  rng = np.random.default_rng(M + depth + Fpad)
  W = 256
  feat = _bf(rng.normal(size=(M, Fpad)).astype(np.float32))
  in_pads = [Fpad] + [W + Fpad if (skip and i - 1 == skip) else W for i in range(1, depth)]
  ws = [_bf(rng.normal(size=(W, k)).astype(np.float32) * math.sqrt(2.0 / k)) for k in in_pads]
  bs = [torch.tensor(rng.normal(size=(W,)).astype(np.float32) * 0.1).cuda() for _ in range(depth)]
  hw = _bf(rng.normal(size=(1, W)).astype(np.float32) / 16)
  hb = torch.tensor([0.37]).cuda()
  # ---- per-layer path (the skip layer's input is [hidden | features], as models.py lays it out)
  acts_ref, bits_ref = [], []
  x = feat
  for i in range(depth):
    wide = skip and i == skip
    out = torch.zeros(M, W + Fpad if wide else W, dtype=torch.bfloat16, device='cuda')
    if wide:
      out[:, W:] = feat
    bits = torch.zeros(M, W // 32, dtype=torch.int32, device='cuda')
    ops.gemm(L.GEMM_FWD, x, ws[i], out[:, :W], m=M, n=W, k=in_pads[i], act=L.ACT_RELU, bias=bs[i], maskbits=bits)
    acts_ref.append(out)
    bits_ref.append(bits)
    x = out
  head_ref = ops.head_fwd(acts_ref[-1][:, :W], hw, hb, 1, W)
  # ---- chained
  acts = [torch.full((M, W + Fpad if (skip and i == skip) else W), -7.0, dtype=torch.bfloat16, device='cuda')
          for i in range(depth)]
  bits = [torch.full((M, W // 32), -1, dtype=torch.int32, device='cuda') for _ in range(depth)]
  head = torch.full((M,), -3.0, device='cuda')
  layers = []
  for i in range(depth):
    ly = dict(w=ws[i], bias=bs[i], out=acts[i][:, :W], maskbits=bits[i])
    if i == 0:
      ly.update(n_stream=Fpad // 64, stream_col0=0, stream_kb0=0)
    else:
      ly.update(n_res=4, res_kb0=0)
      if in_pads[i] == W + Fpad:
        ly.update(n_stream=Fpad // 64, stream_col0=0, stream_kb0=4)
    layers.append(ly)
  desc = ops.chain_desc(L.CHAIN_FWD, M, layers, stream=feat, stream_cols=Fpad, head_w=hw[0].float().contiguous(),
                        head_b=hb, head_out=head)
  ops.mlp_chain(desc)
  torch.cuda.synchronize()
  for i in range(depth):
    a, b = acts[i][:, :W].float(), acts_ref[i][:, :W].float()
    # same operands, same fp32 accumulation; only the k-block order of a skip layer differs
    close(a, b, atol=2e-2, rtol=1.6e-2, msg=f'layer {i} activation')
    exact = float((a == b).float().mean())
    assert exact > (0.999 if not skip else 0.98), (i, exact)
    assert torch.equal(_unpack_bits(bits[i], W), a.cpu() > 0), f'layer {i} mask bits'
    if skip and i == skip:
      assert (acts[i][:, W:] == -7).all()            # the chain never touches the feature columns
  close(head, head_ref[:, 0], atol=2e-3, rtol=2e-3, msg='density head')
  # fp32 reference of the first layer from the same bf16 operands
  ref0 = torch.relu(feat.float() @ ws[0].float().T + bs[0])
  close(acts[0][:, :W].float(), ref0.to(torch.bfloat16).float(), atol=2e-2, rtol=1.6e-2, msg='layer 0 vs fp32')
  # inference form: no stores except the last layer, no masks
  last = torch.zeros(M, W, dtype=torch.bfloat16, device='cuda')
  head2 = torch.zeros(M, device='cuda')
  layers2 = [dict(ly) for ly in layers]
  for i, ly in enumerate(layers2):
    ly.pop('maskbits')
    ly.pop('out')
    if i == depth - 1:
      ly['out'] = last
  ops.mlp_chain(ops.chain_desc(L.CHAIN_FWD, M, layers2, stream=feat, stream_cols=Fpad,
                               head_w=hw[0].float().contiguous(), head_b=hb, head_out=head2))
  torch.cuda.synchronize()
  assert torch.equal(last, acts[-1][:, :W]) and torch.equal(head2, head)


@pytest.mark.parametrize('M,depth', [(512, 4), (16384, 4), (100352, 4), (1000, 4), (8320, 8), (640, 2)])
def test_chain_backward_vs_per_layer(ops, M, depth):
  from multinerf_b200 import lib as L
  rng = np.random.default_rng(7 * M + depth)
  W = 256
  dy_last = _bf(rng.normal(size=(M, W)).astype(np.float32))
  # w_kn[l] = [in_pad, out] (rows beyond 256 = feature rows of a skip layer, never used by the dgrad)
  w_kn = [_bf(rng.normal(size=(W + (128 if l == 2 else 0), W)).astype(np.float32) / 16) for l in range(depth)]
  masks = [torch.tensor(rng.integers(-2 ** 31, 2 ** 31, (M, W // 32)).astype(np.int32)).cuda() for _ in range(depth)]
  # ---- per-layer dgrads
  cur = dy_last
  outs_ref, cs_ref = [], []
  for i in range(depth - 1, 0, -1):
    out = torch.empty(M, W, dtype=torch.bfloat16, device='cuda')
    cs = torch.full((W,), 1.5, device='cuda')
    ops.gemm(L.GEMM_DGRAD, cur, w_kn[i], out, m=M, n=W, k=W, maskbits=masks[i - 1], colsum=cs)
    outs_ref.append(out)
    cs_ref.append(cs)
    cur = out
  # ---- chained
  outs = [torch.full((M, W), -7.0, dtype=torch.bfloat16, device='cuda') for _ in range(depth - 1)]
  css = [torch.full((W,), 1.5, device='cuda') for _ in range(depth - 1)]
  layers = []
  for j, i in enumerate(range(depth - 1, 0, -1)):
    ly = dict(w=w_kn[i], maskbits=masks[i - 1], colsum=css[j], out=outs[j])
    ly.update(dict(n_stream=4, stream_col0=0, stream_kb0=0) if j == 0 else dict(n_res=4, res_kb0=0))
    layers.append(ly)
  ops.mlp_chain(ops.chain_desc(L.CHAIN_BWD, M, layers, stream=dy_last, stream_cols=W))
  torch.cuda.synchronize()
  for j in range(depth - 1):
    a, b = outs[j].float(), outs_ref[j].float()
    close(a, b, atol=3e-2, rtol=1.6e-2, msg=f'dgrad {j}')
    assert float((a == b).float().mean()) > 0.999, j
    close(css[j], cs_ref[j], atol=2e-2 * math.sqrt(M), rtol=2e-3, msg=f'bias gradient {j}')
  # fp32 reference of the first chained layer
  mask0 = _unpack_bits(masks[depth - 2], W).cuda()
  ref = (dy_last.float() @ w_kn[depth - 1][:W].float().T) * mask0
  close(outs[0].float(), ref.to(torch.bfloat16).float(), atol=3e-2, rtol=1.6e-2, msg='dgrad 0 vs fp32')


def test_chain_rejects_bad_descriptors(ops):
  from multinerf_b200 import lib as L
  w = torch.zeros(256, 256, dtype=torch.bfloat16, device='cuda')
  x = torch.zeros(512, 256, dtype=torch.bfloat16, device='cuda')
  with pytest.raises(L.MnrfError):       # the first layer has no resident operand
    ops.mlp_chain(ops.chain_desc(L.CHAIN_FWD, 512, [dict(w=w, n_res=4, out=x)], stream=x, stream_cols=256))
  with pytest.raises(L.MnrfError):       # streamed columns outside the tensor
    ops.mlp_chain(ops.chain_desc(L.CHAIN_FWD, 512, [dict(w=w, n_stream=4, stream_col0=64, out=x)], stream=x,
                                 stream_cols=256))
  d, fl = ops.chain_desc(L.CHAIN_FWD, 512, [dict(w=w, n_stream=4, out=x)], stream=x, stream_cols=256)
  d.width = 128
  with pytest.raises(L.MnrfError):
    ops.mlp_chain((d, fl))


def test_model_chain_matches_per_layer_path(monkeypatch):
  """The same train step with the chained trunks (default) and with the per-layer GEMMs.
  `blender1`: one level of the 8 x 256 NerfMLP (skip connection) -- no resampling between the two paths, so the
  gradients agree to rounding.  `360`: PropMLP chained, and the two paths differ by the summation order of
  the density head (1e-7 relative), which moves the resampled positions of the next level by a few ulps;
  the 2^11-frequency IPE features amplify that, so only a loose bound holds there (the same sensitivity shows
  in the oracle comparison of Dense_0, test_gpu_fullwidth.py)."""
  from multinerf_b200 import configs, lib, models, train_utils, utils
  from test_gpu_model import synth_rays
  lib.require_device()
  for which, tol in (('blender1', 5e-3), ('360', 0.2)):
    grads = []
    for chain in (True, False):
      with monkeypatch.context() as mp:
        if not chain:
          mp.setattr(models.Model, '_use_chain', lambda self, plan, M, impl=0: False)
        bundle = configs.bundle_360() if which == '360' else configs.bundle_blender_256()
        if which == 'blender1':
          bundle.model.num_levels = 1
          bundle.model.num_nerf_samples = 64
        bundle.config.grad_max_norm = 0.0
        B = 128
        rays, rng = synth_rays(77, B, 0.2 if which == '360' else 2.0, 1e6 if which == '360' else 6.0,
                               unit_cube=which == '360')
        target = rng.uniform(0, 1, (B, 3)).astype(np.float32)
        model, variables = models.construct_model(78, rays, bundle)
        n_lv = bundle.model.num_levels
        rand = {'jitter': [torch.tensor(rng.uniform(0, 1, (B, 1)).astype(np.float32)) for _ in range(n_lv)]}
        step_fn = train_utils.create_train_step(model, bundle.config)
        state = train_utils.TrainState(variables)
        state, stats, _ = step_fn(rand, state, utils.Batch(rays=rays, rgb=target), None, 0.5)
        torch.cuda.synchronize()
        grads.append((model.export_grads_flax(), stats.materialize()['loss']))
    (g1, l1), (g0, l0) = grads
    assert abs(l1 - l0) < (1e-4 if which == 'blender1' else 1e-2) * max(1.0, abs(l0)), (which, l1, l0)
    for mname in g1:
      for lname in g1[mname]:
        for leaf in ('kernel', 'bias'):
          a = torch.tensor(g1[mname][lname][leaf]).double().flatten()
          b = torch.tensor(g0[mname][lname][leaf]).double().flatten()
          if float(b.norm()) == 0:
            continue
          rel = float((a - b).norm() / b.norm())
          assert rel < tol, (which, mname, lname, leaf, rel)
