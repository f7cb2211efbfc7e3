"""CPU-only tests of the host logic: the C ABI loads and exports every declared symbol, the
gin subset binds the reference's own config files, layer tables reproduce the published
parameter counts, level schedule, chunked render_image, and the world_size-2 collectives (gloo)."""
import os
import re
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_abi_library_loads_and_exports_header_symbols():
  from multinerf_b200 import lib
  if not os.path.exists(lib.LIB_PATH):
    from multinerf_b200 import build
    build.build()
  l = lib.load()
  assert l.mnrf_abi_version() == 1
  header = open(os.path.join(ROOT, 'include', 'mnrf.h')).read()
  declared = set(re.findall(r'\b(mnrf_[a-z0-9_]+)\s*\(', header))
  declared -= {'mnrf_bf16', 'mnrf_stream'}
  assert declared == set(lib.EXPORTED), declared ^ set(lib.EXPORTED)
  for name in declared:
    assert hasattr(l, name)
  # descriptor struct sizes must match the C side (compiled check via a tiny C program)
  import ctypes, subprocess, tempfile
  src = '#include <stdio.h>\n#include "mnrf.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\\n",sizeof(mnrf_sample_desc),sizeof(mnrf_encode_desc),sizeof(mnrf_gemm_desc),sizeof(mnrf_composite_desc),sizeof(mnrf_loss_desc),sizeof(mnrf_adam_desc),sizeof(mnrf_refdir_desc),sizeof(mnrf_camera_desc),sizeof(mnrf_pack_item),sizeof(mnrf_chain_layer),sizeof(mnrf_chain_desc));return 0;}'
  with tempfile.TemporaryDirectory() as td:
    open(os.path.join(td, 'a.c'), 'w').write(src)
    subprocess.run(['gcc', '-I', os.path.join(ROOT, 'include'), os.path.join(td, 'a.c'), '-o', os.path.join(td, 'a')], check=True)
    sizes = list(map(int, subprocess.run([os.path.join(td, 'a')], capture_output=True, text=True).stdout.split()))
  assert sizes == [ctypes.sizeof(lib.SampleDesc), ctypes.sizeof(lib.EncodeDesc), ctypes.sizeof(lib.GemmDesc),
                   ctypes.sizeof(lib.CompositeDesc), ctypes.sizeof(lib.LossDesc), ctypes.sizeof(lib.AdamDesc),
                   ctypes.sizeof(lib.RefdirDesc), ctypes.sizeof(lib.CameraDesc), ctypes.sizeof(lib.PackItem),
                   ctypes.sizeof(lib.ChainLayer), ctypes.sizeof(lib.ChainDesc)]


def test_no_cpu_fallback():
  from multinerf_b200 import lib, models, configs
  if torch.cuda.is_available():
    pytest.skip('GPU present')
  with pytest.raises(lib.MnrfError):
    models.Model(configs.bundle_360())
  with pytest.raises(lib.MnrfError):
    lib.ptr(torch.zeros(3))


def test_product_never_imports_oracle():
  for dirpath, _, files in os.walk(os.path.join(ROOT, 'multinerf_b200')):
    for f in files:
      if f.endswith('.py'):
        src = open(os.path.join(dirpath, f)).read()
        assert not re.search(r'^\s*(from|import)\s+oracle', src, re.M), f


def test_gin_subset_binds_reference_configs():
  import json
  from multinerf_b200 import configs
  b = configs.bundle_360()
  assert b.config.near == 0.2 and b.config.far == 1e6 and b.model.raydist_fn == 'reciprocal'
  assert b.model.opaque_background and b.nerf_mlp.net_width == 1024 and b.prop_mlp.warp_fn == 'contract'
  assert b.prop_mlp.disable_rgb and b.model.num_levels == 3          # defaults stay
  # the reference's configs/*.gin, byte for byte, and the bindings each one makes (make_golden_configs.py)
  ref = os.path.join(ROOT, 'tests', 'golden', 'configs')
  with open(os.path.join(ROOT, 'tests', 'golden', 'configs.json')) as fh:
    recorded = json.load(fh)
  assert sorted(f for f in os.listdir(ref) if f.endswith('.gin')) == sorted(recorded) and len(recorded) == 13
  fields = {'Config': 'config', 'Model': 'model', 'NerfMLP': 'nerf_mlp', 'PropMLP': 'prop_mlp'}
  for f, cfg in sorted(recorded.items()):      # the shipped files parse unmodified, and every binding we know lands
    got = configs.load_config([os.path.join(ref, f)], search_paths=[ref])
    for sel, v in cfg['bindings']:
      cls, attr = sel.rsplit('.', 1)
      target = getattr(got, fields[cls])
      if hasattr(target, attr):
        assert getattr(target, attr) == (v['ref'].split('.')[-1] if isinstance(v, dict) else v), (f, sel)
  r = configs.load_config([os.path.join(ref, 'blender_refnerf.gin')])
  assert r.nerf_mlp.use_reflections and r.nerf_mlp.deg_view == 5 and r.model.single_mlp
  assert r.config.orientation_loss_target == 'normals_pred' and r.model.resample_padding == 0.01
  raw = configs.load_config([os.path.join(ref, 'llff_raw.gin')])
  assert raw.nerf_mlp.rgb_activation == 'safe_exp' and raw.nerf_mlp.rgb_bias == -5.0
  assert raw.config.data_loss_type == 'rawnerf' and raw.model.ray_shape == 'cylinder'
  raw_test = configs.load_config([os.path.join(ref, 'llff_raw_test.gin')])      # include + override
  assert raw_test.config.factor == 0 and raw_test.config.data_loss_type == 'rawnerf'
  same = configs.load_config([os.path.join(ref, '360.gin')])
  assert same == configs.bundle_360()
  assert configs.load_config([os.path.join(ref, 'blender_256.gin')]) == configs.bundle_blender_256()
  assert r == configs.bundle_blender_refnerf() and raw == configs.bundle_llff_raw()
  b2 = configs.load_config(gin_bindings=['Config.batch_size = 4096', "Model.ray_shape = 'cylinder'",
                                         'NerfMLP.net_activation = @jax.nn.relu', 'Unknown.thing = 3'])
  assert b2.config.batch_size == 4096 and b2.model.ray_shape == 'cylinder' and b2.nerf_mlp.net_activation == 'relu'
  bad = configs.Bundle()
  bad.nerf_mlp.use_reflections = True
  bad.nerf_mlp.disable_density_normals = True
  with pytest.raises(ValueError):
    bad.nerf_mlp.validate()       # internal/models.py:383-385


def test_layer_tables_reproduce_published_param_counts():
  # scripts/generate_tables.ipynb:145 (9,007,493) and the blender_256 row (835,205)
  from multinerf_b200 import configs
  from multinerf_b200.models import MLPPlan
  b = configs.bundle_360()
  n, p = MLPPlan(b.nerf_mlp), MLPPlan(b.prop_mlp)
  assert (n.K, n.L, n.F, n.Fpad) == (21, 12, 504, 512)
  assert n.num_params == 8680580 and p.num_params == 326913 and n.num_params + p.num_params == 9007493
  shapes = [(s.in_dim, s.out_dim) for s in n.specs]
  assert shapes == [(504, 1024)] + [(1024, 1024)] * 4 + [(1528, 1024)] + [(1024, 1024)] * 2 + \
      [(1024, 1), (1024, 256), (283, 128), (128, 3)]
  assert [s.in_pad for s in n.specs][5] == 1536 and n.specs[10].in_pad == 320
  bb = configs.bundle_blender_256()
  assert MLPPlan(bb.nerf_mlp).num_params + MLPPlan(bb.prop_mlp).num_params == 835205
  with pytest.raises(NotImplementedError):
    bb.nerf_mlp.net_activation = 'silu'          # only the ReLU trunk has a CUDA path
    MLPPlan(bb.nerf_mlp)
  # blender_refnerf.gin: 713,230 (scripts/generate_tables.ipynb Ref-NeRF row) and its layer order
  ref = configs.Bundle()
  n = ref.nerf_mlp
  n.net_depth_viewdirs, n.basis_shape, n.basis_subdivisions, n.disable_density_normals = 8, 'octahedron', 1, False
  n.enable_pred_normals = n.use_directional_enc = n.use_reflections = n.enable_pred_roughness = True
  n.use_diffuse_color = n.use_specular_tint = n.use_n_dot_v = True
  n.deg_view, n.bottleneck_width, n.density_bias, n.max_deg_point = 5, 128, 0.5, 16
  rp = MLPPlan(n)
  assert rp.num_params == 713230
  assert [sp.role for sp in rp.specs[8:14]] == ['density', 'grad_pred', 'diffuse', 'tint', 'roughness', 'bottleneck']
  assert (rp.vin_dim, rp.vin_pad, rp.view_concat_after) == (201, 256, [4]) and rp.specs[19].in_dim == 329


def test_level_schedule_matches_reference_constants():
  # SURVEY appendix A: dilation 0.0103125 (level 1) and 0.0026220703125 (level 2); anneal 0.9091
  from multinerf_b200 import configs, models
  m = models.Model.__new__(models.Model)
  m.mcfg = configs.bundle_360().model
  s_near, s_far, sched = models.Model.level_schedule(m, 0.5)
  assert (s_near, s_far) == (0.0, 1.0)
  assert [lv['S'] for lv in sched] == [64, 64, 32]
  assert sched[1]['dilation'] == 0.0103125 and sched[2]['dilation'] == 0.0026220703125
  assert not sched[0]['use_dilation'] and sched[1]['use_dilation']
  assert abs(sched[0]['anneal'] - 10 * 0.5 / (9 * 0.5 + 1)) < 1e-12


def test_learning_rate_matches_reference_run():
  from multinerf_b200 import train_utils
  g = np.load(os.path.join(ROOT, 'tests', 'golden', 'math.npz'))
  for s, lr, lr2 in zip(g['steps'], g['lrs'], g['lrs_nodelay']):
    assert abs(train_utils.learning_rate_decay(int(s), 2e-3, 2e-5, 250000, 512, 0.01) - lr) <= 1e-6 * lr
    assert abs(train_utils.learning_rate_decay(int(s), 1e-3, 1e-5, 500000) - lr2) <= 1e-6 * lr2
  with pytest.raises(ValueError):
    train_utils.learning_rate_decay(1, 0.0, 1e-5, 10)


def test_shard_unshard_and_render_image_chunking():
  from multinerf_b200 import configs, models, utils
  x = np.arange(24, dtype=np.float32).reshape(12, 2)
  assert utils.shard(x, 4).shape == (4, 3, 2)
  np.testing.assert_array_equal(utils.unshard(utils.shard(x, 4)), x)
  np.testing.assert_array_equal(utils.unshard(utils.shard(x, 4), padding=2), x[:-2])
  H, W = 7, 9                           # 63 rays, chunks of 16 -> 3 full + one of 15 (padded to 16 for world 2)
  f = np.float32
  o = np.arange(H * W * 3, dtype=f).reshape(H, W, 3)
  rays = utils.Rays(origins=o, directions=o + 1, viewdirs=o, radii=np.ones((H, W, 1), f),
                    imageplane=np.zeros((H, W, 2), f), lossmult=np.ones((H, W, 1), f),
                    near=np.ones((H, W, 1), f), far=np.ones((H, W, 1), f), cam_idx=np.zeros((H, W, 1), np.int32))
  cfg = configs.Config(render_chunk_size=16, vis_num_rays=4)
  calls = []

  def render_fn(rng, chunk):            # world_size 1: renders the chunk it is given
    calls.append(chunk.origins.shape[0])
    a = torch.tensor(chunk.origins)
    return [{'rgb': a * (lv + 1), 'acc': a[:, 0] * (lv + 1), 'ray_sdist': torch.zeros(4, 3)} for lv in range(2)], None
  out = models.render_image(render_fn, rays, None, cfg, verbose=False)
  assert out['rgb'].shape == (H, W, 3) and out['acc'].shape == (H, W)
  np.testing.assert_array_equal(out['rgb'].numpy(), 2 * o)           # last level is kept
  assert calls == [16, 16, 16, 15] and len(out['ray_sdist']) == 2     # ray_* bundles: all levels

  # world_size 2: each rank is handed its half of the edge-padded chunk; the fake render_fn returns
  # a "gathered" buffer of the padded size, render_image strips the padding
  flat = o.reshape(-1, 3)
  seen = {0: [], 1: []}
  for rank in range(2):
    def fn(rng, chunk, rank=rank):
      seen[rank].append(np.array(chunk.origins))
      n = chunk.origins.shape[0]
      return [{'rgb': torch.zeros(2 * n, 3), 'ray_sdist': torch.zeros(4, 3)}], None
    r = models.render_image(fn, rays, None, cfg, verbose=False, world_size=2, rank=rank)
    assert r['rgb'].shape == (H, W, 3)
  r0, r1 = np.concatenate(seen[0]), np.concatenate(seen[1])
  assert r0.shape[0] == r1.shape[0] == 32            # 3*8 + 8 (last chunk 15 -> padded to 16)
  np.testing.assert_array_equal(r0[:8], flat[:8])
  np.testing.assert_array_equal(r1[:8], flat[8:16])
  np.testing.assert_array_equal(r1[-1], flat[-1])    # edge padding repeats the last ray
  np.testing.assert_array_equal(r1[-2], flat[-1])


def _gloo_worker(rank, world, port, q):
  import torch.distributed as dist
  os.environ['MASTER_ADDR'] = '127.0.0.1'
  os.environ['MASTER_PORT'] = str(port)
  dist.init_process_group('gloo', rank=rank, world_size=world)
  sys.path.insert(0, ROOT)
  from multinerf_b200 import train_utils
  rend = [{'rgb': torch.full((4, 3), float(rank)), 'acc': torch.arange(4.) + 10 * rank,
           'ray_sdist': torch.full((2, 5), float(rank))}]
  g = train_utils.gather_renderings(rend, world)
  # two levels: only the last one travels (render_image keeps nothing else), ray_* bundles stay local
  two = train_utils.gather_renderings([dict(rend[0]), dict(rend[0])], world)
  assert set(two[0]) == {'ray_sdist'} and two[1]['rgb'].shape == (8, 3)
  assert train_utils.gather_renderings([dict(rend[0]), dict(rend[0])], world, all_levels=True)[0]['acc'].shape == (8,)
  # the train step's single flat exchange: gradients + the stats tail in one all-reduce
  from multinerf_b200 import configs, models
  b = configs.bundle_blender_256()
  prm = models.Params({'NerfMLP_0': models.MLPPlan(b.nerf_mlp, True)}, 'cpu', {})
  prm.grads.fill_(float(rank + 1))
  prm.stats_tail.fill_(float(rank))
  assert train_utils.allreduce_flat_(prm, world) == 0.5
  assert float(prm.grads.min()) == float(prm.grads.max()) == 3.0 and float(prm.stats_tail.max()) == 1.0
  q.put((rank, g[0]['rgb'][:, 0].tolist(), g[0]['acc'].tolist(), g[0]['ray_sdist'][0, 0].item()))
  dist.destroy_process_group()


def test_world_size_2_collectives_gloo():
  import torch.multiprocessing as mp
  ctx = mp.get_context('spawn')
  q = ctx.Queue()
  port = 29600 + os.getpid() % 300
  procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
  for p in procs:
    p.start()
  res = sorted(q.get(timeout=60) for _ in range(2))
  for p in procs:
    p.join(30)
  for rank, rgb, acc, rs in res:
    assert rgb == [0.0] * 4 + [1.0] * 4                   # rank r's rows at [r*n, (r+1)*n)
    assert acc == [0., 1., 2., 3., 10., 11., 12., 13.]
    assert rs == float(rank)                              # ray_* bundles stay local


def test_checkpoint_roundtrip_cpu(tmp_path):
  """checkpoints.save/restore/latest on host tensors (state = step + params + Adam moments; layout
  mismatch is an error; `keep` prunes the oldest files) -- train.py:84,219-223 semantics."""
  import torch
  from multinerf_b200 import checkpoints, configs, models, train_utils
  b = configs.bundle_360()
  plans = {'NerfMLP_0': models.MLPPlan(b.nerf_mlp, True), 'PropMLP_0': models.MLPPlan(b.prop_mlp, True)}
  p = models.Params(plans, 'cpu', {})
  g = torch.Generator().manual_seed(0)
  for buf in (p.flat, p.mu, p.nu):
    buf.copy_(torch.randn(buf.shape, generator=g))
  p.step = 7
  state = train_utils.TrainState(p)
  d = str(tmp_path / 'ck')
  assert checkpoints.latest_checkpoint(d) is None
  assert checkpoints.restore_checkpoint(d, state) is state and state.step == 7      # nothing to restore
  for s in (1, 5, 7):
    checkpoints.save_checkpoint(d, state, s, keep=2)
  assert sorted(os.listdir(d)) == ['checkpoint_5', 'checkpoint_7']
  assert checkpoints.latest_checkpoint(d).endswith('checkpoint_7')
  q = models.Params(plans, 'cpu', {})
  st2 = checkpoints.restore_checkpoint(d, train_utils.TrainState(q))
  assert st2.step == 7 and torch.equal(q.flat, p.flat) and torch.equal(q.mu, p.mu) and torch.equal(q.nu, p.nu)
  other = models.Params({'NerfMLP_0': plans['NerfMLP_0']}, 'cpu', {})
  with pytest.raises(ValueError):
    checkpoints.restore_checkpoint(d, train_utils.TrainState(other))


def test_camera_host_helpers():
  """multinerf_b200.camera_utils host one-liners vs the oracle's (camera_utils.py:398-424) and the
  Pixels container (internal/utils.py:31-41)."""
  import torch
  from multinerf_b200 import camera_utils, utils
  from oracle import o_camera
  p = camera_utils.get_pixtocam(123.0, 64, 48)
  np.testing.assert_allclose(p, o_camera.get_pixtocam(123.0, 64, 48).numpy(), atol=1e-15)
  np.testing.assert_allclose(camera_utils.intrinsic_matrix(1.0, 2.0, 3.0, 4.0),
                             o_camera.intrinsic_matrix(1.0, 2.0, 3.0, 4.0).numpy())
  x, y = camera_utils.pixel_coordinates(5, 3)
  ox, oy = o_camera.pixel_coordinates(5, 3)
  assert x.shape == (3, 5) and np.array_equal(x, ox.numpy()) and np.array_equal(y, oy.numpy())
  assert camera_utils.ProjectionType('fisheye') is camera_utils.ProjectionType.FISHEYE
  px = utils.Pixels(pix_x_int=x, pix_y_int=y, lossmult=None, near=None, far=None, cam_idx=None)
  assert px.exposure_idx is None and px.exposure_values is None
  with pytest.raises(lib_error()):
    camera_utils.pixels_to_rays(x, y, p, np.eye(4)[:3], device='cpu')      # no CPU path


def test_bench_dump_outputs_budget_and_sampling(tmp_path):
  """bench.py --dump-outputs: float32 / float64 .npy files, DUMP_BYTES in all at most, small arrays whole,
  the large ones sampled at the same positions on every run."""
  sys.path.insert(0, ROOT)
  import bench
  arrays = {'params': torch.arange(10**7, dtype=torch.float32), 'adam_mu': -torch.arange(10**7, dtype=torch.float32),
            'mses': torch.ones(3, dtype=torch.bfloat16), 'loss': np.float64(0.25)}
  for d in ('a', 'b'):
    bench.dump_outputs(str(tmp_path / d), arrays)
  a = {p.stem: np.load(p) for p in (tmp_path / 'a').glob('*.npy')}
  b = {p.stem: np.load(p) for p in (tmp_path / 'b').glob('*.npy')}
  assert sum(p.stat().st_size for p in (tmp_path / 'a').iterdir()) <= bench.DUMP_BYTES
  assert a['loss'].dtype == np.float64 and float(a['loss']) == 0.25
  assert a['mses'].dtype == np.float32 and a['mses'].tolist() == [1.0] * 3
  assert a['params'].dtype == np.float32 and 0 < a['params'].size < 10**7
  assert np.all(np.diff(a['params']) > 0)                    # positions in index order, no repeats
  np.testing.assert_array_equal(a['adam_mu'], -a['params'])  # same positions for same-size arrays
  for k in a:
    np.testing.assert_array_equal(a[k], b[k])
  import json
  index = json.loads((tmp_path / 'a' / 'dump.json').read_text())['arrays']
  assert index['mses'] == {'shape': [3], 'kept': None} and index['loss'] == {'shape': [], 'kept': None}
  assert index['params']['shape'] == [10**7] and index['params']['kept'] == a['params'].size
  # the sample is traceable: element j of params.npy is params[sample_positions(size, kept)[j]]
  np.testing.assert_array_equal(a['params'], bench.sample_positions(10**7, index['params']['kept']))


def lib_error():
  from multinerf_b200 import lib
  return (lib.MnrfError, RuntimeError, AssertionError)
