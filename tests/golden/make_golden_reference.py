"""Generate tests/golden/reference_model.npz and tests/golden/reference_register.npz by running the
UNMODIFIED reference code of Deep Global Registration on the CPU:

    python tests/golden/make_golden_reference.py --reference <checkout of the reference project>

The reference's model/*.py, core/*.py and util/*.py are imported from that checkout with
  * MinkowskiEngine -> oracle/me_cpu.py (the sparse operators of oracle/sparse_ops.py),
  * open3d          -> the I/O stand-in of shims.py, with registration_icp backed by oracle/icp.py,
and the outputs the parity tests compare with are stored, so that the tests need neither the reference
tree nor MinkowskiEngine:

reference_model.npz (tests/test_oracle_graph_vs_reference.py, tests/test_abi_and_host.py)
  graph{i}_rows / _out      ResUNetBN2C forward of case i of GRAPH_CASES at a seeded sample of rows
  state_dict_shapes         JSON: the reference ResUNetBN2C(1, 32, conv1_kernel_size=7)'s state-dict keys and shapes

reference_register.npz (tests/test_oracle_pipeline_vs_reference.py, tests/test_gpu_reference_on_shim.py)
  reg_{ones,coords}_*       DeepGlobalRegistration.register() of syn.room_pair(7) on REGISTER_CASES: the pose,
                            the printed gate line, the arguments handed to open3d's ICP, and the outputs of
                            preprocess() (sha256 of the arrays) / fcgf_feature_extraction() (sampled rows) of cloud 0
  surface                   JSON: parameter names and default reprs of the class's public methods
  class_T                   register() of syn.room_pair(2, 20000) with syn.make_checkpoint(0)
  demo_T                    the demo flow (two PLY files read with open3d) on syn.room_pair(6, 15000)
  resunet_rows / _out       sampled rows of ResUNetBN2C forward on 6000 random 3-D coordinates
"""
import argparse
import contextlib
import hashlib
import inspect
import io
import json
import os
import sys
import tempfile
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from deepglobalregistration_b200 import io as dio            # noqa: E402
from deepglobalregistration_b200 import shims                # noqa: E402
from deepglobalregistration_b200 import synthetic as syn     # noqa: E402
from oracle import icp as oicp                                # noqa: E402
from oracle import me_cpu                                     # noqa: E402

# (D, cin, cout, conv1 kernel, normalize, n, extent): the cases of tests/test_oracle_graph_vs_reference.py
GRAPH_CASES = [
    (3, 1, 32, 7, True, 600, 7),        # FCGF, 3DMatch setting
    (3, 1, 32, 5, True, 500, 9),        # FCGF, KITTI setting
    (6, 1, 1, 3, False, 300, 2),        # inlier network, 'ones' features
    (6, 6, 1, 3, False, 250, 2),        # inlier network, 'coords' features
]
REGISTER_CASES = [('ones', np.float64), ('coords', np.float32)]
SHIM_EXTENT = (1.8, 1.5, 1.25)
SAMPLE_ROWS = 256                 # feature rows stored per output: a fixed, seeded sample keeps the files small
_REF_PACKAGES = ('model', 'core', 'util')


def sha(a):
  return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def sample_rows(n, seed):
  return np.sort(np.random.default_rng(seed).choice(n, min(n, SAMPLE_ROWS), replace=False)).astype(np.int32)


def graph_inputs(D, cin, cout, k1, n, extent):
  """State dict, coordinates and features of one graph case (built the same way by the test)."""
  sd = syn.resunet_state_dict(D + k1, cin, cout, k1, D)
  g = torch.Generator().manual_seed(1)
  for k in sd:                                  # non-trivial BN statistics so a misplaced norm shows
    if k.endswith('running_mean'):
      sd[k] = 0.1 * torch.randn(sd[k].shape, generator=g)
    if k.endswith('bn.bias'):
      sd[k] = 0.1 * torch.randn(sd[k].shape, generator=g)
  rng = np.random.default_rng(D)
  c = np.unique(rng.integers(-extent, extent, size=(n, D)), axis=0)
  coords = np.concatenate([np.zeros((len(c), 1), np.int64), c], 1).astype(np.int32)
  feats = torch.ones(len(coords), cin) if cin == 1 else torch.randn(len(coords), cin, generator=g)
  return sd, coords, feats


def resunet_inputs():
  sd = syn.resunet_state_dict(5, 1, 32, 7, 3)
  g = np.random.default_rng(0)
  coords = np.unique(g.integers(-12, 12, size=(6000, 3)), axis=0)
  coords = np.concatenate([np.zeros((len(coords), 1), np.int64), coords], 1).astype(np.int32)
  return sd, coords


@contextlib.contextmanager
def reference_modules(ref):
  """The reference's packages importable on a CPU-only machine; yields the registration_icp calls and the
  checkpoints torch.load hands back."""
  restore_me = me_cpu.install()
  o3d = shims._open3d_stub()
  reg = types.ModuleType('open3d.pipelines.registration')
  icp_calls = []

  def registration_icp(source, target, max_correspondence_distance, init=np.eye(4), *a, **k):
    icp_calls.append(dict(init=np.array(init), max_dist=max_correspondence_distance, n_source=len(source.points),
                          n_target=len(target.points)))
    T, info = oicp.icp_point_to_point(np.asarray(source.points), np.asarray(target.points),
                                      max_correspondence_distance, init)
    return types.SimpleNamespace(transformation=T, fitness=info['fitness'], inlier_rmse=info['inlier_rmse'])
  reg.registration_icp = registration_icp
  o3d.pipelines = types.ModuleType('open3d.pipelines')
  o3d.pipelines.registration = o3d.registration = reg
  for k in [k for k in sys.modules if k == 'open3d' or k.startswith('open3d.') or k.split('.')[0] in _REF_PACKAGES]:
    del sys.modules[k]
  sys.modules['open3d'] = o3d
  sys.path.insert(0, ref)
  real_load = torch.load
  preloaded = {}
  # the reference torch.load()s config.weights: hand back the in-memory checkpoint registered for the path
  torch.load = lambda f, *a, **k: preloaded[str(f)] if str(f) in preloaded else real_load(f, *a, **k)
  try:
    yield types.SimpleNamespace(icp_calls=icp_calls, preloaded=preloaded, o3d=o3d)
  finally:
    torch.load = real_load
    sys.path.remove(ref)
    restore_me()


def reference_dgr(env, state, tmp, **kw):
  from core.deep_global_registration import DeepGlobalRegistration
  path = os.path.join(tmp, 'ckpt.pth')
  open(path, 'wb').close()
  env.preloaded[path] = state
  return DeepGlobalRegistration(types.SimpleNamespace(weights=path, clip_weight_thresh=0.05, **kw),
                                device=torch.device('cpu'))


def model_fixtures(ref):
  out = {}
  with reference_modules(ref):
    from model import load_model
    import MinkowskiEngine as ME
    for i, (D, cin, cout, k1, normalize, n, extent) in enumerate(GRAPH_CASES):
      sd, coords, feats = graph_inputs(D, cin, cout, k1, n, extent)
      net = load_model('ResUNetBN2C')(cin, cout, bn_momentum=0.05, conv1_kernel_size=k1, normalize_feature=normalize, D=D)
      net.load_state_dict(sd, strict=True)
      net.eval()
      with torch.no_grad():
        F = net(ME.SparseTensor(feats, coordinates=coords)).F.numpy()
      out[f'graph{i}_rows'] = rows = sample_rows(len(F), i)
      out[f'graph{i}_out'] = F[rows].astype(np.float32)
    net = load_model('ResUNetBN2C')(1, 32, bn_momentum=0.05, conv1_kernel_size=7, normalize_feature=True)
    sd = net.state_dict()
    out['state_dict_shapes'] = json.dumps({k: list(v.shape) for k, v in sd.items()})
  return out


def register_fixtures(ref):
  out = {}
  with reference_modules(ref) as env, tempfile.TemporaryDirectory() as tmp:
    from core.deep_global_registration import DeepGlobalRegistration
    for feature_type, dtype in REGISTER_CASES:
      state = syn.make_checkpoint(1, inlier_feature_type=feature_type)
      xyz0, xyz1, _ = syn.room_pair(7, n_raw=5000, extent=(1.2, 1.0, 0.8))
      xyz0, xyz1 = xyz0.astype(dtype), xyz1.astype(dtype)
      dgr = reference_dgr(env, state, tmp)
      env.icp_calls.clear()
      buf = io.StringIO()
      with contextlib.redirect_stdout(buf):
        T = dgr.register(xyz0, xyz1)
      call, = env.icp_calls
      p0, c0, f0 = dgr.preprocess(xyz0)
      with torch.no_grad():
        F0 = dgr.fcgf_feature_extraction(f0, c0)
      k = f'reg_{feature_type}_'
      out.update({k + 'T': T, k + 'use_icp': dgr.use_icp, k + 'voxel_size': dgr.voxel_size,
                  k + 'printed': [ln for ln in buf.getvalue().splitlines() if 'Weighted sum' in ln][0],
                  k + 'icp_init': call['init'], k + 'icp_max_dist': call['max_dist'],
                  k + 'icp_n_source': call['n_source'], k + 'icp_n_target': call['n_target'],
                  k + 'sha_p0': sha(p0.numpy()), k + 'sha_c0': sha(c0.numpy()), k + 'f0_shape': np.array(f0.shape),
                  k + 'p0_dtype': str(p0.dtype), k + 'c0_dtype': str(c0.dtype),
                  k + 'F0_rows': sample_rows(len(F0), 0), k + 'F0': F0.numpy()[sample_rows(len(F0), 0)]})
      print(f'register {feature_type}: N0={len(c0)} {out[k + "printed"]}', flush=True)

    surface = {}
    for name, f in inspect.getmembers(DeepGlobalRegistration, inspect.isfunction):
      if not name.startswith('_') or name == '__init__':
        surface[name] = [[p.name, p.default is not inspect.Parameter.empty,
                          None if p.default is inspect.Parameter.empty else repr(p.default)]
                         for p in inspect.signature(f).parameters.values()]
    out['surface'] = json.dumps(surface)

    state = syn.make_checkpoint(0)
    xyz0, xyz1, _ = syn.room_pair(2, n_raw=20000, extent=SHIM_EXTENT)
    out['class_T'] = reference_dgr(env, state, tmp).register(xyz0, xyz1)
    print('class_T done', flush=True)

    # demo.py's flow: two PLY files read with open3d, registered, transformed
    xyz0, xyz1, _ = syn.room_pair(6, n_raw=15000, extent=SHIM_EXTENT)
    a, b = os.path.join(tmp, 'a.ply'), os.path.join(tmp, 'b.ply')
    dio.write_ply(a, xyz0, dtype='double')
    dio.write_ply(b, xyz1, dtype='double')
    dgr = reference_dgr(env, state, tmp, pcd0=a, pcd1=b)
    pcd0, pcd1 = env.o3d.io.read_point_cloud(a), env.o3d.io.read_point_cloud(b)
    out['demo_T'] = dgr.register(pcd0, pcd1)
    print('demo_T done', flush=True)

    from model.resunet import ResUNetBN2C
    import MinkowskiEngine as ME
    sd, coords = resunet_inputs()
    net = ResUNetBN2C(1, 32, bn_momentum=0.05, conv1_kernel_size=7, normalize_feature=True, D=3)
    net.load_state_dict(sd)
    net.eval()
    with torch.no_grad():
      F = net(ME.SparseTensor(torch.ones(len(coords), 1), coordinates=coords)).F.numpy()
    out['resunet_n'] = len(coords)
    out['resunet_rows'] = rows = sample_rows(len(F), 1)
    out['resunet_out'] = F[rows].astype(np.float32)
  return out


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--reference', required=True, help='checkout of the reference Deep Global Registration project')
  args = ap.parse_args()
  ref = os.path.abspath(args.reference)
  torch.set_num_threads(min(32, os.cpu_count() or 1))
  for name, fn in (('reference_model.npz', model_fixtures), ('reference_register.npz', register_fixtures)):
    path = os.path.join(HERE, name)
    np.savez_compressed(path, **fn(ref))
    print(f'{path}: {os.path.getsize(path) / 1e6:.2f} MB', flush=True)


if __name__ == '__main__':
  main()
