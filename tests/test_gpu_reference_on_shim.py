"""Boundary b2 (SURVEY 8b): this stack against the reference's own code.

The reference's files are not part of this repository, so nothing here runs them over shims.install(); test names
that say "reference ... on cuda" compare this package's code on cuda with the reference's stored results.

* The open3d stand-in's registration pipeline (o3d_registration.py: registration_icp /
  registration_ransac_based_on_correspondence behind `open3d.pipelines.registration`) called the way
  core/deep_global_registration.py:50-64,317-322 and util/pointcloud.py:15-23 call open3d, against the library
  entry points and the oracle.
* This package's DeepGlobalRegistration and ResUNetBN2C on cuda against what the reference's UNMODIFIED
  `core/deep_global_registration.py::DeepGlobalRegistration`, `model/resunet.py` and demo.py flow returned on the
  same inputs (run on the CPU over the oracle's MinkowskiEngine stand-in; stored in
  tests/golden/reference_register.npz by tests/golden/make_golden_reference.py), and against the oracle."""
import os
import sys
import types

import numpy as np
import pytest
import torch

from deepglobalregistration_b200 import synthetic as syn

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_register.npz')
EXTENT = (1.8, 1.5, 1.25)


@pytest.fixture(scope='module')
def setup():
  from deepglobalregistration_b200 import _abi, shims
  from deepglobalregistration_b200.core.deep_global_registration import DeepGlobalRegistration
  _abi.require_device('cuda')
  state = syn.make_checkpoint(0)
  d = DeepGlobalRegistration(types.SimpleNamespace(weights=state, clip_weight_thresh=0.05, verbose=False))
  saved = sys.modules.pop('open3d', None)
  o3d = shims._open3d_stub()
  if saved is not None:
    sys.modules['open3d'] = saved
  return d, state, o3d, _abi


def _pcd(o3d, xyz_t):
  """util/pointcloud.py:15-23 make_open3d_point_cloud"""
  pcd = o3d.geometry.PointCloud()
  pcd.points = o3d.utility.Vector3dVector(xyz_t.cpu().detach().numpy())
  return pcd


def test_standin_icp_equals_library_and_oracle(setup):
  from oracle import icp as oicp
  d, state, o3d, abi = setup
  xyz0, xyz1, T_gt = syn.room_pair(4, n_raw=20000, extent=EXTENT)
  with torch.no_grad():
    p0, c0, _ = d.preprocess(xyz0, 0, _batch=0)
    p1, c1, _ = d.preprocess(xyz1, 1, _batch=0)
  T0 = T_gt.copy()
  T0[:3, 3] += 0.02                                        # a perturbed start, as after the refinement
  # the reference's call (core/deep_global_registration.py:317-322)
  res = o3d.pipelines.registration.registration_icp(source=_pcd(o3d, p0), target=_pcd(o3d, p1),
                                                    max_correspondence_distance=d.voxel_size * 2, init=T0)
  lib = abi.icp_point_to_point(p0, p1, c1._dgr_manager, d.voxel_size, 2 * d.voxel_size, T0, batch=0).cpu().numpy()
  assert np.allclose(res.transformation, lib[:16].reshape(4, 4), atol=1e-9)
  assert abs(res.fitness - lib[16]) < 1e-12 and abs(res.inlier_rmse - lib[17]) < 1e-12
  T_o, info = oicp.icp_point_to_point(p0.cpu().numpy(), p1.cpu().numpy(), 2 * d.voxel_size, T0)
  te, re = syn.rte_rre(res.transformation, T_o)
  assert te <= 1e-5 and re <= 1e-5, (te, re)
  assert abs(res.fitness - info['fitness']) <= 1e-9 and len(res.correspondence_set) == info['n_corr']
  # a target that is NOT voxelised (several raw points within a quarter of the search radius): refused loudly
  dense = torch.from_numpy(xyz1[:30000]).float().cuda()
  with pytest.raises(NotImplementedError):
    o3d.pipelines.registration.registration_icp(_pcd(o3d, p0), _pcd(o3d, dense), 0.04, T0)


def test_standin_ransac_equals_library(setup):
  d, state, o3d, abi = setup
  P, Q, idx0, idx1, T_gt, inl = syn.correspondence_set(3, n=3000)
  corres = o3d.utility.Vector2iVector(np.stack((idx0, idx1), axis=1))       # :52-53
  res = o3d.pipelines.registration.registration_ransac_based_on_correspondence(
      source=_pcd(o3d, torch.from_numpy(P)), target=_pcd(o3d, torch.from_numpy(Q)), corres=corres,
      max_correspondence_distance=0.1,
      estimation_method=o3d.pipelines.registration.TransformationEstimationPointToPoint(False), ransac_n=4,
      criteria=o3d.pipelines.registration.RANSACConvergenceCriteria(50000, 80000))
  lib = abi.ransac_correspondence(torch.from_numpy(P).cuda(), torch.from_numpy(Q).cuda(),
                                  torch.from_numpy(idx0.astype(np.int32)).cuda(),
                                  torch.from_numpy(idx1.astype(np.int32)).cuda(), 0.1, num_hyp=50000, seed=0).cpu().numpy()
  assert np.allclose(res.transformation, lib[:16].reshape(4, 4), atol=1e-12)
  te, re = syn.rte_rre(res.transformation, T_gt)
  assert te <= 0.02 and re <= 0.02 and res.fitness > 0.25


# ------------------------------------------------------------------------------------------------------------
# against the reference's own files (their outputs on the same inputs, tests/golden/reference_register.npz)
# ------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def reference():
  return np.load(GOLD)


def test_reference_class_on_cuda_equals_ours_and_oracle(reference, setup):
  """This package's register() on cuda vs the reference class's stored register() of the same pair, and vs the
  oracle (the reference class itself does not run here)."""
  from oracle import pipeline as op
  d, state, _, _ = setup
  xyz0, xyz1, _ = syn.room_pair(2, n_raw=20000, extent=EXTENT)
  T_ref = reference['class_T']                              # the reference's register() (use_icp = True)
  d.use_icp = True
  T_ours = d.register(xyz0, xyz1)
  te, re = syn.rte_rre(T_ref, T_ours)
  print(f'register() vs the reference class: TE={te:.2e} m RE={re:.2e} rad')
  assert te <= 1e-3 and re <= 1e-3, (te, re)
  assert float(np.abs(T_ref - T_ours).max()) <= 1e-5, T_ref - T_ours    # RE's arccos is noisy below ~1e-4
  T_o, _ = op.register(state, xyz0, xyz1, use_icp=True)
  te, re = syn.rte_rre(T_ref, T_o)
  assert te <= 1e-3 and re <= 1e-3, (te, re)


def test_reference_resunet_forward_on_cuda_equals_oracle(reference):
  """This package's ResUNetBN2C on cuda vs the oracle and vs the reference model/resunet.py's stored output."""
  from deepglobalregistration_b200 import me as ME
  from deepglobalregistration_b200.model import load_model
  from oracle.resunet import resunet_forward
  sd = syn.resunet_state_dict(5, 1, 32, 7, 3)
  net = load_model('ResUNetBN2C')(1, 32, bn_momentum=0.05, conv1_kernel_size=7, normalize_feature=True, D=3)
  net.load_state_dict(sd)
  net = net.cuda().eval()
  g = np.random.default_rng(0)
  coords = np.unique(g.integers(-12, 12, size=(6000, 3)), axis=0)
  coords = np.concatenate([np.zeros((len(coords), 1), np.int64), coords], 1).astype(np.int32)
  assert len(coords) == int(reference['resunet_n'])
  with torch.no_grad():
    out = net(ME.SparseTensor(torch.ones(len(coords), 1), coordinates=torch.from_numpy(coords), device='cuda')).F
  out = out.cpu()
  want = resunet_forward(sd, coords, torch.ones(len(coords), 1), 7, True)
  assert float((out - want).abs().max()) <= 5e-5
  rows = torch.from_numpy(reference['resunet_rows']).long()
  assert float((out[rows] - torch.from_numpy(reference['resunet_out'])).abs().max()) <= 5e-5


def test_reference_demo_flow_on_two_ply_files(reference, tmp_path, setup):
  """demo.py:28-48 without its download, with this package's class: read two PLY files with (stand-in) open3d,
  register, transform, 'draw'; the pose is compared with the reference's stored result of the same flow."""
  from deepglobalregistration_b200 import io as dio
  d, state, o3d, _ = setup
  xyz0, xyz1, _ = syn.room_pair(6, n_raw=15000, extent=EXTENT)
  dio.write_ply(str(tmp_path / 'a.ply'), xyz0, dtype='double')
  dio.write_ply(str(tmp_path / 'b.ply'), xyz1, dtype='double')
  pcd0 = o3d.io.read_point_cloud(str(tmp_path / 'a.ply'))
  pcd0.estimate_normals()
  pcd1 = o3d.io.read_point_cloud(str(tmp_path / 'b.ply'))
  pcd1.estimate_normals()
  d.use_icp = True
  T01 = d.register(pcd0, pcd1)
  o3d.visualization.draw_geometries([pcd0, pcd1])
  pcd0.transform(T01)
  te, re = syn.rte_rre(T01, reference['demo_T'])           # the reference's demo flow on the same two files
  print(f'demo flow vs the reference: TE={te:.2e} m RE={re:.2e} rad')
  assert te <= 1e-3 and re <= 1e-3, (te, re)
  assert float(np.abs(reference['demo_T'] - T01).max()) <= 1e-5, reference['demo_T'] - T01
  te, re = syn.rte_rre(T01, d.register(xyz0, xyz1))
  assert te <= 1e-5 and re <= 1e-5
