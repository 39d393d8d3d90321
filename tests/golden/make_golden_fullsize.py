"""Generate tests/golden/fullsize_config{2,3}.npz: the CPU oracle (oracle/pipeline.py) run ONCE at
the BASELINE.json sizes, stored as compact taps so that the `-m gpu` parity tests and bench.py's
`parity` block can compare the CUDA path with the oracle at the sizes the benchmark runs at:

  config 2   the bench's own first pair: syn.room_pair(0, n_raw=250_000), checkpoint
             syn.make_checkpoint(0) (voxel 0.05 m, FCGF conv1 k=7)  -> N0 ~ 51k / N1 ~ 40k voxels
  config 3   the full KITTI-shape pair syn.lidar_pair(0), checkpoint
             syn.make_checkpoint(3, voxel_size=0.3, feat_conv1_kernel_size=5) -> ~16k voxels

    python tests/golden/make_golden_fullsize.py [2] [3]          (minutes of CPU per config)

What is stored (everything else is re-derivable from these on the GPU box without the oracle):
  n0, n1                     voxel counts
  sha_*                      sha256 of sel0 / sel1 (int64), coords0 / coords1 / coords6 (int32) bytes
  feat{0,1}_rows, feat_step  every feat_step-th row of the oracle's FCGF features
  idx1                       the oracle's correspondences (int32 [N0])
  knn_safe, gap_safe         np.packbits of the rows whose float64 relative gap between the best and the
                             second-best squared distance exceeds gap_safe (rows with a smaller gap may
                             legitimately flip)
  logit                      float32 [N0] inlier logits of the oracle on ITS correspondences
  wsum, branch               the gate
  T_refined, refine_iters    pose after Procrustes + SE(3) refinement (before ICP)
  T_icp, icp_fitness, icp_rmse, icp_iters   the literal register() return value (use_icp=True)
  seconds                    CPU seconds per stage of this run (threads stated) - the same-config
                             CPU timing quoted in DESIGN.md
The oracle is test infrastructure; this script is the only producer of the fixture.
"""
import hashlib
import json
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from deepglobalregistration_b200 import synthetic as syn   # noqa: E402
from oracle import pipeline as op                           # noqa: E402
from oracle.registration import feature_knn, inlier_weights, se3_refine   # noqa: E402

FEAT_STEP = 16
GAP_SAFE = 2e-3        # relative top-2 gap above which a 5e-5 feature perturbation cannot flip the arg-min


def sha(a):
  return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def knn_gap64(F0, F1, chunk=2048):
  """float64 relative gap (d2_second - d2_best) / (d2_second + 1e-7) per F0 row."""
  A, B = F0.double(), F1.double()
  bn = (B * B).sum(1)
  out = []
  for s in range(0, len(A), chunk):
    a = A[s:s + chunk]
    d2 = ((a * a).sum(1, keepdim=True) + bn[None] - 2.0 * (a @ B.t())).clamp_min(0)
    top = torch.topk(d2, 2, dim=1, largest=False).values
    out.append((top[:, 1] - top[:, 0]) / (top[:, 1] + 1e-7))
  return torch.cat(out).float().numpy()


def case(config):
  if config == 2:
    state = syn.make_checkpoint(0)
    xyz0, xyz1, T_gt = syn.room_pair(0, n_raw=250_000)
  elif config == 3:
    state = syn.make_checkpoint(3, voxel_size=0.3, feat_conv1_kernel_size=5)
    xyz0, xyz1, T_gt = syn.lidar_pair(0)
  else:
    raise ValueError(config)
  return state, xyz0, xyz1, T_gt


def run(config):
  state, xyz0, xyz1, T_gt = case(config)
  cfg = state['config']
  vs = cfg['voxel_size']
  sec = {}

  def timed(name, fn):
    t = time.perf_counter()
    r = fn()
    sec[name] = time.perf_counter() - t
    print(f'  config {config}: {name} {sec[name]:.1f} s', flush=True)
    return r

  p0, c0, sel0 = timed('preprocess0', lambda: op.preprocess(xyz0, vs))
  p1, c1, sel1 = timed('preprocess1', lambda: op.preprocess(xyz1, vs))
  f0 = timed('fcgf0', lambda: op.fcgf(state, c0))
  f1 = timed('fcgf1', lambda: op.fcgf(state, c1))
  idx1 = timed('knn', lambda: feature_knn(f0, f1, cfg['nn_max_n']).numpy())
  gap = knn_gap64(f0, f1)
  c6 = op.inlier_coords(c0, c1, idx1)
  logit = timed('inlier_net', lambda: op.inlier_logits(
      state, c6, op.inlier_features(cfg['inlier_feature_type'], p0, p1, idx1)))
  w = inlier_weights(logit, 0.05)
  wsum = float(w.sum())
  branch = 'procrustes' if wsum >= max(200, len(w) * 0.05) else 'safeguard'
  out = dict(n0=len(c0), n1=len(c1), sha_sel0=sha(sel0.astype(np.int64)), sha_sel1=sha(sel1.astype(np.int64)),
             sha_coords0=sha(c0.astype(np.int32)), sha_coords1=sha(c1.astype(np.int32)),
             sha_coords6=sha(c6.astype(np.int32)), feat_step=FEAT_STEP,
             feat0_rows=f0[::FEAT_STEP].numpy(), feat1_rows=f1[::FEAT_STEP].numpy(),
             idx1=idx1.astype(np.int32), gap_safe=GAP_SAFE, knn_safe=np.packbits(gap > GAP_SAFE),
             logit=logit.reshape(-1).numpy().astype(np.float32),
             wsum=wsum, branch=branch, T_gt=T_gt)
  if branch == 'procrustes':
    R, t, info = timed('refine', lambda: se3_refine(p0, p1[idx1], w, 2 * vs))
    T = np.eye(4)
    T[:3, :3] = R.numpy()
    T[:3, 3] = t.numpy().reshape(3)
    out.update(T_refined=T, refine_iters=int(info['iterations']))
    from oracle.icp import icp_point_to_point
    T_icp, icp_info = timed('icp', lambda: icp_point_to_point(p0, p1, 2 * vs, T))
    out.update(T_icp=T_icp, icp_fitness=float(icp_info['fitness']), icp_rmse=float(icp_info['inlier_rmse']),
               icp_iters=int(icp_info['iterations']))
  sec['total_through_refine'] = sum(v for k, v in sec.items() if k != 'icp')
  out['seconds'] = json.dumps(dict(sec, threads=torch.get_num_threads()))
  path = os.path.join(HERE, f'fullsize_config{config}.npz')
  np.savez_compressed(path, **out)
  print(f'config {config}: N0={len(c0)} N1={len(c1)} wsum={wsum:.1f} branch={branch} '
        f'-> {path} ({os.path.getsize(path) / 1e6:.2f} MB); seconds {out["seconds"]}', flush=True)


if __name__ == '__main__':
  todo = [int(a) for a in sys.argv[1:]] or [3, 2]
  for c in todo:
    run(c)
