"""The oracle's ResUNetBN2C restatement (oracle/resunet.py) against the reference's OWN model code:
model/resunet.py + model/residual_block.py + model/common.py run unmodified on the CPU over oracle/me_cpu.py
(a MinkowskiEngine-shaped module backed by oracle/sparse_ops.py), stored in tests/golden/reference_model.npz
by tests/golden/make_golden_reference.py.  Same sparse operators on both sides, so this isolates - and pins -
the GRAPH: layer order, strides, transposed-convolution pairing, skip concatenation order, norm placement,
final bias and normalisation."""
import os

import numpy as np
import pytest
import torch

from deepglobalregistration_b200 import synthetic as syn
from oracle.resunet import resunet_forward

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_model.npz')


def _cloud(seed, n, D, extent):
  g = np.random.default_rng(seed)
  c = np.unique(g.integers(-extent, extent, size=(n, D)), axis=0)
  return np.concatenate([np.zeros((len(c), 1), np.int64), c], 1).astype(np.int32)


@pytest.mark.parametrize('case,D,cin,cout,k1,normalize,n,extent', [
    (0, 3, 1, 32, 7, True, 600, 7),        # FCGF, 3DMatch setting (scripts/train_3dmatch.sh:19)
    (1, 3, 1, 32, 5, True, 500, 9),        # FCGF, KITTI setting
    (2, 6, 1, 1, 3, False, 300, 2),        # inlier network, 'ones' features
    (3, 6, 6, 1, 3, False, 250, 2),        # inlier network, 'coords' features
], ids=['3-1-32-7-True-600-7', '3-1-32-5-True-500-9', '6-1-1-3-False-300-2', '6-6-1-3-False-250-2'])
def test_reference_graph_equals_oracle_restatement(case, D, cin, cout, k1, normalize, n, extent):
  gold = np.load(GOLD)
  sd = syn.resunet_state_dict(D + k1, cin, cout, k1, D)
  g = torch.Generator().manual_seed(1)
  for k in sd:                                  # non-trivial BN statistics so a misplaced norm shows
    if k.endswith('running_mean'):
      sd[k] = 0.1 * torch.randn(sd[k].shape, generator=g)
    if k.endswith('bn.bias'):
      sd[k] = 0.1 * torch.randn(sd[k].shape, generator=g)
  coords = _cloud(D, n, D, extent)
  feats = torch.ones(len(coords), cin) if cin == 1 else torch.randn(len(coords), cin, generator=g)
  want = resunet_forward(sd, coords, feats, k1, normalize)
  assert want.shape == (len(coords), cout)
  rows = gold[f'graph{case}_rows']
  got = gold[f'graph{case}_out']                # the reference's output at these rows
  assert rows.max() < len(coords) and got.shape == (len(rows), cout)
  want = want.numpy()[rows]
  err = float(np.abs(got - want).max() / (1 + np.abs(want).max()))
  assert err <= 1e-6, err
  assert float(np.abs(want).max()) > 1e-4           # the comparison is not vacuous
