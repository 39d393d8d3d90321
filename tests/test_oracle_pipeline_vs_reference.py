"""oracle/pipeline.py::register against the reference's OWN DeepGlobalRegistration.register():
core/deep_global_registration.py, core/knn.py, core/registration.py, model/*.py, util/*.py run
unmodified end to end on the CPU, with
* MinkowskiEngine  -> oracle/me_cpu.py (sparse operators of oracle/sparse_ops.py),
* open3d           -> the I/O stand-in of shims.py + registration_icp backed by oracle/icp.py,
and what they returned is stored in tests/golden/reference_register.npz (tests/golden/make_golden_reference.py).
The sparse operators and ICP are therefore the oracle's on both sides; what this pins is everything
else the oracle restates by hand: the order of the stages, dtypes, voxelisation and re-flooring, the
6-D coordinate assembly, feature types, the sigmoid / clip / weight-sum gate and its thresholds, the
arguments handed to GlobalRegistration and to ICP."""
import hashlib
import json
import os

import numpy as np
import pytest

from deepglobalregistration_b200 import synthetic as syn
from oracle import pipeline as op

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_register.npz')


def sha(a):
  return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope='module')
def gold():
  return np.load(GOLD)


@pytest.mark.parametrize('feature_type,dtype', [('ones', np.float64), ('coords', np.float32)])
def test_reference_register_equals_oracle_pipeline(gold, feature_type, dtype):
  ref = {k[len(f'reg_{feature_type}_'):]: gold[k] for k in gold.files if k.startswith(f'reg_{feature_type}_')}
  state = syn.make_checkpoint(1, inlier_feature_type=feature_type)
  xyz0, xyz1, _ = syn.room_pair(7, n_raw=5000, extent=(1.2, 1.0, 0.8))
  xyz0, xyz1 = xyz0.astype(dtype), xyz1.astype(dtype)
  # the reference instance: default use_icp = True, voxel size from the checkpoint
  assert bool(ref['use_icp']) is True and float(ref['voxel_size']) == state['config']['voxel_size']
  vs = float(ref['voxel_size'])
  T_o, taps = op.register(state, xyz0, xyz1, clip_weight_thresh=0.05, use_icp=True)
  assert taps['branch'] == 'procrustes'
  assert f"=> Weighted sum {taps['wsum']:.2f} >=" in str(ref['printed'])       # same gate value, same branch
  # what the reference handed to open3d's ICP
  assert float(ref['icp_max_dist']) == 2 * vs and int(ref['icp_n_source']) == len(taps['coords0']) \
      and int(ref['icp_n_target']) == len(taps['coords1'])
  te, re = syn.rte_rre(ref['icp_init'], taps['T_refined'])                   # tap A: before ICP
  assert te <= 1e-3 and re <= 1e-3, (te, re, taps['refine'])
  te, re = syn.rte_rre(ref['T'], T_o)                                        # tap B: the literal return value
  assert te <= 1e-3 and re <= 1e-3, (te, re, taps['icp'])
  # stage taps of the reference's own methods: preprocess(xyz0) and fcgf_feature_extraction
  assert str(ref['p0_dtype']) == 'torch.float32' and str(ref['c0_dtype']) == 'torch.int32'
  assert sha(taps['coords0'].astype(np.int32)) == str(ref['sha_c0'])
  assert sha(taps['xyz0'].astype(np.float32)) == str(ref['sha_p0'])
  assert tuple(ref['f0_shape']) == (len(taps['coords0']), 1)
  rows = ref['F0_rows']
  assert float(np.abs(ref['F0'] - taps['feat0'].numpy()[rows]).max()) <= 1e-6


def test_public_surface_matches_the_reference_class(gold):
  """Same public methods with the same parameter names (and defaults where the reference has them) on
  deepglobalregistration_b200's DeepGlobalRegistration - the drop-in boundary of SURVEY.md 8(b)."""
  import inspect

  from deepglobalregistration_b200.core.deep_global_registration import DeepGlobalRegistration as Ours
  ref_methods = json.loads(str(gold['surface']))
  assert set(ref_methods) == {'__init__', 'preprocess', 'fcgf_feature_extraction', 'fcgf_feature_matching',
                              'inlier_feature_generation', 'inlier_prediction', 'safeguard_registration', 'register'}
  for name, want in ref_methods.items():
    ours = getattr(Ours, name, None)
    assert ours is not None, f'missing method {name}'
    got = inspect.signature(ours).parameters
    public = [p for p in got if not p.startswith('_')]          # ours may add private keyword-only helpers
    assert public == [p for p, _, _ in want], (name, public, want)
    for p, has_default, default in want:
      if has_default and name != '__init__':
        assert repr(got[p].default) == default, (name, p)
  assert str(inspect.signature(Ours.__init__).parameters['device'].default) == 'cuda'
