"""The FP16 tensor-core kNN pre-filter returns exactly what the fp32 brute-force kernel returns (indices and
distances) on inputs that stress its error bound: per-row magnitudes over twelve decades, entries that become
FP16 subnormals after scaling, zero rows, ties, ragged tile edges, many work items per SM, C = 64, and the
benchmark pair's own FCGF features."""
import types

import pytest
import torch

from deepglobalregistration_b200 import synthetic as syn

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def abi():
  from deepglobalregistration_b200 import _abi
  _abi.require_device('cuda')
  return _abi


def _check(abi, F0, F1):
  F0, F1 = F0.cuda().contiguous(), F1.cuda().contiguous()
  i_tc, d_tc = abi.knn_top1(F0, F1, return_distance=True, mode='tc')
  i_ref, d_ref = abi.knn_top1(F0, F1, return_distance=True, mode='simt')
  assert torch.equal(i_tc, i_ref), f'{int((i_tc != i_ref).sum())} rows differ'
  assert torch.equal(d_tc, d_ref)
  return i_tc.cpu()


def _clustered(g, n0, n1, c, n_centres, jitter):
  centres = torch.nn.functional.normalize(torch.randn(n_centres, c, generator=g), dim=1)
  F0 = centres[torch.randint(0, n_centres, (n0,), generator=g)] + jitter * torch.randn(n0, c, generator=g)
  F1 = centres[torch.randint(0, n_centres, (n1,), generator=g)] + jitter * torch.randn(n1, c, generator=g)
  return F0, F1


@pytest.mark.parametrize('c', [32, 64])
def test_row_magnitudes_over_twelve_decades(abi, c):
  g = torch.Generator().manual_seed(1)
  n0, n1 = 3001, 2003
  F0 = torch.randn(n0, c, generator=g) * 10 ** (torch.rand(n0, 1, generator=g) * 12 - 8)
  F1 = torch.randn(n1, c, generator=g) * 10 ** (torch.rand(n1, 1, generator=g) * 12 - 8)
  _check(abi, F0, F1)


def test_fp16_subnormal_entries(abi):
  """One entry of each row near 1, the others 2^-30 .. 2^-40 of it: after the power-of-two scale they fall into
  (or below) the FP16 subnormal range, which only the bound's absolute term covers."""
  g = torch.Generator().manual_seed(2)
  n0, n1, c = 2000, 3000, 32
  F0 = torch.randn(n0, c, generator=g) * 2.0 ** -torch.randint(30, 41, (n0, c), generator=g).float()
  F1 = torch.randn(n1, c, generator=g) * 2.0 ** -torch.randint(30, 41, (n1, c), generator=g).float()
  F0[:, 0] += 1.0
  F1[:, 0] += 1.0
  F1[:, 5] += 2.0 ** -28 * torch.randint(0, 3, (n1,), generator=g).float()
  _check(abi, F0, F1)


def test_zero_rows_duplicates_and_exact_matches(abi):
  g = torch.Generator().manual_seed(3)
  n0, n1, c = 1000, 1500, 32
  F0, F1 = _clustered(g, n0, n1, c, 20, 1e-3)
  F0[:50] = 0.0
  F1[100:110] = 0.0                       # zero columns: a zero row's nearest is column 100
  F1[700] = F1[300]
  F1[1400] = F1[300]
  F0[60:70] = F1[300]                     # exact match, two later duplicates: lowest index wins
  F0[70:80] = F1[1200:1210]
  idx = _check(abi, F0, F1)
  assert torch.equal(idx[:50], torch.full((50,), 100, dtype=torch.int32))
  assert torch.equal(idx[60:70], torch.full((10,), 300, dtype=torch.int32))
  assert torch.equal(idx[70:80], torch.arange(1200, 1210, dtype=torch.int32))


@pytest.mark.parametrize('n1', [1, 255, 257])
def test_ragged_column_counts(abi, n1):
  g = torch.Generator().manual_seed(n1)
  F0, F1 = _clustered(g, 700, n1, 32, 8, 1e-2)
  _check(abi, F0, F1)


def test_many_work_items_per_sm(abi):
  """n0 not a multiple of the row tile, and far more (row tile, column tile) items than SMs."""
  g = torch.Generator().manual_seed(4)
  F0, F1 = _clustered(g, 40_077, 3_001, 32, 50, 1e-3)
  _check(abi, F0, F1)


def test_c64_clustered(abi):
  g = torch.Generator().manual_seed(5)
  F0, F1 = _clustered(g, 10_001, 9_003, 64, 30, 1e-3)
  _check(abi, F0, F1)


def test_clustered_bench_shape(abi):
  """51k x 40k x 32, few tight clusters: hundreds of candidates per row in the second sweep."""
  g = torch.Generator().manual_seed(6)
  F0, F1 = _clustered(g, 51_381, 39_881, 32, 40, 1e-3)
  F0 = torch.nn.functional.normalize(F0, dim=1)
  F1 = torch.nn.functional.normalize(F1, dim=1)
  _check(abi, F0, F1)


def test_bench_pair_fcgf_features(abi):
  """The benchmark's first pair (syn.room_pair(0), 250k raw points per cloud) through the seeded checkpoint's
  FCGF network: the features the benchmark's kNN stage sees."""
  from deepglobalregistration_b200.core.deep_global_registration import DeepGlobalRegistration
  dgr = DeepGlobalRegistration(types.SimpleNamespace(weights=syn.make_checkpoint(0), clip_weight_thresh=0.05,
                                                     verbose=False))
  xyz0, xyz1, _ = syn.room_pair(0, n_raw=250_000)
  with torch.no_grad():
    _, coords0, _ = dgr.preprocess(xyz0, _slot=0)
    _, coords1, _ = dgr.preprocess(xyz1, _slot=1)
    F0, F1 = dgr.fcgf_feature_extraction_pair(coords0, coords1)
  assert F0.shape[0] > 40_000 and F1.shape[0] > 30_000 and F0.shape[1] == 32
  _check(abi, F0, F1)
