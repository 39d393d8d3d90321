"""CPU-side checks: the C-ABI library builds, loads and exports every symbol declared in
include/dgr_b200.h (no compute calls without a GPU); the ME-shaped host API has the
surface the reference touches; product code fails loudly without CUDA."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def built():
  from deepglobalregistration_b200 import build
  return build.build()


def test_library_exports_every_declared_symbol(built):
  header = open(os.path.join(ROOT, 'include', 'dgr_b200.h')).read()
  declared = set(re.findall(r'\b(dgr_[a-z0-9_]+)\s*\(', header))
  declared -= {'dgr_keyspec_t'}
  assert len(declared) >= 25
  lib = ctypes.CDLL(built)
  missing = [s for s in sorted(declared) if not hasattr(lib, s)]
  assert not missing, missing
  from deepglobalregistration_b200 import _abi
  assert set(_abi.SIGNATURES) == declared, set(_abi.SIGNATURES) ^ declared
  assert _abi.lib().dgr_version() == 100
  assert ctypes.sizeof(_abi.KeySpec) == 4 * (2 + 3 * 8)


def test_sm100a_sass_present(built):
  out = os.popen(f'cuobjdump -lelf {built} 2>/dev/null').read()
  assert 'sm_100a' in out


def test_no_cpu_fallback():
  from deepglobalregistration_b200 import _abi
  with pytest.raises(_abi.DgrError):
    _abi.require_device('cpu')
  if not torch.cuda.is_available():
    from deepglobalregistration_b200 import me as ME
    with pytest.raises(Exception):
      ME.SparseTensor(torch.ones(2, 1), coordinates=torch.zeros(2, 4, dtype=torch.int32))


def test_product_never_imports_oracle():
  pkg = os.path.join(ROOT, 'deepglobalregistration_b200')
  for dp, _, files in os.walk(pkg):
    for f in files:
      if f.endswith('.py'):
        src = open(os.path.join(dp, f)).read()
        assert not re.search(r'^\s*(from|import)\s+oracle\b', src, re.M), os.path.join(dp, f)


def test_me_surface_and_state_dict_layout():
  from deepglobalregistration_b200 import shims, synthetic as syn
  ME = shims.install()
  import MinkowskiEngine
  import MinkowskiEngine.MinkowskiFunctional as MEF
  assert MinkowskiEngine is ME and callable(MEF.relu)
  for name in ('SparseTensor', 'MinkowskiNetwork', 'MinkowskiConvolution', 'MinkowskiConvolutionTranspose',
               'KernelGenerator', 'RegionType', 'MinkowskiBatchNorm', 'cat', 'MinkowskiSumPooling',
               'MinkowskiPoolingTranspose', 'MinkowskiInstanceNorm', 'MinkowskiReLU', 'MinkowskiELU'):
    assert hasattr(ME, name), name
  assert callable(ME.utils.sparse_quantize) and callable(ME.utils.batched_coordinates)
  conv = ME.MinkowskiConvolution(3, 8, kernel_size=3, stride=2, has_bias=True, dimension=3)   # 0.4 spelling
  assert conv.kernel.shape == (27, 3, 8) and conv.bias.shape == (1, 8)
  assert ME.MinkowskiConvolution(3, 8, kernel_size=1, dimension=6).kernel.shape == (3, 8)
  assert ME.MinkowskiConvolutionTranspose(4, 2, kernel_size=3, stride=2, dimension=6).kernel.shape == (729, 4, 2)
  bn = ME.MinkowskiBatchNorm(8, momentum=0.05)
  assert set(bn.state_dict()) == {'bn.weight', 'bn.bias', 'bn.running_mean', 'bn.running_var',
                                  'bn.num_batches_tracked'}
  with pytest.raises(NotImplementedError):
    ME.MinkowskiInstanceNorm(8)
  bc = ME.utils.batched_coordinates([torch.zeros(3, 3).int(), torch.ones(2, 3).int()])
  assert bc.shape == (5, 4) and bc[:, 0].tolist() == [0, 0, 0, 1, 1] and bc.dtype == torch.int32
  from deepglobalregistration_b200.model import load_model
  assert load_model('NoSuchNet') is None
  for D, cin, cout, k in ((3, 1, 32, 7), (6, 1, 1, 3)):
    m = load_model('ResUNetBN2C')(cin, cout, conv1_kernel_size=k, D=D)
    sd = syn.resunet_state_dict(0, cin, cout, k, D) if D == 3 else None
    if sd is not None:
      assert m.load_state_dict(sd).missing_keys == []
    n_par = sum(p.numel() for p in m.parameters())
    assert n_par == (8_760_384 if D == 3 else 235_926_689), n_par


def test_kernel_offsets_match_oracle():
  from deepglobalregistration_b200.me.coords import kernel_offsets
  from oracle import sparse_ops as so
  for k, D, s in ((3, 3, 1), (7, 3, 1), (5, 3, 2), (3, 6, 4)):
    assert np.array_equal(kernel_offsets(k, D, s, 'cpu').numpy(), so.kernel_offsets(k, D, s))


def test_reference_model_files_import_against_the_shim():
  """The reference's own ResUNetBN2C (model/resunet.py, state-dict layout stored in tests/golden/reference_model.npz
  by tests/golden/make_golden_reference.py, built over oracle/me_cpu.py) has the same parameters as ours, so both
  accept the same checkpoint.  The reference's files are not part of this repository: nothing is imported over the
  shim here any more; the name is kept so that the check keeps its history."""
  import json

  from deepglobalregistration_b200 import synthetic as syn
  ref = json.loads(str(np.load(os.path.join(ROOT, 'tests', 'golden', 'reference_model.npz'))['state_dict_shapes']))
  from deepglobalregistration_b200.model import load_model
  ours = load_model('ResUNetBN2C')(1, 32, bn_momentum=0.05, conv1_kernel_size=7, normalize_feature=True)
  assert {k: list(v.shape) for k, v in ours.state_dict().items()} == ref
  sd = syn.resunet_state_dict(0, 1, 32, 7, 3)
  assert {k: list(v.shape) for k, v in sd.items()} == ref
  ours.load_state_dict(sd)


def test_native_layer_table_parameter_order():
  """native.network_parameters lists the 66 tensors dgr_net_create documents, in execution order, for this
  package's ResUNetBN2C (whose parameter names and shapes are the reference's: see
  test_reference_model_files_import_against_the_shim)."""
  from deepglobalregistration_b200 import native, synthetic as syn
  from deepglobalregistration_b200.model import load_model
  models = [load_model('ResUNetBN2C')(1, 32, bn_momentum=0.05, conv1_kernel_size=7, normalize_feature=True, D=3)]
  C, T = [None, 32, 64, 128, 256], [None, 64, 64, 64, 128]
  for m in models:
    m.load_state_dict(syn.resunet_state_dict(0, 1, 32, 7, 3))
    m.eval()
    ps = native.network_parameters(m)
    assert len(ps) == 66 and all(p.dtype == torch.float32 and p.is_contiguous() for p in ps)
    assert tuple(ps[0].shape) == (343, 1, 32) and tuple(ps[1].shape) == (32,) and tuple(ps[2].shape) == (32,)
    assert tuple(ps[3].shape) == (27, 32, 32)                       # block1.conv1
    assert tuple(ps[9].shape) == (27, C[1], C[2])                   # conv2 (stride 2)
    assert tuple(ps[36].shape) == (27, C[4], T[4])                  # conv4_tr
    assert tuple(ps[45].shape) == (27, C[3] + T[4], T[3])           # conv3_tr reads cat(decoder, skip)
    assert tuple(ps[63].shape) == (C[1] + T[2], T[1]) and tuple(ps[64].shape) == (T[1], 32) and tuple(ps[65].shape) == (32,)
    # folded BatchNorm: scale = weight / sqrt(var + eps)
    bn = m.norm1.bn
    assert torch.allclose(ps[1], bn.weight / torch.sqrt(bn.running_var + bn.eps))
