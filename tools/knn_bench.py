"""Feature-kNN timings: random unit vectors at three shapes, and the benchmark pair's own FCGF features
(syn.room_pair(0, 250k raw points) through the seeded checkpoint - tightly clustered, unlike random vectors).

--ab alternates the FP16 pre-filter with the TF32 one (DGR_KNN_TF32=1) in the same process."""
import argparse
import os
import sys
import types

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from deepglobalregistration_b200 import _abi
from deepglobalregistration_b200 import synthetic as syn


def time_ms(F0, F1, mode='tc', reps=5):
  for _ in range(2): idx = _abi.knn_top1(F0, F1, mode=mode)
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for _ in range(reps): idx = _abi.knn_top1(F0, F1, mode=mode)
  e1.record(); torch.cuda.synchronize()
  return e0.elapsed_time(e1) / reps, int(idx.long().sum())


def set_tf32(on):
  if on: os.environ['DGR_KNN_TF32'] = '1'
  else: os.environ.pop('DGR_KNN_TF32', None)


def bench_pair_features():
  from deepglobalregistration_b200.core.deep_global_registration import DeepGlobalRegistration
  dgr = DeepGlobalRegistration(types.SimpleNamespace(weights=syn.make_checkpoint(0), clip_weight_thresh=0.05,
                                                     verbose=False))
  xyz0, xyz1, _ = syn.room_pair(0, n_raw=250_000)
  with torch.no_grad():
    _, c0, _ = dgr.preprocess(xyz0, _slot=0)
    _, c1, _ = dgr.preprocess(xyz1, _slot=1)
    F0, F1 = dgr.fcgf_feature_extraction_pair(c0, c1)
  return F0.contiguous(), F1.contiguous()


def candidates_per_row(F0, F1):
  """Columns within the second sweep's bound of each row's minimum, counted on exact distances (the kernel
  compares estimates, so its count differs by the columns inside the estimate error)."""
  nb = float(F1.norm(dim=1).max())
  counts = []
  for s in range(0, F0.shape[0], 4096):
    a = F0[s:s + 4096]
    d2 = torch.cdist(a.double(), F1.double()).square()
    na = a.norm(dim=1).double()
    e = (2 ** -10 * 1.25 + 4e-5) * na * nb + 1e-6 * (na + nb) ** 2 + 1e-7
    counts.append((d2 <= d2.min(dim=1, keepdim=True).values + 4 * e[:, None]).sum(1))
  c = torch.cat(counts).double()
  return float(c.mean()), int(c.max())


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--ab', action='store_true', help='alternate FP16 and TF32 pre-filters')
  ap.add_argument('--rounds', type=int, default=3)
  args = ap.parse_args()
  torch.manual_seed(0)
  cases = []
  for n0, n1, c in ((51381, 39881, 32), (100000, 100000, 32), (50000, 50000, 64)):
    F0 = torch.nn.functional.normalize(torch.randn(n0, c, device='cuda'), dim=1)
    F1 = torch.nn.functional.normalize(torch.randn(n1, c, device='cuda'), dim=1)
    cases.append((f'random {n0}x{n1}x{c}', F0, F1))
  F0, F1 = bench_pair_features()
  cases.append((f'bench pair FCGF {F0.shape[0]}x{F1.shape[0]}x{F0.shape[1]}', F0, F1))
  mean, mx = candidates_per_row(F0, F1)
  print(f'bench pair FCGF: candidates per row under the bound (exact distances): mean {mean:.1f}, max {mx}')
  arms = (('fp16', False), ('tf32', True)) if args.ab else (('default', None),)
  for name, F0, F1 in cases:
    for r in range(args.rounds if args.ab else 1):
      for arm, tf32 in arms:
        if tf32 is not None: set_tf32(tf32)
        ms, chk = time_ms(F0, F1)
        print(f'{arm:7s} knn {name}: {ms:.3f} ms  {F0.shape[0]*F1.shape[0]*F0.shape[1]/ms/1e9:.2f} T pair-terms/s  '
              f'checksum {chk}', flush=True)
    set_tf32(False)
    ms, chk = time_ms(F0, F1, mode='simt', reps=2)
    print(f'simt    knn {name}: {ms:.3f} ms  checksum {chk}', flush=True)


if __name__ == '__main__':
  main()
