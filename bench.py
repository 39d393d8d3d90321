#!/usr/bin/env python
"""bench.py - scan-pairs/sec of DGR's pairwise-registration hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \\
        --master-port P bench.py --gpus N --steps K --warmup W

One "step" = one full register() of one synthetic 3DMatch-shape scan pair (BASELINE.json
configs[1]/[3] shape: ~50k voxels per cloud at 0.05 m, FCGF feature dim 32, ResUNetBN2C for
both networks): voxelise x2 -> FCGF x2 -> feature kNN -> 6-D inlier network -> weights ->
weighted Procrustes + SE(3) refinement (SURVEY 8(d)'s unit).  The ICP fine-tune and the RANSAC
safeguard are built but outside the benchmarked unit on both arms.  Pairs are independent: each rank registers its own pairs (weak scaling) and
the poses are all-gathered over NCCL at the end of the timed region.

Prints ONE JSON line (rank 0).  `value` = pairs/s with the raw scans resident in HBM;
`e2e` = pairs/s through DeepGlobalRegistration.register(host ndarrays) including the H2D
copy of both scans and the D2H read of the pose.  `--impl reference` times the CPU oracle
port of the same path (MinkowskiEngine cannot be installed offline) on a bounded sample.
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time
import types

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)

import numpy as np
import torch

from deepglobalregistration_b200 import synthetic as syn

WORKLOAD = '3dmatch_shape_pair_register'
N_RAW = 250_000               # raw points per scan -> ~50k voxels at 0.05 m
SAMPLE_N_RAW = 8_000          # CPU sample: same generator, ~4k voxels per cloud
SAMPLE_EXTENT = (1.5, 1.2, 1.0)
REF_MIN_N_RAW = 1500          # the reference arm's untimed warm-up sample
VOXEL = 0.05
POOL = 3                      # distinct pairs per rank, cycled over the steps
INFLIGHT = int(os.environ.get('DGR_BENCH_INFLIGHT', '4'))   # pairs in flight per GPU (SURVEY 8e: pipeline pairs per GPU)


_emit = print


def log(*a):
  print(*a, file=sys.stderr, flush=True)


def base_config(n_gpus):
  """The SAME dict on both arms (the driver compares them): anything that differs between the arms
  (voxel counts seen, sample notes) goes into other keys of the line."""
  return {'workload': WORKLOAD, 'n_raw_points_per_scan': N_RAW, 'voxel_size': VOXEL, 'feat_dim': 32,
          'fcgf_model': 'ResUNetBN2C(D=3,conv1_k=7)', 'inlier_model': 'ResUNetBN2C(D=6,conv1_k=3)',
          'conv_arithmetic': 'tcgen05 split products, fp32 accumulate: 3xFP16 hi/lo on the wide layers, 3xTF32 elsewhere (both fp32-accurate: features within 5e-5 of the fp32 oracle at full size); fp32 adds for conv1',
          'parallelism': f'pair-sharded dp{n_gpus}', 'pairs_per_step_per_gpu': 1,
          'excluded_on_both_arms': 'ICP fine-tune and RANSAC safeguard (both built; the benchmarked unit is SURVEY 8(d)\'s: through the SE(3) refinement, and the benchmark pairs take the Procrustes branch)',
          'l2_policy': 'inputs larger than L2: every step streams the 944 MB inlier-net weights '
                       '(L2 = 126 MB) and cycles through %d distinct pairs (the same ones on every rank)' % POOL}


# ------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------
class ClockSampler:
  """SM clock and throttle reasons during the timed region.  Uses NVML in-process (a query costs
  microseconds); spawning nvidia-smi in a loop was measured to stall the CUDA driver for ~200 ms
  per query on these hosts and is only the fallback."""
  Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
       'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
       'clocks_event_reasons.sw_power_cap')

  def __init__(self, index, period=0.1):
    self.rows, self.proc, self.nvml, self.stop_flag = [], None, None, False
    self.period = period
    try:
      import pynvml
      pynvml.nvmlInit()
      self.nvml = pynvml
      # torch's device index follows CUDA_VISIBLE_DEVICES; map through the UUID-free common case
      vis = os.environ.get('CUDA_VISIBLE_DEVICES')
      phys = int(vis.split(',')[index]) if vis and vis.split(',')[index].isdigit() else index
      self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
      self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
      self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
      self.thread.start()
      return
    except Exception as e:   # noqa: BLE001
      log('NVML sampler unavailable (%s); falling back to nvidia-smi' % e)
      self.nvml = None
    try:
      self.proc = subprocess.Popen(['nvidia-smi', '-i', str(index), f'--query-gpu={self.Q}',
                                    '--format=csv,noheader,nounits', '-lms', '500'],
                                   stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      self.thread = threading.Thread(target=self._read, daemon=True)
      self.thread.start()
    except Exception as e:   # noqa: BLE001
      log('clock sampler unavailable:', e)

  def _poll_nvml(self):
    n = self.nvml
    names = {'hw_slowdown': getattr(n, 'nvmlClocksEventReasonHwSlowdown', 0x8),
             'hw_thermal_slowdown': getattr(n, 'nvmlClocksEventReasonHwThermalSlowdown', 0x40),
             'sw_thermal_slowdown': getattr(n, 'nvmlClocksEventReasonSwThermalSlowdown', 0x20),
             'sw_power_cap': getattr(n, 'nvmlClocksEventReasonSwPowerCap', 0x4)}
    get_reasons = getattr(n, 'nvmlDeviceGetCurrentClocksEventReasons',
                          getattr(n, 'nvmlDeviceGetCurrentClocksThrottleReasons', None))
    while not self.stop_flag:
      try:
        sm = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
        mask = int(get_reasons(self.handle)) if get_reasons else 0
        active = [k for k, bit in names.items() if mask & bit]
        self.rows.append((time.time(), sm, active))
      except Exception:   # noqa: BLE001
        pass
      time.sleep(self.period)

  def _read(self):
    names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
    for line in self.proc.stdout:
      f = [x.strip() for x in line.split(',')]
      try:
        self.max_sm = float(f[1])
        self.rows.append((time.time(), float(f[0]),
                          [nm for nm, v in zip(names, f[3:7]) if v.lower().startswith('active')]))
      except (ValueError, IndexError):
        continue

  def stop(self, t0, t1):
    self.stop_flag = True
    if self.proc is not None:
      self.proc.terminate()
    if self.proc is None and self.nvml is None:
      return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable']}
    sm, reasons = [], set()
    for ts, clk, active in self.rows:
      if t0 - 0.05 <= ts <= t1 + 0.15:
        sm.append(clk)
        reasons.update(active)
    return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': getattr(self, 'max_sm', None),
            'samples': len(sm), 'reasons': sorted(reasons),
            'source': 'nvml' if self.nvml is not None else 'nvidia-smi'}


# ------------------------------------------------------------------------------------------
# CPU baseline (oracle port) - also the --impl reference arm
# ------------------------------------------------------------------------------------------
def cgroup_throttled_ms():
  """Cumulative time this container's CPU cgroup has been throttled (ms), or None."""
  for path in ('/sys/fs/cgroup/cpu.stat', '/sys/fs/cgroup/cpu/cpu.stat'):
    try:
      for line in open(path):
        k, v = line.split()
        if k == 'throttled_usec':
          return int(v) / 1e3
        if k == 'throttled_time':
          return int(v) / 1e6
    except Exception:   # noqa: BLE001
      continue
  return None


def effective_cpus():
  """Host threads this process may really use: affinity mask and cgroup CPU quota, not nproc."""
  n = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
  try:
    quota, period = open('/sys/fs/cgroup/cpu.max').read().split()
    if quota != 'max':
      n = min(n, max(1, int(np.ceil(int(quota) / int(period)))))
  except Exception:   # noqa: BLE001
    try:
      q = int(open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us').read())
      p = int(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
      if q > 0:
        n = min(n, max(1, int(np.ceil(q / p))))
    except Exception:   # noqa: BLE001
      pass
  return n


def pin_rank_to_numa_node(local_rank):
  """Keep this rank's host threads on the CPU cores local to its GPU (the box has two sockets: GPUs 0-3 hang
  off one, 4-7 off the other); a rank whose launch threads sit on the far socket pays a cross-socket hop on
  every launch and host read.  Best effort: silently does nothing when the topology cannot be read."""
  try:
    p = torch.cuda.get_device_properties(local_rank)
    path = f'/sys/bus/pci/devices/{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0/local_cpulist'
    cpus = set()
    for part in open(path).read().strip().split(','):
      lo, _, hi = part.partition('-')
      cpus.update(range(int(lo), int(hi or lo) + 1))
    cpus &= os.sched_getaffinity(0)
    if cpus:
      os.sched_setaffinity(0, cpus)
      log(f'[bench] local rank {local_rank}: pinned to {len(cpus)} cores local to the GPU ({min(cpus)}-{max(cpus)})')
  except Exception as e:   # noqa: BLE001
    log(f'[bench] NUMA pinning skipped: {e!r}')


CPU_THREADS = None


def cpu_threads():
  """Threads for the CPU arm: all usable cores, capped at 32 (the per-offset mm / index_add
  of the oracle stop scaling well before that and oversubscription is catastrophic)."""
  global CPU_THREADS
  if CPU_THREADS is None:
    CPU_THREADS = max(1, min(effective_cpus(), 32))
    torch.set_num_threads(CPU_THREADS)
  return CPU_THREADS


def cpu_sample_time(state, seed, reps=1, n_raw=SAMPLE_N_RAW):
  """Seconds per pair of the CPU oracle on the bounded sample."""
  from oracle import pipeline as op
  cpu_threads()
  xyz0, xyz1, _ = syn.room_pair(seed, n_raw=n_raw, extent=SAMPLE_EXTENT)
  ts, info = [], {}
  for _ in range(reps):
    t = time.perf_counter()
    _, taps = op.register(state, xyz0, xyz1)
    ts.append(time.perf_counter() - t)
    info = {'n0': int(len(taps['coords0'])), 'n1': int(len(taps['coords1'])), 'branch': taps['branch']}
  return float(np.median(ts)), info


def sample_desc(info, n_raw=SAMPLE_N_RAW):
  return (f'1 pair of the same generator at {n_raw} raw points/scan -> N0={info["n0"]}, '
          f'N1={info["n1"]} voxels (the workload has ~51k/~40k); pairs/s of the SAMPLE, not extrapolated; '
          'CPU path = oracle port (torch-CPU index_select/mm/index_add per kernel offset, the algorithm '
          "of MinkowskiEngine's CPU backend) + restated kNN / Procrustes / Adam refinement")


def fixture_parity(T, key='T_refined'):
  """TE [m] / RE [rad] of a pose of the bench's first pair (rank 0, seed 0, 250k raw points) against the CPU
  oracle's pose stored in tests/golden/fullsize_config2.npz (tests/golden/make_golden_fullsize.py)."""
  try:
    g = np.load(os.path.join(ROOT, 'tests', 'golden', 'fullsize_config2.npz'))
    te, re = syn.rte_rre(np.asarray(T, np.float64).reshape(4, 4), g[key])
    return {'te_m': te, 're_rad': re, 'tolerance': '1e-3 m / 1e-3 rad (north_star)', 'within_tolerance': bool(te <= 1e-3 and re <= 1e-3),
            'against': 'CPU oracle pose before ICP of the same pair (BASELINE config 2: syn.room_pair(0, 250k raw points), '
                       f'N0={int(g["n0"])}, N1={int(g["n1"])} voxels), fixture tests/golden/fullsize_config2.npz',
            'config': WORKLOAD}
  except Exception as e:   # noqa: BLE001
    return {'te_m': None, 're_rad': None, 'error': repr(e)}


def stage_isolated_parity(dgr, pair_dev):
  """The last stage at the bench's size on the ORACLE's inputs: register the pair once more, take the voxelised
  points from the executor, and run Procrustes + refinement on the oracle's correspondences and weights (fixture).
  End-to-end poses of a random-init network are ill-conditioned (its correspondences are unrelated points; a
  handful of arg-min flips inside the features' rounding noise move the optimum by centimetres), so this is the
  number that isolates the arithmetic; the earlier stages are pinned the same way in
  tests/test_gpu_zzzz_golden_fullsize.py."""
  try:
    from deepglobalregistration_b200 import _abi
    g = np.load(os.path.join(ROOT, 'tests', 'golden', 'fullsize_config2.npz'))
    dgr.register(*pair_dev)
    ctx = dgr._last_ctx
    n0 = dgr.last_info['n0']
    if n0 != int(g['n0']) or dgr.last_info['n1'] != int(g['n1']):
      return {'error': f'voxel counts differ from the fixture: {n0}, {dgr.last_info["n1"]}'}
    xyz = ctx.tap('xyz')
    idx_gpu = ctx.tap('idx1').cpu().numpy()
    flips = int((idx_gpu != g['idx1']).sum())
    _abi.refresh_stream()
    dev = xyz.device
    w, _ = _abi.sigmoid_clip_sum(torch.from_numpy(g['logit']).to(dev).contiguous(), 0.05)
    res = _abi.se3_register(xyz[:n0].contiguous(), xyz[n0:].contiguous(), w.reshape(-1).contiguous(),
                            idx1=torch.from_numpy(g['idx1']).to(dev).int().contiguous(),
                            quantization_size=2 * dgr.voxel_size, break_threshold_ratio=1e-4).cpu().numpy()
    T = np.eye(4)
    T[:3, :3], T[:3, 3] = res[:9].reshape(3, 3), res[9:12]
    te, re = syn.rte_rre(T, g['T_refined'])
    return {'te_m': te, 're_rad': re, 'within_tolerance': bool(te <= 1e-3 and re <= 1e-3),
            'correspondences_differing_from_oracle_end_to_end': flips, 'correspondences': int(n0)}
  except Exception as e:   # noqa: BLE001
    return {'error': repr(e)}


def dump_outputs(dirname, last, last_e2e=None):
  """What the last timed step returned, as float64 .npy files: the 4x4 pose register() hands its caller and the
  inlier weight sum behind the branch choice.  `last_e2e` is the last step of the host-buffer (`e2e`) loop."""
  os.makedirs(dirname, exist_ok=True)
  out = {'pose': last[0], 'weight_sum': [last[2].get('wsum', np.nan)]}
  if last_e2e is not None:
    out.update(pose_e2e=last_e2e[0], weight_sum_e2e=[last_e2e[2].get('wsum', np.nan)])
  for name, a in out.items():
    np.save(os.path.join(dirname, name + '.npy'), np.asarray(a, np.float64))
  log(f'[bench] outputs of the last timed step: {", ".join(sorted(out))} -> {dirname}')


def run_reference(args):
  """The reference's CPU implementation of the path (the oracle port: MinkowskiEngine is not installable
  offline, nothing of the reference compiles into oracle/_ref) on the SAME configuration as the B200 arm:
  full-size pairs of the same generator and seeds.  One such pair is minutes of CPU, so the arm's default is
  one step; it registers exactly K pairs (cpu_baseline.steps_executed) and nothing is extrapolated."""
  rank = int(os.environ.get('RANK', '0'))
  if rank != 0:
    return
  from oracle import pipeline as op
  state = syn.make_checkpoint(0)
  cores = cpu_threads()
  log(f'[bench] reference arm: {cores} threads (nproc {os.cpu_count()}, usable {effective_cpus()})')
  # warm-up: thread pools / allocator on a tiny sample of the same generator (seconds), untimed
  t_warm, _ = cpu_sample_time(state, 100, n_raw=REF_MIN_N_RAW)
  log(f'[bench] reference arm: warm-up sample {t_warm:.1f} s; timing full-size pairs')
  times, info, parity = [], {}, None
  for i in range(args.steps):
    xyz0, xyz1, _ = syn.room_pair(1000 * rank + (i % POOL), n_raw=N_RAW)
    t = time.perf_counter()
    T, taps = op.register(state, xyz0, xyz1)
    times.append(time.perf_counter() - t)
    info = {'n0': int(len(taps['coords0'])), 'n1': int(len(taps['coords1'])), 'branch': taps['branch']}
    if i == 0:
      parity = fixture_parity(T)
    log(f'[bench] reference arm: pair {i} N0={info["n0"]} N1={info["n1"]} {times[-1]:.1f} s')
  if args.dump_outputs:
    dump_outputs(args.dump_outputs, (T, taps['branch'], {'wsum': taps['wsum']}))
  n_exec = len(times)
  dt = float(sum(times))
  val = n_exec / dt
  line = {'impl': 'reference', 'metric': 'scan_pairs_per_sec', 'value': val, 'unit': 'pairs/s',
          'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
          'ms_per_step': 1e3 * dt / n_exec, 'higher_is_better': True, 'scaling': 'weak',
          'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'config': base_config(args.gpus),
          'cpu_baseline': {'value': val, 'unit': 'pairs/s', 'cores': cores, 'kind': 'port',
                           'sample': f'{n_exec} FULL-SIZE pair(s) of the workload (same generator and seeds as the B200 arm: '
                                     f'{N_RAW} raw points per scan -> N0={info["n0"]}, N1={info["n1"]} voxels), not a reduced sample; '
                                     'CPU path = oracle port (torch-CPU index_select/mm/index_add per kernel offset, the algorithm '
                                     "of MinkowskiEngine's CPU backend) + restated kNN / Procrustes / Adam refinement",
                           'steps_executed': n_exec, 'seconds_per_pair': times,
                           'warmup_executed': f'1 pair of {REF_MIN_N_RAW} raw points ({t_warm:.1f} s)'},
          'workload_detail': info, 'parity': parity,
          'e2e': {'value': val, 'unit': 'pairs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
  _emit(json.dumps(line))


# ------------------------------------------------------------------------------------------
# the B200 arm
# ------------------------------------------------------------------------------------------
def run_ours(args):
  import torch.distributed as dist
  from deepglobalregistration_b200 import _abi, sharding
  from deepglobalregistration_b200.core.deep_global_registration import DeepGlobalRegistration

  world = int(os.environ.get('WORLD_SIZE', '1'))
  rank = int(os.environ.get('RANK', '0'))
  local = int(os.environ.get('LOCAL_RANK', '0'))
  if world > 1:
    dist.init_process_group('nccl', device_id=torch.device('cuda', local))
  torch.cuda.set_device(local)
  dev = torch.device('cuda', local)
  pin_rank_to_numa_node(local)

  state = syn.make_checkpoint(0)
  cfg = types.SimpleNamespace(weights=state, clip_weight_thresh=0.05, verbose=False)
  dgr = DeepGlobalRegistration(cfg, device=dev)
  dgr.use_icp = False     # the benchmarked unit is tap A (through the refinement), as on the CPU arm
  inflight = INFLIGHT if dgr._native_ok() else 1

  strong = args.pairs > 0
  if strong:
    # BASELINE config 4: a fixed set of pairs (seeds 0 .. pairs-1) round-robin over the ranks, same total at every N
    seeds = sharding.shard_indices(args.pairs, rank, world)
    n_steps_default = len(seeds)
  else:
    # weak scaling = the per-GPU work is FIXED as N grows: every rank registers the same POOL pairs (its own
    # copies), cycled over the steps.  (Round 1 gave every rank its own seeds; their voxel counts differ by up to
    # 10 %, and with the result gather as a sync point the slowest rank's data then set the 8-GPU time.)
    seeds = list(range(POOL))
    n_steps_default = args.steps
  pool = min(len(seeds), POOL) if not strong else len(seeds)
  log(f'[bench] rank {rank}/{world}: generating {pool} pair(s)')
  pairs_host = [syn.room_pair(sd, n_raw=N_RAW) for sd in seeds[:pool]]
  pairs_dev = [(torch.from_numpy(a).to(dev), torch.from_numpy(b).to(dev)) for a, b, _ in pairs_host]

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  def gather_poses(rows, total):
    # the path's only collective: one all-gather of [pairs, 20] results (NCCL over NVLink)
    return sharding.gather_results(rows, total, device=dev)

  def timed(n_steps, host_inputs):
    """n_steps register() calls (`inflight` pairs in flight) bracketed by barrier + synchronize; device time by
    CUDA events; the result gather is inside the timed region."""
    barrier()
    src = pairs_host if host_inputs else pairs_dev
    pairs = [src[s % pool][:2] for s in range(n_steps)]
    l0 = _abi.lib().dgr_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.perf_counter()
    e0.record()
    out = dgr.register_batch(pairs, inflight=inflight)
    rows = [sharding.pack_result(T, info.get('wsum', 0.0), info.get('iterations', 0), branch) for T, branch, info in out]
    if strong and n_steps == len(seeds):
      gathered = gather_poses(rows, args.pairs)            # the whole fixed set, in pair order
    else:
      gathered = gather_poses(rows, world * len(rows))
    e1.record()
    barrier()
    wall = time.perf_counter() - w0
    ms_local = ms = e0.elapsed_time(e1)
    launches = _abi.lib().dgr_launch_count() - l0
    d2h = sum(info.get('d2h_bytes', 0) for _, _, info in out)
    reads = sum(info.get('host_reads', 0) for _, _, info in out)
    per_rank = None
    if world > 1:
      tm = torch.tensor([ms, wall * 1e3], device=dev, dtype=torch.float64)
      allt = [torch.empty_like(tm) for _ in range(world)]
      dist.all_gather(allt, tm)
      per_rank = [float(t[0]) for t in allt]
      ms, wall = max(per_rank), max(float(t[1]) for t in allt) / 1e3
    done = sorted(info.get('t_done', w0) for _, _, info in out)
    steps_ms = [1e3 * d for d in np.diff([w0] + done)]
    return dict(ms=ms, ms_local=ms_local, wall=wall, launches=launches, d2h=d2h, reads=reads, poses=gathered,
                steps_ms=steps_ms, per_rank_ms=per_rank, last=out[-1])

  def profiled_serial_pass(n_steps):
    """One pair at a time with per-launch CUDA events around every convolution launch (the roofline of the
    dominant kernel); with two pairs in flight the events would time two kernels sharing the GPU."""
    ctx = dgr.native_context(0)
    torch.cuda.synchronize()
    ctx.profile(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    stages = {}
    for s in range(n_steps):
      dgr.register(*pairs_dev[s % pool])
      for k, v in ctx.stage_times().items():
        stages.setdefault(k, []).append(v)
    e1.record()
    torch.cuda.synchronize()
    rows = ctx.profile_read(64 * n_steps + 64)
    ctx.profile(False)
    return rows, e0.elapsed_time(e1), {k: float(np.mean(v)) for k, v in stages.items()}

  # started before the warm-up: the sampler's own start-up (NVML init) must not land in the timed region
  sampler = ClockSampler(local) if rank == 0 and not os.environ.get('DGR_BENCH_NO_SAMPLER') else None
  K = n_steps_default
  log(f'[bench] rank {rank}/{world}: model + {pool} pairs ready ({inflight} in flight), warming up')
  # warm-up: every pair of the pool at least max(W, 3) times on both input paths (arena growth, pinned staging,
  # NCCL channels), then one untimed rehearsal of exactly the timed loops
  n_warm = max(args.warmup, 3) * min(pool, POOL)
  timed(n_warm, host_inputs=False)
  timed(max(min(pool, POOL), 2), host_inputs=True)
  timed(K, host_inputs=False)
  timed(K, host_inputs=True)
  gc.collect()
  log('[bench] warm-up done, timing')

  t_start = time.time()
  thr0 = cgroup_throttled_ms()
  res = timed(K, host_inputs=False)               # `value`: scans resident in HBM
  res_e2e = timed(K, host_inputs=True)            # `e2e`: host buffers in, pose out
  t_end = time.time()
  thr1 = cgroup_throttled_ms()
  clocks = sampler.stop(t_start, t_end) if sampler else None
  if args.dump_outputs and rank == 0:
    dump_outputs(args.dump_outputs, res['last'], res_e2e['last'])
  arena = [dgr.native_context(k).stats() for k in range(inflight)] if dgr._native_ok() else None

  prof_rows, serial_ms, stage_ms, n_prof = None, None, None, min(K, 20)
  if rank == 0 and dgr._native_ok():
    prof_rows, serial_ms, stage_ms = profiled_serial_pass(n_prof)

  # supplementary: the literal reference call (use_icp = True, host arrays in, pose out).  Single-rank
  # only (a failure here must not strand peers in a collective) and never fatal to the contract line.
  e2e_icp = None
  if world == 1 and not strong:
    try:
      dgr.use_icp = True
      timed(2 * pool, host_inputs=True)
      r_icp = timed(K, host_inputs=True)
      e2e_icp = {'value': K / (r_icp['ms'] / 1e3), 'unit': 'pairs/s', 'ms_per_step': r_icp['ms'] / K,
                 'icp_iterations_last_pair': r_icp['last'][2].get('icp_iterations'),
                 'note': 'register() exactly as the reference defaults it: Procrustes + refinement + '
                         'point-to-point ICP; outside the contract value, which is SURVEY 8(d)\'s unit'}
    except Exception as e:   # noqa: BLE001
      log(f'[bench] supplementary ICP timing failed: {e!r}')
    finally:
      dgr.use_icp = False

  if rank != 0:
    if world > 1:
      dist.destroy_process_group()
    return

  n_total = args.pairs if strong else world * K
  value = n_total / (res['ms'] / 1e3)
  e2e = n_total / (res_e2e['ms'] / 1e3)

  # ---- roofline of the dominant kernel (live CUDA events around every launch, serial pass) ------------
  peaks, peak_src = None, 'fallback (B200_PROFILING.md: 6650 GB/s, 1590 TFLOP/s bf16)'
  try:
    peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    peak_src = 'measured (MEASURED_PEAKS.json)'
  except Exception:   # noqa: BLE001
    pass
  hbm_peak = float(peaks['hbm_gbs']) if peaks else 6650.0
  bf16_peak = float(peaks.get('bf16_tflops_sustained', peaks['bf16_tflops'])) if peaks else 1400.0
  roofline, roofline_tensor, kernel_share = None, None, None
  if prof_rows is not None and len(prof_rows):
    names = {0: 'spconv_tc_kernel', 1: 'spconv_fwd_kernel', 2: 'spconv_table_kernel'}
    by = {}
    for ms, flops, nbytes, kind in prof_rows:
      d = by.setdefault(names.get(int(kind), 'other'), [0, 0.0, 0.0, 0.0])
      d[0] += 1
      d[1] += ms
      d[2] += flops
      d[3] += nbytes
    dom = max(by, key=lambda k: by[k][1])
    n, ms, flops, nbytes = by[dom]
    gbs = nbytes / (ms * 1e-3) / 1e9
    tfs = flops / (ms * 1e-3) / 1e12
    traffic = None
    for name in ('r02_spconv_tc_traffic.json', 'r01_spconv_tc_traffic.json'):
      try:   # per-launch DRAM bytes from the committed ncu --set full capture, if present
        traffic = json.load(open(os.path.join(ROOT, 'profiles', name)))['dram_bytes_per_launch']
        break
      except Exception:   # noqa: BLE001
        pass
    roofline = {'kernel': dom, 'bound': 'hbm', 'achieved': gbs, 'peak': hbm_peak, 'unit': 'GB/s',
                'frac': gbs / hbm_peak, 'traffic': traffic, 'peak_source': peak_src,
                'launches_per_step': n / n_prof, 'avg_launch_ms': ms / n,
                'algorithmic_bytes_per_launch': nbytes / n,
                'bytes_model': 'SURVEY 8(d) gather-scatter model: P*(Cin+Cout)*4 + 8*P + K_nonempty*Cin*Cout*4',
                'measured_in': f'a serial pass of {n_prof} steps right after the timed region (one pair at a time, CUDA '
                               'events on the launching stream around every launch); the timed region itself keeps '
                               f'{inflight} pairs in flight, where an event pair would time two kernels sharing the GPU'}
    roofline_tensor = {'kernel': dom, 'bound': 'tensor', 'achieved': tfs, 'peak': bf16_peak, 'unit': 'TFLOP/s',
                       'frac': tfs / bf16_peak, 'algorithmic_flops_per_launch': flops / n,
                       'note': 'algorithmic fp32 FLOPs 2*P*Cin*Cout; the kernel spends 3 TF32 MMAs per product '
                               '(3xTF32) and TF32 runs at half the bf16 rate, so its ceiling is peak/6'}
    kernel_share = {k: v[1] / serial_ms for k, v in by.items()}
    kernel_share['serial_pass_ms_per_step'] = serial_ms / n_prof

  log(f'[bench] value {value:.2f} pairs/s, e2e {e2e:.2f} pairs/s; timing the CPU sample')
  # ---- CPU baseline on a bounded sample --------------------------------------------------------
  cpu_s, info = cpu_sample_time(state, 0, reps=1)
  cpu = {'value': 1.0 / cpu_s, 'unit': 'pairs/s', 'cores': cpu_threads(), 'kind': 'port',
         'sample': sample_desc(info), 'seconds_per_sample_pair': cpu_s}
  try:     # the same-config CPU time: one FULL-SIZE oracle run of this arm's first pair, recorded with the fixture
    g = np.load(os.path.join(ROOT, 'tests', 'golden', 'fullsize_config2.npz'))
    sec = json.loads(str(g['seconds']))
    cpu['full_size_pair'] = {'seconds_through_refine': sec['total_through_refine'], 'threads': sec['threads'],
                             'pairs_per_sec': 1.0 / sec['total_through_refine'],
                             'where': 'build container, recorded by tests/golden/make_golden_fullsize.py; '
                                      '`bench.py --impl reference` times the same full-size pair on this box'}
  except Exception:   # noqa: BLE001
    pass

  # pose of this arm's first pair (timed `value` loop, step 0 = seed 0) against the CPU oracle's pose of the same pair
  parity = {'end_to_end': fixture_parity(res['poses'][0][:16].numpy()),
            'final_stage_on_oracle_inputs': stage_isolated_parity(dgr, pairs_dev[0]) if dgr._native_ok() and not strong else None,
            'config': WORKLOAD,
            'note': 'end_to_end = register() free-running vs the oracle run of the same pair; the checkpoint is random-init, '
                    'so its correspondences are unrelated points and the fitted pose is ill-conditioned: a few arg-min flips '
                    'inside the feature rounding noise move it by centimetres.  final_stage_on_oracle_inputs feeds the '
                    'oracle\'s correspondences and weights to the CUDA Procrustes + refinement; the other stages are pinned '
                    'at this size by tests/test_gpu_zzzz_golden_fullsize.py (bit-exact voxels / 6-D coordinates, features '
                    '<= 5e-5, logits <= 5e-5)'}
  last = res['last'][2]
  detail = dict(n0=last.get('n0'), n1=last.get('n1'), branch=res['last'][1], refine_iterations=last.get('iterations'),
                pairs_in_flight_per_gpu=inflight, native_executor=bool(dgr._native_ok()),
                host_reads_per_pair=res['reads'] / max(len(res['steps_ms']), 1))
  cfg_out = base_config(world)
  h2d = int(sum(a.nbytes + b.nbytes for a, b, _ in pairs_host) / len(pairs_host))
  n_local = len(res['steps_ms'])
  line = {'metric': 'scan_pairs_per_sec', 'value': value, 'unit': 'pairs/s', 'n_gpus': world, 'steps': args.steps,
          'warmup': args.warmup, 'warmup_steps_run': n_warm + max(min(pool, POOL), 2) + 2 * K,
          'ms_per_step': res['ms'] / n_local, 'higher_is_better': True,
          'scaling': 'strong' if strong else 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
          'config': cfg_out,
          'e2e': {'value': e2e, 'unit': 'pairs/s', 'h2d_bytes_per_step': h2d,
                  'd2h_bytes_per_step': int(res_e2e['d2h'] / n_local),
                  'ms_per_step': res_e2e['ms'] / n_local, 'wall_ms_per_step': 1e3 * res_e2e['wall'] / n_local},
          'gpu_launches': int(res['launches']), 'gpu_launches_per_step': res['launches'] / n_local,
          'clocks': clocks, 'roofline': roofline, 'roofline_tensor': roofline_tensor,
          'kernel_share_of_step': kernel_share, 'stage_ms_serial_pass': stage_ms, 'cpu_baseline': cpu, 'parity': parity, 'workload_detail': detail,
          'wall_ms_per_step': 1e3 * res['wall'] / n_local,
          'host_cgroup_throttled_ms_during_timing': (thr1 - thr0) if thr0 is not None and thr1 is not None else None,
          'device_arena': arena,
          'host_threads': {'torch_intraop': torch.get_num_threads(), 'usable_cpus': effective_cpus(),
                           'affinity': sorted(os.sched_getaffinity(0))[:4] + ['...'] if hasattr(os, 'sched_getaffinity') else None},
          'per_rank_ms': {'value': res['per_rank_ms'], 'e2e': res_e2e['per_rank_ms']},
          'step_ms': {'min': min(res['steps_ms']), 'median': float(np.median(res['steps_ms'])),
                      'max': max(res['steps_ms']), 'all': [round(x, 2) for x in res['steps_ms']],
                      'note': 'gaps between consecutive pair completions on rank 0 (pairs overlap)'},
          'e2e_step_ms': {'min': min(res_e2e['steps_ms']), 'median': float(np.median(res_e2e['steps_ms'])),
                          'max': max(res_e2e['steps_ms']), 'all': [round(x, 2) for x in res_e2e['steps_ms']]},
          'e2e_with_icp': e2e_icp,
          'published_reference': '0.69 s/pair without safeguard+ICP (reference assets/results.npz, unknown GPU)'}
  if strong:
    line['pairs_total'] = args.pairs
    line['config']['pairs_total'] = args.pairs
  _emit(json.dumps(line))
  if world > 1:
    dist.destroy_process_group()


def main():
  # keep stdout clean for the ONE JSON line: libraries (NCCL's version banner, ...) write to fd 1
  real_stdout = os.dup(1)
  os.dup2(2, 1)
  global _emit
  _emit = lambda text: os.write(real_stdout, (text + '\n').encode())
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=None,
                  help='timed steps (default 100 for the B200 arm: ~1.5 s per region, so that one ~0.3 s host stall '
                       'of a shared box costs 10-20 %% instead of halving the number; 1 for --impl reference, '
                       'where one full-size pair is minutes of CPU)')
  ap.add_argument('--warmup', type=int, default=3)
  ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
  ap.add_argument('--pairs', type=int, default=0,
                  help='BASELINE config 4: register this many pairs (seeds 0..pairs-1) round-robin over the ranks - '
                       'the same total at every N (strong scaling); 0 = the contract mode (K steps per rank, weak)')
  ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                  help='after the timed steps, write what the last timed step returned (pose, weight sum) as '
                       'DIR/<name>.npy, so that two builds can be compared output for output')
  args = ap.parse_args()
  if args.steps is not None and args.steps < 1:
    ap.error('--steps must be at least 1')
  if args.steps is not None and args.pairs > 0:
    ap.error('--steps and --pairs exclude each other: with --pairs every pair is one timed step')
  if args.steps is None:
    args.steps = 1 if args.impl == 'reference' else 100
  if args.impl == 'reference':
    run_reference(args)
  else:
    run_ours(args)


if __name__ == '__main__':
  main()
