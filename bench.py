#!/usr/bin/env python
"""Benchmark of the WeatherBench2 hot path on B200 (BASELINE.json).

  python bench.py --gpus N --steps K --warmup W          # this framework
  python bench.py --impl reference --gpus N ...          # CPU reference arm
  python bench.py ... --dump-outputs DIR                 # + last-step outputs

The inputs are generated from fixed seeds, so two builds run with the same
arguments can be compared output for output through --dump-outputs.

Prints ONE JSON line (rank 0).  The top-level keys are the contract line for
BASELINE.json configs[1] (fused weighted RMSE + Bias + ACC, 6 variables x 13
levels x 721 x 1440, chunk = 1 init x 10 leads); `workloads` carries the other
north-star configurations, each with its own value / roofline / e2e / clocks:

  crps_sweep      configs[2]: CRPS + spread / skill, 50 members, 3 vars x 13
                  levels x 721 x 1440 per (init, lead) chunk
  regrid          configs[3]: conservative 0.25 -> 1.5 degree, 6 vars x 37
                  levels per time step
  spectrum_sweep  configs[4]: zonal energy spectrum, 37 levels x 5 vars, time
                  mean fused in (+ the 385 MB all-reduce at N > 1); `latsum` =
                  the fused latitude-weighted reduction of the north star

A "step" is one pass of the path over one chunk resident in HBM (inputs >> L2,
so no flush is needed between steps).  Under torchrun every rank owns its own
chunk (weak scaling: chunks are independent, weatherbench2/evaluation.py:
583-599) and the time sums are all-reduced once at the end (the NCCL
equivalent of xbeam.Mean, evaluation.py:740-744).  Every timed region is
bracketed by barrier + synchronize, timed with CUDA events on the stream the
kernels are launched on, max over ranks; SM clocks and throttle reasons are
sampled through NVML every ~2 ms DURING each timed region.

`value` = device-resident throughput; `e2e` = the same workload through the
public operator API with pinned HOST inputs (H2D inside the timed region, D2H
of the result); `roofline` = achieved algorithmic HBM GB/s of the dominant
kernel vs MEASURED_PEAKS.json; `cpu_baseline` = the oracle port on this box's
host cores on a bounded sample.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)

NLAT, NLON, NLEV, NVAR, NLEAD = 721, 1440, 13, 6, 10
VARIABLES = ['geopotential', 'temperature', 'u_component_of_wind',
             'v_component_of_wind', 'specific_humidity', 'vertical_velocity']
LEVELS = [50, 100, 150, 200, 250, 300, 400, 500, 600, 700, 850, 925, 1000]
BYTES_PER_CELL = 12  # f + t + c, float32 (SURVEY.md section 8d)
SLAB = NLAT * NLON

# configs[2]
ENS_M, ENS_NVAR = 50, 3
ENS_FIELDS = ENS_NVAR * NLEV          # fields of one (init, lead) chunk
ENS_BYTES_PER_POINT = 4 * ENS_M + 4   # members + truth
# configs[3]
RG_FIELDS = 6 * 37                    # one time step
RG_TLON, RG_TLAT = 240, 121
RG_BYTES_PER_CELL = 4 + 4 * (RG_TLON * RG_TLAT) / (NLON * NLAT)
# configs[4]
SP_SLOTS = 37 * 5                     # (level, variable) outputs of the time mean
SP_TIMES = 16                         # time steps per launch (12.3 GB)
SP_NK = NLON // 2 + 1
# --dump-outputs: outputs larger than this are sampled (same indices every run)
DUMP_MAX_ELEMS = 1 << 20
DUMP_SEED = 20240101
DUMP_MAX_BYTES = 64 << 20


def _peak_gbs():
  path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  try:
    with open(path) as fh:
      return float(json.load(fh)['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
  except Exception:  # pylint: disable=broad-except
    return 6650.0, 'fallback (B200_PROFILING.md)'


def _ncu_traffic(key):
  """dram bytes per launch of a dominant kernel from the committed ncu capture
  of this command (profiles/r2_traffic.json, written by
  benchmarks/ncu_traffic.py); None if absent."""
  if os.environ.get('WB2_DET_PATH') == 'ldg' and key == 'rmse_acc':
    return None
  for name in ('r2_traffic.json',):
    try:
      with open(os.path.join(ROOT, 'profiles', name)) as fh:
        return float(json.load(fh)[key]['dram_bytes_per_launch'])
    except Exception:  # pylint: disable=broad-except
      pass
  if key == 'rmse_acc':
    try:
      with open(os.path.join(ROOT, 'profiles', 'r1_k1_traffic.json')) as fh:
        return float(json.load(fh)['dram_bytes_per_launch'])
    except Exception:  # pylint: disable=broad-except
      pass
  return None


# ------------------------------------------------------------------------------
# clocks: NVML sampled every ~2 ms from a thread while a region is timed
# ------------------------------------------------------------------------------
class ClockSampler:
  """SM clock + throttle reasons during a timed region.  The headline region
  lasts tens of ms, so `nvidia-smi -lms` (>= 100 ms period) cannot see it;
  NVML is polled directly instead."""
  REASONS = {0x4: 'sw_power_cap', 0x8: 'hw_slowdown', 0x20: 'sw_thermal_slowdown',
             0x40: 'hw_thermal_slowdown', 0x80: 'hw_power_brake_slowdown'}

  def __init__(self, index=0, period_s=0.002):
    self.period = period_s
    self.samples, self.bits, self.power = [], 0, []
    self.stop_flag = threading.Event()
    self.thread = None
    self.handle = None
    self.smax = None
    try:
      import pynvml  # pylint: disable=import-outside-toplevel
      self.nv = pynvml
      pynvml.nvmlInit()
      # CUDA_VISIBLE_DEVICES remaps indices: go through the PCI bus id
      import torch  # pylint: disable=import-outside-toplevel
      p = torch.cuda.get_device_properties(index)
      bus = f'{p.pci_domain_id:08x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0'
      try:
        self.handle = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
      except Exception:  # pylint: disable=broad-except
        self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
      self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(
          self.handle, pynvml.NVML_CLOCK_SM))
      self.reasons_fn = getattr(
          pynvml, 'nvmlDeviceGetCurrentClocksEventReasons',
          getattr(pynvml, 'nvmlDeviceGetCurrentClocksThrottleReasons', None))
    except Exception:  # pylint: disable=broad-except
      self.handle = None

  def _run(self):
    nv, h = self.nv, self.handle
    while not self.stop_flag.is_set():
      try:
        self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
        self.bits |= int(self.reasons_fn(h))
        self.power.append(nv.nvmlDeviceGetPowerUsage(h) / 1000.0)
      except Exception:  # pylint: disable=broad-except
        pass
      time.sleep(self.period)

  def start(self):
    self.samples, self.bits, self.power = [], 0, []
    self.stop_flag.clear()
    if self.handle is not None:
      self.thread = threading.Thread(target=self._run, daemon=True)
      self.thread.start()

  def stop(self):
    if self.handle is None:
      return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable'],
              'samples': 0}
    self.stop_flag.set()
    self.thread.join(timeout=2)
    reasons = sorted(n for b, n in self.REASONS.items() if self.bits & b)
    return {'sm_mhz': float(np.median(self.samples)) if self.samples else None,
            'sm_min_mhz': float(min(self.samples)) if self.samples else None,
            'sm_max_mhz': self.smax, 'reasons': reasons,
            'power_w_max': float(max(self.power)) if self.power else None,
            'samples': len(self.samples), 'source': 'NVML, ~2 ms period'}


def _bind_to_gpu_numa_node(local):
  """Pins this process to the host cores of the GPU's NUMA node BEFORE pinned
  host buffers are allocated, so that the staging memory of every rank is
  local to its GPU's PCIe root (8 ranks streaming from one socket is what held
  the round-1 end-to-end scaling at 0.85)."""
  try:
    import torch  # pylint: disable=import-outside-toplevel
    p = torch.cuda.get_device_properties(local)
    bus = f'{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0'
    with open(f'/sys/bus/pci/devices/{bus}/numa_node') as fh:
      node = int(fh.read().strip())
    if node < 0:
      return {'numa_node': node, 'bound': False}
    with open(f'/sys/devices/system/node/node{node}/cpulist') as fh:
      cpus = set()
      for part in fh.read().strip().split(','):
        a, _, b = part.partition('-')
        cpus.update(range(int(a), int(b or a) + 1))
    allowed = os.sched_getaffinity(0)
    target = cpus & allowed
    if target:
      os.sched_setaffinity(0, target)
    return {'numa_node': node, 'bound': bool(target), 'cores': len(target)}
  except Exception as e:  # pylint: disable=broad-except
    return {'numa_node': None, 'bound': False, 'why': str(e)[:80]}


# ------------------------------------------------------------------------------
# CPU arm: the oracle port (the reference needs xarray / jax, not installed)
# ------------------------------------------------------------------------------
def usable_cores():
  """Host threads this process may actually use: the affinity mask capped by
  the cgroup CPU quota (os.cpu_count() reports the machine, not the lease)."""
  aff = len(os.sched_getaffinity(0))
  quota = None
  for path in ('/sys/fs/cgroup/cpu.max', '/sys/fs/cgroup/cpu/cpu.cfs_quota_us'):
    try:
      with open(path) as fh:
        txt = fh.read().split()
      if path.endswith('cpu.max'):
        if txt[0] != 'max':
          quota = float(txt[0]) / float(txt[1])
      else:
        q = float(txt[0])
        if q > 0:
          with open('/sys/fs/cgroup/cpu/cpu.cfs_period_us') as fh2:
            quota = q / float(fh2.read().split()[0])
      break
    except Exception:  # pylint: disable=broad-except
      continue
  n = aff if quota is None else max(1, min(aff, int(quota + 0.5)))
  return n, {'os_cpu_count': os.cpu_count(), 'sched_getaffinity': aff,
             'cgroup_cpu_quota': quota}


def _lat_lon():
  return np.linspace(-90, 90, NLAT), np.arange(NLON) * 0.25


def _cpu_inputs(kind, seed):
  rs = np.random.RandomState(seed)
  if kind == 'rmse_acc':
    shape = (NLEV, NLAT, NLON)
    return tuple(rs.standard_normal(shape).astype(np.float32) for _ in range(3))
  if kind == 'crps':
    # a latitude band of one field: the port costs the same per point anywhere
    x = rs.standard_normal((ENS_M, 181, NLON)).astype(np.float32)
    t = rs.standard_normal((181, NLON)).astype(np.float32)
    return x, t
  if kind == 'regrid':
    return (rs.standard_normal((6, NLON, NLAT)).astype(np.float32),)
  if kind == 'spectrum':
    return (rs.standard_normal((NLEV, NLAT, NLON)).astype(np.float32),)
  raise ValueError(kind)


def _cpu_compute(kind, data):
  """One bounded sample of `kind` with the oracle (op-for-op restatement of the
  reference) on ONE host thread (BLAS / OpenMP pools are limited to 1, so that
  `cores` means what it says; parallelism comes from the process pool);
  returns (seconds in the path, units processed)."""
  try:
    from threadpoolctl import threadpool_limits  # pylint: disable=import-outside-toplevel
    with threadpool_limits(limits=1):
      return _cpu_compute_1t(kind, data)
  except ImportError:
    return _cpu_compute_1t(kind, data)


def _cpu_compute_1t(kind, data):
  from oracle import wb2_oracle as orc
  lat, lon = _lat_lon()
  if kind == 'rmse_acc':
    f, t, c = data
    dims = ('level', 'latitude', 'longitude')
    t0 = time.perf_counter()
    orc.rmse_sqrt_before_time_avg(f, dims, t, dims, lat, lon)
    orc.bias(f, dims, t, dims, lat, lon)
    orc.acc(f, dims, t, dims, c, dims, lat, lon)
    return time.perf_counter() - t0, f.size
  if kind == 'crps':
    x, t = data
    blat = lat[270:451]
    fd, td = ('realization', 'latitude', 'longitude'), ('latitude', 'longitude')
    t0 = time.perf_counter()
    orc.crps(x, fd, t, td, 'realization', blat, lon)  # skill + spread inside
    orc.ensemble_mean_rmse_sqrt_before_time_avg(x, fd, t, td, 'realization',
                                                blat, lon)
    orc.ensemble_stddev_sqrt_before_time_avg(x, fd, 'realization', blat, lon)
    return time.perf_counter() - t0, t.size
  if kind == 'regrid':
    (x,) = data
    src = orc.Grid(lon, lat)
    tgt = orc.Grid(np.arange(RG_TLON) * 1.5, np.linspace(-90, 90, RG_TLAT))
    t0 = time.perf_counter()
    orc.conservative_regrid(x, src, tgt)
    return time.perf_counter() - t0, x.size
  if kind == 'spectrum':
    (x,) = data
    t0 = time.perf_counter()
    s, _, _, _ = orc.zonal_energy_spectrum(
        x, ('time', 'latitude', 'longitude'), lat, lon)
    s.mean(axis=0)
    return time.perf_counter() - t0, x.size
  raise ValueError(kind)


def _worker(args):
  """One host process of the reference arm: inputs are generated once (not
  timed), then `reps` samples of the path."""
  kind, seed, reps = args
  os.environ.setdefault('OMP_NUM_THREADS', '1')
  data = _cpu_inputs(kind, seed)
  total_t, total_units = 0.0, 0
  for _ in range(reps):
    dt, n = _cpu_compute(kind, data)
    total_t += dt
    total_units += n
  return total_t, total_units


_CPU_DESC = {
    'rmse_acc': ('grid-cells/s', f'1 variable x {NLEV} levels x {NLAT}x{NLON}, '
                 'RMSE+Bias+ACC'),
    'crps': ('grid-points/s', f'{ENS_M} members x 181x{NLON} band, CRPS + '
             'spread/skill + ens-mean RMSE + stddev'),
    'regrid': ('grid-cells/s', f'6 fields {NLON}x{NLAT} -> {RG_TLON}x{RG_TLAT}, '
               'conservative (dense float32 einsum like the reference)'),
    'spectrum': ('grid-cells/s', f'{NLEV} fields x {NLAT}x{NLON}, rfft + power + time '
                 'mean'),
}


def cpu_pool_rate(kind, workers, reps, pool):
  res = pool.map(_worker, [(kind, 100 + i, reps) for i in range(workers)])
  # all processes compute concurrently; the job takes as long as the slowest
  # one spends in the path (input generation is not part of it)
  wall = max(r[0] for r in res)
  return sum(r[1] for r in res) / wall, wall


def cpu_baseline_single(kind='rmse_acc', reps=3):
  """Oracle on one core, bounded sample."""
  data = _cpu_inputs(kind, 0)
  _cpu_compute(kind, data)  # warm-up (page faults, imports)
  tt, units = 0.0, 0
  for _ in range(reps):
    dt, n = _cpu_compute(kind, data)
    tt += dt
    units += n
  unit, desc = _CPU_DESC[kind]
  return {'value': units / tt, 'unit': unit, 'cores': 1, 'kind': 'port',
          'sample': f'{reps} x ({desc}) via oracle/wb2_oracle.py (NumPy '
                    'restatement of the xarray path), time.perf_counter around '
                    'the compute only'}


def run_reference(args):
  """--impl reference: the oracle port on the host cores this lease may use
  (the reference itself needs xarray, which is not installed: kind = "port").
  The worker count is calibrated: the usable-core count and its halves are
  tried once each and the fastest is kept, so an over-subscribed lease does not
  understate the reference (round 1: 128 processes on a 4-core share)."""
  rank = int(os.environ.get('RANK', 0))
  if rank != 0:
    return
  import multiprocessing as mp
  ncores, core_info = usable_cores()
  ctxm = mp.get_context('fork')
  legs = {}
  for kind in ('rmse_acc', 'crps', 'regrid', 'spectrum'):
    cap = min(ncores, 64) if kind == 'crps' else min(ncores, 256)
    cands = sorted({max(1, cap), max(1, cap // 2), max(1, cap // 4)}, reverse=True)
    best = None
    calib = []
    for w in cands:
      with ctxm.Pool(w) as pool:
        cpu_pool_rate(kind, w, 1, pool)  # page faults, imports
        rate, _ = cpu_pool_rate(kind, w, 2, pool)
      calib.append({'workers': w, 'value': rate})
      if best is None or rate > best[1]:
        best = (w, rate)
    w = best[0]
    steps = args.steps if kind == 'rmse_acc' else max(1, min(args.steps, 3))
    with ctxm.Pool(w) as pool:
      for _ in range(max(0, min(args.warmup, 1))):
        cpu_pool_rate(kind, w, 1, pool)
      rate, wall = cpu_pool_rate(kind, w, steps, pool)
    unit, desc = _CPU_DESC[kind]
    legs[kind] = {'value': rate, 'unit': unit, 'workers': w, 'steps': steps,
                  'ms_per_step': 1e3 * wall / steps, 'calibration': calib,
                  'sample': f'{w} processes x {steps} steps x ({desc}) via '
                            'oracle/wb2_oracle.py'}
  main = legs['rmse_acc']
  line = {
      'impl': 'reference', 'metric': 'grid-cells/s', 'value': main['value'],
      'unit': 'grid-cells/s', 'n_gpus': args.gpus, 'steps': args.steps,
      'warmup': args.warmup, 'ms_per_step': main['ms_per_step'],
      'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
      'dtype': 'f32', 'data': 'synthetic',
      'config': dict(_config(args.gpus),
                     reference_step=f"{main['workers']} processes x (1 variable "
                                    f'x {NLEV} levels x {NLAT}x{NLON}) = '
                                    f"{main['workers'] * NLEV * SLAB} cells"),
      'cpu_baseline': {'value': main['value'], 'unit': 'grid-cells/s',
                       'cores': main['workers'], 'kind': 'port',
                       'sample': main['sample'], 'host': core_info,
                       'calibration': main['calibration']},
      'e2e': {'value': main['value'], 'unit': 'grid-cells/s',
              'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
      'workloads': {
          'crps_sweep': _ref_leg(legs['crps']),
          'regrid': _ref_leg(legs['regrid']),
          'spectrum_sweep': _ref_leg(legs['spectrum']),
      },
  }
  print(json.dumps(line))


def _ref_leg(leg):
  return {'value': leg['value'], 'unit': leg['unit'],
          'cpu_baseline': {'value': leg['value'], 'unit': leg['unit'],
                           'cores': leg['workers'], 'kind': 'port',
                           'sample': leg['sample'],
                           'calibration': leg['calibration']},
          'e2e': {'value': leg['value'], 'unit': leg['unit'],
                  'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}


def _config(n_gpus):
  return {'workload': 'configs[1]: RMSE+Bias+ACC, 6 vars x 13 levels x '
                      '721x1440, chunk = 1 init x 10 lead (780 fields, '
                      '9.72 GB f32 per step per GPU)',
          'cells_per_step_per_gpu': NLEAD * NVAR * NLEV * SLAB,
          'regions': 1, 'skipna': False,
          'l2_policy': 'inputs (9.72 GB) >> L2 (126 MB); no flush needed',
          'parallelism': f'chunks sharded over {n_gpus} GPU(s), one NCCL '
                         'all-reduce of the time-sum at the end'}


# ------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------
class Harness:
  """Shared state of the GPU arm: device, stream, process group, timing."""

  def __init__(self, args):
    import torch
    import torch.distributed as dist
    from weatherbench2_b200 import _lib
    self.torch, self.dist, self._lib = torch, dist, _lib
    self.args = args
    self.rank = int(os.environ.get('RANK', 0))
    self.world = int(os.environ.get('WORLD_SIZE', 1))
    self.local = int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(self.local)
    self.numa = _bind_to_gpu_numa_node(self.local)
    if self.world > 1:
      os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
      dist.init_process_group('nccl', device_id=torch.device('cuda', self.local))
    self.dev = torch.device('cuda', self.local)
    os.environ.setdefault('WB2_DEVICE', str(self.local))
    self.ctx = _lib.default_context(self.local)
    # one explicit (non-legacy) stream shared by torch and the library, so that
    # torch.cuda.Event timing sees the kernels
    self.stream = torch.cuda.Stream(device=self.dev)
    torch.cuda.set_stream(self.stream)
    self.ctx.set_stream(self.stream.cuda_stream)
    self.sampler = ClockSampler(self.local)
    self.peak, self.peak_src = _peak_gbs()
    self.outputs = {}  # name -> host array, for --dump-outputs

  def keep(self, name, value):
    """Records what a timed path returned in its last step for
    --dump-outputs: a tensor, an array or an xarray_lite Dataset (one entry
    per variable).  Outputs above DUMP_MAX_ELEMS elements are reduced to a
    fixed, seeded sample of their flattened elements."""
    if not self.args.dump_outputs:
      return
    if hasattr(value, 'keys'):
      for v in value.keys():
        self.keep(f'{name}.{v}', value[v].values)
      return
    torch = self.torch
    if not isinstance(value, (np.ndarray, torch.Tensor)):
      value = np.asarray(value.values)  # an xarray_lite DataArray
    flat = value.reshape(-1)
    if flat.shape[0] > DUMP_MAX_ELEMS:
      rng = np.random.default_rng(DUMP_SEED)
      idx = np.sort(rng.integers(0, flat.shape[0], DUMP_MAX_ELEMS))
      if isinstance(flat, torch.Tensor):
        idx = torch.from_numpy(idx).to(flat.device)
      flat = flat[idx]
      name += '.sample'
    else:
      flat = value
    if isinstance(flat, torch.Tensor):
      flat = flat.cpu().numpy()
    flat = np.asarray(flat)
    if flat.dtype not in (np.float32, np.float64):
      flat = flat.astype(np.float64)
    self.outputs[name] = np.array(flat)

  def dump_outputs(self, out_dir):
    """Writes the recorded outputs as <out_dir>/<name>.npy (rank 0)."""
    total = sum(a.nbytes for a in self.outputs.values())
    assert total <= DUMP_MAX_BYTES, total
    os.makedirs(out_dir, exist_ok=True)
    for name, a in self.outputs.items():
      np.save(os.path.join(out_dir, f'{name}.npy'), a)

  def barrier(self):
    if self.world > 1:
      self.dist.barrier()
    self.torch.cuda.synchronize()

  def max_over_ranks(self, values):
    t = self.torch.tensor(values, device=self.dev, dtype=self.torch.float64)
    if self.world > 1:
      self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
    return [float(x) for x in t.tolist()]

  def time_steps(self, step, tail, steps, warmup):
    """W warm-up steps (+ the tail once), then EXACTLY `steps` steps and the
    tail (time sum + all-reduce) between two events, barrier + synchronize on
    both sides, clocks sampled in between.  Returns (ms_total, ms_kernels,
    launches, clocks), times = max over ranks."""
    torch = self.torch
    for i in range(warmup):
      step(i)
    tail(warm=True)
    self.barrier()
    if self.rank == 0:  # one NVML poller per box (8 of them contend in the driver)
      self.sampler.start()
    launches0 = self.ctx.launch_count
    ev0 = torch.cuda.Event(enable_timing=True)
    evk = torch.cuda.Event(enable_timing=True)
    ev1 = torch.cuda.Event(enable_timing=True)
    self.barrier()
    ev0.record()
    for i in range(steps):
      step(warmup + i)
    evk.record()
    tail(warm=False)
    ev1.record()
    self.barrier()
    clocks = self.sampler.stop() if self.rank == 0 else None
    launches = self.ctx.launch_count - launches0
    mine = [ev0.elapsed_time(ev1), ev0.elapsed_time(evk)]
    ms_total, ms_kernels = self.max_over_ranks(mine)
    if clocks is not None and self.world > 1:
      # spread of the per-rank kernel times (the job time is the max)
      lo = self.max_over_ranks([-mine[1]])[0]
      clocks['kernel_ms_per_step_min_max_over_ranks'] = [
          -lo / max(steps, 1), ms_kernels / max(steps, 1)]
    elif self.world > 1:
      self.max_over_ranks([-mine[1]])
    return ms_total, ms_kernels, int(launches), clocks

  def time_host(self, fn, steps):
    """End-to-end region: host clock around `steps` synchronous operator calls
    (each returns with the result in host memory), max over ranks."""
    self.barrier()
    if self.rank == 0:
      self.sampler.start()
    t0 = time.perf_counter()
    out = None
    for i in range(steps):
      out = fn(i)
    self.torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    clocks = self.sampler.stop() if self.rank == 0 else None
    (dt,) = self.max_over_ranks([dt])
    return dt, out, clocks

  def roofline(self, key, kernel, alg_bytes, kernel_ms):
    achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
    return {'bound': 'hbm', 'achieved': achieved, 'peak': self.peak,
            'unit': 'GB/s', 'frac': achieved / self.peak,
            'traffic': _ncu_traffic(key), 'peak_source': self.peak_src,
            'kernel': kernel, 'kernel_ms': kernel_ms,
            'algorithmic_bytes_per_launch': alg_bytes}

  def pinned_from(self, tensor):
    """Pinned host copy of a device tensor (its shape), NUMA-local."""
    h = self.ctx.pinned_empty(tuple(tensor.shape), np.float32)
    self._lib.check(self.ctx.lib.wb2_memcpy_d2h(
        self.ctx.handle, h.ctypes.data, tensor.data_ptr(), h.nbytes))
    return h

  def free_pinned(self, *arrays):
    for h in arrays:
      self.ctx.host_free(h.ctypes.data)


def bench_rmse_acc(h):
  """configs[1]; returns the top-level contract keys."""
  torch, _lib, ctx, args = h.torch, h._lib, h.ctx, h.args
  from weatherbench2_b200 import _spatial as sp
  nfield = NLEAD * NVAR * NLEV
  gen = torch.Generator(device=h.dev)
  gen.manual_seed(802701 + h.rank)
  f, t, c = (torch.randn((nfield, NLAT, NLON), device=h.dev, dtype=torch.float32,
                         generator=gen) for _ in range(3))
  lat, lon = _lat_lon()
  (_, spec), = sp.build_weights(ctx, lat, lon, [None], 'lat_lon', NLON)
  base = min(f.data_ptr(), t.data_ptr(), c.data_ptr())
  offs = [np.arange(nfield, dtype=np.int64) * SLAB + (x.data_ptr() - base) // 4
          for x in (f, t, c)]
  total = args.warmup + args.steps
  out = torch.zeros((total, nfield, _lib.DET_NSTAT), device=h.dev,
                    dtype=torch.float64)

  def step(i):
    ctx.det_metrics(base, base, base, _lib.F32, offs[0], offs[1], offs[2],
                    spec, False, out[i].data_ptr())

  def tail(warm):
    # time mean over the steps of this rank, then ONE all-reduce (sum, count)
    s = out[:args.warmup].sum(dim=0) if warm else out[args.warmup:].sum(dim=0)
    if h.world > 1:
      h.dist.all_reduce(s)

  ms_total, ms_kernels, launches, clocks = h.time_steps(step, tail, args.steps,
                                                        args.warmup)
  cells = nfield * SLAB
  # sanity (cheap, on rank 0): statistic 6 is the weight sum = nlat * nlon
  wsum = float(out[args.warmup, 0, 6].item())
  assert abs(wsum - SLAB) < 1e-3 * SLAB, wsum
  h.keep('rmse_acc.stats', out[args.warmup + args.steps - 1])
  line = {
      'metric': 'grid-cells/s',
      'value': h.world * cells * args.steps / (ms_total * 1e-3),
      'unit': 'grid-cells/s', 'n_gpus': h.world, 'steps': args.steps,
      'warmup': args.warmup, 'ms_per_step': ms_total / args.steps,
      'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
      'dtype': 'f32', 'data': 'synthetic', 'config': _config(h.world),
      'clocks': clocks, 'gpu_launches': launches,
      'roofline': h.roofline(
          'rmse_acc', ('det_metrics_kernel<float,4,CLIM> (LDG path)'
                       if os.environ.get('WB2_DET_PATH') == 'ldg' else
                       'det_tma_kernel<CLIM,!SKIPNA> (TMA ring)') + ' + finalize',
          cells * BYTES_PER_CELL, ms_kernels / args.steps),
  }
  if not args.no_e2e:
    line['e2e'] = e2e_rmse_acc(h, f, t, c)
  return line


def e2e_rmse_acc(h, f, t, c):
  """A sweep over init times through evaluation._metric_and_region_loop on
  pinned-HOST datasets: chunk i = 1 init x 10 leads, its truth is the by-init
  gather truth.sel(time=valid_time) of a host record and its climatology the
  day-of-year lookup.  Inside `ctx.slab_cache()` the truth / climatology slabs
  that consecutive chunks share stay in HBM, so in steady state only the
  forecast and ONE new valid time cross PCIe per chunk."""
  import pandas as pd
  from weatherbench2_b200 import config, evaluation, metrics
  from weatherbench2_b200 import xarray_lite as xl
  args, ctx = h.args, h.ctx
  nsteps = max(1, args.e2e_steps)
  ntime = NLEAD + nsteps + 1  # + 1 warm-up chunk
  per_time = NVAR * NLEV
  # host record: forecast of one chunk, truth / climatology of `ntime` valid
  # times (times beyond the resident chunk reuse its slabs -- same bytes)
  hf = h.pinned_from(f.view(NLEAD, NVAR, NLEV, NLAT, NLON))
  ht = ctx.pinned_empty((ntime, NVAR, NLEV, NLAT, NLON), np.float32)
  hc = ctx.pinned_empty((ntime, NVAR, NLEV, NLAT, NLON), np.float32)
  for k in range(ntime):
    src = (k % NLEAD) * per_time
    for dst, dev in ((ht, t), (hc, c)):
      h._lib.check(ctx.lib.wb2_memcpy_d2h(
          ctx.handle, dst[k].ctypes.data,
          dev[src:src + per_time].data_ptr(), dst[k].nbytes))
  lat, lon = _lat_lon()
  day = np.timedelta64(1, 'D').astype('timedelta64[ns]')
  t0 = np.datetime64('2020-01-01T00', 'ns')
  times = t0 + np.arange(ntime) * day
  lead = np.arange(NLEAD) * day
  levels = np.array(LEVELS)
  tdims = ('time', 'level', 'latitude', 'longitude')
  cdims = ('dayofyear', 'level', 'latitude', 'longitude')
  truth_src = xl.Dataset({v: (tdims, ht[:, i]) for i, v in enumerate(VARIABLES)},
                         {'time': times, 'level': levels, 'latitude': lat,
                          'longitude': lon})
  clim = xl.Dataset({v: (cdims, hc[:, i]) for i, v in enumerate(VARIABLES)},
                    {'dayofyear': pd.DatetimeIndex(times).dayofyear.values,
                     'level': levels, 'latitude': lat, 'longitude': lon})
  eval_config = config.Eval(
      metrics={'rmse': metrics.RMSESqrtBeforeTimeAvg(), 'bias': metrics.Bias(),
               'acc': metrics.ACC(climatology=clim)}, temporal_mean=False)
  fdims = ('init_time', 'lead_time', 'level', 'latitude', 'longitude')

  def chunk(i):
    init = times[i:i + 1]
    fcoords = {'init_time': init, 'lead_time': lead, 'level': levels,
               'latitude': lat, 'longitude': lon,
               'valid_time': (('init_time', 'lead_time'),
                              init[:, None] + lead[None, :])}
    forecast = xl.Dataset({v: (fdims, hf[None, :, k]) for k, v in
                           enumerate(VARIABLES)}, fcoords)
    truth = evaluation.select_truth_at_valid_time(truth_src, forecast)
    return evaluation._metric_and_region_loop(  # pylint: disable=protected-access
        forecast, truth, eval_config, skipna=False, compute_chunk=True)

  cells = NLEAD * per_time * SLAB
  with ctx.slab_cache():
    ctx.reset_transfer_stats()
    chunk(0)  # cold chunk: staging buffers, the first 10 valid times
    cold = ctx.transfer_stats()
    ctx.reset_transfer_stats()
    dt, res, clocks = h.time_host(lambda i: chunk(1 + i), nsteps)
    st = ctx.transfer_stats()
  h.keep('rmse_acc.e2e', res)
  d2h = sum(res[v].values.nbytes for v in res.keys())
  h.free_pinned(hf, ht, hc)
  return {'value': h.world * cells * nsteps / dt, 'unit': 'grid-cells/s',
          'h2d_bytes_per_step': int(st['h2d_bytes'] // nsteps),
          'd2h_bytes_per_step': int(max(d2h, st['d2h_bytes'] // nsteps)),
          'cold_chunk_h2d_bytes': int(cold['h2d_bytes']),
          'slab_cache': {'hits_per_step': st['cache_hits'] // nsteps,
                         'misses_per_step': st['cache_misses'] // nsteps},
          'steps': nsteps, 'ms_per_step': 1e3 * dt / nsteps, 'clocks': clocks,
          'host_numa': h.numa,
          'api': 'evaluation._metric_and_region_loop(RMSE+Bias+ACC) per init-time '
                 'chunk on pinned-host datasets inside ctx.slab_cache() -> '
                 'wb2_det_metrics_host (truth / climatology slabs resident in '
                 'HBM across chunks; forecast + 1 new valid time per chunk)'}


def bench_crps(h):
  """configs[2]: CRPS + spread / skill + ensemble-mean (R)MSE / variance from
  one read of the 50 members (K2)."""
  torch, _lib, ctx, args = h.torch, h._lib, h.ctx, h.args
  from weatherbench2_b200 import _spatial as sp
  gen = torch.Generator(device=h.dev)
  gen.manual_seed(802702 + h.rank)
  x = torch.randn((ENS_M, ENS_FIELDS, NLAT, NLON), device=h.dev,
                  dtype=torch.float32, generator=gen)
  sig = torch.randn((1, ENS_FIELDS, NLAT, NLON), device=h.dev,
                    dtype=torch.float32, generator=gen)
  x += sig  # members share a signal (SURVEY.md section 8d)
  del sig
  t = torch.randn((ENS_FIELDS, NLAT, NLON), device=h.dev, dtype=torch.float32,
                  generator=gen)
  lat, lon = _lat_lon()
  (_, spec), = sp.build_weights(ctx, lat, lon, [None], 'lat_lon', NLON)
  base = min(x.data_ptr(), t.data_ptr())
  off_x = (np.arange(ENS_FIELDS, dtype=np.int64) * SLAB +
           (x.data_ptr() - base) // 4)
  off_t = (np.arange(ENS_FIELDS, dtype=np.int64) * SLAB +
           (t.data_ptr() - base) // 4)
  total = args.warmup + args.steps
  out = torch.zeros((total, ENS_FIELDS, _lib.ENS_NSTAT), device=h.dev,
                    dtype=torch.float64)

  def step(i):
    ctx.ens_metrics(base, base, _lib.F32, ENS_M, ENS_FIELDS * SLAB, off_x,
                    off_t, spec, False, out[i].data_ptr())

  def tail(warm):
    s = out[:args.warmup].sum(dim=0) if warm else out[args.warmup:].sum(dim=0)
    if h.world > 1:
      h.dist.all_reduce(s)

  ms_total, ms_kernels, launches, clocks = h.time_steps(step, tail, args.steps,
                                                        args.warmup)
  points = ENS_FIELDS * SLAB
  wsum = float(out[args.warmup, 0, 5].item())
  assert abs(wsum - SLAB) < 1e-3 * SLAB, wsum
  h.keep('crps_sweep.stats', out[args.warmup + args.steps - 1])
  entry = {
      'workload': f'configs[2]: CRPS + spread/skill + ens-mean (R)MSE + variance, '
                  f'{ENS_M} members, {ENS_NVAR} vars x {NLEV} levels x '
                  f'{NLAT}x{NLON} per (init, lead) chunk ({ENS_FIELDS} fields, '
                  '8.26 GB f32 per step per GPU)',
      'value': h.world * points * args.steps / (ms_total * 1e-3),
      'unit': 'grid-points/s (a point carries the 50 member values)',
      'member_cells_per_s': h.world * points * ENS_M * args.steps / (ms_total * 1e-3),
      'ms_per_step': ms_total / args.steps, 'scaling': 'weak',
      'gpu_launches': launches, 'clocks': clocks,
      'roofline': h.roofline('crps_sweep', 'ens_pair_kernel<50> (two points per lane, packed '
                             'f32x2 sorting network) + finalize',
                             points * ENS_BYTES_PER_POINT,
                             ms_kernels / args.steps),
  }
  if not args.no_e2e:
    entry['e2e'] = e2e_crps(h, x, t)
  return entry


def e2e_crps(h, x, t):
  """The chunk through evaluation._metric_and_region_loop with the CRPS +
  spread / skill eval config on pinned-HOST datasets -> wb2_ens_metrics_host
  (204 B per grid point cross PCIe: this path is PCIe-bound by construction)."""
  from weatherbench2_b200 import config, evaluation, metrics
  from weatherbench2_b200 import xarray_lite as xl
  args, ctx = h.args, h.ctx
  nsteps = max(1, args.e2e_steps)
  hx = h.pinned_from(x.view(ENS_M, ENS_NVAR, NLEV, NLAT, NLON))
  ht = h.pinned_from(t.view(ENS_NVAR, NLEV, NLAT, NLON))
  lat, lon = _lat_lon()
  levels = np.array(LEVELS)
  names = VARIABLES[:ENS_NVAR]
  t0 = np.array(['2020-01-01T00'], dtype='datetime64[ns]')
  fdims = ('realization', 'time', 'level', 'latitude', 'longitude')
  tdims = ('time', 'level', 'latitude', 'longitude')
  coords = {'time': t0, 'level': levels, 'latitude': lat, 'longitude': lon}
  forecast = xl.Dataset({v: (fdims, hx[:, None, i]) for i, v in enumerate(names)},
                        dict(coords, realization=np.arange(ENS_M)))
  truth = xl.Dataset({v: (tdims, ht[None, i]) for i, v in enumerate(names)},
                     coords)
  eval_config = config.Eval(
      metrics={'crps': metrics.CRPS(), 'crps_spread': metrics.CRPSSpread(),
               'crps_skill': metrics.CRPSSkill(),
               'ensemble_mean_rmse': metrics.EnsembleMeanRMSESqrtBeforeTimeAvg(),
               'ensemble_stddev': metrics.EnsembleStddevSqrtBeforeTimeAvg()},
      temporal_mean=False)

  def one(_):
    return evaluation._metric_and_region_loop(  # pylint: disable=protected-access
        forecast, truth, eval_config, skipna=False, compute_chunk=True)

  one(0)
  ctx.reset_transfer_stats()
  dt, res, clocks = h.time_host(one, nsteps)
  st = ctx.transfer_stats()
  h.keep('crps_sweep.e2e', res)
  d2h = sum(res[v].values.nbytes for v in res.keys())
  h.free_pinned(hx, ht)
  points = ENS_FIELDS * SLAB
  return {'value': h.world * points * nsteps / dt,
          'unit': 'grid-points/s',
          'h2d_bytes_per_step': int(st['h2d_bytes'] // nsteps),
          'd2h_bytes_per_step': int(max(d2h, st['d2h_bytes'] // nsteps)),
          'steps': nsteps, 'ms_per_step': 1e3 * dt / nsteps, 'clocks': clocks,
          'pcie_gbs': st['h2d_bytes'] / dt / 1e9,
          'api': 'evaluation._metric_and_region_loop(CRPS, CRPSSpread, CRPSSkill, '
                 'EnsembleMeanRMSE, EnsembleStddev) on pinned-host datasets -> '
                 'wb2_ens_metrics_host (one pass for all five)'}


def bench_regrid(h):
  """configs[3]: ConservativeRegridder 0.25 -> 1.5 degree (K5)."""
  torch, ctx, args = h.torch, h.ctx, h.args
  from weatherbench2_b200 import regridding as rg
  lat, lon = _lat_lon()
  src = rg.Grid.from_degrees(lon, lat)
  tgt = rg.Grid.from_degrees(np.arange(RG_TLON) * 1.5,
                             np.linspace(-90, 90, RG_TLAT))
  regridder = rg.ConservativeRegridder(src, tgt)
  gen = torch.Generator(device=h.dev)
  gen.manual_seed(802703 + h.rank)
  # the reference's layout: (..., lon, lat), latitude contiguous
  x = torch.randn((RG_FIELDS, NLON, NLAT), device=h.dev, dtype=torch.float32,
                  generator=gen)
  out = torch.empty((RG_FIELDS, RG_TLON, RG_TLAT), device=h.dev,
                    dtype=torch.float32)

  def step(_):
    regridder.regrid_device(ctx, x.data_ptr(), out.data_ptr(), RG_FIELDS)

  ms_total, ms_kernels, launches, clocks = h.time_steps(
      step, lambda warm: None, args.steps, args.warmup)
  cells = RG_FIELDS * SLAB
  assert bool(torch.isfinite(out).all().item())
  h.keep('regrid.out', out)
  entry = {
      'workload': f'configs[3]: ConservativeRegridder 0.25 -> 1.5 degree '
                  f'({NLAT}x{NLON} -> {RG_TLAT}x{RG_TLON}), 6 vars x 37 levels per '
                  f'time step ({RG_FIELDS} fields, 0.92 GB f32 per step per GPU; '
                  'no collective: outputs stay time-sharded)',
      'value': h.world * cells * args.steps / (ms_total * 1e-3),
      'unit': 'source grid-cells/s', 'ms_per_step': ms_total / args.steps,
      'scaling': 'weak', 'gpu_launches': launches, 'clocks': clocks,
      'l2_policy': 'input 0.92 GB per step >> L2 (126 MB)',
      'roofline': h.roofline('regrid', 'regrid_kernel (banded 7x7 stencil)',
                             cells * RG_BYTES_PER_CELL, ms_kernels / args.steps),
  }
  if not args.no_e2e:
    nsteps = max(1, args.e2e_steps)
    hx = h.pinned_from(x)
    # warm-up; two results alive at once, so that the pinned result pool holds
    # the two buffers a loop `out = f()` alternates between
    w1 = regridder.regrid_array(hx)
    w2 = regridder.regrid_array(hx)
    del w1, w2
    ctx.reset_transfer_stats()
    dt, res, eclocks = h.time_host(lambda _: regridder.regrid_array(hx), nsteps)
    st = ctx.transfer_stats()
    assert res.shape == (RG_FIELDS, RG_TLON, RG_TLAT)
    h.keep('regrid.e2e', res)
    h.free_pinned(hx)
    entry['e2e'] = {
        'value': h.world * cells * nsteps / dt, 'unit': 'source grid-cells/s',
        'h2d_bytes_per_step': int(st['h2d_bytes'] // nsteps),
        'd2h_bytes_per_step': int(st['d2h_bytes'] // nsteps), 'steps': nsteps,
        'ms_per_step': 1e3 * dt / nsteps, 'clocks': eclocks,
        'pcie_gbs': st['h2d_bytes'] / dt / 1e9,
        'api': 'ConservativeRegridder.regrid_array(pinned-host array) -> '
               'wb2_regrid_conservative_host (result to pageable host memory)'}
  return entry


def bench_spectrum(h):
  """configs[4]: ZonalEnergySpectrum with the script's time mean fused in (K4),
  plus the north-star variant with the latitude-weighted reduction fused."""
  torch, ctx, args = h.torch, h.ctx, h.args
  from weatherbench2_b200 import derived_variables as dvs
  from weatherbench2_b200 import _spatial as sp
  gen = torch.Generator(device=h.dev)
  gen.manual_seed(802704 + h.rank)
  nfield = SP_TIMES * SP_SLOTS
  x = torch.randn((nfield, NLAT, NLON), device=h.dev, dtype=torch.float32,
                  generator=gen)
  lat, lon = _lat_lon()
  circ = dvs.ZonalEnergySpectrum('u')._circumference(lat)  # pylint: disable=protected-access
  acc = torch.zeros((SP_SLOTS, NLAT, SP_NK), device=h.dev, dtype=torch.float32)
  red = torch.zeros((SP_SLOTS, SP_NK), device=h.dev, dtype=torch.float32)
  w = sp.lat_weights(lat)
  scale_red = circ * w / w.sum()

  def step(_):
    ctx.zonal_spectrum(x.data_ptr(), nfield, NLAT, NLON, circ, acc.data_ptr(),
                       True, SP_SLOTS)

  def tail(warm):
    del warm
    if h.world > 1:  # xbeam.Mean(['time']) across ranks: one 385 MB all-reduce
      h.dist.all_reduce(acc)

  ms_total, ms_kernels, launches, clocks = h.time_steps(step, tail, args.steps,
                                                        args.warmup)
  cells = nfield * SLAB
  assert bool(torch.isfinite(acc).all().item())
  h.keep('spectrum_sweep.time_sum', acc)
  entry = {
      'workload': f'configs[4]: zonal energy spectrum, rFFT along lon={NLON}, 37 '
                  f'levels x 5 vars, {SP_TIMES} time steps per launch '
                  f'({nfield} fields, 12.3 GB f32 per step per GPU), time mean '
                  'fused in; at N > 1 one 385 MB NCCL all-reduce of the time sum '
                  'at the end',
      'value': h.world * cells * args.steps / (ms_total * 1e-3),
      'unit': 'grid-cells/s', 'ms_per_step': ms_total / args.steps,
      'scaling': 'weak', 'gpu_launches': launches, 'clocks': clocks,
      'roofline': h.roofline(
          'spectrum_sweep', 'spectrum_pfa_kernel<9x16x5, time-sum> (packed f32x2 '
          'prime-factor FFT, TMA-staged rows)', cells * 4, ms_kernels / args.steps),
  }

  def step_red(_):
    ctx.zonal_spectrum_latsum(x.data_ptr(), nfield, NLAT, NLON, scale_red,
                              red.data_ptr(), SP_SLOTS)

  def tail_red(warm):
    del warm
    if h.world > 1:
      h.dist.all_reduce(red)

  ms_total, ms_kernels, launches, rclocks = h.time_steps(
      step_red, tail_red, args.steps, args.warmup)
  h.keep('spectrum_sweep.latsum', red)
  entry['latsum'] = {
      'what': 'north-star variant: rFFT + power + latitude-weighted meridional '
              'reduction (get_lat_weights) + time mean fused, nothing per-latitude '
              'is written',
      'value': h.world * cells * args.steps / (ms_total * 1e-3),
      'unit': 'grid-cells/s', 'ms_per_step': ms_total / args.steps,
      'gpu_launches': launches, 'clocks': rclocks,
      'roofline': h.roofline('spectrum_latsum', 'spectrum_pfa_kernel<9x16x5, '
                             'latsum> + finalize', cells * 4,
                             ms_kernels / args.steps)}
  if not args.no_e2e:
    from weatherbench2_b200 import xarray_lite as xl
    nsteps = max(1, args.e2e_steps)
    hx = h.pinned_from(x.view(SP_TIMES, SP_SLOTS, NLAT, NLON))
    ds = xl.Dataset(
        {'u': (('time', 'level_var', 'latitude', 'longitude'), hx)},
        {'time': np.arange(SP_TIMES), 'level_var': np.arange(SP_SLOTS),
         'latitude': lat, 'longitude': lon})
    op = dvs.ZonalEnergySpectrum('u')
    w1 = op.compute(ds, time_sum_dim='time')  # warm-up (see bench_regrid)
    w2 = op.compute(ds, time_sum_dim='time')
    del w1, w2
    ctx.reset_transfer_stats()
    dt, res, eclocks = h.time_host(
        lambda _: op.compute(ds, time_sum_dim='time'), nsteps)
    st = ctx.transfer_stats()
    assert res.shape == (SP_SLOTS, NLAT, SP_NK)
    h.keep('spectrum_sweep.e2e', res)
    h.free_pinned(hx)
    entry['e2e'] = {
        'value': h.world * cells * nsteps / dt, 'unit': 'grid-cells/s',
        'h2d_bytes_per_step': int(st['h2d_bytes'] // nsteps),
        'd2h_bytes_per_step': int(st['d2h_bytes'] // nsteps), 'steps': nsteps,
        'ms_per_step': 1e3 * dt / nsteps, 'clocks': eclocks,
        'pcie_gbs': st['h2d_bytes'] / dt / 1e9,
        'api': "ZonalEnergySpectrum('u').compute(pinned-host dataset, "
               "time_sum_dim='time') -> wb2_zonal_spectrum_host (accumulator in "
               'HBM, only the time sum comes back)'}
  return entry


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=20)
  ap.add_argument('--warmup', type=int, default=3)
  ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
  ap.add_argument('--e2e-steps', type=int, default=3)
  ap.add_argument('--no-e2e', action='store_true')
  ap.add_argument('--no-cpu', action='store_true')
  ap.add_argument('--workloads', default='crps,regrid,spectrum',
                  help='comma-separated subset of crps,regrid,spectrum (the '
                       'configs[1] line always runs); "none" skips them')
  ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                  help='after the timed steps, write what each timed path '
                       'returned in its last step as DIR/<name>.npy (rank 0; '
                       'outputs above 2**20 elements as a fixed, seeded '
                       'sample; at most 64 MB in all)')
  args = ap.parse_args()
  if args.impl == 'reference':
    run_reference(args)
    return
  args.warmup = max(args.warmup, 3)
  h = Harness(args)
  torch = h.torch
  line = bench_rmse_acc(h)
  torch.cuda.empty_cache()
  wanted = [] if args.workloads == 'none' else args.workloads.split(',')
  workloads = {}
  for key, name, fn in (('crps', 'crps_sweep', bench_crps),
                        ('regrid', 'regrid', bench_regrid),
                        ('spectrum', 'spectrum_sweep', bench_spectrum)):
    if key in wanted:
      if h.world == 1:
        try:
          workloads[name] = fn(h)
        except Exception as e:  # pylint: disable=broad-except
          # a failed workload must not take the contract line with it (under
          # torchrun an exception ends the job anyway: ranks meet in collectives)
          workloads[name] = {'error': f'{type(e).__name__}: {e}'[:400]}
      else:
        workloads[name] = fn(h)
      torch.cuda.empty_cache()
  line['workloads'] = workloads
  if h.rank == 0 and not args.no_cpu:
    line['cpu_baseline'] = cpu_baseline_single('rmse_acc')
    for key, name in (('crps', 'crps_sweep'), ('regrid', 'regrid'),
                      ('spectrum', 'spectrum_sweep')):
      if name in workloads:
        workloads[name]['cpu_baseline'] = cpu_baseline_single(key, reps=2)
    line['cpu_baseline']['host'] = usable_cores()[1]
  if h.rank == 0:
    if args.dump_outputs:
      h.dump_outputs(args.dump_outputs)
    print(json.dumps(line))
  if h.world > 1:
    h.dist.destroy_process_group()


if __name__ == '__main__':
  main()
