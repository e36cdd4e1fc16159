"""Multi-GPU evaluation: chunks of init times are sharded over the ranks of a
`torch.distributed` process group (one process per GPU) and the time mean is
formed with ONE all-reduce of [sum, count] at the end.

This replaces the Beam pipeline of the reference for the hot path
(weatherbench2/evaluation.py:693-744): `xbeam.DatasetToChunks` -> rank-local
chunk loop, `EvaluateChunk` -> `_metric_and_region_loop(compute_chunk=True)`,
`xbeam.Mean(dim, skipna)` -> all-reduce(sum) of per-rank partial sums and
counts.  Chunks are independent (no data-path collective); the payload of the
reduce is a few KB.
"""
from __future__ import annotations

import typing as t

import numpy as np

from weatherbench2_b200 import xarray_lite as xl


def shard_indices(n: int, rank: int, world: int) -> np.ndarray:
  """Contiguous, balanced block of chunk indices owned by `rank`."""
  per, extra = divmod(n, world)
  start = rank * per + min(rank, extra)
  return np.arange(start, start + per + (1 if rank < extra else 0))


def _dist():
  import torch.distributed as dist  # pylint: disable=import-outside-toplevel
  return dist


def _nccl_device(device=None):
  """The CUDA device this rank's collectives run on: the caller's choice, else
  the device of the rank's wb2 context (LOCAL_RANK) -- NOT torch's current
  device, which is cuda:0 on every rank unless the launcher set it."""
  import torch  # pylint: disable=import-outside-toplevel
  if device is not None:
    return torch.device(device)
  from weatherbench2_b200 import _lib  # pylint: disable=import-outside-toplevel
  return torch.device('cuda', _lib.default_context().device)


def all_reduce_sum(arrays: list, group=None, device=None) -> list:
  """Sum-all-reduce a list of float64 NumPy arrays in one collective.
  NCCL needs device tensors; gloo (CPU tests) takes host tensors."""
  import torch  # pylint: disable=import-outside-toplevel
  dist = _dist()
  if not (dist.is_available() and dist.is_initialized()):
    return arrays
  flat = np.concatenate([np.asarray(a, dtype=np.float64).ravel()
                         for a in arrays]) if arrays else np.zeros(0)
  backend = dist.get_backend(group)
  tensor = torch.from_numpy(flat.copy())
  if backend == 'nccl':
    tensor = tensor.to(_nccl_device(device))
  dist.all_reduce(tensor, op=dist.ReduceOp.SUM, group=group)
  flat = tensor.cpu().numpy()
  out, pos = [], 0
  for a in arrays:
    n = int(np.prod(np.shape(a))) if np.shape(a) else 1
    out.append(flat[pos:pos + n].reshape(np.shape(a)))
    pos += n
  return out


class TimeMeanAccumulator:
  """Accumulates per-chunk results along `avg_dim` as (sum, count) so that
  mean(dim, skipna) can be finished after a cross-rank reduction
  (weatherbench2/metrics.py:133-138 semantics: NaN propagates unless skipna).
  """

  def __init__(self, avg_dim: str, skipna: bool):
    self.avg_dim = avg_dim
    self.skipna = skipna
    self.sums: dict = {}
    self.counts: dict = {}
    self.meta: dict = {}

  def add(self, chunk: xl.Dataset):
    for name in chunk.keys():
      da = chunk[name]
      if self.avg_dim not in da.dims:
        raise ValueError(f'{name} has no {self.avg_dim!r} dimension')
      ax = da.dims.index(self.avg_dim)
      v = da.values.astype(np.float64)
      if self.skipna:
        ok = ~np.isnan(v)
        s = np.where(ok, v, 0.0).sum(axis=ax)
        c = ok.sum(axis=ax).astype(np.float64)
      else:
        s = v.sum(axis=ax)
        c = np.full(s.shape, v.shape[ax], dtype=np.float64)
      if name in self.sums:
        self.sums[name] = self.sums[name] + s
        self.counts[name] = self.counts[name] + c
      else:
        self.sums[name] = s
        self.counts[name] = c
        dims = tuple(d for d in da.dims if d != self.avg_dim)
        coords = {k: cc for k, cc in da.coords.items()
                  if all(d in dims for d in cc.dims)}
        self.meta[name] = (dims, coords)

  def finish(self, group=None, device=None) -> xl.Dataset:
    names = sorted(self.sums)
    reduced = all_reduce_sum([self.sums[n] for n in names] +
                             [self.counts[n] for n in names], group, device)
    out = xl.Dataset()
    k = len(names)
    for i, n in enumerate(names):
      s, c = reduced[i], reduced[k + i]
      with np.errstate(invalid='ignore', divide='ignore'):
        mean = np.where(c > 0, s / np.where(c > 0, c, 1.0), np.nan)
      dims, coords = self.meta[n]
      out[n] = xl.DataArray(mean, dims, coords, n)
    return out


def _gather_chunks(per_chunk: list, indices: list, chunk_dim: str, world: int,
                   group=None, device=None) -> xl.Dataset:
  """All ranks' per-chunk results, concatenated along `chunk_dim` in chunk
  order (the un-reduced output of the reference's pipeline when
  `temporal_mean=False`).  Variables without `chunk_dim` (it was averaged or
  never present) are taken from the first chunk."""
  pairs = list(zip(indices, per_chunk))
  if world > 1:
    dist = _dist()
    payload = [(i, {k: (ds[k].dims, ds[k].values) for k in ds.keys()},
                {k: (c.dims, c.values) for k, c in ds.coords.items()})
               for i, ds in pairs]
    gathered = [None] * world
    if dist.get_backend(group) == 'nccl':
      import torch  # pylint: disable=import-outside-toplevel
      # all_gather_object stages the pickles on torch's CURRENT device
      with torch.cuda.device(_nccl_device(device)):
        dist.all_gather_object(gathered, payload, group=group)
    else:
      dist.all_gather_object(gathered, payload, group=group)
    pairs = []
    for part in gathered:
      for i, data_vars, coords in part:
        pairs.append((i, xl.Dataset(data_vars, coords)))
  pairs.sort(key=lambda p: p[0])
  if not pairs:
    return xl.Dataset()
  parts = [ds for _, ds in pairs]
  if all(chunk_dim in parts[0][k].dims for k in parts[0].keys()):
    return xl.concat(parts, chunk_dim)
  out = xl.Dataset(attrs=parts[0].attrs)
  for k in parts[0].keys():
    if chunk_dim in parts[0][k].dims:
      out[k] = xl.concat([xl.Dataset({k: p[k]}) for p in parts], chunk_dim)[k]
    else:
      out[k] = parts[0][k]
  return out


def _truth_for_chunk(truth, fc, chunk_dim, select_truth):
  """Truth of one forecast chunk.  By-valid chunks (`chunk_dim == 'time'`) are
  aligned BY LABEL like the reference's xarray arithmetic -- the truth record
  may be longer than the forecast's or start elsewhere -- never by position;
  forecast times without a truth label raise KeyError (an inner join would
  silently shorten the time mean).

  The by-valid truth is a lazily gathered view of the truth record, not a
  per-chunk copy: the slab cache keys truth slabs by host address, and a copy
  freed after one chunk can be reallocated at the same address for the next
  one with other contents."""
  tr = select_truth(truth, fc)
  if chunk_dim == 'time' and 'time' in truth.dims and 'time' in fc.coords:
    times = fc.coords['time'].values
    pos = xl._lookup(truth.coords['time'].values, times)  # pylint: disable=protected-access
    tr = xl.Dataset(attrs=truth.attrs)
    for k in truth.keys():
      v = truth[k]
      tr[k] = v if 'time' not in v.dims else xl.LazyGather(
          v, {'time': (('time',), pos)},
          extra_coords={'time': xl.Coord(('time',), times)})
  return tr


def evaluate_sharded(forecast: xl.Dataset, truth: xl.Dataset, eval_config,
                     skipna: bool = False, chunk_dim: str = 'init_time',
                     chunk_size: int = 1, group=None, device=None,
                     loop_fn: t.Optional[t.Callable] = None,
                     select_truth: t.Optional[t.Callable] = None,
                     prefetch: int = 0, num_threads: int = 2,
                     temporal_mean: bool = True) -> xl.Dataset:
  """Time-mean metric results with the chunks of `chunk_dim` sharded over the
  process group.  Every rank returns the full (identical) result.

  forecast: by-init forecast (dims init_time, lead_time, ...) with a
    `valid_time` coordinate (evaluation.apply_time_conventions), or a by-valid
    one with `time`; truth: dataset with a `time` dimension.
  loop_fn / select_truth are injectable for tests; they default to
  evaluation._metric_and_region_loop and
  evaluation.select_truth_at_valid_time.
  prefetch > 0: this rank's forecast chunks come from a feeder.ChunkFeeder that
  reads `prefetch` chunks ahead into pinned host buffers with `num_threads`
  reader threads (the DatasetToChunks replacement, evaluation.py:693-705), so
  the read of chunk i+1 overlaps the kernels of chunk i and the H2D copies run
  at the PCIe rate.
  temporal_mean=False (config.Eval.temporal_mean, evaluation.py:733-744): no
  reduction -- the per-chunk results are gathered from all ranks and
  concatenated along `chunk_dim` in chunk order.
  """
  from weatherbench2_b200 import evaluation  # pylint: disable=import-outside-toplevel
  dist = _dist()
  if dist.is_available() and dist.is_initialized():
    rank, world = dist.get_rank(group), dist.get_world_size(group)
  else:
    rank, world = 0, 1
  cache_scope = None
  if loop_fn is None:
    # product path: keep the truth / climatology slabs that repeat from chunk
    # to chunk resident in HBM for the duration of the sweep (host inputs only;
    # the datasets are not modified while we hold them)
    from weatherbench2_b200 import _lib  # pylint: disable=import-outside-toplevel
    cache_scope = _lib.default_context().slab_cache()
  loop_fn = loop_fn or evaluation._metric_and_region_loop  # pylint: disable=protected-access
  if select_truth is None:
    select_truth = (evaluation.select_truth_at_valid_time
                    if chunk_dim == 'init_time' else (lambda tr, fc: tr))
  n = forecast.sizes[chunk_dim]
  nchunks = (n + chunk_size - 1) // chunk_size
  acc = TimeMeanAccumulator(chunk_dim, skipna)
  import contextlib  # pylint: disable=import-outside-toplevel
  mine = [int(ci) for ci in shard_indices(nchunks, rank, world)]
  if prefetch > 0:
    from weatherbench2_b200 import feeder  # pylint: disable=import-outside-toplevel
    chunks = (c for _, c in feeder.ChunkFeeder(
        forecast, chunk_dim, chunk_size, indices=mine, depth=prefetch,
        num_threads=num_threads, pin=cache_scope is not None))
  else:
    chunks = (forecast.isel({chunk_dim: slice(
        ci * chunk_size, min(n, (ci + 1) * chunk_size))}) for ci in mine)
  per_chunk = []
  with (cache_scope if cache_scope is not None else contextlib.nullcontext()):
    for fc in chunks:
      tr = _truth_for_chunk(truth, fc, chunk_dim, select_truth)
      res = loop_fn(fc, tr, eval_config, skipna=skipna, compute_chunk=True)
      if temporal_mean:
        acc.add(res)
      else:
        per_chunk.append(xl.from_xarray(res))
  if not temporal_mean:
    return _gather_chunks(per_chunk, mine, chunk_dim, world, group, device)
  if not acc.sums:
    # a rank without chunks still has to take part in the collective with the
    # right payload shape: evaluate nothing, contribute zeros
    fc = forecast.isel({chunk_dim: slice(0, 1)})
    tr = _truth_for_chunk(truth, fc, chunk_dim, select_truth)
    probe = loop_fn(fc, tr, eval_config, skipna=skipna, compute_chunk=True)
    acc.add(probe)
    for k in acc.sums:
      acc.sums[k] = np.zeros_like(acc.sums[k])
      acc.counts[k] = np.zeros_like(acc.counts[k])
  return acc.finish(group, device)
