"""TEST INFRASTRUCTURE: a NumPy stand-in for `_lib.Context` that lets the CPU
suite drive the Python operator layer end to end (evaluate_in_memory ->
_metric_and_region_loop -> metrics.batch -> _spatial.run_* -> C ABI call)
without a GPU.

It interprets the SAME raw arguments the operators hand to the C ABI -- base
addresses, element-offset tables, the wb2_weights factorisation, member strides
-- by reading host memory at those addresses, and produces the raw statistics
`include/wb2b200.h` documents.  What it checks is therefore the host logic
(offset tables, gathers, region factors, result assembly); the arithmetic of
the CUDA kernels is checked by the `-m gpu` tests against the oracle.  It is
never importable from the package: the product has no CPU path.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import hashlib

import numpy as np

from weatherbench2_b200 import _lib


def _view(addr: int, n: int, dtype) -> np.ndarray:
  dtype = np.dtype(dtype)
  buf = (C.c_char * (n * dtype.itemsize)).from_address(int(addr))
  return np.frombuffer(buf, dtype=dtype, count=n)


def _slab(base: int, off: int, w: _lib.WeightSpec, dtype,
          native: bool = False) -> np.ndarray:
  es = np.dtype(dtype).itemsize
  span = (w.nrow - 1) * w.row_stride + w.ncol
  flat = _view(base + int(off) * es, span, dtype)
  rows = np.lib.stride_tricks.as_strided(
      flat, shape=(w.nrow, w.ncol), strides=(w.row_stride * es, es),
      writeable=False)
  return rows.copy() if native else rows.astype(np.float64)


class FakeContext:
  """'Device' memory is host memory; compute entries are NumPy."""

  def __init__(self):
    self._bufs: dict = {}
    self.calls: list = []
    self.h2d_bytes = 0
    self._cached = None  # host address -> digest of the slab, in slab_cache()

  # -- memory -------------------------------------------------------------------
  def malloc(self, nbytes: int) -> int:
    buf = np.zeros(max(int(nbytes), 8), dtype=np.uint8)
    self._bufs[buf.ctypes.data] = buf
    return buf.ctypes.data

  def free(self, ptr) -> None:
    self._bufs.pop(int(ptr), None)

  def to_device(self, arr: np.ndarray) -> int:
    arr = np.ascontiguousarray(arr)
    ptr = self.malloc(arr.nbytes)
    _view(ptr, arr.nbytes, np.uint8)[...] = arr.view(np.uint8).reshape(-1)
    self.h2d_bytes += arr.nbytes
    return ptr

  def from_device(self, ptr, shape, dtype) -> np.ndarray:
    n = int(np.prod(shape)) if len(shape) else 1
    return _view(ptr, n, dtype).reshape(shape).copy()

  def synchronize(self) -> None:
    pass

  @property
  def launch_count(self) -> int:
    """Kernel launches the real library makes for the calls so far (the GPU
    tests assert 'ONE pass serves all metrics / regions' through it): reduction
    entries = main kernel + finalize, the threshold entry passes of 4 / 2 / 1
    thresholds + finalize, map entries one kernel."""
    n = 0
    for call in self.calls:
      if call[0] in ('det_metrics', 'det_metrics_vector', 'ens_metrics',
                     'energy_score', 'gaussian_metrics'):
        n += 2
      elif call[0] == 'ens_threshold_metrics':
        nq = call[2]  # passes of 4, then 2, then 1 thresholds; + finalize
        n += nq // 4 + (nq % 4 >= 2) + nq % 2 + 1
      else:
        n += 1
    return n

  @contextlib.contextmanager
  def slab_cache(self, nbytes=None):
    """Holds the library's slab-cache contract: the truth / climatology slabs
    a *_host entry reads are keyed by host address, so an address that comes
    back with other contents inside the scope (a freed per-chunk copy
    reallocated in place) would be served stale by the library.  Re-entrant,
    like Context.slab_cache."""
    del nbytes
    if self._cached is not None:
      yield self
      return
    self._cached = {}
    try:
      yield self
    finally:
      self._cached = None

  def _check_cached(self, base, offs, w, dtype):
    if self._cached is None:
      return
    es = np.dtype(dtype).itemsize
    for off in offs:
      addr = base + int(off) * es
      digest = hashlib.blake2b(
          _slab(base, off, w, dtype, native=True).tobytes()).digest()
      assert self._cached.setdefault(addr, digest) == digest, (
          f'slab cache: host address {addr:#x} reused with other contents')

  def pinned_result(self, shape, dtype):
    return np.empty(shape, dtype=dtype)

  # -- weights ------------------------------------------------------------------
  def _weights(self, w: _lib.WeightSpec) -> np.ndarray:
    """W[r, row, col] exactly as the header defines it."""
    seg_of_col = np.zeros(w.ncol, dtype=int)
    for k in range(w.nseg):
      seg_of_col[w.seg_start[k]:w.seg_start[k + 1]] = k
    colw = (np.ones(w.ncol) if w.col_w is None
            else w.col_w.astype(np.float64))
    out = (w.row_w[:, :, None] * w.seg_w[:, seg_of_col][:, None, :] *
           colw[None, None, :])
    if w.cell_w_dev:
      cell = _view(w.cell_w_dev, w.nrow * w.ncol, np.float32).reshape(
          w.nrow, w.ncol).astype(np.float64)
      out = out * cell[None]
    return out

  @staticmethod
  def _wsum(W, value, skipna, zero_skip):
    """(sum W*value, sum W*[valid]) with the skipna / where(w>0, 0) rules."""
    if zero_skip:
      value = np.where(W > 0, value, 0.0)
    valid = ~np.isnan(value)
    if skipna:
      return (np.where(valid, value, 0.0) * W).sum(), (W * valid).sum()
    return (value * W).sum(), W.sum()

  # -- K1 -----------------------------------------------------------------------
  def det_metrics(self, f, t, c, dtype, off_f, off_t, off_c, weights, skipna,
                  out, host=False):
    self.calls.append(('det_metrics', int(off_f.size), weights.nregion, host))
    dt = np.float32 if dtype == _lib.F32 else np.float64
    if host:
      self._check_cached(t, off_t, weights, dt)
      if c:
        self._check_cached(c, off_c, weights, dt)
    W = self._weights(weights)
    res = np.zeros((off_f.size, weights.nregion, _lib.DET_NSTAT))
    for i in range(off_f.size):
      fs = _slab(f, off_f[i], weights, dt)
      ts = _slab(t, off_t[i], weights, dt)
      with np.errstate(invalid='ignore'):  # inf - inf in masked-out cells
        d = fs - ts
      vals = [d * d, np.abs(d), d]
      if c:
        cs = _slab(c, off_c[i], weights, dt)
        fa, ta = fs - cs, ts - cs
        vals += [fa * ta, fa * fa, ta * ta]
      for r in range(weights.nregion):
        zs = weights.zero_skip
        for k, v in enumerate(vals):
          s, ws = self._wsum(W[r], v, skipna, zs)
          res[i, r, k] = s
          if k == 0:
            res[i, r, 6] = ws
          elif k == 3:
            res[i, r, 7] = ws
          elif k == 4:
            res[i, r, 8] = ws
          elif k == 5:
            res[i, r, 9] = ws
    _view(out, res.size, np.float64)[...] = res.reshape(-1)

  # -- K2 -----------------------------------------------------------------------
  def ens_metrics(self, x, t, dtype, nmember, member_stride, off_x, off_t,
                  weights, skipna, out):
    self.calls.append(('ens_metrics', int(off_x.size), weights.nregion))
    dt = np.float32 if dtype == _lib.F32 else np.float64
    W = self._weights(weights)
    M = int(nmember)
    res = np.zeros((off_x.size, weights.nregion, _lib.ENS_NSTAT))
    for i in range(off_x.size):
      skill, spread, mse, var, deb = self._ens_point(
          x, t, dt, M, member_stride, off_x[i], off_t[i], weights, skipna)
      for r in range(weights.nregion):
        for k, v in enumerate([skill, spread, mse, var, deb]):
          s, ws = self._wsum(W[r], v, skipna, weights.zero_skip)
          res[i, r, k] = s
          res[i, r, 5 + k] = ws
    _view(out, res.size, np.float64)[...] = res.reshape(-1)

  @staticmethod
  def _ens_point(x, t, dt, M, member_stride, off_x, off_t, geometry, skipna):
    """The five point-wise statistics of WB2_ENS_NSTAT's list."""
    es = np.dtype(dt).itemsize
    mean_fn = np.nanmean if skipna else np.mean
    xs = np.stack([_slab(x + m * member_stride * es, off_x, geometry, dt)
                   for m in range(M)])
    ts = _slab(t, off_t, geometry, dt)
    with np.errstate(invalid='ignore'), _quiet():
      skill = mean_fn(np.abs(ts[None] - xs), axis=0)
      if M < 2:
        spread = np.zeros_like(ts)
      else:
        order = np.sort(xs, axis=0)  # NaN last, like np.argsort
        rank = np.arange(1, M + 1, dtype=np.float64)[:, None, None]
        if skipna:
          n = (~np.isnan(xs)).sum(axis=0).astype(np.float64)
          spread = 2.0 * np.nansum((2 * rank - M - 1) * order, axis=0) / np.where(
              n > 0, n, np.nan) / (M - 1)
        else:
          spread = 2.0 * ((2 * rank - M - 1) * order).mean(axis=0) / (M - 1)
      xbar = mean_fn(xs, axis=0)
      mse = (ts - xbar) ** 2
      if M > 1:
        var = (np.nanvar if skipna else np.var)(xs, axis=0, ddof=1)
      else:
        var = np.full_like(ts, np.nan)
      deb = mse - var / M
    return [skill, spread, mse, var, deb]

  def ens_metrics_host(self, x, t, nmember, member_stride, off_x, off_t,
                       weights, skipna, out):
    self._check_cached(t, off_t, weights, np.float32)
    self.ens_metrics(x, t, _lib.F32, nmember, member_stride, off_x, off_t,
                     weights, skipna, out)

  def det_metrics_vector(self, fu, fv, tu, tv, dtype, off_fu, off_fv, off_tu,
                         off_tv, weights, skipna, out):
    self.calls.append(('det_metrics_vector', int(off_fu.size), weights.nregion))
    dt = np.float32 if dtype == _lib.F32 else np.float64
    W = self._weights(weights)
    res = np.zeros((off_fu.size, weights.nregion, _lib.DET_NSTAT))
    for i in range(off_fu.size):
      du = _slab(fu, off_fu[i], weights, dt) - _slab(tu, off_tu[i], weights, dt)
      dv = _slab(fv, off_fv[i], weights, dt) - _slab(tv, off_tv[i], weights, dt)
      for r in range(weights.nregion):
        res[i, r, 0], res[i, r, 6] = self._wsum(W[r], du * du + dv * dv, skipna,
                                                weights.zero_skip)
    _view(out, res.size, np.float64)[...] = res.reshape(-1)

  # -- K3 -----------------------------------------------------------------------
  def energy_score(self, x, t, dtype, nmember, member_stride, off_x, off_t,
                   weights, out):
    self.calls.append(('energy_score', int(off_x.size), weights.nregion))
    dt = np.float32 if dtype == _lib.F32 else np.float64
    es = np.dtype(dt).itemsize
    W = self._weights(weights)
    M = int(nmember)
    res = np.zeros((off_x.size, weights.nregion, 4, M))
    for i in range(off_x.size):
      xs = [_slab(x + m * member_stride * es, off_x[i], weights, dt)
            for m in range(M)]
      ts = _slab(t, off_t[i], weights, dt)
      for r in range(weights.nregion):
        for m in range(M):
          res[i, r, 0, m], res[i, r, 2, m] = self._wsum(
              W[r], (xs[m] - ts) ** 2, False, weights.zero_skip)
          if m < M - 1:
            res[i, r, 1, m], res[i, r, 3, m] = self._wsum(
                W[r], (xs[m] - xs[m + 1]) ** 2, False, weights.zero_skip)
    _view(out, res.size, np.float64)[...] = res.reshape(-1)

  # -- K6 / K6e -----------------------------------------------------------------
  @staticmethod
  def _geometry(nrow, ncol, row_stride):
    return _lib.WeightSpec(nrow, ncol, np.ones((1, nrow)), [0, ncol],
                           np.ones((1, 1)), row_stride=row_stride)

  def det_maps(self, f, t, dtype, stat, nout, ngroup, off_f, off_t, nrow, ncol,
               row_stride, skipna, out):
    self.calls.append(('det_maps', int(nout), int(ngroup)))
    dt = np.float32 if dtype == _lib.F32 else np.float64
    g = self._geometry(nrow, ncol, row_stride)
    res = np.empty((nout, nrow, ncol), dtype=dt)
    for j in range(nout):
      terms = []
      for k in range(ngroup):
        # the kernel forms the point-wise term in the input precision
        d = (_slab(f, off_f[j * ngroup + k], g, dt, native=True) -
             _slab(t, off_t[j * ngroup + k], g, dt, native=True))
        terms.append([d, d * d, np.abs(d)][stat].astype(np.float64))
      with _quiet():
        res[j] = (np.nanmean if skipna else np.mean)(np.stack(terms), axis=0)
    _view(out, res.size, dt)[...] = res.reshape(-1)

  def ens_maps(self, x, t, dtype, nmember, member_stride, nout, ngroup, off_x,
               off_t, nrow, ncol, row_stride, stat_mask, skipna, out):
    self.calls.append(('ens_maps', int(nout), int(ngroup), int(stat_mask)))
    dt = np.float32 if dtype == _lib.F32 else np.float64
    g = self._geometry(nrow, ncol, row_stride)
    sel = [b for b in range(6) if stat_mask >> b & 1]
    res = np.empty((len(sel), nout, nrow, ncol), dtype=np.float32)
    for j in range(nout):
      terms = []
      for k in range(ngroup):
        point = self._ens_point(x, t, dt, nmember, member_stride,
                                off_x[j * ngroup + k], off_t[j * ngroup + k], g,
                                skipna)
        point.append(point[0] - 0.5 * point[1])
        terms.append(np.stack([point[b] for b in sel]))
      with _quiet():
        res[:, j] = (np.nanmean if skipna else np.mean)(np.stack(terms), axis=0)
    _view(out, res.size, np.float32)[...] = res.reshape(-1)

  # -- K7: threshold / Gaussian metrics -------------------------------------------
  # (point-wise scores from the oracle: this stand-in checks the operand
  # staging, the threshold tables and the result assembly, not the arithmetic)
  @staticmethod
  def _threshold_fields(nthreshold, thr_a, off_a, thr_b, off_b, z, field, nfield,
                        g):
    out = []
    for k in range(nthreshold):
      if thr_b:
        mean = _slab(thr_a, off_a[field], g, np.float32)
        std = _slab(thr_b, off_b[field], g, np.float32)
        out.append(mean + np.float64(z[k]) * std)
      else:
        out.append(_slab(thr_a, np.asarray(off_a).reshape(
            nthreshold, nfield)[k, field], g, np.float32))
    return out

  @staticmethod
  def _ens_threshold_point(xs, ts, thr, skipna):
    from oracle import wb2_oracle as orc  # pylint: disable=import-outside-toplevel
    with np.errstate(invalid='ignore', divide='ignore'), _quiet():
      return [orc.ens_brier_pointwise(xs, ts, thr, 0, False, skipna),
              orc.ens_brier_pointwise(xs, ts, thr, 0, True, skipna),
              orc.ens_ignorance_pointwise(xs, ts, thr, 0, skipna),
              orc.ens_rps_part_pointwise(xs, ts, thr, 0, skipna)]

  def ens_threshold_metrics(self, x, t, nmember, member_stride, off_x, off_t,
                            nthreshold, thr_a, off_a, thr_b, off_b, z, weights,
                            skipna, out):
    self.calls.append(('ens_threshold_metrics', int(off_x.size), nthreshold))
    W = self._weights(weights)
    nfield = off_x.size
    res = np.zeros((nfield, nthreshold, weights.nregion, 8))
    for i in range(nfield):
      xs = np.stack([_slab(x + m * member_stride * 4, off_x[i], weights,
                           np.float32) for m in range(nmember)])
      ts = _slab(t, off_t[i], weights, np.float32)
      thrs = self._threshold_fields(nthreshold, thr_a, off_a, thr_b, off_b, z,
                                    i, nfield, weights)
      for k, thr in enumerate(thrs):
        for r in range(weights.nregion):
          for q, v in enumerate(self._ens_threshold_point(xs, ts, thr, skipna)):
            res[i, k, r, q], res[i, k, r, 4 + q] = self._wsum(
                W[r], v, skipna, weights.zero_skip)
    _view(out, res.size, np.float64)[...] = res.reshape(-1)

  def ens_threshold_maps(self, x, t, nmember, member_stride, nout, ngroup,
                         off_x, off_t, nthreshold, thr_a, off_a, thr_b, off_b,
                         z, nrow, ncol, row_stride, stat, skipna, out):
    self.calls.append(('ens_threshold_maps', int(nout), int(ngroup), stat))
    g = self._geometry(nrow, ncol, row_stride)
    nfield = nout * ngroup
    res = np.empty((nthreshold, nout, nrow, ncol), dtype=np.float32)
    for j in range(nout):
      terms = [[] for _ in range(nthreshold)]
      for q in range(ngroup):
        i = j * ngroup + q
        xs = np.stack([_slab(x + m * member_stride * 4, off_x[i], g, np.float32)
                       for m in range(nmember)])
        ts = _slab(t, off_t[i], g, np.float32)
        thrs = self._threshold_fields(nthreshold, thr_a, off_a, thr_b, off_b,
                                      z, i, nfield, g)
        for k, thr in enumerate(thrs):
          terms[k].append(self._ens_threshold_point(xs, ts, thr, skipna)[stat])
      with _quiet():
        for k in range(nthreshold):
          res[k, j] = (np.nanmean if skipna else np.mean)(np.stack(terms[k]),
                                                          axis=0)
    _view(out, res.size, np.float32)[...] = res.reshape(-1)

  def gaussian_metrics(self, mean, std, t, off_mean, off_std, off_t, nthreshold,
                       thr_a, off_a, thr_b, off_b, z, weights, skipna, out):
    from oracle import wb2_oracle as orc  # pylint: disable=import-outside-toplevel
    self.calls.append(('gaussian_metrics', int(off_mean.size), nthreshold))
    W = self._weights(weights)
    nfield = off_mean.size
    nt = max(nthreshold, 1)
    res = np.zeros((nfield, nt, weights.nregion, 8))
    for i in range(nfield):
      f = _slab(mean, off_mean[i], weights, np.float32)
      sd = _slab(std, off_std[i], weights, np.float32)
      ts = _slab(t, off_t[i], weights, np.float32)
      if nthreshold == 0:
        point = [{0: orc.gaussian_crps_pointwise(f, sd, ts), 1: sd * sd}]
      else:
        thrs = self._threshold_fields(nthreshold, thr_a, off_a, thr_b, off_b,
                                      z, i, nfield, weights)
        point = [{0: orc.gaussian_brier_pointwise(f, sd, ts, thr),
                  2: orc.gaussian_ignorance_pointwise(f, sd, ts, thr),
                  3: orc.gaussian_rps_part_pointwise(f, sd, ts, thr)}
                 for thr in thrs]
      for k, stats in enumerate(point):
        for r in range(weights.nregion):
          for q, v in stats.items():
            res[i, k, r, q], res[i, k, r, 4 + q] = self._wsum(
                W[r], v, skipna, weights.zero_skip)
    _view(out, res.size, np.float64)[...] = res.reshape(-1)

  # -- K9: SEEPS maps --------------------------------------------------------------
  def seeps_maps(self, f, t, wet, p1, nout, ngroup, off_f, off_t, off_wet_f,
                 off_wet_t, nrow, ncol, row_stride, wet_row_stride,
                 dry_threshold, min_p1, max_p1, skipna, out):
    from oracle import wb2_oracle as orc  # pylint: disable=import-outside-toplevel
    self.calls.append(('seeps_maps', int(nout), int(ngroup)))
    g = self._geometry(nrow, ncol, row_stride)
    gw = self._geometry(nrow, ncol, wet_row_stride)
    p1a = _view(p1, nrow * ncol, np.float32).reshape(nrow, ncol).astype(
        np.float64)
    res = np.empty((nout, nrow, ncol), dtype=np.float32)
    for j in range(nout):
      terms = []
      for q in range(ngroup):
        i = j * ngroup + q
        with _quiet():
          terms.append(orc.seeps_pointwise(
              _slab(f, off_f[i], g, np.float32),
              _slab(t, off_t[i], g, np.float32),
              _slab(wet, off_wet_f[i], gw, np.float32),
              _slab(wet, off_wet_t[i], gw, np.float32), p1a,
              float(dry_threshold) * 1000.0, float(min_p1), float(max_p1)))
      with _quiet():
        res[j] = (np.nanmean if skipna else np.mean)(np.stack(terms), axis=0)
    _view(out, res.size, np.float32)[...] = res.reshape(-1)

  # -- K10: rank histogram ------------------------------------------------------------
  def rank_histogram(self, x, t, nmember, member_stride, nout, ngroup, off_x,
                     off_t, nrow, ncol, row_stride, nbins, random_ties, seed,
                     out):
    self.calls.append(('rank_histogram', int(nout), int(ngroup), int(nbins)))
    g = self._geometry(nrow, ncol, row_stride)
    rs = np.random.RandomState(int(seed) % (2**32))
    width = (nmember + 1) // nbins
    res = np.zeros((nout, nrow, ncol, nbins), dtype=np.float32)
    for j in range(nout):
      for q in range(ngroup):
        i = j * ngroup + q
        xs = np.stack([_slab(x + m * member_stride * 4, off_x[i], g, np.float32)
                       for m in range(nmember)])
        ts = _slab(t, off_t[i], g, np.float32)
        with np.errstate(invalid='ignore'):
          # NaN sorts last: members that are NaN never precede the truth
          below = (xs < ts[None]).sum(axis=0)
          if np.isnan(ts).any():
            below = np.where(np.isnan(ts), (~np.isnan(xs)).sum(axis=0), below)
          equal = (xs == ts[None]).sum(axis=0)
        if random_ties:  # truth placed uniformly among the members equal to it
          below = below + (rs.rand(*below.shape) * (equal + 1)).astype(int)
        bins = below // width
        res[j] += np.eye(nbins, dtype=np.float32)[bins] / ngroup
    _view(out, res.size, np.float32)[...] = res.reshape(-1)

  # -- K5 / K8: regridding -----------------------------------------------------------
  @staticmethod
  def _dense(csr: _lib.CsrSpec) -> np.ndarray:
    w = np.zeros((csr.n_tgt, csr.n_src))
    for i in range(csr.n_tgt):
      lo, hi = csr.row_ptr[i], csr.row_ptr[i + 1]
      w[i, csr.col_idx[lo:hi]] = csr.val[lo:hi]
      if csr.nan_row[i]:
        w[i] = np.nan
    return w

  def regrid_conservative(self, src, dst, nfield, src_stride, dst_stride, lon_w,
                          lat_w):
    self.calls.append(('regrid_conservative', int(nfield)))
    wlon, wlat = self._dense(lon_w), self._dense(lat_w)
    ns = lon_w.n_src * lat_w.n_src
    nt = lon_w.n_tgt * lat_w.n_tgt
    for i in range(nfield):
      x = _view(src + i * src_stride * 4, ns, np.float32).reshape(
          lon_w.n_src, lat_w.n_src).astype(np.float64)
      ok = ~np.isnan(x)
      with np.errstate(invalid='ignore', divide='ignore'):
        num = np.einsum('ab,cd,bd->ac', wlon, wlat, np.where(ok, x, 0.0))
        den = np.einsum('ab,cd,bd->ac', wlon, wlat, ok.astype(np.float64))
        res = num / den
      _view(dst + i * dst_stride * 4, nt, np.float32)[...] = res.astype(
          np.float32).reshape(-1)

  def regrid_conservative_host(self, *args):
    self.regrid_conservative(*args)

  def regrid_gather(self, src, dst, nfield, src_stride, dst_stride, nsource,
                    indices):
    self.calls.append(('regrid_gather', int(nfield)))
    idx = np.asarray(indices)
    if idx.size and (idx.min() < 0 or idx.max() >= nsource):
      raise _lib.Wb2Error('wb2_regrid_gather: index out of range')
    for i in range(nfield):
      x = _view(src + i * src_stride * 4, nsource, np.float32)
      _view(dst + i * dst_stride * 4, idx.size, np.float32)[...] = x[idx]

  def regrid_bilinear(self, src, dst, nfield, src_stride, dst_stride,
                      source_shape, lon_taps, lat_taps):
    self.calls.append(('regrid_bilinear', int(nfield)))
    nlon_s, nlat_s = source_shape

    def lerp(a, i0, i1, frac, axis):
      i0, i1 = np.asarray(i0), np.asarray(i1)
      lo = np.take(a, np.maximum(i0, 0), axis=axis)
      hi = np.take(a, np.maximum(i1, 0), axis=axis)
      shape = [1, 1]
      shape[axis] = -1
      fr = np.asarray(frac, dtype=np.float32).reshape(shape)
      val = lo + fr * (hi - lo)
      outside = ((i0 < 0) | (i1 < 0)).reshape(shape)
      return np.where(outside, np.float32(np.nan), val).astype(np.float32)

    for i in range(nfield):
      x = _view(src + i * src_stride * 4, nlon_s * nlat_s, np.float32).reshape(
          nlon_s, nlat_s)
      y = lerp(x, *lat_taps, axis=1)   # latitude first, then longitude
      y = lerp(y, *lon_taps, axis=0)
      _view(dst + i * dst_stride * 4, y.size, np.float32)[...] = y.reshape(-1)

  # -- K4: zonal spectrum -------------------------------------------------------------
  @staticmethod
  def _spectra(x, nfield, nrow, ncol, scale):
    a = _view(x, nfield * nrow * ncol, np.float32).reshape(nfield, nrow, ncol)
    fk = np.fft.rfft(a.astype(np.float64), axis=-1, norm='forward')
    s = np.abs(fk) ** 2
    s[..., 1:] *= 2
    return s * np.asarray(scale, dtype=np.float64)[None, :, None]

  def zonal_spectrum(self, x, nfield, nrow, ncol, scale, out, accumulate=False,
                     nfield_out=0):
    self.calls.append(('zonal_spectrum', int(nfield), bool(accumulate)))
    s = self._spectra(x, nfield, nrow, ncol, scale)
    nk = ncol // 2 + 1
    if not accumulate:
      _view(out, s.size, np.float32)[...] = s.astype(np.float32).reshape(-1)
      return
    acc = _view(out, nfield_out * nrow * nk, np.float32).reshape(
        nfield_out, nrow, nk)
    for i in range(nfield):  # ADDED to slot i % nfield_out
      acc[i % nfield_out] += s[i].astype(np.float32)

  def zonal_spectrum_host(self, x, nfield, nrow, ncol, scale, out,
                          accumulate=False, nfield_out=0):
    if accumulate:  # the host entry OVERWRITES with the sum
      nk = ncol // 2 + 1
      _view(out, nfield_out * nrow * nk, np.float32)[...] = 0
    self.zonal_spectrum(x, nfield, nrow, ncol, scale, out, accumulate,
                        nfield_out)

  def zonal_spectrum_latsum(self, x, nfield, nrow, ncol, scale, out,
                            nfield_out):
    self.calls.append(('zonal_spectrum_latsum', int(nfield), int(nfield_out)))
    s = self._spectra(x, nfield, nrow, ncol, scale).sum(axis=1)
    res = np.zeros((nfield_out, ncol // 2 + 1))
    for i in range(nfield):
      res[i % nfield_out] += s[i]
    _view(out, res.size, np.float32)[...] = res.astype(np.float32).reshape(-1)

  def zonal_spectrum_latsum_host(self, *args):
    self.zonal_spectrum_latsum(*args)

  # -- derived variables / preprocessing ------------------------------------------------
  def wind_speed(self, u, v, out, n):
    self.calls.append(('wind_speed', int(n)))
    a, b = _view(u, n, np.float32), _view(v, n, np.float32)
    _view(out, n, np.float32)[...] = np.sqrt(a * a + b * b)

  def ens_mean(self, x, nmember, member_stride, off_x, slab, skipna, out):
    self.calls.append(('ens_mean', int(np.size(off_x)), int(nmember)))
    off_x = np.asarray(off_x)
    res = _view(out, off_x.size * slab, np.float32).reshape(off_x.size, slab)
    for i, off in enumerate(off_x):
      xs = np.stack([_view(x + (int(off) + m * member_stride) * 4, slab,
                           np.float32) for m in range(nmember)])
      with _quiet():
        res[i] = (np.nanmean if skipna else np.mean)(
            xs.astype(np.float64), axis=0).astype(np.float32)

  def spectrum_interp(self, spec, nfield, nrow, nk, freq_table, freqs, out):
    self.calls.append(('spectrum_interp', int(nfield)))
    a = _view(spec, nfield * nrow * nk, np.float32).reshape(nfield, nrow, nk)
    table = np.asarray(freq_table, dtype=np.float64).reshape(nrow, nk)
    fr = np.asarray(freqs, dtype=np.float64)
    res = _view(out, nfield * nrow * fr.size, np.float32).reshape(
        nfield, nrow, fr.size)
    for i in range(nfield):
      for r in range(nrow):
        res[i, r] = np.interp(fr, table[r], a[i, r].astype(np.float64),
                              left=np.nan, right=np.nan)

  def __getattr__(self, name):
    raise AttributeError(
        f'FakeContext has no emulation of {name!r}: this code path needs the '
        'GPU tests')


@contextlib.contextmanager
def _quiet():
  import warnings  # pylint: disable=import-outside-toplevel
  with warnings.catch_warnings():
    warnings.simplefilter('ignore', RuntimeWarning)
    yield


_installed = 0  # depth of the installed() blocks being executed


def active() -> bool:
  """Whether the stand-in is installed: test bodies shared with the GPU suite
  then keep to host inputs, even on a machine that has a GPU."""
  return _installed > 0


@contextlib.contextmanager
def installed():
  """Makes `_lib.default_context()` return a FakeContext inside the block."""
  global _installed
  fake = FakeContext()
  saved = _lib.default_context
  _lib.default_context = lambda device=None: fake
  _installed += 1
  try:
    yield fake
  finally:
    _installed -= 1
    _lib.default_context = saved
