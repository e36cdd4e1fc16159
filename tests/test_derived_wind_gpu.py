"""GPU tests of the WindSpeed derived variable
(weatherbench2/derived_variables.py:77-99): bit-identical to NumPy, and usable
as `Eval.derived_variables` in the metric / region loop
(weatherbench2/evaluation.py:401-405)."""
import numpy as np
import pytest

import fake_ctx
from oracle import wb2_oracle as orc

pytestmark = pytest.mark.gpu


def _uv(shape, seed):
  rs = np.random.RandomState(seed)
  return (rs.normal(scale=8, size=shape).astype(np.float32),
          rs.normal(scale=8, size=shape).astype(np.float32))


def test_wind_speed_is_bit_identical_to_numpy():
  import torch
  from weatherbench2_b200 import derived_variables as dv, xarray_lite as xl
  dims = ('time', 'level', 'latitude', 'longitude')
  u, v = _uv((3, 2, 19, 36), 0)
  u[0, 0, 0, 0] = np.nan
  coords = {'time': np.arange(3), 'level': np.array([500, 850]),
            'latitude': np.linspace(-90, 90, 19),
            'longitude': np.linspace(0, 360, 36, endpoint=False)}
  ds = xl.Dataset({'u_component_of_wind': (dims, u),
                   'v_component_of_wind': (dims, v)}, coords)
  ws = dv.WindSpeed(u_name='u_component_of_wind', v_name='v_component_of_wind')
  assert ws.base_variables == ['u_component_of_wind', 'v_component_of_wind']
  got = ws.compute(ds)
  want = np.sqrt(u**2 + v**2)
  assert got.dims == dims and got.dtype == np.float32
  np.testing.assert_array_equal(got.values, want)
  if not torch.cuda.is_available() or fake_ctx.active():
    # the stand-in context reads host memory: NumPy inputs only
    return
  dev = xl.Dataset(
      {'u_component_of_wind': (dims, torch.from_numpy(u).cuda()),
       'v_component_of_wind': (dims, torch.from_numpy(v).cuda())}, coords)
  got = ws.compute(dev)
  assert got.data.is_cuda
  np.testing.assert_array_equal(got.data.cpu().numpy(), want)


def test_wind_speed_as_eval_derived_variable():
  from weatherbench2_b200 import config, derived_variables as dv, evaluation
  from weatherbench2_b200 import metrics, xarray_lite as xl
  dims = ('time', 'level', 'latitude', 'longitude')
  lat = np.linspace(-90, 90, 19)
  lon = np.linspace(0, 360, 36, endpoint=False)
  coords = {'time': np.arange(4), 'level': np.array([500, 850]),
            'latitude': lat, 'longitude': lon}
  fu, fv = _uv((4, 2, 19, 36), 1)
  tu, tv = _uv((4, 2, 19, 36), 2)
  names = ('u_component_of_wind', 'v_component_of_wind')
  fds = xl.Dataset({names[0]: (dims, fu), names[1]: (dims, fv)}, coords)
  tds = xl.Dataset({names[0]: (dims, tu), names[1]: (dims, tv)}, coords)
  ec = config.Eval(
      metrics={'mse': metrics.MSE()},
      derived_variables={'wind_speed': dv.WindSpeed(u_name=names[0],
                                                    v_name=names[1])})
  res = evaluation._metric_and_region_loop(fds, tds, ec, skipna=False)  # pylint: disable=protected-access
  fs, ts = np.sqrt(fu**2 + fv**2), np.sqrt(tu**2 + tv**2)
  want, wd = orc.mse(fs, dims, ts, dims, lat, lon)
  want, wd = orc.time_mean(want, wd, avg_dim='time')
  got = res['wind_speed'].isel(metric=0)
  a, b, _ = orc.align(np.asarray(got.values), got.dims, want, wd)
  np.testing.assert_allclose(a, b, rtol=1e-5)
