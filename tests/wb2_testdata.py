"""NumPy restatement of the reference's test-data recipes (no xarray needed).

Follows weatherbench2/schema.py:62-115 (mock_truth_data / mock_forecast_data:
dims ('time','level','longitude','latitude'), latitude fastest, float32 zeros;
forecast prepends 'prediction_timedelta' then 'realization'),
weatherbench2/utils.py:290-295 (random_like: one RandomState(seed), .normal per
variable in dict order -> float64) and weatherbench2/test_utils.py:52-63
(insert_nan).  A "dataset" here is {'vars': {name: (dims, array)},
'coords': {name: array}}.
"""
import numpy as np
import pandas as pd


def mock_truth_data(*, variables_3d=('geopotential',), variables_2d=(),
                    levels=(500, 700, 850),
                    spatial_resolution_in_degrees=10.0,
                    time_start='2020-01-01', time_stop='2021-01-01',
                    time_resolution='1 day', dtype=np.float32):
  num_lat = round(180 / spatial_resolution_in_degrees) + 1
  num_lon = round(360 / spatial_resolution_in_degrees)
  freq = pd.Timedelta(time_resolution)
  coords = {
      'time': pd.date_range(time_start, time_stop, freq=freq,
                            inclusive='left').values,
      'latitude': np.linspace(-90, 90, num_lat),
      'longitude': np.linspace(0, 360, num_lon, endpoint=False),
      'level': np.array(levels),
  }
  dims_3d = ('time', 'level', 'longitude', 'latitude')
  shape_3d = tuple(coords[d].size for d in dims_3d)
  data = {k: (dims_3d, np.zeros(shape_3d, dtype)) for k in variables_3d}
  if not data:
    del coords['level']
  dims_2d = ('time', 'longitude', 'latitude')
  shape_2d = tuple(coords[d].size for d in dims_2d)
  data.update({k: (dims_2d, np.zeros(shape_2d, dtype)) for k in variables_2d})
  return {'vars': data, 'coords': coords}


def mock_forecast_data(*, lead_start='0 day', lead_stop='10 day',
                       lead_resolution='1 day', ensemble_size=None, **kwargs):
  lead = pd.timedelta_range(pd.Timedelta(lead_start), pd.Timedelta(lead_stop),
                            freq=pd.Timedelta(lead_resolution)).values
  ds = mock_truth_data(**kwargs)
  out = {}
  for k, (dims, arr) in ds['vars'].items():
    arr = np.broadcast_to(arr, (lead.size,) + arr.shape).copy()
    dims = ('prediction_timedelta',) + dims
    if ensemble_size is not None:
      arr = np.broadcast_to(arr, (ensemble_size,) + arr.shape).copy()
      dims = ('realization',) + dims
    out[k] = (dims, arr)
  coords = dict(ds['coords'])
  coords['prediction_timedelta'] = lead
  if ensemble_size is not None:
    coords['realization'] = np.arange(ensemble_size)
  return {'vars': out, 'coords': coords}


def random_like(ds, seed=0):
  rs = np.random.RandomState(seed)
  return {
      'vars': {k: (d, rs.normal(size=v.shape)) for k, (d, v) in
               ds['vars'].items()},
      'coords': dict(ds['coords']),
  }


def insert_nan(ds, frac_nan=0.1, seed=802701):
  rng = np.random.RandomState(seed)
  out = {}
  for k, (d, v) in ds['vars'].items():
    mask = rng.rand(*v.shape) < frac_nan
    out[k] = (d, np.where(mask, np.nan, v))
  return {'vars': out, 'coords': dict(ds['coords'])}


def get_random_truth_and_forecast(variables=('geopotential',),
                                  ensemble_size=None, seed=802701,
                                  lead_start='0 day', lead_stop='10 day',
                                  **data_kwargs):
  """weatherbench2/metrics_test.py:28-58."""
  kw = dict(variables_3d=variables, variables_2d=[], time_start='2019-12-01',
            time_stop='2019-12-02', spatial_resolution_in_degrees=30,
            time_resolution='3 hours')
  kw.update(data_kwargs)
  truth = random_like(mock_truth_data(**kw), seed=seed)
  forecast = random_like(
      mock_forecast_data(ensemble_size=ensemble_size, lead_start=lead_start,
                         lead_stop=lead_stop, **kw), seed=seed + 1)
  return truth, forecast


def host_and_device(x):
  """The array as the operators may receive it: NumPy, and -- when a GPU is
  present -- a CUDA tensor (the stand-in context of fake_ctx.py has no device
  memory: it sees the NumPy case only)."""
  yield x
  import torch
  import fake_ctx
  if torch.cuda.is_available() and not fake_ctx.active():
    yield torch.from_numpy(x).cuda()
