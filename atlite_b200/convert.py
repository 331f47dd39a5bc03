"""Reference-facing API of the hot path: ``convert_and_aggregate`` and the
``pv`` / ``wind`` / ``heat_demand`` wrappers, with the reference's signatures,
argument meaning, warnings and errors (convert.py:59-276, 421-471, 665-744,
857-936), executing on the GPU through ``libatlite_b200.so``.

Instead of building a lazy dask graph of ~60 ufunc passes and a per-chunk
``dense * csr.T`` product, a known ``convert_func`` is mapped to a fused
operator (physics + shape reduce in one kernel).  Unknown ``convert_func``
callables keep the reference's plugin protocol: they are evaluated by the
caller's code and only the aggregation runs on the GPU (``atl_spmm``).
"""

from __future__ import annotations

import logging
import re
import types
import warnings
from pathlib import Path

import numpy as np
import pandas as pd
import scipy.sparse as sp

from . import _lib, engine
from .labelled import HAVE_XARRAY, DataArray, is_dataarray, make_dataarray
from .orientation import get_orientation
from .resource import (
    EfficiencyTable,
    get_cspinstallationconfig,
    get_solarpanelconfig,
    get_windturbineconfig,
    windturbine_smooth,
)

if HAVE_XARRAY:  # pragma: no cover
    import xarray as xr

logger = logging.getLogger(__name__)

_SOLAR_WARNING = """The calculation method and handling of solar position variables will change.
    The solar position will in the future be a permanent variables of a cutout.
    Recreate your cutout to remove this warning and permanently include the solar position variables into your cutout."""


# --------------------------------------------------------------------------
# dataset access helpers (xarray.Dataset or atlite_b200.labelled.Dataset)
# --------------------------------------------------------------------------


def _has(ds, name):
    return name in ds


def _coord(ds, name):
    v = ds[name]
    return np.asarray(getattr(v, "values", v))


def _raw(ds, name):
    """(time, y, x) array of a variable: torch CUDA tensor for a device-resident
    cutout, else a NumPy array."""
    if hasattr(ds, "raw"):
        arr = ds.raw(name)
        dims = ds.dims_of(name)
        if dims != ("time", "y", "x")[-len(dims):]:
            raise ValueError(f"variable {name!r} must have dims (time, y, x), has {dims}")
        return arr
    da = ds[name]
    if da.ndim == 3:
        da = da.transpose("time", "y", "x")
    return np.asarray(da.values)


def _grid_shape(ds):
    return len(_coord(ds, "y")), len(_coord(ds, "x"))


def _is_dask_backed(ds):
    """Lazily loaded cutout: a dask-backed xarray dataset (what ``Cutout(path)`` opens,
    cutout.py:142-154) or an ``atlite_b200.LazyDataset``."""
    if getattr(ds, "lazy", False):
        return True
    if not HAVE_XARRAY or hasattr(ds, "raw"):
        return False
    try:
        from dask.array.core import Array

        return any(isinstance(ds[v].data, Array) for v in ds.data_vars)
    except Exception:  # noqa: BLE001
        return False


def _to_host(a):
    if engine._is_torch(a):
        return a.detach().cpu().numpy()
    return np.asarray(a)


# --------------------------------------------------------------------------
# fused operator specs
# --------------------------------------------------------------------------


def _solar_source(ds):
    """SolarPosition: getter vs computation (pv/solar_position.py:54-67) -> (SOLAR_* value,
    names of the stored solar position fields)."""
    if _has(ds, "solar_azimuth") and _has(ds, "solar_altitude"):
        dt = np.dtype(str(_raw(ds, "solar_altitude").dtype).replace("torch.", ""))
        return (_lib.SOLAR_STORED_F64 if dt == np.float64 else _lib.SOLAR_STORED_F32), \
            ["solar_altitude", "solar_azimuth"]
    warnings.warn(_SOLAR_WARNING, DeprecationWarning)
    return _lib.SOLAR_COMPUTED, []


class _Spec:
    """A known conversion bound to a cutout: can reduce to buses, or produce
    per-cell values / their time sum.  A subclass sets its operator ``op`` and its
    input ``fields`` (name -> (time, y, x) array or None, through ``_set_fields``)."""

    time_labels = None  # output time coordinate
    name = None
    units = None

    def __init__(self, ds):
        self.ny, self.nx = _grid_shape(ds)
        self.time_labels = pd.DatetimeIndex(_coord(ds, "time"))

    def _set_fields(self, fields):
        self.fields = fields
        self.pitch = engine.pitch_of(fields.values(), self.nx)

    def _device_fields(self):
        """Host arrays -> device tensors (per-cell output paths only)."""
        torch = engine._torch()
        dev = f"cuda:{engine.current_device()}"
        return {
            k: (v if v is None or engine._is_torch(v) else torch.from_numpy(np.ascontiguousarray(v)).to(dev))
            for k, v in self.fields.items()
        }

    def reduce(self, plan):
        return self.op.reduce(plan, self.fields)

    def cells(self, timesum=False):
        """Per-cell values (time, y, x), or with ``timesum`` the NaN-skipping per-cell time sum
        and the number of valid steps per cell, stacked (2, y, x)."""
        return self.op.cells(self._device_fields(), timesum=timesum)


class _PvSpec(_Spec):
    name = "specific generation"

    def __init__(self, ds, panel, orientation, tracking=None, trigon_model="simple",
                 clearsky_model="simple", output="panel", thermal=(0.0, 0.0, 0.0)):
        super().__init__(ds)
        ny, nx = self.ny, self.nx
        self.ds = ds
        lon, lat = _coord(ds, "lon").astype(np.float64), _coord(ds, "lat").astype(np.float64)
        solar_src, solar_names = _solar_source(ds)

        # SurfaceOrientation (pv/orientation.py:104-109, 177-183)
        if tracking not in _lib.TRACKING:
            raise AssertionError(
                "Values describing tracking system must be None for no tracking,"
                "'horizontal' for 1-axis horizontal tracking,"
                "tilted_horizontal' for 1-axis horizontal tracking of tilted panle,"
                "vertical' for 1-axis vertical tracking, or 'dual' for 2-axis tracking"
            )
        lon_r = DataArray(np.radians(lon), {"x": _coord(ds, "x")}, ("x",), "lon")
        lat_r = DataArray(np.radians(lat), {"y": _coord(ds, "y")}, ("y",), "lat")
        o = orientation(lon_r, lat_r, None)

        def table(v, nm):
            """slope / azimuth of the callback (pv/orientation.py:107) -> scalar, (y,) or (y, x)."""
            if hasattr(v, "dims") and hasattr(v, "transpose") and getattr(v, "ndim", 0) >= 1:
                dims = tuple(v.dims)
                if not set(dims) <= {"y", "x"}:
                    raise NotImplementedError(
                        f"orientation {nm} varies along {dims}; only (y, x)-dependent orientations are "
                        "supported (the orientation may not depend on time / the solar position)")
                v = v.transpose(*[d for d in ("y", "x") if d in dims])
                arr = np.asarray(v.values, dtype=np.float64)
                return arr[None, :] * np.ones((ny, 1)) if dims == ("x",) else arr
            arr = np.asarray(getattr(v, "values", v), dtype=np.float64)
            if arr.ndim == 0 or arr.shape == (ny,) or arr.shape == (ny, nx):
                return arr
            if arr.shape == (nx,):
                return arr[None, :] * np.ones((ny, 1))
            raise NotImplementedError(
                f"orientation {nm} must be a scalar, vary with latitude (y), or be a (y, x) array; "
                f"got shape {arr.shape}")

        slope, azimuth = table(o["slope"], "slope"), table(o["azimuth"], "azimuth")

        # TiltedIrradiation inputs (pv/irradiation.py:202-213)
        if _has(ds, "influx"):
            irr_branch = _lib.IRR_INFLUX
            cm = clearsky_model
            if cm is None:
                cm = "enhanced" if _has(ds, "temperature") and _has(ds, "humidity") else "simple"
            if cm not in _lib.CLEARSKY:
                raise KeyError("`clearsky model` must be chosen from 'simple' and 'enhanced'")
            clearsky = _lib.CLEARSKY[cm]
        elif _has(ds, "influx_direct") and _has(ds, "influx_diffuse"):
            irr_branch, clearsky = _lib.IRR_DIRECT_DIFFUSE, 0
        else:
            raise AssertionError(
                "Need either influx or influx_direct and influx_diffuse in the "
                "dataset. Check your cutout and dataset module."
            )
        if _has(ds, "albedo"):
            albedo_src = _lib.ALBEDO_VAR
        elif _has(ds, "outflux"):
            albedo_src = _lib.ALBEDO_OUTFLUX
        else:
            raise AssertionError(
                "Need either albedo or outflux as a variable in the dataset. "
                "Check your cutout and dataset module."
            )
        trigon = _lib.TRIGON_SIMPLE if trigon_model == "simple" else _lib.TRIGON_HAY_DAVIES

        names = ["influx_toa", "temperature"]
        if output in ("total", "direct", "diffuse", "ground") and not _has(ds, "temperature"):
            names = ["influx_toa"]  # irradiation needs no temperature (convert.py:748-767)
        names += ["influx"] if irr_branch == _lib.IRR_INFLUX else ["influx_direct", "influx_diffuse"]
        if irr_branch == _lib.IRR_INFLUX and clearsky == 1:
            names.append("humidity")
        names.append("albedo" if albedo_src == _lib.ALBEDO_VAR else "outflux")
        fields = {n: _raw(ds, n) for n in names + solar_names}
        fields.setdefault("temperature", fields["influx_toa"])  # unused placeholder
        self._set_fields(fields)
        self.op = engine.PvOp(
            ny=ny, nx=nx, time=self.time_labels, lon=lon, lat=lat, slope=slope, azimuth=azimuth,
            tracking=tracking, trigon_model=trigon, clearsky_model=clearsky,
            irr_branch=irr_branch, albedo_src=albedo_src, solar_src=solar_src, panel=panel,
            output=output, thermal=thermal, pitch=self.pitch,
        )


class _IrradiationSpec(_PvSpec):
    """convert_irradiation (convert.py:748-767): the PV operator without the panel."""

    units = "W m**-2"

    def __init__(self, ds, orientation, tracking=None, irradiation="total", trigon_model="simple",
                 clearsky_model="simple"):
        if irradiation not in ("total", "direct", "diffuse", "ground"):
            raise ValueError(f"irradiation must be total, direct, diffuse or ground, not {irradiation!r}")
        super().__init__(ds, None, orientation, tracking, trigon_model, clearsky_model, output=irradiation)
        self.name = f"{irradiation} tilted"


class _SolarThermalSpec(_PvSpec):
    """convert_solar_thermal (convert.py:550-573)."""

    def __init__(self, ds, orientation, trigon_model, clearsky_model, c0, c1, t_store):
        super().__init__(ds, None, orientation, None, trigon_model, clearsky_model,
                         output="solar_thermal", thermal=(c0, c1, t_store))
        self.name = None


class _PointwiseSpec(_Spec):
    """Pointwise function of one (time, y, x) variable."""

    def __init__(self, ds, var, shift=0.0, nan_to_zero=False, poly=None, cell_scale=None, name=None):
        super().__init__(ds)
        if not _has(ds, var):
            raise KeyError(var)
        self._set_fields({var: _raw(ds, var)})
        self.name = name
        self.op = engine.PointwiseOp(ny=self.ny, nx=self.nx, shift=shift, nan_to_zero=nan_to_zero, poly=poly,
                                     cell_scale=cell_scale, pitch=self.pitch)


def _temperature_spec(ds):
    return _PointwiseSpec(ds, "temperature", shift=-273.15, name="temperature")


def _soil_temperature_spec(ds):
    return _PointwiseSpec(ds, "soil temperature", shift=-273.15, nan_to_zero=True, name="soil temperature")


def _dewpoint_temperature_spec(ds):
    return _PointwiseSpec(ds, "dewpoint temperature", shift=-273.15, name="dewpoint temperature")


def _cop_spec(ds, source, sink_T, c0, c1, c2):
    assert source in ["air", "soil"], NotImplementedError("'source' must be one of  ['air', 'soil']")
    if source == "air":  # convert.py:343-350
        d = (6.81, -0.121, 0.000630)
        var, nz = "temperature", False
    else:  # convert.py:351-358
        d = (8.77, -0.150, 0.000734)
        var, nz = "soil temperature", True
    c0, c1, c2 = (dv if v is None else v for v, dv in zip((c0, c1, c2), d))
    return _PointwiseSpec(ds, var, shift=-273.15, nan_to_zero=nz, poly=(sink_T, c0, c1, c2))


def _runoff_spec(ds, weight_with_height=True):
    scale = None
    if weight_with_height:
        if not _has(ds, "height"):
            raise KeyError(
                "runoff(weight_with_height=True) needs the static 'height' variable (datasets/era5.py:65-81: "
                "geopotential z / g0); prepare the cutout with the 'height' feature "
                "(atlite_b200.era5.get_data_height) or pass weight_with_height=False"
            )
        h = _raw(ds, "height")
        scale = _to_host(h)
        if scale.ndim == 3:
            scale = scale[0]
        scale = np.ascontiguousarray(scale[:, : _grid_shape(ds)[1]])  # drop row padding
    return _PointwiseSpec(ds, "runoff", cell_scale=scale, name="runoff")


class _CspSpec(_Spec):
    """convert_csp (convert.py:940-972)."""

    name = "specific generation"
    units = "kWh/kW_ref"

    def __init__(self, ds, installation):
        super().__init__(ds)
        tech = installation["technology"]
        if tech not in _lib.CSP_TECH:
            raise ValueError(f'Unknown CSP technology option "{tech}".')
        solar_src, solar_names = _solar_source(ds)
        eff = EfficiencyTable.from_any(installation["efficiency"])
        self._set_fields({n: _raw(ds, n) for n in ["influx_direct"] + solar_names})
        self.op = engine.CspOp(
            ny=self.ny, nx=self.nx, time=self.time_labels, lon=_coord(ds, "lon").astype(np.float64),
            lat=_coord(ds, "lat").astype(np.float64), solar_src=solar_src,
            technology=_lib.CSP_TECH[tech], r_irradiance=installation["r_irradiance"],
            altitude=eff.altitude, azimuth=eff.azimuth, efficiency=eff.values, pitch=self.pitch,
        )


class _WindSpec(_Spec):
    name = "specific generation"
    units = "MWh/MWp"

    def __init__(self, ds, turbine, interpolation_method="logarithmic"):
        super().__init__(ds)
        V, POW, hub_height, P = (turbine[k] for k in ("V", "POW", "hub_height", "P"))
        to_name = f"wnd{int(hub_height):0d}m"
        aux = None
        from_height = hub_height
        if _has(ds, to_name):  # fast lane, wind.py:75-78
            method = _lib.WIND_NONE
            wnd = _raw(ds, to_name)
        else:
            names = list(ds.data_vars) if hasattr(ds, "data_vars") else list(ds)
            heights = np.asarray([int(s[3:-1]) for s in names if re.match(r"wnd\d+m", str(s))])
            if len(heights) == 0:
                raise AssertionError("Wind speed is not in dataset")
            from_height = heights[np.argmin(np.abs(heights - hub_height))]
            wnd = _raw(ds, f"wnd{int(from_height):0d}m")
            if interpolation_method == "logarithmic":
                if not _has(ds, "roughness"):
                    raise RuntimeError(
                        "The logarithmic interpolation method requires surface roughness (roughness);\n"
                        "make sure you choose a compatible dataset like ERA5"
                    )
                method, aux = _lib.WIND_LOG, _raw(ds, "roughness")
            elif interpolation_method == "power":
                if not _has(ds, "wnd_shear_exp"):
                    raise RuntimeError(
                        "The power law interpolation method requires a wind shear exponent (wnd_shear_exp);\n"
                        "make sure you choose a compatible dataset like ERA5 and update your cutout"
                    )
                method, aux = _lib.WIND_POWER, _raw(ds, "wnd_shear_exp")
            else:
                raise ValueError(
                    f"Interpolation method must be 'logarithmic' or 'power',  but is: {interpolation_method}"
                )
        self.wnd, self.aux = wnd, aux
        self._set_fields({"wnd": wnd, "aux": aux})
        self.op = engine.WindOp(
            ny=self.ny, nx=self.nx, V=np.asarray(V, float), POW_norm=np.asarray(POW, float) / P,
            method=method, from_height=from_height, to_height=hub_height, pitch=self.pitch,
        )

    def reduce(self, plan):
        return self.op.reduce(plan, self.wnd, self.aux)


def day_bins(time, hour_shift):
    """Calendar-day bins of ``time + hour_shift`` (``resample(time="1D")``,
    convert.py:408-412).  Returns (day labels, offsets[n_days+1] into time)."""
    t = pd.DatetimeIndex(time) + pd.Timedelta(hours=hour_shift)
    if len(t) == 0:
        return pd.DatetimeIndex([]), np.zeros(1, dtype=np.int64)
    if not t.is_monotonic_increasing:
        raise ValueError("time axis must be sorted for the daily heat-demand bins")
    days = t.floor("D")
    labels = pd.date_range(days[0], days[-1], freq="D")
    offsets = np.searchsorted(days.values, labels.values, side="left")
    offsets = np.append(offsets, len(t)).astype(np.int64)
    return labels, offsets


class _HeatSpec(_Spec):
    name = "heat_demand"
    cooling = False

    def __init__(self, ds, threshold, a, constant, hour_shift):
        super().__init__(ds)
        self.temp = _raw(ds, "temperature")
        self.time_labels, self.day_start = day_bins(_coord(ds, "time"), hour_shift)
        self._set_fields({"temperature": self.temp})
        self.op = engine.HeatOp(ny=self.ny, nx=self.nx, threshold=threshold, a=a, constant=constant,
                                cooling=self.cooling, pitch=self.pitch)

    def reduce(self, plan):
        return self.op.reduce(plan, self.temp, self.day_start)

    def cells(self, timesum=False):
        return self.op.cells(self._device_fields(), self.day_start, timesum=timesum)


class _CoolingSpec(_HeatSpec):
    """convert_cooling_demand (convert.py:475-491): a * (Tmean - threshold)."""

    name = "cooling_demand"
    cooling = True


# --------------------------------------------------------------------------
# convert_* callables (plugin protocol, convert.py:198)
# --------------------------------------------------------------------------


def _wrap_cells(ds, spec, values):
    coords = {"time": spec.time_labels, "y": _coord(ds, "y"), "x": _coord(ds, "x")}
    attrs = {"units": spec.units} if spec.units else {}
    return make_dataarray(_to_host(values), ("time", "y", "x"), coords, attrs, spec.name)


def convert_pv(ds, panel, orientation, tracking=None, trigon_model="simple", clearsky_model="simple"):
    """Per-cell PV capacity factors (time, y, x); convert.py:840-854."""
    spec = _PvSpec(ds, panel, orientation, tracking, trigon_model, clearsky_model)
    return _wrap_cells(ds, spec, spec.cells())


def convert_wind(ds, turbine, interpolation_method="logarithmic"):
    """Per-cell wind capacity factors (time, y, x); convert.py:634-662."""
    spec = _WindSpec(ds, turbine, interpolation_method)
    return _wrap_cells(ds, spec, spec.cells())


def convert_heat_demand(ds, threshold, a, constant, hour_shift):
    """Per-cell daily heat demand (day, y, x); convert.py:405-418."""
    spec = _HeatSpec(ds, threshold, a, constant, hour_shift)
    return _wrap_cells(ds, spec, spec.cells())


def convert_irradiation(ds, orientation, tracking=None, irradiation="total", trigon_model="simple",
                        clearsky_model="simple"):
    """Per-cell tilted irradiation (time, y, x); convert.py:748-767."""
    spec = _IrradiationSpec(ds, orientation, tracking, irradiation, trigon_model, clearsky_model)
    return _wrap_cells(ds, spec, spec.cells())


def convert_solar_thermal(ds, orientation, trigon_model, clearsky_model, c0, c1, t_store):
    """Per-cell solar thermal collector output; convert.py:550-573."""
    spec = _SolarThermalSpec(ds, orientation, trigon_model, clearsky_model, c0, c1, t_store)
    return _wrap_cells(ds, spec, spec.cells())


def convert_temperature(ds):
    """Outside temperature in deg C; convert.py:292-298."""
    spec = _temperature_spec(ds)
    return _wrap_cells(ds, spec, spec.cells())


def convert_soil_temperature(ds):
    """Soil temperature in deg C, 0 over sea; convert.py:306-316."""
    spec = _soil_temperature_spec(ds)
    return _wrap_cells(ds, spec, spec.cells())


def convert_dewpoint_temperature(ds):
    """Dewpoint temperature in deg C; convert.py:324-329."""
    spec = _dewpoint_temperature_spec(ds)
    return _wrap_cells(ds, spec, spec.cells())


def convert_coefficient_of_performance(ds, source, sink_T, c0, c1, c2):
    """Heat pump COP; convert.py:338-366."""
    spec = _cop_spec(ds, source, sink_T, c0, c1, c2)
    return _wrap_cells(ds, spec, spec.cells())


def convert_cooling_demand(ds, threshold, a, constant, hour_shift):
    """Per-cell daily cooling demand; convert.py:475-491."""
    spec = _CoolingSpec(ds, threshold, a, constant, hour_shift)
    return _wrap_cells(ds, spec, spec.cells())


def convert_csp(ds, installation):
    """Per-cell CSP specific generation; convert.py:940-972."""
    spec = _CspSpec(ds, installation)
    return _wrap_cells(ds, spec, spec.cells())


def convert_runoff(ds, weight_with_height=True):
    """Runoff (optionally weighted with height); convert.py:1028-1034."""
    spec = _runoff_spec(ds, weight_with_height)
    return _wrap_cells(ds, spec, spec.cells())


_SPECS = {
    "convert_pv": _PvSpec, "convert_wind": _WindSpec, "convert_heat_demand": _HeatSpec,
    "convert_irradiation": _IrradiationSpec, "convert_solar_thermal": _SolarThermalSpec,
    "convert_temperature": _temperature_spec, "convert_soil_temperature": _soil_temperature_spec,
    "convert_dewpoint_temperature": _dewpoint_temperature_spec,
    "convert_coefficient_of_performance": _cop_spec, "convert_cooling_demand": _CoolingSpec,
    "convert_runoff": _runoff_spec, "convert_csp": _CspSpec,
}


# identity -> spec: this package's own convert_* objects ...
_REGISTRY = {globals()[_n]: _s for _n, _s in _SPECS.items()}


def _reference_registry():
    """... plus the reference's, when the caller has imported it (``atlite.convert``
    in sys.modules): a script written against the reference passes
    ``atlite.convert.convert_pv`` etc. as ``convert_func``."""
    import sys

    mod = sys.modules.get("atlite.convert")
    if mod is None:
        return {}
    return {getattr(mod, n): s for n, s in _SPECS.items() if callable(getattr(mod, n, None))}


def _known_spec(convert_func):
    """Fused operator for a KNOWN converter, matched by identity (never by name: a user
    plugin that happens to be called ``convert_pv`` keeps the plugin protocol)."""
    try:
        spec = _REGISTRY.get(convert_func)
        return spec if spec is not None else _reference_registry().get(convert_func)
    except TypeError:  # unhashable callable
        return None


# --------------------------------------------------------------------------
# time-partitioned execution: several GPUs from one process, lazily loaded cutouts
# --------------------------------------------------------------------------


PART_BYTES = 1 << 30  # input bytes per time part of a lazily loaded cutout


def _time_slice(ds, lo, hi):
    """Steps [lo, hi) of a cutout dataset (views for in-memory data; for a dask-backed
    xarray dataset still lazy: only these steps are read when the part is converted)."""
    if hasattr(ds, "isel_time"):
        return ds.isel_time(lo, hi)
    return ds.isel(time=slice(lo, hi))


def _bytes_per_step(ds):
    ny, nx = _grid_shape(ds)
    names = list(ds.data_vars) if hasattr(ds, "data_vars") else list(ds)
    if hasattr(ds, "dims_of"):
        n3 = sum(1 for n in names if len(ds.dims_of(n)) == 3)
    else:
        n3 = sum(1 for n in names if len(ds[n].dims) == 3)  # xarray: metadata only, nothing is read
    return max(1, n3) * ny * nx * 4


def _is_host_resident(ds):
    """No variable lives on a GPU (device-resident cutouts are single-device objects)."""
    if not hasattr(ds, "raw") or getattr(ds, "lazy", False):
        return True
    return not any(engine._is_torch(ds.raw(n)) and ds.raw(n).is_cuda for n in ds.keys())


def _partition(ds, n_time, devices, lazy, day_offsets=None):
    """Contiguous time parts [(lo, hi, device)], in time order.  In-memory cutouts get one
    part per device; lazily loaded ones (dask-backed) parts of ~1 GiB of input, cut on the
    dataset's own time chunks (cutout.py:143: {"time": 100}), so a cutout that does not
    fit the host memory streams through it.  ``day_offsets`` (heat / cooling demand):
    part boundaries are snapped to calendar-day starts of the shifted axis."""
    from .dist import shard_bounds

    n_dev = len(devices)
    if n_time == 0:
        return [(0, 0, devices[0])]
    cuts = [0]
    if lazy:
        unit = 100
        try:
            ch = ds.chunks.get("time") if hasattr(ds.chunks, "get") else None
            if ch:
                unit = max(1, int(ch[0]))
        except Exception:  # noqa: BLE001
            pass
        k = max(1, int(round(PART_BYTES / (unit * _bytes_per_step(ds)))))
        per_dev = [shard_bounds(n_time, n_dev, r, align=unit) for r in range(n_dev)]
        for lo, hi in per_dev:
            for c in range(lo + unit * k, hi, unit * k):
                cuts.append(c)
            if hi > cuts[-1]:
                cuts.append(hi)
    else:
        per_dev = [shard_bounds(n_time, n_dev, r) for r in range(n_dev)]
        cuts += [hi for lo, hi in per_dev if hi > lo]
    owner_of = lambda lo: next(devices[r] for r, (a, b) in enumerate(per_dev) if a <= lo < b)  # noqa: E731
    if day_offsets is not None:  # snap to day starts (first step of a day of the shifted axis)
        offs = np.asarray(day_offsets)
        snapped = sorted({int(offs[np.argmin(np.abs(offs - c))]) for c in cuts[1:-1]} | {0, n_time})
        cuts = snapped
    cuts = sorted(set(cuts))
    return [(lo, hi, owner_of(min(lo, n_time - 1))) for lo, hi in zip(cuts[:-1], cuts[1:]) if hi > lo]


def _run_partitioned(ds, spec_cls, convert_kwds, parts, run, workers_per_device):
    """Convert every time part on its device (one host thread per device, two for lazily
    loaded data so that reading part i+1 overlaps the GPU work on part i) and return the
    per-part results in time order.  ``run(spec, device) -> result`` does the per-part work."""
    from concurrent.futures import ThreadPoolExecutor

    torch = engine._torch()
    devices = sorted({d for _, _, d in parts})
    pools = {d: ThreadPoolExecutor(workers_per_device, thread_name_prefix=f"atl-dev{d}") for d in devices}
    caught = warnings.catch_warnings(record=True)
    log = caught.__enter__()  # the worker threads' warnings are re-issued once by the caller's thread
    warnings.simplefilter("always")

    def work(lo, hi, dev):
        torch.cuda.set_device(dev)  # per-thread current device
        spec = spec_cls(_time_slice(ds, lo, hi), **convert_kwds)
        res = run(spec, dev)
        # only the labels travel on: the spec owns the part's input (up to PART_BYTES of decoded
        # fields, or its device copy), which must not outlive the part -- a lazily loaded cutout
        # larger than the host memory is the point of converting part by part
        return res, types.SimpleNamespace(units=getattr(spec, "units", None), name=spec.name,
                                          time_labels=spec.time_labels)

    try:
        futs = [pools[d].submit(work, lo, hi, d) for lo, hi, d in parts]
        out = [f.result() for f in futs]
    finally:
        for p in pools.values():
            p.shutdown(wait=True)
        caught.__exit__(None, None, None)
    seen = set()
    for w in log:
        key = (w.category, str(w.message))
        if key not in seen:
            seen.add(key)
            warnings.warn_explicit(w.message, w.category, w.filename, w.lineno)
    return out


# --------------------------------------------------------------------------
# orchestration
# --------------------------------------------------------------------------


def _aggregate_time_np(values, method, axis):
    if method == "sum":
        return np.nansum(values, axis=axis)
    if method == "mean":
        return np.nanmean(values, axis=axis)
    return values


def _finish_results(res, caps, agg, bus_major):
    """The tail of convert_and_aggregate (convert.py:259-271) on a (time, bus) float32 result:
    float64, ``/ capacity.where(capacity != 0)`` then ``fillna(0)`` when ``caps`` is given
    (per_unit), time aggregation (``agg`` = "sum" / "mean", NaN-skipping like xarray's) or the
    (bus, time) layout of NumPy-backed cutouts.  A device result is finished ON the device --
    for a year x 3000 buses these are four passes over 210 MB and a strided transpose that cost
    the host several times the conversion kernel -- and only the final array crosses PCIe."""
    if engine._is_torch(res):
        torch = engine._torch()
        r = res.to(torch.float64)
        if caps is not None:
            c = torch.as_tensor(np.where(caps != 0, caps, np.nan), dtype=torch.float64, device=r.device)
            r = r / c[None, :]
            r = torch.where(torch.isnan(r), torch.zeros((), dtype=r.dtype, device=r.device), r)
        if agg == "sum":
            r = torch.nansum(r, dim=0)
        elif agg == "mean":
            r = torch.nanmean(r, dim=0)
        elif bus_major:
            r = r.T.contiguous()
        return r.cpu().numpy()
    results = np.asarray(res).astype(np.float64)
    if caps is not None:
        with np.errstate(divide="ignore", invalid="ignore"):
            results = results / np.where(caps != 0, caps, np.nan)[None, :]
        results = np.where(np.isnan(results), 0.0, results)
    if agg is not None:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", RuntimeWarning)  # mean of an all-NaN column is NaN, silently
            return _aggregate_time_np(results, agg, 0)
    return np.ascontiguousarray(results.T) if bus_major else results


def _ensure_index(index, n):
    """utils.py:22-36 ensure_coords: pandas Index -> (dim name, Index)."""
    if index is None:
        index = pd.RangeIndex(n)
    if isinstance(index, pd.MultiIndex):
        return index.name or "dim_0", index
    if isinstance(index, pd.Index):
        return index.name or "dim_0", index
    if HAVE_XARRAY and isinstance(index, xr.Coordinates):
        if len(index.dims) > 1:
            raise ValueError(f"index must have a single dimension, not: {index.dims}")
        d = list(index.dims)[0]
        return d, index.to_index()
    raise ValueError(f"index must be a pandas index or xarray coordinates, not: {index}")


def _layout_values(layout, ds):
    """layout.reindex_like(cutout.data).stack(spatial=[y, x])  (convert.py:244)."""
    y, x = _coord(ds, "y"), _coord(ds, "x")
    if HAVE_XARRAY and isinstance(layout, xr.DataArray):
        lay = layout.reindex(y=y, x=x).transpose("y", "x")
        return np.asarray(lay.values, dtype=np.float64).reshape(-1)
    lay = layout.transpose("y", "x")
    iy = pd.Index(np.asarray(lay.coords["y"])).get_indexer(y)
    ix = pd.Index(np.asarray(lay.coords["x"])).get_indexer(x)
    vals = np.asarray(lay.values, dtype=np.float64)
    out = vals[np.clip(iy, 0, None)][:, np.clip(ix, 0, None)]
    out[iy < 0, :] = np.nan
    out[:, ix < 0] = np.nan
    return out.reshape(-1)


def _aggregate_time_arg(aggregate_time, capacity_factor, capacity_factor_timeseries):
    """``aggregate_time`` after the deprecated ``capacity_factor*`` flags (convert.py:183-217);
    the warnings point at the caller of ``convert_and_aggregate``."""
    if aggregate_time not in ("sum", "mean", "legacy", None):
        raise ValueError(
            f"aggregate_time must be 'sum', 'mean', 'legacy', or None, got {aggregate_time!r}"
        )
    if aggregate_time == "legacy":
        warnings.warn(
            "aggregate_time='legacy' is deprecated and will be removed in a "
            "future release. Pass 'sum', 'mean', or None explicitly.",
            FutureWarning,
            stacklevel=3,
        )
    if capacity_factor or capacity_factor_timeseries:
        if aggregate_time != "legacy":
            raise ValueError(
                "Cannot use 'aggregate_time' together with deprecated "
                "'capacity_factor' or 'capacity_factor_timeseries'."
            )
        if capacity_factor:
            warnings.warn(
                "capacity_factor is deprecated. Use aggregate_time='mean' instead.",
                FutureWarning,
                stacklevel=3,
            )
            aggregate_time = "mean"
        if capacity_factor_timeseries:
            warnings.warn(
                "capacity_factor_timeseries is deprecated. Use aggregate_time=None instead.",
                FutureWarning,
                stacklevel=3,
            )
            aggregate_time = None
    return aggregate_time


def _aggregation_matrix(cutout, ds, matrix, index, layout, shapes, shapes_crs):
    """``matrix`` / ``shapes`` / ``layout`` / ``index`` -> (CSR aggregation matrix, bus dim name,
    bus index) (convert.py:233-255)."""
    if matrix is not None:
        if shapes is not None:
            raise ValueError("Passing matrix and shapes is ambiguous. Pass only one of them.")
        if is_dataarray(matrix):
            coords = matrix.indexes[matrix.dims[1]].to_frame(index=False)
            if not np.array_equal(coords[["x", "y"]], cutout.grid[["x", "y"]]):
                raise ValueError(
                    "Matrix spatial coordinates not aligned with cutout spatial coordinates."
                )
            if index is None:
                index = matrix
            matrix = matrix.values
        if not matrix.ndim == 2:
            raise ValueError("Matrix not 2-dimensional.")
        matrix = sp.csr_matrix(matrix)

    if shapes is not None:
        if isinstance(shapes, pd.Series) or hasattr(shapes, "geometry"):
            if index is None:
                index = shapes.index
        matrix = cutout.indicatormatrix(shapes, shapes_crs).tocsr()

    if layout is not None:
        assert is_dataarray(layout)
        lay = _layout_values(layout, ds)
        if matrix is None:
            matrix = sp.csr_matrix(lay[None, :])
        else:
            # csr(matrix) * spdiag(layout) (convert.py:249) scales column j by layout[j]: done on the
            # entries directly (6 ms instead of the 44 ms sparse product at 1440 x 720 -> 3000 shapes)
            m0 = sp.csr_matrix(matrix)
            matrix = sp.csr_matrix((m0.data.astype(np.float64) * lay[m0.indices], m0.indices, m0.indptr), shape=m0.shape)

    assert isinstance(matrix, sp.csr_matrix)
    dim, idx = _ensure_index(index, matrix.shape[0])
    return matrix, dim, idx


class _PluginSpec:
    """A plugin's (time, y, x) result on the reduce path: only the aggregation runs on the GPU
    (``atl_spmm``).  A result computed from a row-padded device cutout keeps the padding."""

    def __init__(self, da):
        self.da = da
        self.values = da if engine._is_torch(da) else getattr(da, "values", da)
        self.pitch = int(self.values.shape[-1]) if engine._is_torch(self.values) and self.values.ndim == 3 else None
        self.name = getattr(da, "name", None)

    def reduce(self, plan):
        return plan.spmm(self.values if engine._is_torch(self.values) else np.asarray(self.values))

    @property
    def time_labels(self):
        if hasattr(self.da, "coords"):
            return pd.Index(np.asarray(self.da.coords["time"]))
        return pd.RangeIndex(len(self.values))


def _joined(res):
    """Per-part [(values, labels)] -> (values, time labels) joined along time."""
    if len(res) == 1:
        return res[0][0], res[0][1].time_labels
    labels = pd.Index(np.concatenate([np.asarray(m.time_labels) for _, m in res]))
    if isinstance(res[0][1].time_labels, pd.DatetimeIndex):
        labels = pd.DatetimeIndex(labels)
    return np.concatenate([v for v, _ in res], axis=0), labels


def convert_and_aggregate(
    cutout,
    convert_func,
    matrix=None,
    index=None,
    layout=None,
    shapes=None,
    shapes_crs=4326,
    per_unit=False,
    return_capacity=False,
    aggregate_time="legacy",
    capacity_factor=False,
    capacity_factor_timeseries=False,
    show_progress=False,
    dask_kwargs={},
    **convert_kwds,
):
    """Convert and aggregate a weather-based renewable generation time-series.

    Same contract as the reference (convert.py:59-276): ``matrix`` (N x S, in
    ``cutout.grid`` order), ``shapes`` or ``layout`` select spatial
    aggregation; ``per_unit`` / ``return_capacity``; ``aggregate_time`` in
    {"sum", "mean", "legacy", None}; deprecated ``capacity_factor*`` flags.
    ``show_progress`` and ``dask_kwargs`` are accepted and ignored (the result
    is computed eagerly on the GPU and returned loaded).
    """
    aggregate_time = _aggregate_time_arg(aggregate_time, capacity_factor, capacity_factor_timeseries)
    func_name = convert_func.__name__.replace("convert_", "")
    logger.info(f"Convert and aggregate '{func_name}'.")
    ds = cutout.data
    ny, nx = _grid_shape(ds)
    spec_cls = _known_spec(convert_func)
    shard = getattr(cutout, "time_shard", None)  # multi-GPU time sharding (dist.py)
    devices = list(getattr(cutout, "devices", None) or [])
    lazy = _is_dask_backed(ds)
    # several GPUs from this one process, and/or a lazily loaded (dask-backed) cutout that
    # is converted time part by time part instead of being materialised whole
    partitioned = spec_cls is not None and (len(devices) > 1 or lazy) and _is_host_resident(ds)
    if partitioned and shard is not None:
        raise ValueError("a cutout is either time-sharded across processes (time_shard=) or fanned "
                         "out to several devices by one process (devices=), not both")
    spec = da = parts = None
    if partitioned:
        day_offsets = None
        if spec_cls in (_HeatSpec, _CoolingSpec):
            day_offsets = day_bins(_coord(ds, "time"), convert_kwds.get("hour_shift", 0.0))[1]
        parts = _partition(ds, len(_coord(ds, "time")), devices or [engine.current_device()], lazy, day_offsets)
    else:
        if len(devices) == 1:
            engine._torch().cuda.set_device(devices[0])
        if spec_cls is not None:
            spec = spec_cls(ds, **convert_kwds)
        else:  # plugin protocol: the callable produces the (time, y, x) field itself
            da = convert_func(ds, **convert_kwds)

    def execute(spec, run):
        """[(result, labels)] of ``run(spec, device)`` per time part.  In-process: ``spec`` on
        the caller's thread, its result left where it was computed; partitioned: a spec per
        part on its device, its result moved to the host."""
        if parts is None:
            return [(run(spec, None), spec)]
        return _run_partitioned(ds, spec_cls, convert_kwds, parts, lambda sp_, dev: _to_host(run(sp_, dev)),
                                2 if lazy else 1)

    if all(v is None for v in [layout, shapes, matrix]):
        if per_unit or return_capacity:
            raise ValueError(
                "One of `matrix`, `shapes` and `layout` must be "
                "given for `per_unit` or `return_capacity`"
            )
        agg = "sum" if aggregate_time == "legacy" else aggregate_time
        if da is not None:
            if agg == "sum":
                return da.sum("time", keep_attrs=True)
            if agg == "mean":
                return da.mean("time", keep_attrs=True)
            return da
        res = execute(spec, lambda sp_, dev: sp_.cells(timesum=agg is not None))
        meta = res[0][1]
        coords_yx = {"y": _coord(ds, "y"), "x": _coord(ds, "x")}
        attrs = {"units": meta.units} if meta.units else {}
        if agg is None:
            vals, labels = _joined(res)
            vals = _to_host(vals)
            if shard is not None:
                vals, labels = shard.gather_time(vals, labels)
            return make_dataarray(vals, ("time", "y", "x"), {"time": labels, **coords_yx}, attrs, meta.name)
        # NaN-skipping time sum and the number of valid steps per cell (da.sum / da.mean
        # over "time" skip NaN, convert.py:51-56; an all-NaN cell has mean NaN, sum 0)
        planes = [(v[0], v[1]) for v, _ in res]
        if shard is not None:
            planes = [shard.sum_planes(*planes[0])]
        total = sum(_to_host(t).astype(np.float64) for t, _ in planes)
        if agg == "mean":
            count = sum(_to_host(c).astype(np.float64) for _, c in planes)
            with np.errstate(divide="ignore", invalid="ignore"):
                total = np.where(count > 0, total / count, np.nan)
        return make_dataarray(total, ("y", "x"), coords_yx, attrs, meta.name)

    matrix, dim, idx = _aggregation_matrix(cutout, ds, matrix, index, layout, shapes, shapes_crs)
    if da is not None:
        spec = _PluginSpec(da)
    digest = engine.matrix_digest(matrix)
    res = execute(spec, lambda sp_, dev: sp_.reduce(engine.get_plan(matrix, ny, nx, device=dev, pitch=sp_.pitch,
                                                              digest=digest)))  # (time, bus) float32
    name = res[0][1].name
    res, time_labels = _joined(res)
    if shard is not None:
        res, time_labels = shard.gather_time(res, time_labels)
    capacity = caps = None
    if per_unit or return_capacity:
        caps = np.asarray(matrix.sum(-1)).flatten()
        capacity = make_dataarray(caps, (dim,), {dim: idx}, {"units": "MW"})
    units = "p.u." if per_unit else "MW"

    # dim order mirrors aggregate.py: (time, bus) for dask-backed cutouts
    # (:24-32), (bus, time) for NumPy-backed ones (:34-35)
    agg = aggregate_time if aggregate_time != "legacy" else None
    bus_major = agg is None and not lazy
    results = _finish_results(res, caps if per_unit else None, agg, bus_major)
    if agg is not None:
        out = make_dataarray(results, (dim,), {dim: idx}, {"units": units}, name)
    elif not bus_major:
        out = make_dataarray(results, ("time", dim), {"time": time_labels, dim: idx}, {"units": units}, name)
    else:
        out = make_dataarray(results, (dim, "time"), {dim: idx, "time": time_labels}, {"units": units}, name)
    if return_capacity:
        return out, capacity
    return out


# --------------------------------------------------------------------------
# technology wrappers
# --------------------------------------------------------------------------


def heat_demand(cutout, threshold=15.0, a=1.0, constant=0.0, hour_shift=0.0, **params):
    """Daily heat demand by the degree-day approximation (convert.py:421-471)."""
    return cutout.convert_and_aggregate(
        convert_func=convert_heat_demand,
        threshold=threshold,
        a=a,
        constant=constant,
        hour_shift=hour_shift,
        **params,
    )


def wind(cutout, turbine, smooth=False, add_cutout_windspeed=False,
         interpolation_method="logarithmic", **params):
    """Wind generation time-series (convert.py:665-744)."""
    turbine = get_windturbineconfig(turbine, add_cutout_windspeed=add_cutout_windspeed)
    if smooth:
        turbine = windturbine_smooth(turbine, params=smooth)
    return cutout.convert_and_aggregate(
        convert_func=convert_wind,
        turbine=turbine,
        interpolation_method=interpolation_method,
        **params,
    )


def pv(cutout, panel, orientation, tracking=None, clearsky_model=None, **params):
    """PV generation time-series (convert.py:857-936)."""
    if isinstance(panel, (str, Path)):
        panel = get_solarpanelconfig(panel)
    if not callable(orientation):
        orientation = get_orientation(orientation)
    return cutout.convert_and_aggregate(
        convert_func=convert_pv,
        panel=panel,
        orientation=orientation,
        tracking=tracking,
        clearsky_model=clearsky_model,
        **params,
    )


# --------------------------------------------------------------------------
# further technology wrappers on the same path (SURVEY.md section 8 f3)
# --------------------------------------------------------------------------


def temperature(cutout, **params):
    """convert.py:301-302"""
    return cutout.convert_and_aggregate(convert_func=convert_temperature, **params)


def soil_temperature(cutout, **params):
    """convert.py:319-320"""
    return cutout.convert_and_aggregate(convert_func=convert_soil_temperature, **params)


def dewpoint_temperature(cutout, **params):
    """convert.py:332-335"""
    return cutout.convert_and_aggregate(convert_func=convert_dewpoint_temperature, **params)


def coefficient_of_performance(cutout, source="air", sink_T=55.0, c0=None, c1=None, c2=None, **params):
    """Air- or ground-sourced heat pump COP (convert.py:369-401)."""
    return cutout.convert_and_aggregate(
        convert_func=convert_coefficient_of_performance,
        source=source, sink_T=sink_T, c0=c0, c1=c1, c2=c2, **params,
    )


def cooling_demand(cutout, threshold=23.0, a=1.0, constant=0.0, hour_shift=0.0, **params):
    """Daily cooling demand by the degree-day approximation (convert.py:494-546)."""
    return cutout.convert_and_aggregate(
        convert_func=convert_cooling_demand,
        threshold=threshold, a=a, constant=constant, hour_shift=hour_shift, **params,
    )


def solar_thermal(cutout, orientation={"slope": 45.0, "azimuth": 180.0}, trigon_model="simple",
                  clearsky_model="simple", c0=0.8, c1=3.0, t_store=80.0, **params):
    """Solar thermal collector time series (convert.py:576-630)."""
    if not callable(orientation):
        orientation = get_orientation(orientation)
    return cutout.convert_and_aggregate(
        convert_func=convert_solar_thermal,
        orientation=orientation, trigon_model=trigon_model, clearsky_model=clearsky_model,
        c0=c0, c1=c1, t_store=t_store, **params,
    )


def irradiation(cutout, orientation, irradiation="total", tracking=None, clearsky_model=None, **params):
    """Total / direct / diffuse / ground irradiation on a tilted surface (convert.py:770-836)."""
    if not callable(orientation):
        orientation = get_orientation(orientation)
    return cutout.convert_and_aggregate(
        convert_func=convert_irradiation,
        orientation=orientation, tracking=tracking, irradiation=irradiation,
        clearsky_model=clearsky_model, **params,
    )


def csp(cutout, installation, technology=None, **params):
    """CSP generation time-series from direct radiation (convert.py:975-1024)."""
    if isinstance(installation, (str, Path)):
        installation = get_cspinstallationconfig(installation)
    if technology is not None:
        installation = dict(installation, technology=technology)
    return cutout.convert_and_aggregate(convert_func=convert_csp, installation=installation, **params)


def runoff(cutout, smooth=None, lower_threshold_quantile=None, normalize_using_yearly=None, **params):
    """Runoff aggregated to buses with the reference's optional post-processing
    (rolling mean, lower-quantile cut, yearly normalisation; convert.py:1037-1084)."""
    result = cutout.convert_and_aggregate(convert_func=convert_runoff, **params)
    res, cap = (result if isinstance(result, tuple) else (result, None))
    if "time" not in res.dims or (smooth is None and lower_threshold_quantile is None
                                  and normalize_using_yearly is None):
        return result
    tax = list(res.dims).index("time")
    vals = np.asarray(res.values, dtype=np.float64)
    if smooth is not None:
        if smooth is True:
            smooth = 24 * 7
        frame = pd.DataFrame(np.moveaxis(vals, tax, 0).reshape(vals.shape[tax], -1))
        sm = frame.rolling(smooth, min_periods=1).mean().values
        vals = np.moveaxis(sm.reshape(np.moveaxis(vals, tax, 0).shape), 0, tax)
    if lower_threshold_quantile is not None:
        if lower_threshold_quantile is True:
            lower_threshold_quantile = 5e-3
        lower = pd.Series(vals.ravel()).quantile(lower_threshold_quantile)
        vals = np.where(vals >= lower, vals, 0.0)
    if normalize_using_yearly is not None:
        idx = normalize_using_yearly.index
        idx = idx.year if isinstance(idx, pd.DatetimeIndex) else idx.astype(int)
        tyears = pd.DatetimeIndex(np.asarray(res.coords["time"])).year
        full = pd.Series(tyears).value_counts().loc[lambda x: x > 8700].index.intersection(idx)
        assert len(full), "Need at least a full year of data (more is better)"
        sel = (tyears >= min(full)) & (tyears <= max(full))
        norm = normalize_using_yearly.copy()
        norm.index = idx
        target = norm.loc[min(full):max(full)].sum()
        other = [d for d in res.dims if d != "time"][0]
        target = target.reindex(pd.Index(np.asarray(res.coords[other]))).values
        have = np.take(vals, np.flatnonzero(sel), axis=tax).sum(axis=tax)
        factor = target / have
        vals = vals * (factor[:, None] if tax == 1 else factor[None, :])
    out = make_dataarray(vals, tuple(res.dims), {d: np.asarray(res.coords[d]) for d in res.dims},
                         dict(res.attrs), getattr(res, "name", None))
    return (out, cap) if cap is not None else out
