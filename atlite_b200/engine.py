"""Handle wrappers over the C ABI: aggregation plans and the pv / wind / heat
operators.  Arrays may be NumPy (host) or torch CUDA tensors (device-resident
cutout); host arrays go through the library's streaming entry points
(``atl_*_reduce_host``), device tensors through the kernel entry points.
"""

from __future__ import annotations

import ctypes as C
import threading
from collections import OrderedDict

import numpy as np
import pandas as pd
import scipy.sparse as sp

from . import _lib


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _torch():
    import torch

    return torch


def current_device():
    try:
        torch = _torch()
        if torch.cuda.is_available():
            return torch.cuda.current_device()
    except Exception:  # noqa: BLE001
        pass
    return 0


def _stream_ptr():
    torch = _torch()
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _dptr(x):
    if x is None:
        return None
    if _is_torch(x):
        assert x.is_cuda and x.is_contiguous()
        return C.c_void_p(x.data_ptr())
    raise TypeError("device pointer requested for a non-torch array")


def _hptr(x):
    if x is None:
        return None
    assert isinstance(x, np.ndarray) and x.flags["C_CONTIGUOUS"]
    return C.c_void_p(x.ctypes.data)


def host_f32(a):
    """C-contiguous float32 view/copy of a host array."""
    a = np.asarray(a)
    if a.dtype != np.float32 or not a.flags["C_CONTIGUOUS"]:
        a = np.ascontiguousarray(a, dtype=np.float32)
    return a


def pitch_of(arrays, nx):
    """Row pitch (elements) of a set of (time, y, x) fields: the last dimension of
    device tensors (``Cutout.to_device`` pads rows to a multiple of 4), ``nx`` for
    host arrays."""
    p = None
    for a in arrays:
        if a is None or getattr(a, "ndim", 0) != 3:
            continue
        w = int(a.shape[-1])
        if p is not None and w != p:
            raise ValueError("fields of one call must share the same row pitch")
        p = w
    p = nx if p is None else p
    if p < nx:
        raise ValueError(f"fields are narrower ({p}) than the grid ({nx})")
    if p != nx and not any(_is_torch(a) for a in arrays if a is not None):
        raise ValueError("host arrays must be unpadded (last dimension == nx)")
    return p


def time_ns(time):
    """datetime-like sequence -> contiguous int64 nanoseconds since the epoch (UTC)."""
    idx = pd.DatetimeIndex(np.asarray(time))
    return np.ascontiguousarray(idx.as_unit("ns").asi8, dtype=np.int64)


class Plan:
    """Device-side aggregation plan built from an (n_bus, S) CSR matrix."""

    def __init__(self, matrix, ny, nx, device=None, pitch=None):
        lib = _lib.load()
        m = sp.csr_matrix(matrix)
        m.sum_duplicates()
        if m.shape[1] != ny * nx:
            raise ValueError(
                f"matrix has {m.shape[1]} columns but the cutout grid has {ny}x{nx}={ny * nx} cells"
            )
        self.shape = m.shape
        self.grid = (ny, nx)
        self.device = current_device() if device is None else device
        self._indptr = np.ascontiguousarray(m.indptr, dtype=np.int64)
        self._indices = np.ascontiguousarray(m.indices, dtype=np.int32)
        self._data = np.ascontiguousarray(m.data, dtype=np.float64)
        h = C.c_void_p()
        self.pitch = nx if pitch is None else int(pitch)
        _lib.check(
            lib.atl_plan_create_pitched(
                self.device, ny, nx, self.pitch, m.shape[0],
                _lib.ptr(self._indptr), _lib.ptr(self._indices), _lib.ptr(self._data),
                C.byref(h),
            )
        )
        self.handle = h
        info = _lib.PlanInfo()
        _lib.check(lib.atl_plan_info(h, C.byref(info)))
        self.info = {f[0]: getattr(info, f[0]) for f in _lib.PlanInfo._fields_}
        self.n_bus = m.shape[0]

    def __del__(self):
        h = getattr(self, "handle", None)
        if h:
            try:
                _lib.load().atl_plan_destroy(h)
            except Exception:  # noqa: BLE001
                pass
            self.handle = None

    def spmm(self, dense):
        """(nt, ny, nx) | (nt, S) per-cell values (host or device) -> (nt, n_bus) float32."""
        torch = _torch()
        if not _is_torch(dense):
            dense = torch.from_numpy(host_f32(dense)).to(f"cuda:{self.device}")
        dense = dense.contiguous().to(torch.float32)
        nt = dense.shape[0]
        ny, nx = self.grid
        ok = (dense.ndim == 3 and tuple(dense.shape[1:]) == (ny, self.pitch)) or \
             (dense.ndim == 2 and dense.shape[1] == ny * self.pitch)
        if not ok:
            raise ValueError(f"per-cell values have shape {tuple(dense.shape)}; this plan expects "
                             f"(time, {ny}, {self.pitch}) or (time, {ny * self.pitch})")
        if dense.device.type != "cuda" or dense.device.index != self.device:
            raise ValueError(f"per-cell values live on {dense.device}, the plan on cuda:{self.device}")
        out = torch.zeros((nt, self.n_bus), dtype=torch.float32, device=dense.device)
        if nt == 0:
            return out
        _lib.check(_lib.load().atl_spmm(self.handle, _dptr(dense), nt, _dptr(out), _stream_ptr()))
        return out


_PLAN_CACHE: "OrderedDict[tuple, Plan]" = OrderedDict()
_PLAN_LOCK = threading.Lock()
_PLAN_CACHE_SIZE = 4  # per device


def matrix_digest(m):
    """Content key of a CSR matrix for the plan cache: three 128-bit hashes (indptr, indices,
    data; ``atl_hash128``) next to shape, nnz and dtypes.  A collision would silently reuse a
    wrong plan, hence 3 x 128 bits; the hash sits on the critical path of every call, hence
    not hashlib (blake2b: 23 ms for the 15 MB of 1440 x 720 -> 3000 shapes; this: ~3 ms)."""
    lib = _lib.load()
    parts = []
    for seed, a in enumerate((m.indptr, m.indices, m.data)):
        b = np.ascontiguousarray(a)
        out = (C.c_uint64 * 2)()
        _lib.check(lib.atl_hash128(b.ctypes.data_as(C.c_void_p), b.nbytes, seed, out))
        parts += [int(out[0]), int(out[1]), b.nbytes, str(b.dtype)]
    return (m.shape, m.nnz, tuple(parts))


def get_plan(matrix, ny, nx, device=None, pitch=None, digest=None):
    """Plans are cached (LRU, 4 entries per device): the typical workflow evaluates many
    technologies against the same shapes.  Thread-safe (one host thread per GPU in the
    single-process multi-GPU path); ``digest`` = a precomputed ``matrix_digest``."""
    m = sp.csr_matrix(matrix)
    device = current_device() if device is None else device
    pitch = nx if pitch is None else int(pitch)
    key = (device, ny, nx, pitch) + (matrix_digest(m) if digest is None else digest)
    with _PLAN_LOCK:
        plan = _PLAN_CACHE.get(key)
        if plan is not None:
            _PLAN_CACHE.move_to_end(key)
            return plan
    plan = Plan(m, ny, nx, device, pitch)  # built outside the lock: devices build concurrently
    with _PLAN_LOCK:
        _PLAN_CACHE[key] = plan
        mine = [k for k in _PLAN_CACHE if k[0] == device]
        for k in mine[:-_PLAN_CACHE_SIZE]:
            del _PLAN_CACHE[k]
    return plan


def _first(fields):
    return next(a for a in fields.values() if a is not None)


class _Op:
    """A fused operator, ``atl_<_name>_*`` of the C ABI.  A subclass declares its fields:
    ``_struct`` is the ctypes struct of field pointers (None: one bare field pointer) and
    ``_f64`` the fields that may be float64 (stored solar position).  ``_slab`` forms the
    arguments that follow the fields in the C call."""

    _name = None
    _struct = None
    _f64 = ()

    def _bind(self, ny, nx, device, pitch):
        _lib.load()
        self.device = current_device() if device is None else device
        self.ny, self.nx = ny, nx
        self.pitch = int(pitch) or nx

    def _create(self, cfg):
        h = C.c_void_p()
        _lib.check(getattr(_lib.load(), f"atl_{self._name}_create")(self.device, C.byref(cfg), C.byref(h)))
        self.handle = h

    def __del__(self):
        h = getattr(self, "handle", None)
        if h:
            try:
                getattr(_lib.load(), f"atl_{self._name}_destroy")(h)
            except Exception:  # noqa: BLE001
                pass
            self.handle = None

    @staticmethod
    def _all_device(arrs):
        kinds = {_is_torch(a) for a in arrs if a is not None}
        if len(kinds) > 1:
            raise ValueError("mixing host (NumPy) and device (torch) fields in one call")
        return kinds.pop() if kinds else False

    def _dev(self, a, f64_ok=False):
        """Device field -> contiguous tensor, after checking what the kernels assume
        about it: (time, ny, pitch) layout on this operator's GPU, float32 (float64
        for stored solar position).  The C ABI takes raw pointers, so this is the
        only place a wrong shape can be caught."""
        torch = _torch()
        if a.ndim != 3 or tuple(a.shape[1:]) != (self.ny, self.pitch):
            raise ValueError(f"field has shape {tuple(a.shape)}, expected (time, {self.ny}, {self.pitch})")
        if a.dtype != torch.float32 and not (f64_ok and a.dtype == torch.float64):
            raise TypeError(f"device fields must be float32, got {a.dtype}")
        if a.device.type != "cuda" or a.device.index != self.device:
            raise ValueError(f"field lives on {a.device}, operator on cuda:{self.device}")
        return a.contiguous()

    def _host(self, a, f64_ok=False):
        a = np.asarray(a)
        if a.ndim != 3 or a.shape[1:] != (self.ny, self.nx):
            raise ValueError(f"field has shape {a.shape}, expected (time, {self.ny}, {self.nx})")
        if f64_ok and a.dtype == np.float64:
            return np.ascontiguousarray(a)
        return host_f32(a)

    def _pack(self, fields, dev):
        """Checked fields -> (the C call's field argument, the arrays it points into)."""
        check, ptr = (self._dev, _dptr) if dev else (self._host, _hptr)
        names = list(fields) if self._struct is None else [n for n, _ in self._struct._fields_]
        keep = {n: check(fields[n], f64_ok=n in self._f64) for n in names if fields.get(n) is not None}
        if self._struct is None:
            (a,) = keep.values()
            return ptr(a), keep
        f = self._struct()
        for n in names:
            setattr(f, n, ptr(keep[n]).value if n in keep else None)
        return C.byref(f), keep

    def _call(self, kind, fields, slab, n, plan=None, chunk=0):
        """``atl_<op>_<kind>`` on ``fields`` (name -> (time, y, x) array or None), ``slab`` = the
        arguments after the fields, ``n`` = output steps.  kind "reduce": (n, n_bus) float32,
        a torch CUDA tensor for device fields, an ndarray for host fields (``*_reduce_host``
        streams them in slabs of ``chunk``); "cells": (n, ny, nx); "timesum": (2, ny, nx) =
        NaN-skipping sum | valid steps.  Per-cell outputs take device fields only."""
        dev = self._all_device(fields.values()) if kind == "reduce" else True
        first = _first(fields)
        shape = (2, self.ny, self.nx) if kind == "timesum" else \
            (n, plan.n_bus) if kind == "reduce" else (n, self.ny, self.nx)
        if n == 0 or first.shape[0] == 0:
            # e.g. a rank whose time shard is empty: no kernel is launched (empty tensors
            # have NULL data pointers)
            if _is_torch(first):
                torch = _torch()
                return torch.zeros(shape, dtype=torch.float32, device=first.device)
            return np.zeros(shape, dtype=np.float32)
        arg, keep = self._pack(fields, dev)
        head = (self.handle, plan.handle) if kind == "reduce" else (self.handle,)
        if not dev:
            out = np.empty(shape, dtype=np.float32)
            _lib.check(getattr(_lib.load(), f"atl_{self._name}_reduce_host")(*head, arg, *slab, _hptr(out), chunk))
            return out
        torch = _torch()
        if kind == "timesum":
            out = torch.zeros(shape, dtype=torch.float32, device=first.device)
            outs = (_dptr(out[0]), _dptr(out[1]))
        else:
            out = torch.empty(shape, dtype=torch.float32, device=first.device)
            outs = (_dptr(out),)
        _lib.check(getattr(_lib.load(), f"atl_{self._name}_{kind}")(*head, arg, *slab, *outs, _stream_ptr()))
        return out

    def _slab(self, fields):
        """(the C call's arguments after the fields, output steps) for whole fields."""
        nt = _first(fields).shape[0]
        return (nt,), nt

    def reduce(self, plan, fields, chunk_steps=0):
        slab, n = self._slab(fields)
        return self._call("reduce", fields, slab, n, plan, chunk_steps)

    def cells(self, fields, timesum=False):
        """Per-cell values (nt, ny, nx) or their time sum (2, ny, nx); device fields only."""
        slab, n = self._slab(fields)
        return self._call("timesum" if timesum else "cells", fields, slab, n)


class PvOp(_Op):
    """convert_pv (convert.py:840-854) operator; see include/atlite_b200.h."""

    _name, _struct, _f64 = "pv", _lib.PvFields, ("solar_altitude", "solar_azimuth")

    def __init__(self, *, ny, nx, time, lon, lat, slope, azimuth, tracking, trigon_model,
                 clearsky_model, irr_branch, albedo_src, solar_src, panel=None, time_shift="0h",
                 altitude_threshold=1.0, output="panel", thermal=(0.0, 0.0, 0.0), device=None, pitch=0):
        self._bind(ny, nx, device, pitch)
        self._time = time_ns(time)
        self.nt = len(self._time)
        self._lon, self._lat = _lib.as_f64(lon), _lib.as_f64(lat)
        slope, azimuth = np.asarray(slope, dtype=np.float64), np.asarray(azimuth, dtype=np.float64)
        self.orientation_2d = slope.ndim == 2 or azimuth.ndim == 2
        oshape = (ny, nx) if self.orientation_2d else (ny,)
        # (ny,) tables broadcast along x when the other one is 2-D
        self._slope = np.ascontiguousarray(np.broadcast_to(slope[:, None] if (self.orientation_2d and slope.ndim == 1) else slope, oshape))
        self._az = np.ascontiguousarray(np.broadcast_to(azimuth[:, None] if (self.orientation_2d and azimuth.ndim == 1) else azimuth, oshape))
        cfg = _lib.PvConfig()
        cfg.ny, cfg.nx, cfg.nt = ny, nx, self.nt
        cfg.time_ns = _lib.ptr(self._time).value
        cfg.time_shift_ns = int(pd.to_timedelta(time_shift).value)
        cfg.lon_deg, cfg.lat_deg = _lib.ptr(self._lon).value, _lib.ptr(self._lat).value
        cfg.slope_rad, cfg.azimuth_rad = _lib.ptr(self._slope).value, _lib.ptr(self._az).value
        cfg.tracking = _lib.TRACKING[tracking]
        cfg.trigon_model = trigon_model
        cfg.clearsky_model = clearsky_model
        cfg.irr_branch, cfg.albedo_src, cfg.solar_src = irr_branch, albedo_src, solar_src
        cfg.pitch = int(pitch)
        cfg.orientation_2d = 1 if self.orientation_2d else 0
        cfg.output = _lib.OUTPUT[output]
        for i, v in enumerate(thermal):
            cfg.thermal[i] = float(v)
        cfg.altitude_threshold_deg = altitude_threshold
        model = "huld" if panel is None else panel.get("model", "huld")
        if model not in _lib.PANEL:
            raise AssertionError(f"Unknown panel model: {model}")
        cfg.panel_model = _lib.PANEL[model]
        if panel is None:
            vals = []
        elif model == "huld":
            vals = [panel["c_temp_amb"], panel["c_temp_irrad"], panel["r_tmod"], panel["r_irradiance"]]
            vals += [panel[f"k_{i}"] for i in range(1, 7)]
            vals += [panel.get("inverter_efficiency", 1.0)]
        else:
            vals = [panel[k] for k in ("A", "B", "C", "D", "NOCT", "Tamb", "Intc", "Tstd", "ta", "threshold")]
            vals += [panel.get("inverter_efficiency", 1.0)]
        for i, v in enumerate(vals):
            cfg.panel[i] = float(v)
        self._create(cfg)

    def reduce(self, plan, fields, t0=0, nt=None, chunk_steps=0):
        """(nt, n_bus) float32: torch CUDA tensor for device fields, ndarray for host fields."""
        nt = _first(fields).shape[0] if nt is None else nt
        return self._call("reduce", fields, (t0, nt), nt, plan, chunk_steps)

    def _slab(self, fields):
        nt = _first(fields).shape[0]
        return (0, nt), nt


class WindOp(_Op):
    """convert_wind (convert.py:634-662) operator."""

    _name, _struct = "wind", _lib.WindFields

    def __init__(self, *, ny, nx, V, POW_norm, method, from_height, to_height, device=None, pitch=0):
        self._bind(ny, nx, device, pitch)
        self._V, self._P = _lib.as_f64(V), _lib.as_f64(POW_norm)
        cfg = _lib.WindConfig()
        cfg.ny, cfg.nx, cfg.method = ny, nx, method
        cfg.from_height, cfg.to_height = float(from_height), float(to_height)
        cfg.pitch = int(pitch)
        cfg.n_knots = len(self._V)
        cfg.V, cfg.POW_norm = _lib.ptr(self._V).value, _lib.ptr(self._P).value
        self._create(cfg)

    def reduce(self, plan, wnd, aux=None, chunk_steps=0):
        return super().reduce(plan, {"wnd": wnd, "aux": aux}, chunk_steps)


class HeatOp(_Op):
    """convert_heat_demand (convert.py:405-418) operator."""

    _name = "heat"

    def __init__(self, *, ny, nx, threshold, a, constant, cooling=False, device=None, pitch=0):
        self._bind(ny, nx, device, pitch)
        cfg = _lib.HeatConfig()
        cfg.ny, cfg.nx = ny, nx
        cfg.threshold_c, cfg.a, cfg.constant = float(threshold), float(a), float(constant)
        cfg.cooling = 1 if cooling else 0
        cfg.pitch = int(pitch)
        self._create(cfg)

    def reduce(self, plan, temperature, day_start, chunk_days=0):
        ds = np.ascontiguousarray(day_start, dtype=np.int64)
        return self._call("reduce", {"temperature": temperature}, (_lib.ptr(ds), len(ds) - 1), len(ds) - 1,
                          plan, chunk_days)

    def cells(self, fields, day_start, timesum=False):
        ds = np.ascontiguousarray(day_start, dtype=np.int64)
        return self._call("timesum" if timesum else "cells", fields, (_lib.ptr(ds), len(ds) - 1), len(ds) - 1)


class PointwiseOp(_Op):
    """Pointwise function of one field (temperature family, COP, runoff x height);
    see include/atlite_b200.h."""

    _name = "pointwise"

    def __init__(self, *, ny, nx, shift=0.0, nan_to_zero=False, poly=None, cell_scale=None, device=None, pitch=0):
        self._bind(ny, nx, device, pitch)
        cfg = _lib.PointwiseConfig()
        cfg.ny, cfg.nx = ny, nx
        cfg.shift = float(shift)
        cfg.pitch = int(pitch)
        cfg.nan_to_zero = 1 if nan_to_zero else 0
        cfg.poly = 0 if poly is None else 1
        if poly is not None:
            cfg.sink, cfg.c0, cfg.c1, cfg.c2 = (float(v) for v in poly)
        self._scale = None
        if cell_scale is not None:
            self._scale = host_f32(cell_scale)
            if self._scale.shape != (ny, nx):
                raise ValueError(f"cell_scale must have shape {(ny, nx)}, has {self._scale.shape}")
            cfg.cell_scale = self._scale.ctypes.data
        self._create(cfg)


class CspOp(_Op):
    """convert_csp (convert.py:940-972) operator."""

    _name, _struct, _f64 = "csp", _lib.CspFields, ("solar_altitude", "solar_azimuth")

    def __init__(self, *, ny, nx, time, lon, lat, solar_src, technology, r_irradiance, altitude, azimuth,
                 efficiency, time_shift="0h", dni_altitude_threshold=3.75, device=None, pitch=0):
        self._bind(ny, nx, device, pitch)
        self._time = time_ns(time)
        self._lon, self._lat = _lib.as_f64(lon), _lib.as_f64(lat)
        self._alt, self._az, self._eff = _lib.as_f64(altitude), _lib.as_f64(azimuth), _lib.as_f64(efficiency)
        cfg = _lib.CspConfig()
        cfg.ny, cfg.nx, cfg.nt = ny, nx, len(self._time)
        cfg.time_ns = _lib.ptr(self._time).value
        cfg.time_shift_ns = int(pd.to_timedelta(time_shift).value)
        cfg.lon_deg, cfg.lat_deg = _lib.ptr(self._lon).value, _lib.ptr(self._lat).value
        cfg.solar_src = solar_src
        cfg.pitch = int(pitch)
        cfg.technology = technology
        cfg.r_irradiance = float(r_irradiance)
        cfg.dni_altitude_threshold_deg = float(dni_altitude_threshold)
        cfg.n_alt, cfg.n_az = len(self._alt), len(self._az)
        cfg.altitude_rad, cfg.azimuth_rad = _lib.ptr(self._alt).value, _lib.ptr(self._az).value
        cfg.efficiency = _lib.ptr(self._eff).value
        self._create(cfg)

    _slab = PvOp._slab  # t0 = 0, nt
