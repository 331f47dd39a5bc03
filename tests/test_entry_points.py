"""The C entry points of the five fused operators share one call sequence: every argument
check, then the device, then the launch.

CPU part: a malformed call is refused with ATL_ERR_INVALID and its message before the
library touches the device.  Heat and pointwise operators (without ``cell_scale``) are
created without any CUDA call, so this runs on a machine without a GPU.  No plan pointer is
ever made up here: with no device there is no real plan to point at.

GPU part: kernel launches per call for every operator and entry kind on a tiling plan, the
same plan in deterministic mode and a plan that does not tile (two-pass fallback); and a
host entry point refusing a row-padded operator.
"""

import ctypes as C

import numpy as np
import pandas as pd
import pytest
import scipy.sparse as sp

import atlite_b200 as ab
from atlite_b200 import _lib, engine, synthetic as syn

ATL_ERR_INVALID = -1
NY, NX, NT = 40, 64, 48


def _invalid(rc, message):
    assert rc == ATL_ERR_INVALID, (rc, _lib.load().atl_last_error())
    assert _lib.load().atl_last_error().decode() == message


@pytest.fixture
def heat_op():
    cfg = _lib.HeatConfig()
    cfg.ny, cfg.nx, cfg.threshold_c, cfg.a = NY, NX, 15.0, 1.0
    h = C.c_void_p()
    assert _lib.load().atl_heat_create(0, C.byref(cfg), C.byref(h)) == 0
    yield h
    _lib.load().atl_heat_destroy(h)


@pytest.fixture
def pointwise_op():
    cfg = _lib.PointwiseConfig()
    cfg.ny, cfg.nx = NY, NX
    h = C.c_void_p()
    assert _lib.load().atl_pointwise_create(0, C.byref(cfg), C.byref(h)) == 0
    yield h
    _lib.load().atl_pointwise_destroy(h)


# host buffers stand in for the valid arguments: every call below is refused before any is read
FIELD = np.zeros((NT, NY, NX), np.float32)
OUT = np.zeros((2, NY, NX), np.float32)
DAYS = np.array([0, 24, 48], np.int64)
NOT_MONOTONE = np.array([0, 30, 24], np.int64)


def _p(a):
    return None if a is None else a.ctypes.data


@pytest.mark.parametrize("kind", ["cells", "timesum"])
@pytest.mark.parametrize("fault", ["field", "out", "days", "not_monotone"])
def test_heat_per_cell_refusals(heat_op, kind, fault):
    field = None if fault == "field" else FIELD
    out = None if fault == "out" else OUT
    days = None if fault == "days" else NOT_MONOTONE if fault == "not_monotone" else DAYS
    fn = getattr(_lib.load(), f"atl_heat_{kind}")
    args = [heat_op, _p(field), _p(days), 2, _p(out)] + ([_p(OUT[1])] if kind == "timesum" else []) + [None]
    _invalid(fn(*args), "day offsets not monotone" if fault == "not_monotone" else "NULL argument")


@pytest.mark.parametrize("kind", ["cells", "timesum"])
@pytest.mark.parametrize("fault", ["field", "out"])
def test_pointwise_per_cell_refusals(pointwise_op, kind, fault):
    field = None if fault == "field" else FIELD
    out = None if fault == "out" else OUT
    fn = getattr(_lib.load(), f"atl_pointwise_{kind}")
    args = [pointwise_op, _p(field), NT, _p(out)] + ([_p(OUT[1])] if kind == "timesum" else []) + [None]
    _invalid(fn(*args), "NULL argument")


def test_reduce_without_plan_is_refused(heat_op, pointwise_op):
    lib = _lib.load()
    red = np.zeros((NT, 3), np.float32)
    _invalid(lib.atl_heat_reduce(heat_op, None, _p(FIELD), _p(DAYS), 2, _p(red), None), "NULL plan")
    _invalid(lib.atl_heat_reduce_host(heat_op, None, _p(FIELD), _p(DAYS), 2, _p(red), 0), "NULL argument")
    _invalid(lib.atl_pointwise_reduce(pointwise_op, None, _p(FIELD), NT, _p(red), None), "NULL argument")
    _invalid(lib.atl_pointwise_reduce_host(pointwise_op, None, _p(FIELD), NT, _p(red), 0), "NULL argument")


# ---------------------------------------------------------------- GPU


def _operators(time):
    lon = np.linspace(0.0, 16.0, NX)
    lat = np.linspace(30.0, 40.0, NY)
    return {
        "pv": engine.PvOp(ny=NY, nx=NX, time=time, lon=lon, lat=lat, slope=np.full(NY, 0.5),
                          azimuth=np.full(NY, np.pi), tracking=None, trigon_model=0, clearsky_model=0,
                          irr_branch=0, albedo_src=0, solar_src=0, panel=ab.get_solarpanelconfig("CSi")),
        "wind": engine.WindOp(ny=NY, nx=NX, V=[0.0, 3.0, 12.0, 25.0, 25.0], POW_norm=[0.0, 0.0, 1.0, 1.0, 0.0],
                              method=_lib.WIND_LOG, from_height=100.0, to_height=100.0),
        "heat": engine.HeatOp(ny=NY, nx=NX, threshold=15.0, a=1.0, constant=0.0),
        "pointwise": engine.PointwiseOp(ny=NY, nx=NX, shift=-273.15),
        "csp": engine.CspOp(ny=NY, nx=NX, time=time, lon=lon, lat=lat, solar_src=0, technology=0,
                            r_irradiance=950.0, altitude=np.linspace(0.0, 1.5, 4),
                            azimuth=np.linspace(0.0, 6.0, 4), efficiency=np.full(16, 0.5)),
    }


def _fields(name, make):
    one = lambda: make(np.random.default_rng(0).uniform(1.0, 300.0, (NT, NY, NX)).astype(np.float32))  # noqa: E731
    return {
        "pv": lambda: {k: one() for k in ("influx_toa", "influx_direct", "influx_diffuse", "albedo", "temperature")},
        "wind": lambda: {"wnd": one(), "aux": one()},
        "heat": lambda: {"temperature": one()},
        "pointwise": lambda: {"temperature": one()},
        "csp": lambda: {"influx_direct": one()},
    }[name]()


def _run(op, name, kind, fields, plan):
    if name == "heat":
        if kind == "reduce":
            return op.reduce(plan, fields["temperature"], DAYS)
        return op.cells(fields, DAYS, timesum=kind == "timesum")
    if kind == "reduce":
        return op.reduce(plan, fields) if name != "wind" else op.reduce(plan, fields["wnd"], fields["aux"])
    return op.cells(fields, timesum=kind == "timesum")


# kernel launches of one call: the fused kernel; + the slot gather in deterministic mode; the
# per-cell kernel + the CSR gather for a plan that does not tile; one kernel per per-cell call
LAUNCHES = {"tiling": 1, "deterministic": 2, "two_pass": 2, "cells": 1, "timesum": 1}


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["pv", "wind", "heat", "pointwise", "csp"])
def test_launches_per_call(name):
    import torch

    ops = _operators(pd.date_range("2013-06-01", periods=NT, freq="h"))
    op = ops[name]
    tiling = engine.Plan(syn.make_shapes(NX, NY, 12), NY, NX)
    identity = engine.Plan(sp.identity(NY * NX, format="csr"), NY, NX)
    assert tiling.info["fused"] == 1 and identity.info["fused"] == 0
    dev = _fields(name, lambda a: torch.from_numpy(a).cuda())
    host = _fields(name, lambda a: a)
    got = {}
    for where, fields in (("device", dev), ("host", host)):
        for plan_name, plan in (("tiling", tiling), ("deterministic", tiling), ("two_pass", identity)):
            prev = ab.set_deterministic(plan_name == "deterministic")
            try:
                torch.cuda.synchronize()
                n0 = _lib.launch_count()
                _run(op, name, "reduce", fields, plan)
                got[f"{where} reduce {plan_name}"] = _lib.launch_count() - n0
            finally:
                ab.set_deterministic(prev)
    for kind in ("cells", "timesum"):
        n0 = _lib.launch_count()
        _run(op, name, kind, dev, None)
        got[kind] = _lib.launch_count() - n0
    torch.cuda.synchronize()
    want = {k: LAUNCHES[k.split()[-1]] for k in got}
    assert got == want


@pytest.mark.gpu
def test_host_entry_refuses_padded_operator():
    """The host ring holds ny * nx elements per step, the kernels index a padded operator's
    fields with ny * pitch.  The plan is empty, so no kernel would read a field even if the
    refusal were missing."""
    pitch = NX + 2
    op = engine.PointwiseOp(ny=NY, nx=NX, pitch=pitch)
    plan = engine.Plan(sp.csr_matrix((3, NY * NX)), NY, NX, pitch=pitch)
    assert plan.info["fused"] == 1 and plan.info["n_active_tiles"] == 0
    field = np.zeros((NT, NY, pitch), np.float32)
    out = np.full((NT, 3), np.nan, np.float32)
    rc = _lib.load().atl_pointwise_reduce_host(op.handle, plan.handle, _p(field), NT, _p(out), 0)
    _invalid(rc, "host entry points take unpadded fields (operator pitch must be nx)")
