"""convert_and_aggregate's orchestration on a fake operator layer, without a GPU.

A fake converter is registered like a known one; its spec reduces with a NumPy sparse
product and produces per-cell values and NaN-skipping time sums.  The plan cache and
``torch.cuda.set_device`` are stubbed.  What is checked is everything around the
operators: the in-process and the partitioned execution (several devices, a lazily
loaded cutout in several parts, heat-like specs on day starts), the plugin protocol,
time aggregation, the aggregation matrix built from ``matrix`` / ``layout`` / ``index``,
``per_unit`` / ``return_capacity``, and the dims, coordinates, ``units`` and ``name`` of
the results.  All values are multiples of 1/8 with small sums, so float32 sums are exact
in any order and partitioned results must equal in-process ones bit for bit.
"""

import types
import warnings

import numpy as np
import pandas as pd
import pytest
import scipy.sparse as sp

import atlite_b200 as ab
from atlite_b200 import convert, engine, labelled

NY, NX, NT = 3, 4, 30


def _data():
    rng = np.random.default_rng(7)
    v = (rng.integers(0, 16, (NT, NY, NX)) / 8.0).astype(np.float32)
    v[:, 0, 1] = np.nan  # NaN in every step: mean NaN, sum 0
    v[5, 2, 2] = np.nan  # NaN in one step
    coords = {
        "time": pd.date_range("2013-01-01 00:00", periods=NT, freq="3h"),  # 8 steps a day, 3.75 days
        "y": np.arange(NY) * 0.5 + 50.0,
        "x": np.arange(NX) * 0.5 + 5.0,
    }
    coords["lat"], coords["lon"] = coords["y"], coords["x"]
    return v, coords


def _dataset():
    v, coords = _data()
    return labelled.Dataset({"v": v}, coords=coords)


def _lazy():
    v, coords = _data()
    return labelled.LazyDataset({"v": lambda lo, hi: v[lo:hi]}, coords=coords, time_chunk=4)


class FakeSpec:
    """What a known converter's spec offers the orchestration, computed with NumPy."""

    name, units = "fake thing", "kW"

    def __init__(self, ds, scale=1.0):
        self.field = np.asarray(ds.raw("v")) * np.float32(scale)
        self.time_labels = pd.DatetimeIndex(np.asarray(ds.coords["time"]))
        self.pitch = NX

    def reduce(self, plan):
        nt = self.field.shape[0]
        return np.asarray(plan.m @ self.field.reshape(nt, -1).T).T.astype(np.float32)

    def cells(self, timesum=False):
        if not timesum:
            return self.field.copy()
        return np.stack([np.nansum(self.field, axis=0), (~np.isnan(self.field)).sum(0)]).astype(np.float32)

    def cells_timesum(self):
        sc = self.cells(timesum=True)
        return sc[0], sc[1]


class FakeDailySpec(FakeSpec):
    """Heat-like: one value per calendar day of the shifted time axis (the daily mean)."""

    name, units = "fake daily", None

    def __init__(self, ds, scale=1.0, hour_shift=0.0):
        super().__init__(ds, scale)
        self.time_labels, self.day_start = convert.day_bins(np.asarray(ds.coords["time"]), hour_shift)
        ds_ = self.day_start
        self.field = np.stack([self.field[a:b].mean(0) for a, b in zip(ds_[:-1], ds_[1:])]).astype(np.float32)


def fake_convert(ds, scale=1.0):
    raise AssertionError("a registered converter is never called")


def fake_daily_convert(ds, scale=1.0, hour_shift=0.0):
    raise AssertionError("a registered converter is never called")


def plugin_convert(ds, scale=1.0):
    """A user's convert_func: returns the labelled (time, y, x) field itself."""
    vals = np.asarray(ds.raw("v")) * np.float32(scale)
    coords = {"time": np.asarray(ds.coords["time"]), "y": ds.coords["y"], "x": ds.coords["x"]}
    return labelled.make_dataarray(vals, ("time", "y", "x"), coords, {"units": "kW"}, "plugin thing")


class FakePlan:
    def __init__(self, matrix, ny, nx, device=None, pitch=None, digest=None):
        assert (ny, nx) == (NY, NX) and pitch in (None, NX)
        self.m = sp.csr_matrix(matrix)
        self.n_bus = self.m.shape[0]
        self.device = device

    def spmm(self, dense):
        dense = np.asarray(dense, dtype=np.float32)
        return np.asarray(self.m @ dense.reshape(dense.shape[0], -1).T).T.astype(np.float32)


@pytest.fixture
def fake_layer(monkeypatch):
    fake_torch = types.SimpleNamespace(cuda=types.SimpleNamespace(set_device=lambda d: None))
    monkeypatch.setattr(engine, "_torch", lambda: fake_torch)
    monkeypatch.setattr(engine, "get_plan", FakePlan)
    monkeypatch.setattr(engine, "matrix_digest", lambda m: ("digest", m.shape, m.nnz))
    monkeypatch.setitem(convert._REGISTRY, fake_convert, FakeSpec)
    monkeypatch.setitem(convert._REGISTRY, fake_daily_convert, FakeDailySpec)
    monkeypatch.setattr(convert, "_HeatSpec", FakeDailySpec)  # heat-like: parts snap to day starts


MODES = ["in-process", "devices", "lazy", "plugin"]


def _run(monkeypatch, mode, daily=False, **kw):
    if mode == "lazy":
        monkeypatch.setattr(convert, "PART_BYTES", 4 * 2 * convert._bytes_per_step(_lazy()))  # 8-step parts
        cutout = ab.Cutout(data=_lazy())
    else:
        cutout = ab.Cutout(data=_dataset(), devices=[0, 1] if mode == "devices" else None)
    func = plugin_convert if mode == "plugin" else fake_daily_convert if daily else fake_convert
    with warnings.catch_warnings(record=True) as log:
        warnings.simplefilter("always")
        out = cutout.convert_and_aggregate(func, scale=2.0, **kw)
    return out, [str(w.message) for w in log]


def _values(mode, daily=False, hour_shift=0.0):
    v, coords = _data()
    v = v * np.float32(2.0)
    labels = pd.DatetimeIndex(coords["time"])
    if daily:
        labels, offs = convert.day_bins(coords["time"], hour_shift)
        v = np.stack([v[a:b].mean(0) for a, b in zip(offs[:-1], offs[1:])]).astype(np.float32)
    return v, labels


def _matrix():
    m = np.zeros((4, NY * NX))
    m[0, [0, 1, 2]] = [1.0, 0.5, 0.25]  # holds the all-NaN cell (0, 1)
    m[1, 5:9] = 0.5
    m[3, [9, 10, 11, 4]] = [2.0, 1.0, 1.0, 0.125]  # holds the one-step NaN cell (2, 2)
    return sp.csr_matrix(m)  # bus 2 has zero capacity


def _coord(out, d):
    return np.asarray(out.coords[d])


def _check(out, dims, values, coords, units, name):
    assert tuple(out.dims) == dims
    got = np.asarray(out.values)
    assert got.shape == values.shape
    np.testing.assert_array_equal(got, values)  # NaN where expected, bit-equal elsewhere
    for d, c in coords.items():
        np.testing.assert_array_equal(_coord(out, d), np.asarray(c))
    assert out.attrs.get("units") == units
    assert out.name == name


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("aggregate_time", [None, "sum", "mean", "legacy"])
def test_per_cell_results(fake_layer, monkeypatch, mode, aggregate_time):
    out, warned = _run(monkeypatch, mode, aggregate_time=aggregate_time)
    assert any("legacy" in w for w in warned) == (aggregate_time == "legacy")
    v, labels = _values(mode)
    _, coords = _data()
    yx = {"y": coords["y"], "x": coords["x"]}
    name, units = ("plugin thing", "kW") if mode == "plugin" else ("fake thing", "kW")
    if aggregate_time is None:
        _check(out, ("time", "y", "x"), v, {"time": labels, **yx}, units, name)
        return
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        want = np.nanmean(v.astype(np.float64), 0) if aggregate_time == "mean" else np.nansum(v, 0)
        if mode == "plugin":  # the plugin's own da.sum / da.mean over time
            want = np.nanmean(v, 0) if aggregate_time == "mean" else np.nansum(v, 0)
    assert np.isnan(want[0, 1]) == (aggregate_time == "mean") and want[2, 2] == want[2, 2]
    _check(out, ("y", "x"), want, yx, units, name)


@pytest.mark.parametrize("hour_shift", [0.0, 5.0])
@pytest.mark.parametrize("mode", ["in-process", "devices", "lazy"])
def test_daily_specs_are_cut_on_day_starts(fake_layer, monkeypatch, mode, hour_shift):
    out, _ = _run(monkeypatch, mode, daily=True, matrix=_matrix(), aggregate_time=None, hour_shift=hour_shift)
    v, labels = _values(mode, daily=True, hour_shift=hour_shift)
    res = (_matrix() @ v.reshape(len(v), -1).T).astype(np.float32).astype(np.float64)
    if mode == "lazy":
        _check(out, ("time", "dim_0"), res.T, {"time": labels, "dim_0": np.arange(4)}, "MW", "fake daily")
    else:
        _check(out, ("dim_0", "time"), res, {"time": labels, "dim_0": np.arange(4)}, "MW", "fake daily")


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("aggregate_time", [None, "sum", "mean"])
@pytest.mark.parametrize("options", ["plain", "per_unit", "capacity", "index", "layout", "layout_only"])
def test_bus_results(fake_layer, monkeypatch, mode, aggregate_time, options):
    m = _matrix()
    kw = dict(matrix=m, aggregate_time=aggregate_time)
    dim, idx = "dim_0", pd.RangeIndex(4)
    _, coords = _data()
    lay = (np.arange(NY * NX).reshape(NY, NX) % 3 + 1) / 2.0
    if options == "per_unit":
        kw["per_unit"] = True
    elif options == "capacity":
        kw.update(per_unit=True, return_capacity=True)
    elif options == "index":
        dim, idx = "bus", pd.Index(["a", "b", "c", "d"], name="bus")
        kw["index"] = idx
    elif options in ("layout", "layout_only"):
        kw["layout"] = labelled.DataArray(lay, {"y": coords["y"], "x": coords["x"]}, ("y", "x"))
        if options == "layout_only":
            del kw["matrix"]
    out, _ = _run(monkeypatch, mode, **kw)
    if options == "capacity":
        out, capacity = out
    else:
        assert not isinstance(out, tuple)

    mm = m if options != "layout_only" else sp.csr_matrix(np.ones((1, NY * NX)))
    if options in ("layout", "layout_only"):
        mm = sp.csr_matrix(mm.multiply(lay.reshape(1, -1)))
        dim, idx = "dim_0", pd.RangeIndex(mm.shape[0])
    caps = np.asarray(mm.sum(-1)).ravel()
    v, labels = _values(mode)
    res = np.asarray(mm @ v.reshape(NT, -1).T).T.astype(np.float32).astype(np.float64)  # (time, bus)
    units = "MW"
    if kw.get("per_unit"):
        units = "p.u."
        with np.errstate(divide="ignore", invalid="ignore"):
            res = res / np.where(caps != 0, caps, np.nan)[None, :]
        res = np.where(np.isnan(res), 0.0, res)
    name = "plugin thing" if mode == "plugin" else "fake thing"
    if aggregate_time is not None:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", RuntimeWarning)
            want = np.nansum(res, 0) if aggregate_time == "sum" else np.nanmean(res, 0)
        _check(out, (dim,), want, {dim: idx}, units, name)
    elif mode == "lazy":  # lazily loaded cutouts: (time, bus)
        _check(out, ("time", dim), res, {"time": labels, dim: idx}, units, name)
    else:  # in-memory cutouts: (bus, time)
        _check(out, (dim, "time"), res.T, {"time": labels, dim: idx}, units, name)
    if options == "capacity":
        _check(capacity, (dim,), caps, {dim: idx}, "MW", None)
        assert caps[2] == 0.0


def test_matrix_arguments_are_checked_after_the_spec_is_built(fake_layer, monkeypatch):
    """The spec (or a plugin's field) is built first, then the aggregation arguments are validated."""
    built = []

    class Spec(FakeSpec):
        def __init__(self, ds, scale=1.0):
            built.append(True)
            super().__init__(ds, scale)

    monkeypatch.setitem(convert._REGISTRY, fake_convert, Spec)
    with pytest.raises(ValueError, match="ambiguous"):
        _run(monkeypatch, "in-process", matrix=_matrix(), shapes=[object()])
    assert built == [True]
    with pytest.raises(ValueError, match="per_unit"):
        _run(monkeypatch, "in-process", per_unit=True)
    assert built == [True, True]
