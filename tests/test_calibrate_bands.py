"""Calibration against a benchmark flood map on the device and over row bands (device.calibrate, bands.calibrate_bands,
BandRunner.load_flood / log_indices / calibrate, pipeline_files(flood=...)).

CPU: the host merge of per-band extrema against np.unique, the band driver with NumPy stand-in bands (LocalExchange and
gloo) against a NumPy restatement of the reference's calibration, and argument validation of the new entry points.
GPU: the extrema, fused histogram and class-map kernels against np.unique and the materialising path, KAT-1 through
device.calibrate, k logical bands against one GPU, and the files against pipeline_files."""
import filecmp
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from helpers import PX, avaliacao, binary_map, example_inputs, min_max_scale, misaligned

UNDER = {"under": True, "over": False}


# ---- NumPy restatements ------------------------------------------------------------------------------------------
def np_extrema(a):
    """dtb_eval_extrema of one part: lo, second lo, hi, distinct non-NaN values (capped at 2), NaN seen"""
    a = np.asarray(a, np.float64).reshape(-1)
    v = np.unique(a[~np.isnan(a)])
    out = np.zeros(5)
    out[:2][:min(2, len(v))] = v[:2]
    out[2] = v[-1] if len(v) else 0.0
    out[3], out[4] = min(2, len(v)), float(np.isnan(a).any())
    return out


def np_unique_ends(x):
    e = np.unique(x)
    return float(e[1]), float(e[-1])


def remapped(flood):
    """the benchmark after avaliacao's first call in the reference (1 -> 2, -100 -> 0, evaluation.py:149-150); helpers'
    avaliacao restates the 1 -> 2 only"""
    return np.where(flood == -100, 0, flood)


def np_calibration(desc, flood, under):
    """helpers.calibration for both directions (evaluation.py:12-87)"""
    fit = lambda t: avaliacao(binary_map(desc, t, UNDER[under]), flood)[1]
    f1, f2, f3 = fit(0.25), fit(0.50), fit(0.75)
    if f3 > f2:
        it, best = (75, f3) if f3 > f1 else (25, f1)
    else:
        it, best = (50, f2) if f2 > f1 else (25, f1)
    th = None
    for i in range(it - 20, it + 30, 10):
        v = fit(i / 100)
        if v >= best:
            best, th = v, i
    it = th
    for i in range(it - 5, it + 6):
        v = fit(i / 100)
        if v > best:
            best, th = v, i
    for scale in (1000, 10000):
        it = th * 10
        th = it
        for i in range(it - 10, it + 11):
            v = fit(i / scale)
            if v > best:
                best, th = v, i
    return th / 10000


def reference(x, flood, under, nodata=-100):
    """example.py:113-147 on the whole raster: (mn, mx, threshold, correctness, fit, class map)"""
    mn, mx = np_unique_ends(x)
    with np.errstate(all="ignore"):
        desc = min_max_scale(x.astype(np.float64), mn, mx, nodata)
        fl = remapped(flood).astype(np.int64)
        th = np_calibration(desc, fl, under)
        c, f, cls = avaliacao(binary_map(desc, th, UNDER[under]), fl)
    return mn, mx, th, float(c), float(f), cls


def scaled(v, mn, mx, nodata):
    v = np.asarray(v, np.float64)
    with np.errstate(all="ignore"):
        return np.where((v == nodata) | np.isnan(v), np.nan, (v - mn) / (mx - mn))


class NumpyBand:
    """calibrate_bands' band interface over NumPy rows (the kernels' semantics restated)"""

    def __init__(self, index, desc, flood):
        self.index, self.desc, self.flood = index, desc, flood
        self.cls = None

    def extrema(self, descriptor):
        return torch.from_numpy(np_extrema(self.desc))

    def corner(self, descriptor):
        return torch.tensor([float(self.desc[0, 0])], dtype=torch.float64)

    def _bits(self, mn, mx, corner, nodata):
        s = scaled(self.desc, mn, mx, nodata).reshape(-1)
        nd = scaled(corner, mn, mx, nodata)
        usable = ~np.isnan(s) & (s != nd)
        f = self.flood.reshape(-1).astype(np.int64)
        c = np.where(f == 1, 2, np.where(f == -100, 0, f))
        return s, usable, f, c

    def histogram(self, descriptor, mn, mx, corner, thresholds, under, nodata, hist):
        s, usable, f, c = self._bits(mn, mx, corner, nodata)
        th, k = np.asarray(thresholds, np.float64), len(thresholds)
        j = np.searchsorted(th, s, side="left" if under == "under" else "right")
        j = np.where(usable, j, k if under == "under" else 0)
        ok = ((f >= 0) & (f <= 3)) | (f == -100)
        h = np.zeros(4 * 33, np.int64)
        np.add.at(h, (c * 33 + j)[ok], 1)
        hist += torch.from_numpy(h)

    def class_map(self, descriptor, mn, mx, corner, threshold, under, nodata):
        s, usable, f, c = self._bits(mn, mx, corner, nodata)
        with np.errstate(invalid="ignore"):
            b = usable & ((s <= threshold) if under == "under" else (s >= threshold))
        self.cls = (b + c).reshape(self.desc.shape)


def hand_like(rows, cols, seed, dtype=np.float32, corner_valid=False, nan=False):
    """a HAND-like descriptor (0 .. ~25 m, -100 nodata border and blobs, a few NaN) and a benchmark flood map
    (HAND <= 3 m with random flips, some -100 cells, a few values outside 0..3)"""
    rng = np.random.default_rng(seed)
    h = rng.gamma(1.5, 3.0, (rows, cols))
    if dtype == np.int16:
        h = np.round(h)
    h = h.astype(dtype)
    if not corner_valid:
        h[0, :], h[:, 0] = -100, -100
    h[rows // 3:rows // 3 + 4, cols // 2:cols // 2 + 7] = -100
    if nan and dtype == np.float32:
        h[rng.random((rows, cols)) < 0.002] = np.nan
    flood = (h <= 3).astype(np.int8)
    flip = rng.random((rows, cols)) < 0.08
    flood[flip] = 1 - flood[flip]
    flood[rng.random((rows, cols)) < 0.03] = -100
    flood[rng.random((rows, cols)) < 0.003] = 5
    return h, flood


# ---- CPU: host merge of per-band extrema ---------------------------------------------------------------------------
def _special_raster(dtype, seed, rows=37, cols=29):
    rng = np.random.default_rng(seed)
    if dtype == np.int16:
        x = rng.integers(-120, 200, (rows, cols)).astype(np.int16)
        x[rng.random((rows, cols)) < 0.2] = -100
        x[rng.random((rows, cols)) < 0.05] = 0
    else:
        x = (rng.standard_normal((rows, cols)) * 10).astype(np.float32)
        for v, p in ((np.nan, 0.03), (np.inf, 0.01), (-np.inf, 0.01), (0.0, 0.02), (-0.0, 0.02), (-100.0, 0.2)):
            x[rng.random((rows, cols)) < p] = v
    return x


def _splits(rows, k, rng):
    cuts = sorted(rng.choice(np.arange(1, rows), k - 1, replace=False).tolist()) if k > 1 else []
    return [0] + cuts + [rows]


@pytest.mark.parametrize("dtype", [np.float32, np.int16])
@pytest.mark.parametrize("k", [1, 2, 3, 4, 5])
def test_merged_band_extrema_equal_np_unique_ends(dtype, k):
    from descriptools_b200 import evaluation

    rng = np.random.default_rng(k)
    for seed in range(6):
        x = _special_raster(dtype, 100 * k + seed)
        if seed == 1:
            x[:9] = -100                     # an all-nodata band
        if seed == 2 and dtype == np.float32:
            x[5:20] = 7.5                    # one-value bands
            x[20:] = np.nan
        if seed == 3:
            x[:] = -100
            x[3, 4] = 2
        edges = _splits(x.shape[0], k, rng) if seed != 4 else list(range(min(k, x.shape[0]))) + [x.shape[0]]  # one-row bands
        rows = [np_extrema(x[a:b]) for a, b in zip(edges, edges[1:])]
        want = np_unique_ends(x)
        got = evaluation.unique_ends(np.stack(rows))
        np.testing.assert_array_equal(np.array(got), np.array(want), err_msg=f"seed {seed}")


def test_fewer_than_two_values_raise():
    from descriptools_b200 import evaluation

    for x in (np.full((4, 3), -100, np.float32), np.full((4, 3), np.nan, np.float32), np.array([[0.0, -0.0]], np.float32)):
        with pytest.raises(ValueError):
            evaluation.unique_ends(np.stack([np_extrema(x[:2]), np_extrema(x[2:])]) if len(x) > 1 else np_extrema(x))
    # one value and NaN: np.unique has two elements, mn and mx are NaN
    mn, mx = evaluation.unique_ends(np_extrema(np.array([[3.0, np.nan]], np.float32)))
    assert np.isnan(mn) and np.isnan(mx)


# ---- CPU: the driver with NumPy stand-ins ----------------------------------------------------------------------
# (name, dtype, valid corner cell, NaN cells: mx = np.unique(x)[-1] is NaN then, and every scaled cell with it)
CASES = [("f32", np.float32, False, False), ("i16", np.int16, False, False), ("corner", np.float32, True, False),
         ("nan", np.float32, False, True)]


def _case(name):
    _, dtype, corner, nan = next(c for c in CASES if c[0] == name)
    return hand_like(260, 90, seed=len(name), dtype=dtype, corner_valid=corner, nan=nan)


def _check(res, classes, x, flood, under):
    mn, mx, th, c, f, cls = reference(x, flood, under)
    np.testing.assert_array_equal([res["mn"], res["mx"]], [mn, mx])
    assert res["threshold"] == th
    np.testing.assert_array_equal([res["correctness"], res["fit"]], [c, f])
    got = np.concatenate(classes, 0)
    np.testing.assert_array_equal(got, cls)
    assert res["counts"] == tuple(int((cls == k).sum()) for k in range(4))


@pytest.mark.parametrize("under", ["under", "over"])
@pytest.mark.parametrize("name", [c[0] for c in CASES])
@pytest.mark.parametrize("k", [1, 2, 3, 4])
def test_calibrate_bands_local_stand_ins(name, under, k):
    from descriptools_b200 import bands

    x, flood = _case(name)
    e = bands.band_edges(x.shape[0], k)
    bs = [NumpyBand(i, x[e[i]:e[i + 1]], flood[e[i]:e[i + 1]]) for i in range(k)]
    res = bands.calibrate_bands(bs, bands.LocalExchange(k), "hand", under)
    _check(res, [b.cls for b in bs], x, flood, under)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _gloo_worker(rank, world, port, q):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        import torch.distributed as dist

        dist.init_process_group("gloo", rank=rank, world_size=world)
        from descriptools_b200 import bands

        x_ = bands.DistExchange()
        out = {}
        for name, *_ in CASES:
            x, flood = _case(name)
            e = bands.band_edges(x.shape[0], world)
            for under in ("under", "over"):
                b = NumpyBand(rank, x[e[rank]:e[rank + 1]], flood[e[rank]:e[rank + 1]])
                out[name, under] = (bands.calibrate_bands([b], x_, "hand", under), b.cls)
        dist.barrier()
        dist.destroy_process_group()
        q.put((rank, "ok", out))
    except Exception:  # pragma: no cover
        import traceback

        q.put((rank, "fail", traceback.format_exc()))


@pytest.mark.parametrize("world", [2, 3])
def test_calibrate_bands_over_gloo(world):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gloo_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = sorted((q.get(timeout=600) for _ in procs), key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
    for rank, status, info in results:
        assert status == "ok", f"rank {rank}: {info}"
    for name, *_ in CASES:
        x, flood = _case(name)
        for under in ("under", "over"):
            res = [info[name, under][0] for _, _, info in results]
            assert all(repr(r) == repr(res[0]) for r in res)
            _check(res[0], [info[name, under][1] for _, _, info in results], x, flood, under)


# ---- CPU: argument validation and the host prefix sums --------------------------------------------------------------
def test_new_entry_points_validate_without_a_device():
    import ctypes

    from descriptools_b200 import _lib

    L = _lib.lib
    th = (ctypes.c_double * 3)(0.1, 0.2, 0.3)
    bad = (ctypes.c_double * 3)(0.1, 0.1, 0.3)
    nws = L.dtb_eval_extrema_workspace_bytes()
    assert nws > 0
    assert L.dtb_eval_extrema(None, 0, 10, 1, 1, nws, None) == -1
    assert L.dtb_eval_extrema(1, 0, 10, None, 1, nws, None) == -1
    assert L.dtb_eval_extrema(1, 0, 0, 1, 1, nws, None) == -1
    assert L.dtb_eval_extrema(1, 1, 10, 1, 1, nws, None) == -1      # f64: not a calibrated descriptor type
    assert L.dtb_eval_extrema(1, 7, 10, 1, 1, nws, None) == -1
    assert L.dtb_eval_extrema(1, 0, 10, 1, 1, nws - 1, None) == -3
    args = lambda **kw: [kw.get(k, v) for k, v in dict(desc=1, dt=0, flood=1, n=10, mn=0.0, mx=1.0, nd=-100.0, corner=-100.0,
                                                      th=th, k=3, under=1, hist=1, st=None).items()]
    assert L.dtb_eval_hist(*args(desc=None)) == -1
    assert L.dtb_eval_hist(*args(flood=None)) == -1
    assert L.dtb_eval_hist(*args(hist=None)) == -1
    assert L.dtb_eval_hist(*args(th=None)) == -1
    assert L.dtb_eval_hist(*args(n=0)) == -1
    assert L.dtb_eval_hist(*args(k=0)) == -1 and L.dtb_eval_hist(*args(k=33)) == -1
    assert L.dtb_eval_hist(*args(th=bad)) == -1
    assert L.dtb_eval_hist(*args(dt=1)) == -1 and L.dtb_eval_hist(*args(dt=5)) == -1
    assert L.dtb_eval_class_scaled(None, 0, 1, 10, 0.0, 1.0, -100.0, -100.0, 0.5, 1, 1, None) == -1
    assert L.dtb_eval_class_scaled(1, 0, None, 10, 0.0, 1.0, -100.0, -100.0, 0.5, 1, 1, None) == -1
    assert L.dtb_eval_class_scaled(1, 0, 1, 10, 0.0, 1.0, -100.0, -100.0, 0.5, 1, None, None) == -1
    assert L.dtb_eval_class_scaled(1, 3, 1, 10, 0.0, 1.0, -100.0, -100.0, 0.5, 1, 1, None) == -1
    out = (ctypes.c_int64 * 4)()
    assert L.dtb_eval_counts_from_hist(None, 1, 1, out) == -1
    h = np.zeros(4 * 33, np.uint64)
    assert L.dtb_eval_counts_from_hist(h.ctypes.data, 0, 1, out) == -1
    assert L.dtb_eval_counts_from_hist(h.ctypes.data, 33, 1, out) == -1
    assert L.dtb_eval_counts_from_hist(h.ctypes.data, 1, 1, None) == -1


@pytest.mark.parametrize("under", ["under", "over"])
def test_counts_from_hist_equal_direct_counts(under):
    from descriptools_b200 import evaluation

    rng = np.random.default_rng(5)
    d = rng.random(4000)
    d[rng.random(4000) < 0.05] = np.nan
    f = rng.choice(np.array([0, 1, 2, 3, -100, 7]), 4000)
    th = np.sort(rng.choice(np.linspace(0.0, 1.0, 101), 17, replace=False))
    b = NumpyBand(0, d.reshape(40, 100), f.reshape(40, 100))
    hist = torch.zeros(4 * 33, dtype=torch.int64)
    b.histogram("x", 0.0, 1.0, float("nan"), th, under, -100, hist)
    got = evaluation.counts_from_hist(hist.numpy(), len(th), under)
    fl = np.where(f == -100, 0, f)
    for i, t in enumerate(th):
        with np.errstate(invalid="ignore"):
            bin_ = np.where(np.isnan(d), 0, (d <= t) if under == "under" else (d >= t))
        cls = bin_ + np.where(fl == 1, 2, fl)
        assert got[i].tolist() == [int((cls == c).sum()) for c in range(4)], t


# ---- GPU: the kernels ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.int16])
def test_extrema_kernel_equals_np_unique(dtype):
    from descriptools_b200 import device

    for seed in range(5):
        x = _special_raster(dtype, seed, rows=67 + seed, cols=31 + 2 * seed)  # lengths not a multiple of 4
        if seed == 1:
            x[:] = -100
            x[3, 4] = 2
        if seed == 2 and dtype == np.float32:
            x[:] = np.nan
            x[0, 1] = -0.0
            x[5, 5] = 0.0
        t = torch.from_numpy(x).cuda()
        for v in (t, misaligned(t)):
            got = device.eval_extrema(v).cpu().numpy()
            want = np_extrema(x)
            want[:3] = want[:3] + 0.0  # -0 -> +0
            np.testing.assert_array_equal(got, want, err_msg=f"seed {seed}")
            assert not np.signbit(got[:3][got[:3] == 0]).any()
    big = _special_raster(dtype, 9, rows=2049, cols=1999)
    np.testing.assert_array_equal(device.eval_extrema(torch.from_numpy(big).cuda()).cpu().numpy(), np_extrema(big) + 0.0)


def _materialised_counts(x, flood, mn, mx, ths, under):
    """dtb_minmax_scale + dtb_eval_counts on the f64 raster (binary_map's nodata = its cell (0, 0))"""
    from descriptools_b200 import evaluation

    s = evaluation.minMaxScale(x, mn, mx, -100)
    st = torch.from_numpy(s).cuda()
    ctr = evaluation._Counter(st, True, float(s[0, 0]), torch.from_numpy(evaluation_remap(flood)).cuda(), under)
    return ctr.counts(ths), s


def evaluation_remap(flood):
    f = flood.copy()
    f[f == 1] = 2
    f[f == -100] = 0
    return f


@pytest.mark.gpu
@pytest.mark.parametrize("under", ["under", "over"])
@pytest.mark.parametrize("name", [c[0] for c in CASES])
def test_fused_histogram_and_class_map_equal_the_materialising_path(name, under):
    from descriptools_b200 import device, evaluation

    x, flood = _case(name)
    x = np.ascontiguousarray(np.tile(x, (3, 5)))  # larger than one block's share
    flood = np.ascontiguousarray(np.tile(flood, (3, 5)))
    mn, mx = np_unique_ends(x)
    xt, ft = torch.from_numpy(x).cuda(), torch.from_numpy(flood).cuda()
    for ths in ([0.25], list(np.linspace(0.0, 0.62, 32)), [i / 10000 for i in range(110, 131)]):
        want, s = _materialised_counts(x, flood, mn, mx, ths, under)
        for xv, fv in ((xt, ft), (misaligned(xt), ft), (xt, misaligned(ft))):
            hist = torch.zeros(4 * 33, dtype=torch.int64, device="cuda")
            device.eval_hist(xv, fv, mn, mx, float(x[0, 0]), ths, under, hist)
            device.eval_hist(xv, fv, mn, mx, float(x[0, 0]), ths, under, hist)  # it adds
            got = evaluation.counts_from_hist(hist.cpu().numpy() // 2, len(ths), under)
            np.testing.assert_array_equal(got, want)
        th = ths[len(ths) // 2]
        cls = device.eval_class(xt, ft, mn, mx, float(x[0, 0]), th, under).cpu().numpy()
        b = evaluation.binary_map(s, th, under)
        _, _, want_cls = evaluation.avaliacao(b, flood.copy())
        np.testing.assert_array_equal(cls, want_cls.astype(np.int8))
    assert torch.equal(ft.cpu(), torch.from_numpy(flood))


@pytest.mark.gpu
def test_kat1_through_device_calibrate():
    from descriptools_b200 import device, flowhand

    ex = example_inputs()
    _, _, hand = flowhand.flow_hand_index(ex["dem"], ex["fdr"], ex["river"], PX)
    assert hand.dtype == np.int16
    flood = torch.from_numpy(ex["flood"]).cuda()
    before = flood.clone()
    res = device.calibrate(torch.from_numpy(hand).cuda(), flood, "under")
    assert res["threshold"] == 0.012
    assert res["correctness"] == 0.8581615676712259 and res["fit"] == 0.7240945135019289
    np.testing.assert_array_equal(res["class_map"].cpu().numpy().astype(np.uint8), ex["hand_class"])
    assert torch.equal(flood, before)
    e = np.unique(hand)
    assert (res["mn"], res["mx"]) == (float(e[1]), float(e[-1]))
    res8 = device.calibrate(torch.from_numpy(hand).cuda(), flood.view(torch.uint8), "under")  # uint8 is read as int8
    assert res8["threshold"] == 0.012
    with pytest.raises(ValueError):
        device.calibrate(torch.full((8, 8), -100, dtype=torch.int16, device="cuda"), flood[:8, :8])


# ---- GPU: bands against one GPU ---------------------------------------------------------------------------------------
def _flood_file(path, hand, seed):
    """a benchmark flood map for a HAND raster: HAND <= 3 m with random flips and some -100 cells (uint8: 156)"""
    import descriptools_b200.raster as rio

    rng = np.random.default_rng(seed)
    f = ((hand <= 3) & (hand != -100)).astype(np.int8)
    flip = rng.random(hand.shape) < 0.05
    f[flip] = 1 - f[flip]
    f[rng.random(hand.shape) < 0.02] = -100
    with rio.open(path, "w", width=hand.shape[1], height=hand.shape[0], dtype="uint8", compress="lzw", tiled=True,
                  blockxsize=128, blockysize=128, nodata=0) as dst:
        dst.write(f.view(np.uint8))
    return f


@pytest.mark.gpu
@pytest.mark.parametrize("holes", [True, False])
def test_bands_calibrate_equal_one_gpu(tmp_path, holes):
    from descriptools_b200 import bands, device, evaluation, pipeline

    import helpers

    rows, cols, thr = 700, 530, 300
    dem = helpers.synth(rows, cols, 17, holes=holes)
    one = pipeline.run_device(torch.from_numpy(dem).cuda(), PX, thr)
    flood = _flood_file(tmp_path / "flood.tif", one["hand"].cpu().numpy(), 3)
    ft = torch.from_numpy(flood).cuda()
    ref = {d: device.calibrate(one[d], ft, u) for d, u in (("hand", "under"), ("gfi", "over"))}
    for d, u in (("hand", "under"), ("gfi", "over")):  # the drop-in on host copies
        h = one[d].cpu().numpy()
        e = np.unique(h)
        s = evaluation.minMaxScale(h, e[1], e[-1], -100)
        fl = flood.copy()
        th = evaluation.calibration(s, fl, u)
        c, f, cls = evaluation.avaliacao(evaluation.binary_map(s, th, u), fl)
        assert (th, c, f) == (ref[d]["threshold"], ref[d]["correctness"], ref[d]["fit"]), d
        np.testing.assert_array_equal(cls.astype(np.int8), ref[d]["class_map"].cpu().numpy())
    rad = device.slope_to_radians(one["slope"])
    ti, mti = device.ti_mti(one["acc"], rad, PX, 0.1)
    ln = device.ln_hl_H(one["hand"], one["acc"], 0.4, 0.1, PX)
    for k in (1, 2, 3, 4):
        runner = bands.BandRunner(rows, cols, PX, thr, 0.4, 0.1, nbands=k)
        runner.load([torch.from_numpy(dem[a:b].copy()) for a, b in zip(runner.edges, runner.edges[1:])])
        runner.step()
        runner.load_flood(tmp_path / "flood.tif")
        runner.log_indices(0.1)
        for d, u in (("hand", "under"), ("gfi", "over")):
            res = runner.calibrate(d, u)
            want = {key: v for key, v in ref[d].items() if key != "class_map"}
            assert res == want, (k, d)
            got = torch.cat([o[d + "_class"] for o in runner.outputs()], 0)
            assert torch.equal(got, ref[d]["class_map"]), (k, d)
        for name, t in (("ti", ti), ("mti", mti), ("lnhlh", ln)):
            got = torch.cat([o[name] for o in runner.outputs()], 0)
            assert torch.equal(got.view(torch.int32), t.view(torch.int32)), (k, name)


def test_runner_refuses_a_flood_map_of_another_shape_or_type(tmp_path):
    import descriptools_b200.raster as rio
    from descriptools_b200 import bands

    for name, shape, dt in (("shape", (64, 60), "uint8"), ("type", (128, 60), "int16")):
        with rio.open(tmp_path / f"{name}.tif", "w", width=shape[1], height=shape[0], dtype=dt, compress="lzw", tiled=True,
                      blockxsize=64, blockysize=64) as dst:
            dst.write(np.zeros(shape, dt))
    runner = bands.BandRunner.__new__(bands.BandRunner)  # no device needed: the checks come before any band is read
    runner.rows, runner.cols, runner.bands = 128, 60, []
    with pytest.raises(ValueError):
        runner.load_flood(tmp_path / "shape.tif")
    with pytest.raises(TypeError):
        runner.load_flood(tmp_path / "type.tif")


# ---- GPU: files -------------------------------------------------------------------------------------------------------
EXTRA = ("ti", "mti", "lnhlh", "hand_class")


def _raw_dem_and_flood(base):
    """a raw DEM file (pits to fill, nodata holes across band seams) and a flood map file for its HAND"""
    import descriptools_b200.raster as rio
    from descriptools_b200 import pipeline

    import oracle

    dem, flood = base / "raw.tif", base / "flood.tif"
    if not dem.exists():
        raw = oracle.synth_dem(700, 530, 0, 29)
        raw[170:215, 40:120] = -9999.0
        raw[319, 200:330] = -9999.0
        raw[505:520, 100:140] = -9999.0
        with rio.open(dem, "w", width=530, height=700, dtype="float32", compress="lzw", predictor=3, tiled=True, blockxsize=128,
                      blockysize=128, nodata=-9999.0, transform=rio.Affine(PX, 0, 500000.0, 0, -PX, 7000000.0)) as dst:
            dst.write(raw)
        pipeline.pipeline_files(dem, base / "hand_only", river_threshold=300, px=PX, condition=True, outputs=("hand",))
        _flood_file(flood, rio.open(base / "hand_only" / "hand.tif").read(1), 8)
    return dem, flood


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 4])
def test_band_files_with_calibration_equal_pipeline_files(tmp_path_factory, tmp_path, k):
    from PIL import Image

    from descriptools_b200 import bands, pipeline

    base = tmp_path_factory.getbasetemp()
    dem, flood = _raw_dem_and_flood(base)
    ref = base / "ref_calib"
    if not ref.exists():
        got = pipeline.pipeline_files(dem, ref, river_threshold=300, px=PX, condition=True, flood=flood,
                                      outputs=pipeline.STAGE_OUTPUTS + EXTRA)
        (ref / "calibration.txt").write_text(repr(got["calibration"]))
    runner = bands.BandRunner(700, 530, PX, 300, 0.4, 0.1, nbands=k)
    runner.load_file(dem, condition=True)
    runner.load_flood(flood)
    runner.step()
    runner.log_indices(0.1)
    res = runner.calibrate("hand", "under")
    assert repr(res) == (ref / "calibration.txt").read_text()
    paths = runner.write_files(tmp_path / "out", outputs=EXTRA)
    for name, p in paths.items():
        assert filecmp.cmp(ref / f"{name}.tif", p, shallow=False), name
    cls = torch.cat([o["hand_class"] for o in runner.outputs()], 0).cpu().numpy()
    Image.MAX_IMAGE_PIXELS = None
    np.testing.assert_array_equal(np.asarray(Image.open(paths["hand_class"])), cls.astype(np.uint8))
    assert set(np.unique(cls)) <= {0, 1, 2, 3}


@pytest.mark.gpu
def test_pipeline_files_defaults_are_unchanged(tmp_path):
    from descriptools_b200 import pipeline

    dem, _ = _raw_dem_and_flood(tmp_path)
    paths = pipeline.pipeline_files(dem, tmp_path / "out", river_threshold=300, px=PX, condition=True)
    assert sorted(paths) == sorted(pipeline.STAGE_OUTPUTS)
    with pytest.raises(ValueError):
        pipeline.pipeline_files(dem, tmp_path / "x", river_threshold=300, px=PX, outputs=("hand_class",))


def _nccl_worker(rank, world, port, dem, flood, out_dir, q):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        import torch.distributed as dist

        torch.cuda.set_device(rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
        from descriptools_b200 import bands

        runner = bands.BandRunner(700, 530, PX, 300, 0.4, 0.1)
        runner.load_file(dem, condition=True)
        runner.load_flood(flood)
        runner.step()
        runner.log_indices(0.1)
        res = runner.calibrate("hand", "under")
        runner.write_files(out_dir, outputs=EXTRA)
        dist.barrier()
        dist.destroy_process_group()
        q.put((rank, "ok", repr(res)))
    except Exception:  # pragma: no cover
        import traceback

        q.put((rank, "fail", traceback.format_exc()))


@pytest.mark.gpu
def test_band_files_with_calibration_two_processes_nccl(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from descriptools_b200 import pipeline

    dem, flood = _raw_dem_and_flood(tmp_path)
    got = pipeline.pipeline_files(dem, tmp_path / "ref", river_threshold=300, px=PX, condition=True, flood=flood, outputs=EXTRA)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, str(dem), str(flood), str(tmp_path / "out"), q)) for r in range(2)]
    for p in procs:
        p.start()
    results = sorted((q.get(timeout=600) for _ in procs), key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
    for rank, status, info in results:
        assert status == "ok", f"rank {rank}: {info}"
        assert info == repr(got["calibration"])
    for name in EXTRA:
        assert filecmp.cmp(tmp_path / "ref" / f"{name}.tif", tmp_path / "out" / f"{name}.tif", shallow=False), name
