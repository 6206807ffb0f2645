"""Depression filling over row bands (bands.fill_rounds, dtb_fill_band_f32): the banded fill equals the single-raster
fill (dtb_fill_depressions_f32) and the oracle's priority flood bit for bit.

CPU: the round loop over DistExchange (gloo) and LocalExchange with the NumPy stand-in tests/fill_band_sim.py, and the
argument checks of the C entry points.  GPU: k logical bands on one GPU, a raw DEM file through load_file(condition=True)
and the whole chain, and two processes over NCCL where two GPUs are visible."""
import functools
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import oracle
from fill_band_sim import FillBandSim

PX = 12.5


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _bowl(rows, cols):
    """one depression spanning every band; its only low outlet is on the bottom edge, in the last band"""
    r = np.arange(rows, dtype=np.float64)[:, None]
    c = np.arange(cols, dtype=np.float64)[None, :]
    z = (50.0 + 0.01 * ((r - rows / 2) ** 2 + (c - cols / 2) ** 2)).astype(np.float32)
    z[rows - 1, cols // 2] = 10.0
    return z


@functools.lru_cache(maxsize=None)
def _dem(kind):
    """the test rasters (read-only: callers copy)"""
    if kind == "synth":         # raw; cols not a multiple of 32; 4 bands of exactly 64 rows
        d = oracle.synth_dem(256, 333, 0, 7)
    elif kind == "nodata":      # holes across the seam at row 192, nodata rows right above the seams at 128 and 192
        d = oracle.synth_dem(384, 300, 0, 11)
        d[150:230, 50:120] = -100
        d[127, 150:260] = -100
        d[191, 200:280] = -100
        d[300:310, 0:40] = np.nan
    elif kind == "bowl":
        d = _bowl(256, 256)
    elif kind == "noise":       # pits everywhere
        d = (np.random.default_rng(3).random((320, 200)) * 10).astype(np.float32)
    elif kind == "filled":
        d = oracle.priority_flood_eps(oracle.synth_dem(320, 250, 0, 5))
    else:
        raise KeyError(kind)
    d.setflags(write=False)
    return d


@functools.lru_cache(maxsize=None)
def _want(kind):
    w = oracle.priority_flood_eps(_dem(kind).copy())
    w.setflags(write=False)
    return w


# ---- CPU: the round loop with the NumPy stand-in ----------------------------------------------------------
def _sim_bands(dem, edges, indices):
    n = len(edges) - 1
    return [FillBandSim(dem, edges[i], edges[i + 1], i == 0, i == n - 1) for i in indices]


@functools.lru_cache(maxsize=None)
def _sim_rounds(kind, k):
    """rounds of the k-band fill with the stand-in.  Every SOLVE ends at its band's unique fixed point for the halo rows
    it was given, whatever order the cells are relaxed in, so the sequence of rounds is the algorithm's own: the device's
    tiles, the stand-in's Jacobi sweeps, one process or k must all stop in this round."""
    from descriptools_b200 import bands

    dem = _dem(kind)
    bs = _sim_bands(dem, bands.band_edges(dem.shape[0], k), range(k))
    info = bands.fill_rounds(bs, bands.LocalExchange(k))
    np.testing.assert_array_equal(np.concatenate([b.band for b in bs], 0), _want(kind))
    return info["rounds"]


def _gloo_worker(rank, world, port, kinds, q):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        import torch.distributed as dist

        dist.init_process_group("gloo", rank=rank, world_size=world)
        from descriptools_b200 import bands

        x = bands.DistExchange()
        out = {}
        for kind in kinds:
            dem = _dem(kind)
            edges = bands.band_edges(dem.shape[0], world)
            (b,) = _sim_bands(dem, edges, [rank])
            info = bands.fill_rounds([b], x)
            out[kind] = (b.band.copy(), info["rounds"], b.ws is None)
        dist.barrier()
        dist.destroy_process_group()
        q.put((rank, "ok", out))
    except Exception:  # pragma: no cover
        import traceback

        q.put((rank, "fail", traceback.format_exc()))


@pytest.mark.parametrize("world", [2, 3])
def test_fill_rounds_gloo_match_oracle(world):
    """one band per process over torch.distributed (gloo): the stacked bands == oracle.priority_flood_eps"""
    kinds = ["synth", "nodata", "bowl"]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gloo_worker, args=(r, world, port, kinds, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = sorted(q.get(timeout=600) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    for rank, status, info in results:
        assert status == "ok", f"rank {rank}: {info}"
    for kind in kinds:
        got = np.concatenate([info[kind][0] for _, _, info in results], 0)
        np.testing.assert_array_equal(got, _want(kind), err_msg=kind)
        assert {info[kind][1] for _, _, info in results} == {_sim_rounds(kind, world)}, kind  # the same rounds as in one process
        assert all(info[kind][2] for _, _, info in results)  # workspace released


@pytest.mark.parametrize("k", [1, 2, 3, 4])
@pytest.mark.parametrize("kind", ["synth", "bowl", "noise", "filled"])
def test_fill_rounds_local_match_oracle(kind, k):
    """k bands in one process (LocalExchange) with the stand-in"""
    from descriptools_b200 import bands

    dem = _dem(kind)
    edges = bands.band_edges(dem.shape[0], k)
    bs = _sim_bands(dem, edges, range(k))
    info = bands.fill_rounds(bs, bands.LocalExchange(k))
    np.testing.assert_array_equal(np.concatenate([b.band for b in bs], 0), _want(kind))
    assert len(info["passes"]) == k
    if kind == "filled":
        np.testing.assert_array_equal(_want(kind), dem)
    if k == 1:
        assert info["rounds"] == 1


def test_fill_rounds_cap_raises():
    from descriptools_b200 import bands

    dem = _dem("bowl")
    bs = _sim_bands(dem, bands.band_edges(dem.shape[0], 4), range(4))
    with pytest.raises(RuntimeError, match="did not converge"):
        bands.fill_rounds(bs, bands.LocalExchange(4), max_rounds=1)
    assert all(b.ws is None for b in bs)


def test_fill_band_argument_validation_needs_no_device():
    import ctypes

    from descriptools_b200 import _lib

    L = _lib.lib
    assert L.dtb_fill_band_workspace_bytes(100, 70) == L.dtb_fill_workspace_bytes(100, 70)
    assert L.dtb_fill_band_workspace_bytes(0, 70) == 0
    p, s = ctypes.c_int(0), ctypes.c_int(0)
    ws = L.dtb_fill_band_workspace_bytes(100, 70)
    args = lambda **kw: dict(dict(dem=1, rows=100, cols=70, above=1, below=1, mode=_lib.DTB_FILL_SOLVE, ws=1, nbytes=ws), **kw)

    def call(**kw):
        a = args(**kw)
        return L.dtb_fill_band_f32(a["dem"], a["rows"], a["cols"], a["above"], a["below"], a["mode"], a["ws"], a["nbytes"],
                                   ctypes.byref(p), ctypes.byref(s), None)

    assert call(dem=None) == -1
    assert call(ws=None) == -1
    assert call(rows=0) == -1 and call(cols=-3) == -1
    assert call(above=2) == -1 and call(below=-1) == -1
    assert call(mode=7) == -1
    assert call(nbytes=ws - 1) == -3
    assert call(mode=_lib.DTB_FILL_INIT, nbytes=16) == -3


# ---- GPU: k logical bands on one GPU ----------------------------------------------------------------------
def _runner_fill(dem, k):
    from descriptools_b200 import bands

    rows, cols = dem.shape
    runner = bands.BandRunner(rows, cols, PX, 100, nbands=k)
    runner.load([torch.from_numpy(dem[a:b].copy()) for a, b in zip(runner.edges, runner.edges[1:])])
    info = runner.fill_depressions()
    torch.cuda.synchronize()
    got = torch.cat([b.dem for b in runner.bands], 0).cpu().numpy()
    assert all(b.ws_fill is None for b in runner.bands)
    return got, info


@functools.lru_cache(maxsize=None)
def _single_gpu(kind):
    from descriptools_b200 import device

    t = torch.from_numpy(_dem(kind).copy()).cuda()
    device.fill_depressions(t)
    return t.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 3, 4])
@pytest.mark.parametrize("kind", ["synth", "nodata", "bowl", "noise", "filled"])
def test_band_fill_equals_single_gpu_and_oracle(kind, k):
    """BandRunner(nbands=k).fill_depressions() == device.fill_depressions == oracle.priority_flood_eps, bit for bit"""
    dem = _dem(kind)
    got, info = _runner_fill(dem, k)
    single = _single_gpu(kind)
    np.testing.assert_array_equal(single, _want(kind))
    np.testing.assert_array_equal(got, single)
    assert len(info["passes"]) == k and all(p > 0 for p in info["passes"])
    # the device stops in the round the algorithm does (see _sim_rounds): a kernel that lowered a seam row without
    # flagging it, or a driver that exchanged stale rows, would stop elsewhere or not match bit for bit
    assert info["rounds"] == _sim_rounds(kind, k)
    if kind == "filled":
        np.testing.assert_array_equal(got, dem)
    if k == 1:
        assert info["rounds"] == 1
    elif kind == "filled":
        # one round only without seams: with seams, INIT's row-scan bound lies above the surface on the seam rows, so the
        # first SOLVE lowers them and the neighbours need another round
        assert info["rounds"] > 1


@pytest.mark.gpu
def test_load_file_condition_then_step_equals_single_gpu(tmp_path):
    """a raw DEM GeoTIFF -> load_file(condition=True) over 3 bands -> step(): all seven rasters == pipeline.run_device on
    the single-GPU-filled DEM"""
    import descriptools_b200.raster as rio
    from descriptools_b200 import bands, device, pipeline

    raw = oracle.synth_dem(448, 330, 0, 19)
    hole = np.zeros(raw.shape, bool)
    hole[120:170, 40:90] = True   # across the seam at row 128 (3 bands: 0, 128, 320, 448)
    hole[319, 100:200] = True     # a nodata row right above the seam at row 320
    p = tmp_path / "raw.tif"
    with rio.open(p, "w", width=330, height=448, dtype="float32", compress="lzw", predictor=3, tiled=True, blockxsize=128,
                  blockysize=128, nodata=-9999.0) as dst:
        dst.write(np.where(hole, np.float32(-9999.0), raw))
    clean = torch.from_numpy(np.where(hole, np.float32(-100), raw)).cuda()
    device.fill_depressions(clean)
    assert (clean.cpu().numpy() != np.where(hole, np.float32(-100), raw)).sum() > 50  # there were pits
    ref = pipeline.run_device(clean, PX, 300)
    runner = bands.BandRunner(448, 330, PX, 300, 0.4, 0.1, nbands=3)
    assert runner.edges == [0, 128, 320, 448]
    runner.load_file(p, condition=True)
    np.testing.assert_array_equal(torch.cat([b.dem for b in runner.bands], 0).cpu().numpy(), clean.cpu().numpy())
    runner.step()
    torch.cuda.synchronize()
    outs = runner.outputs()
    for name in ("slope", "d8", "acc", "idx", "fdist", "hand", "gfi"):
        got = torch.cat([o[name] for o in outs], 0).cpu().numpy()
        np.testing.assert_array_equal(got, ref[name].cpu().numpy(), err_msg=name)


def _nccl_worker(rank, world, port, kinds, q):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        import torch.distributed as dist

        torch.cuda.set_device(rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
        from descriptools_b200 import bands

        out = {}
        for kind in kinds:
            dem = _dem(kind)
            rows, cols = dem.shape
            runner = bands.BandRunner(rows, cols, PX, 100)
            (b,) = runner.bands
            runner.load([torch.from_numpy(dem[b.r0:b.r1].copy())])
            info = runner.fill_depressions()
            out[kind] = (b.dem.cpu().numpy(), info["rounds"])
        dist.barrier()
        dist.destroy_process_group()
        q.put((rank, "ok", out))
    except Exception:  # pragma: no cover
        import traceback

        q.put((rank, "fail", traceback.format_exc()))


@pytest.mark.gpu
def test_band_fill_two_processes_nccl():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    kinds = ["nodata", "bowl"]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, kinds, q)) for r in range(2)]
    for p in procs:
        p.start()
    results = sorted(q.get(timeout=600) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    for rank, status, info in results:
        assert status == "ok", f"rank {rank}: {info}"
    for kind in kinds:
        got = np.concatenate([info[kind][0] for _, _, info in results], 0)
        np.testing.assert_array_equal(got, _want(kind), err_msg=kind)
        assert results[0][2][kind][1] == results[1][2][kind][1]
