"""Shared test helpers: golden loaders, the example.py glue, synthetic DEMs, the fused HAND check against
the oracle and a NumPy restatement of the reference's evaluation.py steps used by KAT-1 (evaluation.py:5-9,
12-87, 90-123, 126-171)."""
import hashlib
import os

import numpy as np

import oracle

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
PX = 12.5
RTOL, ATOL = 1e-5, 1e-6


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def load(name):
    return dict(np.load(os.path.join(GOLDEN, name), allow_pickle=False))


def example_inputs():
    z = load("example_inputs.npz")
    shape = tuple(int(v) for v in z["shape"])
    flood = np.unpackbits(z["flood_bits"])[: shape[0] * shape[1]].reshape(shape).astype(np.int8)
    fac = z["fac"].astype(np.int64)
    river = np.where(fac > 128000, 1, 0).astype(np.int8)  # example.py:52
    return dict(dem=z["dem"], fdr=z["fdr"], fac=fac, river=river, flood=flood, hand_class=z["hand_class"])


def synth(rows, cols, seed, holes=True):
    """a conditioned float32 DEM (recipe dtb-synth-v1 + priority flood), with -100 blobs unless holes=False"""
    dem = oracle.synth_dem(rows, cols, 0, seed)
    if holes:
        rng = np.random.default_rng(seed)
        for _ in range(6):
            r, c = int(rng.integers(2, rows - 12)), int(rng.integers(2, cols - 12))
            dem[r:r + int(rng.integers(1, 10)), c:c + int(rng.integers(1, 10))] = -100
        dem[rows // 2, :5] = -100
    return oracle.priority_flood_eps(dem)


def serpentine_d8(rows, cols):
    """one channel through every row, east on even rows, west on odd ones, down at the row ends; it leaves the raster
    below its last cell"""
    d8 = np.zeros((rows, cols), np.uint8)
    for r in range(rows):
        east = r % 2 == 0
        d8[r, :] = 1 if east else 16
        d8[r, cols - 1 if east else 0] = 4
    return d8


def listed_tiles(rows, cols):
    """tiles the compact HAND tile pass handed to the 64-bit pass in the last fused call on a raster of this shape: the
    counter sits in word 32 of the HAND workspace header (csrc/hand.cu, OVF_SLOT)"""
    import torch

    from descriptools_b200 import device
    from descriptools_b200._lib import lib

    ws = device.workspace.get(lib.dtb_hand_workspace_bytes(rows, cols), "hand")
    return int(ws[128:132].view(torch.int32).item())


def misaligned(t):
    """the same values in a contiguous view that starts one element (2, 4 or 8 bytes) into its buffer: not 16-byte
    aligned, so the pointwise and stencil launchers take their scalar / generic kernels"""
    import torch

    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    v = buf[1:].view(t.shape)
    v.copy_(t)
    assert v.data_ptr() % 16 != 0
    return v


def hand_fused_vs_oracle(d8, dem, thr, px=PX, n=0.4, b=0.1, size=None):
    """fused flow accumulation + HAND (entry_done) on a D8 grid against the oracle, with GFI parameters (n, b, size)
    (size defaults to px, as example.py:87 passes it); returns the kernel profile"""
    import torch

    from descriptools_b200 import _lib, device

    size = px if size is None else size
    acc_ref, _ = oracle.flow_accumulation(d8)
    river = (acc_ref > thr).astype(np.int8)
    f_ref, i_ref, h_ref = oracle.flow_hand_index(dem, d8, river, px)
    with np.errstate(all="ignore"):
        g_ref = oracle.gfi(h_ref, acc_ref, i_ref, n, b, size)
    t8, td = torch.from_numpy(d8).cuda(), torch.from_numpy(dem).cuda()
    _lib.profile_enable(True)
    try:
        acc = device.flow_accumulation(t8, fuse_hand_threshold=thr)
        out = device.hand(t8, td, px, acc=acc, river_threshold=thr, gfi_params=(n, b, size), entry_done=True)
        torch.cuda.synchronize()
        prof = _lib.profile_collect()
    finally:
        _lib.profile_enable(False)
    assert out["hand"].dtype == td.dtype
    np.testing.assert_array_equal(acc.cpu().numpy(), acc_ref)
    np.testing.assert_array_equal(out["idx"].cpu().numpy(), i_ref)
    np.testing.assert_array_equal(out["hand"].cpu().numpy(), h_ref)
    np.testing.assert_allclose(out["fdist"].cpu().numpy(), f_ref, rtol=RTOL, atol=0)
    np.testing.assert_allclose(out["gfi"].cpu().numpy(), g_ref, rtol=RTOL, atol=ATOL)
    return prof


# ---- evaluation.py restatement (KAT-1 only) -------------------------------------------
def min_max_scale(mat, mn, mx, nodata):  # evaluation.py:5-9
    scaled = np.where(mat == nodata, np.nan, mat)
    return np.where(np.isnan(mat), scaled, (scaled - mn) / (mx - mn))


def binary_map(desc, th, under=True):  # evaluation.py:90-123
    d = np.where(desc == desc[0, 0], np.nan, desc)
    hit = (d <= th) if under else (d >= th)
    return np.where(np.isnan(d), 0, np.where(hit, 1, 0))


def avaliacao(binary, flood):  # evaluation.py:126-171
    cmp_ = np.where(flood == 1, 2, flood)
    cls = binary + cmp_
    tn, fp, fn, tp = [(cls == k).sum() for k in range(4)]
    c = tp / (tp + fn)
    f = tp / (tp + fn + fp)
    return c, f, cls


def calibration(desc, flood):  # evaluation.py:12-87, direction 'under'
    fit = lambda t: avaliacao(binary_map(desc, t), flood)[1]
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
