"""evaluation.py -- drop-in for descriptools/evaluation.py (reference: evaluation.py:5-211).

Min-max scaling, threshold calibration, binary map and the performance indexes of a terrain descriptor against a
benchmark flood map.  The reference evaluates one threshold per full-raster NumPy pass (61 passes per calibration,
evaluation.py:32-85); here the rasters go to the device once and every stage of the search is ONE pass that yields the
confusion counts of all its thresholds (csrc/evaluation.cu).  Same names, arguments, return values and side effects
as the reference -- including `avaliacao` / `calibration` rewriting the benchmark array in place
(1 -> 2, -100 -> 0: evaluation.py:149-150).
"""
import ctypes

import numpy as np
import torch

from . import device
from ._lib import check, lib


def _dev_desc(descriptor_matrix):
    """descriptor on the device (float32 stays float32, everything else is compared as float64) + its nodata value"""
    d = np.asarray(descriptor_matrix)
    if d.dtype != np.float32:
        d = d.astype(np.float64, copy=False)
    d = np.ascontiguousarray(d)
    nodata = float(d.flat[0])  # binary_map: descriptor_matrix == descriptor_matrix[0, 0] -> NaN (evaluation.py:111)
    device.require_cuda()
    return torch.from_numpy(d).cuda(), nodata, d.dtype == np.float64


def _remap_inplace(comparison_flood_map):
    comparison_flood_map[comparison_flood_map == 1] = 2      # evaluation.py:149
    comparison_flood_map[comparison_flood_map == -100] = 0   # evaluation.py:150


def _flood_dev(comparison):
    c = np.asarray(comparison)
    if c.dtype != np.int8:
        if c.size and (c.min() < -128 or c.max() > 127):
            raise ValueError("benchmark flood map values must fit int8")
        c = c.astype(np.int8)
    return torch.from_numpy(np.ascontiguousarray(c)).cuda()


class _Counter:
    """confusion counts of a list of thresholds in one device pass"""

    def __init__(self, desc_t, is_f64, nodata, flood_t, under):
        self.d, self.is_f64, self.nodata, self.f = desc_t, is_f64, nodata, flood_t
        self.under = 1 if under == "under" else 0
        self.ws = torch.empty(4 * 33 * 8, dtype=torch.uint8, device=desc_t.device)

    def counts(self, thresholds):
        th = np.asarray(thresholds, np.float64)
        if not self.is_f64:
            # NumPy compares a float32 descriptor with a Python-float threshold in float32 (the scalar is cast down,
            # evaluation.py:32-85 under NEP 50): round the thresholds the same way before the f64 comparison on the device
            th = th.astype(np.float32).astype(np.float64)
        order = np.argsort(th, kind="stable")
        th = th[order]
        uniq, inv = np.unique(th, return_inverse=True)  # the kernel wants strictly ascending thresholds
        out = np.zeros((len(uniq), 4), np.int64)
        for a in range(0, len(uniq), 32):
            part = np.ascontiguousarray(uniq[a:a + 32])
            res = np.zeros((len(part), 4), np.int64)
            check(lib.dtb_eval_counts(self.d.data_ptr(), 1 if self.is_f64 else 0, self.f.data_ptr(), self.d.numel(), self.nodata,
                                      part.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), len(part), self.under,
                                      res.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), self.ws.data_ptr(), self.ws.numel(),
                                      torch.cuda.current_stream().cuda_stream), "dtb_eval_counts")
            out[a:a + len(part)] = res
        back = np.empty(len(th), np.int64)
        back[order] = inv
        return out[back]  # row i <-> thresholds[i]: (tn, fp, fn, tp)


def minMaxScale(mat, mn, mx, nodata):
    """evaluation.py:5-9: nodata -> NaN, the rest (mat - mn) / (mx - mn); float64."""
    m = np.ascontiguousarray(mat)
    kinds = {np.dtype(np.float32): 0, np.dtype(np.float64): 1, np.dtype(np.int16): 2}
    if m.dtype not in kinds:
        m = m.astype(np.float64)
    device.require_cuda()
    t = torch.from_numpy(m).cuda()
    out = torch.empty(m.shape, dtype=torch.float64, device=t.device)
    check(lib.dtb_minmax_scale(t.data_ptr(), kinds[m.dtype], t.numel(), float(mn), float(mx), float(nodata), out.data_ptr(),
                               torch.cuda.current_stream().cuda_stream), "dtb_minmax_scale")
    return out.cpu().numpy()


def search_threshold(counts):
    """The threshold search of calibration (evaluation.py:32-87): five stages of thresholds on the scaled descriptor, the
    first three in steps of 0.25, then 0.1, 0.01, 0.001 and 0.0001 around the best so far, with the reference's tie rules
    (the stage-1 pick, `>=` in stage 2, `>` after it).  `counts(thresholds)` -> (len, 4) int64 rows (tn, fp, fn, tp), one
    call per stage: the drop-in, device.calibrate and the row-band driver differ only in where those counts come from.

    Returns (threshold, correctness index, fit index, (tn, fp, fn, tp)) at the threshold, taken from the last stage's
    counts: the final threshold is always a member of that stage's list (its centre, if nothing beats it)."""
    def fits(c):
        # fit index: tp / (tp + fn + fp)  (evaluation.py:192-211); numpy int division like the reference
        with np.errstate(divide="ignore", invalid="ignore"):
            return c[:, 3] / (c[:, 3] + c[:, 2] + c[:, 1])

    f1, f2, f3 = fits(counts([25 / 100, 50 / 100, 75 / 100]))  # evaluation.py:32-37
    if f3 > f2:
        fit_index, iteration_value = (f3, 75) if f3 > f1 else (f1, 25)
    else:
        fit_index, iteration_value = (f2, 50) if f2 > f1 else (f1, 25)
    threshold = None
    steps = list(range(iteration_value - 20, iteration_value + 30, 10))  # evaluation.py:54-59
    for i, v in zip(steps, fits(counts([i / 100 for i in steps]))):
        if v >= fit_index:
            fit_index, threshold = v, i
    iteration_value = threshold
    steps = list(range(iteration_value - 5, iteration_value + 6, 1))  # evaluation.py:61-66
    for i, v in zip(steps, fits(counts([i / 100 for i in steps]))):
        if v > fit_index:
            fit_index, threshold = v, i
    for scale in (1000, 10000):  # evaluation.py:68-85
        iteration_value = threshold * 10
        threshold = iteration_value
        steps = list(range(iteration_value - 10, iteration_value + 11, 1))
        last = counts([i / scale for i in steps])
        for i, v in zip(steps, fits(last)):
            if v > fit_index:
                fit_index, threshold = v, i
    tn, fp, fn, tp = (int(v) for v in last[steps.index(threshold)])
    with np.errstate(divide="ignore", invalid="ignore"):
        correctness_index = np.int64(tp) / np.int64(fn + tp)          # evaluation.py:174-190
        fit = np.int64(tp) / np.int64(tp + fn + fp)
    return threshold / 10000, float(correctness_index), float(fit), (tn, fp, fn, tp)


def calibration(descriptor_matrix, comparison_matrix, under):
    """Best threshold for the linear binary classification -- evaluation.py:12-87 (same search, same tie rules).
    Like the reference it leaves `comparison_matrix` remapped in place (1 -> 2, -100 -> 0)."""
    d, nodata, is_f64 = _dev_desc(descriptor_matrix)
    _remap_inplace(comparison_matrix)  # what the first avaliacao call of the reference does (evaluation.py:32)
    k = _Counter(d, is_f64, nodata, _flood_dev(comparison_matrix), under)
    return search_threshold(k.counts)[0]


def counts_from_hist(hist, k: int, under) -> np.ndarray:
    """(k, 4) int64 (tn, fp, fn, tp) of the k thresholds a 4 x 33 histogram of dtb_eval_hist was taken for (host only)"""
    h = np.ascontiguousarray(np.asarray(hist).reshape(-1), dtype=np.int64)
    if h.size != 4 * 33:
        raise ValueError("a calibration histogram has 4 x 33 entries")
    out = np.zeros((k, 4), np.int64)
    check(lib.dtb_eval_counts_from_hist(h.ctypes.data, int(k), 1 if under == "under" else 0,
                                        out.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))), "dtb_eval_counts_from_hist")
    return out


def unique_ends(extrema):
    """(mn, mx) = (np.unique(x)[1], np.unique(x)[-1]) (example.py:113-115) from the extrema rows of the parts of x (rows of
    dtb_eval_extrema: lo, second lo, hi, distinct non-NaN values capped at 2, NaN seen).  np.unique keeps one NaN and sorts
    it last, so a NaN anywhere makes mx NaN, and mn is NaN when only one non-NaN value exists.  Fewer than two values
    raise ValueError (the reference's IndexError at elements[1])."""
    e = np.asarray(extrema, dtype=np.float64).reshape(-1, 5)
    cnt = e[:, 3].astype(np.int64)
    small = np.unique(np.concatenate([e[cnt >= 1, 0], e[cnt >= 2, 1]]))[:2]  # two smallest distinct values of the union
    has_nan = bool((e[:, 4] != 0).any())
    if len(small) + has_nan < 2:
        raise ValueError("the descriptor has fewer than two distinct values: np.unique(descriptor)[1] does not exist")
    mn = small[1] if len(small) >= 2 else np.nan
    mx = np.nan if has_nan else e[cnt >= 1, 2].max()
    return float(mn), float(mx)


def binary_map(descriptor_matrix, threshold, under):
    """evaluation.py:90-123: 1 where the descriptor is on the flooded side of the threshold, 0 elsewhere / nodata."""
    d, nodata, is_f64 = _dev_desc(descriptor_matrix)
    out = torch.empty(d.shape, dtype=torch.int8, device=d.device)
    if not is_f64:
        threshold = float(np.float32(threshold))  # float32 descriptor: NumPy compares in float32 (see _Counter.counts)
    check(lib.dtb_eval_class_map(d.data_ptr(), 1 if is_f64 else 0, None, d.numel(), nodata, float(threshold),
                                 1 if under == "under" else 0, out.data_ptr(), None, torch.cuda.current_stream().cuda_stream),
          "dtb_eval_class_map")
    return out.cpu().numpy().astype(np.int64)  # np.where(..., 1, 0) is int64 in the reference


def avaliacao(descriptor_flood_map, comparison_flood_map):
    """Correctness index, fit index and the class map (0 tn, 1 fp, 2 fn, 3 tp) -- evaluation.py:126-171.
    Rewrites `comparison_flood_map` in place like the reference (1 -> 2, -100 -> 0)."""
    _remap_inplace(comparison_flood_map)
    b = np.ascontiguousarray(descriptor_flood_map)
    device.require_cuda()
    bt = torch.from_numpy(b.astype(np.float32)).cuda()  # 0/1 map: threshold 0.5, 'over'
    ft = _flood_dev(comparison_flood_map)
    counts = _Counter(bt, False, float("nan"), ft, "over").counts([0.5])[0]
    cls = torch.empty(bt.shape, dtype=torch.int8, device=bt.device)
    check(lib.dtb_eval_class_map(bt.data_ptr(), 0, ft.data_ptr(), bt.numel(), float("nan"), 0.5, 0, None, cls.data_ptr(),
                                 torch.cuda.current_stream().cuda_stream), "dtb_eval_class_map")
    with np.errstate(divide="ignore", invalid="ignore"):
        correctness_index = counts[3] / (counts[2] + counts[3])        # evaluation.py:174-190
        fit_index = counts[3] / (counts[3] + counts[2] + counts[1])    # evaluation.py:192-211
    result = cls.cpu().numpy().astype(np.result_type(b.dtype, np.asarray(comparison_flood_map).dtype))
    return correctness_index, fit_index, result
