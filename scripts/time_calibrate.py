"""Calibration of HAND against a flood map: the fused device path (device.calibrate: extrema pass, 5 histogram passes that
min-max scale on load, class map) against the materialising path (dtb_minmax_scale to a float64 raster, 5 x dtb_eval_counts
on it, the float64 class map), alternating in one run, timed with CUDA events.

Input: the conditioned synthetic DEM (dtb-synth-v1) at each size, HAND from pipeline.run_device, and a seeded synthetic
benchmark: HAND <= 3 m, 5 % of the cells flipped, 2 % set to -100.  Both paths must give the same threshold, counts and
class map.  Achieved GB/s use the algorithmic bytes per cell (f32 HAND, int8 benchmark, int8 class map):
fused: extrema 4, histogram 4 + 1 per pass, class map 4 + 1 + 1 = 35 B/cell for the calibration;
materialising: scale 4 + 8, counts 8 + 1 per pass, class map 8 + 1 + 1 = 67 B/cell (plus the 8 B/cell raster it holds).

    python scripts/time_calibrate.py [out.json] [sizes, default 10000,40000] [reps, default 5]
"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from descriptools_b200 import device, evaluation, pipeline  # noqa: E402
from descriptools_b200._lib import check, lib  # noqa: E402

PX, THR = 12.5, 2000


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()[0]
        info["power_limit"], info["max_sm_clock"] = (v.strip() for v in q.split(","))
    except Exception as e:  # noqa: BLE001
        info["power_limit"] = f"unavailable ({e})"
    return info


class Timer:
    def __init__(self):
        self.ms = {}

    def __call__(self, name, fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        b.synchronize()
        self.ms.setdefault(name, []).append(a.elapsed_time(b))
        return out


def fused(hand, flood, tm):
    """device.calibrate step by step, each step timed (the host work between passes included in 'calibrate' only)"""
    ext = tm("extrema", lambda: device.eval_extrema(hand))
    mn, mx = evaluation.unique_ends(ext.cpu().numpy())
    corner = float(hand[0, 0])
    hist = torch.zeros(4 * 33, dtype=torch.int64, device=hand.device)
    stage = [0]

    def counts(ths):
        hist.zero_()
        tm(f"hist_{stage[0]}", lambda: device.eval_hist(hand, flood, mn, mx, corner, ths, "under", hist))
        stage[0] += 1
        return evaluation.counts_from_hist(hist.cpu().numpy(), len(ths), "under")

    th, c, f, cnt = evaluation.search_threshold(counts)
    cls = tm("class_map", lambda: device.eval_class(hand, flood, mn, mx, corner, th, "under"))
    return th, cnt, cls


def materialising(hand, flood, scaled, tm):
    """the float64 path: np.unique's ends from the extrema pass (not timed here), then dtb_minmax_scale, the counts of every
    stage on the scaled raster (dtb_eval_counts, synchronous) and the f64 class map"""
    mn, mx = evaluation.unique_ends(device.eval_extrema(hand).cpu().numpy())
    st = torch.cuda.current_stream().cuda_stream
    tm("scale_f64", lambda: check(lib.dtb_minmax_scale(hand.data_ptr(), 0, hand.numel(), mn, mx, -100.0, scaled.data_ptr(), st),
                                  "dtb_minmax_scale"))
    nd = float(scaled[0, 0])
    ctr = evaluation._Counter(scaled, True, nd, flood, "under")
    stage = [0]

    def counts(ths):
        out = tm(f"counts_f64_{stage[0]}", lambda: ctr.counts(ths))
        stage[0] += 1
        return out

    th, c, f, cnt = evaluation.search_threshold(counts)
    cls = torch.empty(hand.shape, dtype=torch.int8, device=hand.device)
    tm("class_map_f64", lambda: check(lib.dtb_eval_class_map(scaled.data_ptr(), 1, flood.data_ptr(), scaled.numel(), nd, th, 1, None,
                                                             cls.data_ptr(), st), "dtb_eval_class_map"))
    return th, cnt, cls


def run(n, reps):
    dem = device.conditioned_dem(n, n)
    res = pipeline.run_device(dem, PX, THR)
    hand = res["hand"]
    del res, dem
    torch.cuda.empty_cache()
    g = torch.Generator(device="cuda").manual_seed(20261022)
    flood = ((hand <= 3) & (hand != -100)).to(torch.int8)
    flip = torch.rand(hand.shape, generator=g, device="cuda") < 0.05
    flood[flip] = 1 - flood[flip]
    flood[torch.rand(hand.shape, generator=g, device="cuda") < 0.02] = -100
    del flip
    scaled = torch.empty(hand.shape, dtype=torch.float64, device="cuda")
    cells = hand.numel()
    # warm-up of both paths, and the check that they agree
    tf, tmat = Timer(), Timer()
    a = fused(hand, flood, tf)
    b = materialising(hand, flood, scaled, tmat)
    assert a[0] == b[0] and a[1] == b[1], (a[:2], b[:2])
    assert torch.equal(a[2], b[2])
    whole = Timer()
    tf, tmat = Timer(), Timer()
    for _ in range(reps):  # alternating
        whole("fused_calibrate", lambda: device.calibrate(hand, flood, "under"))
        whole("materialising_calibrate", lambda: materialising(hand, flood, scaled, tmat))
        fused(hand, flood, tf)
    med = lambda v: float(np.median(v))
    bytes_per = {"extrema": 4, "class_map": 6, "scale_f64": 12, "class_map_f64": 10}
    kern = {}
    for name, v in {**tf.ms, **tmat.ms}.items():
        b = bytes_per.get(name, 5 if name.startswith("hist_") else 9)
        kern[name] = {"ms": med(v), "GB_per_s": b * cells / med(v) / 1e6, "bytes_per_cell": b}
    out = {"cells": cells, "threshold": a[0], "counts": list(a[1]), "kernels": kern,
           "fused_calibrate_ms": med(whole.ms["fused_calibrate"]), "materialising_calibrate_ms": med(whole.ms["materialising_calibrate"]),
           "fused_bytes_per_cell": 35, "materialising_bytes_per_cell": 67}
    for k in ("fused", "materialising"):
        ms = out[f"{k}_calibrate_ms"]
        out[f"{k}_calibrate_GB_per_s"] = out[f"{k}_bytes_per_cell"] * cells / ms / 1e6
    del scaled, hand, flood
    torch.cuda.empty_cache()
    return out


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else None
    sizes = [int(s) for s in (sys.argv[2] if len(sys.argv) > 2 else "10000,40000").split(",")]
    reps = int(sys.argv[3]) if len(sys.argv) > 3 else 5
    device.require_cuda()
    result = {"card": card(), "reps": reps, "timing": "CUDA events, median of the alternating repetitions; whole calls include "
              "their host syncs (one per stage)", "sizes": {}}
    for n in sizes:
        result["sizes"][f"{n}x{n}"] = run(n, reps)
        print(json.dumps({f"{n}x{n}": result["sizes"][f"{n}x{n}"]}), flush=True)
    if path:
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
        with open(path, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
