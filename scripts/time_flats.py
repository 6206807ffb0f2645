"""Device time of the exact fill, flat resolution and the epsilon fill on the synthetic DEM quantised to 0.1 m (which
makes flats), at each size given (default 10000 and 40000, square).  Each size is first run once untimed, which loads
the modules and leaves every workspace allocated at that size, so no timed window allocates; then REPS (3) repetitions,
each on a freshly generated DEM, exact route then epsilon route.  CUDA events around each call; every call ends in a
device synchronise (the fills and resolve_flats read flags back), so the event times are the calls' own.  Prints the
card's name, power limit and top SM clock, then one JSON line per size with the median and range over the repetitions.

    python scripts/time_flats.py [N ...]
"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from descriptools_b200 import device  # noqa: E402


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    r = fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1), r


def quantised(n):
    dem = device.synth_dem(n, n)
    dem.mul_(10).round_().div_(10)
    return dem


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else torch.cuda.get_device_name()


REPS = 3


def one_round(n, px):
    """(times in ms, counts) of one exact route and one epsilon route at n x n, each on a fresh DEM"""
    dem = quantised(n)
    t, c = {}, {}
    t["exact_fill"], c["exact_fill_passes"] = timed(lambda: device.fill_depressions(dem, epsilon=False))
    _, d8 = device.slope_d8(dem, px, want_slope=False)
    c["flat_cells"] = int(((d8 == 0) & (dem > -100)).sum())
    before = d8.clone()
    t["resolve_flats"], left = timed(lambda: device.resolve_flats(dem, d8))
    c["codes_written"] = int((d8 != before).sum())
    del before
    dem = quantised(n)
    t["eps_fill"], c["eps_fill_passes"] = timed(lambda: device.fill_depressions(dem))
    _, d8 = device.slope_d8(dem, px, want_slope=False)
    t["resolve_flats_no_flat"], left_eps = timed(lambda: device.resolve_flats(dem, d8))  # one pass over the codes
    assert left == 0 and left_eps == 0
    return t, c


def main():
    sizes = [int(a) for a in sys.argv[1:]] or [10000, 40000]
    px = 12.5
    print(json.dumps({"card": card()}), flush=True)
    for n in sizes:
        one_round(n, px)  # warm-up: modules loaded, workspaces of this size allocated
        runs = [one_round(n, px) for _ in range(REPS)]
        row = dict(rows=n, cols=n, reps=REPS, **runs[0][1])
        for k in runs[0][0]:
            v = sorted(r[0][k] for r in runs)
            row[k + "_ms"] = round(v[len(v) // 2], 3)
            row[k + "_ms_range"] = [round(v[0], 3), round(v[-1], 3)]
        row["peak_gb"] = round(torch.cuda.max_memory_allocated() / 1e9, 1)
        print(json.dumps(row), flush=True)
        device.workspace.release()
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
