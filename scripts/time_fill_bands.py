"""Depression filling over row bands against the single-GPU fill, on a raw (unfilled) dtb-synth-v1 DEM.

    torchrun --nproc_per_node N scripts/time_fill_bands.py [--rows 40000] [--cols 40000] [--out FILE.json]
    python scripts/time_fill_bands.py --local-bands K [...]       (K logical bands on one GPU)

Every rank synthesises only its own rows (device.synth_dem(rows, cols, row0)) and BandRunner.fill_depressions() fills
them; the time is a host clock from a barrier to the end of the call (which ends in a device synchronise on every rank).
Then every rank fills the whole DEM on its own GPU with device.fill_depressions (timed the same way) and compares its
band with the matching rows bit for bit: `verified`.  Rank 0 prints one JSON line and writes it to --out."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist

from descriptools_b200 import bands, device


def gpu_info():
    """name and power limit of every GPU of the node (read-only query)"""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout
        return [dict(zip(("index", "name", "power_limit_w"), (s.strip() for s in line.split(",")))) for line in out.splitlines() if line]
    except (OSError, subprocess.SubprocessError):
        return [{"name": torch.cuda.get_device_name(), "power_limit_w": "unknown"}]


class TimedBand:
    """a Band whose fill calls (synchronous) are timed with the host clock"""

    def __init__(self, b):
        self.b, self.dev, self.init_s, self.solve_s = b, b.dev, 0.0, []

    def fill_halo_items(self):
        return self.b.fill_halo_items()

    def fill_init(self):
        t0 = time.perf_counter()
        self.b.fill_init()
        self.init_s = time.perf_counter() - t0

    def fill_solve(self):
        t0 = time.perf_counter()
        r = self.b.fill_solve()
        self.solve_s.append(time.perf_counter() - t0)
        return r

    def fill_release(self):
        self.b.fill_release()


def local_bands(a):
    """K logical bands on one GPU (LocalExchange), one after the other: rounds, passes and the result are those of K
    GPUs (each SOLVE ends at its band's unique fixed point for the halos it was given); the times are those of one GPU
    doing every band's work -- the wall time on K GPUs is not measured here.  Every band call is timed (host clock around
    synchronous calls)."""
    runner = bands.BandRunner(a.rows, a.cols, 12.5, 128000, nbands=a.local_bands)
    for b in runner.bands:
        b.dem.copy_(device.synth_dem(b.rows, a.cols, b.r0))
    # warm-up: module load
    w = device.synth_dem(256, 256)
    device.fill_depressions(w)
    tb = [TimedBand(b) for b in runner.bands]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    info = bands.fill_rounds(tb, runner.x)
    torch.cuda.synchronize()
    serial_s = time.perf_counter() - t0
    init_s = [round(t.init_s, 4) for t in tb]
    solve_s = [[round(x, 4) for x in t.solve_s] for t in tb]
    got = [(b.r0, b.r1, b.dem.clone()) for b in runner.bands]
    del runner, tb
    torch.cuda.empty_cache()
    full = device.synth_dem(a.rows, a.cols)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    single_passes = device.fill_depressions(full)
    torch.cuda.synchronize()
    single_s = time.perf_counter() - t0
    same = all(bool(torch.equal(full[r0:r1], d)) for r0, r1, d in got)
    res = {"what": "depression filling over row bands, K logical bands on one GPU (LocalExchange) vs device.fill_depressions",
           "dem": f"dtb-synth-v1 raw, {a.rows} x {a.cols}", "bands": a.local_bands, "rounds": info["rounds"],
           "passes_per_band": info["passes"], "one_gpu_all_bands_s": round(serial_s, 3),
           "init_s_per_band": init_s, "solve_s_per_band_per_round": solve_s, "single_gpu_fill_s": round(single_s, 3), "single_gpu_passes": single_passes,
           "verified": same, "gpu": gpu_info(), "torch": torch.__version__}
    line = json.dumps(res)
    print(line, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=40000)
    ap.add_argument("--cols", type=int, default=40000)
    ap.add_argument("--local-bands", type=int, default=0, help="K > 0: K logical bands on one GPU, no torchrun")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.local_bands > 0:
        local_bands(a)
        return
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()

    # warm-up: module load and the NCCL peers, on a raster of one 64-row band per rank
    small = bands.BandRunner(64 * world, 256, 12.5, 100)
    small.bands[0].dem.copy_(device.synth_dem(64, 256, 64 * rank))
    small.fill_depressions()
    del small

    runner = bands.BandRunner(a.rows, a.cols, 12.5, 128000)
    (b,) = runner.bands
    b.dem.copy_(device.synth_dem(b.rows, a.cols, b.r0))
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    dist.barrier()
    t0 = time.perf_counter()
    info = runner.fill_depressions()
    torch.cuda.synchronize()
    band_s = time.perf_counter() - t0
    peak_gb = torch.cuda.max_memory_allocated() / 1e9
    mine = b.dem.clone()
    r0, r1 = b.r0, b.r1
    del runner, b
    torch.cuda.empty_cache()

    full = device.synth_dem(a.rows, a.cols)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    single_passes = device.fill_depressions(full)
    torch.cuda.synchronize()
    single_s = time.perf_counter() - t0
    same = bool(torch.equal(full[r0:r1], mine))
    del full, mine
    device.workspace.release()

    me = {"rank": rank, "rows": [r0, r1], "fill_s": round(band_s, 3), "passes": info["passes"][0], "peak_alloc_gb": round(peak_gb, 2),
          "single_gpu_fill_s": round(single_s, 3), "single_gpu_passes": single_passes, "verified": same, "rounds": info["rounds"]}
    everyone = [None] * world
    dist.all_gather_object(everyone, me)
    if rank == 0:
        res = {"what": "depression filling over row bands (BandRunner.fill_depressions) vs device.fill_depressions on one GPU",
               "dem": f"dtb-synth-v1 raw, {a.rows} x {a.cols}", "gpus": world, "rounds": info["rounds"],
               "band_fill_s": max(e["fill_s"] for e in everyone), "single_gpu_fill_s": everyone[0]["single_gpu_fill_s"],
               "single_gpu_passes": everyone[0]["single_gpu_passes"], "verified": all(e["verified"] for e in everyone),
               "per_rank": everyone, "gpu": gpu_info(), "torch": torch.__version__}
        line = json.dumps(res)
        print(line, flush=True)
        if a.out:
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "w") as f:
                f.write(line + "\n")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
