"""The chain's seven rasters written from row bands (BandRunner.write_raster) against pipeline_files' write phase on one GPU.

    torchrun --nproc_per_node N scripts/time_band_files.py [--rows 40000] [--cols 40000] [--out FILE.json]
    python scripts/time_band_files.py --local-bands K [...]       (K logical bands on one GPU)

Every band synthesises its own rows of a raw dtb-synth-v1 DEM, fills it (fill_depressions) and runs step(); then each
raster is written with the metadata pipeline_files uses (pipeline.output_meta: LZW, 256 x 256 tiles, predictor 3 / 2).
Per raster: the file's bytes, the encode time (the device encoder of every local band, host clock around synchronous
calls), and the whole write_raster call (host clock from a barrier; it ends when the file is closed); write = whole -
encode is the hand-off, the collectives, the copies to pinned memory and the file writes.  Files go to --dir (default:
a temporary directory) and are written without fsync, as pipeline_files does.
With --local-bands, every raster is also written from the whole raster on the same GPU with
raster.write_from_device(encode="device") -- pipeline_files' write phase -- timed the same way, and the two files are
compared byte for byte (`identical`).  Rank 0 prints one JSON line and writes it to --out."""
import argparse
import filecmp
import json
import os
import shutil
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist

from descriptools_b200 import bands, device, pipeline
from descriptools_b200 import raster as rio

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from time_fill_bands import gpu_info  # noqa: E402


class TimedEncoder:
    """bands.device_encoder with a host clock around every call (synchronised: the streams are encoded)"""

    def __init__(self):
        self.s = 0.0

    def __call__(self, lay, t, c0, c1):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = bands.device_encoder(lay, t, c0, c1)
        torch.cuda.synchronize()
        self.s += time.perf_counter() - t0
        return r


def run_chain(a, runner):
    for b in runner.bands:
        b.dem.copy_(device.synth_dem(b.rows, a.cols, b.r0))
    runner.fill_depressions()
    runner.step()
    torch.cuda.synchronize()


def write_bands(runner, path, name, x):
    per_band = [o[name] for o in runner.outputs()]
    enc = TimedEncoder()
    if isinstance(x, bands.DistExchange):
        dist.barrier()
    t0 = time.perf_counter()
    bands.write_raster(runner.bands, x, path, per_band, pipeline.output_meta(name, per_band[0].dtype.is_floating_point), encoder=enc)
    torch.cuda.synchronize()
    total = time.perf_counter() - t0
    return dict(bytes=os.path.getsize(path), encode_s=round(enc.s, 3), write_s=round(total - enc.s, 3), total_s=round(total, 3))


def emit(a, res):
    line = json.dumps(res)
    print(line, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


def local_bands(a, out_dir):
    """K logical bands on one GPU, one after the other: the times are those of one GPU doing every band's work (wall
    times on K GPUs are not measured here)"""
    runner = bands.BandRunner(a.rows, a.cols, 12.5, 128000, nbands=a.local_bands)
    run_chain(a, runner)
    # warm-up: module load, the encoder on a small raster
    small = torch.zeros((512, 512), dtype=torch.float32, device="cuda")
    rio.write_from_device(os.path.join(out_dir, "warm.tif"), small, encode="device", **pipeline.output_meta("slope", True))
    rasters, total = {}, {"bands_s": 0.0, "single_gpu_s": 0.0}
    for name in pipeline.STAGE_OUTPUTS:
        p_band, p_one = os.path.join(out_dir, f"{name}_bands.tif"), os.path.join(out_dir, f"{name}_one.tif")
        r = write_bands(runner, p_band, name, runner.x)
        whole = torch.cat([o[name] for o in runner.outputs()], 0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rio.write_from_device(p_one, whole, encode="device", **pipeline.output_meta(name, whole.dtype.is_floating_point))
        torch.cuda.synchronize()
        r["single_gpu_write_from_device_s"] = round(time.perf_counter() - t0, 3)
        del whole
        r["identical"] = filecmp.cmp(p_band, p_one, shallow=False)
        os.remove(p_band)
        os.remove(p_one)
        rasters[name] = r
        total["bands_s"] += r["total_s"]
        total["single_gpu_s"] += r["single_gpu_write_from_device_s"]
    emit(a, {"what": "seven chain rasters written from K logical row bands on one GPU (bands.write_raster, LocalExchange) vs "
                     "raster.write_from_device(encode='device') of the whole raster (pipeline_files' write phase)",
             "dem": f"dtb-synth-v1 raw, filled, {a.rows} x {a.cols}", "bands": a.local_bands, "meta": "LZW, 256 x 256 tiles, predictor 3 / 2",
             "rasters": rasters, "bands_total_s": round(total["bands_s"], 3), "single_gpu_total_s": round(total["single_gpu_s"], 3),
             "identical": all(r["identical"] for r in rasters.values()), "gpu": gpu_info(), "torch": torch.__version__})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=40000)
    ap.add_argument("--cols", type=int, default=40000)
    ap.add_argument("--local-bands", type=int, default=0, help="K > 0: K logical bands on one GPU, no torchrun")
    ap.add_argument("--dir", default=None, help="where the files go (shared by all ranks); default: a temporary directory")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.local_bands > 0:
        out_dir = a.dir or tempfile.mkdtemp(prefix="band_files_")
        os.makedirs(out_dir, exist_ok=True)
        try:
            local_bands(a, out_dir)
        finally:
            if a.dir is None:
                shutil.rmtree(out_dir, ignore_errors=True)
        return
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    out_dir = [a.dir or (tempfile.mkdtemp(prefix="band_files_") if rank == 0 else None)]
    dist.broadcast_object_list(out_dir, src=0)
    out_dir = out_dir[0]
    runner = bands.BandRunner(a.rows, a.cols, 12.5, 128000)
    run_chain(a, runner)
    write_bands(runner, os.path.join(out_dir, "warm.tif"), "d8", runner.x)  # warm-up: module load, NCCL peers
    torch.cuda.reset_peak_memory_stats()
    rasters = {}
    for name in pipeline.STAGE_OUTPUTS:
        p = os.path.join(out_dir, f"{name}.tif")
        r = write_bands(runner, p, name, runner.x)
        dist.barrier()
        if rank == 0:
            os.remove(p)
        rasters[name] = r
    me = {"rank": rank, "rows": [runner.bands[0].r0, runner.bands[0].r1], "rasters": rasters,
          "peak_alloc_gb": round(torch.cuda.max_memory_allocated() / 1e9, 2)}
    everyone = [None] * world
    dist.all_gather_object(everyone, me)
    if rank == 0:
        if a.dir is None:
            shutil.rmtree(out_dir, ignore_errors=True)
        emit(a, {"what": "seven chain rasters written from row bands, one per GPU (bands.write_raster over NCCL)",
                 "dem": f"dtb-synth-v1 raw, filled, {a.rows} x {a.cols}", "gpus": world, "meta": "LZW, 256 x 256 tiles, predictor 3 / 2",
                 "total_s": round(sum(max(e["rasters"][n]["total_s"] for e in everyone) for n in pipeline.STAGE_OUTPUTS), 3),
                 "per_rank": everyone, "gpu": gpu_info(), "torch": torch.__version__})
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
