#!/usr/bin/env python
"""bench.py -- DEM Mcells/s for slope -> D8 -> flow accumulation -> HAND -> GFI (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--rows R --cols C] [--dump-outputs DIR]

A "step" is one pass of the whole chain over one synthetic hydrologically conditioned DEM
(recipe dtb-synth-v1, generated and depression-filled on the device before timing).  At N=1 the
workload is BASELINE.json configs[2]: 40 000 x 40 000 f32, full chain, one B200.  At N>1 the same
DEM is sharded into N contiguous row bands (configs[3]; "scaling": "strong").

  value  : cells / time with the DEM already resident in HBM (CUDA events, max over ranks)
  e2e    : same metric through the host API (pinned NumPy DEM in, all seven rasters out),
           host<->device copies inside the timed region
  roofline : dominant stage, algorithmic bytes (SURVEY.md 8d) / CUDA-event time vs measured HBM peak
  cpu_baseline : the oracle port (oracle/dt_oracle.c, OpenMP) on a bounded sample, rank 0, N=1

  verified : device-side identities of the timed result (csrc/verify.cu), summed over ranks

--dump-outputs DIR (1 GPU) writes the seven rasters of the last timed step as DIR/<name>.npy, integer rasters as float64
(exact) and the others as float32: whole when they fit in 60 MiB, else the same seeded sample of cells from every raster.
The DEM depends only on --rows / --cols, so two builds run with the same arguments can be compared output for output.

--impl reference times the reference's own CPU path on the host cores: the unmodified reference installed under
baseline/_ref (pip --target, git-ignored, travels with the snapshot) through its compiled Numba CPU-jit twins
(baseline/ref_bench.py, kind "reference", 1 core: they are serial loops); D8 and flow accumulation, which the
reference does not implement, are timed with the oracle port and reported separately.  If numba or baseline/_ref is
missing the arm falls back to the oracle port over the whole chain (kind "port") and says why.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

PX, RIVER_THR, N_GFI, B_GFI = 12.5, 128000, 0.4, 0.1
# SURVEY.md 8(d), int32 indices.  HAND + GFI are ONE fused pass here: its compulsory traffic is the 25 B of the HAND row
# (d8 1 + acc 4 + dem 4 in, gather dem[idx] 4, idx + fdist + hand 12 out) plus the 4 B GFI raster and the acc[idx] gather
# 4 B = 33 B, not the 41 B of SURVEY's two separate kernels (which re-read hand and idx).
BYTES_PER_CELL = {"slope_d8": 9, "flowacc": 5, "hand_gfi": 33}
CHAIN_BYTES = 55  # the chain figure keeps SURVEY's per-stage sum (9 + 5 + 25 + 16): it is the published roofline target
# algorithmic bytes per cell of the individual kernels (DESIGN.md section 4): what one launch must move
KERNEL_BYTES = {
    "slope_d8_tma_kernel": 9,      # dem 4 R, slope 4 W, d8 1 W
    "fa_tile_kernel": 5,           # d8 1 R, acc 4 W
    "fa_tile_finish_kernel<hand>": 1,  # d8 1 R (+ the acc runs an entry path touches); fused with HAND's entry pass
    "hand_tile_kernel": 33,        # d8 1, acc 4, dem 4 R; gathers dem[idx] 4 + acc[idx] 4; idx, fdist, hand, gfi 16 W
    "hand_tile_kernel<table>": 30, # successor table 2 R instead of d8 + acc (fused chain)
}
# what the dominant kernel cannot avoid moving through DRAM: table 2 + dem 4 in, four rasters 16 out (the dem[idx] / acc[idx]
# gathers are resolved once per tile exit and served by L2)
KERNEL_COMPULSORY_BYTES = {"hand_tile_kernel<table>": 22, "slope_d8_tma_kernel": 9, "fa_tile_kernel": 7}
DUMP_BYTES, DUMP_SEED = 60 << 20, 0  # --dump-outputs: data bytes of all files (< 64 MB), seed of the sampled cells
SAMPLE_ROWS = SAMPLE_COLS = 3072  # bounded CPU sample of the OpenMP port
REF_SAMPLE = 1536                    # bounded sample of the single-threaded reference (about 1 s per step)
GPU_REF_SAMPLE = 4096                # the reference's own Numba-CUDA kernels on the same GPU


def measured_hbm_peak():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """SM clocks / throttle reasons sampled during the timed region (NVML; nvidia-smi as a fallback --
    spawning nvidia-smi every 200 ms perturbs kernel submission, an in-process NVML query does not)."""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.stop = index, [], threading.Event()
        self.t = threading.Thread(target=self._run, daemon=True)
        self.nvml = None
        try:
            import pynvml

            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        sm = n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(self.h, n.NVML_CLOCK_SM)
        r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        flag = lambda name: "Active" if r & getattr(n, name, 0) else "Not Active"
        return [str(sm), str(mx), flag("nvmlClocksThrottleReasonHwSlowdown"), flag("nvmlClocksThrottleReasonHwThermalSlowdown"),
                flag("nvmlClocksThrottleReasonSwThermalSlowdown"), flag("nvmlClocksThrottleReasonSwPowerCap")]

    def _run(self):
        while not self.stop.is_set():
            try:
                if self.nvml is not None:
                    self.rows.append(self._sample_nvml())
                else:
                    out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                         capture_output=True, text=True, timeout=5).stdout.strip()
                    if out:
                        self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.02 if self.nvml is not None else 0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.t.join(timeout=6)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows if len(r) >= 6)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def _subprocess_json(cmd, timeout):
    env = dict(os.environ, OMP_NUM_THREADS=str(os.cpu_count() or 1), NUMBA_NUM_THREADS=str(os.cpu_count() or 1))
    env.pop("NUMBA_ENABLE_CUDASIM", None)
    r = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=timeout)
    if r.returncode != 0:
        raise RuntimeError((r.stderr or r.stdout).strip().splitlines()[-1][:300] if (r.stderr or r.stdout).strip() else f"rc {r.returncode}")
    out = json.loads(r.stdout.strip().splitlines()[-1])
    if "error" in out:
        raise RuntimeError(out["error"])
    return out


def cpu_port(steps, warmup):
    """the oracle port over the chain, timed in a process of its own (oracle/cpu_bench.py: no torch in the process,
    OpenMP team = all host cores even under torchrun, which exports OMP_NUM_THREADS=1)"""
    cmd = [sys.executable, os.path.join(REPO, "oracle", "cpu_bench.py"), str(SAMPLE_ROWS), str(SAMPLE_COLS), str(steps), str(warmup),
           str(PX), str(RIVER_THR), str(N_GFI), str(B_GFI)]
    r = _subprocess_json(cmd, 1800)
    sample = f"{SAMPLE_ROWS}x{SAMPLE_COLS} f32 dtb-synth-v1 DEM per step, river = acc > {RIVER_THR}; oracle/dt_oracle.c with OpenMP"
    return {"value": r["cells"] * len(r["seconds"]) / sum(r["seconds"]) / 1e6, "unit": "Mcells/s", "cores": r["cores"], "kind": "port",
            "sample": sample, "seconds": r["seconds"]}


def cpu_reference(steps, warmup, mode="cpu", n=REF_SAMPLE):
    """the unmodified reference (baseline/_ref) in a process of its own: baseline/ref_bench.py"""
    cmd = [sys.executable, os.path.join(REPO, "baseline", "ref_bench.py"), mode, str(n), str(n), str(steps), str(warmup), str(PX),
           str(RIVER_THR), str(N_GFI), str(B_GFI)]
    r = _subprocess_json(cmd, 3000)
    what = ("slope_sequential_jit + fdist_indexes_sequential_jit + hand_calculator + geomorphic_flood_index_sequential_jit (1 core)"
            if mode == "cpu" else "sloper + flow_hand_index + gfi_calculator: its Numba-CUDA kernels, host arrays in / out per call")
    sample = (f"{n}x{n} f32 dtb-synth-v1 DEM per step, river = acc > {RIVER_THR}; reference {what}; D8 + flow accumulation (absent "
              f"from the reference) by oracle/dt_oracle.c on {r['port_cores']} cores, included")
    out = {"value": r["cells"] * len(r["seconds"]) / sum(r["seconds"]) / 1e6, "unit": "Mcells/s", "cores": r["cores"],
           "kind": "reference", "sample": sample, "seconds": r["seconds"], "stage_seconds": r["stage_seconds"],
           "reference_only_value": r["cells"] * len(r["seconds"]) / sum(r["reference_seconds"]) / 1e6, "numba": r.get("numba")}
    if "device" in r:
        out["device"] = r["device"]
    return out


def cpu_baseline(steps, warmup):
    """reference if it runs on this box, else the port -- and why"""
    try:
        return cpu_reference(steps, warmup)
    except Exception as ex:
        out = cpu_port(steps, warmup)
        out["fallback_reason"] = "reference CPU path unavailable: " + repr(ex)[:200]
        return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_baseline(args.steps, args.warmup)
    secs = r.pop("seconds")
    dt = sum(secs)
    val = r["value"]
    line = {
        "impl": "reference", "metric": "DEM Mcells/s slope->D8->flowacc->HAND->GFI", "value": val, "unit": "Mcells/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(len(secs), 1),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args), "sample": r["sample"]},
        "cpu_baseline": r,
        "e2e": {"value": val, "unit": "Mcells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def _time_launches(run, reps=10, warm=3):
    import torch

    for _ in range(warm):
        run()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        run()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def stencil_config1(peak):
    """BASELINE.json configs[1]: synthetic 10k x 10k f32 DEM, fused slope + D8 only, 1 GPU (inputs + outputs 0.9 GB > L2).
    Headline: the conditioned DEM at the chain's px = 12.5.  Beside it, so that the figure is not a best case: a px whose
    100/px is not a power of two (general cardinal product), the unconditioned DEM (pits), and nodata holes (16 %)."""
    import torch

    from descriptools_b200 import device

    n = 10000
    raw = device.synth_dem(n, n)
    dem = raw.clone()
    device.fill_depressions(dem)
    holes = dem.clone()
    g = torch.Generator(device="cpu").manual_seed(7)
    k = 10
    cy, cx = (torch.rand(k * k, generator=g) * n).long().tolist(), (torch.rand(k * k, generator=g) * n).long().tolist()
    rr = (40 + torch.rand(k * k, generator=g) * 360).long().tolist()
    for y, x, r in zip(cy, cx, rr):
        y0, y1, x0, x1 = max(0, y - r), min(n, y + r + 1), max(0, x - r), min(n, x + r + 1)
        yy = torch.arange(y0, y1, device="cuda").view(-1, 1) - y
        xx = torch.arange(x0, x1, device="cuda").view(1, -1) - x
        holes[y0:y1, x0:x1][(yy * yy + xx * xx) <= r * r] = -100.0
    slope = torch.empty((n, n), dtype=torch.float32, device="cuda")
    d8 = torch.empty((n, n), dtype=torch.uint8, device="cuda")

    def timed(t, px):
        def run():
            device.check(device.lib.dtb_slope_d8(t.data_ptr(), 0, n, n, 0, n, px, slope.data_ptr(), d8.data_ptr(),
                                                 torch.cuda.current_stream().cuda_stream), "dtb_slope_d8")
        ms = _time_launches(run)
        gbs = 9 * n * n / (ms * 1e-3) / 1e9
        return {"ms": ms, "achieved_gbs": gbs, "frac": gbs / peak}

    head = timed(dem, PX)
    out = {"workload": "synthetic 10000x10000 f32 DEM (depression-filled), fused slope + D8 stencil, px = 12.5", "ms": head["ms"],
           "mcells_s": n * n / head["ms"] / 1e3, "bytes_per_cell": 9, "achieved_gbs": head["achieved_gbs"], "frac": head["frac"],
           "variants": {"px_30 (100/px not a power of two)": timed(dem, 30.0), "unconditioned (pits)": timed(raw, PX),
                        "nodata_holes (%.1f %% nodata)" % (100 * float((holes <= -100).float().mean())): timed(holes, PX)}}
    return out


def extra_kernels(peak):
    """the kernels outside the headline chain (SURVEY.md 8d bytes): downslope, TI + MTI, ln(hl/H), calibration counts --
    10k x 10k, CUDA-event time of the call, algorithmic bytes / time against the HBM peak"""
    import torch

    from descriptools_b200 import device, pipeline

    n = 10000
    dem = device.conditioned_dem(n, n)
    res = pipeline.run_device(dem, PX, 2000)
    slope_rad = device.slope_to_radians(res["slope"])
    cells = n * n
    out = {}

    def rec(name, ms, bpc, note):
        gbs = bpc * cells / (ms * 1e-3) / 1e9
        out[name] = {"ms": ms, "bytes_per_cell": bpc, "achieved_gbs": gbs, "frac": gbs / peak, "note": note}

    rec("downslope_kernel", _time_launches(lambda: device.downslope(dem, res["d8"], PX, 5.0), reps=5, warm=2), 9,
        "dem 4 + d8 1 in, f32 out; plus the walks: ~180 moves per cell on this DEM (5 B each, served by L2), issue-bound (~40 instructions per move), see @workload")
    rec("ti_mti_kernel", _time_launches(lambda: device.ti_mti(res["acc"], slope_rad, PX, 0.1), reps=5, warm=2), 16,
        "acc 4 + slope 4 in, TI + MTI out; f64 tan + two short logs")
    rec("lnhlh_kernel", _time_launches(lambda: device.ln_hl_H(res["hand"], res["acc"], N_GFI, B_GFI, PX), reps=5, warm=2), 12,
        "hand 4 + acc 4 in, f32 out; two short logs (ln b + n ln x - ln y)")
    rec("slope_rad_kernel", _time_launches(lambda: device.slope_to_radians(res["slope"]), reps=5, warm=2), 8, "f32 in, f32 out; atanf")
    try:
        from descriptools_b200 import evaluation as ev

        desc = res["hand"]
        bench_map = (res["acc"] > 2000).to(torch.int8)
        ths = torch.linspace(0.0, 30.0, 32, dtype=torch.float64).tolist()
        ctr = ev._Counter(desc, False, -100.0, bench_map, "under")
        rec("eval_counts_kernel", _time_launches(lambda: ctr.counts(ths), reps=5, warm=2), 5,
            "descriptor 4 + benchmark 1 in; 32 thresholds per pass (evaluation.py:32-85 makes one pass per threshold)")
    except Exception as ex:  # the calibration module's device entry is optional here
        out["eval_counts_kernel"] = {"error": repr(ex)[:160]}
    del res, dem, slope_rad
    device.workspace.release()
    torch.cuda.empty_cache()
    return out


def dump_outputs(outs, path):
    """--dump-outputs: the rasters in `outs` as path/<name>.npy (see the module docstring)"""
    import numpy as np
    import torch

    wide = {k: torch.float64 if t.dtype in (torch.int32, torch.int64) else torch.float32 for k, t in outs.items()}
    per_cell = sum(8 if d == torch.float64 else 4 for d in wide.values())
    n = next(iter(outs.values())).numel()
    cells = None
    if n * per_cell > DUMP_BYTES:
        rng = np.random.default_rng(DUMP_SEED)
        cells = torch.from_numpy(np.unique(rng.integers(0, n, DUMP_BYTES // per_cell))).cuda()
    os.makedirs(path, exist_ok=True)
    for k, t in outs.items():
        v = t if cells is None else t.reshape(-1)[cells]
        np.save(os.path.join(path, k + ".npy"), v.to(wide[k]).cpu().numpy())


def workload_name(args):
    cond = "not depression-filled" if getattr(args, "unconditioned", False) else "depression-filled"
    return f"synthetic {args.rows}x{args.cols} f32 DEM (dtb-synth-v1, {cond}), full slope->D8->flowacc->HAND->GFI chain"


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from descriptools_b200 import _lib, device, pipeline

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs is for one GPU")
    torch.cuda.set_device(local)
    from descriptools_b200 import bands as _bands

    numa_cpus = _bands.bind_to_gpu_numa(local)  # before any pinned allocation: host rasters next to this rank's GPU
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rows, cols = args.rows, args.cols
    n_cells = rows * cols

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ev = lambda: torch.cuda.Event(enable_timing=True)
    stage_ms = {k: 0.0 for k in BYTES_PER_CELL}

    if world == 1:
        dem = device.conditioned_dem(rows, cols)
        torch.cuda.synchronize()
        int_dt = torch.int32 if n_cells < 2**31 else torch.int64

        outs = pipeline.alloc_outputs(rows, cols)  # the seven rasters, allocated once and rewritten by every pass

        def step(timed):
            e = [ev() for _ in range(4)]
            e[0].record()
            slope, d8 = device.slope_d8(dem, PX, out=outs)
            e[1].record()
            acc = device.flow_accumulation(d8, dtype=int_dt, fuse_hand_threshold=RIVER_THR, out=outs)
            e[2].record()
            out = device.hand(d8, dem, PX, acc=acc, river_threshold=RIVER_THR, gfi_params=(N_GFI, B_GFI, PX), idx_dtype=int_dt,
                              entry_done=True, out=outs)
            e[3].record()
            return e, None

        runner = None
    else:
        from descriptools_b200 import bands

        # rank 0 generates and depression-fills the WHOLE DEM on its own GPU before anything else is allocated (untimed):
        # at 100 000 x 100 000 that is 40 GB + 50 GB of workspace on one 180 GB B200, 5.5 s (profiles/r2_fill_100k.txt) --
        # the same conditioning as the 1-GPU workload, whatever the number of bands.  --unconditioned keeps the old
        # per-rank synthesis without filling (pits end flow paths early; not the headline workload).
        full = None
        if rank == 0 and not args.unconditioned:
            full = device.conditioned_dem(rows, cols)
            device.workspace.release()
            torch.cuda.empty_cache()
        runner = bands.BandRunner(rows, cols, PX, RIVER_THR, N_GFI, B_GFI)
        band = runner.bands[0]
        if args.unconditioned:
            band.dem.copy_(device.synth_dem(band.rows, cols, band.r0))
        elif rank == 0:
            for i in range(1, world):
                dist.send(full[runner.edges[i]:runner.edges[i + 1]], dst=i)  # row slices are contiguous
            band.dem.copy_(full[runner.edges[0]:runner.edges[1]])
            del full
            torch.cuda.empty_cache()
        else:
            dist.recv(band.dem, src=0)
        torch.cuda.synchronize()

        def step(timed):
            e = [ev() for _ in range(4)]
            runner.step(e, check=False)  # verified once after the timed loop (runner.check_deferred below)
            return e, None

    for _ in range(args.warmup):
        step(False)
    barrier()
    launches0 = _lib.launch_count()
    _lib.profile_enable(True)  # CUDA events around every kernel launch of the timed region (roofline of the top kernel)
    t_start, t_end = ev(), ev()
    with ClockSampler(local) as clk:
        t_start.record()
        events = []
        for _ in range(args.steps):
            e, keep = step(True)
            events.append(e)
        t_end.record()
        barrier()
    launches = _lib.launch_count() - launches0
    if runner is not None:
        runner.check_deferred()  # every boundary solve of the timed steps resolved (else the run is invalid: raises)
    kernel_ms = _lib.profile_collect()
    _lib.profile_enable(False)
    # ---- the timed result itself is checked: device-side identities (csrc/verify.cu), summed over the bands ----
    if world == 1:
        cnt = device.chain_check(outs["d8"], outs["acc"], RIVER_THR, idx=outs["idx"], dem=dem, hand=outs["hand"])
    else:
        o = runner.bands[0].outputs()
        cnt = device.chain_check(o["d8"], o["acc"], RIVER_THR, idx=o["idx"], dem=runner.bands[0].dem, hand=o["hand"],
                                 row0=runner.bands[0].r0, total_rows=rows)
        dist.all_reduce(cnt)
    verdict = device.chain_verdict(cnt.tolist())
    if args.dump_outputs:
        dump_outputs(outs, args.dump_outputs)
    ms = t_start.elapsed_time(t_end)
    for e in events:
        for i, k in enumerate(stage_ms):
            stage_ms[k] += e[i].elapsed_time(e[i + 1])
    if world > 1:
        t = torch.tensor([ms] + [stage_ms[k] for k in stage_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t[0])
        for i, k in enumerate(stage_ms):
            stage_ms[k] = float(t[1 + i])
    ms_step = ms / args.steps
    value = n_cells / (ms_step * 1e-3) / 1e6
    keep = None
    per_rank_kernel_ms = None
    if world > 1:  # load balance across bands: every rank's kernel time per step
        mine = torch.tensor([sum(v[0] for v in kernel_ms.values()) / args.steps], device="cuda", dtype=torch.float64)
        allk = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allk, mine)
        per_rank_kernel_ms = [round(float(t[0]), 3) for t in allk]

    # ---- downslope index at the workload size (not part of the headline chain): one timed call -----------------
    downslope_ms = None
    if world == 1 and not args.no_cpu:
        try:
            device.downslope(dem, outs["d8"], PX, 5.0)
            downslope_ms = _time_launches(lambda: device.downslope(dem, outs["d8"], PX, 5.0), reps=1, warm=0)
        except Exception:
            downslope_ms = None
        torch.cuda.empty_cache()

    # ---- end-to-end through the host API: pinned DEM in, seven rasters out ----------------------
    e2e = None
    if world == 1:
        try:
            dts = pipeline.output_dtypes(np.float32, n_cells)
            dem_host = torch.empty((rows, cols), dtype=torch.float32, pin_memory=True)
            dem_host.copy_(dem)
            pinned = {k: torch.empty((rows, cols), dtype=getattr(torch, np.dtype(v).name), pin_memory=True) for k, v in dts.items()}
            del dem, outs
            device.workspace.release()
            torch.cuda.empty_cache()
            for _ in range(2):  # warm-up (device allocations, workspaces, first touch of the pinned buffers)
                pipeline.pipeline(dem_host, PX, RIVER_THR, N_GFI, B_GFI, pinned_out=pinned, chunks=16)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            k_e2e = max(1, min(args.steps, 3))
            for _ in range(k_e2e):
                pipeline.pipeline(dem_host, PX, RIVER_THR, N_GFI, B_GFI, pinned_out=pinned, chunks=16)
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) / k_e2e
            e2e = {"value": n_cells / dt / 1e6, "unit": "Mcells/s", "h2d_bytes_per_step": n_cells * 4,
                   "d2h_bytes_per_step": int(sum(np.dtype(v).itemsize for v in dts.values())) * n_cells, "steps": k_e2e,
                   "ms_per_step": dt * 1e3}
            del pinned, dem_host
            pipeline.release_buffers()
        except Exception as ex:  # host RAM too small for the pinned staging buffers
            e2e = {"value": None, "unit": "Mcells/s", "error": repr(ex)[:200]}
    elif runner is not None and args.no_e2e:
        e2e = {"value": None, "unit": "Mcells/s", "skipped": "--no-e2e"}
    elif runner is not None:
        # every rank: pinned band DEM in, its seven band rasters out; wall clock between barriers, max over ranks
        try:
            band = runner.bands[0]
            outs = band.outputs()
            dem_host = torch.empty((band.rows, cols), dtype=torch.float32, pin_memory=True)
            dem_host.copy_(band.dem)
            pinned = {k: torch.empty(tuple(t.shape), dtype=t.dtype, pin_memory=True) for k, t in outs.items()}

            def host_step():
                runner.step_host([dem_host], [pinned])  # finished rasters stream back while the next stage computes

            host_step()
            host_step()
            barrier()
            k_e2e = max(1, min(args.steps, 3))
            t0 = time.perf_counter()
            for _ in range(k_e2e):
                host_step()
            barrier()
            dt = torch.tensor([(time.perf_counter() - t0) / k_e2e], device="cuda", dtype=torch.float64)
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            dt = float(dt[0])
            d2h = sum(t.numel() * t.element_size() for t in outs.values())
            tot = torch.tensor([band.rows * cols * 4, d2h], device="cuda", dtype=torch.int64)
            dist.all_reduce(tot)
            e2e = {"value": n_cells / dt / 1e6, "unit": "Mcells/s", "h2d_bytes_per_step": int(tot[0]),
                   "d2h_bytes_per_step": int(tot[1]), "steps": k_e2e, "ms_per_step": dt * 1e3}
            del pinned, dem_host
        except Exception as ex:
            e2e = {"value": None, "unit": "Mcells/s", "error": repr(ex)[:200]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_kind = measured_hbm_peak()
    peak_total = peak * world
    stages = {}
    for k, b in BYTES_PER_CELL.items():
        t_ms = stage_ms[k] / args.steps
        gbs = b * n_cells / (t_ms * 1e-3) / 1e9 if t_ms > 0 else 0.0
        stages[k] = {"ms": t_ms, "bytes_per_cell": b, "achieved_gbs": gbs, "frac": gbs / peak_total}
    # dominant kernel: algorithmic bytes of one launch / its average launch duration (events on its stream)
    cells_launch = n_cells // world  # rank 0's band
    kernels = {}
    for name, (tot_ms, n) in kernel_ms.items():
        avg = tot_ms / max(n, 1)
        b = KERNEL_BYTES.get(name)
        kernels[name] = {"ms_per_step": tot_ms / args.steps, "launches_per_step": n / args.steps, "avg_launch_ms": avg}
        if b is not None and avg > 0:
            kernels[name].update(bytes_per_cell=b, achieved_gbs=b * cells_launch / (avg * 1e-3) / 1e9)
    dom = max(kernels, key=lambda k: kernels[k]["ms_per_step"]) if kernels else None
    traffic = None
    try:  # ncu --set full capture of the same kernel (profiles/): dram bytes read + written per cell
        tr = json.load(open(os.path.join(REPO, "profiles", "traffic.json")))
        traffic = tr[dom]["dram_bytes_per_cell"] * cells_launch
    except Exception:
        pass
    dk = kernels.get(dom, {})
    roofline = {"bound": "hbm", "kernel": dom, "achieved": dk.get("achieved_gbs"), "peak": peak, "unit": "GB/s",
                "frac": (dk.get("achieved_gbs") or 0.0) / peak, "traffic": traffic, "peak_kind": peak_kind + " (burst copy)",
                "bytes_per_launch": (dk.get("bytes_per_cell") or 0) * cells_launch, "avg_launch_ms": dk.get("avg_launch_ms"),
                "chain_frac": CHAIN_BYTES * n_cells / (ms_step * 1e-3) / 1e9 / peak_total, "stages": stages, "kernels": kernels}
    cb = KERNEL_COMPULSORY_BYTES.get(dom)
    if cb is not None and dk.get("avg_launch_ms"):
        # the same kernel against the bytes it cannot avoid moving through DRAM (gathers that L2 serves left out)
        roofline["compulsory"] = {"bytes_per_cell": cb, "achieved_gbs": cb * cells_launch / (dk["avg_launch_ms"] * 1e-3) / 1e9}
        roofline["compulsory"]["frac"] = roofline["compulsory"]["achieved_gbs"] / peak
    if per_rank_kernel_ms is not None:
        roofline["per_rank_kernel_ms"] = per_rank_kernel_ms
    if world == 1 and not args.no_cpu:
        roofline["stencil_10k"] = stencil_config1(peak)
        roofline["extra"] = extra_kernels(peak)
        if downslope_ms:
            roofline["extra"]["downslope_kernel@workload"] = {
                "ms": downslope_ms, "mcells_s": n_cells / downslope_ms / 1e3,
                "note": "delta = 5 m on the 0.02 m/cell tilt of dtb-synth-v1: ~180 D8 moves per cell (measured on the host, "
                        "profiles/r2_downslope_walks.txt), two dependent L2 gathers each -- the walk, not the 9 B/cell of "
                        "compulsory traffic, is the work; SIMT efficiency of one-cell-per-lane is 85 % here"}

    line = {
        "metric": "DEM Mcells/s slope->D8->flowacc->HAND->GFI", "value": value, "unit": "Mcells/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args), "rows": rows, "cols": cols, "px": PX, "river_threshold": RIVER_THR,
                   "parallelism": "1 GPU" if world == 1 else f"{world} row bands", "l2": "inputs larger than L2 (no flush needed)",
                   "host_cores_bound": len(numa_cpus) if numa_cpus else None},
        "clocks": clk.summary(), "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline,
        "verified": verdict["verified"], "verification": verdict,
    }
    if world == 1 and not args.no_cpu:
        r = cpu_baseline(1, 1)
        r.pop("seconds", None)
        line["cpu_baseline"] = r
        if r["kind"] == "reference":  # the OpenMP port beside it (what round 1 reported): a much stronger CPU arm
            try:
                pr = cpu_port(1, 1)
                pr.pop("seconds", None)
                line["cpu_baseline_port"] = pr
            except Exception as ex:
                line["cpu_baseline_port"] = {"error": repr(ex)[:200]}
        try:  # the reference's own Numba-CUDA kernels on this very GPU, through its public entry points
            g = cpu_reference(2, 1, mode="gpu", n=GPU_REF_SAMPLE)
            g.pop("seconds", None)
            g["kind"] = "reference numba-cuda"
            line["gpu_baseline"] = g
        except Exception as ex:
            line["gpu_baseline"] = {"error": repr(ex)[:200]}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=40000)
    ap.add_argument("--cols", type=int, default=40000)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--unconditioned", action="store_true",
                    help="N>1 only: every rank synthesises its band, no depression filling (sizes no single GPU can condition)")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-API leg (pinned staging buffers may exceed host RAM)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the rasters of the last timed step to DIR/<name>.npy (1 GPU)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
