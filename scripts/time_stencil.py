"""Fused slope + D8 stencil alone (BASELINE configs[1]): CUDA-event time per launch on 10k x 10k DEMs -- conditioned
(depression-filled), unconditioned (pits), and conditioned with nodata holes, all on the TMA kernel; and the conditioned
DEM on the generic kernel three ways: viewed 4 bytes off 16-byte alignment, cropped to an odd width (N - 1 columns), and
rounded to int16 -- plus a bit-exact check of a 2048 x 2048 crop of each, through the same kernel, against the oracle.
Calls dtb_slope_d8 directly, so it times whichever libdtb200 is built.

    python scripts/time_stencil.py [N=10000] [reps=20]
"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import oracle
from descriptools_b200 import device
from descriptools_b200._lib import DTB_F32, DTB_I16

PX = 12.5


def holes(dem):
    """nodata blobs (~8 % of the raster): discs of radius 40..400 cells on a fixed grid of centres"""
    n, m = dem.shape
    out = dem.clone()
    g = torch.Generator(device="cpu").manual_seed(7)
    k = max(4, n // 1000)
    cy = (torch.rand(k * k, generator=g) * n).long()
    cx = (torch.rand(k * k, generator=g) * m).long()
    rr = (40 + torch.rand(k * k, generator=g) * 360).long()
    for y, x, r in zip(cy.tolist(), cx.tolist(), rr.tolist()):
        y0, y1, x0, x1 = max(0, y - r), min(n, y + r + 1), max(0, x - r), min(m, x + r + 1)
        yy = torch.arange(y0, y1, device=dem.device).view(-1, 1) - y
        xx = torch.arange(x0, x1, device=dem.device).view(1, -1) - x
        out[y0:y1, x0:x1][(yy * yy + xx * xx) <= r * r] = -100.0
    return out


def misaligned(t):
    """the same values in a contiguous view that starts 4 bytes into its buffer (not 16-byte aligned)"""
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    v = buf[1:].view(t.shape)
    v.copy_(t)
    return v


def slope_d8(dem, slope, d8):
    rows, cols = dem.shape
    dt = DTB_I16 if dem.dtype == torch.int16 else DTB_F32
    device.check(device.lib.dtb_slope_d8(dem.data_ptr(), dt, rows, cols, 0, rows, PX, slope.data_ptr(), d8.data_ptr(),
                                         torch.cuda.current_stream().cuda_stream), "dtb_slope_d8")


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 10000
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 20
    raw = device.synth_dem(n, n)
    cond = raw.clone()
    device.fill_depressions(cond)
    same = lambda t: t  # noqa: E731
    # name: (DEM, the form it is launched in -- applied to the timed DEM and to its parity crop alike)
    cases = {"conditioned": (cond, same), "unconditioned": (raw, same), "nodata_holes": (holes(cond), same),
             "generic_f32_misaligned": (cond, misaligned),
             "generic_f32_odd_width": (cond, lambda t: t[:, :-1].contiguous()),
             "generic_i16": (cond, lambda t: t.round().to(torch.int16))}
    res = {"n": n}
    for name, (base, form) in cases.items():
        dem = form(base)
        slope = torch.empty(dem.shape, dtype=torch.float32, device="cuda")
        d8 = torch.empty(dem.shape, dtype=torch.uint8, device="cuda")
        for _ in range(3):
            slope_d8(dem, slope, d8)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            slope_d8(dem, slope, d8)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        pits = float(((d8 == 0) & (dem > -100)).float().mean())
        # parity on a crop (own halo: the crop is a raster of its own)
        c = min(n, 2048)
        r0 = (n - c) // 2
        crop = form(base[r0:r0 + c, r0:r0 + c].contiguous())
        s_c = torch.empty(crop.shape, dtype=torch.float32, device="cuda")
        d_c = torch.empty(crop.shape, dtype=torch.uint8, device="cuda")
        slope_d8(crop, s_c, d_c)
        s_ref, d_ref = oracle.slope_d8(crop.cpu().numpy(), PX)
        ok_s = bool(np.array_equal(s_c.cpu().numpy(), s_ref))
        ok_d = bool(np.array_equal(d_c.cpu().numpy(), d_ref))
        nbytes = dem.numel() * (dem.element_size() + 5)  # DEM in, slope (4 B) and D8 (1 B) out
        res[name] = {"ms": round(ms, 4), "gbs": round(nbytes / ms / 1e6, 1), "frac_6560": round(nbytes / ms / 1e6 / 6560, 3),
                     "aligned16": dem.data_ptr() % 16 == 0, "cols": dem.shape[1], "dtype": str(dem.dtype).replace("torch.", ""),
                     "slope_exact": ok_s, "d8_exact": ok_d, "nodata_frac": round(float((dem <= -100).float().mean()), 4),
                     "code0_valid_frac": round(pits, 5)}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
