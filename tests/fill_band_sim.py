"""Test-only stand-in for Band's depression-filling calls (dtb_fill_band_f32, include/dtb200.h): the INIT bound and the
SOLVE relaxation restated in NumPy, so that bands.fill_rounds -- halo exchange, rounds, stop test -- runs on CPU with
gloo.  The relaxation here is Jacobi over the whole band, not tiles, so pass and round counts differ from the device;
the fixed point does not."""
import numpy as np
import torch

ND = np.float32(-100)
INF = np.float32(np.inf)


def succ(x):
    """next float32 up, as succ() in csrc/synth.cu (0 and NaN -> the smallest subnormal)"""
    x = np.asarray(x, np.float32)
    u = x.view(np.uint32)
    return np.where(x > 0, u + np.uint32(1), np.where(x < 0, u - np.uint32(1), np.uint32(1))).astype(np.uint32).view(np.float32)


def is_nd(z):
    return (z == ND) | np.isnan(z)


class FillBandSim:
    """rows [r0, r1) of `dem` as one band; buf is the (rows + 2) x cols view the device call works on"""

    def __init__(self, dem, r0, r1, first, last):
        self.rows, self.cols = r1 - r0, dem.shape[1]
        self.first, self.last = first, last
        self.dev = torch.device("cpu")
        self.buf = torch.full((self.rows + 2, self.cols), float("nan"), dtype=torch.float32)
        self.buf[1:self.rows + 1] = torch.from_numpy(np.array(dem[r0:r1]))
        self.ws = None

    @property
    def band(self):
        return self.buf[1:self.rows + 1].numpy()

    def fill_halo_items(self):
        r = self.rows
        return self.buf[1], self.buf[r], self.buf[0], self.buf[r + 1]

    def fill_init(self):
        b = self.buf.numpy()
        R, C = self.rows, self.cols
        z = b[1:R + 1].copy()
        pad = np.full((R + 2, C + 2), np.nan, np.float32)  # outside the raster: never read (those cells are seeds)
        pad[:, 1:-1] = b
        fixed = is_nd(z)
        fixed[:, 0] = fixed[:, -1] = True
        if self.first:
            fixed[0] = True
        if self.last:
            fixed[-1] = True
        for dr in (-1, 0, 1):
            for dc in (-1, 0, 1):
                nb = is_nd(pad[1 + dr:1 + dr + R, 1 + dc:1 + dc + C])
                if dr == -1 and self.first:
                    nb[0] = False
                if dr == 1 and self.last:
                    nb[-1] = False
                fixed |= nb
        w = z.copy()
        if self.first:  # column scan from the raster top
            prev = np.zeros(C, np.float32)
            for r in range(R):
                w[r] = np.where(fixed[r], z[r], np.maximum(z[r], succ(prev)))
                prev = w[r]
        else:
            w[:] = np.where(fixed, z, INF)
        for r in range(R):  # west-to-east row scan
            prev = np.float32(0)
            for c in range(C):
                if not fixed[r, c]:
                    w[r, c] = min(w[r, c], max(z[r, c], succ(prev)))
                prev = w[r, c]
        b[1:R + 1] = w
        self.ws = (z, fixed)

    def fill_solve(self):
        b = self.buf.numpy()
        R, C = self.rows, self.cols
        z, fixed = self.ws
        w = b[1:R + 1]
        first0, last0 = w[0].copy(), w[-1].copy()
        passes = 0
        while True:
            pad = np.full((R + 2, C + 2), INF, np.float32)
            pad[1:-1, 1:-1] = w
            if not self.first:
                pad[0, 1:-1] = b[0]
            if not self.last:
                pad[-1, 1:-1] = b[R + 1]
            m = np.full((R, C), INF, np.float32)
            for dr in (-1, 0, 1):
                for dc in (-1, 0, 1):
                    if dr or dc:
                        m = np.fmin(m, pad[1 + dr:1 + dr + R, 1 + dc:1 + dc + C])
            new = np.where(fixed, w, np.minimum(w, np.maximum(z, succ(m))))
            passes += 1
            if np.array_equal(new, w, equal_nan=True):
                break
            w[:] = new
        seam = not (np.array_equal(first0, w[0], equal_nan=True) and np.array_equal(last0, w[-1], equal_nan=True))
        return passes, int(seam)

    def fill_release(self):
        self.ws = None
