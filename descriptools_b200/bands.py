"""bands.py -- the chain sharded into row bands, one band per GPU (SURVEY.md 8e).

The reference scales a raster by a *serial* loop over tiles on one GPU (slope.py:126-147 ships a 1-cell halo
with each tile; flowhand.py:282-402 pre-resolves separator lines and hands them to the tiles as look-up rows).
Here the same decomposition runs in parallel, one process per GPU (torch.distributed / NCCL):

  * slope + D8      : 2 DEM rows exchanged with each neighbour (send/recv); the band computes the codes of its halo row itself;
  * flow accumulation: every band runs its tile pass and node sweep with zero inflow and emits a boundary
                      summary (dtb_flowacc_band, DTB_FA_SUMMARY); the summaries are all-gathered and every rank
                      solves the (small) boundary graph (`solve_flowacc_boundary`) for the inflow carried by its
                      halo rows; a second node sweep + the final tile pass finish the band;
  * HAND / GFI      : same pattern (dtb_hand band modes + `solve_hand_boundary`); paths may cross seams many
                      times, so the solve is real pointer jumping over the boundary nodes.

Band seams sit on multiples of 64 rows (the tile edge of the device kernels).  Results are bit-identical to the
single-GPU run.  The boundary solvers are pure torch (device-agnostic) so the whole driver can be exercised on
CPU with gloo, with the per-band kernels replaced by a stand-in (tests/test_bands_cpu.py); `LocalExchange` runs
k logical bands on ONE GPU through the very same kernels and solvers (tests/test_gpu_parity.py).
"""
from __future__ import annotations

import bisect
import ctypes

import numpy as np
import torch

TILE = 64
KIND_RIVER, KIND_FAIL, KIND_EXIT = 1, 2, 3
CNT_SAT = 32767
FAIL_STATE = -(1 << 63)  # kind 2 in bits 63..62 of an int64


def band_edges(rows: int, nbands: int) -> list[int]:
    """Row ranges [e[i], e[i+1]) of the bands; interior seams on multiples of 64 rows."""
    if nbands < 1:
        raise ValueError("nbands must be >= 1")
    edges = [0]
    for i in range(1, nbands):
        e = int(round(i * rows / nbands / TILE)) * TILE
        edges.append(min(max(e, edges[-1]), rows))
    edges.append(rows)
    if any(b <= a for a, b in zip(edges, edges[1:])):
        raise ValueError(f"{rows} rows cannot be cut into {nbands} bands with seams on multiples of {TILE}")
    return edges


# ---- boundary solvers (rank 0; pure torch, any device) -------------------------------------------
# Whole-array ops only (no data-dependent shapes) and a fixed number of pointer-doubling rounds, so a solve
# enqueues without any host sync.  Each solver also returns a 0-d flag tensor that is non-zero if a chain of
# more than 2**ROUNDS seam crossings (or a cycle across seams) was left unresolved; the driver checks the
# flags once per step and repeats the step with more rounds in that (pathological) case.
ROUNDS = 6


_solver_bufs = {}


def _solver_buffers(solver: str, dev, out_shape: tuple, ws_bytes: int):
    """(workspace, int64 output, int32 unresolved flag) of a library solve, allocated on the first call for (solver, device,
    shape) and reused after: a solve captured in a CUDA graph (_GraphedSolver) replays into the same buffers"""
    key = (solver, dev.index, out_shape)
    if key not in _solver_bufs:
        _solver_bufs[key] = (torch.empty(ws_bytes, dtype=torch.uint8, device=dev), torch.empty(out_shape, dtype=torch.int64, device=dev),
                             torch.zeros(1, dtype=torch.int32, device=dev))
    return _solver_bufs[key]


def forest_accumulate(nxt: torch.Tensor, base: torch.Tensor, rounds: int = ROUNDS):
    """out[i] = base[i] + sum of out[j] over j with nxt[j] == i  (nxt < 0: none).  Returns (out, unresolved flag).
    CUDA tensors: the library's last-arriver sweep (dtb_forest_accumulate); CPU tensors: pointer doubling in torch."""
    if nxt.is_cuda:
        from ._lib import check, lib

        n = nxt.numel()
        nxt, base = nxt.contiguous(), base.contiguous()
        ws, out, flag = _solver_buffers("forest", nxt.device, (n,), lib.dtb_forest_workspace_bytes(n))
        check(lib.dtb_forest_accumulate(nxt.data_ptr(), base.data_ptr(), n, out.data_ptr(), flag.data_ptr(), ws.data_ptr(),
                                        ws.numel(), torch.cuda.current_stream(nxt.device).cuda_stream), "dtb_forest_accumulate")
        return out, flag[0] != 0
    s, a = base.clone(), nxt.clone()
    zero = torch.zeros_like(s)
    for _ in range(rounds):
        live = a >= 0
        tgt = a.clamp(min=0)
        s = s + torch.zeros_like(s).index_add_(0, tgt, torch.where(live, s, zero))
        a = torch.where(live, a[tgt], a)
    return s, (a >= 0).any()


_plan_cache = {}


def _plan(n: int, cols: int, dev):
    """static index tensors of the boundary graph: node (b, side, c) -> (b*2+side)*cols + c"""
    key = (n, cols, str(dev))
    p = _plan_cache.get(key)
    if p is None:
        b = torch.arange(n, device=dev).view(n, 1, 1).expand(n, 2, cols)
        side = torch.arange(2, device=dev).view(1, 2, 1).expand(n, 2, cols)
        c = torch.arange(cols, device=dev).view(1, 1, cols).expand(n, 2, cols)
        b2 = torch.where(side == 0, b - 1, b + 1)           # band on the other side of the seam
        p = dict(c=c.contiguous(), s2=(1 - side).contiguous(), b2ok=((b2 >= 0) & (b2 < n)).contiguous(),
                 b2c=b2.clamp(0, n - 1).contiguous(), node=torch.arange(2 * n * cols, device=dev))
        p["nb"], p["nside"] = p["node"] // (2 * cols), (p["node"] // cols) % 2
        _plan_cache[key] = p
    return p


def solve_flowacc_boundary(summ: torch.Tensor, rounds: int = ROUNDS):
    """summ int64 [N, 6, cols]: exit_above, exit_below, term_above, term_below, d8 first row, d8 last row.
    Returns (inflow int64 [N, 2, cols]: (acc+1) carried by the halo row above / below each band, flag)."""
    n, _, cols = summ.shape
    if summ.is_cuda:  # the library's solve (dtb_flowacc_boundary_solve); the torch form below serves CPU tensors
        from ._lib import check, lib

        summ = summ.contiguous()
        ws, inflow, flag = _solver_buffers("flowacc", summ.device, (n, 2, cols), lib.dtb_flowacc_boundary_workspace_bytes(n, cols))
        check(lib.dtb_flowacc_boundary_solve(summ.data_ptr(), n, cols, inflow.data_ptr(), flag.data_ptr(), ws.data_ptr(), ws.numel(),
                                             torch.cuda.current_stream(summ.device).cuda_stream), "dtb_flowacc_boundary_solve")
        return inflow, flag[0] != 0
    p = _plan(n, cols, summ.device)
    base = summ[:, 0:2, :]
    term = summ[:, 2:4, :]
    code = summ[:, 4:6, :]
    # column shift of the move across the seam: NW/SW -1, N/S 0, NE/SE +1 (flowhand.py:801-824)
    dc = ((code == 128) | (code == 2)).to(torch.int64) - ((code == 32) | (code == 8)).to(torch.int64)
    c2 = p["c"] + dc
    is_exit = (base > 0) & p["b2ok"] & (c2 >= 0) & (c2 < cols)
    t = term[p["b2c"], p["s2"], c2.clamp(0, cols - 1)]          # where the landing cell's in-band path leaves
    nxt = torch.where(is_exit & (t >= 0), (p["b2c"] * 2 + ((t >> 30) & 1)) * cols + (t & 0x3FFFFFFF), torch.full_like(t, -1))
    f, flag = forest_accumulate(nxt.reshape(-1), base.reshape(-1), rounds)
    f = f.view(n, 2, cols)
    inflow = torch.zeros((n, 2, cols), dtype=torch.int64, device=summ.device)
    inflow[1:, 0, :] = f[:-1, 1, :]                             # above band b = last row of band b-1
    inflow[:-1, 1, :] = f[1:, 0, :]                             # below band b = first row of band b+1
    return inflow, flag


def solve_hand_boundary(summ: torch.Tensor, rounds: int = ROUNDS):
    """summ int64 [N, 8, cols]: (state, idx, z-bits, acc) of the first row, then of the last row.
    Returns (int64 [N, 8, cols]: resolved (state, idx, z-bits, acc) of the halo row above, then below; flag)."""
    n, _, cols = summ.shape
    dev = summ.device
    if summ.is_cuda:  # the library's pointer jumping (dtb_hand_boundary_solve); the torch form below serves CPU tensors
        from ._lib import check, lib

        summ = summ.contiguous()
        ws, res, flag = _solver_buffers("hand", dev, (n, 8, cols), lib.dtb_hand_boundary_workspace_bytes(n, cols))
        check(lib.dtb_hand_boundary_solve(summ.data_ptr(), n, cols, int(rounds), res.data_ptr(), flag.data_ptr(), ws.data_ptr(),
                                          ws.numel(), torch.cuda.current_stream(dev).cuda_stream), "dtb_hand_boundary_solve")
        return res, flag[0] != 0
    p = _plan(n, cols, dev)
    st = torch.stack([summ[:, 0, :], summ[:, 4, :]], 1).reshape(-1)          # node (b, side, c)
    pay = torch.stack([summ[:, 1:4, :], summ[:, 5:8, :]], 1)                 # [N, 2, 3, cols]
    pay = pay.permute(0, 1, 3, 2).reshape(-1, 3)
    kind = (st >> 62) & 3
    nd = (st >> 47) & 0x7FFF
    nc = (st >> 32) & 0x7FFF
    ptr = st & 0xFFFFFFFF
    kind = torch.where(st == 0, KIND_FAIL, kind)                             # not an entry: never referenced
    t_side, t_col = (ptr >> 30) & 1, ptr & 0x3FFFFFFF
    b2 = torch.where(t_side == 0, p["nb"] - 1, p["nb"] + 1)
    ok = (kind == KIND_EXIT) & (b2 >= 0) & (b2 < n) & (t_col < cols)
    tgt = torch.where(ok, (b2.clamp(0, n - 1) * 2 + (1 - t_side)) * cols + t_col.clamp(max=cols - 1), -1)
    kind = torch.where((kind == KIND_EXIT) & ~ok, KIND_FAIL, kind)
    src = p["node"]                                                          # whose payload the node ends up with
    for _ in range(rounds):
        live = kind == KIND_EXIT
        t = tgt.clamp(min=0)
        nd = torch.where(live, (nd + nd[t]).clamp(max=CNT_SAT), nd)
        nc = torch.where(live, (nc + nc[t]).clamp(max=CNT_SAT), nc)
        kind, tgt, src = torch.where(live, kind[t], kind), torch.where(live, tgt[t], tgt), torch.where(live, src[t], src)
    flag = (kind == KIND_EXIT).any()
    kind = torch.where(kind == KIND_EXIT, KIND_FAIL, kind)                   # cycle across seams
    state = ((kind << 62) | (nd << 47) | (nc << 32)).view(n, 2, cols)
    pay = pay[src].view(n, 2, cols, 3)
    res = torch.zeros((n, 8, cols), dtype=torch.int64, device=dev)
    res[:, 0, :] = FAIL_STATE
    res[:, 4, :] = FAIL_STATE
    res[1:, 0, :] = state[:-1, 1, :]                                         # above band b = last row of band b-1
    res[1:, 1:4, :] = pay[:-1, 1].permute(0, 2, 1)
    res[:-1, 4, :] = state[1:, 0, :]                                         # below band b = first row of band b+1
    res[:-1, 5:8, :] = pay[1:, 0].permute(0, 2, 1)
    return res, flag


# ---- one band on one device ------------------------------------------------------------------------
class Band:
    """Device buffers and kernel calls of one row band (rows [r0, r1) of a `grows` x `cols` raster)."""

    def __init__(self, index: int, nbands: int, r0: int, r1: int, grows: int, cols: int, px: float, thr: int, n_gfi: float,
                 b_gfi: float, device, force_int64: bool = False):
        from ._lib import lib

        self.lib = lib
        self.index, self.nbands, self.r0, self.r1, self.grows, self.cols = index, nbands, r0, r1, grows, cols
        self.rows = r1 - r0
        self.px, self.thr, self.n_gfi, self.b_gfi = float(px), int(thr), float(n_gfi), float(b_gfi)
        self.dev = device
        self.first, self.last = index == 0, index == nbands - 1
        self.int_dt = torch.int32 if grows * cols < 2**31 and not force_int64 else torch.int64
        rows = self.rows
        f32, u8, i64 = torch.float32, torch.uint8, torch.int64
        mk = lambda shape, dt: torch.empty(shape, dtype=dt, device=device)
        # two halo rows of elevations on each side: the band computes the D8 codes of its one halo row of codes itself
        # (the same inputs give the neighbour's own codes bit for bit), so a step needs ONE exchange, not two
        self.dem_buf = torch.full((rows + 4, cols), float("nan"), dtype=f32, device=device)   # halo rows 0,1 and rows+2,rows+3
        self.d8_buf = torch.zeros((rows + 2, cols), dtype=u8, device=device)                  # halo rows 0 and rows+1
        self.slope_buf = mk((rows + 2, cols), f32)
        self.slope = self.slope_buf[1:rows + 1]
        self.acc = mk((rows, cols), self.int_dt)
        self.fdist, self.hand, self.gfi = mk((rows, cols), f32), mk((rows, cols), f32), mk((rows, cols), f32)
        self.idx = mk((rows, cols), self.int_dt)
        self.ws_fa = mk((lib.dtb_flowacc_workspace_bytes(rows, cols),), u8)
        self.ws_hand = mk((lib.dtb_hand_workspace_bytes(rows, cols),), u8)
        self.fa_exit = torch.zeros((2, cols), dtype=i64, device=device)
        self.fa_term = torch.full((2, cols), -2, dtype=torch.int32, device=device)
        self.fa_inflow = torch.zeros((2, cols), dtype=i64, device=device)
        self.hand_sum = torch.zeros((8, cols), dtype=i64, device=device)
        self.hand_res = torch.zeros((8, cols), dtype=i64, device=device)
        self.ws_fill = None  # depression filling only: allocated by fill_init, freed by fill_release
        self.flood = None    # benchmark flood map rows (int8), load_flood
        self.extra = {}      # ti, mti, lnhlh, <descriptor>_class: allocated on first use (log_indices, calibrate)
        self.slope_rad = None

    # views
    @property
    def dem(self):
        return self.dem_buf[2:self.rows + 2]

    @property
    def d8(self):
        return self.d8_buf[1:self.rows + 1]

    def _stream(self):
        return torch.cuda.current_stream(self.dev).cuda_stream

    def _check(self, code, what):
        from ._lib import check

        check(code, what)

    # stages
    def slope_d8(self, part: str = "all"):
        """rows 1 .. rows+2 of the elevation buffer = the band plus one halo row on each side (whose slope is discarded).
        part="interior": only the rows whose 3-row window lies inside the band (they need no halo: the driver runs them
        while the halo exchange is in flight); part="edges": the two rows at each end, once the halo has arrived."""
        r = self.rows
        spans = {"all": [(1, r + 3)], "interior": [(3, r + 1)], "edges": [(1, 3), (r + 1, r + 3)]}[part]
        for a, b in spans:
            if b <= a:
                continue
            self._check(self.lib.dtb_slope_d8(self.dem_buf.data_ptr(), 0, r + 4, self.cols, a, b, self.px,
                                              self.slope_buf[a - 1:].data_ptr(), self.d8_buf[a - 1:].data_ptr(), self._stream()),
                        "dtb_slope_d8")

    def _fa_args(self, mode):
        from ._lib import DTB_I32, DTB_I64, FlowaccArgs

        a = FlowaccArgs()
        a.d8, a.rows, a.cols = self.d8.data_ptr(), self.rows, self.cols
        a.halo_above = 0 if self.first else self.d8_buf[0].data_ptr()
        a.halo_below = 0 if self.last else self.d8_buf[self.rows + 1].data_ptr()
        a.acc, a.acc_dtype, a.nodata_fill = self.acc.data_ptr(), DTB_I64 if self.int_dt == torch.int64 else DTB_I32, -100
        a.mode = mode
        # the tile passes keep their successor table in the HAND workspace, and the last one also does HAND's
        # entry-node pass (river = acc > threshold) into it
        a.hand_ws, a.hand_ws_bytes, a.hand_river_threshold = self.ws_hand.data_ptr(), self.ws_hand.numel(), self.thr
        return a

    def flowacc_summary(self) -> torch.Tensor:
        """int64 [6, cols]: exit_above, exit_below, term_above, term_below, d8 first row, d8 last row."""
        from ._lib import DTB_FA_SUMMARY

        a = self._fa_args(DTB_FA_SUMMARY)
        if not self.first:
            a.exit_above, a.term_above = self.fa_exit[0].data_ptr(), self.fa_term[0].data_ptr()
        if not self.last:
            a.exit_below, a.term_below = self.fa_exit[1].data_ptr(), self.fa_term[1].data_ptr()
        self._check(self.lib.dtb_flowacc_band(ctypes.byref(a), self.ws_fa.data_ptr(), self.ws_fa.numel(), self._stream()),
                    "dtb_flowacc_band(summary)")
        return torch.cat([self.fa_exit, self.fa_term.to(torch.int64), self.d8[0:1].to(torch.int64),
                          self.d8[self.rows - 1:self.rows].to(torch.int64)], 0)

    def flowacc_finish(self, inflow: torch.Tensor | None):
        """inflow int64 [2, cols] from the boundary solve; None = the band is the whole raster (one call)."""
        from ._lib import DTB_FA_FINISH, DTB_FA_FULL

        if inflow is not None:
            self.fa_inflow.copy_(inflow)
        a = self._fa_args(DTB_FA_FINISH if inflow is not None else DTB_FA_FULL)
        a.inflow_above = 0 if self.first else self.fa_inflow[0].data_ptr()
        a.inflow_below = 0 if self.last else self.fa_inflow[1].data_ptr()
        self._check(self.lib.dtb_flowacc_band(ctypes.byref(a), self.ws_fa.data_ptr(), self.ws_fa.numel(), self._stream()),
                    "dtb_flowacc_band(finish)")

    def _hand_args(self, mode):
        from ._lib import DTB_F32, DTB_I32, DTB_I64, HandArgs, HandBand

        a, b = HandArgs(), HandBand()
        idt = DTB_I64 if self.int_dt == torch.int64 else DTB_I32
        a.fdr, a.acc, a.acc_dtype, a.river_threshold = self.d8.data_ptr(), self.acc.data_ptr(), idt, self.thr
        a.dem, a.dem_dtype, a.rows, a.cols, a.px = self.dem.data_ptr(), DTB_F32, self.rows, self.cols, self.px
        a.idx_dtype = idt
        a.gfi_n, a.gfi_b, a.gfi_size = self.n_gfi, self.b_gfi, self.px
        b.mode, b.row_offset = mode, self.r0
        a.entry_done = 1
        b.above.halo = 0 if self.first else self.d8_buf[0].data_ptr()
        b.below.halo = 0 if self.last else self.d8_buf[self.rows + 1].data_ptr()
        a.band = ctypes.pointer(b)
        return a, b

    def hand_summary(self) -> torch.Tensor:
        """int64 [8, cols]: (state, idx, z-bits, acc) of the first row, then of the last row."""
        from ._lib import DTB_HAND_SUMMARY

        a, b = self._hand_args(DTB_HAND_SUMMARY)
        s = self.hand_sum
        if not self.first:
            b.above.sum_state, b.above.sum_idx, b.above.sum_z, b.above.sum_acc = (s[k].data_ptr() for k in range(4))
        if not self.last:
            b.below.sum_state, b.below.sum_idx, b.below.sum_z, b.below.sum_acc = (s[k].data_ptr() for k in range(4, 8))
        self._check(self.lib.dtb_hand(ctypes.byref(a), self.ws_hand.data_ptr(), self.ws_hand.numel(), self._stream()),
                    "dtb_hand(summary)")
        return s

    def hand_finish(self, res: torch.Tensor | None):
        """res int64 [8, cols] from the boundary solve; None = the band is the whole raster (one call)."""
        from ._lib import DTB_HAND_FINISH, DTB_HAND_FULL

        if res is not None:
            self.hand_res.copy_(res)
        a, b = self._hand_args(DTB_HAND_FINISH if res is not None else DTB_HAND_FULL)
        r = self.hand_res
        if not self.first:
            b.above.res_state, b.above.res_idx, b.above.res_z, b.above.res_acc = (r[k].data_ptr() for k in range(4))
        if not self.last:
            b.below.res_state, b.below.res_idx, b.below.res_z, b.below.res_acc = (r[k].data_ptr() for k in range(4, 8))
        a.fdist, a.idx, a.hand, a.gfi = self.fdist.data_ptr(), self.idx.data_ptr(), self.hand.data_ptr(), self.gfi.data_ptr()
        self._check(self.lib.dtb_hand(ctypes.byref(a), self.ws_hand.data_ptr(), self.ws_hand.numel(), self._stream()),
                    "dtb_hand(finish)")

    def outputs(self) -> dict:
        return dict(slope=self.slope, d8=self.d8, acc=self.acc, fdist=self.fdist, idx=self.idx, hand=self.hand, gfi=self.gfi,
                    **self.extra)

    def _extra(self, name, dtype):
        if name not in self.extra:
            self.extra[name] = torch.empty((self.rows, self.cols), dtype=dtype, device=self.dev)
        return self.extra[name]

    def log_indices(self, n_top: float):
        """TI and MTI (topoindexes.py:109-167, slope in radians as example.py:63-64 makes it) and ln(hl/H) (gfi.py:297-346,
        size = px) of the band's rows: pointwise, no exchange"""
        from ._lib import DTB_I32, DTB_I64

        n = self.rows * self.cols
        idt = DTB_I64 if self.int_dt == torch.int64 else DTB_I32
        if self.slope_rad is None:
            self.slope_rad = torch.empty((self.rows, self.cols), dtype=torch.float32, device=self.dev)
        rad = self.slope_rad
        ti, mti, ln = self._extra("ti", torch.float32), self._extra("mti", torch.float32), self._extra("lnhlh", torch.float32)
        self._check(self.lib.dtb_slope_to_radians(self.slope.data_ptr(), n, rad.data_ptr(), self._stream()), "dtb_slope_to_radians")
        self._check(self.lib.dtb_ti_mti(self.acc.data_ptr(), idt, rad.data_ptr(), n, self.px, float(n_top), ti.data_ptr(), mti.data_ptr(),
                                        self._stream()), "dtb_ti_mti")
        self._check(self.lib.dtb_lnhlh(self.hand.data_ptr(), 0, self.acc.data_ptr(), idt, n, self.n_gfi, self.b_gfi, self.px, ln.data_ptr(),
                                       self._stream()), "dtb_lnhlh")

    # calibration (calibrate_bands)
    def _descriptor(self, name):
        t = self.outputs().get(name)
        if t is None or t.dtype != torch.float32:
            raise ValueError(f"{name!r} is not a float32 raster of the bands (calibrate hand, gfi, ti, mti, lnhlh, ...)")
        if self.flood is None:
            raise RuntimeError("calibration needs the benchmark flood map: load_flood() first")
        return t

    def extrema(self, descriptor: str) -> torch.Tensor:
        """float64 [5]: the band's part of np.unique's two ends (device.eval_extrema)"""
        from . import device

        return device.eval_extrema(self._descriptor(descriptor))

    def corner(self, descriptor: str) -> torch.Tensor:
        """float64 [1]: the band's first cell (band 0: the raster's cell (0, 0), binary_map's nodata)"""
        return self._descriptor(descriptor)[0, :1].to(torch.float64)

    def histogram(self, descriptor, mn, mx, corner, thresholds, under, nodata, hist):
        """add the band's scaled confusion histogram into hist (device.eval_hist)"""
        from . import device

        device.eval_hist(self._descriptor(descriptor), self.flood, mn, mx, corner, thresholds, under, hist, nodata)

    def class_map(self, descriptor, mn, mx, corner, threshold, under, nodata):
        """the band's rows of the class map, kept as `<descriptor>_class` (int8)"""
        from . import device

        d = self._descriptor(descriptor)
        device.eval_class(d, self.flood, mn, mx, corner, threshold, under, nodata, out=self._extra(descriptor + "_class", torch.int8))

    # depression filling (fill_rounds): the (rows + 2) x cols view dem_buf[1:rows+3], one halo row per side
    def fill_halo_items(self):
        """(first row, last row, halo row above, halo row below) for the exchange's halo()"""
        r = self.rows
        return self.dem_buf[2], self.dem_buf[r + 1], self.dem_buf[1], self.dem_buf[r + 2]

    def _fill(self, mode) -> tuple[int, int]:
        passes, seam = ctypes.c_int(0), ctypes.c_int(0)
        self._check(self.lib.dtb_fill_band_f32(self.dem_buf[1].data_ptr(), self.rows, self.cols, 0 if self.first else 1,
                                               0 if self.last else 1, mode, self.ws_fill.data_ptr(), self.ws_fill.numel(),
                                               ctypes.byref(passes), ctypes.byref(seam), self._stream()), "dtb_fill_band_f32")
        return int(passes.value), int(seam.value)

    def fill_init(self):
        """halo rows = the neighbours' DEM rows: seed mask, then an upper bound of the fill written into the band.  The
        workspace (5 bytes per cell: elevations + seed mask) lives until fill_release()."""
        from ._lib import DTB_FILL_INIT

        self.ws_fill = torch.empty(self.lib.dtb_fill_band_workspace_bytes(self.rows, self.cols), dtype=torch.uint8, device=self.dev)
        self._fill(DTB_FILL_INIT)

    def fill_solve(self) -> tuple[int, int]:
        """halo rows = the neighbours' current seam rows: relax the band to its fixed point -> (passes, seam row lowered)"""
        from ._lib import DTB_FILL_SOLVE

        return self._fill(DTB_FILL_SOLVE)

    def fill_release(self):
        self.ws_fill = None


# ---- depression filling over bands -------------------------------------------------------------------
FILL_MAX_ROUNDS = 10000


def fill_rounds(bands, x, max_rounds: int = FILL_MAX_ROUNDS) -> dict:
    """Priority-flood+epsilon filling of the raster held by `bands` (this process's bands; `x` the exchange), bit-identical
    to the single-raster fill (dtb_fill_depressions_f32).

    The fill is the unique fixed point of W(c) = max(z(c), min over the 8 neighbours of succ(W(n))), and relaxing any
    upper bound converges to it, so the bands relax block-Jacobi: every band starts from an upper bound built from its
    own rows (fill_init), then each round exchanges the seam rows and every band relaxes to its own fixed point with its
    halo rows held constant (fill_solve).  A round in which no band lowered a cell of its first or last row leaves every
    band fixed under halos equal to its neighbours' current rows: the whole raster is then the fixed point.

    A band is anything with fill_halo_items / fill_init / fill_solve / fill_release (tests pass NumPy stand-ins).
    Returns {"rounds": n, "passes": [relaxation passes of each local band]}."""
    items = [b.fill_halo_items() for b in bands]
    x.halo(items)  # the DEM rows next to the seams: a cell beside nodata across a seam is a seed
    passes = [0] * len(bands)
    try:
        for b in bands:
            b.fill_init()
        for rnd in range(1, max_rounds + 1):
            x.halo(items)
            moved = 0
            for k, b in enumerate(bands):
                p, s = b.fill_solve()
                passes[k] += p
                moved += s
            if int(x.all_sum(torch.tensor([moved], dtype=torch.int64))[0]) == 0:
                return {"rounds": rnd, "passes": passes}
    finally:
        for b in bands:
            b.fill_release()
    raise RuntimeError(f"depression filling over bands did not converge in {max_rounds} rounds")


# ---- calibration over bands --------------------------------------------------------------------------------
def calibrate_bands(bands, x, descriptor: str = "hand", under: str = "under", nodata: float = -100) -> dict:
    """Calibrate the raster `descriptor` held by `bands` (this process's bands; `x` the exchange) against the benchmark
    flood map the bands hold: the numbers device.calibrate gives on the whole raster, and every band's rows of its class
    map, with no rank holding more than its band.

      1. every band's extrema (two smallest distinct values, largest, NaN seen) are gathered and merged on the host by
         np.unique's rule (evaluation.unique_ends) -> mn, mx; band 0 broadcasts the raw value of cell (0, 0);
      2. per stage of the threshold search (evaluation.search_threshold) every band adds its scaled histogram into one
         buffer, which is summed over the ranks (all_sum) and turned into the stage's counts on the host;
      3. every band writes its rows of the class map at the threshold found.

    A band is anything with extrema / corner / histogram / class_map (tests pass NumPy stand-ins).
    Returns {"threshold", "correctness", "fit", "mn", "mx", "counts": (tn, fp, fn, tp)}."""
    from . import evaluation

    if under not in ("under", "over"):
        raise ValueError("under must be 'under' or 'over'")
    ext = x.gather([b.extrema(descriptor) for b in bands])
    mn, mx = evaluation.unique_ends(ext.cpu().numpy())
    corner = bands[0].corner(descriptor) if bands[0].index == 0 else torch.zeros(1, dtype=torch.float64, device=ext.device)
    x.broadcast(corner, 0)
    corner = float(corner.cpu()[0])
    hist = torch.zeros(4 * 33, dtype=torch.int64, device=ext.device)

    def counts(thresholds):
        hist.zero_()
        for b in bands:
            b.histogram(descriptor, mn, mx, corner, thresholds, under, nodata, hist)
        return evaluation.counts_from_hist(x.all_sum(hist).cpu().numpy(), len(thresholds), under)

    th, c, f, cnt = evaluation.search_threshold(counts)
    for b in bands:
        b.class_map(descriptor, mn, mx, corner, th, under, nodata)
    return dict(threshold=th, correctness=c, fit=f, mn=mn, mx=mx, counts=cnt)


# ---- raster files from bands -------------------------------------------------------------------------
TIFF_HEADER_BYTES = 16   # the writer reserves them for the header; the chunks follow back to back, each padded to even length
WRITE_PIECE_BYTES = 64 << 20


def device_encoder(lay, raster, c0: int, c1: int):
    """write_raster's default encoder: chunks [c0, c1) of `raster` (a device tensor holding rows [lay.row_lo, lay.row_hi)
    of the file) encoded on its device -> (streams back to back, each padded with a zero byte to even length, as a device
    uint8 tensor; their sizes, np.int64)"""
    from . import raster as rio

    parts, sizes = [], []
    cur = torch.cuda.current_stream(raster.device)
    for _, _, blob, s, io in rio.encode_groups(lay, raster, c0, c1):
        with torch.cuda.stream(io):
            part = blob.clone()
        part.record_stream(cur)
        parts.append(part)
        sizes.append(s)
    return torch.cat(parts), np.concatenate(sizes)


def _window(lay, lo: int, hi: int):
    from ._lib import TiffLayout

    w = TiffLayout.from_buffer_copy(lay)
    w.row_lo, w.row_hi = lo, hi
    return w


def write_plan(edges: list[int], chunk_rows: int, rows: int):
    """Who encodes what when row bands [edges[i], edges[i+1]) write a file of `chunk_rows`-row chunk-rows.
    Chunk-row k belongs to the band that holds its first row.  Returns (own, sends):
      own[i] = (k0, k1, straddle): band i encodes chunk-rows [k0, k1) from its own rows, and chunk-row `straddle` (or None),
               which runs past its last row, from a staging buffer its successors fill;
      sends  = [(src band, dst band, first row, end row)]: a band whose first row falls inside a chunk-row sends its rows of
               that chunk-row to the owner (all of them if the band lies inside the chunk-row)."""
    own, sends = [], []
    for i in range(len(edges) - 1):
        r0, r1 = edges[i], edges[i + 1]
        k0, k1 = -(-r0 // chunk_rows), -(-r1 // chunk_rows)
        straddle = k1 - 1 if k0 < k1 and min(k1 * chunk_rows, rows) > r1 else None
        own.append((k0, k1 if straddle is None else k1 - 1, straddle))
        if r0 % chunk_rows:
            k = r0 // chunk_rows
            sends.append((i, bisect.bisect_right(edges, k * chunk_rows) - 1, r0, min(r1, (k + 1) * chunk_rows)))
    return own, sends


def write_raster(bands, x, path, per_band, meta: dict, encoder=None, piece_bytes: int = WRITE_PIECE_BYTES) -> int:
    """Write one raster held as row bands into one GeoTIFF, every band encoding and writing its own chunks: no rank
    ever holds more than its band plus one chunk-row.  The file is byte for byte the one
    raster.write_from_device(encode="device") writes from the whole raster.

    `bands` are this process's bands (anything with index / grows / cols), `x` the exchange, per_band[k] the
    contiguous (rows, cols) tensor of local band k, `meta` as for raster.open(path, "w", ...) (width, height and dtype
    default to the tensors').  `encoder(layout, tensor, c0, c1) -> (packed streams, sizes)` encodes chunks [c0, c1) of a
    row window (layout.row_lo / row_hi); the default is the device kernel (device_encoder), so only stored or LZW
    files with predictor 1-3 can be written.

      1. hand-off: a band whose first row falls inside a chunk-row sends its rows of it to the band that owns it
         (write_plan), which assembles that chunk-row in a staging buffer;
      2. every band encodes the chunks it owns (they stay where the encoder put them);
      3. one collective of the per-chunk sizes: every rank computes every chunk's offset (16 header bytes, then the
         streams in chunk order, each padded to even length);
      4. the rank holding band 0 created the file (main writer, tags) before that collective; the others open part
         writers and write their chunks at their offsets, then a collective of the write status; the main writer
         records the others' chunks and closes (the IFD), and its close status is shared.
    Any failure on any rank raises on every rank and leaves no file.  Returns the bytes of header and chunks."""
    from . import raster as rio

    grows, cols = bands[0].grows, bands[0].cols
    meta = dict(meta)
    meta.setdefault("width", cols)
    meta.setdefault("height", grows)
    meta.setdefault("dtype", str(per_band[0].dtype).replace("torch.", ""))
    if (int(meta["height"]), int(meta["width"])) != (grows, cols):
        raise rio.RasterError(f"{path}: the bands hold a {grows} x {cols} raster, meta describes {meta['height']} x {meta['width']}")
    lay, across, n = rio.layout_of(meta)
    if encoder is None:
        from ._lib import lib as cuda_lib

        if int(cuda_lib.dtb_tiff_encode_bound(ctypes.byref(lay))) == 0:
            raise rio.RasterError("row bands write stored or LZW chunks (predictor 1-3) encoded on the device, not this file")
        encoder = device_encoder
    ch = lay.chunk_rows
    edges = band_edges(grows, x.nbands)
    own, sends = write_plan(edges, ch, grows)
    local = {b.index: t for b, t in zip(bands, per_band)}
    for b, t in zip(bands, per_band):
        if tuple(t.shape) != (edges[b.index + 1] - edges[b.index], cols) or not t.is_contiguous():
            raise rio.RasterError(f"{path}: band {b.index} must be a contiguous tensor of its {edges[b.index + 1] - edges[b.index]} x {cols} rows")

    # 1. the rows of straddling chunk-rows go to their owners
    stage = {}
    for i, (_, _, k) in enumerate(own):
        if k is not None and i in local:
            a = k * ch
            t = local[i]
            stage[i] = torch.empty((min(a + ch, grows) - a, cols), dtype=t.dtype, device=t.device)
            stage[i][:edges[i + 1] - a].copy_(t[a - edges[i]:])
    x.handoff([(src, dst, local[src][a - edges[src]:e - edges[src]] if src in local else None,
                stage[dst][a - a // ch * ch:e - a // ch * ch] if dst in local else None) for src, dst, a, e in sends])

    # 2. encode what this process owns; 3. the sizes of every chunk
    main, err, mine = None, None, []
    try:
        if 0 in local:
            main = rio.DatasetWriter(path, **meta)
        for i in sorted(local):
            k0, k1, k = own[i]
            if k1 > k0:
                mine.append((k0 * across, k1 * across) + tuple(encoder(_window(lay, edges[i], edges[i + 1]), local[i], k0 * across, k1 * across)))
            if k is not None:
                a = k * ch
                mine.append((k * across, (k + 1) * across) + tuple(encoder(_window(lay, a, a + stage[i].shape[0]), stage[i], k * across,
                                                                           (k + 1) * across)))
        stage.clear()
    except Exception as e:  # noqa: BLE001 -- reported to every rank below
        err = e
    vec = torch.zeros(n + 1, dtype=torch.int64)
    vec[0] = 0 if err is None else 1
    for c0, c1, _, s in mine:
        vec[1 + c0:1 + c1] = torch.from_numpy(np.asarray(s, dtype=np.int64))
    vec = x.all_sum(vec)

    def fail(what, e):
        if main is not None:
            main.abort()
        raise rio.RasterError(f"{path}: {what}" + (f" ({e})" if e is not None else "")) from e

    if vec[0] > 0:
        fail(f"encoding failed on {int(vec[0])} rank(s)", err)
    sizes = vec[1:].numpy()
    if (sizes <= 0).any():
        fail("a chunk was encoded by no band", None)
    aligned = (sizes + 1) & ~1
    offsets = TIFF_HEADER_BYTES + np.cumsum(aligned) - aligned
    total = int(TIFF_HEADER_BYTES + aligned.sum())

    # 4. every rank writes its chunks at their offsets
    part = None
    try:
        if mine and main is None:
            part = rio.DatasetWriter(path, part=True, **meta)
        w = main if main is not None else part
        if w is not None:
            got = w.chunk_layout()[0]
            if any(getattr(got, f) != getattr(lay, f) for f in ("rows", "cols", "bps", "predictor", "compression", "tiled", "chunk_rows", "chunk_cols")):
                raise rio.RasterError("the writer settled on another chunk layout")
        for c0, c1, packed, s in mine:
            rio.write_packed(w, c0, packed, s, piece_bytes, offsets=offsets[c0:c1])
        if part is not None:
            part.close()
        err = None
    except Exception as e:  # noqa: BLE001
        err = e
        if part is not None:
            part.abort()
    bad = int(x.all_sum(torch.tensor([0 if err is None else 1], dtype=torch.int64))[0])
    if bad:
        fail(f"writing failed on {bad} rank(s)", err)
    # 5. the main writer records the other ranks' chunks and writes the IFD
    if main is not None:
        try:
            written = np.zeros(n, bool)
            for c0, c1, _, _ in mine:
                written[c0:c1] = True
            edge = np.flatnonzero(np.diff(np.concatenate([[1], written.view(np.int8), [1]])))
            for c0, c1 in zip(edge[::2], edge[1::2]):  # runs of chunks other ranks wrote
                main.place_chunks(int(c0), offsets[c0:c1], sizes[c0:c1])
            main.close()
            err = None
        except Exception as e:  # noqa: BLE001
            err = e
            main.abort()
    bad = int(x.all_sum(torch.tensor([0 if main is None or err is None else 1], dtype=torch.int64))[0])
    if bad:
        main = None
        fail("closing the file failed", err)
    return total


# ---- exchange back-ends ----------------------------------------------------------------------------
class _GraphedSolver:
    """A boundary solver replayed as a CUDA graph: on CUDA tensors a solve is one library call of about ten kernel
    launches and memsets, whose launch overhead (not their run time) every rank would otherwise spend between the two
    collectives."""

    def __init__(self):
        self.cache = {}

    def __call__(self, solver, stacked_in: torch.Tensor, rounds: int):
        """stacked_in int64 [N, k, cols] -> (out, flag); CPU tensors take the eager path."""
        if not stacked_in.is_cuda:
            return solver(stacked_in, rounds)
        key = (solver.__name__, tuple(stacked_in.shape), rounds, stacked_in.device.index)
        ent = self.cache.get(key)
        if ent is None:
            static_in = stacked_in.clone()
            side = torch.cuda.Stream(device=stacked_in.device)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):  # warm-up outside capture (allocator, lazy init)
                    solver(static_in, rounds)
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                out, flag = solver(static_in, rounds)
            ent = self.cache[key] = (graph, static_in, out, flag)
        graph, static_in, out, flag = ent
        static_in.copy_(stacked_in)
        graph.replay()
        return out, flag


class _Exchange:
    """Where the bands live, as the band driver sees it: `nbands`, the indices of the bands this process holds
    (`local_bands`), row exchanges between bands (halo, handoff), small collectives (all_sum, broadcast) and the
    boundary solves.  `flags` collects the unresolved flag of every solve until the driver checks them."""

    def __init__(self, nbands: int, local_bands):
        self.nbands, self.local_bands = nbands, local_bands
        self.flags = []
        self.graphed = _GraphedSolver()

    def solve(self, per_band, solver, rounds=ROUNDS):
        """per_band: the summaries of this process's bands.  Every band's summary is gathered here and this process solves
        the (small) boundary graph itself, keeping its own bands' answers: one collective per solve, and no rank waits
        for rank 0 to prepare and scatter."""
        res, flag = self.graphed(solver, self.gather(per_band), rounds)
        self.flags.append(flag.clone())
        return [res[i].clone() for i in self.local_bands]


class LocalExchange(_Exchange):
    """All bands live in this process (tests; k logical bands on one GPU)."""

    def __init__(self, nbands):
        super().__init__(nbands, range(nbands))

    def halo(self, items):
        """items[i] = (first_row, last_row, halo_above_dst, halo_below_dst) of band i"""
        for i, (_, _, above, below) in enumerate(items):
            if i > 0:
                above.copy_(items[i - 1][1])
            if i + 1 < len(items):
                below.copy_(items[i + 1][0])

    def handoff(self, items):
        """items = [(src band, dst band, rows to send, where they go)]: row blocks between bands (write_raster)"""
        for _, _, send, recv in items:
            recv.copy_(send)

    def all_sum(self, t: torch.Tensor) -> torch.Tensor:
        """one process: the sum is t"""
        return t

    def broadcast(self, t: torch.Tensor, band: int):
        """one process: t already holds band `band`'s rows"""

    def gather(self, per_band):
        """the tensors of every band, stacked in band order"""
        return torch.stack(per_band, 0)


class DistExchange(_Exchange):
    """One band per rank over torch.distributed (NCCL on GPUs, gloo in the CPU tests)."""

    def __init__(self, group=None):
        import torch.distributed as dist

        self.dist, self.group = dist, group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        super().__init__(self.world, [self.rank])
        # NCCL reduces device tensors only: all_sum takes a host tensor through this GPU
        self.dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend(group) == "nccl" else None

    def _peer(self, r: int) -> int:
        """the global rank of rank r of the group: what P2POp and broadcast take"""
        return r if self.group is None else self.dist.get_global_rank(self.group, r)

    def halo(self, items):
        """items = [(first_row, last_row, halo_above_dst, halo_below_dst)] of this rank's band"""
        (first_row, last_row, above, below), = items
        r, blocks = self.rank, []
        if r > 0:
            blocks += [(r, r - 1, first_row, None), (r - 1, r, None, above)]
        if r + 1 < self.world:
            blocks += [(r, r + 1, last_row, None), (r + 1, r, None, below)]
        self.handoff(blocks)

    def handoff(self, items):
        """items = [(src band, dst band, rows to send or None, where they go or None)]: point-to-point row blocks between
        bands; a rank posts the sends of its band and the receives into its buffers, in the order of `items`"""
        d, ops = self.dist, []
        for src, dst, send, recv in items:
            if src == self.rank:
                ops.append(d.P2POp(d.isend, send, self._peer(dst), self.group))
            if dst == self.rank:
                ops.append(d.P2POp(d.irecv, recv, self._peer(src), self.group))
        if ops:
            for w in d.batch_isend_irecv(ops):
                w.wait()

    def all_sum(self, t: torch.Tensor) -> torch.Tensor:
        """t summed over the ranks, on t's device"""
        d = t if self.dev is None else t.to(self.dev)
        self.dist.all_reduce(d, group=self.group)
        return d.to(t.device)

    def broadcast(self, t: torch.Tensor, band: int):
        """t on every rank := t on the rank holding band `band`"""
        self.dist.broadcast(t, src=self._peer(band), group=self.group)

    def gather(self, per_band):
        """the tensors of every band (one per rank, same shape), stacked in band order on every rank"""
        (mine,), d = per_band, self.dist
        mine = mine.contiguous()
        everyone = torch.empty((self.world,) + tuple(mine.shape), dtype=mine.dtype, device=mine.device)
        if mine.is_cuda:
            d.all_gather_into_tensor(everyone.view(-1), mine.view(-1), group=self.group)
        else:  # gloo (the CPU tests)
            d.all_gather(list(everyone.unbind(0)), mine, group=self.group)
        return everyone


def bind_to_gpu_numa(device_index: int) -> list[int] | None:
    """Pin this process to the CPU cores next to its GPU (NVML's affinity mask) BEFORE it allocates pinned host buffers:
    cudaHostAlloc places the pages on the calling thread's NUMA node, and a host raster that sits on the other socket
    crosses the inter-socket link on every H2D / D2H copy.  Returns the cores, or None if NVML / the mask is unavailable."""
    import os

    try:
        import pynvml

        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[device_index]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else device_index
        h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1]
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return allowed
    except Exception:
        return None


# ---- the driver --------------------------------------------------------------------------------------
class BandRunner:
    """Runs the chain over row bands.  `exchange=None` picks torch.distributed (one band per rank)."""

    def __init__(self, rows, cols, px, river_threshold, n_gfi=0.4, b_gfi=0.1, nbands=None, exchange=None, device=None,
                 force_int64=False):
        if exchange is None:
            exchange = DistExchange() if nbands is None else LocalExchange(nbands)
        self.x = exchange
        self.nbands = exchange.nbands
        self.rows, self.cols = rows, cols
        self.edges = band_edges(rows, self.nbands)
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device())
        self.bands = [Band(i, self.nbands, self.edges[i], self.edges[i + 1], rows, cols, px, river_threshold, n_gfi, b_gfi, device,
                           force_int64) for i in exchange.local_bands]
        self.geo = {}  # crs / transform of the DEM load_file read: the defaults of write_raster / write_files

    def load(self, dem_rows: list[torch.Tensor]):
        """dem_rows[k]: the DEM rows of local band k (device or host tensor)"""
        for b, d in zip(self.bands, dem_rows):
            b.dem.copy_(d, non_blocking=True)

    def fill_depressions(self, max_rounds: int = FILL_MAX_ROUNDS) -> dict:
        """Fill the depressions of the loaded DEM in place, band by band (fill_rounds): the result equals
        device.fill_depressions on the whole raster, bit for bit, and no rank holds more than its band (plus a 5 bytes
        per cell workspace for the duration of the call).  Returns {"rounds": n, "passes": [per local band]}."""
        return fill_rounds(self.bands, self.x, max_rounds)

    def load_file(self, path, decode: str = "auto", nodata=None, condition: bool = False):
        """Every local band decodes its own rows of a float32 DEM GeoTIFF straight into its device buffer
        (raster.read_to_device(rows=...): with decode="device" only the band's compressed tiles cross PCIe); the file's
        nodata value (or `nodata`) becomes the path's sentinel -100, as example.py:42-43 does on the host.
        `condition=True` then fills the DEM's depressions over the bands (fill_depressions), for DEMs no GIS has
        conditioned yet."""
        from . import raster

        with raster.open(path) as src:
            if src.shape != (self.rows, self.cols):
                raise ValueError(f"{path}: raster is {src.shape}, the runner was built for {(self.rows, self.cols)}")
            if src.dtypes[0] != "float32":
                raise TypeError(f"{path}: row bands take float32 DEMs, the file holds {src.dtypes[0]}")
            nd = src.nodata if nodata is None else nodata
            self.geo = dict(crs=src.crs, transform=src.transform)
            for b in self.bands:
                from . import device as _device

                raster.read_to_device(src, out=b.dem, rows=(b.r0, b.r1), decode=decode)
                _device.nodata_to_sentinel(b.dem, nd)
        if condition:
            self.fill_depressions()

    def load_flood(self, path):
        """Every local band reads its rows of a benchmark flood map GeoTIFF (uint8 or int8, the DEM's shape) to its device,
        kept as int8 (what example.py:106's .astype("int8") makes of it) for calibrate()."""
        from . import raster

        with raster.open(path) as src:
            if src.shape != (self.rows, self.cols):
                raise ValueError(f"{path}: flood map is {src.shape}, the runner was built for {(self.rows, self.cols)}")
            dt = src.dtypes[0]
            if dt not in ("uint8", "int8"):
                raise TypeError(f"{path}: the flood map must be uint8 or int8, the file holds {dt}")
            for b in self.bands:
                t = torch.empty((b.rows, self.cols), dtype=getattr(torch, dt), device=b.dev)
                raster.read_to_device(src, out=t, rows=(b.r0, b.r1))
                b.flood = t.view(torch.int8)

    def calibrate(self, descriptor: str = "hand", under: str = "under", nodata: float = -100) -> dict:
        """Calibrate a float32 raster of the bands (after step(); "hand" with "under" as example.py:136 does, "gfi" with
        "over", or ti / mti / lnhlh after log_indices()) against the flood map of load_flood (calibrate_bands).  The
        class map becomes the output `<descriptor>_class`.  Returns the threshold, correctness and fit indexes, mn, mx
        and the counts at the threshold, equal to device.calibrate on the whole raster."""
        return calibrate_bands(self.bands, self.x, descriptor, under, nodata)

    def log_indices(self, n_top: float = 0.1):
        """TI and MTI (example.py:63-69) and ln(hl/H) (example.py:91, with the runner's GFI exponent and scale, size = px)
        of every local band after step(): the outputs `ti`, `mti` and `lnhlh`."""
        for b in self.bands:
            b.log_indices(n_top)

    def step(self, events=None, hook=None, check=True):
        """One pass of the chain; `events` (4 CUDA events) are recorded at the stage boundaries and `hook(i)` is
        called after stage i (1 slope+D8, 2 flow accumulation, 3 HAND/GFI) has been enqueued.

        check=True waits for the step and verifies that every boundary solve resolved (repeating the step with more
        pointer-doubling rounds if not).  check=False only enqueues: the caller must call `check_deferred()` before
        trusting the results (a back-to-back loop keeps the GPU busy that way; one host sync per step costs ~5 %
        at 8 GPUs)."""
        if not check:
            self._step(events, ROUNDS, hook)
            return
        rounds = ROUNDS
        while True:
            self.x.flags.clear()
            self._step(events, rounds, hook)
            if not self._unresolved():
                return
            rounds += 6  # a chain of more than 2**rounds seam crossings: repeat the step with more doubling rounds
            if rounds > 32:  # the library's limit (dtb_hand_boundary_solve); 2**32 crossings cannot happen without a cycle
                raise RuntimeError("band boundary graph did not resolve (cycle across band seams)")

    def check_deferred(self):
        """after step(check=False) calls: raise if any boundary solve since the last check was left unresolved"""
        bad = self._unresolved()
        self.x.flags.clear()
        if bad:
            raise RuntimeError("a band boundary solve did not resolve within the default rounds: rerun with step(check=True)")

    def _unresolved(self) -> bool:
        """one host sync per step: did every boundary solve resolve?  (all ranks must agree on repeating)"""
        flags = self.x.flags
        bad = torch.stack([f.to(torch.int32) for f in flags]).sum() if flags else None
        # (with one band per rank every rank has solved the same boundary graphs: the flags agree without a collective)
        return bool(bad.item()) if bad is not None else False

    def step_host(self, dem_host: list, pinned_out: list):
        """Host in / host out: dem_host[k] (pinned) is band k's DEM rows, pinned_out[k] a dict of pinned tensors for its
        seven rasters.  Every finished raster streams back on a copy stream while the next stage computes."""
        main = torch.cuda.current_stream(self.bands[0].dev)
        if not hasattr(self, "_down"):
            self._down = torch.cuda.Stream(device=self.bands[0].dev)
        down = self._down
        for b, h in zip(self.bands, dem_host):
            b.dem.copy_(h, non_blocking=True)
        ready = {1: ("slope", "d8"), 2: ("acc",), 3: ("idx", "fdist", "hand", "gfi")}

        def hook(i):
            ev = torch.cuda.Event()
            ev.record(main)
            down.wait_event(ev)
            with torch.cuda.stream(down):
                for b, pin in zip(self.bands, pinned_out):
                    o = b.outputs()
                    for name in ready[i]:
                        pin[name].copy_(o[name], non_blocking=True)

        self.step(hook=hook)
        down.synchronize()
        main.synchronize()

    def _step(self, events, rounds, hook=None):
        def rec(i):
            if events is not None:
                events[i].record()
            if hook is not None and i > 0:
                hook(i)

        B = self.bands
        rec(0)
        items = [(b.dem_buf[2:4], b.dem_buf[b.rows:b.rows + 2], b.dem_buf[0:2], b.dem_buf[b.rows + 2:b.rows + 4]) for b in B]
        if B[0].dem_buf.is_cuda and min(b.rows for b in B) > 4:
            # the exchange runs on its own stream while the stencil does every row that needs no halo.  It writes only
            # halo rows, which those rows do not read, and reads only DEM rows (its neighbours' ones, for local bands),
            # which the stencil does not write
            main = torch.cuda.current_stream(B[0].dev)
            if not hasattr(self, "_comm"):
                self._comm = torch.cuda.Stream(device=B[0].dev)
            self._comm.wait_stream(main)  # the halo rows may still be read by the previous step's kernels
            with torch.cuda.stream(self._comm):
                self.x.halo(items)
            for b in B:
                b.slope_d8("interior")
            main.wait_stream(self._comm)
            for b in B:
                b.slope_d8("edges")
        else:
            self.x.halo(items)
            for b in B:
                b.slope_d8()
        rec(1)
        if self.nbands == 1:
            B[0].flowacc_finish(None)
        else:
            inflow = self.x.solve([b.flowacc_summary() for b in B], solve_flowacc_boundary, rounds)
            for b, f in zip(B, inflow):
                b.flowacc_finish(f)
        rec(2)
        if self.nbands == 1:
            B[0].hand_finish(None)
        else:
            res = self.x.solve([b.hand_summary() for b in B], solve_hand_boundary, rounds)
            for b, r in zip(B, res):
                b.hand_finish(r)
        rec(3)

    def downslope(self, delta: float, max_moves: int = 0, halo_rows: int = 1024) -> list[torch.Tensor]:
        """Downslope index of every local band (downslope.py:317-376), after step() (it needs the D8 codes).

        A downslope walk is cut by the drop it has reached, not by a band seam, and cannot be pointer-jumped; but it is
        local (hundreds of moves).  The reference's scheme -- tiles, then a global second pass over whatever left its
        tile, flagged -50 (downslope.py:366-374, 526-529) -- becomes: every band walks inside a window of its own rows
        plus `halo_rows` rows of DEM + D8 from each neighbour (one exchange); walks that would leave the window are
        flagged -50 and counted, and as long as any rank counts one the halo is widened (x4) and the flagged bands walk
        again.  No rank holds more than its band plus halo, unless a walk spans a whole neighbouring band: only then
        does the driver fall back to replicating DEM + D8 (5 bytes per cell) on every rank."""
        from ._lib import check, lib

        dev = self.bands[0].dev
        h = max(int(halo_rows), 1)
        while True:
            items, wins = [], []
            for b in self.bands:
                ha = 0 if b.first else min(h, self.edges[b.index] - self.edges[b.index - 1])
                hb = 0 if b.last else min(h, self.edges[b.index + 2] - self.edges[b.index + 1])
                wd = torch.empty((ha + b.rows + hb, self.cols), dtype=torch.float32, device=dev)
                w8 = torch.empty((ha + b.rows + hb, self.cols), dtype=torch.uint8, device=dev)
                wd[ha:ha + b.rows].copy_(b.dem)
                w8[ha:ha + b.rows].copy_(b.d8)
                mine = min(h, b.rows)
                items.append(((b.dem[:mine], b.d8[:mine]), (b.dem[b.rows - mine:], b.d8[b.rows - mine:]),
                              (wd[:ha], w8[:ha]), (wd[ha + b.rows:], w8[ha + b.rows:])))
                wins.append((wd, w8, ha, hb))
            for k in range(2):  # elevations, then codes
                self.x.halo([(it[0][k].contiguous(), it[1][k].contiguous(), it[2][k], it[3][k]) for it in items])
            outs, esc = [], torch.zeros(1, dtype=torch.int64, device=dev)
            complete = True
            for b, (wd, w8, ha, hb) in zip(self.bands, wins):
                out = torch.empty((b.rows, self.cols), dtype=torch.float32, device=dev)
                check(lib.dtb_downslope_window(wd.data_ptr(), 0, w8.data_ptr(), ha + b.rows + hb, self.cols, ha, ha + b.rows, b.px,
                                               float(delta), int(max_moves), out.data_ptr(), 0 if b.first else 1, 0 if b.last else 1,
                                               esc.data_ptr(), b._stream()), "dtb_downslope_window")
                outs.append(out)
                complete &= (b.first or ha == self.edges[b.index] - self.edges[b.index - 1]) and \
                            (b.last or hb == self.edges[b.index + 2] - self.edges[b.index + 1])
            state = self.x.all_sum(torch.stack([esc[0], torch.tensor(0 if complete else 1, dtype=torch.int64, device=dev)]))
            escaped, widenable = (int(v) for v in state.tolist())
            if escaped == 0:
                return outs
            if not widenable:  # every window already holds its whole neighbours: a walk spans more than a band
                return self._downslope_replicated(delta, max_moves)
            h *= 4

    def _downslope_replicated(self, delta: float, max_moves: int = 0) -> list[torch.Tensor]:
        """fallback of downslope(): DEM + D8 of the whole raster on every rank (one broadcast per band), each rank walks
        its own rows over it.  Exact for any walk length."""
        from ._lib import check, lib

        dev = self.bands[0].dev
        full_dem = torch.empty((self.rows, self.cols), dtype=torch.float32, device=dev)
        full_d8 = torch.empty((self.rows, self.cols), dtype=torch.uint8, device=dev)
        mine = {b.index: b for b in self.bands}
        for i in range(self.nbands):
            a, e = self.edges[i], self.edges[i + 1]
            if i in mine:
                full_dem[a:e].copy_(mine[i].dem)
                full_d8[a:e].copy_(mine[i].d8)
            self.x.broadcast(full_dem[a:e], i)
            self.x.broadcast(full_d8[a:e], i)
        outs = []
        for b in self.bands:
            out = torch.empty((b.rows, self.cols), dtype=torch.float32, device=dev)
            check(lib.dtb_downslope_rows(full_dem.data_ptr(), 0, full_d8.data_ptr(), self.rows, self.cols, b.r0, b.r1, b.px,
                                         float(delta), int(max_moves), out.data_ptr(), b._stream()), "dtb_downslope_rows")
            outs.append(out)
        return outs

    def outputs(self) -> list[dict]:
        return [b.outputs() for b in self.bands]

    def write_raster(self, path, per_band: list, **meta) -> int:
        """One GeoTIFF from a raster held as this process's bands (per_band[k]: local band k's rows, e.g. what downslope()
        returns), every rank writing its own chunks (write_raster): byte for byte what raster.write_from_device(
        encode="device") writes from the whole raster.  `meta` as for raster.open(path, "w", ...); crs and transform
        default to the DEM's from load_file.  Every rank calls it; the file system must be shared by all of them."""
        meta = {**self.geo, **meta}
        return write_raster(self.bands, self.x, path, per_band, meta)

    def write_files(self, out_dir, outputs=None, compress: str = "lzw", blocksize: int = 256, **geo) -> dict:
        """The chain's rasters of the last step() as `out_dir/<name>.tif`, with the metadata pipeline.pipeline_files uses
        (pipeline.output_meta) and the DEM's georeferencing from load_file (or `geo`): the files are byte for byte those
        pipeline_files writes on one GPU.  `outputs` defaults to the seven chain rasters; ti, mti, lnhlh (log_indices) and
        <descriptor>_class (calibrate; uint8, nodata 0, as example.py:205-206 writes it) may be listed.  Returns {name: path}."""
        import os

        from .pipeline import STAGE_OUTPUTS, output_meta

        os.makedirs(out_dir, exist_ok=True)
        paths = {}
        outs = self.outputs()
        for name in (STAGE_OUTPUTS if outputs is None else outputs):
            if name not in outs[0]:
                raise ValueError(f"{name!r} is not an output of the bands (log_indices() / calibrate() add ti, mti, lnhlh and *_class)")
            per_band = [o[name].view(torch.uint8) if name.endswith("_class") else o[name] for o in outs]
            paths[name] = os.path.join(out_dir, name + ".tif")
            self.write_raster(paths[name], per_band, **output_meta(name, per_band[0].dtype.is_floating_point, compress, blocksize), **geo)
        return paths
