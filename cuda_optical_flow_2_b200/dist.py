"""Multi-GPU host logic for the pyramidal LK path: one process per GPU over torch.distributed.

The reference is single-GPU (SURVEY.md 2.1: no streams, no NCCL, no threads); both modes here are new:

* frame-batch sharding -- pairs are independent, so rank r takes a contiguous block of the batch and
  runs the whole path on its own GPU.  No data-path collective; only timings / statistics are
  gathered at the end.  (`shard_range`, `flow_pairs_sharded`)
* row strips -- one very large pair is cut into horizontal strips.  Strips nest across pyramid
  levels (bounds are fixed on the coarsest level and doubled per finer level), every level needs
  its neighbours' image rows (stencil halo + warp reach) and the next-coarser level's cumulative
  flow rows.  `NativeStrips` runs a whole pair from the library (csrc/strips.cu): the sender's
  kernels store the halo rows straight into the receiver's memory over NVLink, one exchange per
  pyramid level.  The result is bit-identical to the 1-GPU result as long as no warp sample
  reaches past the rows held; the kernel raises a flag otherwise and `NativeStrips.check()` turns
  it into an error instead of returning different numbers.

torch is used for device memory, streams and the process group only; all arithmetic is in the
C-ABI library.  `StripPlan` restates the strip schedule in plain Python: it is unit-tested on CPU
and is the reference the library's schedule is tested against.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Tuple

from ._lib import WARP_BILINEAR


# ------------------------------------------------------------------------------------------ frame batch
def shard_range(n_items: int, world: int, rank: int) -> Tuple[int, int]:
    """Contiguous block [lo, hi) of n_items for `rank`; sizes differ by at most one."""
    if world < 1 or not 0 <= rank < world:
        raise ValueError("bad world/rank")
    base, rem = divmod(n_items, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def flow_pairs_sharded(ctx, prev, next, w: int, levels: int, win: int, warp_mode: int = WARP_BILINEAR,
                       flow_scale: float = 1.0, world: int = 1, rank: int = 0, stream: int = 0):
    """Run this rank's block of a (n, h, pitch) uint8 CUDA batch; returns (lo, hi, flows) with flows the
    residual-flow tensors of the local pairs.  Every rank holds (or is given) only its own block."""
    lo, hi = shard_range(prev.shape[0], world, rank)
    if hi == lo:
        return lo, hi, []
    flows = ctx.flow_pairs_device(prev[lo:hi].contiguous(), next[lo:hi].contiguous(), w, levels, win, warp_mode=warp_mode,
                                  flow_scale=flow_scale, stream=stream)
    return lo, hi, flows


# ------------------------------------------------------------------------------------------ row strips
@dataclass
class LevelStrip:
    """Geometry of one pyramid level on one rank (all rows are GLOBAL row numbers of that level)."""
    w: int
    h: int          # height of the whole level
    y0: int         # rows this rank owns (and produces flow for): [y0, y1)
    y1: int
    by0: int        # rows its image buffers hold: own rows plus halo, clipped to the image: [by0, by1)
    by1: int
    cy0: int        # rows of the NEXT-COARSER level's cumulative flow its buffer holds: [cy0, cy1)
    cy1: int

    @property
    def own_rows(self) -> int:
        return self.y1 - self.y0

    @property
    def buf_rows(self) -> int:
        return self.by1 - self.by0


class StripPlan:
    """Row-strip schedule of a W x H pair over `world` ranks.

    Bounds are set on the coarsest level (floor(r*H_c/world)) and doubled per finer level so that a
    rank's strip at level k sits exactly on top of its strip at level k+1; the last rank also takes
    the rows that odd heights leave over.  `reach` is the largest vertical warp displacement (in
    rows of the level being warped) the halo must absorb.
    """

    def __init__(self, W: int, H: int, levels: int, win: int, world: int, reach: int = 16):
        if world < 1 or levels < 1 or win % 2 == 0:
            raise ValueError("bad strip plan arguments")
        self.W, self.H, self.levels, self.win, self.world, self.reach = W, H, levels, win, world, reach
        self.r = win // 2
        hc = H >> (levels - 1)
        if hc < world:  # as ofb_strips_plan_query: every rank owns at least one row of the coarsest level
            raise ValueError(f"coarsest level has {hc} rows, cannot cut it into {world} strips")
        self.coarse_bounds = [(rk * hc) // world for rk in range(world)] + [hc]
        # image halo: 3x3 stencil + window radius + one row of even-row alignment + warp reach + bilinear tap
        self.img_halo = self.r + 2 + reach + 2
        # coarser cumulative-flow halo: rows (y >> 1) for every image-buffer row that can be warped or composed
        self.cum_halo = (self.r + 2) // 2 + 1

    def level(self, k: int, rank: int) -> LevelStrip:
        sh = self.levels - 1 - k
        w, h = self.W >> k, self.H >> k
        y0 = self.coarse_bounds[rank] << sh
        y1 = h if rank == self.world - 1 else self.coarse_bounds[rank + 1] << sh
        by0, by1 = max(0, y0 - self.img_halo), min(h, y1 + self.img_halo)
        if k < self.levels - 1:
            hc = self.H >> (k + 1)
            # the kernel looks up cum[(y >> 1)] for the rows it warps (its W tile: own rows -r-2 .. +r+1)
            cy0 = max(0, ((y0 - self.r - 2) >> 1))
            cy1 = min(hc, ((y1 + self.r + 1) >> 1) + 1)
        else:
            cy0 = cy1 = 0
        return LevelStrip(w, h, y0, y1, by0, by1, cy0, cy1)

    def halo_messages(self, k: int, rank: int) -> List[Tuple[int, int, int, int]]:
        """Image rows this rank must SEND at level k: list of (peer, first_row, last_row_exclusive, tag).
        A peer needs the part of its buffer [by0, by1) that this rank owns."""
        me = self.level(k, rank)
        out = []
        for peer in range(self.world):
            if peer == rank:
                continue
            pl = self.level(k, peer)
            lo, hi = max(me.y0, pl.by0), min(me.y1, pl.by1)
            if lo < hi:
                out.append((peer, lo, hi, k))
        return out

    def cum_messages(self, k: int, rank: int) -> List[Tuple[int, int, int, int]]:
        """Rows of cum_{k+1} this rank must SEND before level k is solved (it owns them at level k+1)."""
        if k >= self.levels - 1:
            return []
        mine = self.level(k + 1, rank)
        out = []
        for peer in range(self.world):
            if peer == rank:
                continue
            pl = self.level(k, peer)
            lo, hi = max(mine.y0, pl.cy0), min(mine.y1, pl.cy1)
            if lo < hi:
                out.append((peer, lo, hi, 100 + k))
        return out

    def validate(self) -> None:
        for k in range(self.levels):
            covered = 0
            for rk in range(self.world):
                ls = self.level(k, rk)
                if ls.y0 != covered:
                    raise AssertionError(f"level {k}: strips do not tile the image")
                if ls.own_rows < 1:
                    raise AssertionError(f"level {k}: rank {rk} owns no rows")
                covered = ls.y1
            if covered != (self.H >> k):
                raise AssertionError(f"level {k}: strips do not cover the image")


class NativeStrips:
    """The row-strip runner (csrc/strips.cu): the schedule of StripPlan, a whole pair enqueued from C++ on one stream.
    The halo rows move through peer memory: the sender's kernels store them straight into the receiver's memory over
    NVLink and raise epoch flags there.  transport "peer": ranks in separate processes, connected
    over CUDA IPC (`torch.distributed` is used once, to hand round the IPC handles); "local": ranks living in this process
    (connect_local, tests).

    fb_reach (an int >= 0) makes a handle that can also run checked pairs (run_fb: the forward-backward consistency check
    of Context.flow_pairs_fb_device on the strips): a rank's check may sample backward rows up to fb_reach rows beyond its
    own."""

    def __init__(self, ctx, w: int, h: int, levels: int, win: int, world: int, rank: int, device, warp_mode: int = WARP_BILINEAR,
                 flow_scale: float = 1.0, reach: int = 16, transport: str = "peer", fb_reach: Optional[int] = None):
        import ctypes as C

        import torch

        from . import _lib as L

        if transport not in ("peer", "local"):
            raise ValueError(f"strip transport must be 'peer' or 'local', not {transport!r}")
        self.torch, self.C, self.L, self.lib, self.ctx = torch, C, L, L.load(), ctx
        self.w, self.h, self.levels, self.dev, self.world, self.rank = w, h, levels, device, world, rank
        self.flow_scale = flow_scale
        self._transport = transport
        hnd = C.c_void_p()
        self.fb_reach = fb_reach
        if fb_reach is None:
            L.check(self.lib.ofb_strips_create(ctx._h, w, h, levels, win, warp_mode, C.c_float(flow_scale), world, rank, reach,
                                               C.byref(hnd)))
        else:
            L.check(self.lib.ofb_strips_create_fb(ctx._h, w, h, levels, win, warp_mode, C.c_float(flow_scale), world, rank, reach,
                                                  int(fb_reach), C.byref(hnd)))
        self._h = hnd
        if world > 1 and transport == "peer":
            import torch.distributed as dist

            blob = (C.c_ubyte * 128)()
            L.check(self.lib.ofb_strips_peer_handle(self._h, C.cast(blob, C.c_void_p)))
            mine = torch.tensor(list(blob), dtype=torch.uint8, device=device)
            every = torch.empty(world * 128, dtype=torch.uint8, device=device)
            dist.all_gather_into_tensor(every, mine)
            blobs = (C.c_ubyte * (world * 128))(*every.cpu().tolist())
            L.check(self.lib.ofb_strips_peer_connect(self._h, C.cast(blobs, C.c_void_p)))
            dist.barrier()  # nobody pushes before everybody has mapped its neighbours

    def input_rows(self):
        """(prev, next) uint8 torch views (own_rows, pitch) of where the own rows of level 0 live inside the runner:
        fill them in place and pass them to run() to save the upload copy."""
        C = self.C
        pp, pn, pitch = C.c_void_p(), C.c_void_p(), C.c_size_t()
        self.L.check(self.lib.ofb_strips_input(self._h, C.byref(pp), C.byref(pn), C.byref(pitch)))
        y0, y1 = self.own_rows(0)

        def view(ptr):
            class _H:
                __cuda_array_interface__ = {"shape": ((y1 - y0) * pitch.value,), "typestr": "|u1", "data": (ptr, False), "version": 3}

            return self.torch.as_tensor(_H(), device=self.dev).view(y1 - y0, pitch.value)

        return view(pp.value), view(pn.value)

    def set_total(self, on: bool) -> None:
        self.L.check(self.lib.ofb_strips_set_total(self._h, 1 if on else 0))

    def set_fused(self, on: bool) -> None:
        """Peer-memory transport: cumulative-flow halo rows pushed by the level kernels themselves (default) or by
        separate copy / wait kernels."""
        self.L.check(self.lib.ofb_strips_set_fused(self._h, 1 if on else 0))

    def arena(self) -> int:
        p = self.C.c_void_p()
        self.L.check(self.lib.ofb_strips_peer_arena(self._h, self.C.byref(p)))
        return p.value

    @staticmethod
    def connect_local(ranks) -> None:
        """Peer-memory transport between NativeStrips objects of ONE process (ranks[r] is rank r)."""
        import ctypes as C

        arenas = (C.c_void_p * len(ranks))(*[r.arena() for r in ranks])
        for r in ranks:
            r.L.check(r.lib.ofb_strips_peer_connect_local(r._h, arenas))

    def own_rows(self, level: int = 0):
        y0, y1 = self.C.c_int(), self.C.c_int()
        self.L.check(self.lib.ofb_strips_own_rows(self._h, level, self.C.byref(y0), self.C.byref(y1)))
        return y0.value, y1.value

    def run(self, prev_own, next_own, stream: int = 0) -> None:
        """prev_own / next_own: (own_rows, pitch) uint8 CUDA tensors (or row-sliced views) of level 0."""
        self.L.check(self.lib.ofb_strips_run_device(self._h, prev_own.data_ptr(), next_own.data_ptr(), prev_own.stride(0),
                                                    self.C.c_void_p(stream)))

    def run_phase(self, prev_own, next_own, phase: int, stream: int = 0) -> None:
        """One of the 2 * levels phases of a pair (peer-memory transport); see run_local_sequenced."""
        self.L.check(self.lib.ofb_strips_run_phase_device(self._h, prev_own.data_ptr(), next_own.data_ptr(), prev_own.stride(0),
                                                          int(phase), self.C.c_void_p(stream)))

    @staticmethod
    def run_local_sequenced(ranks, inputs, stream: int = 0) -> None:
        """One pair on ranks that live in ONE process and share ONE device (connect_local): phase p of every rank is
        enqueued on `stream` before phase p + 1 of any, so every flag a kernel waits for has been raised by a kernel
        AHEAD of it in the stream.  (Ranks that spin on each other from separate streams of one GPU are not
        guaranteed to be co-scheduled; across GPUs each rank simply calls run().)"""
        for phase in range(2 * ranks[0].levels):
            for ns, (pin, nin) in zip(ranks, inputs):
                ns.run_phase(pin, nin, phase, stream)

    def run_fb(self, prev_own, next_own, alpha: float = 0.01, beta: float = 0.5, want_err2: bool = False, stream: int = 0) -> None:
        """One checked pair (a handle made with fb_reach): both directions on one pyramid build, then the check of the own
        rows; results in own_fb()."""
        self.L.check(self.lib.ofb_strips_run_fb_device(self._h, prev_own.data_ptr(), next_own.data_ptr(), prev_own.stride(0),
                                                       self.C.c_float(alpha), self.C.c_float(beta), 1 if want_err2 else 0,
                                                       self.C.c_void_p(stream)))

    def run_fb_phase(self, prev_own, next_own, phase: int, alpha: float = 0.01, beta: float = 0.5, want_err2: bool = False,
                     stream: int = 0) -> None:
        """One of the 4 * levels + 1 phases of a checked pair; see run_local_sequenced_fb."""
        self.L.check(self.lib.ofb_strips_run_fb_phase_device(self._h, prev_own.data_ptr(), next_own.data_ptr(), prev_own.stride(0),
                                                             self.C.c_float(alpha), self.C.c_float(beta), 1 if want_err2 else 0,
                                                             int(phase), self.C.c_void_p(stream)))

    @staticmethod
    def run_local_sequenced_fb(ranks, inputs, alpha: float = 0.01, beta: float = 0.5, want_err2: bool = False,
                               stream: int = 0) -> None:
        """run_local_sequenced for a checked pair."""
        for phase in range(4 * ranks[0].levels + 1):
            for ns, (pin, nin) in zip(ranks, inputs):
                ns.run_fb_phase(pin, nin, phase, alpha, beta, want_err2, stream)

    def own_fb(self):
        """Torch views (no copy) of the own rows of level 0 after a checked pair: (forward total (rows, w, 2), backward
        total (rows, w, 2), status (rows, w) uint8 FB_* codes, err2 (rows, w); err2 is written only by pairs run with
        want_err2)."""
        C = self.C
        f, b, s, e = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_void_p()
        self.L.check(self.lib.ofb_strips_fb_result(self._h, C.byref(f), C.byref(b), C.byref(s), C.byref(e)))
        y0, y1 = self.own_rows(0)
        rows = y1 - y0

        class _H:
            __cuda_array_interface__ = {"shape": (rows * self.w,), "typestr": "|u1", "data": (s.value, False), "version": 3}

        status = self.torch.as_tensor(_H(), device=self.dev).view(rows, self.w)
        return (_device_view(self.torch, f.value, (rows, self.w, 2), self.dev),
                _device_view(self.torch, b.value, (rows, self.w, 2), self.dev), status,
                _device_view(self.torch, e.value, (rows, self.w), self.dev))

    def check(self, stream: int = 0, allow_unchecked: bool = False) -> None:
        """Synchronises; raises if any pair since the last check went wrong (the flag is sticky), and clears the flag.
        allow_unchecked: accept checked pairs with FB_UNCHECKED pixels (their other outputs are still exact)."""
        v = self.C.c_int()
        self.L.check(self.lib.ofb_strips_check(self._h, self.C.c_void_p(stream), self.C.byref(v)))
        if v.value & 2:
            raise RuntimeError("a neighbour's halo rows did not arrive (peer-memory transport timed out)")
        if v.value & 1:
            raise RuntimeError("a warp sample reached past the exchanged halo rows: raise `reach`")
        if v.value & 4 and not allow_unchecked:
            raise RuntimeError("the check needed backward flow rows beyond those held (FB_UNCHECKED pixels): raise `fb_reach`")

    def own_flow(self, level: int, total: bool = False):
        """A torch view (no copy) of the own rows of the residual (or cumulative) flow of `level`."""
        f, t = self.C.c_void_p(), self.C.c_void_p()
        self.L.check(self.lib.ofb_strips_result(self._h, level, self.C.byref(f), self.C.byref(t)))
        y0, y1 = self.own_rows(level)
        n = (y1 - y0) * (self.w >> level) * 2
        ptr = t.value if total else f.value
        return _device_view(self.torch, ptr, (y1 - y0, self.w >> level, 2), self.dev)

    def close(self) -> None:
        """Collective across the ranks of a multi-process run: nobody frees the memory its neighbours write into before
        everybody has finished (the library additionally waits for the neighbours' last acknowledgements)."""
        if getattr(self, "_h", None):
            if self.world > 1 and self._transport != "local":
                import torch.distributed as dist

                if dist.is_available() and dist.is_initialized():
                    self.torch.cuda.synchronize(self.dev)
                    dist.barrier()
            self.lib.ofb_strips_destroy(self._h)
            self._h = None

    def __del__(self):
        # (no collective from a finaliser: only the library-side bounded wait)
        try:
            if getattr(self, "_h", None):
                self.lib.ofb_strips_destroy(self._h)
                self._h = None
        except Exception:
            pass


def _device_view(torch, ptr: int, shape, device):
    """float32 torch tensor over device memory owned by the library (valid while its owner lives)."""
    n = 1
    for d in shape:
        n *= d

    class _Holder:
        __cuda_array_interface__ = {"shape": (n,), "typestr": "<f4", "data": (ptr, False), "version": 3}

    return torch.as_tensor(_Holder(), device=device).view(*shape)
