"""Device-side resampling engine: thin Python object over the C ABI (include/plsb200.h).

PyTorch is used for device memory, streams and (in `dist.py`) torch.distributed only; every number is
produced by the hand-written kernels of libplsb200.so.  There is no CPU path: constructing an Engine
without a CUDA device raises.
"""
import os
import threading

import numpy as np
import torch

from . import _lib
from ._lib import lib, check

F64 = torch.float64
F32 = torch.float32
I32 = torch.int32


def check_choice(name, value, allowed):
    """ValueError unless `value` is one of `allowed` (the values of one option)."""
    if value not in allowed:
        raise ValueError(f"{name} must be one of {allowed}, got {value!r}")


def _require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError(
            "plspy_b200 needs a CUDA device (B200, sm_100a): its resampling path is hand-written CUDA "
            "with no CPU fallback."
        )


class Engine:
    """Holds X (N x p, float64, or float32 with x_storage="fp32") on one GPU together with its Gram matrix and runs the batched kernels.

    Replaces, for one analysis, the per-iteration bodies of `_permutation_test` / `_bootstrap_test`
    (plspy/core/bootstrap_permutation.py:323-452, 537-675).
    """

    PRECISIONS = ("fp64", "tf32x3", "tf32x3+gram")
    X_STORAGES = ("fp64", "fp32")
    SHARDS = ("resamples", "voxels")
    GRAM_TF32_MAX_ROWS = 320

    def __init__(self, X, device=None, precision="fp64", x_storage="fp64", shard="resamples"):
        """precision: "fp64" (exact mode, FP64 DMMA) or "tf32x3" (fast mode: the bootstrap moment GEMM runs on the
        tcgen05 tensor cores with the 3xTF32 split; every N-space quantity -- Gram matrix, permutation p-values,
        Tdistrib, U_hat -- stays FP64) or "tf32x3+gram" (fast mode whose Gram matrix G = X X^T is ALSO formed on the
        tcgen05 tensor cores with the 3xTF32 split: permuted singular values then carry
        a relative error of ~1e-6 instead of being exact, inside the fast mode's tolerance of 1e-5, and a permutation
        p-value can differ by one count where a permuted value ties with the observed one at that level; designs
        beyond 320 rows keep the exact Gram kernel).

        x_storage: "fp64" (default) holds X as float64; "fp32" holds `X.astype(float32)` (a float32 input as it is, a
        float64 one rounded once) and never allocates a float64 copy of X: the task-method kernels widen each element
        where they load it, so every result equals, bit for bit, the "fp64" result for the widened float32 matrix.
        Half the device memory and half the HBM traffic of every pass over X.  The behaviour / multiblock kernels
        (cell_standardize, rb_boot, half_gram, gram_stacked) take float64 operands only.

        shard: the layout of X in a multi-process run.  "resamples" (default): every rank holds the whole of X.
        "voxels" (task methods): every rank is handed the whole host matrix and holds only its columns
        `voxel_range` = dist.voxel_shard(p); `p` is then the width of that slice and `p_total` the width of X.  The
        Gram matrix (`G`) and `xv` become collectives: the partial product of the slice plus one all-reduce, so every
        rank must call them at the same point.  With one process (or inside dist.local_only) the two layouts are the
        same."""
        _require_cuda()
        check_choice("precision", precision, self.PRECISIONS)
        check_choice("x_storage", x_storage, self.X_STORAGES)
        check_choice("shard", shard, self.SHARDS)
        from . import dist
        self.shard = shard
        self._world = dist.world()
        self.voxel_sharded = shard == "voxels" and self._world[1] > 1
        p_total = int(X.shape[1]) if len(X.shape) == 2 else 0
        self.voxel_range = dist.voxel_shard(p_total, *self._world) if self.voxel_sharded else (0, p_total)
        self.p_total = p_total
        self.x_storage = x_storage
        self._xdt = F32 if x_storage == "fp32" else F64
        self.gram_tf32 = precision == "tf32x3+gram"
        self.precision = "tf32x3" if self.gram_tf32 else precision
        self._tf32_ranges = None
        self._ximage = None
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self._pending = None          # [(v0, v1, event)]: voxel ranges of X still being uploaded (see _upload_x)
        self._X = self._upload_x(X)
        if self._X.dim() != 2:
            raise ValueError("X must be 2-dimensional")
        self.N, self.p = int(self._X.shape[0]), int(self._X.shape[1])     # p: the width held here
        self.ldx = int(self._X.stride(0))
        self._G = None
        self._xv_next = None          # the V of a later xv(V) whose product comes out of the Gram launch (prepare_xv)
        self._xv_done = None          # (V, X V) of that launch
        self.kernel_events = None     # set to {} to record CUDA events around named kernels (bench.py)
        self.on_mark = None           # optional callable(name) invoked at every _mark (bench.py: clock sampling)
        self.h2d_bytes = 0 if (torch.is_tensor(X) and X.is_cuda) else self._X.numel() * self._X.element_size()

    def _xp(self, v0=0):
        """Address of column v0 of the device copy of X (float32 or float64 elements)."""
        return self._X.data_ptr() + self._X.element_size() * v0

    def _xfn(self, name, M=None):
        """(function, name) of the entry point `name` reading M (default X), or of its float32 twin when M is float32:
        `_x32` goes before the `_f64` suffix, in place of a trailing `_x`, or at the end."""
        if (self._X if M is None else M).dtype == F32:
            base, f64 = (name[:-4], "_f64") if name.endswith("_f64") else (name.removesuffix("_x"), "")
            name = f"{base}_x32{f64}"
        return getattr(lib, "plsb200_" + name), name

    def _x_stream(self, v0=0, v1=None):
        """The voxel ranges (lo, hi) of X clipped to [v0, v1), each yielded once the current stream waits for its upload."""
        v1 = self.p if v1 is None else v1
        cur = torch.cuda.current_stream(self.device)
        for a, b, ev in self._x_ranges():
            lo, hi = max(a, v0), min(b, v1)
            if lo >= hi:
                continue
            if ev is not None:
                cur.wait_event(ev)
            yield lo, hi

    def _column_blocks(self, K, part):
        """A result of K > KMAX independent columns from `part(k0, k1)`, the result(s) of columns [k0, k1) <= KMAX wide."""
        parts = [part(k0, min(K, k0 + self.KMAX)) for k0 in range(0, K, self.KMAX)]
        if isinstance(parts[0], tuple):
            return tuple(torch.cat(blocks, dim=1) for blocks in zip(*parts))
        return torch.cat(parts, dim=1)

    def _collective(self):
        """The world this voxel-sharded engine was cut for must be the current one: a voxel-sharded engine used inside
        dist.local_only (or in another process group) would silently compute on its slice alone."""
        from . import dist
        if self.voxel_sharded and dist.world() != self._world:
            raise RuntimeError(f"this engine holds the voxels {self.voxel_range} of {self.p_total} for rank "
                               f"{self._world[0]} of {self._world[1]}; it cannot be used outside that process group")
        return dist

    def gather_voxels(self, T):
        """The p_total x ... tensor whose rows [v0, v1) are the voxel rows `T` of every rank (voxel-sharded: ONE
        all-gather, COLLECTIVE); T itself otherwise."""
        if not self.voxel_sharded:
            return T
        dist = self._collective()
        return dist.gather_spans(T, [dist.voxel_shard(self.p_total, r, self._world[1]) for r in range(self._world[1])])

    def _need_whole_x(self, what):
        """The behaviour / multiblock kernels need every voxel of X (shard="voxels" is for mct / cst)."""
        if self.voxel_sharded:
            raise _lib.PlsB200Error(f"{what}: needs the whole of X, this engine holds the voxels {self.voxel_range} "
                                    "(shard='voxels' applies to the task methods mct and cst)")

    @staticmethod
    def _need_f64(M, what):
        """The behaviour / multiblock kernels read float64 operands only (x_storage="fp32" is for mct / cst)."""
        if M is not None and M.dtype != F64:
            raise _lib.PlsB200Error(f"{what}: needs a float64 data matrix, got {M.dtype} (x_storage='fp32' applies to "
                                    "the task methods mct and cst)")

    # ------------------------------------------------------------------ plumbing
    PIPELINED_UPLOAD_MIN_BYTES = 64 << 20
    UPLOAD_FIRST_VOXELS = 148 * 128      # first range of a pipelined upload: one full wave of 128-voxel tiles

    @property
    def X(self):
        """The device copy of X.  If a pipelined upload is still in flight the current stream is made to wait for
        all of it first (kernels that can start on the voxel ranges already uploaded use `_x_ranges` instead)."""
        if self._pending is not None:
            self._start_upload()
            cur = torch.cuda.current_stream(self.device)
            cur.wait_event(self._pending[-1][2])       # the copy stream is in order: the last event covers all
            self._pending = None
        return self._X

    def _x_ranges(self):
        """Voxel ranges of X with the event after which each is on the device ([(0, p, None)] when X is resident)."""
        if self._pending is None:
            return [(0, self.p, None)]
        self._start_upload()
        return list(self._pending)

    @property
    def upload_in_flight(self):
        return self._pending is not None

    def _upload_pipelined(self, Xh):
        """Pinned host X -> device in two voxel ranges (see _start_upload) on a copy stream, one event per range, so that the
        voxel-tiled kernels (Gram partials, TF32 split, bootstrap moment GEMM) can start on the first range while
        the rest is still crossing PCIe.  The copies are only enqueued at the first use of X (`_start_upload`):
        host->device copies execute in issue order, so the small uploads of an analysis (index matrices, V, weights)
        must be issued before the 480 MB of X or they would wait behind it -- and with them the first kernels."""
        v0, v1 = self.voxel_range   # (the columns this rank holds: all of them unless voxel-sharded)
        self._x_host = Xh            # keep the pinned source alive until the copies have been consumed
        self._pending = []           # empty list = upload not started yet
        return torch.empty((int(Xh.shape[0]), v1 - v0), dtype=Xh.dtype, device=self.device)

    def _start_upload(self):
        if self._pending is None or len(self._pending) > 0:
            return
        Xh, Xd = self._x_host, self._X
        n, p = int(Xd.shape[0]), int(Xd.shape[1])
        c0, ph = self.voxel_range[0], int(Xh.shape[1])       # first column held here, host row length
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(device=self.device)
        side = self._copy_stream
        side.wait_stream(torch.cuda.current_stream(self.device))
        # Exact mode -- two voxel ranges: a first one of one full wave of the FP64 moment GEMM (148 SMs x 128 voxels = whole
        # waves of its 64-voxel tiles), whose GEMM (~20 ms) starts after ~1 ms of upload and covers the transfer of the
        # rest; four equal ranges made four launches of 15.84 waves each, 0.65 waves = 2.2 ms of tail per analysis
        # (e2e 222.0 -> 220.3 ms).  Fast mode -- four equal ranges: its GEMM takes 2.5 ms per tenth of X against 0.9 ms
        # of upload, so a small first range would leave the GPU idle for most of the second range's transfer
        # (measured: e2e 34.1 -> 36.8 ms with the two ranges of the exact mode).
        if self.precision == "fp64":
            first = self.UPLOAD_FIRST_VOXELS if p >= 4 * self.UPLOAD_FIRST_VOXELS else -(-(p // 2) // 256) * 256
            bounds = [0, first, p] if 0 < first < p else [0, p]
        else:
            step = -(-(-(-p // 4)) // 256) * 256          # whole pairs of 128-voxel tiles
            bounds = list(range(0, p, step)) + [p]
        pend = []
        es = Xd.element_size()
        with torch.cuda.device(self.device):
            for v0, v1 in zip(bounds[:-1], bounds[1:]):
                # (torch's copy_ of a column block goes through a contiguous temporary and synchronises)
                check(lib.plsb200_copy2d_h2d(Xd.data_ptr() + es * v0, es * p, Xh.data_ptr() + es * (c0 + v0), es * ph,
                                             es * (v1 - v0), n, side.cuda_stream), "copy2d_h2d")
                ev = torch.cuda.Event()
                ev.record(side)
                pend.append((v0, v1, ev))
        Xd.record_stream(side)
        self._pending = pend

    def _upload_x(self, X):
        """X -> device.  In a multi-process run X is replicated (every rank is handed the same host matrix), so
        each rank uploads only its 1/world share of the rows over PCIe and the ranks exchange the shares with one
        all-gather over NVLink: eight ranks pulling the same 480 MB through the host's memory system at the same
        time took 17 ms each, a share plus the all-gather takes 2.  Voxel-sharded, each rank uploads only its columns
        (`voxel_range`) by the same paths and nothing is gathered."""
        from . import dist
        size = dist.world()[1]
        dt = self._xdt
        cols = self.voxel_sharded and len(X.shape) == 2
        v0, v1 = self.voxel_range
        if dt == F64 and torch.is_tensor(X) and X.dtype == torch.float32 and X.dim() == 2:
            # float32 storage (plspy_b200/io.py): half the bytes over PCIe, widened on the device
            x32 = (X[:, v0:v1] if cols else X).to(self.device, non_blocking=True).contiguous()
            out = torch.empty(x32.shape, dtype=F64, device=self.device)
            with torch.cuda.device(self.device):
                check(lib.plsb200_widen_f32_f64(x32.data_ptr(), out.data_ptr(), x32.numel(), self._stream()),
                      "widen_f32_f64")
            return out
        on_host = not (torch.is_tensor(X) and X.is_cuda)
        whole = size == 1 or cols                     # this rank uploads everything it holds over PCIe itself
        if (whole and on_host and torch.is_tensor(X) and X.dim() == 2 and X.dtype == dt and X.is_pinned()
                and X.is_contiguous() and X.shape[0] * (v1 - v0) * X.element_size() >= self.PIPELINED_UPLOAD_MIN_BYTES):
            return self._upload_pipelined(X)
        if (whole and on_host and len(X.shape) == 2 and not torch.is_tensor(X)
                and X.dtype == (np.float64 if dt == F64 else np.float32) and X.flags.c_contiguous
                and X.shape[0] * (v1 - v0) * X.itemsize >= self.PIPELINED_UPLOAD_MIN_BYTES
                and self.PAGEABLE_UPLOAD_THREADS > 1):
            return self._upload_pageable(X)
        if cols:
            return self.to_device(X[:, v0:v1], dt)
        if size == 1 or not on_host or len(X.shape) != 2:
            return self.to_device(X, dt)
        n = int(X.shape[0])
        lo, hi = dist.shard(n)
        part = self.to_device(X[lo:hi], dt)
        if part.shape[0] == 0:
            part = torch.zeros((0, int(X.shape[1])), dtype=dt, device=self.device)
        return dist.gather_rows(part, n, lo).contiguous()

    PAGEABLE_UPLOAD_THREADS = int(os.environ.get("PLSB200_UPLOAD_THREADS", str(max(1, min(8, (os.cpu_count() or 2) // 2)))))
    STAGING_BLOCK_BYTES = 32 << 20
    _staging = {}                    # pinned staging buffers, shared by the engines of a process
    _staging_lock = threading.Lock()

    def _upload_pageable(self, X):
        """A large PAGEABLE host matrix (what `PLS(X numpy, ...)` hands over).  The driver stages a pageable
        host->device copy through its own pinned buffer on one host thread: 43 ms = 11 GB/s for the 480 MB of the bench
        design, more than the whole fast-mode GEMM, and calling it from several threads or streams changes nothing (the
        copies serialise: measured 43 ms with 1, 2, 4 and 8 threads).  Here the staging is done by this library: row
        blocks are copied into two pinned buffers by a few threads (numpy's copy loop releases the GIL) and leave them
        by asynchronous DMA, so the host copy of block i+1 overlaps the transfer of block i: 16 ms with 4 threads, 14 ms
        with 8 (tools/time_upload.py)."""
        with Engine._staging_lock:
            return self._upload_pageable_locked(X)

    def _upload_pageable_locked(self, X):
        import concurrent.futures
        v0, v1 = self.voxel_range
        n, p = int(X.shape[0]), v1 - v0
        dt = self._xdt
        out = torch.empty((n, p), dtype=dt, device=self.device)
        nt = max(1, self.PAGEABLE_UPLOAD_THREADS)
        rows = max(1, self.STAGING_BLOCK_BYTES // (X.itemsize * p))
        bufs = Engine._staging.get(dt)
        if bufs is None or bufs[0].numel() < rows * p:            # one pair per process and dtype, grown when a row is longer
            bufs = Engine._staging[dt] = [torch.empty(rows * p, dtype=dt).pin_memory() for _ in range(2)]
        side = getattr(self, "_copy_stream", None)
        if side is None:
            side = self._copy_stream = torch.cuda.Stream(device=self.device)
        cur = torch.cuda.current_stream(self.device)
        side.wait_stream(cur)
        free = [None, None]                                       # event after which a staging buffer may be refilled
        with concurrent.futures.ThreadPoolExecutor(nt) as pool:
            for b, r0 in enumerate(range(0, n, rows)):
                r1 = min(n, r0 + rows)
                buf = bufs[b % 2][:(r1 - r0) * p].view(r1 - r0, p)
                if free[b % 2] is not None:
                    free[b % 2].synchronize()
                dst = buf.numpy()
                cuts = [r0 + (r1 - r0) * i // nt for i in range(nt + 1)]
                list(pool.map(lambda i: np.copyto(dst[cuts[i] - r0:cuts[i + 1] - r0], X[cuts[i]:cuts[i + 1], v0:v1]),
                              range(nt)))
                with torch.cuda.stream(side):
                    out[r0:r1].copy_(buf, non_blocking=True)
                    free[b % 2] = torch.cuda.Event()
                    free[b % 2].record(side)
        for ev in free:                      # the staging buffers are shared: drained before anybody refills them
            if ev is not None:
                ev.synchronize()
        cur.wait_stream(side)
        out.record_stream(side)
        return out

    def to_device(self, a, dtype):
        if torch.is_tensor(a):
            t = a
        else:
            t = torch.from_numpy(np.ascontiguousarray(a))
        if t.dtype != dtype:
            t = t.to(dtype)
        if not t.is_cuda:
            t = t.to(self.device, non_blocking=True)
        elif t.device != self.device:
            t = t.to(self.device)
        return t.contiguous()

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def to_host_async(self, *tensors, side=False):
        """Enqueue device -> host copies into pinned staging buffers (torch's caching host allocator) and return
        a function that waits for them (one event synchronisation) and hands back numpy arrays; None passes
        through.  Lets the caller keep enqueuing GPU work before it blocks.  `side=True` issues the copies on a
        second stream (after everything enqueued so far), so that they overlap the kernels enqueued next."""
        cur = torch.cuda.current_stream(self.device)
        stream = cur
        if side:
            if getattr(self, "_copy_stream", None) is None:
                self._copy_stream = torch.cuda.Stream(device=self.device)
            stream = self._copy_stream
            stream.wait_stream(cur)
        staged = []
        with torch.cuda.stream(stream):
            for t in tensors:
                if t is None:
                    staged.append(None)
                    continue
                h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
                h.copy_(t, non_blocking=True)
                if side:
                    t.record_stream(stream)
                staged.append(h)
        done = torch.cuda.Event()
        done.record(stream)

        def wait():
            done.synchronize()
            out = [None if h is None else h.numpy() for h in staged]
            return out[0] if len(out) == 1 else out
        return wait

    def to_host(self, *tensors):
        """Device -> host through pinned staging buffers, one synchronisation for the whole batch."""
        return self.to_host_async(*tensors)()

    def _empty(self, *shape, dtype=F64):
        return torch.empty(*shape, dtype=dtype, device=self.device)

    def _ws(self, nbytes):
        return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=self.device)

    @staticmethod
    def _p(t):
        return t.data_ptr() if t is not None else None

    def _mark(self, name):
        """CUDA event on the launching stream, kept only when kernel_events is enabled."""
        if self.kernel_events is None:
            return
        if self.on_mark is not None:
            self.on_mark(name)
        ev = torch.cuda.Event(enable_timing=True)
        ev.record(torch.cuda.current_stream(self.device))
        self.kernel_events.setdefault(name, []).append(ev)

    def kernel_ms(self, name):
        """Durations (ms) of the launches bracketed by _mark(name) pairs; call after a synchronize."""
        ev = (self.kernel_events or {}).get(name, [])
        return [ev[i].elapsed_time(ev[i + 1]) for i in range(0, len(ev) - 1, 2)]

    # ------------------------------------------------------------------ kernels
    def gram_of(self, M):
        """K1: M M^T for a device matrix M (rows x p)."""
        n, p, ld = int(M.shape[0]), int(M.shape[1]), int(M.stride(0))
        fn, what = self._xfn("gram_f64", M)
        with torch.cuda.device(self.device):
            ws = self._ws(lib.plsb200_gram_f64_workspace(n, p))
            G = self._empty(n, n)
            check(fn(self._p(M), n, p, ld, self._p(G), self._p(ws), ws.numel(), self._stream()), what)
        return G

    def gram_stacked(self, M1, M2):
        """Gram matrix of the row stack [M1; M2] ((n1 + n2) x p) without building it (multiblock: [X; Zb])."""
        n1, n2, p = int(M1.shape[0]), int(M2.shape[0]), int(M1.shape[1])
        assert int(M2.shape[1]) == p
        self._need_f64(M1, "gram_stacked"); self._need_f64(M2, "gram_stacked"); self._need_whole_x("gram_stacked")
        with torch.cuda.device(self.device):
            ws = self._ws(lib.plsb200_gram_f64_workspace(n1 + n2, p))
            G = self._empty(n1 + n2, n1 + n2)
            check(lib.plsb200_gram_stacked_f64(self._p(M1), n1, int(M1.stride(0)), self._p(M2), n2, int(M2.stride(0)), p,
                                               self._p(G), self._p(ws), ws.numel(), self._stream()), "gram_stacked_f64")
        return G

    @property
    def G(self):
        """G = X X^T (N x N), computed once per engine.  Voxel-sharded: the Gram matrix of this rank's columns plus one
        all-reduce of N x N doubles (COLLECTIVE at its first use)."""
        if self._G is None:
            if self.p == 0:
                self._G = torch.zeros(self.N, self.N, dtype=F64, device=self.device)
            elif self.gram_tf32 and self.N <= self.GRAM_TF32_MAX_ROWS:
                self._G = self._gram_tf32()
            elif self._xv_next is not None:
                self._G = self._gram_xv()
            elif self._pending is None:
                self._G = self.gram_of(self.X)
            else:       # partial Gram matrices of the voxel ranges as they arrive, summed in a fixed order
                G = None
                for v0, v1 in self._x_stream():
                    Gc = self.gram_of(self._X[:, v0:v1])
                    G = Gc if G is None else G.add_(Gc)
                self._G = G
            if self.voxel_sharded:
                self._collective().allreduce_sum_(self._G)
        return self._G

    def _gram_tf32(self, v0=0, v1=None):
        """K1 fast mode: G of the voxels [v0, v1) on the tcgen05 tensor cores, voxel range by voxel range as X arrives
        (TF32 split of a range into the Gram kernel's operand image, then its partial Gram, accumulated in a fixed
        order)."""
        G = self._empty(self.N, self.N)
        split, what = self._xfn("gram_tf32_split")
        with torch.cuda.device(self.device):
            for i, (v0, v1) in enumerate(self._x_stream(v0, v1)):
                pc = v1 - v0
                img = self._ws(lib.plsb200_gram_tf32_image_bytes(self.N, pc))
                nb = lib.plsb200_gram_tf32_workspace(self.N, pc)
                ws = self._ws(nb)
                self._mark("gram_tf32")
                check(split(self._xp(v0), self.N, pc, self.ldx, self._p(img), self._stream()), what)
                check(lib.plsb200_gram_tf32(self._p(img), self.N, pc, self._p(G), 1 if i else 0, self._p(ws), nb,
                                            self._stream()), "gram_tf32")
                self._mark("gram_tf32")
        return G

    def gram_collective(self):
        """COLLECTIVE in a multi-process run (every rank must call it at the same point): G from the partial Gram
        matrix of this rank's voxel range plus one all-reduce of N x N doubles, instead of every rank forming the whole
        G redundantly -- the Gram is the largest piece of per-rank work that does not shrink with the shard of
        resamples.  Single process, G already there, a voxel-sharded engine (whose G is collective anyway) or
        PLSB200_SHARD_GRAM=0: the plain property."""
        from . import dist
        rank, size = dist.world()
        if (self._G is None and size > 1 and not self.voxel_sharded and self.p >= 4096 * size
                and os.environ.get("PLSB200_SHARD_GRAM", "1") != "0"):
            cut = [(self.p * r // size) // 64 * 64 for r in range(size)] + [self.p]
            if self.gram_tf32 and self.N <= self.GRAM_TF32_MAX_ROWS:
                self.X                                      # (the whole of X is on the device from here on)
                G = self._gram_tf32(cut[rank], cut[rank + 1])
            else:
                G = self.gram_of(self.X[:, cut[rank]:cut[rank + 1]])
            dist.allreduce_sum_(G)
            self._G = G
        return self.G

    def prepare_xv(self, V):
        """Announces the V (p x K) of a later `xv(V)`.  If G is not formed yet, X is float64, whole and resident, G is
        exact, and the stack [X; V^T] has the same row tiles as X (plsb200_gram_stack_fuses), G is then formed as the
        Gram matrix of that stack in one launch: its X block is bit-identical to `gram_of(X)` (same tiles, same voxel splits; a row of G only
        reads its own two rows of the stack) and its X-V^T block is X V, which `xv(V)` returns without a pass of its
        own over X.  Otherwise nothing changes.  Returns whether the product will come from the Gram launch."""
        V = self.to_device(V, F64)
        K = int(V.shape[1])
        fused = (self._G is None and self._pending is None and not self.voxel_sharded and self._X.dtype == F64
                 and not (self.gram_tf32 and self.N <= self.GRAM_TF32_MAX_ROWS) and self.p > 0
                 and V.dim() == 2 and int(V.shape[0]) == self.p and lib.plsb200_gram_stack_fuses(self.N, K) == 1)
        self._xv_next = V if fused else None
        return fused

    def _gram_xv(self):
        V, self._xv_next = self._xv_next, None
        Gs = self.gram_stacked(self.X, V.T.contiguous())
        self._xv_done = (V, Gs[:self.N, self.N:].contiguous())
        return Gs[:self.N, :self.N].contiguous()

    def xv(self, V):
        """XL = X @ V (N x K) for V of p_total x K.  Voxel-sharded: the product of this rank's columns with its rows of V
        plus one all-reduce of N x K doubles (COLLECTIVE).  The V of `prepare_xv`: the product of the Gram launch."""
        V = self.to_device(V, F64)
        if self._xv_next is V:
            self.G
        if self._xv_done is not None and self._xv_done[0] is V:
            return self._xv_done[1]
        K = int(V.shape[1])
        if self.voxel_sharded:
            if int(V.shape[0]) != self.p_total:
                raise ValueError(f"xv: V must have {self.p_total} rows, got {int(V.shape[0])}")
            V = V[self.voxel_range[0]:self.voxel_range[1]].contiguous()
        X = self.X
        if self.p == 0:
            out = torch.zeros(self.N, K, dtype=F64, device=self.device)
        else:
            fn, what = self._xfn("xv_f64", X)
            with torch.cuda.device(self.device):
                ws = self._ws(lib.plsb200_xv_f64_workspace(self.N, self.p, K))
                out = self._empty(self.N, K)
                check(fn(self._p(X), self.N, self.p, self.ldx, self._p(V), K, self._p(out), self._p(ws), ws.numel(),
                         self._stream()), what)
        if self.voxel_sharded:
            self._collective().allreduce_sum_(out)
        return out

    def nspace_coef(self, G, C, Lmat=None):
        """d2[r,k] = C_r[:,k]^T G C_r[:,k] for explicit per-resample coefficients C (R x N x K)."""
        R, N, K = int(C.shape[0]), int(C.shape[1]), int(C.shape[2])
        d2 = self._empty(R, K)
        T = None; Kt = 0
        if Lmat is not None:
            Lmat = self.to_device(Lmat, F64); Kt = int(Lmat.shape[0]); T = self._empty(R, Kt, K)
        with torch.cuda.device(self.device):
            check(lib.plsb200_nspace_coef_f64(self._p(G), N, self._p(C), K, R, self._p(Lmat), Kt, self._p(d2),
                                              self._p(T), self._stream()), "nspace_coef_f64")
        return d2, T

    def nspace_coef_gram(self, G, C):
        """B[r] = C_r^T G C_r (R x K x K) for explicit per-resample coefficients C (R x N x K)."""
        R, N, K = int(C.shape[0]), int(C.shape[1]), int(C.shape[2])
        d2 = self._empty(R, K); B = self._empty(R, K, K)
        with torch.cuda.device(self.device):
            check(lib.plsb200_nspace_coef_gram_f64(self._p(G), N, self._p(C), K, R, self._p(d2), self._p(B),
                                                   self._stream()), "nspace_coef_gram_f64")
        return B

    def pack_coef(self, E, idx):
        """The per-resample coefficients C_r = scatter(E, idx_r) packed in the B-fragment order of the exact bootstrap
        GEMM (one pack serves `boot_moments` and the tensor-core N-space pass).  Returns None when the shape has no
        packed form (K > 24)."""
        E = self.to_device(E, F64); idx = self.to_device(idx, I32)
        R, K = int(idx.shape[0]), int(E.shape[1])
        if K > self.KMAX or R == 0:
            return None
        with torch.cuda.device(self.device):
            nbytes = lib.plsb200_boot_coef_bytes(self.N, K, R)
            if nbytes == 0:
                return None
            coef = self._ws(nbytes)
            check(lib.plsb200_boot_coef_pack_f64(self._p(E), self.N, K, self._p(idx), R, self._p(coef),
                                                 self._stream()), "boot_coef_pack_f64")
        return {"coef": coef, "R": R, "K": K}

    def nspace(self, E, idx, Lmat=None, packed=None):
        """d2[r,k] = ||X^T C_r[:,k]||^2 and (optionally) T[r] = Lmat G C_r diag(1/sqrt(d2)).  Designs up to 320 rows
        and 24 columns run on the FP64 tensor cores from the packed coefficients (`packed`: a `pack_coef` result to
        reuse), the rest on the FMA kernel."""
        E = self.to_device(E, F64); idx = self.to_device(idx, I32)
        R, K = int(idx.shape[0]), int(E.shape[1])
        assert idx.shape[1] == self.N and E.shape[0] == self.N
        d2 = self._empty(R, K)
        T = None; Kt = 0
        if Lmat is not None:
            Lmat = self.to_device(Lmat, F64); Kt = int(Lmat.shape[0])
            assert Lmat.shape[1] == self.N
            T = self._empty(R, Kt, K)
        G = self.G
        ws_bytes = lib.plsb200_nspace_dmma_f64_workspace(self.N, K, Kt, R) if R > 0 else 0
        if ws_bytes:
            if packed is None or packed["R"] != R or packed["K"] != K:
                packed = self.pack_coef(E, idx)
            if packed is not None:
                with torch.cuda.device(self.device):
                    ws = self._ws(ws_bytes)
                    self._mark("nspace")
                    check(lib.plsb200_nspace_dmma_f64(self._p(G), self.N, self._p(Lmat), Kt, self._p(packed["coef"]), K,
                                                      R, self._p(d2), self._p(T), self._p(ws), ws.numel(),
                                                      self._stream()), "nspace_dmma_f64")
                    self._mark("nspace")
                return d2, T
        with torch.cuda.device(self.device):
            check(lib.plsb200_nspace_f64(self._p(G), self.N, self._p(E), K, self._p(idx), R, self._p(Lmat), Kt,
                                         self._p(d2), self._p(T), self._stream()), "nspace_f64")
        return d2, T

    def nspace_gram(self, E, idx):
        """B[r] = C_r^T G C_r (R x K x K), C_r = scatter(E, idx_r): Gram matrix of the resampled cross-block matrix."""
        E = self.to_device(E, F64); idx = self.to_device(idx, I32)
        R, K = int(idx.shape[0]), int(E.shape[1])
        d2 = self._empty(R, K); B = self._empty(R, K, K)
        G = self.G
        with torch.cuda.device(self.device):
            check(lib.plsb200_nspace_gram_f64(self._p(G), self.N, self._p(E), K, self._p(idx), R, self._p(d2),
                                              self._p(B), self._stream()), "nspace_gram_f64")
        return B

    def quad_form(self, G, C):
        """C^T G C (K x K) for a device Gram matrix G (N x N) and coefficients C (N x K): the K x K products of the
        device-side original analysis, on the N-space kernel (no library GEMM)."""
        C = self.to_device(C, F64).contiguous()
        N, K = int(C.shape[0]), int(C.shape[1])
        if (2 * N * K + K) * 8 + N * 4 <= 200 * 1024:         # one column chunk: the kernel writes the full K x K block
            ident = torch.arange(N, dtype=I32, device=self.device)[None].contiguous()
            d2 = self._empty(1, K); B = self._empty(1, K, K)
            with torch.cuda.device(self.device):
                check(lib.plsb200_nspace_gram_f64(self._p(G), N, self._p(C), K, self._p(ident), 1, self._p(d2),
                                                  self._p(B), self._stream()), "nspace_gram_f64")
            return B[0]
        # column chunks: T = C^T (G C) diag(1 / sqrt(d2)) from the kernel, un-normalised again (d2 = 0 <=> zero column)
        d2, T = self.nspace_coef(G, C[None], Lmat=C.T.contiguous())
        return T[0] * torch.sqrt(torch.clamp(d2[0], min=0.0))[None, :]

    def perm_count(self, d2, s_ref, totcov_ref, thresh, counts=None, mb_total=None):
        d2 = self.to_device(d2, F64)
        R, K = int(d2.shape[0]), int(d2.shape[1])
        s_ref = self.to_device(s_ref, F64); totcov_ref = self.to_device(totcov_ref, F64)
        if mb_total is not None:
            mb_total = self.to_device(mb_total, F64)
        if counts is None:
            counts = torch.zeros(2 * K, dtype=torch.int64, device=self.device)
        s_hat = self._empty(R, K)
        with torch.cuda.device(self.device):
            check(lib.plsb200_perm_count_f64(self._p(d2), R, K, self._p(s_ref), self._p(totcov_ref), float(thresh),
                                             self._p(mb_total), self._p(counts), self._p(s_hat), self._stream()),
                  "perm_count_f64")
        return counts, s_hat

    def uhat(self, XL, Lop, idx, R=None):
        """Lop . XL[idx_r] per resample.  XL is (N x K) shared, or (R x N x K) one latent matrix per resample;
        idx may be None (identity)."""
        XL = self.to_device(XL, F64); Lop = self.to_device(Lop, F64)
        idx = self.to_device(idx, I32) if idx is not None else None
        per = XL.dim() == 3
        if R is None:
            R = int(idx.shape[0]) if idx is not None else int(XL.shape[0])
        N, K, Ku = int(XL.shape[-2]), int(XL.shape[-1]), int(Lop.shape[0])
        out = self._empty(R, Ku, K)
        with torch.cuda.device(self.device):
            check(lib.plsb200_uhat_f64(self._p(XL), N * K if per else 0, N, K, self._p(Lop), Ku, self._p(idx), R,
                                       self._p(out), self._stream()), "uhat_f64")
        return out

    def scatter_coef(self, E, idx):
        E = self.to_device(E, F64); idx = self.to_device(idx, I32)
        R, N, K = int(idx.shape[0]), int(E.shape[0]), int(E.shape[1])
        C = self._empty(R, N, K)
        with torch.cuda.device(self.device):
            check(lib.plsb200_scatter_coef_f64(self._p(E), N, K, self._p(idx), R, self._p(C), self._stream()),
                  "scatter_coef_f64")
        return C

    def coef_project(self, C1, d2, Uc):
        Uc = self.to_device(Uc, F64)
        R, N, M, K = int(C1.shape[0]), int(C1.shape[1]), int(C1.shape[2]), int(Uc.shape[1])
        C2 = self._empty(R, N, K)
        with torch.cuda.device(self.device):
            check(lib.plsb200_coef_project_f64(self._p(C1), N, M, self._p(d2), self._p(Uc), K, R, self._p(C2),
                                               self._stream()), "coef_project_f64")
        return C2


    def _ximage_of(self, i, v0, v1, ev):
        """TF32 hi/lo planes of the voxel range [v0, v1) of X in the tile order of the tcgen05 kernel (fast mode),
        built once per engine and range."""
        if self._ximage is None:
            self._ximage = {}
        if i not in self._ximage:
            if ev is not None:
                torch.cuda.current_stream(self.device).wait_event(ev)
            with torch.cuda.device(self.device):
                img = self._ws(lib.plsb200_tf32_ximage_bytes(self.N, v1 - v0))
                split, what = self._xfn("tf32_split_x")
                check(split(self._xp(v0), self.N, v1 - v0, self.ldx, self._p(img), self._stream()), what)
            self._ximage[i] = (v0, v1, img)
        return self._ximage[i][2]

    def _boot_moments_tf32(self, E, idx, pivot, R, K):
        with torch.cuda.device(self.device):
            nbytes = lib.plsb200_boot_coef_bytes_tf32(self.N, K, R)
            if nbytes == 0:
                raise _lib.PlsB200Error(f"boot_moments (tf32x3): unsupported shape N={self.N} K={K} R={R}")
            coef = self._ws(nbytes)
            check(lib.plsb200_boot_coef_pack_tf32(self._p(E), self.N, K, self._p(idx), R, self._p(coef),
                                                  self._stream()), "boot_coef_pack_tf32")
            s1 = self._empty(self.p, K); s2 = self._empty(self.p, K)
            # the voxel ranges of the first call stay the unit of work for later calls (their images are cached)
            if self._tf32_ranges is None:
                self._tf32_ranges = self._x_ranges()
            for i, (v0, v1, ev) in enumerate(self._tf32_ranges):
                img = self._ximage_of(i, v0, v1, ev)         # split of range i, then straight away its GEMM
                pc = v1 - v0
                ws = self._ws(lib.plsb200_boot_moments_tf32_workspace(self.N, pc, K, R))
                self._mark("boot_moments")
                check(lib.plsb200_boot_moments_tf32(self._p(img), self.N, pc, self._p(coef), K, R,
                                                    None if pivot is None else pivot.data_ptr() + 8 * v0 * K,
                                                    s1.data_ptr() + 8 * v0 * K, s2.data_ptr() + 8 * v0 * K,
                                                    self._p(ws), ws.numel(), self._stream()), "boot_moments_tf32")
                self._mark("boot_moments")
        return s1, s2

    KMAX = 24   # columns per boot_moments launch

    def boot_moments(self, E, idx, pivot=None, packed=None):
        """K4: sum_r (VS_r - pivot), sum_r (VS_r - pivot)^2 with VS_r = X^T scatter(E, idx_r); p x K each.
        `packed`: a `pack_coef` result for the same (E, idx) to reuse in the exact mode."""
        E = self.to_device(E, F64); idx = self.to_device(idx, I32)
        R, K = int(idx.shape[0]), int(E.shape[1])
        if pivot is not None:
            pivot = self.to_device(pivot, F64)
        if K > self.KMAX:
            return self._column_blocks(K, lambda k0, k1: self.boot_moments(
                E[:, k0:k1].contiguous(), idx, None if pivot is None else pivot[:, k0:k1].contiguous()))
        self._x_ranges()          # (starts a deferred upload of X now: every small input is already on its way)
        if self.p == 0:           # the empty voxel slice of a voxel-sharded rank
            return self._empty(0, K), self._empty(0, K)
        if self.precision == "tf32x3":
            return self._boot_moments_tf32(E, idx, pivot, R, K)
        with torch.cuda.device(self.device):
            if packed is None or packed["R"] != R or packed["K"] != K:
                packed = self.pack_coef(E, idx)
            if packed is None:
                raise _lib.PlsB200Error(f"boot_moments: unsupported shape N={self.N} K={K} R={R}")
            coef = packed["coef"]
            s1 = self._empty(self.p, K); s2 = self._empty(self.p, K)
            fn, what = self._xfn("boot_moments_f64")
            for v0, v1 in self._x_stream():             # one launch per voxel range still arriving, else one in all
                pc = v1 - v0
                ws = self._ws(lib.plsb200_boot_moments_f64_workspace(self.N, pc, K, R))
                self._mark("boot_moments")
                check(fn(self._xp(v0), self.N, pc, self.ldx, self._p(coef), K, R,
                         None if pivot is None else pivot.data_ptr() + 8 * v0 * K,
                         s1.data_ptr() + 8 * v0 * K, s2.data_ptr() + 8 * v0 * K,
                         self._p(ws), ws.numel(), self._stream()), what)
                self._mark("boot_moments")
        return s1, s2

    QUAD_MAX_ROWS = 320     # designs the collapsed bootstrap's register-resident quadratic-form kernel holds

    def boot_cov(self, E, idx, max_bytes=1 << 30):
        """Partial sums of the collapsed bootstrap over the resamples in `idx`, pivoted at the original coefficients
        (d_r = scatter(E, idx_r) - E): S1 = sum_r d_r (N x K) and S2[k] = sum_r d_rk d_rk^T (K x N x N).  They add up
        over any split of the resamples (a multi-process run all-reduces them).  N-space only -- X is not read.
        Per chunk of resamples (at most `max_bytes` of workspace) the K matrices [d_1k ... d_Rk; 1 ... 1] ((N + 1) x R)
        go through the FP64 Gram kernel: their Gram matrix holds S2[k] and, in its last column, S1[:, k].  Chunks
        are summed in a fixed order."""
        E = self.to_device(E, F64); idx = self.to_device(idx, I32)
        R, N, K = int(idx.shape[0]), int(E.shape[0]), int(E.shape[1])
        S = torch.zeros(K, N + 1, N + 1, dtype=F64, device=self.device)
        rc = max(1, min(R, int(max_bytes // (8 * (N * K + K * (N + 1))))))
        Et = E.T.contiguous()
        for r0 in range(0, R, rc):
            n = min(rc, R - r0)
            C = self.scatter_coef(E, idx[r0:r0 + n])                      # n x N x K
            M = torch.ones(K, N + 1, n, dtype=F64, device=self.device)
            M[:, :N, :].copy_(C.permute(2, 1, 0)).sub_(Et[:, :, None])
            del C
            for k in range(K):
                S[k] += self.gram_of(M[k])
            del M
        return S[:, :N, N].T.contiguous(), S[:, :N, :N].contiguous()

    def boot_quad(self, Sig, v0=0, v1=None):
        """Collapsed bootstrap: q[v,k] = x_v^T Sig[k] x_v for the voxels v0 <= v < v1 ((v1 - v0) x K).  With
        Sig[k] = R . Cov_r(c_rk), (sum = 0, sumsq = q) are the moments `boot_finalize` turns into standard errors.
        One launch per voxel range of a pipelined upload, each after its range has arrived.  Designs of at most
        320 rows."""
        Sig = self.to_device(Sig, F64)
        K, N = int(Sig.shape[0]), int(Sig.shape[1])
        v1 = self.p if v1 is None else int(v1)
        if N != self.N or tuple(Sig.shape) != (K, N, N):
            raise ValueError(f"boot_quad: Sig must be K x {self.N} x {self.N}")
        if K > self.KMAX:
            return self._column_blocks(K, lambda k0, k1: self.boot_quad(Sig[k0:k1], v0, v1))
        q = self._empty(max(v1 - v0, 0), K)
        if v1 <= v0:
            return q
        with torch.cuda.device(self.device):
            nbytes = lib.plsb200_boot_quad_coef_bytes(N, K)
            if nbytes == 0:
                raise _lib.PlsB200Error(f"boot_quad: unsupported shape N={N} K={K} (N <= {self.QUAD_MAX_ROWS})")
            coef = self._ws(nbytes)
            check(lib.plsb200_boot_quad_coef_pack_f64(self._p(Sig), N, K, self._p(coef), self._stream()),
                  "boot_quad_coef_pack_f64")
            fn, what = self._xfn("boot_quad_f64")
            for lo, hi in self._x_stream(v0, v1):
                ws = self._ws(lib.plsb200_boot_quad_f64_workspace(N, hi - lo, K))
                self._mark("boot_quad")
                check(fn(self._xp(lo), N, hi - lo, self.ldx, self._p(coef), K, q.data_ptr() + 8 * (lo - v0) * K,
                         self._p(ws), ws.numel(), self._stream()), what)
                self._mark("boot_quad")
        return q

    def boot_draw_check(self, idx, layout):
        """A one-element int32 device tensor, nonzero unless every draw in `idx` keeps each row in its cell and uses one
        subject map for all conditions (the structure of resample.bootstrap_indices).  `layout`: the int32 row layout of
        plsb200_boot_counts_f64."""
        idx = self.to_device(idx, I32); layout = self.to_device(layout, I32)
        R = int(idx.shape[0])
        ns = int(layout.numel()) - 2 * self.N
        bad = torch.zeros(1, dtype=I32, device=self.device)
        with torch.cuda.device(self.device):
            check(lib.plsb200_boot_counts_f64(self._p(idx), self.N, R, self._p(layout), ns, None, 0, self._p(bad),
                                              self._stream()), "boot_counts_f64")
        return bad

    def boot_count_gram(self, idx, layout):
        """Factored collapsed bootstrap, N-space part of the resamples in `idx`: the (ns + 1)-square Gram matrix of
        [m_r - 1; 1] over the draws (m_r: draws of each subject).  Integer entries, so exact in any summation order; a
        multi-process run all-reduces it."""
        idx = self.to_device(idx, I32); layout = self.to_device(layout, I32)
        R = int(idx.shape[0])
        ns = int(layout.numel()) - 2 * self.N
        counts = self._empty(ns + 1, R)
        with torch.cuda.device(self.device):
            check(lib.plsb200_boot_counts_f64(self._p(idx), self.N, R, self._p(layout), ns, self._p(counts), R, None,
                                              self._stream()), "boot_counts_f64")
        return self.gram_of(counts)

    def boot_factor(self, Mg, R_total, gstart):
        """L (ns x (ns - G)) with L L^T = sum_r (m_r - 1)(m_r - 1)^T - s1 s1^T / R_total from `boot_count_gram`'s
        matrix (summed over every resample); one CTA, no host synchronisation."""
        gstart = self.to_device(gstart, I32)
        ns, G = int(Mg.shape[0]) - 1, int(gstart.numel()) - 1
        L = self._empty(ns, ns - G)
        with torch.cuda.device(self.device):
            ws = self._ws(lib.plsb200_boot_factor_f64_workspace(ns, G))
            check(lib.plsb200_boot_factor_f64(self._p(Mg), ns, int(R_total), self._p(gstart), G, self._p(L), self._p(ws),
                                              ws.numel(), self._stream()), "boot_factor_f64")
        return L

    def boot_factor_quad(self, E, L, sid, v0=0, v1=None):
        """q[v,k] = sum_j (x_v^T c_jk)^2 with c_jk[n] = E[n,k] L[sid[n], j], for the voxels v0 <= v < v1: the bootstrap
        moment GEMM on the J columns of L as pseudo-resamples (no pivot).  With L L^T the draw-count covariance this is
        the q of `boot_quad`.  One launch per voxel range of a pipelined upload, each after its range has arrived."""
        E = self.to_device(E, F64); sid = self.to_device(sid, I32)
        K, J = int(E.shape[1]), int(L.shape[1])
        v1 = self.p if v1 is None else int(v1)
        if K > self.KMAX:
            return self._column_blocks(K, lambda k0, k1: self.boot_factor_quad(E[:, k0:k1].contiguous(), L, sid, v0, v1))
        q = self._empty(max(v1 - v0, 0), K)
        if v1 <= v0:
            return q
        s1 = self._empty(v1 - v0, K)                 # sum_j x_v^T c_jk: not needed, the kernel writes it
        with torch.cuda.device(self.device):
            nbytes = lib.plsb200_boot_factor_coef_bytes(self.N, K, J)
            if nbytes == 0:
                raise _lib.PlsB200Error(f"boot_factor_quad: unsupported shape N={self.N} K={K} J={J} (the factored "
                                        "pack needs 1 <= K <= 24 and J >= 1)")
            coef = self._ws(nbytes)
            check(lib.plsb200_boot_factor_pack_f64(self._p(E), self.N, K, self._p(L), J, self._p(sid), self._p(coef),
                                                   self._stream()), "boot_factor_pack_f64")
            fn, what = self._xfn("boot_moments_f64")
            for lo, hi in self._x_stream(v0, v1):
                ws = self._ws(lib.plsb200_boot_moments_f64_workspace(self.N, hi - lo, K, J))
                off = 8 * (lo - v0) * K
                self._mark("boot_moments")
                check(fn(self._xp(lo), self.N, hi - lo, self.ldx, self._p(coef), K, J, None, s1.data_ptr() + off,
                         q.data_ptr() + off, self._p(ws), ws.numel(), self._stream()), what)
                self._mark("boot_moments")
        return q

    def boot_finalize(self, s1, s2, R_total, numer=None):
        K = int(s1.shape[1])
        se = self._empty(self.p, K)
        br = self._empty(self.p, K) if numer is not None else None
        if numer is not None:
            numer = self.to_device(numer, F64)
        if self.p == 0:
            return se, br
        with torch.cuda.device(self.device):
            check(lib.plsb200_boot_finalize_f64(self._p(s1), self._p(s2), self.p, K, int(R_total), self._p(numer),
                                                self._p(se), self._p(br), self._stream()), "boot_finalize_f64")
        return se, br

    def colstd(self, A):
        A = self.to_device(A, F64)
        R = int(A.shape[0]); M = int(A.numel() // R)
        out = self._empty(*A.shape[1:])
        with torch.cuda.device(self.device):
            check(lib.plsb200_colstd_f64(self._p(A), R, M, self._p(out), self._stream()), "colstd_f64")
        return out

    def percentile_interval(self, A, conf=(0.05, 0.95)):
        """Element-wise percentile interval over the first axis of a (B x ...) stack (resample.py:171-222, MATLAB
        prctile convention); returns (lower, upper) device tensors shaped like A[0]."""
        A = self.to_device(A, F64)
        B = int(A.shape[0]); M = int(A.numel() // B)
        lo = self._empty(*A.shape[1:]); hi = self._empty(*A.shape[1:])
        with torch.cuda.device(self.device):
            nb = lib.plsb200_percentile_f64_workspace(B)
            ws = self._ws(nb)
            check(lib.plsb200_percentile_f64(self._p(A), B, M, M, 1, float(conf[0]), float(conf[1]), self._p(lo),
                                             self._p(hi), self._p(ws), nb, self._stream()), "percentile_f64")
        return lo, hi

    def percentile_interval_bc(self, A, orig, conf=(0.05, 0.95)):
        """Bias-corrected percentile interval (Efron) over the first axis of a (B x ...) stack: `orig`, shaped like
        A[0], holds the original value theta of every element; prop = #{samples <= theta} / B and the bounds are taken
        at the levels Phi(2 Phi^-1(prop) + Phi^-1(q)) (DESIGN.md section 5.8).  Returns (lower, upper, prop) device
        tensors shaped like A[0]; lower / upper are NaN where prop is 0 or 1."""
        A = self.to_device(A, F64)
        orig = self.to_device(orig, F64)
        if tuple(orig.shape) != tuple(A.shape[1:]):
            raise ValueError(f"orig has shape {tuple(orig.shape)}, the elements of the stack {tuple(A.shape[1:])}")
        B = int(A.shape[0]); M = int(A.numel() // B)
        lo, hi, prop = (self._empty(*A.shape[1:]) for _ in range(3))
        with torch.cuda.device(self.device):
            nb = lib.plsb200_percentile_f64_workspace(B)
            ws = self._ws(nb)
            check(lib.plsb200_percentile_bc_f64(self._p(A), B, M, M, 1, self._p(orig), float(conf[0]), float(conf[1]),
                                                self._p(lo), self._p(hi), self._p(prop), self._p(ws), nb,
                                                self._stream()), "percentile_bc_f64")
        return lo, hi, prop

    def percentile_interval_bca(self, A, orig, accel, conf=(0.05, 0.95)):
        """Bias-corrected and accelerated percentile interval (BCa, Efron 1987) over the first axis of a (B x ...)
        stack: `orig` and `accel`, shaped like A[0], hold the original value theta and the acceleration a of every
        element.  prop and z0 = Phi^-1(prop) are those of `percentile_interval_bc`; with w = z0 + Phi^-1(q) the bounds
        are taken at the levels Phi(z0 + w / (1 - a w)) (DESIGN.md section 5.8).  Returns (lower, upper, prop) device
        tensors shaped like A[0]; lower / upper are NaN where prop is 0 or 1 and where 1 - a w <= 0, and q = 0 / 1
        give the minimum / maximum.  With a = 0 the bounds are those of `percentile_interval_bc`."""
        A = self.to_device(A, F64)
        orig = self.to_device(orig, F64)
        accel = self.to_device(accel, F64)
        for name, t in (("orig", orig), ("accel", accel)):
            if tuple(t.shape) != tuple(A.shape[1:]):
                raise ValueError(f"{name} has shape {tuple(t.shape)}, the elements of the stack {tuple(A.shape[1:])}")
        B = int(A.shape[0]); M = int(A.numel() // B)
        lo, hi, prop = (self._empty(*A.shape[1:]) for _ in range(3))
        with torch.cuda.device(self.device):
            nb = lib.plsb200_percentile_f64_workspace(B)
            ws = self._ws(nb)
            check(lib.plsb200_percentile_bca_f64(self._p(A), B, M, M, 1, self._p(orig), self._p(accel), float(conf[0]),
                                                 float(conf[1]), self._p(lo), self._p(hi), self._p(prop), self._p(ws),
                                                 nb, self._stream()), "percentile_bca_f64")
        return lo, hi, prop

    def _salience_chunks(self, E, idx, max_bytes, reduce, extra_series=0):
        """Streams the bootstrap salience distribution VS[r] = X^T scatter(E, idx_r) without holding the R x p x K
        cube: voxel chunks of at most `max_bytes` are made explicit series-major and handed to
        `reduce(cube, R, v0, v1, ws, nb)` (ws: nb bytes of percentile workspace), then dropped.  `extra_series`
        samples per element that `reduce` holds next to the chunk count against `max_bytes` too."""
        E = self.to_device(E, F64); idx = self.to_device(idx, I32)
        R, K = int(idx.shape[0]), int(E.shape[1])
        vc = max(128, min(self.p, int(max_bytes // ((R + extra_series) * K * 8)) // 128 * 128))
        X = self.X
        series, what = self._xfn("salience_series_f64", X)
        nb = lib.plsb200_percentile_f64_workspace(R)
        with torch.cuda.device(self.device):
            ws = self._ws(nb)
            for v0 in range(0, self.p, vc):
                v1 = min(self.p, v0 + vc)
                # series-major chunk [voxel][k][resample]: the sort reads every series as one contiguous run (the
                # resample-major cube read in place with a stride of the chunk size cost 23-41 ms per chunk against 17)
                cube = self._empty(v1 - v0, K, R)
                check(series(self._xp(v0), self.N, v1 - v0, self.ldx, self._p(E), K, self._p(idx), R, self._p(cube),
                             self._stream()), what)
                reduce(cube, R, v0, v1, ws, nb)
                del cube

    def salience_percentiles(self, E, idx, conf=(0.05, 0.95), max_bytes=4 << 30):
        """Percentile interval of every element of the bootstrap salience distribution VS[r] = X^T scatter(E, idx_r)
        (what `confidence_interval(right_sv_sampled)` would give) without holding the R x p x K cube: voxel chunks
        of at most `max_bytes` are made explicit (`salience`), reduced to their two bounds and dropped.
        Returns (lower, upper), p x K device tensors."""
        K = int(E.shape[1])
        lo = self._empty(self.p, K); hi = self._empty(self.p, K)

        def reduce(cube, R, v0, v1, ws, nb):
            check(lib.plsb200_percentile_f64(self._p(cube), R, (v1 - v0) * K, 1, R, float(conf[0]), float(conf[1]),
                                             lo.data_ptr() + 8 * v0 * K, hi.data_ptr() + 8 * v0 * K, self._p(ws), nb,
                                             self._stream()), "percentile_f64")
        self._salience_chunks(E, idx, max_bytes, reduce)
        return lo, hi

    def salience_percentiles_bc(self, E, idx, orig, conf=(0.05, 0.95), max_bytes=4 << 30):
        """Bias-corrected percentile interval (`percentile_interval_bc`) of every element of the same streamed
        distribution; `orig` (p x K, this engine's voxels) is the original salience of every element.
        Returns (lower, upper, prop), p x K device tensors."""
        K = int(E.shape[1])
        orig = self.to_device(orig, F64)
        if tuple(orig.shape) != (self.p, K):
            raise ValueError(f"orig has shape {tuple(orig.shape)}, the saliences {(self.p, K)}")
        lo, hi, prop = (self._empty(self.p, K) for _ in range(3))

        def reduce(cube, R, v0, v1, ws, nb):
            off = 8 * v0 * K
            check(lib.plsb200_percentile_bc_f64(self._p(cube), R, (v1 - v0) * K, 1, R, orig.data_ptr() + off,
                                                float(conf[0]), float(conf[1]), lo.data_ptr() + off,
                                                hi.data_ptr() + off, prop.data_ptr() + off, self._p(ws), nb,
                                                self._stream()), "percentile_bc_f64")
        self._salience_chunks(E, idx, max_bytes, reduce)
        return lo, hi, prop

    def salience_percentiles_bca(self, E, idx, orig, jack, conf=(0.05, 0.95), max_bytes=4 << 30):
        """Bias-corrected and accelerated percentile interval (`percentile_interval_bca`) of every element of the same
        streamed distribution.  `orig` (p x K, this engine's voxels) is the original salience of every element;
        `jack` = (C, goff): C (J x N x K) the coefficients of the J leave-one-subject-out saliences X^T C_j, and goff
        (G + 1 offsets) the groups of the J subjects.  Per voxel chunk the bootstrap cube and the jackknife cube
        (voxel x K x J, `salience_coef_series_f64`) are made explicit -- `max_bytes` bounds the two together -- the
        stratified jackknife acceleration of every element is formed (`jack_accel_f64`, pivot at `orig`) and the
        chunk is sorted.  Returns (lower, upper, prop, accel), p x K device tensors."""
        K = int(E.shape[1])
        orig = self.to_device(orig, F64)
        if tuple(orig.shape) != (self.p, K):
            raise ValueError(f"orig has shape {tuple(orig.shape)}, the saliences {(self.p, K)}")
        Cj = self.to_device(jack[0], F64); goff = self.to_device(jack[1], I32)
        J, G = int(Cj.shape[0]), int(goff.shape[0]) - 1
        if tuple(Cj.shape) != (J, self.N, K):
            raise ValueError(f"jackknife coefficients of shape {tuple(Cj.shape)}, need (J, {self.N}, {K})")
        lo, hi, prop, accel = (self._empty(self.p, K) for _ in range(4))
        jfn, jwhat = self._xfn("salience_coef_series_f64", self.X)

        def reduce(cube, R, v0, v1, ws, nb):
            off, n = 8 * v0 * K, (v1 - v0) * K
            jc = self._empty(v1 - v0, K, J)
            check(jfn(self._xp(v0), self.N, v1 - v0, self.ldx, self._p(Cj), K, J, self._p(jc), self._stream()), jwhat)
            check(lib.plsb200_jack_accel_f64(self._p(jc), n, J, self._p(goff), G, orig.data_ptr() + off,
                                             accel.data_ptr() + off, self._stream()), "jack_accel_f64")
            del jc
            check(lib.plsb200_percentile_bca_f64(self._p(cube), R, n, 1, R, orig.data_ptr() + off,
                                                 accel.data_ptr() + off, float(conf[0]), float(conf[1]),
                                                 lo.data_ptr() + off, hi.data_ptr() + off, prop.data_ptr() + off,
                                                 self._p(ws), nb, self._stream()), "percentile_bca_f64")
        self._salience_chunks(E, idx, max_bytes, reduce, extra_series=J)
        return lo, hi, prop, accel

    def salience(self, E, idx, M=None):
        """Explicit VS[r] = M^T scatter(E, idx_r) (R x p x K), M = X by default -- small R only."""
        E = self.to_device(E, F64); idx = self.to_device(idx, I32)
        M = self.X if M is None else M
        n, p, ld = int(M.shape[0]), int(M.shape[1]), int(M.stride(0))
        R, K = int(idx.shape[0]), int(E.shape[1])
        out = self._empty(R, p, K)
        if p == 0:
            return out
        fn, what = self._xfn("salience_f64", M)
        with torch.cuda.device(self.device):
            check(fn(self._p(M), n, p, ld, self._p(E), K, self._p(idx), R, self._p(out), self._stream()), what)
        return out

    def salience_window(self, E, idx):
        """The task-method saliences VS[r] = X^T scatter(E, idx_r) over a voxel window: returns `fill(v0, v1, out)`,
        which writes voxels [v0, v1) of this engine's columns into `out` (R x (v1 - v0) x K, contiguous float64) with
        `salience_f64` (or its float32 twin) read in place through the row stride of X.  E and the index matrix are
        uploaded once, here; the values are those of `salience` bit for bit."""
        E = self.to_device(E, F64); idx = self.to_device(idx, I32)
        R, K = int(idx.shape[0]), int(E.shape[1])
        X = self.X
        fn, what = self._xfn("salience_f64", X)

        def fill(v0, v1, out):
            with torch.cuda.device(self.device):
                check(fn(self._xp(v0), self.N, v1 - v0, self.ldx, self._p(E), K, self._p(idx), R, self._p(out),
                         self._stream()), what)
        return fill

    def stream_chunks(self, fill, B, K, max_bytes, v_offset=0):
        """Generator over the B x p x K cube that `fill(v0, v1, out)` computes window by window (out: B x (v1 - v0) x K,
        contiguous float64 on the device), in voxel chunks of at most `max_bytes` (at least one voxel): yields
        (v_offset + v0, v_offset + v1, chunk), chunk a float64 numpy array B x (v1 - v0) x K that stays valid until the
        next step.  Two device buffers and two pinned host buffers: chunk c is copied on the side stream (the one of
        `to_host_async(side=True)`) while chunk c+1 is computed, and is yielded once its copy has finished; chunk c+1
        is then copied while the caller reads chunk c.  Closing the generator early waits for the work in flight and
        frees the buffers."""
        p = self.p
        vc = max(1, min(p, int(max_bytes) // (B * K * 8)))
        spans = [(v0, min(p, v0 + vc)) for v0 in range(0, p, vc)]
        if not spans:
            return
        cur = torch.cuda.current_stream(self.device)
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(device=self.device)
        side = self._copy_stream
        n = B * vc * K
        dev = [self._empty(n) for _ in range(min(2, len(spans)))]
        host = [torch.empty(n, dtype=F64, pin_memory=True) for _ in dev]
        computed = [torch.cuda.Event() for _ in dev]
        copied = [torch.cuda.Event() for _ in dev]

        def launch(c):          # compute chunk c on the current stream, then copy it on the side stream
            v0, v1 = spans[c]
            i, m = c % 2, B * (v1 - v0) * K
            with torch.cuda.stream(cur):
                fill(v0, v1, dev[i][:m].view(B, v1 - v0, K))
                computed[i].record(cur)
            side.wait_event(computed[i])
            with torch.cuda.stream(side):
                host[i][:m].copy_(dev[i][:m], non_blocking=True)
                copied[i].record(side)
        try:
            launch(0)
            for c, (v0, v1) in enumerate(spans):
                if c + 1 < len(spans):
                    # chunk c+1 is computed while chunk c is copied, and copied while the caller reads chunk c: its
                    # buffers held chunk c-1, whose copy finished before chunk c-1 was yielded and which the caller
                    # has let go of by asking for the next step
                    launch(c + 1)
                copied[c % 2].synchronize()
                yield v_offset + v0, v_offset + v1, host[c % 2][:B * (v1 - v0) * K].numpy().reshape(B, v1 - v0, K)
        finally:
            side.synchronize()
            cur.synchronize()
            del dev, host

    # ------------------------------------------------------------------ split-half (K3)
    def sym_eig(self, A):
        """Batched symmetric eigendecomposition (B x K x K, K <= 112): evals descending, evecs in columns.
        Raises if a matrix did not converge within the solver's sweep limit."""
        A = self.to_device(A, F64)
        B, K = int(A.shape[0]), int(A.shape[1])
        ev = self._empty(B, K); U = self._empty(B, K, K)
        status = torch.empty(B, dtype=I32, device=self.device)
        with torch.cuda.device(self.device):
            check(lib.plsb200_sym_eig_f64(self._p(A), K, B, self._p(ev), self._p(U), self._p(status), self._stream()),
                  "sym_eig_f64")
        self._check_converged(status, "sym_eig")
        return ev, U

    def _check_converged(self, status, what):
        """One scalar read-back (the callers read the results back right after anyway): the Jacobi solvers flag
        matrices that hit their sweep limit and such results must not be consumed."""
        bad = int(status.sum().item())
        if bad:
            raise _lib.PlsB200Error(f"{what}: the Jacobi eigensolver did not converge for {bad} of {status.numel()} "
                                    "matrices")

    def split_gram(self, idx1, idx2, A1, A2):
        """S11, S12, S22 (S x K x K) of the half-sample cross-block matrices M_h = A_h X[idx_h]."""
        idx1 = self.to_device(idx1, I32); idx2 = self.to_device(idx2, I32)
        A1 = self.to_device(A1, F64); A2 = self.to_device(A2, F64)
        S, n1, n2, K = int(idx1.shape[0]), int(idx1.shape[1]), int(idx2.shape[1]), int(A1.shape[0])
        assert A1.shape[1] == n1 and A2.shape == (K, n2) and idx2.shape[0] == S
        out = [self._empty(S, K, K) for _ in range(3)]
        G = self.G
        with torch.cuda.device(self.device):
            check(lib.plsb200_split_gram_f64(self._p(G), self.N, self._p(idx1), n1, self._p(idx2), n2, S, self._p(A1),
                                             self._p(A2), K, self._p(out[0]), self._p(out[1]), self._p(out[2]),
                                             self._stream()), "split_gram_f64")
        return out

    def split_svd(self, S11, S12, S22):
        """(s_train, s_test, u_repro, v_repro, s2) from the Gram blocks (see include/plsb200.h)."""
        S, K = int(S11.shape[0]), int(S11.shape[1])
        s1 = self._empty(S, K); s2 = self._empty(S, K)
        st = self._empty(S, K, K); ur = self._empty(S, K, K); vr = self._empty(S, K, K)
        status = torch.empty(S, dtype=I32, device=self.device)
        with torch.cuda.device(self.device):
            ws = self._ws(lib.plsb200_split_svd_f64_workspace(K, S))
            check(lib.plsb200_split_svd_f64(self._p(S11), self._p(S12), self._p(S22), K, S, self._p(s1), self._p(st),
                                            self._p(ur), self._p(vr), self._p(s2), self._p(status), self._p(ws),
                                            ws.numel(), self._stream()), "split_svd_f64")
        self._check_converged(status, "split_svd")
        return s1, st, ur, vr, s2

    # ------------------------------------------------------------------ behaviour PLS (K5)
    def cell_standardize(self, cell_start, want_z=True, M=None):
        """Xc = M - block means, Z = block z-score(M) / sqrt(n) (both rows x p, dense); M defaults to X."""
        cs = self.to_device(np.asarray(cell_start, dtype=np.int32), I32)
        M = self.X if M is None else M
        self._need_f64(M, "cell_standardize"); self._need_whole_x("cell_standardize")
        n, p, ld = int(M.shape[0]), int(M.shape[1]), int(M.stride(0))
        Xc = self._empty(n, p)
        Z = self._empty(n, p) if want_z else None
        with torch.cuda.device(self.device):
            check(lib.plsb200_cell_standardize_f64(self._p(M), n, p, ld, self._p(cs), int(cs.numel()) - 1,
                                                   self._p(Xc), self._p(Z), self._stream()), "cell_standardize_f64")
        return Xc, Z

    def rb_coef(self, Y, idx, cell_start, U, scatter, want_yz=False):
        Y = self.to_device(Y, F64); U = self.to_device(U, F64)
        cs = self.to_device(np.asarray(cell_start, dtype=np.int32), I32)
        idx = self.to_device(idx, I32) if idx is not None else None
        nb = int(Y.shape[1])
        # number of resampled rows = length of an index vector (half-samples are shorter than Y)
        N = int(idx.shape[1]) if idx is not None else int(Y.shape[0])
        R = int(idx.shape[0]) if idx is not None else 1
        Kc = int(U.shape[1])
        if int(cs[-1].item()) != N:
            raise ValueError(f"rb_coef: blocks cover {int(cs[-1].item())} rows, index vectors have {N}")
        if scatter and N != int(Y.shape[0]):
            raise ValueError("rb_coef: scatter mode needs full-length index vectors")
        Q = self._empty(R, N, Kc)
        W = self._empty(R, N) if scatter else None
        Yz = self._empty(R, N, nb) if want_yz else None
        with torch.cuda.device(self.device):
            check(lib.plsb200_rb_coef_f64(self._p(Y), N, nb, self._p(idx), R, self._p(cs), int(cs.numel()) - 1,
                                          self._p(U), Kc, int(bool(scatter)), self._p(Q), self._p(W), self._p(Yz),
                                          self._stream()), "rb_coef_f64")
        return Q, W, Yz

    def rb_boot(self, Xc, Q, W, cell_start, pivot=None, unit_cells=0, max_ws_bytes=2 << 30, want_t=True, X2=None,
                vs_out=None):
        """p-space pass over all bootstraps in Q: returns (sum, sumsq) of VS - pivot (p x K),
        T (R x N x K) = Xc @ VS_b (None when want_t is False) and nrm2 (R x K).  `vs_out`: an R x p x K float64 device
        tensor that receives the saliences VS_b themselves (the reference's right_sv_sampled); with want_t=False the
        call is the p-space pass alone.
        Runs on the FP64 tensor path (plsb200_rb_boot_dmma_f64) when the design fits its register-resident
        fragments, else on the general FMA kernel.  `X2`: the data matrix is the row stack [Xc; X2] (not built: the
        kernels take the two row segments; multiblock bootstraps pass [Xcb; X])."""
        self._need_f64(Xc, "rb_boot"); self._need_f64(X2, "rb_boot"); self._need_whole_x("rb_boot")
        cs_host = np.ascontiguousarray(np.asarray(cell_start, dtype=np.int32))
        R, N, K = int(Q.shape[0]), int(Q.shape[1]), int(Q.shape[2])
        p = int(Xc.shape[1])
        n1 = int(Xc.shape[0])
        ld2 = int(X2.stride(0)) if X2 is not None else p
        if n1 + (int(X2.shape[0]) if X2 is not None else 0) != N:
            raise ValueError("rb_boot: coefficient rows do not match the data matrix")
        if vs_out is not None and (vs_out.dtype != F64 or tuple(vs_out.shape) != (R, p, K) or not vs_out.is_contiguous()
                                   or vs_out.device != torch.device(self.device)):
            raise ValueError(f"rb_boot: vs_out must be a contiguous float64 tensor of shape {(R, p, K)} on {self.device}")
        ncell = int(cs_host.size) - 1
        s1 = torch.zeros(p, K, dtype=F64, device=self.device); s2 = torch.zeros_like(s1)
        T = self._empty(R, N, K) if want_t else None
        nrm2 = self._empty(R, K)
        if pivot is not None:
            pivot = self.to_device(pivot, F64)
        Xc = Xc.contiguous()
        per = lib.plsb200_rb_boot_dmma_f64_workspace(N, p, K, 1, cs_host.ctypes.data, ncell, int(unit_cells),
                                                     int(want_t))
        if per and not getattr(self, "force_rb_fma", False):
            self.last_rb_path = "dmma"
            nbt = max(1, min(R, int(max_ws_bytes // per)))
            ws_bytes = lib.plsb200_rb_boot_dmma_f64_workspace(N, p, K, nbt, cs_host.ctypes.data, ncell,
                                                              int(unit_cells), int(want_t))
            with torch.cuda.device(self.device):
                ws = self._ws(ws_bytes)
                self._mark("rb_boot")
                for b0 in range(0, R, nbt):
                    n = min(nbt, R - b0)
                    check(lib.plsb200_rb_boot_dmma_vs_f64(self._p(Xc), N, p, self._p(X2), n1, ld2, self._p(Q), self._p(W), K,
                                                          b0, n, cs_host.ctypes.data, ncell, int(unit_cells),
                                                          self._p(pivot), self._p(s1), self._p(s2), self._p(T),
                                                          self._p(nrm2), self._p(vs_out), self._p(ws), ws.numel(),
                                                          self._stream()), "rb_boot_dmma_f64")
                self._mark("rb_boot")
            return s1, s2, T, nrm2
        # design outside the tensor-core kernel's buckets (more than 16 blocks or 384 rows after padding every block to a
        # multiple of 4): the general FMA kernel is an order of magnitude slower -- say so once instead of silently
        if not getattr(self, "force_rb_fma", False) and not getattr(Engine, "_warned_rb_fma", False):
            import warnings
            Engine._warned_rb_fma = True
            warnings.warn(f"plspy_b200: behaviour / multiblock bootstrap with {ncell} blocks and {N} rows runs on the "
                          "general FMA kernel (the DMMA kernel holds up to 16 blocks / 384 padded rows): expect ~10x "
                          "less throughput", RuntimeWarning, stacklevel=3)
        self.last_rb_path = "fma"
        cs = self.to_device(cs_host, I32)
        if T is None:
            T = self._empty(R, N, K)
        per = lib.plsb200_rb_boot_f64_workspace(N, p, K, 1)
        nbt = max(1, min(R, int(min(max_ws_bytes, 512 << 20) // max(per, 1))))
        with torch.cuda.device(self.device):
            ws = self._ws(per * nbt)
            self._mark("rb_boot")
            for b0 in range(0, R, nbt):
                n = min(nbt, R - b0)
                check(lib.plsb200_rb_boot_vs_f64(self._p(Xc), N, p, self._p(X2), n1, ld2, self._p(Q), self._p(W), K, b0, n,
                                                 self._p(cs), ncell, int(unit_cells), self._p(pivot), self._p(s1),
                                                 self._p(s2), self._p(T), self._p(nrm2), self._p(vs_out), self._p(ws),
                                                 ws.numel(), self._stream()), "rb_boot_f64")
            self._mark("rb_boot")
        return s1, s2, (T if want_t else None), nrm2

    def rb_salience(self, Xc, Q, W, cell_start, unit_cells=0, X2=None):
        """The export-only p-space pass of `rb_boot` over a voxel window: returns `fill(v0, v1, out)`, which writes the
        saliences VS_b of voxels [v0, v1) of every bootstrap in Q into `out` (R x (v1 - v0) x K, contiguous float64),
        bit-identical to the `vs_out` of `rb_boot`.  Runs on the DMMA kernel when the design fits it (its coefficients
        are packed once, here, for every window) and on the FMA kernel otherwise or with `force_rb_fma`, like
        `rb_boot`.  `X2`: the data matrix is the row stack [Xc; X2]."""
        self._need_f64(Xc, "rb_salience"); self._need_f64(X2, "rb_salience"); self._need_whole_x("rb_salience")
        cs_host = np.ascontiguousarray(np.asarray(cell_start, dtype=np.int32))
        R, N, K = int(Q.shape[0]), int(Q.shape[1]), int(Q.shape[2])
        n1, ld1 = int(Xc.shape[0]), int(Xc.stride(0))
        ld2 = int(X2.stride(0)) if X2 is not None else ld1
        if n1 + (int(X2.shape[0]) if X2 is not None else 0) != N:
            raise ValueError("rb_salience: coefficient rows do not match the data matrix")
        ncell = int(cs_host.size) - 1
        nbytes = lib.plsb200_rb_salience_dmma_f64_workspace(N, K, R, cs_host.ctypes.data, ncell, int(unit_cells))
        if nbytes and not getattr(self, "force_rb_fma", False):
            self.last_rb_path = "dmma"
            with torch.cuda.device(self.device):
                ws = self._ws(nbytes)
                check(lib.plsb200_rb_salience_dmma_pack_f64(self._p(Q), self._p(W), N, K, R, cs_host.ctypes.data, ncell,
                                                            int(unit_cells), self._p(ws), ws.numel(), self._stream()),
                      "rb_salience_dmma_pack_f64")

            def fill(v0, v1, out):
                with torch.cuda.device(self.device):
                    check(lib.plsb200_rb_salience_dmma_f64(self._p(Xc), N, ld1, self._p(X2), n1, ld2, v0, v1, K, R,
                                                           cs_host.ctypes.data, ncell, int(unit_cells), self._p(out),
                                                           self._p(ws), ws.numel(), self._stream()),
                          "rb_salience_dmma_f64")
            return fill
        self.last_rb_path = "fma"
        cs = self.to_device(cs_host, I32)

        def fill(v0, v1, out):
            with torch.cuda.device(self.device):
                check(lib.plsb200_rb_salience_f64(self._p(Xc), N, ld1, self._p(X2), n1, ld2, v0, v1, self._p(Q),
                                                  self._p(W), K, R, self._p(cs), ncell, int(unit_cells), self._p(out),
                                                  self._stream()), "rb_salience_f64")
        return fill

    def rb_lvcorr(self, T, nrm2, Yz, idx, cell_start, nb):
        cs = self.to_device(np.asarray(cell_start, dtype=np.int32), I32)
        idx = self.to_device(idx, I32) if idx is not None else None
        R, N, K = int(T.shape[0]), int(T.shape[1]), int(T.shape[2])
        ncell = int(cs.numel()) - 1
        LV = self._empty(R, ncell * nb, K)
        with torch.cuda.device(self.device):
            check(lib.plsb200_rb_lvcorr_f64(self._p(T), self._p(nrm2), self._p(Yz), self._p(idx), N, nb, K, R,
                                            self._p(cs), ncell, self._p(LV), self._stream()), "rb_lvcorr_f64")
        return LV

    def half_gram(self, Xstd, Xlin, ids, Q, cells, unit_cells, max_ws_bytes=256 << 20, dense=False):
        """Split-half Gram blocks in p-space: ids (S x 2 x nmax int32), Q (S x 2 x nmax x K),
        cells (2 x (ncell+1) int32 position offsets).  Returns S3 (S x 3 x K x K) = [S11, S12, S22].
        The windowed kernel (half_gram.cu, DMMA Gram) is used: the non-zero column window of every block is read
        off Q (blocks wider than 8 columns become several segments); `dense=True` forces the older FMA kernel of
        rb.cu (K <= 24), kept as the in-library cross-check."""
        self._need_f64(Xstd, "half_gram"); self._need_f64(Xlin, "half_gram"); self._need_whole_x("half_gram")
        ids = self.to_device(ids, I32); Q = self.to_device(Q, F64)
        cells_h = np.asarray(cells.cpu() if torch.is_tensor(cells) else cells, dtype=np.int32)
        S, nmax, K = int(ids.shape[0]), int(ids.shape[2]), int(Q.shape[3])
        ncell = int(cells_h.shape[1]) - 1
        p = int(Xstd.shape[1])
        S3 = self._empty(S, 3, K, K)
        if dense:
            cells_d = self.to_device(cells_h, I32)
            per = lib.plsb200_half_gram_f64_workspace(p, K, 1)
            ns = max(1, min(S, int(max_ws_bytes // max(per, 1))))
            with torch.cuda.device(self.device):
                ws = self._ws(per * ns)
                for s0 in range(0, S, ns):
                    n = min(ns, S - s0)
                    check(lib.plsb200_half_gram_f64(self._p(Xstd), self._p(Xlin), p, self._p(ids), self._p(Q),
                                                    self._p(cells_d), ncell, int(unit_cells), nmax, K, s0, n,
                                                    self._p(S3), self._p(ws), ws.numel(), self._stream()),
                          "half_gram_f64")
            return S3
        nz = (Q != 0).any(dim=0).cpu().numpy()                      # 2 x nmax x K: columns a position ever feeds
        segs = [[], []]       # (pos_begin, pos_end, col0, width, unit, offset of the packed coefficients in doubles)
        nq = 2
        for h in range(2):
            off = 0
            for c in range(ncell):
                b, e = int(cells_h[h, c]), int(cells_h[h, c + 1])
                cols = np.flatnonzero(nz[h, b:e].any(axis=0)) if e > b else []
                if len(cols) == 0:
                    continue
                for c0 in range(int(cols[0]), int(cols[-1]) + 1, 8):
                    w = min(8, int(cols[-1]) + 1 - c0)
                    wq = 1 if w <= 1 else (2 if w == 2 else (4 if w <= 4 else 8))     # doubles per position
                    segs[h].append((b, e, c0, w, int(c >= ncell - unit_cells), off))
                    off += (e - b) * wq
                    off += off & 1                                                   # 16-byte aligned segments
            nq = max(nq, off)
        nseg = max(len(segs[0]), len(segs[1]), 1)
        table = np.zeros((2, nseg, 6), dtype=np.int32)
        for h in range(2):
            if segs[h]:
                table[h, :len(segs[h])] = np.array(segs[h], dtype=np.int32)
        segs_d = self.to_device(table, I32)
        per = lib.plsb200_half_gram_win_f64_workspace(p, K, 1)
        ns = max(1, min(S, int(max_ws_bytes // max(per, 1))))
        with torch.cuda.device(self.device):
            ws = self._ws(per * ns)
            for s0 in range(0, S, ns):
                n = min(ns, S - s0)
                check(lib.plsb200_half_gram_win_f64(self._p(Xstd), self._p(Xlin), p, self._p(ids), self._p(Q),
                                                    self._p(segs_d), nseg, nq, nmax, K, s0, n, self._p(S3),
                                                    self._p(ws), ws.numel(), self._stream()), "half_gram_win_f64")
        return S3
