"""Host <-> device transfers for host matrices (plumbing; the reference has no device boundary, this replaces its
zero-copy ``InRAMDataHandler.fetch``, ``illico/utils/registry.py:97-100``).

Four cases:
  * a large float32 matrix that is mostly zeros (what a dense ``adata.X`` is), in pageable memory -- or in pinned memory
    when this host feeds a single GPU: the staging threads SQUEEZE the row chunks (bit mask + non-zero values,
    ``illico_host_pack_rows_f32``) instead of copying them, an eighth of the bytes crosses PCIe and
    ``illico_unpack_rows_f32`` rebuilds the rows in HBM (:func:`_h2d_2d_packed`; DESIGN.md section 4);
  * pinned source (``torch.Tensor.pin_memory()`` behind the ndarray, or ``cudaHostRegister``-ed memory): one asynchronous
    ``cudaMemcpy2DAsync`` straight from the user's buffer -- also for a column shard ``X[:, lb:ub]`` of a C-order matrix
    (a strided source), which is how the genes are split across GPUs;
  * pageable source (what ``adata.X`` normally is): worker threads copy row chunks into a ring of pinned staging
    buffers (numpy releases the GIL in the copy loop) and enqueue each chunk's ``cudaMemcpyAsync`` on their own stream,
    so that the host-side copies of several threads and the DMA of earlier chunks overlap; the caller keeps working on
    the host meanwhile and joins with :meth:`Pending.finish`;
  * results: each GPU writes its ``results[:, lb:ub, :]`` slab straight into ONE pinned ``[G, N, 3]`` host array with a
    strided device-to-host copy.
"""
from __future__ import annotations

import os
import threading
import warnings

import numpy as np
import torch

from . import _lib

CHUNK_BYTES = int(os.environ.get("ILLICO_STAGE_CHUNK_MB", "32")) << 20
_rings: dict = {}
_rings_lock = threading.Lock()
CONCURRENT_UPLOADS = 1     # GPUs this process is feeding at once (asymptotic_wilcoxon(devices=...) sets it): the cores are shared
LAST_UPLOAD: dict = {}     # the last packed upload: chunks squeezed / sent as they are, bytes that crossed the link


def stage_threads() -> int:
    env = os.environ.get("ILLICO_STAGE_THREADS")
    if env:
        return max(1, int(env))
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", "1") or 1)
    return max(1, min(8, (os.cpu_count() or 8) // max(1, local_world)))


def pack_threads() -> int:
    """Threads that squeeze row chunks for the packed upload: the scan runs at memory speed only with most cores on it
    (8 threads: 0.157 s per K562 upload, 14 of 16 cores: 0.084 s), two are left to the caller and the driver."""
    env = os.environ.get("ILLICO_STAGE_THREADS")
    if env:
        return max(1, int(env))
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", "1") or 1) * max(1, CONCURRENT_UPLOADS)
    return max(1, min(32, ((os.cpu_count() or 8) - 2) // max(1, local_world)))


def is_pinned(a: np.ndarray) -> bool:
    """True when the array's memory is page-locked and known to CUDA (asynchronous DMA is possible from it)."""
    try:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")          # read-only arrays: we only read
            return bool(torch.from_numpy(a[:1] if a.ndim else a.reshape(1)).is_pinned())
    except Exception:
        return False


# ---- NUMA placement ------------------------------------------------------------------------------------------------
def numa_cpus_for_device(index: int):
    """CPUs of the NUMA node the GPU hangs off (sysfs), or None when unknown / single node."""
    try:
        bus = torch.cuda.get_device_properties(index).pci_bus_id
        dev = torch.cuda.get_device_properties(index).pci_device_id
        dom = torch.cuda.get_device_properties(index).pci_domain_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0/numa_node"
        with open(path) as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        return cpus if cpus and cpus != allowed else None
    except Exception:
        return None


def bind_thread_to_device_node(index: int) -> None:
    """Runs the calling thread on the CPUs next to GPU ``index`` (first touch then places its pinned buffers there)."""
    cpus = numa_cpus_for_device(index)
    if cpus:
        try:
            os.sched_setaffinity(0, cpus)
        except Exception:
            pass


# ---- strided copies through the C ABI (cudaMemcpy2DAsync) -------------------------------------------------------------
def copy2d_async(dst_ptr: int, dpitch: int, src_ptr: int, spitch: int, width_bytes: int, height: int, kind: str, stream) -> None:
    lib = _lib.load()
    rc = lib.illico_memcpy2d_async(dst_ptr, dpitch, src_ptr, spitch, width_bytes, height, {"h2d": 1, "d2h": 2, "d2d": 3}[kind],
                                   stream.cuda_stream)
    _lib.check(rc, "illico_memcpy2d_async")


class _Ring:
    """Per (device, thread slot) pinned staging buffers, created once per process (page-locking 32 MB costs ~10 ms)."""

    def __init__(self, device, n_threads):
        self.device = device
        self.bufs = [[None, None] for _ in range(n_threads)]
        self.events = [[None, None] for _ in range(n_threads)]
        self.streams = [None] * n_threads
        self.busy = False

    def slot(self, t, k):
        if self.bufs[t][k] is None or self.bufs[t][k].numel() != CHUNK_BYTES:
            self.bufs[t][k] = torch.empty(CHUNK_BYTES, dtype=torch.uint8, pin_memory=True)
        return self.bufs[t][k]

    def stream(self, t):
        if self.streams[t] is None:
            self.streams[t] = torch.cuda.Stream(device=self.device)
        return self.streams[t]

    def dev_slot(self, t, k):
        """Device-side landing buffer of a packed chunk (same size as the pinned one)."""
        if not hasattr(self, "dev"):
            self.dev = [[None, None] for _ in range(len(self.bufs))]
        if self.dev[t][k] is None or self.dev[t][k].numel() != CHUNK_BYTES:
            self.dev[t][k] = torch.empty(CHUNK_BYTES, dtype=torch.uint8, device=self.device)
        return self.dev[t][k]


def _acquire_ring(device, n_threads) -> _Ring:
    """A free ring of the pool (a new one when every ring is in use: concurrent uploads never share staging buffers)."""
    key = (str(device), n_threads)
    with _rings_lock:
        pool = _rings.setdefault(key, [])
        for r in pool:
            if not r.busy:
                r.busy = True
                return r
        r = _Ring(device, n_threads)
        r.busy = True
        pool.append(r)
        return r


def _release_ring(ring) -> None:
    with _rings_lock:
        ring.busy = False


class Pending:
    """A host-to-device upload in flight.  :meth:`finish` joins the staging threads and makes the current stream of the
    device wait for the copies; until then the destination must not be read."""

    def __init__(self, device, threads=(), events=(), ring=None):
        self.device, self.threads, self.events, self._ring = device, list(threads), list(events), ring
        self.error = None
        self._done = False

    def finish(self):
        if self._done:
            return
        for t in self.threads:
            t.join()
        if self._ring is not None:
            _release_ring(self._ring)      # the buffers' events say when their last DMA is over
            self._ring = None
        self._done = True
        if getattr(self, "stats", None) is not None:
            LAST_UPLOAD.clear()
            LAST_UPLOAD.update(self.stats)
        if self.error is not None:
            raise self.error
        cur = torch.cuda.current_stream(self.device)
        for ev in self.events:
            if ev is not None:
                cur.wait_event(ev)


def h2d_2d(dst: torch.Tensor, src: np.ndarray, n_threads: int | None = None, allow_pack: bool = True) -> Pending:
    """Starts the copy of the 2-D host array ``src`` (any row stride, unit column stride) into the contiguous device
    tensor ``dst`` of the same shape and dtype.  Returns at once; see :class:`Pending`."""
    device = dst.device
    n, b = src.shape
    item = src.dtype.itemsize
    assert dst.is_contiguous() and tuple(dst.shape) == (n, b) and dst.element_size() == item
    if n == 0 or b == 0:
        return Pending(device)
    if src.strides[1] != item or src.strides[0] < 0:
        src = np.ascontiguousarray(src)
    cur = torch.cuda.current_stream(device)
    row_bytes = b * item
    pinned_src = is_pinned(src)
    # A pinned source is squeezed while this host feeds at most FOUR GPUs: plain DMA needs no CPU at all, but the links
    # of 2 / 4 GPUs together carry 111 / 115 GB/s on the measured box and its cores scan ~135 GB/s of raw matrix into an
    # eighth of the bytes (two ranks, each its own K562 matrix: 0.201 -> 0.140 s; one matrix split over two: 0.093 ->
    # 0.075 s); eight links carry 186 GB/s and win.  A pageable source has to be touched by the CPU anyway.
    feeding = int(os.environ.get("LOCAL_WORLD_SIZE", "1") or 1) * max(1, CONCURRENT_UPLOADS)
    if allow_pack and (not pinned_src or feeding <= 4 or os.environ.get("ILLICO_PACK_UPLOAD") == "1") and _pack_wanted(src, n, b):
        return _h2d_2d_packed(dst, src, n_threads)
    if pinned_src:
        if src.strides[0] == b * item:      # contiguous: one linear asynchronous copy
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                dst.copy_(torch.from_numpy(src), non_blocking=True)
        else:                               # a column shard of a wider matrix: strided DMA
            copy2d_async(dst.data_ptr(), b * item, src.__array_interface__["data"][0], src.strides[0], b * item, n, "h2d", cur)
        return Pending(device)
    if n * row_bytes <= (4 << 20) or row_bytes > CHUNK_BYTES:   # small (or absurdly wide rows): the driver's own staged copy
        dst.copy_(torch.from_numpy(np.ascontiguousarray(src)), non_blocking=True)
        return Pending(device)
    T = n_threads or stage_threads()
    rows_per_chunk = max(1, CHUNK_BYTES // row_bytes)
    n_chunks = -(-n // rows_per_chunk)
    T = max(1, min(T, n_chunks))
    ring = _acquire_ring(device, T)
    counter = iter(range(n_chunks))
    counter_lock = threading.Lock()
    pending = Pending(device, ring=ring)
    final_events = [None] * T
    dst_bytes = dst.view(torch.uint8).view(n, row_bytes) if item != 1 else dst.view(n, row_bytes)
    dev_index = device.index if device.index is not None else torch.cuda.current_device()
    start_event = torch.cuda.Event()
    start_event.record(cur)                   # the destination may still be in use by earlier work on this stream

    def worker(t):
        try:
            bind_thread_to_device_node(dev_index)
            with torch.cuda.device(device):
                st = ring.stream(t)
                st.wait_event(start_event)
                k = 0
                while True:
                    with counter_lock:
                        c = next(counter, None)
                    if c is None:
                        break
                    r0 = c * rows_per_chunk
                    r1 = min(n, r0 + rows_per_chunk)
                    ev = ring.events[t][k]
                    if ev is not None:
                        ev.synchronize()          # the DMA out of this staging buffer has finished
                    buf = ring.slot(t, k)
                    view = buf[: (r1 - r0) * row_bytes]
                    hv = view.numpy().view(src.dtype).reshape(r1 - r0, b)
                    np.copyto(hv, src[r0:r1])     # GIL released inside; strided sources are gathered row by row
                    with torch.cuda.stream(st):
                        dst_bytes[r0:r1].copy_(view.view(r1 - r0, row_bytes), non_blocking=True)
                        ev = torch.cuda.Event()
                        ev.record(st)
                    ring.events[t][k] = ev
                    final_events[t] = ev
                    k ^= 1
        except BaseException as e:  # surfaced by finish()
            pending.error = e

    threads = [threading.Thread(target=worker, args=(t,), daemon=True) for t in range(T)]
    pending.threads, pending.events = threads, final_events
    for th in threads:
        th.start()
    return pending


# ---- packed upload (float32, mostly zeros) -----------------------------------------------------------------------------
def _pack_wanted(src: np.ndarray, n: int, b: int) -> bool:
    """A large float32 matrix whose sampled rows are mostly zeros goes up packed (``ILLICO_PACK_UPLOAD``: 0 never,
    1 whenever the layout allows, default: when the sampled density is at most 0.3)."""
    mode = os.environ.get("ILLICO_PACK_UPLOAD", "auto")
    if mode == "0" or src.dtype != np.float32 or b < 64 or n * b * 4 < (64 << 20) or b * 4 > CHUNK_BYTES // 2:
        return False
    if mode == "1":
        return True
    rows = np.linspace(0, n - 1, num=min(n, 48), dtype=np.int64)
    sample = src[rows][:, :: max(1, b // 2048)]                 # at most ~100k elements, spread over the matrix
    return float(np.count_nonzero(sample)) <= 0.3 * sample.size


def _h2d_2d_packed(dst: torch.Tensor, src: np.ndarray, n_threads: int | None) -> Pending:
    """The upload of a mostly-zero float32 matrix with the host threads squeezing the row chunks (bit mask + non-zero
    values, ``illico_host_pack_rows_f32``) instead of copying them: the packed chunk crosses PCIe (about 1/8 of the bytes
    at 10 % density) and ``illico_unpack_rows_f32`` rebuilds the rows in the destination.  The threads share one queue
    of chunks.  (A worker sending chunks of a pinned source as they are, beside the squeeze threads, measured slower on
    the K562 matrix: the squeeze threads slow down ten-fold while plain DMA out of the same pinned pages is running;
    0.17 s against 0.10 s with the threads alone.)"""
    lib = _lib.load()
    device = dst.device
    n, b = src.shape
    W = (b + 31) // 32
    row_bytes = b * 4
    rows_per_chunk = max(1, CHUNK_BYTES // row_bytes)          # a chunk that does not squeeze still fits its buffer
    n_chunks = -(-n // rows_per_chunk)
    T = max(1, min(n_threads or pack_threads(), n_chunks))
    ring = _acquire_ring(device, T)
    counter = iter(range(n_chunks))
    counter_lock = threading.Lock()
    pending = Pending(device, ring=ring)
    final_events = [None] * T
    cur = torch.cuda.current_stream(device)
    dev_index = device.index if device.index is not None else torch.cuda.current_device()
    start_event = torch.cuda.Event()
    start_event.record(cur)
    src_ptr, src_stride = src.__array_interface__["data"][0], src.strides[0]
    hdr_bytes = (rows_per_chunk * W * 4 + (rows_per_chunk + 1) * 4 + 63) & ~63
    vals_cap = (CHUNK_BYTES - hdr_bytes) // 4
    dst_ptr = dst.data_ptr()
    stats = {"packed": 0, "raw": 0, "bytes": 0}
    pending.stats = stats

    def take():
        with counter_lock:
            return next(counter, None)

    def worker(t):
        try:
            bind_thread_to_device_node(dev_index)
            with torch.cuda.device(device):
                st = ring.stream(t)
                st.wait_event(start_event)
                k = 0
                while True:
                    c = take()
                    if c is None:
                        break
                    r0 = c * rows_per_chunk
                    r1 = min(n, r0 + rows_per_chunk)
                    nr = r1 - r0
                    ev = ring.events[t][k]
                    if ev is not None:
                        ev.synchronize()          # the DMA out of this staging buffer has finished
                    buf = ring.slot(t, k)
                    base = buf.data_ptr()
                    off_bytes = nr * W * 4
                    nnz = lib.illico_host_pack_rows_f32(src_ptr + r0 * src_stride, src_stride // 4, nr, b, base, base + off_bytes,
                                                        base + hdr_bytes, vals_cap)      # (ctypes releases the GIL)
                    with torch.cuda.stream(st):
                        if nnz >= 0:
                            used = hdr_bytes + nnz * 4
                            dbuf = ring.dev_slot(t, k)
                            dbuf[:used].copy_(buf[:used], non_blocking=True)
                            d0 = dbuf.data_ptr()
                            _lib.check(lib.illico_unpack_rows_f32(d0, d0 + off_bytes, d0 + hdr_bytes, nr, b, dst_ptr + r0 * row_bytes,
                                                                  b, st.cuda_stream), "illico_unpack_rows_f32")
                            stats["packed"] += 1
                            stats["bytes"] += used
                        else:                     # a dense chunk: as it is
                            hv = buf[: nr * row_bytes].numpy().view(np.float32).reshape(nr, b)
                            np.copyto(hv, src[r0:r1])
                            dst.view(torch.uint8).view(n, row_bytes)[r0:r1].copy_(buf[: nr * row_bytes].view(nr, row_bytes), non_blocking=True)
                            stats["raw"] += 1
                            stats["bytes"] += nr * row_bytes
                        ev = torch.cuda.Event()
                        ev.record(st)
                    ring.events[t][k] = ev
                    final_events[t] = ev
                    # (one staging buffer per thread is enough here: the DMA of a packed chunk -- ~4 MB -- takes a
                    # fortieth of the time the next squeeze does, and page-locking a second 32 MB buffer per thread
                    # would double what the first call pays for the ring)
        except BaseException as e:  # surfaced by finish()
            pending.error = e

    threads = [threading.Thread(target=worker, args=(t,), daemon=True) for t in range(T)]
    pending.threads, pending.events = threads, final_events
    for th in threads:
        th.start()
    return pending


def h2d_1d(dst: torch.Tensor, src: np.ndarray, n_threads: int | None = None) -> Pending:
    """1-D variant (the arrays of a sparse matrix)."""
    src = np.ascontiguousarray(src).reshape(-1)
    n = src.size
    if n == 0:
        return Pending(dst.device)
    width = max(1, min(n, (CHUNK_BYTES // 4) // src.dtype.itemsize))
    rows = n // width
    if rows >= 1 and rows * width == n:
        return h2d_2d(dst.view(rows, width), src.reshape(rows, width), n_threads, allow_pack=False)   # (stored values: nothing to squeeze)
    # ragged tail: body as a 2-D copy, tail directly
    body = rows * width
    p = h2d_2d(dst[:body].view(rows, width), src[:body].reshape(rows, width), n_threads, allow_pack=False) if rows else Pending(dst.device)
    dst[body:].copy_(torch.from_numpy(src[body:]), non_blocking=True)
    return p


def d2h_slab(host: torch.Tensor, dev_slab: torch.Tensor, gene_lb: int, kind: str = "d2h") -> None:
    """Enqueues ``host[:, gene_lb:gene_lb + nb] = dev_slab`` (``host`` pinned ``[G, N, ...]``, ``dev_slab`` contiguous
    ``[G, nb, ...]`` of the same dtype on a GPU; the results ``[G, N, 3]`` or the score plane ``[G, N]``) on the current
    stream of the slab's device: one strided device-to-host copy.  ``kind="d2d"``: ``host`` is a device tensor instead
    (possibly on another GPU)."""
    G, N = host.shape[:2]
    nb = dev_slab.shape[1]
    assert dev_slab.shape[0] == G and dev_slab.shape[2:] == host.shape[2:] and dev_slab.dtype == host.dtype
    assert dev_slab.is_contiguous() and host.is_contiguous()
    if nb == 0:
        return
    rec = host[0, 0].numel() * host.element_size()      # bytes per (group, gene)
    cur = torch.cuda.current_stream(dev_slab.device)
    copy2d_async(host.data_ptr() + gene_lb * rec, N * rec, dev_slab.data_ptr(), nb * rec, nb * rec, G, kind, cur)

