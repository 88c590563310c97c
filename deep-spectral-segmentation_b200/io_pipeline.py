"""Host I/O around the GPU stages (SURVEY 8f rank 2). The reference decodes with 8 DataLoader worker processes
(extract/extract.py:60) and writes one .pth per image synchronously (:113, :244); at the rates the kernels run
(thousands of images per second) both would dominate. Here:

  * ``ImagePrefetcher``  runs ``load(i)`` (a file decode or a ``torch.load``) on a thread pool (cv2 / PIL and file
                          reads release the GIL) with a bounded look-ahead, yielding items in order;
  * ``BatchAssembler``   decode threads colour-swap each image straight into a row of a page-locked batch of its shape
                          and hand over completed batches, so that the host->device copy is asynchronous and no staging
                          copy is made (extract_features, extract_all);
  * ``ProcessWriter``    runs ``torch.save`` (the reference's dict layouts, so ``torch.load`` consumers are unaffected)
                          on writer PROCESSES, fed one message per GPU batch: torch.save is ~0.1-0.4 ms of pure Python per
                          file, and writer threads would take the interpreter lock away from the thread that feeds the GPU
                          (measured: the main thread spent 1.4 ms per image waiting for the lock).

Pure host code: nothing here touches the device."""
from __future__ import annotations

import os
import queue
import threading
from collections import deque
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path
from typing import Callable, Iterator, List, Optional, Sequence

import torch


def available_cpus() -> int:
    """CPUs this process may actually use: the scheduler affinity mask and the cgroup CPU quota (cpu.max of cgroup v2,
    cfs_quota_us of v1), not os.cpu_count(). On the B200 hosts a container sees 128 hardware threads and has a quota of
    16: with 32 decode threads the whole process group was throttled for ~100 ms at a time (cpu.stat nr_throttled), which
    stalled the thread that feeds the GPU as well."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    try:
        quota, period = Path("/sys/fs/cgroup/cpu.max").read_text().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        try:
            quota = int(Path("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read_text())
            period = int(Path("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read_text())
            if quota > 0 and period > 0:
                n = min(n, max(1, quota // period))
        except (OSError, ValueError):
            pass
    return max(1, n)


def default_workers(cap: int = 32, reserve: int = 4) -> int:
    """Decode threads: DSS_IO_DECODE_THREADS, else the usable CPUs minus ``reserve`` (the thread that feeds the GPU and
    the writer processes), at most ``cap``."""
    env = os.environ.get("DSS_IO_DECODE_THREADS")
    if env:
        return max(1, int(env))
    cpus = available_cpus()
    return max(1, min(cap, cpus - reserve if cpus > 2 * reserve else cpus - 1))


_LIMITED = False


def limit_library_threads() -> None:
    """Called before this module starts its own decode threads: OpenCV's internal pool is switched off
    (cv2.setNumThreads(1): every cvtColor / resize would otherwise fan out over a pool sized by os.cpu_count(), 128
    spinning threads on a 16-CPU quota) and torch's intra-op pool is capped at the usable CPUs. The parallelism of the
    host pipeline is the decode threads themselves."""
    global _LIMITED
    if _LIMITED:
        return
    _LIMITED = True
    try:
        import cv2
        cv2.setNumThreads(1)
    except ImportError:
        pass
    cpus = available_cpus()
    if torch.get_num_threads() > cpus:
        torch.set_num_threads(cpus)


class ImagePrefetcher:
    """Iterates ``load(i)`` for i in ``indices`` in order, keeping up to ``lookahead`` loads in flight on a thread pool."""

    def __init__(self, load: Callable[[int], object], indices: Sequence[int], num_workers: Optional[int] = None,
                 lookahead: Optional[int] = None):
        self.load, self.indices = load, list(indices)
        self.num_workers = num_workers if num_workers is not None else default_workers()
        self.lookahead = lookahead if lookahead is not None else 4 * max(1, self.num_workers)

    def __len__(self):
        return len(self.indices)

    def __iter__(self) -> Iterator:
        if self.num_workers <= 0:
            for i in self.indices:
                yield self.load(i)
            return
        limit_library_threads()
        with ThreadPoolExecutor(self.num_workers, thread_name_prefix="dss-decode") as pool:
            pending: deque = deque()
            it = iter(self.indices)
            try:
                for i in it:
                    pending.append(pool.submit(self.load, i))
                    if len(pending) >= self.lookahead:
                        yield pending.popleft().result()
                while pending:
                    yield pending.popleft().result()
            finally:
                for f in pending:
                    f.cancel()


class HostBatch:
    """One page-locked batch being filled by the decode workers (BatchAssembler)."""
    __slots__ = ("key", "slot", "host", "np", "capacity", "items", "assigned", "filled", "closed")

    def __init__(self, key, slot, host, capacity):
        self.key, self.slot, self.host, self.np, self.capacity = key, slot, host, host.numpy(), capacity
        self.items: List[tuple] = []          # (path, dataset index) per row
        self.assigned = self.filled = 0
        self.closed = False


class BatchAssembler:
    """Decode threads that write straight into page-locked batches, grouped by image shape.

    Each worker takes the next dataset index, decodes the file (cv2 releases the interpreter lock), asks for a row of the
    open batch of that image's shape and colour-swaps the pixels directly into that row: no per-image hand-over to the
    consuming thread, no temporary RGB image, no staging copy. The consumer iterates over COMPLETED batches (in
    completion order) and gives each one back with ``release`` once its host->device copy has finished; workers block
    while all ``slots`` batches of a shape are in use, which bounds the page-locked memory.

    ``load(i)`` -> (pixels uint8 [H, W, 3] numpy, is_bgr, path, index). A batch is completed when it is full, when more
    than ``max_pending`` images sit in partly filled batches (the largest one is closed) or when the input is exhausted."""

    def __init__(self, load: Callable, indices: Sequence[int], capacity: int, num_workers: Optional[int] = None,
                 slots: int = 4, full_size_shapes: int = 12, small_capacity: int = 8, max_pending: Optional[int] = None):
        self.load, self.indices = load, list(indices)
        self.capacity, self.slots = max(1, int(capacity)), max(2, int(slots))
        self.num_workers = num_workers if num_workers is not None else default_workers()
        self.full_size_shapes, self.small_capacity = full_size_shapes, small_capacity
        self.max_pending = max_pending if max_pending is not None else 8 * self.capacity
        self._cv = threading.Condition()
        self._it = iter(self.indices)
        self._open = {}            # shape -> HostBatch being filled
        self._rings = {}           # shape -> {"cap": rows, "free": [slot...], "bufs": [tensor...]}
        self._pending = 0          # rows assigned in open batches
        self._ready: "queue.Queue" = queue.Queue()
        self._live = 0
        self._stop = False
        self.alloc_seconds = 0.0
        # summed over the decode threads (seconds): file decode, waiting for a free batch of the image's shape, colour
        # swap into the page-locked row
        self.worker_seconds = {"decode": 0.0, "wait_for_batch": 0.0, "convert": 0.0}
        self.trace: Optional[list] = [] if os.environ.get("DSS_IO_TRACE") else None   # (seconds, event, detail)
        self.threads: List[threading.Thread] = []

    # -- called with self._cv held
    def _close(self, b: HostBatch):
        b.closed = True
        self._open.pop(b.key, None)
        self._pending -= b.assigned
        if self.trace is not None:
            import time as _t
            self.trace.append((_t.perf_counter(), "closed", id(b)))
        if b.filled == b.assigned:
            self._ready.put(b)

    def _assign(self, key, path, index):
        import time as _t
        with self._cv:
            while True:
                if self._stop:
                    raise RuntimeError("BatchAssembler stopped")
                b = self._open.get(key)
                if b is None:
                    ring = self._rings.get(key)
                    if ring is None:
                        cap = self.capacity if len(self._rings) < self.full_size_shapes else min(self.capacity, self.small_capacity)
                        ring = self._rings[key] = {"cap": cap, "free": [], "bufs": []}
                    if not ring["free"] and len(ring["bufs"]) < self.slots:
                        t0 = _t.perf_counter()   # page-locked allocation (torch's caching host allocator): lazily, per slot
                        ring["bufs"].append(torch.empty(ring["cap"], key[0], key[1], 3, dtype=torch.uint8,
                                                        pin_memory=torch.cuda.is_available()))
                        ring["free"].append(len(ring["bufs"]) - 1)
                        self.alloc_seconds += _t.perf_counter() - t0
                    if not ring["free"]:
                        if self.trace is not None:
                            self.trace.append((_t.perf_counter(), "no_free_batch", len(ring["bufs"])))
                        self._cv.wait(0.5)
                        continue
                    slot = ring["free"].pop()
                    b = self._open[key] = HostBatch(key, slot, ring["bufs"][slot], ring["cap"])
                    if self.trace is not None:
                        self.trace.append((_t.perf_counter(), "opened", id(b)))
                row = b.assigned
                b.assigned += 1
                b.items.append((path, index))
                self._pending += 1
                if b.assigned == b.capacity:
                    self._close(b)
                elif self._pending > self.max_pending:
                    self._close(max(self._open.values(), key=lambda g: g.assigned))
                return b, row

    def _worker(self):
        import time as _t
        import numpy as np
        t_dec = t_wait = t_conv = 0.0
        try:
            while True:
                with self._cv:
                    i = next(self._it, None) if not self._stop else None
                if i is None:
                    break
                t0 = _t.perf_counter()
                pixels, is_bgr, path, index = self.load(i)
                t1 = _t.perf_counter()
                b, row = self._assign((int(pixels.shape[0]), int(pixels.shape[1])), path, index)
                t2 = _t.perf_counter()
                t_dec += t1 - t0
                t_wait += t2 - t1
                dst = b.np[row]
                if is_bgr:
                    import cv2
                    out = cv2.cvtColor(pixels, cv2.COLOR_BGR2RGB, dst=dst)
                    if out is not dst and not np.shares_memory(out, dst):   # cv2 reallocates when dst does not fit
                        np.copyto(dst, out)
                else:
                    np.copyto(dst, pixels)
                t_conv += _t.perf_counter() - t2
                with self._cv:
                    b.filled += 1
                    if b.closed and b.filled == b.assigned:
                        if self.trace is not None:
                            self.trace.append((_t.perf_counter(), "ready", id(b)))
                        self._ready.put(b)
        except BaseException as e:  # noqa: BLE001  (re-raised by the consumer)
            self._ready.put(e)
        finally:
            with self._cv:
                self.worker_seconds["decode"] += t_dec
                self.worker_seconds["wait_for_batch"] += t_wait
                self.worker_seconds["convert"] += t_conv
                self._live -= 1
                if self._live == 0:     # input exhausted and every row written: hand over the partly filled batches
                    for b in list(self._open.values()):
                        self._close(b)

    def __iter__(self) -> Iterator[HostBatch]:
        total = len(self.indices)
        if total == 0:
            return
        limit_library_threads()
        n = max(1, min(self.num_workers, total))
        self._live = n
        self.threads = [threading.Thread(target=self._worker, name=f"dss-decode-{t}", daemon=True) for t in range(n)]
        import time as _t
        if self.trace is not None:
            self.trace.append((_t.perf_counter(), "starting_threads", n))
        for t in self.threads:
            t.start()
        if self.trace is not None:
            self.trace.append((_t.perf_counter(), "threads_started", n))
        got = 0
        try:
            while got < total:
                b = self._ready.get()
                if isinstance(b, BaseException):
                    raise b
                got += b.assigned
                if self.trace is not None:
                    self.trace.append((_t.perf_counter(), "consumer_got", id(b)))
                yield b
        finally:
            with self._cv:
                self._stop = True
                self._cv.notify_all()
            for t in self.threads:
                t.join(timeout=10)

    def release(self, b: HostBatch) -> None:
        """The consumer is done with the batch's page-locked memory (its host->device copy has completed)."""
        with self._cv:
            self._rings[b.key]["free"].append(b.slot)
            if self.trace is not None:
                import time as _t
                self.trace.append((_t.perf_counter(), "released", id(b)))
            self._cv.notify_all()


# ---------------------------------------------------------------------------------------------------------------
def _materialise(arrays, j, extra, fields) -> dict:
    """The dict of one writer item: ``extra`` plus, for each key of ``fields``, row j of an array of ``arrays`` (see
    ProcessWriter) or a 0-d tensor."""
    import numpy as np
    obj = dict(extra)
    for key, (how, val) in fields.items():
        if how == "slice":            # tensor arrays[val][j]
            obj[key] = torch.from_numpy(np.array(arrays[val][j]))
        elif how == "slice1":         # tensor arrays[val][j:j+1] (keeps the leading batch dimension of 1)
            obj[key] = torch.from_numpy(np.array(arrays[val][j:j + 1]))
        elif how == "np_slice":       # numpy array arrays[val][j]
            obj[key] = np.array(arrays[val][j])
        elif how == "tensor0d":       # 0-d int64 tensor
            obj[key] = torch.tensor(int(val))
        else:
            raise ValueError(how)
    return obj


def save_item(arrays, item) -> None:
    """torch.save of one writer item (path, row j, extra, fields) to a temporary file that is then renamed to ``path``:
    a crash never leaves a truncated file for skip-if-exists to trust. The directory must exist."""
    path, j, extra, fields = item
    tmp = f"{path}.tmp{os.getpid()}"
    torch.save(_materialise(arrays, j, extra, fields), tmp)
    os.replace(tmp, path)


def _writer_process_main(q, errq, doneq):
    torch.set_num_threads(1)
    try:
        while True:
            msg = q.get()
            if msg is None:
                return
            arrays, items = msg
            made = set()
            for item in items:
                parent = os.path.dirname(item[0])
                if parent not in made:      # one mkdir per directory and message, not per file
                    os.makedirs(parent, exist_ok=True)
                    made.add(parent)
                save_item(arrays, item)
            doneq.put(len(items))
    except BaseException as e:  # noqa: BLE001
        import traceback
        errq.put(f"{e!r}\n{traceback.format_exc()}")


class ProcessWriter:
    """Writer processes for the per-image .pth files. ``submit_batch(arrays, items)``: ``arrays`` maps names to numpy
    arrays with a leading batch dimension (sent once per batch), ``items`` is a list of (path, row j, extra dict, fields)
    where fields maps dict keys to ("slice" | "slice1" | "np_slice", array name) or ("tensor0d", int); the worker builds
    each dict and torch.saves it. Started with the 'spawn' method (no fork of a process that holds a CUDA context and
    running threads). Importing torch in the children takes a second or two, so the pool is PERSISTENT: make_writer()
    hands out the same processes to every command of this interpreter; leaving its ``with`` block only waits until
    everything that was submitted has been written (``flush``)."""

    def __init__(self, num_procs: int = 4, max_pending: int = 16):
        import multiprocessing as mp
        ctx = mp.get_context("spawn")
        self.q = ctx.Queue(max_pending)
        self.errq = ctx.Queue()
        self.doneq = ctx.Queue()
        self.procs = [ctx.Process(target=_writer_process_main, args=(self.q, self.errq, self.doneq), daemon=True)
                      for _ in range(max(1, num_procs))]
        for p_ in self.procs:
            p_.start()
        self.submitted = 0
        self.done = 0

    def _check(self):
        if not self.errq.empty():
            raise RuntimeError("writer process failed: " + self.errq.get())
        if any(not p_.is_alive() for p_ in self.procs):
            raise RuntimeError("a writer process died")

    def submit_batch(self, arrays, items) -> None:
        self._check()
        n = len(self.procs)
        # split the batch over the writers in contiguous row ranges; each message carries only its rows of the arrays
        rows = sorted(it_[1] for it_ in items)
        per = -(-len(rows) // n)
        for w in range(n):
            sel = rows[w * per:(w + 1) * per]
            if not sel:
                continue
            lo, hi = sel[0], sel[-1] + 1
            part = [(path, j - lo, extra, fields) for path, j, extra, fields in items if lo <= j < hi]
            self.q.put(({name: a[lo:hi] for name, a in arrays.items()}, part))
            self.submitted += len(part)

    def flush(self, timeout: float = 600.0) -> int:
        import queue as _q
        import time as _t
        t0 = _t.monotonic()
        while self.done < self.submitted:
            try:
                self.done += self.doneq.get(timeout=0.5)
            except _q.Empty:
                self._check()
                if _t.monotonic() - t0 > timeout:
                    raise RuntimeError("writer processes did not finish in time")
        self._check()
        return self.done

    def shutdown(self):
        for _ in self.procs:
            self.q.put(None)
        for p_ in self.procs:
            p_.join(timeout=10)

    def __enter__(self):
        return self

    def __exit__(self, exc_type, exc, tb):
        if exc_type is None:
            self.flush()
        return False


_WRITER_POOL = {}


def make_writer(workers: int = 4) -> ProcessWriter:
    """The persistent ProcessWriter with ``workers`` processes (started on first use, restarted if one has died)."""
    pool = _WRITER_POOL.get(workers)
    if pool is None or any(not p_.is_alive() for p_ in pool.procs):
        pool = _WRITER_POOL[workers] = ProcessWriter(workers)
    return pool
