"""Host-side mirror of the jxl-rs decoder API for the VarDCT hot path.

Reference shape (jxl/src/api/decoder.rs:33-266, data_types.rs:154, image/output_buffer.rs:26):
    JxlDecoder::process(input, buffers, runner)  ->  pixels in JxlOutputBuffer
Here a *batch* of frames is decoded per call (one crossing of the host/device
boundary per batch, SURVEY §3.5). PyTorch supplies device memory, pinned host
memory and streams only; all compute is in libjxgpu.so.
"""
import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import abi


@dataclass
class JxlPixelFormat:
    """jxl/src/api/data_types.rs:154 (colour part only)."""
    color_type: str = "RGB"          # "RGB" | "RGBA"
    data_format: str = "U8"          # "U8" | "U16" | "F16" | "F32" (JxlDataFormat, 16-bit samples in native endianness)

    def abi_format(self):
        if self.data_format == "U8":
            return abi.FORMAT_RGBA_U8 if self.color_type == "RGBA" else abi.FORMAT_RGB_U8
        if self.color_type == "RGB" and self.data_format in ("F32", "U16", "F16"):
            return {"F32": abi.FORMAT_RGB_F32, "U16": abi.FORMAT_RGB_U16, "F16": abi.FORMAT_RGB_F16}[self.data_format]
        raise ValueError(f"unsupported pixel format {self}")


class ParsedFrame:
    """A .jxl file run through the host front-end (headers, TOC, LfGlobal, LF
    groups, HfGlobal): what a Rust host has in `Frame` when it reaches
    decode_and_render_hf_groups (frame/render.rs:143)."""

    def __init__(self, data: bytes, threads: int = 1):
        """threads > 1: the frame's LF groups are decoded on that many host threads (one large image); batches of
        many frames keep 1 and parse frames in parallel instead."""
        self._lib = abi.load_library()
        self._h = C.c_void_p()
        self.info = abi.JxgImageInfo()
        abi.check(self._lib, self._lib.jxg_parse_file_mt(data, len(data), int(threads), C.byref(self._h),
                                                          C.byref(self.info)))

    @property
    def width(self):
        """Output (display-orientation) width: what the caller's buffer must hold."""
        return self.info.width

    @property
    def height(self):
        return self.info.height

    def desc(self, output_format):
        d = abi.JxgFrameDesc()
        hf, off, ln, n = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_uint32()
        abi.check(self._lib, self._lib.jxg_parsed_desc(self._h, output_format, C.byref(d), C.byref(hf), C.byref(off),
                                                       C.byref(ln), C.byref(n)))
        return d, hf, off, ln, n.value

    def __del__(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.jxg_parsed_free(self._h)
            self._h = C.c_void_p()


class JxgContext:
    """One per GPU / rank (jxg_init)."""

    def __init__(self, device: int = 0):
        self._lib = abi.load_library()
        self._h = C.c_void_p()
        abi.check(self._lib, self._lib.jxg_init(device, C.byref(self._h)))
        self.device = device

    def close(self):
        if self._h.value:
            self._lib.jxg_shutdown(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Batch:
    """jxg_batch_*: frames decoded together by one kernel pipeline."""

    def __init__(self, ctx: JxgContext, n_hint: int = 0, staging_threads: int = 0):
        """staging_threads > 0: large input copies are deferred to run() and done by that many host threads
        (jxg_batch_set_deferred_copy); the ParsedFrames added are kept alive by this object."""
        self._lib = ctx._lib
        self._ctx = ctx
        self._h = C.c_void_p()
        abi.check(self._lib, self._lib.jxg_batch_begin(ctx._h, n_hint, C.byref(self._h)))
        self._keep = []
        self.frames = []
        if staging_threads > 0:
            abi.check(self._lib, self._lib.jxg_batch_set_deferred_copy(self._h, staging_threads))

    def add(self, frame: ParsedFrame, out_ptr: int, row_stride: int, fmt: int, out_is_device: bool):
        abi.check(self._lib, self._lib.jxg_batch_add_parsed(self._h, frame._h, fmt, C.c_void_p(out_ptr), row_stride,
                                                            1 if out_is_device else 0))
        self.frames.append(frame)

    def add_desc(self, desc, hf, off, ln, n, out_ptr, row_stride, out_is_device):
        abi.check(self._lib, self._lib.jxg_batch_add_frame(self._h, C.byref(desc), hf, off, ln, n, C.c_void_p(out_ptr),
                                                           row_stride, 1 if out_is_device else 0))

    def set_debug_stop(self, stage: int):
        abi.check(self._lib, self._lib.jxg_batch_set_debug_stop(self._h, stage))

    STAGES = ["memset", "entropy", "dequant_idct", "gaborish", "epf0", "epf1", "epf2", "xyb_store"]

    def set_profile(self, on: bool):
        abi.check(self._lib, self._lib.jxg_batch_set_profile(self._h, 1 if on else 0))

    def stage_times(self):
        ms = (C.c_float * 8)()
        abi.check(self._lib, self._lib.jxg_batch_stage_times(self._h, ms, 8))
        return dict(zip(self.STAGES, [float(v) for v in ms]))

    def stage_marks(self):
        """Absolute device times (ms) of the 9 stage events of the last run, then of the run's first event (before the
        H2D copy) and its last one (behind the D2H copies) (jxg_batch_stage_marks)."""
        ms = (C.c_float * 11)()
        abi.check(self._lib, self._lib.jxg_batch_stage_marks(self._h, ms, 11))
        return [float(v) for v in ms]

    def run(self, stream_ptr: int = 0):
        abi.check(self._lib, self._lib.jxg_batch_run(self._h, C.c_void_p(stream_ptr)))

    def rerun_device(self, stream_ptr: int = 0):
        abi.check(self._lib, self._lib.jxg_batch_rerun_device(self._h, C.c_void_p(stream_ptr)))

    def wait(self):
        f, g = C.c_uint32(), C.c_uint32()
        abi.check(self._lib, self._lib.jxg_batch_wait(self._h, C.byref(f), C.byref(g)))

    def stats(self):
        k, h, d, ms = C.c_uint64(), C.c_uint64(), C.c_uint64(), C.c_float()
        self._lib.jxg_batch_stats(self._h, C.byref(k), C.byref(h), C.byref(d), C.byref(ms))
        return {"kernel_launches": k.value, "h2d_bytes": h.value, "d2h_bytes": d.value, "device_ms": ms.value}

    def read_coeffs(self, f: int):
        n = self.frames[f].info.num_groups * 3 * 65536
        out = np.empty(n, np.int32)
        abi.check(self._lib, self._lib.jxg_batch_read_coeffs(self._h, f, out.ctypes.data_as(C.c_void_p), n))
        return out.reshape(self.frames[f].info.num_groups, 3, 65536)

    def read_xyb(self, f: int, stage: int):
        w, h = self.frames[f].info.coded_width, self.frames[f].info.coded_height
        ps, pr = (w + 7) // 8 * 8, (h + 7) // 8 * 8
        out = np.empty(3 * ps * pr, np.float32)
        abi.check(self._lib, self._lib.jxg_batch_read_xyb(self._h, f, stage, out.ctypes.data_as(C.c_void_p), out.size))
        return out.reshape(3, pr, ps)

    def close(self):
        if self._h.value:
            if self._ctx._h.value:  # a batch that outlives its context is abandoned, not freed through it
                self._lib.jxg_batch_end(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def decode_files(ctx: JxgContext, files, pixel_format: JxlPixelFormat = JxlPixelFormat(), to_host: bool = True):
    """Decodes a list of .jxl byte strings; returns a list of torch tensors
    (H x W x C). Host results land in pinned memory (JxlOutputBuffer analogue)."""
    import torch
    fmt = pixel_format.abi_format()
    cpus = effective_cpus()
    per_file = max(1, cpus // max(1, len(files)))
    if len(files) > 1:
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(max_workers=min(cpus, len(files))) as ex:
            frames = list(ex.map(lambda f: ParsedFrame(f, per_file), files))
    else:
        frames = [ParsedFrame(f, per_file) for f in files]
    batch = Batch(ctx, len(frames))
    outs = []
    try:  # a corrupt frame must not leave the context with a live batch
        for fr in frames:
            ch = 4 if fmt == abi.FORMAT_RGBA_U8 else 3
            dt = {abi.FORMAT_RGB_F32: torch.float32, abi.FORMAT_RGB_U16: torch.uint16, abi.FORMAT_RGB_F16: torch.float16}.get(fmt, torch.uint8)
            if to_host:
                t = torch.empty((fr.height, fr.width, ch), dtype=dt).pin_memory()
            else:
                t = torch.empty((fr.height, fr.width, ch), dtype=dt, device=f"cuda:{ctx.device}")
            outs.append(t)
            batch.add(fr, t.data_ptr(), fr.width * ch * t.element_size(), fmt, not to_host)
        batch.run()
        batch.wait()
    finally:
        batch.close()
    return outs


def device_streams(device: int = 0):
    """The per-device stage streams (JXG_STAGE_STREAMS) are gone: every batch runs on one stream, its context's or the
    caller's. Callers of the old name get this error instead of an AttributeError."""
    raise abi.JxgError(-2, "the stage-stream mode was removed; batches run on their context's stream or the caller's")


def _parse_cpulist(text):
    cpus = set()
    for part in text.strip().split(","):
        if not part:
            continue
        lo, _, hi = part.partition("-")
        cpus.update(range(int(lo), int(hi or lo) + 1))
    return cpus


def gpu_numa_cpus(device: int, sysfs: str = "/sys"):
    """(numa_node, set of CPUs) of the NUMA node the GPU's PCIe root hangs off, or (None, None) when the platform does
    not say (single-node hosts report -1)."""
    import os
    lib = abi.load_library()
    buf = C.create_string_buffer(32)
    if lib.jxg_device_pci_bus_id(device, buf, 32) != 0:
        return None, None
    try:
        node = int(open(os.path.join(sysfs, "bus/pci/devices", buf.value.decode(), "numa_node")).read())
        if node < 0:
            return None, None
        return node, _parse_cpulist(open(os.path.join(sysfs, f"devices/system/node/node{node}/cpulist")).read())
    except (OSError, ValueError):
        return None, None


def bind_to_gpu_numa_node(device: int):
    """Restricts the calling thread (and every thread it starts afterwards: worker pools, the dispatcher) to the
    CPUs of the GPU's NUMA node. Call it before the pools and the pinned buffers are created: pinned pages are
    allocated on the node of the thread that asks for them, and H2D / D2H copies through a remote node cross the
    inter-socket link (the end-to-end scaling collapse of round 1 at 8 GPUs). Returns a description for logs."""
    import os
    node, cpus = gpu_numa_cpus(device)
    if not cpus:
        return {"numa_node": None, "bound": False}
    try:
        allowed = os.sched_getaffinity(0)
        want = cpus & allowed
        if want:
            os.sched_setaffinity(0, want)
            return {"numa_node": node, "bound": True, "cpus": len(want)}
    except (AttributeError, OSError):
        pass
    return {"numa_node": node, "bound": False}


def effective_cpus() -> int:
    """Host threads this process can really run at once: min(cpu_count, affinity mask, cgroup v2/v1 CPU quota)."""
    import math
    import os
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, math.ceil(int(quota) / int(period))))
    except (OSError, ValueError):
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0 and p > 0:
                n = min(n, max(1, math.ceil(q / p)))
        except (OSError, ValueError):
            pass
    return max(1, n)


class PipelinedDecoder:
    """Streaming decode of many batches. `submit()` only queues a batch: its files start parsing on the worker
    pool at once (so parsing of batch k+1.. overlaps everything else) and a dispatcher thread stages each batch
    (parallel copies into the pinned blob), launches it on one of `depth` contexts (own CUDA stream, staging
    arena and device pools, used round-robin) and retires the oldest one when all contexts are busy. Host
    front-end work of batch k+1 therefore overlaps the kernels and the D2H copies of batch k; the output copies of
    all contexts leave on the device's one first-in-first-out D2H stream, so batches retire in launch order.
    This is the serving-shaped entry point (many independent images in flight). bench.py runs it with depth 5."""

    def __init__(self, device: int = 0, depth: int = 3, workers: int = 0, staging_threads: int = 4, parse_ahead: int = 2):
        import os
        import queue
        import threading
        from collections import deque
        from concurrent.futures import ThreadPoolExecutor
        self.ctxs = [JxgContext(device) for _ in range(depth)]
        self.depth = depth
        self.staging_threads = staging_threads
        self.workers = workers or min(64, effective_cpus())
        self.pool = ThreadPoolExecutor(max_workers=self.workers)
        self.inflight = deque()
        self.k = 0
        self.last_stats = {"h2d_bytes": 0, "d2h_bytes": 0, "kernel_launches": 0}
        self._jobs = queue.Queue()
        self._ahead = threading.Semaphore(depth + parse_ahead)  # bounds parsed-but-not-yet-launched batches
        self._error = None
        self.trace = None  # set to [] to record the dispatcher timeline
        self.retire_trace = []  # with trace on: (start, seconds in wait / stats / close) of every retired batch
        self.marks = None  # set to [] to record the device timeline of every batch (stage event times)
        self.marks_ref_host = None  # time.perf_counter() at the device timeline's zero (set with the first marks)
        self._thread = threading.Thread(target=self._dispatch, daemon=True)
        self._thread.start()

    def _retire(self):
        import time
        b = self.inflight.popleft()
        t0 = time.perf_counter()
        try:
            b.wait()
            t1 = time.perf_counter()
            self.last_stats = b.stats()
            if self.marks is not None:
                tcall = time.perf_counter()
                self.marks.append(b.stage_marks())
                if self.marks_ref_host is None:  # the library's reference event was recorded inside that first call
                    self.marks_ref_host = tcall
        finally:
            t2 = time.perf_counter()
            b.close()
        if self.trace is not None:  # ("retire", start, event wait, stats + marks, close)
            self.retire_trace.append((t0, t1 - t0, t2 - t1, time.perf_counter() - t2))

    def _launch(self, futs, outs, fmt, out_is_device):
        import time
        t0 = time.perf_counter()
        if len(self.inflight) == self.depth:
            self._retire()
        t1 = time.perf_counter()
        ctx = self.ctxs[self.k % self.depth]
        self.k += 1
        b = Batch(ctx, len(futs), self.staging_threads)
        if self.marks is not None:
            b.set_profile(True)
        try:
            frames = [fut.result() for fut in futs]
            t2 = time.perf_counter()
            for fr, (ptr, stride) in zip(frames, outs):
                b.add(fr, ptr, stride, fmt, out_is_device)
            t3 = time.perf_counter()
            b.run()
        except Exception:
            b.close()
            raise
        self.inflight.append(b)
        if self.trace is not None:  # host-side timeline of the dispatcher (seconds): start, retire, parse wait, add, run
            self.trace.append((t0, t1 - t0, t2 - t1, t3 - t2, time.perf_counter() - t3))

    def _dispatch(self):
        while True:
            job = self._jobs.get()
            try:
                if job is None:
                    return
                if isinstance(job, tuple) and job[0] == "drain":
                    try:
                        while self.inflight:
                            self._retire()
                    except Exception as e:  # noqa: BLE001 - reported to the caller of drain()
                        self._error = self._error or e
                    job[1].set()
                    continue
                try:
                    if self._error is None:
                        self._launch(*job)
                except Exception as e:  # noqa: BLE001
                    self._error = self._error or e
                finally:
                    self._ahead.release()
            finally:
                self._jobs.task_done()

    def submit(self, files, outs, fmt: int = abi.FORMAT_RGB_U8, out_is_device: bool = False):
        """files: list of .jxl byte strings; outs: list of (data_ptr, row_stride). Returns once the batch is
        queued; its outputs are complete after drain() (or once `depth` later batches have been launched)."""
        self._ahead.acquire()
        # fewer files than workers (one large image): the spare workers decode LF groups inside each file
        per_file = max(1, self.workers // max(1, len(files)))
        futs = [self.pool.submit(ParsedFrame, f, per_file) for f in files]
        self._jobs.put((futs, list(outs), fmt, out_is_device))

    def drain(self):
        import threading
        ev = threading.Event()
        self._jobs.put(("drain", ev))
        ev.wait()
        if self._error is not None:
            e, self._error = self._error, None
            raise e

    def decode(self, files, outs, fmt: int = abi.FORMAT_RGB_U8, out_is_device: bool = False):
        self.submit(files, outs, fmt, out_is_device)
        self.drain()

    def close(self):
        try:
            self.drain()
        finally:
            self._jobs.put(None)
            self._thread.join()
            self.pool.shutdown()
            for c in self.ctxs:
                c.close()


class ModularParsedFrame:
    """A Modular-encoded .jxl file run through the host front-end (headers, TOC, LfGlobal with the global MA tree,
    section 0, ModularLF streams, group headers): the state a Rust host holds when it reaches the ModularHF groups."""

    def __init__(self, data: bytes):
        self._lib = abi.load_library()
        self._h = C.c_void_p()
        self.info = abi.JxgImageInfo()
        abi.check(self._lib, self._lib.jxg_modular_parse_file(data, len(data), C.byref(self._h), C.byref(self.info)))

    @property
    def width(self):
        return self.info.width

    @property
    def height(self):
        return self.info.height

    def __del__(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.jxg_modular_parsed_free(self._h)
            self._h = C.c_void_p()


class ModularBatch:
    """jxg_modular_batch_*: Modular frames whose group streams are decoded together on the GPU."""

    def __init__(self, ctx: JxgContext, lanes_per_warp: int = 1):
        self._lib = ctx._lib
        self._ctx = ctx
        self._h = C.c_void_p()
        abi.check(self._lib, self._lib.jxg_modular_batch_begin(ctx._h, C.byref(self._h)))
        abi.check(self._lib, self._lib.jxg_modular_batch_set_lanes(self._h, lanes_per_warp))
        self.frames = []

    def add(self, frame: ModularParsedFrame, out_ptr: int, row_stride: int, out_is_device: bool):
        abi.check(self._lib, self._lib.jxg_modular_batch_add(self._h, frame._h, C.c_void_p(out_ptr), row_stride,
                                                             1 if out_is_device else 0))
        self.frames.append(frame)

    def run(self, stream_ptr: int = 0):
        abi.check(self._lib, self._lib.jxg_modular_batch_run(self._h, C.c_void_p(stream_ptr)))

    def rerun_device(self, stream_ptr: int = 0):
        abi.check(self._lib, self._lib.jxg_modular_batch_rerun_device(self._h, C.c_void_p(stream_ptr)))

    def wait(self):
        bf, bg = C.c_uint32(), C.c_uint32()
        abi.check(self._lib, self._lib.jxg_modular_batch_wait(self._h, C.byref(bf), C.byref(bg)))

    def stats(self):
        h2d, d2h, launches = C.c_uint64(), C.c_uint64(), C.c_uint64()
        ms = (C.c_float * 2)()
        abi.check(self._lib, self._lib.jxg_modular_batch_stats(self._h, C.byref(h2d), C.byref(d2h), C.byref(launches), ms))
        return {"h2d_bytes": h2d.value, "d2h_bytes": d2h.value, "kernel_launches": launches.value, "device_ms": ms[0],
                "decode_ms": ms[1]}

    def read_planes(self, f: int):
        import numpy as np
        fr = self.frames[f]
        out = np.zeros((3, fr.info.coded_height, fr.info.coded_width), np.int32)
        abi.check(self._lib, self._lib.jxg_modular_batch_read_planes(self._h, f, out.ctypes.data, out.size))
        return out

    def close(self):
        if self._h and self._h.value:
            if self._ctx._h.value:  # a batch that outlives its context is abandoned, not freed through it
                self._lib.jxg_modular_batch_end(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def decode_modular_files(ctx: JxgContext, files, to_host: bool = True, lanes_per_warp: int = 1):
    """Decodes a list of Modular .jxl byte strings on the GPU; returns H x W x 3 uint8 torch tensors."""
    import torch
    frames = [ModularParsedFrame(f) for f in files]
    batch = ModularBatch(ctx, lanes_per_warp)
    outs = []
    try:
        for fr in frames:
            if to_host:
                t = torch.empty((fr.height, fr.width, 3), dtype=torch.uint8).pin_memory()
            else:
                t = torch.empty((fr.height, fr.width, 3), dtype=torch.uint8, device=f"cuda:{ctx.device}")
            outs.append(t)
            batch.add(fr, t.data_ptr(), fr.width * 3, not to_host)
        batch.run()
        batch.wait()
    finally:
        batch.close()
    return outs
