"""Fake device layer for dry runs of bench.py on the CPU (tests/test_bench_dry_run.py and its two-rank driver)."""
import ctypes


class _FakeEvent:
    def __init__(self, enable_timing=False):
        pass

    def record(self, stream=None):
        pass

    def elapsed_time(self, other):
        return 1.0


class _FakeStream:
    cuda_stream = 0

    def __init__(self, device=None):
        pass


def install(setattr_fn, fail_e2e=False, gloo=False):
    """setattr_fn(obj, name, value): monkeypatch.setattr in pytest, plain setattr in a driver script."""
    import torch
    import bench
    from jxl_rs_b200 import decoder
    import jxl_rs_b200 as j

    setattr_fn(torch.cuda, "is_available", lambda: True)
    setattr_fn(torch.cuda, "set_device", lambda d: None)
    setattr_fn(torch.cuda, "synchronize", lambda *a, **k: None)
    setattr_fn(torch.cuda, "Stream", _FakeStream)
    setattr_fn(torch.cuda, "Event", _FakeEvent)
    setattr_fn(torch.cuda, "ExternalStream", lambda ptr, *a, **k: _FakeStream())
    for mod in (decoder, j):
        setattr_fn(mod, "device_streams", lambda device=0: (1, 2))
    setattr_fn(torch.cuda, "current_stream", lambda *a, **k: _FakeStream())
    setattr_fn(torch.cuda, "mem_get_info", lambda *a, **k: (150 << 30, 180 << 30))
    real_empty, real_tensor = torch.empty, torch.tensor
    setattr_fn(torch, "empty", lambda *a, **k: real_empty(*a, **{x: y for x, y in k.items() if x != "device"}))
    setattr_fn(torch, "tensor", lambda *a, **k: real_tensor(*a, **{x: y for x, y in k.items() if x != "device"}))
    setattr_fn(torch.Tensor, "pin_memory", lambda self: self)

    class FakeCtx:
        def __init__(self, device=0):
            self.device = device

        def close(self):
            pass

    class FakeBatch:
        """Every run fills the batch's outputs with its running count (runs: n, reruns: 100 + n), so that a dump shows
        which step wrote it."""
        runs = 0
        reruns = 0

        def __init__(self, ctx, n=0, staging_threads=0):
            self.n = 0
            self.outs = []

        def add(self, fr, ptr, stride, fmt, out_is_device):
            assert fr.width > 0 and ptr != 0 and stride >= fr.width * 3
            self.n += 1
            self.outs.append((ptr, stride * fr.height))

        def _fill(self, value):
            for ptr, nbytes in self.outs:
                ctypes.memset(ptr, value & 0xff, nbytes)

        def set_profile(self, on):
            pass

        def run(self, stream_ptr=0):
            FakeBatch.runs += 1
            if fail_e2e and FakeBatch.runs > 6:  # the device-resident leg runs --inflight (5) batches once; later runs belong to the end-to-end leg
                raise RuntimeError("injected failure of the end-to-end leg")
            self._fill(FakeBatch.runs)

        def rerun_device(self, stream_ptr=0):
            FakeBatch.reruns += 1
            self._fill(100 + FakeBatch.reruns)

        def wait(self):
            pass

        def stage_times(self):
            return {"memset": 0.1, "entropy": 3.0, "dequant_idct": 1.0, "epf2": 1.2}

        def stats(self):
            return {"h2d_bytes": 1000, "d2h_bytes": 2000, "kernel_launches": 7, "device_ms": 5.5}

        def close(self):
            pass

    for mod in (decoder, j):
        setattr_fn(mod, "JxgContext", FakeCtx)
        setattr_fn(mod, "Batch", FakeBatch)
    setattr_fn(bench.ClockSampler, "start", lambda self: None)
    if gloo:  # multi-rank dry run: same collectives over gloo with CPU tensors
        import torch.distributed as dist
        real_init = dist.init_process_group
        setattr_fn(dist, "init_process_group", lambda backend, **kw: real_init("gloo"))
    return bench


