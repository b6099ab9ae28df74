#!/usr/bin/env python3
"""Benchmark of the B200 VarDCT decode hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # our CUDA path
  python bench.py --impl reference --gpus N --steps K ...   # CPU arm (oracle port of the jxl-rs CPU path)
  python bench.py --gpus 1 --steps K --dump-outputs DIR     # also write the last step's pixels, to compare two builds

A "step" decodes one batch of synthetic VarDCT frames. Default = BASELINE config 2: 64 frames of 3840x2160 per GPU,
seeds 2000 + rank*frames + i, 1.19 bits per pixel of file (0.94 of them HF sections), mixed transforms, Gaborish on,
EPF iters 2. `--config 3 | 4 | 5` select the other BASELINE configurations (512 x 1080p sharded over the ranks,
one 16384^2 frame with EPF iters 3, 8 x 4096^2 lossless Modular) with the same JSON line. `value` = whole-job MP/s with the parsed frame state and HF bitstreams
already resident in HBM (timed with CUDA events on the launching stream, max over ranks);
`e2e` = the same metric through the public API from HOST .jxl bytes to HOST pixels in pinned
memory (host front-end parse + H2D + kernels + D2H inside the timed region).
Weak scaling: every rank decodes its own batch; no data-path collective (frames are independent).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "vardct_4k_batch_decode_mpixels_per_s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5],
                    help="BASELINE.json configuration: 2 = 64 x 3840x2160 per GPU (default, the metric's own), 3 = 512 x "
                         "1920x1080 sharded over the ranks (strong scaling), 4 = one 16384x16384 frame with EPF iters 3, "
                         "5 = 8 x 4096x4096 lossless Modular")
    ap.add_argument("--frames", type=int, default=None, help="frames per GPU (default: the configuration's)")
    ap.add_argument("--width", type=int, default=None)
    ap.add_argument("--height", type=int, default=None)
    ap.add_argument("--distance", type=float, default=0.5, help="synthetic quantiser knob (0.5 = 1.19 bpp of file at 4K)")
    ap.add_argument("--profile", type=int, default=1, help="transform mix of the synthetic writer")
    ap.add_argument("--epf", type=int, default=None)
    ap.add_argument("--lf-tree", type=int, default=0, choices=[0, 1],
                    help="coding of the LF image in the synthetic frames: 0 = one Gradient leaf per channel (default "
                         "workload), 1 = libjxl-like weighted-predictor tree (3x the host front-end work per frame)")
    ap.add_argument("--unique", type=int, default=0, help="encode only this many distinct frames and repeat them (0 = all distinct)")
    ap.add_argument("--cpu-sample-frames", type=int, default=4)
    ap.add_argument("--inflight", type=int, default=5, help="resident batches alternated by the device-resident loop")
    ap.add_argument("--e2e-depth", type=int, default=5, help="contexts (batches in flight) of the end-to-end leg's PipelinedDecoder")
    ap.add_argument("--chunk", type=int, default=16, help="frames per chunk of the pipelined end-to-end decode")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the pixels the last step decoded (rank 0; a fixed, seeded sample of "
                         "pixel positions, the same in every frame) as float32 DIR/<name>.npy, under 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA path's outputs; --impl reference keeps none")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cfg = {2: (64, 3840, 2160, 2), 3: (max(1, 512 // world), 1920, 1080, 2), 4: (1, 16384, 16384, 3), 5: (8, 4096, 4096, 0)}[args.config]
    args.frames = cfg[0] if args.frames is None else args.frames
    args.width = cfg[1] if args.width is None else args.width
    args.height = cfg[2] if args.height is None else args.height
    args.epf = cfg[3] if args.epf is None else args.epf
    args.scaling = "strong" if args.config == 3 else "weak"
    return args


def frame_seeds(n, rank):
    """Frame i of rank r uses seed 2000 + r*n + i: ranks decode disjoint frames (weak scaling, no collective)."""
    return [2000 + rank * n + i for i in range(n)]


def host_cores():
    """Host threads really available to this process (cgroup CPU quota and affinity included; the GPU boxes of this
    pool expose 128 logical CPUs but grant 16)."""
    from jxl_rs_b200.decoder import effective_cpus
    return effective_cpus()


def rank_cores():
    """This rank's share of the host threads when several ranks run on the node (one process per GPU)."""
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", os.environ.get("WORLD_SIZE", "1")))
    return max(2, host_cores() // max(1, local_world))


def kernel_traffic(kernel, frames):
    """ncu dram__bytes_read + dram__bytes_write of the dominant kernel per launch (profiles/r02_traffic.json, else the
    round-1 capture; taken at 64 frames and scaled linearly to the batch size), or None when no capture exists."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        try:
            t = json.load(open(os.path.join(ROOT, "profiles", name)))[kernel]
            return t["dram_bytes_per_launch"] * frames / t["frames"]
        except Exception:
            continue
    return None


def make_frames(args, rank):
    """Synthetic .jxl byte strings for this rank (outside every timed region)."""
    import synth
    n = args.frames
    uniq = n if args.unique <= 0 else min(args.unique, n)
    seeds = frame_seeds(n, rank)[:uniq]
    workers = max(1, min(uniq, rank_cores()))
    synth.set_threads(max(1, rank_cores() // workers))  # one large image: the writer splits its own loops
    with ThreadPoolExecutor(max_workers=workers) as ex:
        files = list(ex.map(lambda s: synth.encode_synthetic(args.width, args.height, s, args.distance, args.epf, 1, args.profile,
                                                             getattr(args, "lf_tree", 0)), seeds))
    return [files[i % uniq] for i in range(n)]


class ClockSampler:
    """nvidia-smi clock / throttle-reason samples during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1]))
                mx.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def algorithmic_bytes(info_list, width, height, bpp_out=3):
    """BASELINE.md §5: compulsory bytes per frame, each item touched once."""
    total = 0
    xb, yb = (width + 7) // 8, (height + 7) // 8
    for info in info_list:
        total += info.hf_bytes + 12 * xb * yb + 7 * xb * yb + 2 * ((xb + 7) // 8) * ((yb + 7) // 8) + width * height * bpp_out
    return total


_CPU_POOLS = {}


def cpu_decode_batch(files, threads_total):
    """Oracle (CPU port of the jxl-rs path) over a list of files; returns seconds. Frame-parallel first — one worker per
    frame, the way a batch caller of jxl-rs fans out over images — and only the threads left over split a frame's
    groups / row bands (jxl-rs's per-group fan-out, frame/render.rs:461-479)."""
    from jxl_rs_b200 import abi
    from tests import oracle_binding as ob
    lib = ob.load()
    # the port's AVX2 forms of the IDCTs, Gaborish, EPF 1 / 2 and the sRGB store (bit-identical to its scalar definitions,
    # tests/test_cpu_paths.py): the reference runs these stages as SIMD, a scalar stand-in would flatter the GPU by ~3x
    lib.jxo_set_fast_cpu(1)
    par = max(1, min(len(files), threads_total))
    base, extra = divmod(threads_total, par)  # frames i < extra get one thread more
    jobs = [(f, max(1, base + (1 if i < extra else 0))) for i, f in enumerate(files)]
    try:
        ex = _CPU_POOLS.get(par)
        if ex is None:  # workers live across steps: the port keeps its plane buffers per thread
            ex = _CPU_POOLS[par] = ThreadPoolExecutor(max_workers=par)
        t0 = time.perf_counter()
        list(ex.map(lambda job: ob.decode_file(job[0], abi.FORMAT_RGB_U8, threads=job[1]), jobs))
        return time.perf_counter() - t0
    finally:
        lib.jxo_set_fast_cpu(0)  # the checker default


def cpu_sample_size(args, cores):
    """Frames per step of the CPU legs: at least one per granted core (so that no core idles while another frame's row
    bands are being split), at most the batch; one large image (config 4) is one frame for all cores."""
    return max(1, min(args.frames, max(args.cpu_sample_frames, cores)))


DUMP_BYTES = 20 << 20  # per dumped array: two arrays and their pixel index stay under 64 MB


def sample_index(height, width, frames):
    """Row-major pixel positions that --dump-outputs keeps of every frame: all of them when they fit DUMP_BYTES, else a
    sorted sample drawn with a fixed seed, so that every run and every build of the project keeps the same ones."""
    import numpy as np
    k = min(height * width, DUMP_BYTES // (frames * 3 * 4))
    return np.sort(np.random.default_rng(0).choice(height * width, k, replace=False))


def output_sample(outs):
    """float32 (frames, samples, 3): the pixels at sample_index() of one step's H x W x 3 output tensors."""
    import numpy as np
    import torch
    h, w, _ = outs[0].shape
    idx = torch.from_numpy(sample_index(h, w, len(outs))).to(outs[0].device)
    return np.stack([o.reshape(-1, 3)[idx].cpu().numpy() for o in outs]).astype(np.float32)


def write_outputs(out_dir, samples, height, width):
    """samples: name -> output_sample() array; written as out_dir/<name>.npy next to out_dir/pixel_index.npy."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    frames = len(next(iter(samples.values())))
    np.save(os.path.join(out_dir, "pixel_index.npy"), sample_index(height, width, frames).astype(np.float64))
    for name, a in samples.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def workload_text(args, n):
    return (f"batch of {n} synthetic {args.width}x{args.height} VarDCT frames per GPU (BASELINE config {args.config}), "
            f"distance {args.distance}, transform profile {args.profile}, Gaborish on, EPF iters {args.epf}, RGB u8 out")


def run_reference(args, rank, world):
    """CPU arm: the reference is Rust and cannot be built in this image (no cargo), so this times the
    oracle port of the same path (kind="port") with all host threads, on a bounded sample per step."""
    if rank != 0:
        return
    if args.config == 5:
        return run_reference_modular(args)
    cores = host_cores()
    sample = cpu_sample_size(args, cores)
    a2 = argparse.Namespace(**vars(args))
    a2.frames = sample
    a2.unique = 0
    files = make_frames(a2, 0)
    mp = args.width * args.height * sample / 1e6
    for _ in range(max(1, min(args.warmup, 1))):
        cpu_decode_batch(files, cores)
    times = [cpu_decode_batch(files, cores) for _ in range(args.steps)]
    sec = sum(times) / len(times)
    v = mp / sec
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "MP/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_text(args, args.frames) + f"; CPU oracle port (C++ restatement of the jxl-rs CPU path; IDCT / Gaborish / EPF / store in their AVX2 forms, entropy decode and dequantisation scalar), "
                               f"{sample} frames per step decoded frame-parallel on {cores} host threads",
                   "frames_per_step": sample, "same_config": sample == args.frames, "mp_per_s_per_core": v / cores},
        "cpu_baseline": {"value": v, "unit": "MP/s", "cores": cores, "kind": "port", "simd": "AVX2 IDCT / Gaborish / EPF / store forms of the port (bit-identical to its scalar definitions)",
                         "sample": f"{sample} frames of {args.width}x{args.height} per step, {args.steps} steps"},
        "e2e": {"value": v, "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def modular_files(args, rank):
    import synth
    seeds = [500 + rank * args.frames + i for i in range(args.frames)]
    with ThreadPoolExecutor(max_workers=max(1, min(len(seeds), rank_cores()))) as ex:
        return list(ex.map(lambda sd: synth.encode_modular(args.width, args.height, sd, 6, 0, 1), seeds))


def cpu_decode_modular(files, threads):
    from tests import oracle_binding as ob
    ob.load()
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=max(1, min(len(files), threads))) as ex:
        list(ex.map(ob.decode_modular_file, files))
    return time.perf_counter() - t0


def run_reference_modular(args):
    cores = host_cores()
    a2 = argparse.Namespace(**vars(args))
    a2.frames = max(1, min(args.frames, cores))
    files = modular_files(a2, 0)
    cpu_decode_modular(files[:1], 1)
    times = [cpu_decode_modular(files, cores) for _ in range(args.steps)]
    sec = sum(times) / len(times)
    v = args.width * args.height * len(files) / 1e6 / sec
    print(json.dumps({
        "impl": "reference", "metric": "modular_lossless_batch_decode_mpixels_per_s", "value": v, "unit": "MP/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "i32", "data": "synthetic",
        "config": {"workload": f"{len(files)} x {args.width}x{args.height} lossless Modular frames (BASELINE config 5: RCT YCoCg, "
                               "property tree), CPU checker (scalar sub-bitstream decoder), one frame per thread"},
        "cpu_baseline": {"value": v, "unit": "MP/s", "cores": cores, "kind": "port", "simd": "AVX2 IDCT / Gaborish / EPF / store forms of the port (bit-identical to its scalar definitions)", "sample": f"{len(files)} frames per step"},
        "e2e": {"value": v, "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def run_modular(args, rank, world, local_rank, numa):
    """BASELINE config 5: a batch of lossless 8-bit RGB Modular frames per GPU (group size 256, RCT YCoCg, property
    tree), device-resident and end to end (host parse + H2D + kernels + D2H), bit-exact against the source pictures."""
    import numpy as np
    import torch
    import torch.distributed as dist
    import jxl_rs_b200 as j
    import synth
    files = modular_files(args, rank)
    n, W, H = len(files), args.width, args.height
    mp = W * H * n / 1e6
    with ThreadPoolExecutor(max_workers=max(1, min(n, rank_cores()))) as ex:
        frames = list(ex.map(j.ModularParsedFrame, files))
    ctx = j.JxgContext(local_rank)
    dev_out = [torch.empty((H, W, 3), dtype=torch.uint8, device=f"cuda:{local_rank}") for _ in range(n)]
    b = j.ModularBatch(ctx, 2)  # two streams per warp: 7 % faster than one on this workload (profiles/r02q_modular_and_bench.log)
    for fr, o in zip(frames, dev_out):
        b.add(fr, o.data_ptr(), W * 3, True)
    b.run()
    b.wait()
    ok = bool(np.array_equal(dev_out[0].cpu().numpy(), synth.modular_source(W, H, 500 + rank * n)))
    for _ in range(args.warmup):
        b.rerun_device()
        b.wait()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    dev_ms, decode_ms = 0.0, 0.0
    for _ in range(args.steps):
        b.rerun_device()
        b.wait()
        st = b.stats()
        dev_ms += st["device_ms"]  # CUDA events on the launching stream around the whole step
        decode_ms += st["decode_ms"]
    clocks = sampler.stop()
    launches = b.stats()["kernel_launches"]
    b.close()
    dumps = {"device_rgb": output_sample(dev_out)} if args.dump_outputs and rank == 0 else None
    barrier()
    # end to end: bytes -> parse -> batch -> pixels in pinned host memory
    host_out = [torch.empty((H, W, 3), dtype=torch.uint8).pin_memory() for _ in range(n)]

    def e2e_step():
        with ThreadPoolExecutor(max_workers=max(1, min(n, rank_cores()))) as ex:
            frs = list(ex.map(j.ModularParsedFrame, files))
        mb = j.ModularBatch(ctx, 2)  # two streams per warp: 7 % faster than one on this workload (profiles/r02q_modular_and_bench.log)
        try:
            for fr, o in zip(frs, host_out):
                mb.add(fr, o.data_ptr(), W * 3, False)
            mb.run()
            mb.wait()
            return mb.stats()
        finally:
            mb.close()

    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        est = e2e_step()
    torch.cuda.synchronize()
    e2e_sec = time.perf_counter() - t0
    t = torch.tensor([dev_ms, e2e_sec], dtype=torch.float64, device=f"cuda:{local_rank}")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms_max, e2e_sec_max = float(t[0].item()), float(t[1].item())
    ctx.close()
    if dumps is not None:
        dumps["e2e_rgb"] = output_sample(host_out)
        write_outputs(args.dump_outputs, dumps, H, W)
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        sec_bytes = sum(fr.info.hf_bytes for fr in frames)
        alg_bytes = sec_bytes + 3 * W * H * n  # SURVEY §8(d): section bytes + RGB8 output
        ms_per_step = dev_ms_max / args.steps
        value = mp * world / (ms_per_step / 1e3)
        kernel_ms = decode_ms / args.steps
        cores = host_cores()
        sample = files[:max(1, min(n, cores))]
        cpu_sec = cpu_decode_modular(sample, cores)
        cpu_v = W * H * len(sample) / 1e6 / cpu_sec
        print(json.dumps({
            "metric": "modular_lossless_batch_decode_mpixels_per_s", "value": value, "unit": "MP/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "i32", "data": "synthetic",
            "config": {"workload": f"batch of {n} synthetic {W}x{H} lossless Modular frames per GPU (BASELINE config 5: 8-bit RGB, "
                                   "group size 256, RCT YCoCg, property tree, no Squeeze)", "frames_per_gpu": n,
                       "bit_exact_vs_source": ok, "alg_bytes_per_step": alg_bytes, "numa": numa,
                       "l2_policy": "planes of one step (i32, 12 B/px = 1.6 GB) exceed the 126 MB L2; no explicit flush"},
            "roofline": {"bound": "hbm", "kernel": "k_modular_decode", "achieved": alg_bytes / (kernel_ms / 1e3) / 1e9, "peak": peak,
                         "unit": "GB/s", "frac": alg_bytes / (kernel_ms / 1e3) / 1e9 / peak, "traffic": None, "kernel_ms": kernel_ms,
                         "peak_source": "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"},
            "cpu_baseline": {"value": cpu_v, "unit": "MP/s", "cores": cores, "kind": "port", "simd": "AVX2 IDCT / Gaborish / EPF / store forms of the port (bit-identical to its scalar definitions)",
                             "sample": f"{len(sample)} frames, CPU checker, {cpu_sec:.1f} s"},
            "e2e": {"value": mp * world * args.steps / e2e_sec_max, "unit": "MP/s", "h2d_bytes_per_step": est["h2d_bytes"],
                    "d2h_bytes_per_step": est["d2h_bytes"], "ms_per_step": e2e_sec_max / args.steps * 1e3},
            "gpu_launches": int(launches * args.steps), "clocks": clocks}))
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import jxl_rs_b200 as j
    from jxl_rs_b200 import abi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the hot path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    # Threads and pinned buffers of this rank stay on the NUMA node of its GPU (before any pool or pinned tensor exists).
    try:
        numa = j.bind_to_gpu_numa_node(local_rank)
    except Exception as e:  # noqa: BLE001 - a platform without the sysfs entries just runs unbound
        numa = {"numa_node": None, "bound": False, "error": repr(e)}
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if args.config == 5:
        return run_modular(args, rank, world, local_rank, numa)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    files = make_frames(args, rank)
    ctx = j.JxgContext(local_rank)
    n = len(files)
    mp_per_step = args.width * args.height * n / 1e6
    stream = torch.cuda.Stream(device=local_rank)
    sptr = stream.cuda_stream

    # ---------------- device-resident throughput ----------------
    # Two copies of the batch stay resident on two contexts (own CUDA stream + buffer pools each) and the
    # timed steps alternate between them, so that consecutive steps overlap on the device (entropy decode of
    # one batch is latency-bound and leaves issue slots to the transforms/filters of the other).
    with ThreadPoolExecutor(max_workers=min(n, rank_cores())) as ex:
        per_file = max(1, rank_cores() // max(1, len(files)))  # one large image: LF groups in parallel
        frames = list(ex.map(lambda f: j.ParsedFrame(f, per_file), files))
    # resident batches: as asked, but never more than fit the device (pools per batch ~ 48 B per pixel: coefficient lists at
    # worst-case capacity, two XYB plane sets, output, varblock descriptors); config 3 (1.06 GP per batch) gets 3, not 5
    free_b, _total_b = torch.cuda.mem_get_info(local_rank)
    per_batch = 48.0 * args.width * args.height * n + (1 << 30)
    depth = max(1, min(args.inflight, int(0.8 * free_b / per_batch)))
    e2e_cap = depth
    ctxs = [ctx] + [j.JxgContext(local_rank) for _ in range(depth - 1)]
    dev_out = [[torch.empty((fr.height, fr.width, 3), dtype=torch.uint8, device=f"cuda:{local_rank}") for fr in frames]
               for _ in range(depth)]
    batches = []
    for c, outs in zip(ctxs, dev_out):
        b = j.Batch(c, n)
        for fr, o in zip(frames, outs):
            b.add(fr, o.data_ptr(), fr.width * 3, abi.FORMAT_RGB_U8, True)
        b.set_profile(True)
        b.run()
        b.wait()
        batches.append(b)
    batch = batches[0]
    # Every resident batch runs on its own torch stream (JXG_STAGE_STREAMS=1: on the library's two stage streams), so that
    # torch events bracket the kernels on the launching streams.
    staged = os.environ.get("JXG_STAGE_STREAMS", "0") not in ("", "0")
    if staged:
        e_ptr, p_ptr = j.device_streams(local_rank)
        first_stream, last_streams = torch.cuda.ExternalStream(e_ptr), [torch.cuda.ExternalStream(p_ptr)]
        sptrs = [0] * depth
    else:
        streams = [torch.cuda.Stream(device=local_rank) for _ in range(depth)]
        first_stream, last_streams = streams[0], streams
        sptrs = [st_.cuda_stream for st_ in streams]
    for i in range(args.warmup):
        batches[i % depth].rerun_device(sptrs[i % depth])
    for b in batches:
        b.wait()
    # per-stage times of one batch running alone (CUDA events on the launching stream)
    batch.rerun_device(sptrs[0])
    batch.wait()
    stage_acc = batch.stage_times()
    single_ms = batch.stats()["device_ms"]
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev0 = torch.cuda.Event(enable_timing=True)
    ev_end = [torch.cuda.Event(enable_timing=True) for _ in last_streams]
    torch.cuda.synchronize()
    ev0.record(first_stream)  # the device is idle: this is the start of all K steps
    for i in range(args.steps):
        batches[i % depth].rerun_device(sptrs[i % depth])
    for e, st_ in zip(ev_end, last_streams):
        e.record(st_)
    for b in batches:
        b.wait()
    torch.cuda.synchronize()
    dev_ms = max(ev0.elapsed_time(e) for e in ev_end)  # first launch to the last kernel of the last step, device clock
    clocks = sampler.stop()
    st = batch.stats()
    launches_per_step = st["kernel_launches"]
    infos = [fr.info for fr in frames]
    alg_bytes = algorithmic_bytes(infos, args.width, args.height)
    barrier()
    t = torch.tensor([dev_ms], dtype=torch.float64, device=f"cuda:{local_rank}")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms_max = float(t.item())
    for b in batches:
        b.close()
    for c in ctxs[1:]:
        c.close()
    dumps = {"device_rgb": output_sample(dev_out[(args.steps - 1) % depth])} if args.dump_outputs and rank == 0 else None
    del dev_out

    # ---------------- end to end through the public API (host bytes -> host pixels) ----------------
    # K batches stream through PipelinedDecoder (2 contexts): parse + staging of batch k+1 overlap the kernels
    # and D2H copies of batch k; every batch's pixels are in pinned host memory before the clock stops.
    e2e_depth = max(1, min(args.e2e_depth, e2e_cap))  # contexts of the pipelined decoder = host output sets (a set is rewritten only after its batch retired)
    host_out = [[torch.empty((fr.height, fr.width, 3), dtype=torch.uint8).pin_memory() for fr in frames] for _ in range(e2e_depth)]
    outs = [[(o.data_ptr(), fr.width * 3) for o, fr in zip(ho, frames)] for ho in host_out]
    del frames
    ctx.close()
    # A failure of the end-to-end leg must not lose the device-resident measurement (nor dead-lock the other ranks at
    # a barrier): it is reported as e2e.value = null with the error text.
    e2e_err, dec, e2e_sec, h2d, d2h = None, None, float("nan"), 0, 0
    if os.environ.get("JXG_BENCH_SKIP_E2E"):  # sweeps of the device-resident leg only (tools/gpu_sweep.sh)
        e2e_err = RuntimeError("end-to-end leg skipped (JXG_BENCH_SKIP_E2E)")
    try:
        if e2e_err is not None:
            raise e2e_err
        dec = j.PipelinedDecoder(local_rank, depth=e2e_depth, workers=min(64, rank_cores()),
                                 staging_threads=max(2, min(8, rank_cores() // 2)))
        for i in range(e2e_depth + 1):  # every context has sized its pools and pinned arena before the clock starts
            dec.submit(files, outs[i % e2e_depth], abi.FORMAT_RGB_U8)
        dec.drain()
    except Exception as e:  # noqa: BLE001
        e2e_err = e
    barrier()
    if e2e_err is None:
        try:
            t0 = time.perf_counter()
            for i in range(args.steps):
                dec.submit(files, outs[i % e2e_depth], abi.FORMAT_RGB_U8)
            dec.drain()
            torch.cuda.synchronize()
            e2e_sec = time.perf_counter() - t0
            h2d, d2h = dec.last_stats["h2d_bytes"], dec.last_stats["d2h_bytes"]
        except Exception as e:  # noqa: BLE001
            e2e_err = e
    # The host link itself: one plain pinned D2H / H2D copy of a batch's worth of bytes, all ranks at once (they share the
    # host's root complexes and memory). The end-to-end leg cannot be faster than its D2H bytes over this rate.
    link = {"d2h_gbs": None, "h2d_gbs": None}
    try:
        nbytes = sum(o.numel() for o in host_out[0])
        dev_buf = torch.empty(nbytes, dtype=torch.uint8, device=f"cuda:{local_rank}")
        host_buf = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
        for name, dst, src in (("d2h_gbs", host_buf, dev_buf), ("h2d_gbs", dev_buf, host_buf)):
            dst.copy_(src, non_blocking=True)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                dst.copy_(src, non_blocking=True)
            e1.record()
            torch.cuda.synchronize()
            link[name] = 3 * nbytes / (e0.elapsed_time(e1) / 1e3) / 1e9
        del dev_buf, host_buf
    except Exception as e:  # noqa: BLE001
        link["error"] = repr(e)
    barrier()
    t = torch.tensor([0.0 if e2e_err is not None else e2e_sec, 1.0 if e2e_err is not None else 0.0], dtype=torch.float64,
                     device=f"cuda:{local_rank}")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)  # slowest rank; and "did any rank fail"
    e2e_sec_max, any_failed = float(t[0].item()), float(t[1].item()) > 0
    if dec is not None:
        try:
            dec.close()
        except Exception as e:  # noqa: BLE001
            e2e_err = e2e_err or e
    e2e_ok = not any_failed and e2e_sec_max > 0
    if dumps is not None:
        if e2e_ok:
            dumps["e2e_rgb"] = output_sample(host_out[(args.steps - 1) % e2e_depth])
        write_outputs(args.dump_outputs, dumps, args.height, args.width)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"
        ms_per_step = dev_ms_max / args.steps
        value = mp_per_step * world / (ms_per_step / 1e3)
        kernels = {k: v for k, v in stage_acc.items() if k != "memset" and v > 0}
        dom = max(kernels, key=kernels.get) if kernels else None
        dom_ms = kernels.get(dom, 0.0) if dom else 0.0
        achieved = alg_bytes / (dom_ms / 1e3) / 1e9 if dom_ms > 0 else None
        pipeline_gbs = alg_bytes / (ms_per_step / 1e3) / 1e9
        # CPU baseline on a bounded sample (oracle port, all host threads, at least one frame per thread)
        cores = host_cores()
        sample = cpu_sample_size(args, cores)
        cpu_sec = cpu_decode_batch(files[:sample], cores)
        cpu_v = args.width * args.height * sample / 1e6 / cpu_sec
        line = {
            "metric": METRIC, "value": value, "unit": "MP/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {
                "workload": workload_text(args, n) + f" ({sum(len(f) for f in files) * 8 / (args.width * args.height * n):.2f} bits per "
                            f"pixel of file, {sum(i.hf_bytes for i in infos) * 8 / (args.width * args.height * n):.2f} of them HF sections), "
                            "LF image coded with " + ("a libjxl-like weighted-predictor tree" if args.lf_tree else "one Gradient leaf per channel"),
                "frames_per_gpu": n, "unique_frames": args.unique or n,
                "l2_policy": "working set per step (coefficients + XYB planes, >10 GB) far exceeds the 126 MB L2; no explicit flush",
                "sharding": "frames partitioned by rank, no data-path collective",
                "stage_ms_single_batch": stage_acc, "single_batch_ms": single_ms, "batches_in_flight": depth,
                "e2e_pipeline": f"whole batches on {e2e_depth} contexts (host parse / staging of later batches overlaps the kernels and the D2H copies of earlier ones; output copies leave on one first-in-first-out stream)",
                "host_cores": cores, "host_cores_per_rank": rank_cores(), "numa": numa,
                "pipeline_alg_gbs": pipeline_gbs,
                "alg_bytes_per_step": alg_bytes,
            },
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": (achieved / peak) if achieved else None, "traffic": kernel_traffic(dom, n), "peak_source": peak_src,
                         "kernel_ms": dom_ms},
            "cpu_baseline": {"value": cpu_v, "unit": "MP/s", "cores": cores, "kind": "port", "simd": "AVX2 IDCT / Gaborish / EPF / store forms of the port (bit-identical to its scalar definitions)",
                             "sample": f"{sample} frames of {args.width}x{args.height}, oracle port, {cpu_sec:.1f} s"},
            "e2e": ({"value": mp_per_step * world * args.steps / e2e_sec_max, "unit": "MP/s", "h2d_bytes_per_step": h2d,
                     "d2h_bytes_per_step": d2h, "ms_per_step": e2e_sec_max / args.steps * 1e3,
                     "frac_of_device_resident": (mp_per_step * world * args.steps / e2e_sec_max) / value,
                     "host_link_gbs_rank0": link,
                     "link_bound_mp_per_s": (link["d2h_gbs"] * 1e9 / (d2h / mp_per_step / 1e6) / 1e6 * world
                                             if link.get("d2h_gbs") and d2h else None)} if e2e_ok else
                    {"value": None, "unit": "MP/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                     "error": repr(e2e_err) if e2e_err else "end-to-end leg failed on another rank"}),
            "gpu_launches": int(launches_per_step * args.steps),
            "clocks": clocks,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
