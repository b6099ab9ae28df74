"""CPU-only checks: oracle self-verification on the reference's real bitstreams, synthetic writer round trips,
the C-ABI library surface, and the frame-sharding logic under a world_size-2 gloo group."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from jxl_rs_b200 import abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REAL = ["zoltan_tasi_unsplash.jxl", "green_queen_vardct_e3.jxl", "progressive_ac.jxl", "has_permutation.jxl",         "opsin_inverse.jxl", "3x3_srgb_lossy.jxl", "basic.jxl", "lossy_with_icc.jxl", "grayscale.jxl"]


def _cuda_device_visible():
    """Whether jxg_init can find a device: asked of the CUDA runtime, since a machine may expose its GPU under any
    /dev/nvidia<N> node, not necessarily nvidia0."""
    import torch
    return torch.cuda.is_available()


@pytest.mark.parametrize("name", REAL)
def test_oracle_self_verifies_on_reference_fixtures(golden_dir, name):
    """Every ANS stream must end in state 0x130000, every block must consume exactly its non-zero count and no section
    may be over-read (ans.rs:441, group.rs:574, bit_reader.rs:109): the decode returns 0 only then."""
    from tests import oracle_binding as ob
    data = open(os.path.join(golden_dir, "jxl", name), "rb").read()
    out, taps = ob.decode_file(data, abi.FORMAT_RGB_U8, taps=True, threads=4)
    assert out.shape[2] == 3 and np.isfinite(taps["xyb_filtered"]).all()


ALPHA = ["3x3a_srgb_lossy.jxl", "alpha_premultiplied.jxl", "dice.jxl", "squeeze_alpha.jxl", "upsampled_alpha.jxl"]


@pytest.mark.parametrize("name", ALPHA)
def test_vardct_frames_with_extra_channels_decode_their_colour(golden_dir, name):
    """Extra channels (alpha) are Modular sub-bitstreams around the colour data (modular/mod.rs:258-400); the front-end
    steps over them (LfGlobal section 0, ModularLF per LF group) and the hot path decodes the colour channels — the
    reference's "extra channel not requested" output. Everything behind a skipped stream (HF metadata, HfGlobal, the
    AC streams) only self-verifies if the skip ended on the right bit."""
    from tests import oracle_binding as ob
    data = open(os.path.join(golden_dir, "jxl", name), "rb").read()
    out, taps = ob.decode_file(data, abi.FORMAT_RGB_U8, taps=True, threads=4)
    assert out.shape[2] == 3 and np.isfinite(taps["xyb_filtered"]).all()
    if name == "3x3a_srgb_lossy.jxl":  # the same nine pixels as the file without alpha
        plain = open(os.path.join(golden_dir, "jxl", "3x3_srgb_lossy.jxl"), "rb").read()
        assert np.array_equal(out, ob.decode_file(plain, abi.FORMAT_RGB_U8)[0])
    # truncating inside the skipped data must be reported, not read past
    assert ob.load().jxo_t_parse_ok(data[: len(data) // 3], len(data) // 3) != 0


def test_oracle_detects_corruption(golden_dir):
    from tests import oracle_binding as ob
    data = bytearray(open(os.path.join(golden_dir, "jxl", "green_queen_vardct_e3.jxl"), "rb").read())
    for i in range(len(data) - 3000, len(data) - 2000):
        data[i] ^= 0x5A
    with pytest.raises(abi.JxgError):
        ob.decode_file(bytes(data))


def _srgb_exact(x):
    return np.where(x < 0.0031308, 12.92 * x, 1.055 * np.power(np.maximum(x, 1e-9), 1 / 2.4) - 0.055)


@pytest.mark.parametrize("case", [(8, 8, 1, 1.0, 2, 1, 0, 0), (256, 256, 1000, 0.5, 2, 1, 1, 0), (300, 200, 7, 0.5, 3, 0, 2, 0),
                                  (640, 480, 9, 0.3, 0, 1, 1, 0), (512, 512, 77, 0.5, 0, 0, 3, 0), (600, 520, 78, 0.5, 2, 1, 3, 1),
                                  (400, 300, 79, 0.5, 2, 1, 1, 1)])
def test_synthetic_writer_round_trip(case):
    """The writer's forward transforms / entropy coder and the oracle's decoder were written independently:
    a decode that reproduces the source image (PSNR) pins the transform conventions end to end."""
    import synth
    from tests import oracle_binding as ob
    w, h, seed, dist, epf, gab, prof, ent = case
    data = synth.encode_synthetic(w, h, seed, dist, epf, gab, prof, 0, ent)
    out, _ = ob.decode_file(data, abi.FORMAT_RGB_F32, threads=4)
    assert out.shape == (h, w, 3) and np.isfinite(out).all()
    assert 0.0 < out.mean() < 1.0 and out.std() > 0.01
    assert ob.file_info(data).width == w
    # the source picture of the writer (linear RGB, 8-bit rendering) against the decode (sRGB-encoded float)
    src = _srgb_exact(synth.modular_source(w, h, seed) / 255.0)
    mse = float(np.mean((out.astype(np.float64) - src) ** 2))
    assert 10 * np.log10(1.0 / mse) > (24.0 if w <= 8 else 30.0), f"PSNR {10 * np.log10(1.0 / mse):.1f} dB"


def test_orientation_is_applied_like_the_reference_save_stage():
    """headers/image_metadata.rs:85-96 display_pixel, written here as numpy flips / transposes of the identity decode."""
    import synth
    from tests import oracle_binding as ob
    base, _ = ob.decode_file(synth.encode_synthetic(200, 120, 5, 0.5, 2, 1, 1), abi.FORMAT_RGB_U8)
    want = {1: base, 2: base[:, ::-1], 3: base[::-1, ::-1], 4: base[::-1], 5: base.transpose(1, 0, 2),
            6: np.rot90(base, k=-1), 7: base.transpose(1, 0, 2)[::-1, ::-1], 8: np.rot90(base, k=1)}
    for o in range(1, 9):
        data = synth.encode_synthetic(200, 120, 5, 0.5, 2, 1, 1, orientation=o)
        info = ob.file_info(data)
        assert (info.coded_width, info.coded_height, info.orientation) == (200, 120, o)
        assert (info.width, info.height) == ((120, 200) if o >= 5 else (200, 120))
        out, _ = ob.decode_file(data, abi.FORMAT_RGB_U8)
        assert np.array_equal(out, want[o]), f"orientation {o}"


def test_scope_guards_refuse_what_the_path_cannot_reproduce(golden_dir):
    """A frame the path cannot render like the reference must be refused (JXG_ERR_UNSUPPORTED), never decoded to
    different pixels: noise synthesis (render/stages/noise.rs), multi-frame files, absurd dimensions."""
    from tests import oracle_binding as ob
    lib = abi.load_library()
    data = open(os.path.join(golden_dir, "jxl", "noise.jxl"), "rb").read()
    h, info = C.c_void_p(), abi.JxgImageInfo()
    assert lib.jxg_parse_file(data, len(data), C.byref(h), C.byref(info)) == -2
    assert b"noise" in lib.jxg_last_error()
    with pytest.raises(abi.JxgError) as e:
        ob.decode_file(data)
    assert e.value.code == -2


def test_entropy_variants_of_the_writer_decode_identically():
    """The same quantised frame coded four ways — ANS, prefix codes, and both with LZ77 copies — is the same picture."""
    import synth
    from tests import oracle_binding as ob
    outs = [ob.decode_file(synth.encode_synthetic(600, 400, 5, 0.5, 2, 1, 1, 0, ent), abi.FORMAT_RGB_U8)[0] for ent in range(4)]
    for o in outs[1:]:
        assert np.array_equal(o, outs[0])
    lz = _frame_census(synth.encode_synthetic(600, 400, 5, 0.5, 2, 1, 1, 0, 2))
    assert lz["lz77"] == 1


def _frame_census(data):
    """Transform types used by first blocks and the entropy code of pass 0, from the descriptor the front-end hands
    to the hot path (no GPU involved)."""
    import jxl_rs_b200 as j
    fr = j.ParsedFrame(data)
    d, _, _, _, _ = fr.desc(abi.FORMAT_RGB_U8)
    nb = ((fr.info.coded_width + 7) // 8) * ((fr.info.coded_height + 7) // 8)
    tm = np.ctypeslib.as_array(C.cast(d.transform_map, C.POINTER(C.c_uint8)), (nb,)).copy()
    types = np.bincount(tm[tm >= 128] & 127, minlength=27)
    p0 = d.passes[0]
    census = {"types": types, "use_prefix": int(p0.use_prefix), "clusters": int(p0.num_clusters), "lz77": int(p0.lz77_enabled)}
    if p0.use_prefix:
        e = np.ctypeslib.as_array(C.cast(p0.huff_entries, C.POINTER(C.c_uint32)), (p0.huff_entries_len,)).copy()
        off = np.ctypeslib.as_array(C.cast(p0.huff_offset, C.POINTER(C.c_uint32)), (p0.num_clusters,)).copy()
        roots = np.concatenate([e[o:o + 256] for o in off])
        census["second_level_roots"] = int(((roots & 0xff) > 8).sum())
    return census


def test_profile_3_places_the_128_and_256_transform_families():
    """SURVEY §8 a11: DCT128X128 ... DCT256X256 (types 21..26) must all occur in the frame the parity tests use."""
    import synth
    c = _frame_census(synth.encode_synthetic(1024, 768, 31, 0.5, 2, 1, 3))
    assert all(c["types"][t] > 0 for t in range(21, 27)), c["types"]
    assert c["types"][18] > 0 and c["types"][5] > 0 and c["types"][0] > 0  # and the smaller families around them


def test_prefix_variant_exercises_the_second_level_tables():
    """SURVEY §8 a6: prefix-coded AC streams with codes longer than the 8-bit root table (huffman.rs:446-457) and many
    clusters — not the 1x1 / one-cluster prefix files of the reference's fixture set."""
    import synth
    c = _frame_census(synth.encode_synthetic(1024, 768, 32, 0.5, 2, 1, 1, 0, 1))
    assert c["use_prefix"] == 1 and c["clusters"] >= 16 and c["second_level_roots"] > 0, c


def test_c_abi_exports_every_declared_symbol():
    """libjxgpu.so loads without a GPU and exports every function include/jxg.h declares (no compute calls here)."""
    lib = abi.load_library()
    header = open(os.path.join(ROOT, "include", "jxg.h")).read()
    declared = set(re.findall(r"\b(jxg_[a-z0-9_]+)\s*\(", header))
    assert declared == set(abi.EXPORTS), declared ^ set(abi.EXPORTS)
    for sym in declared:
        assert hasattr(lib, sym), sym
    if not _cuda_device_visible():
        h = C.c_void_p()
        assert lib.jxg_init(0, C.byref(h)) == -21  # JXG_ERR_NO_DEVICE: no CPU fallback
        assert b"no CPU fallback" in lib.jxg_last_error()


def test_header_is_plain_c_and_links_from_c(tmp_path):
    """include/jxg.h is the boundary a Rust / C host binds: it must compile as C99 (no C++ in the signatures) and a C program
    must link against libjxgpu.so and reach an entry point (jxg_init without a GPU returns JXG_ERR_NO_DEVICE)."""
    src = tmp_path / "abi.c"
    src.write_text('#include <stdio.h>\n#include "jxg.h"\n'
                   'int main(void) { void* ctx = 0; int r = jxg_init(0, &ctx); printf("%d %d\\n", JXG_ABI_VERSION, r);'
                   ' if (r == 0) jxg_shutdown(ctx); return 0; }\n')
    exe = tmp_path / "abi"
    libdir = os.path.dirname(abi.library_path())
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"), str(src),
                    "-o", str(exe), "-L", libdir, "-ljxgpu", "-Wl,-rpath," + libdir], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()
    assert int(out[0]) == abi.JXG_ABI_VERSION
    assert int(out[1]) == (0 if _cuda_device_visible() else -21)


def test_c_example_builds_and_fails_loudly_without_a_gpu(tmp_path, golden_dir):
    """examples/decode_files.c (the C host of the file front-end) compiles as pedantic C99, links, and on a box without a
    GPU stops at jxg_init with the library's own message - there is no CPU decode behind the ABI. With a GPU it decodes the
    file to <file>.ppm."""
    import shutil
    exe = tmp_path / "decode_files"
    libdir = os.path.dirname(abi.library_path())
    subprocess.run(["gcc", "-std=c99", "-O1", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "examples", "decode_files.c"), "-o", str(exe), "-L", libdir, "-ljxgpu",
                    "-Wl,-rpath," + libdir], check=True)
    src = tmp_path / "3x3_srgb_lossy.jxl"  # the example writes its output next to its input
    shutil.copy(os.path.join(golden_dir, "jxl", src.name), src)
    r = subprocess.run([str(exe), str(src)], capture_output=True, text=True)
    if not _cuda_device_visible():
        assert r.returncode == 1 and "no CPU fallback" in r.stderr
    else:
        assert r.returncode == 0, r.stderr
        assert (tmp_path / (src.name + ".ppm")).read_bytes().startswith(b"P6\n3 3\n255\n")


def test_product_does_not_touch_the_oracle():
    """Nothing under jxl_rs_b200/ may import, link or execute oracle/."""
    for dirpath, _, files in os.walk(os.path.join(ROOT, "jxl_rs_b200")):
        for f in files:
            if f.endswith((".py", ".cc", ".cu", ".h", "Makefile")):
                txt = open(os.path.join(dirpath, f), errors="replace").read()
                assert "oracle" not in txt.lower() or "test_product" in f, os.path.join(dirpath, f)
    out = subprocess.run(["ldd", abi.library_path()], capture_output=True, text=True).stdout
    assert "oracle" not in out


def test_frame_sharding_world_size_2_gloo(tmp_path):
    """The multi-GPU path partitions whole frames by rank with no data-path collective; this runs the partition +
    max-over-ranks reduction of bench.py under a 2-process gloo group."""
    script = tmp_path / "shard.py"
    script.write_text(
        "import os, sys, torch, torch.distributed as dist\n"
        f"sys.path.insert(0, {ROOT!r})\n"
        "import bench, argparse\n"
        "dist.init_process_group('gloo')\n"
        "r, w = dist.get_rank(), dist.get_world_size()\n"
        "seeds = bench.frame_seeds(8, r)\n"
        "all_seeds = [None] * w\n"
        "dist.all_gather_object(all_seeds, seeds)\n"
        "flat = sum(all_seeds, [])\n"
        "assert len(set(flat)) == 8 * w, flat\n"
        "t = torch.tensor([10.0 + r], dtype=torch.float64)\n"
        "dist.all_reduce(t, op=dist.ReduceOp.MAX)\n"
        "assert t.item() == 10.0 + w - 1\n"
        "dist.barrier(); dist.destroy_process_group()\n")
    import socket
    with socket.socket() as sk:  # a free port: other jobs on the host may hold any fixed one
        sk.bind(("127.0.0.1", 0))
        port = str(sk.getsockname()[1])
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT=port)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", port, str(script)], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]


def test_effective_cpus_is_sane():
    """Thread-pool sizing honours affinity and cgroup quotas (the GPU boxes show 128 CPUs and grant 16)."""
    import os
    from jxl_rs_b200.decoder import effective_cpus
    n = effective_cpus()
    assert 1 <= n <= (os.cpu_count() or 1)


def test_front_end_survives_corrupt_files(golden_dir):
    """Truncated / bit-flipped / spliced files must come back as an error code (or parse), never crash the process:
    the host front-end is the part of the product that touches untrusted bytes first."""
    import ctypes as C
    import glob
    from jxl_rs_b200 import abi
    from tests.fuzz_util import mutants
    lib = abi.load_library()
    paths = sorted(glob.glob(os.path.join(golden_dir, "jxl", "*.jxl")))
    parsed = errors = 0
    for _, data in mutants(paths, seed=1234, count=160):
        for parse, free in ((lib.jxg_parse_file, lib.jxg_parsed_free), (lib.jxg_modular_parse_file, lib.jxg_modular_parsed_free)):
            h, info = C.c_void_p(), abi.JxgImageInfo()
            r = parse(data, len(data), C.byref(h), C.byref(info))
            if r == 0:
                parsed += 1
                free(h)
            else:
                errors += 1
                assert r in abi.ERRORS, r
    assert errors > 0 and parsed >= 0


@pytest.mark.parametrize("name", REAL + ["green_queen_modular_e3.jxl", "lz77_flower.jxl", "tree_max_property_20.jxl", "grayscale_public_university.jxl",
                                         "alpha_premultiplied.jxl", "dice.jxl", "squeeze_alpha.jxl", "upsampled_alpha.jxl"])
def test_specialised_walks_match_the_generic_loop_on_reference_fixtures(golden_dir, name):
    """Same differential check on the reference's real files (libjxl trees: property walks, prefix codes, LZ77,
    weighted predictor), VarDCT front-end and Modular frames."""
    from tests import oracle_binding as ob
    lib = ob.load()
    data = open(os.path.join(golden_dir, "jxl", name), "rb").read()
    vardct = name in REAL or "alpha" in name or name == "dice.jxl"
    dec = (lambda d: ob.decode_file(d, abi.FORMAT_RGB_U8)[0]) if vardct else ob.decode_modular_file
    try:
        fast = dec(data)
        lib.jxo_t_force_generic_walk(1)
        slow = dec(data)
    finally:
        lib.jxo_t_force_generic_walk(0)
    assert np.array_equal(fast, slow)


def test_specialised_modular_walks_match_the_generic_loop():
    """Host front-end fast paths (static-leaf rows, direct-table ANS reader with unchecked refills, lazy-property
    walk) against the generic all-properties loop (decode/channel.rs FullTree semantics): same LF image and HF
    metadata, hence bit-identical coefficients and pixels, on a frame big enough (49 152 blocks, two LF groups wide)
    that the direct-table reader and the checked tail rows both run."""
    import synth
    from tests import oracle_binding as ob
    lib = ob.load()
    f = synth.encode_synthetic(2304 + 40, 1024 + 24, 4242, 0.5, 2, 1, 1)
    try:
        fast, taps_fast = ob.decode_file(f, abi.FORMAT_RGB_F32, taps=True)
        lib.jxo_t_force_generic_walk(1)
        slow, taps_slow = ob.decode_file(f, abi.FORMAT_RGB_F32, taps=True)
    finally:
        lib.jxo_t_force_generic_walk(0)
    assert np.array_equal(taps_fast["coeffs"], taps_slow["coeffs"])
    assert np.array_equal(fast, slow)
    # the same frame with the LF image coded like libjxl does (channel prefix + weighted-predictor subtree: the
    # single-property table walk): same LF samples, so the same pixels, through both walks
    fw = synth.encode_synthetic(2304 + 40, 1024 + 24, 4242, 0.5, 2, 1, 1, lf_tree=1)
    assert fw != f
    try:
        fast_w, _ = ob.decode_file(fw, abi.FORMAT_RGB_F32)
        lib.jxo_t_force_generic_walk(1)
        slow_w, _ = ob.decode_file(fw, abi.FORMAT_RGB_F32)
    finally:
        lib.jxo_t_force_generic_walk(0)
    assert np.array_equal(fast_w, fast) and np.array_equal(slow_w, fast)
    # Modular frames: group streams of 65 536 samples per channel through the same walks
    for tk in (0, 1):
        m = synth.encode_modular(700, 530, 11, 6, 0, tk)
        try:
            a = ob.decode_modular_file(m)
            lib.jxo_t_force_generic_walk(1)
            b = ob.decode_modular_file(m)
        finally:
            lib.jxo_t_force_generic_walk(0)
        assert np.array_equal(a, b) and np.array_equal(a, synth.modular_source(700, 530, 11))


def test_multithreaded_lf_groups_give_the_same_parse():
    """jxg_parse_file_mt: the LF groups of one frame decoded on several threads (frame_info.rs:505-520) must hand the
    hot path exactly the state the serial parse does — also when buffers come back from the pool with stale contents
    (the parses below recycle each other's planes), and a corrupt LF group must still be reported."""
    import synth
    from tests import oracle_binding as ob
    lib = ob.load()
    lib.jxo_t_parse_digest.restype = C.c_uint64
    lib.jxo_t_parse_digest.argtypes = [C.c_char_p, C.c_size_t, C.c_int]
    f = synth.encode_synthetic(4200, 2100, 99, 0.7, 2, 1, 1)  # 3 x 2 LF groups
    g = synth.encode_synthetic(4200, 2100, 100, 0.7, 2, 1, 1)
    ref_f, ref_g = lib.jxo_t_parse_digest(f, len(f), 1), lib.jxo_t_parse_digest(g, len(g), 1)
    assert ref_f != 0 and ref_g != 0 and ref_f != ref_g
    for threads in (2, 3, 8):
        assert lib.jxo_t_parse_digest(f, len(f), threads) == ref_f
        assert lib.jxo_t_parse_digest(g, len(g), threads) == ref_g
    assert lib.jxo_t_parse_digest(f, len(f), 1) == ref_f
    # serial parses pair LF groups (two sub-bitstreams in lockstep through the direct-table reader): the same state as
    # one group at a time, for plain and for libjxl-like (weighted-predictor, i.e. unpairable) LF coding, and for a
    # frame whose paired groups have different widths and heights
    for data in (f, g, synth.encode_synthetic(4200, 2100, 99, 0.7, 2, 1, 1, lf_tree=1),
                 synth.encode_synthetic(2048 + 8 * 9, 2048 + 8 * 3, 7, 0.7, 2, 1, 0)):
        paired = lib.jxo_t_parse_digest(data, len(data), 1)
        try:
            lib.jxo_t_pair_lf_groups(0)
            single = lib.jxo_t_parse_digest(data, len(data), 1)
            lib.jxo_t_force_generic_walk(1)
            generic = lib.jxo_t_parse_digest(data, len(data), 1)
        finally:
            lib.jxo_t_pair_lf_groups(1)
            lib.jxo_t_force_generic_walk(0)
        assert paired != 0 and paired == single == generic
    # many LF groups per thread: the worker threads take them in lockstep pairs too (10 groups, 2 threads)
    wide = synth.encode_synthetic(8200, 2056, 3, 1.5, 2, 1, 0)
    assert lib.jxo_t_parse_digest(wide, len(wide), 2) == lib.jxo_t_parse_digest(wide, len(wide), 1) != 0
    bad = bytearray(f)
    bad[len(f) // 40] ^= 0x55  # inside the LF-group sections (they come first and are ~5 % of the file)
    bad = bytes(bad)
    assert lib.jxo_t_parse_digest(bad, len(bad), 4) in (0, lib.jxo_t_parse_digest(bad, len(bad), 1))


def test_pipelined_decoder_host_logic_with_a_fake_device(monkeypatch):
    """The host side of PipelinedDecoder (worker pool, parse-ahead, dispatcher thread, per-file LF-group threads for
    single large images, error propagation) with the device context and batch replaced by recorders: no GPU needed."""
    import synth
    from jxl_rs_b200 import decoder

    calls = []

    class FakeCtx:
        def __init__(self, device):
            self.device = device

        def close(self):
            pass

    class FakeBatch:
        def __init__(self, ctx, n, staging_threads=0):
            self.frames = []

        def add(self, fr, ptr, stride, fmt, out_is_device):
            self.frames.append((fr.width, fr.height, ptr, stride))

        def run(self, stream_ptr=0):
            calls.append(list(self.frames))

        def wait(self):
            pass

        def stats(self):
            return {"h2d_bytes": 1, "d2h_bytes": 2, "kernel_launches": 3}

        def close(self):
            pass

    monkeypatch.setattr(decoder, "JxgContext", FakeCtx)
    monkeypatch.setattr(decoder, "Batch", FakeBatch)
    seen_threads = []
    real_parsed = decoder.ParsedFrame

    class SpyParsed(real_parsed):
        def __init__(self, data, threads=1):
            seen_threads.append(threads)
            super().__init__(data, threads)

    monkeypatch.setattr(decoder, "ParsedFrame", SpyParsed)
    files = [synth.encode_synthetic(64 + 8 * i, 48, 10 + i, 1.0, 2, 1, 0) for i in range(3)]
    dec = decoder.PipelinedDecoder(0, depth=2, workers=6)
    try:
        for _ in range(4):
            dec.submit(files, [(100 + i, 7) for i in range(3)])
        dec.drain()
        assert len(calls) == 4 and all(len(c) == 3 for c in calls)
        assert calls[0][1][:2] == (72, 48) and calls[0][2][2:] == (102, 7)
        assert set(seen_threads) == {2}  # 6 workers / 3 files
        dec.decode(files[:1], [(5, 5)])
        assert seen_threads[-1] == 6 and dec.last_stats["kernel_launches"] == 3
        # a corrupt file surfaces at drain() as the front-end's error, and the decoder stays usable
        dec.submit([files[0][:40]], [(1, 1)])
        with pytest.raises(abi.JxgError):
            dec.drain()
        dec.decode(files[:2], [(1, 1), (2, 2)])
    finally:
        dec.close()


@pytest.mark.parametrize("w,h,epf,profile,fmt", [(520, 300, 2, 1, 0), (333, 271, 1, 2, 1), (1024, 768, 2, 3, 0), (300, 200, 3, 1, 0),
                                                 (64, 40, 2, 0, 0)])
def test_fast_cpu_forms_are_bit_identical_to_the_scalar_oracle(w, h, epf, profile, fmt):
    """The AVX2 forms the CPU baseline of bench.py runs (8-lane IDCTs, Gaborish, EPF 1 / 2, sRGB u8 store: every lane runs
    the scalar sequence) against the plain restatement that serves as the checker: coefficients aside, every plane and
    every output byte must be equal."""
    import synth
    from jxl_rs_b200 import abi
    from tests import oracle_binding as ob
    lib = ob.load()
    data = synth.encode_synthetic(w, h, 90 + w, 0.5, epf, 1, profile)
    f = abi.FORMAT_RGBA_U8 if fmt else abi.FORMAT_RGB_U8
    try:
        lib.jxo_set_fast_cpu(0)
        a, ta = ob.decode_file(data, f, taps=True, threads=2)
        lib.jxo_set_fast_cpu(1)
        ob.decode_file(synth.encode_synthetic(w + 72, h + 40, 3, 0.5, 2, 1, 1), f, threads=1)  # stale pixels of a larger frame
        b, tb = ob.decode_file(data, f, taps=True, threads=1)                                    # in this thread's plane pool
        b2, _ = ob.decode_file(data, f, threads=2)
    finally:
        lib.jxo_set_fast_cpu(0)
    assert np.array_equal(ta["xyb_idct"], tb["xyb_idct"])
    assert np.array_equal(ta["xyb_filtered"], tb["xyb_filtered"])
    assert np.array_equal(a, b) and np.array_equal(a, b2)
