"""CPU tests of the drop-in boundary: the C-ABI library loads, exports every symbol the headers declare,
keeps the z_stream layout, and the entry points that need no device behave like the reference.
(No compute calls: there is no GPU here and the library has no CPU fallback.)"""
import ctypes
import os
import re

import pytest

import oracle_lib as O
import zlib_rs_b200 as Z

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared(header, macro):
    src = open(os.path.join(ROOT, "include", header)).read()
    return sorted(set(re.findall(macro + r"[^;(]*?\b(\w+)\s*\(", src)) - {"__attribute__"})


def test_library_exports_every_declared_symbol():
    L = Z.lib()
    names = _declared("zlib_b200.h", "ZB_EXPORT") + _declared("zb_engine.h", "ZB_API")
    assert len(names) > 60
    missing = [n for n in names if not hasattr(L, n)]
    assert not missing, missing
    # north_star's mandatory surface (SURVEY.md 8b)
    for n in ("deflateInit2_", "deflate", "deflateEnd", "inflateInit2_", "inflate", "inflateEnd", "compress2", "uncompress",
              "crc32", "adler32"):
        assert n in names


def test_z_stream_layout():
    # zlib-rs/src/c_api.rs:56-71: 112 bytes on LP64
    assert ctypes.sizeof(Z.ZStream) == 112
    assert Z.ZStream.total_in.offset == 16 and Z.ZStream.next_out.offset == 24 and Z.ZStream.state.offset == 56
    assert Z.ZStream.data_type.offset == 88 and Z.ZStream.adler.offset == 96


def test_version_rule():
    # libz-rs-sys/src/lib.rs:2133-2145
    L = Z.lib()
    s = Z.ZStream()
    assert L.zlibVersion().startswith(b"1.3.0-zlib-rs-0.6.7")
    assert L.deflateInit2_(ctypes.byref(s), 6, 8, 15, 8, 0, b"2.0", 112) == Z.Z_VERSION_ERROR
    assert L.deflateInit2_(ctypes.byref(s), 6, 8, 15, 8, 0, None, 112) == Z.Z_VERSION_ERROR
    assert L.deflateInit2_(ctypes.byref(s), 6, 8, 15, 8, 0, Z.ZLIB_VERSION, 111) == Z.Z_VERSION_ERROR
    assert L.inflateInit2_(ctypes.byref(s), 15, b"0.9", 112) == Z.Z_VERSION_ERROR
    assert L.deflateInit2_(None, 6, 8, 15, 8, 0, Z.ZLIB_VERSION, 112) == Z.Z_STREAM_ERROR


def test_parameter_errors_before_device_use():
    # zlib-rs/src/deflate.rs:282-312, inflate.rs:2298-2327
    L = Z.lib()
    s = Z.ZStream()
    for lvl, wb, mem, strat in ((10, 15, 8, 0), (6, 16, 8, 0), (6, 7, 8, 0), (6, 15, 0, 0), (6, 15, 10, 0), (6, 15, 8, 5), (6, -8, 8, 0),
                                (6, -16, 8, 0)):
        assert L.deflateInit2_(ctypes.byref(s), lvl, 8, wb, mem, strat, Z.ZLIB_VERSION, 112) == Z.Z_STREAM_ERROR, (lvl, wb, mem, strat)
    assert L.deflateInit2_(ctypes.byref(s), 6, 7, 15, 8, 0, Z.ZLIB_VERSION, 112) == Z.Z_STREAM_ERROR  # method
    assert L.inflateInit2_(ctypes.byref(s), 7, Z.ZLIB_VERSION, 112) == Z.Z_STREAM_ERROR
    assert L.inflateInit2_(ctypes.byref(s), -16, Z.ZLIB_VERSION, 112) == Z.Z_STREAM_ERROR
    s2 = Z.ZStream()
    assert L.deflate(ctypes.byref(s2), 0) == Z.Z_STREAM_ERROR      # NULL state
    assert L.deflateEnd(ctypes.byref(s2)) == Z.Z_STREAM_ERROR
    assert L.inflate(ctypes.byref(s2), 0) == Z.Z_STREAM_ERROR
    assert L.inflateEnd(ctypes.byref(s2)) == Z.Z_STREAM_ERROR
    assert L.deflate(None, 0) == Z.Z_STREAM_ERROR


def test_no_device_is_loud_not_a_fallback():
    L = Z.lib()
    if L.zb_device_count() > 0:
        pytest.skip("a GPU is present")
    s = Z.ZStream()
    assert L.deflateInit2_(ctypes.byref(s), 6, 8, 15, 8, 0, Z.ZLIB_VERSION, 112) == Z.Z_MEM_ERROR
    assert s.msg == b"no CUDA device"
    assert L.inflateInit2_(ctypes.byref(s), 15, Z.ZLIB_VERSION, 112) == Z.Z_MEM_ERROR
    n = ctypes.c_ulong(100)
    assert L.compress2(ctypes.create_string_buffer(100), ctypes.byref(n), b"abc", 3, 6) == Z.Z_MEM_ERROR
    with pytest.raises(RuntimeError):
        Z.Engine(0)


def test_null_buffer_checksums_and_combine_algebra():
    # libz-rs-sys/src/lib.rs:150-155, 307-312; combine: crc32/combine.rs, adler32.rs:58-87
    L = Z.lib()
    assert L.crc32_z(123, None, 10) == 0 and L.adler32_z(77, None, 10) == 1
    Lo = O.lib()
    for a, b, n in ((1, 1, 0), (0x12345678, 0x9abcdef0, 1), (0xdeadbeef, 0x0badf00d, 5552), (5, 7, 1 << 33)):
        assert L.crc32_combine64(a, b, n) == Lo.zo_crc32_combine(a, b, n)
        assert L.crc32_combine_op(a, b, L.crc32_combine_gen64(n)) == Lo.zo_crc32_combine(a, b, n)
        assert L.adler32_combine64(a % 65521 | ((a >> 16) % 65521) << 16, b % 65521 | ((b >> 16) % 65521) << 16, n) == \
            Lo.zo_adler32_combine(a % 65521 | ((a >> 16) % 65521) << 16, b % 65521 | ((b >> 16) % 65521) << 16, n)
    assert L.zError(-3) == b"data error" and L.zError(-5) == b"buffer error"
    # deflate::compress_bound's documented values (zlib-rs/src/deflate.rs:2966-2968) and the oracle's restatement
    assert (L.compressBound(1024), L.compressBound(4096), L.compressBound(65536)) == (1161, 4617, 73737)
    Lo.zo_compress_bound.restype = ctypes.c_size_t
    Lo.zo_compress_bound.argtypes = [ctypes.c_size_t]
    for n in (0, 1, 8, 9, 100, 1 << 20, 15736320):
        assert L.compressBound(n) == Lo.zo_compress_bound(n)


def test_c_client_links_and_fails_loudly_without_a_device(tmp_path):
    """tests/c_client/pipe_client.c: a plain C program (header + -lz_b200) with zpipe's call sequence.  Without a CUDA device
    deflateInit returns Z_MEM_ERROR ("no CUDA device") -- never a CPU path; on the GPU box the same binary round-trips a file
    (tests/test_gpu_parity.py::test_c_client_round_trip)."""
    import subprocess, os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.check_call(["make", "-C", os.path.join(root, "tests", "c_client")], stdout=subprocess.DEVNULL)
    import torch
    if torch.cuda.is_available():
        return
    f = tmp_path / "in.bin"
    f.write_bytes(b"hello hello hello" * 100)
    r = subprocess.run([os.path.join(root, "tests", "c_client", "_build", "pipe_client"), str(f)], capture_output=True, text=True)
    assert r.returncode == 77 and "no CUDA device" in r.stderr


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU restatement on the host cores) prints one JSON line with the contract's keys."""
    import json, os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "GiB/s" and line["higher_is_better"] is True and line["n_gpus"] == 1
    assert line["metric"] == "deflate_level6_raw_input_throughput_silesia_small_tar" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] == 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]


def test_reference_zpipe_compiles_and_links_unchanged():
    """The reference's own C client (libz-rs-sys-cdylib/zpipe.c) builds against include/zlib.h and links with -lz_b200 without a
    source change: build() compiles it (oracle/Makefile, target `ref`) into oracle/_ref/zpipe_ref, which
    tests/test_gpu_stream.py runs.  Skipped where build() had no zlib-rs source tree to compile it from."""
    import subprocess
    exe = os.path.join(ROOT, "oracle", "_ref", "zpipe_ref")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/zpipe_ref was not built (no zlib-rs source tree at build time)")
    needed = subprocess.run(["readelf", "-d", exe], capture_output=True, text=True).stdout
    assert "[libz_b200.so]" in needed and "[libz.so" not in needed
    syms = subprocess.run(["nm", "-D", "--undefined-only", exe], capture_output=True, text=True).stdout
    for f in ("deflateInit_", "deflate", "deflateEnd", "inflateInit_", "inflate", "inflateEnd"):
        assert (" " + f + "\n") in syms or (" " + f + "@") in syms or f in syms
