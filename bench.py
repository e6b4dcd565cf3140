#!/usr/bin/env python3
"""bench.py -- headline benchmark of the B200 DEFLATE engine: prints one JSON line.

metric  : deflate level-6 GiB/s of raw input on silesia-small.tar (BASELINE.json), zlib wrapper, windowBits 15,
          one deflate(Z_FINISH)-equivalent call per stream -- configs[1].
step    : every rank compresses one copy of silesia-small.tar (15,736,320 B).  N ranks = N independent streams
          ("weak" scaling: per-GPU work is fixed); with N > 1 the compressed segments are all-gathered over NCCL.
value   : device-timed (CUDA events), input and output resident in HBM.
e2e     : the same job through the zlib C ABI (compress2) with pinned HOST buffers, copies inside the timed region.
roofline: k_match (the dominant kernel): algorithmic bytes = the raw input each full launch must read once.
--impl reference : the reference's CPU implementation of the path (the oracle restatement -- zlib-rs itself cannot
          be built here, see DESIGN.md) on the host cores, same workload.
--dump-outputs DIR : after the timed steps, what the last timed step handed its caller -- the compressed stream as
          DIR/compressed.npy (one float32 per byte) and its adler32 as DIR/adler32.npy (float64) -- so that two builds can be
          compared output for output (the input is the same file on every run).
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

GIB = float(1 << 30)
METRIC = "deflate_level6_raw_input_throughput_silesia_small_tar"


def load_tar():
    from corpus import silesia_tar
    return silesia_tar()


ORACLE_FLAGS = {"native": "-O3 -march=native (built on this host by bench.py: make -C oracle native)",
                "portable": "-O3 -march=x86-64-v2 (oracle/Makefile default; the native build failed on this host)"}
_oracle = {}


def oracle_compress_fn():
    """The CPU arm: oracle/ (C restatement of zlib-rs) compiled for THIS host's instruction set; falls back to the portable build
    the tests use.  Returns (compress(data, level) -> (rc, bytes), flags description)."""
    if "fn" in _oracle:
        return _oracle["fn"], _oracle["flags"]
    import shutil
    import tempfile
    import oracle_lib as O
    fn, flags = O.compress, ORACLE_FLAGS["portable"]
    try:
        tmp = tempfile.mkdtemp(prefix="zoracle_native_")  # built per run outside the tree, which may be read-only
        try:
            subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "native", "NATIVE_DIR=" + tmp],
                                  stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            L = ctypes.CDLL(os.path.join(tmp, "libzoracle_native_host.so"))
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
        sz = ctypes.c_size_t
        L.zo_compress_ex.argtypes = [ctypes.c_char_p, ctypes.POINTER(sz), ctypes.c_char_p, sz] + [ctypes.c_int] * 5

        def native(data, level=6):
            cap = len(data) + len(data) // 8 + 1024
            dst = ctypes.create_string_buffer(cap)
            n = sz(cap)
            rc = L.zo_compress_ex(dst, ctypes.byref(n), bytes(data), len(data), level, 15, 8, 0, 4)
            return rc, dst.raw[: n.value]

        probe = (b"oracle self check %d " * 4000) % tuple(range(4000))
        rc, out = native(probe, 6)
        assert rc == 0 and out == O.compress(probe, 6)[1]
        # the code is scalar C, so the instruction set hardly matters: take whichever build is faster on this host
        def best_of(f):
            b = 1e9
            for _ in range(3):
                t = time.perf_counter(); f(probe * 8, 6); b = min(b, time.perf_counter() - t)
            return b
        if best_of(native) <= best_of(O.compress):
            fn, flags = native, ORACLE_FLAGS["native"]
        else:
            flags = "-O3 -march=x86-64-v2 (faster on this host than the -march=native build, both timed)"
    except Exception:
        pass
    _oracle["fn"], _oracle["flags"] = fn, flags
    return fn, flags


def workload(n_streams):
    """config.workload, the same string in both arms."""
    return ("deflate level 6, windowBits 15, memLevel 8, default strategy; %d x silesia-small.tar (15736320 B each), "
            "one compress2 / deflate(Z_FINISH) per stream" % n_streams)


def dump_outputs(d, compressed, adler):
    """--dump-outputs: the compressed stream (one float32 per byte, 25 MiB for silesia-small.tar at level 6) and its adler32."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, "compressed.npy"), np.frombuffer(bytes(compressed), dtype=np.uint8).astype(np.float32))
    np.save(os.path.join(d, "adler32.npy"), np.array([adler], dtype=np.float64))


def cpu_sample(tar, reps=2):
    """Single host thread, whole tar, best of `reps` (BASELINE.md: CPU-baseline plan)."""
    comp, _ = oracle_compress_fn()
    best = 1e9
    for _ in range(reps):
        t = time.perf_counter()
        rc, out = comp(tar, 6)
        best = min(best, time.perf_counter() - t)
    assert rc == 0
    return len(tar) / best / GIB, len(out)


class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw"

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.stop = False
        self.t = None

    def _run(self):
        while not self.stop:
            try:
                o = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                   capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([x.strip() for x in o.split(",")])
            except Exception:
                pass
            time.sleep(0.15)

    def start(self):
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def finish(self):
        self.stop = True
        if self.t:
            self.t.join(timeout=6)
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = []
        for i, name in ((2, "hw_slowdown"), (3, "hw_thermal_slowdown"), (4, "sw_thermal_slowdown"), (5, "sw_power_cap")):
            if any(len(r) > i and r[i].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    tar = load_tar()
    comp, oflags = oracle_compress_fn()
    n_streams = args.gpus
    cores = os.cpu_count() or 1
    threads = min(n_streams, cores)
    from concurrent.futures import ThreadPoolExecutor

    def one(_):
        rc, out = comp(tar, 6)  # ctypes releases the GIL
        assert rc == 0
        return out

    with ThreadPoolExecutor(max_workers=threads) as ex:
        for _ in range(args.warmup):
            list(ex.map(one, range(n_streams)))
        t0 = time.perf_counter()
        for _ in range(args.steps):
            outs = list(ex.map(one, range(n_streams)))
        dt = (time.perf_counter() - t0) / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outs[0], int.from_bytes(outs[0][-4:], "big"))  # a zlib stream ends with its adler32
    value = n_streams * len(tar) / dt / GIB
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "GiB/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "silesia-small.tar (reference corpus, committed as data/silesia-small.tar.gz)",
        "config": {"workload": workload(n_streams),
                   "impl_note": "C restatement of zlib-rs (oracle/), not the Rust binary: no Rust toolchain in this image; scalar code "
                                "(no AVX2 compare256 / PCLMUL), so zlib-rs itself would be faster", "build": oflags,
                   "host_cpus": cores},
        "cpu_baseline": {"value": value, "unit": "GiB/s", "cores": threads, "kind": "port",
                         "sample": "%d full streams per step, one host thread per stream" % n_streams, "build": oflags},
        "e2e": {"value": value, "unit": "GiB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import zlib_rs_b200 as Z
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    eng = Z.Engine(local)
    tar = load_tar()
    N = len(tar)
    W = max(args.warmup, 3)
    K = args.steps

    # rotating inputs (10 copies = 157 MB > 126 MB L2) so the raw bytes come from HBM every step
    ROT = 10
    host = torch.frombuffer(bytearray(tar), dtype=torch.uint8)
    ins = []
    for _ in range(ROT):
        t = torch.zeros(N + 4096, dtype=torch.uint8, device=dev)
        t[:N].copy_(host)
        ins.append(t)
    cap = int(Z.lib().zb_deflate_bound(N)) + 64
    cap = (cap + 255) & ~255
    out_t = torch.zeros(cap, dtype=torch.uint8, device=dev)
    gather_state = {"t": None, "seg": 0}
    torch.cuda.synchronize()

    def gather_segments(seg_t, seg_len):
        """One all-gather of the segment sizes, one of the segment bytes (padded to the largest segment, 256-byte granules)."""
        sizes = torch.tensor([seg_len], dtype=torch.int64, device=dev)
        all_sizes = torch.zeros(world, dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(all_sizes, sizes)
        mx = (int(all_sizes.max().item()) + 255) & ~255
        if gather_state["t"] is None or gather_state["seg"] < mx:
            gather_state["t"], gather_state["seg"] = torch.zeros(mx * world, dtype=torch.uint8, device=dev), mx
        g = gather_state["t"][: mx * world]
        dist.all_gather_into_tensor(g, seg_t[:mx])
        return g, all_sizes, mx

    cpu_b = None
    if rank == 0 and world == 1:
        v, _ = cpu_sample(tar, reps=2)
        cpu_b = {"value": v, "unit": "GiB/s", "cores": 1, "kind": "port", "build": oracle_compress_fn()[1],
                 "sample": "whole silesia-small.tar, level 6, best of 2, single host thread (oracle restatement of zlib-rs, scalar)"}
        try:  # orientation only (BASELINE.md): stock zlib 1.3 on the same core -- other algorithms, other bytes
            import zlib as _z
            t_ = time.perf_counter()
            _z.compress(tar, 6)
            cpu_b["stock_zlib_1_3_GiBps"] = len(tar) / (time.perf_counter() - t_) / GIB
            cpu_b["host_cpus"] = os.cpu_count()
        except Exception:
            pass

    def step(i, timed):
        src = ins[i % ROT]
        _, res = eng.deflate(src.data_ptr(), n=N, level=6, src_on_device=True, dst=out_t.data_ptr(), dst_cap=cap, dst_on_device=True)
        ms = res.gpu_ms
        if world > 1:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            gather_segments(out_t, int(res.out_bytes))
            e1.record()
            torch.cuda.synchronize()
            ms += e0.elapsed_time(e1)
        return ms, res

    for i in range(W):
        ms, res = step(i, False)
    out_bytes = int(res.out_bytes)
    launches = int(res.gpu_launches) + (2 if world > 1 else 0)
    sampler = ClockSampler(local)
    sampler.start()
    if dist:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    dev_ms = 0.0
    for i in range(K):
        ms, res = step(W + i, True)
        dev_ms += ms
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    if args.dump_outputs and rank == 0:  # out_t is reused below, so the last timed step's stream is read back now
        dump_outputs(args.dump_outputs, out_t[: int(res.out_bytes)].cpu().numpy(), int(res.check))
    ms_per_step = dev_ms / K
    if dist:
        t = torch.tensor([ms_per_step], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_per_step = float(t.item())

    # e2e through the zlib C ABI with pinned host buffers (wall clock around compress2)
    pin_in = torch.empty(N, dtype=torch.uint8).pin_memory()
    pin_in.copy_(host)
    bound = int(Z.lib().compressBound(N))
    pin_out = torch.empty(bound, dtype=torch.uint8).pin_memory()
    L = Z.lib()
    e2e_t = []
    for i in range(W + K):
        n = ctypes.c_ulong(bound)
        t1 = time.perf_counter()
        rc = L.compress2(pin_out.data_ptr(), ctypes.byref(n), pin_in.data_ptr(), N, 6)
        dt = time.perf_counter() - t1
        assert rc == 0
        if i >= W:
            e2e_t.append(dt)
    e2e_ms = sum(e2e_t) / len(e2e_t) * 1e3
    if dist:
        t = torch.tensor([e2e_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    clocks = sampler.finish()

    # roofline of the dominant kernel, timed live with CUDA events around each launch group
    roof = None
    if rank == 0:
        eng.set_profile(True)
        _, res = eng.deflate(ins[0].data_ptr(), n=N, level=6, src_on_device=True, dst=out_t.data_ptr(), dst_cap=cap, dst_on_device=True)
        prof = eng.get_profile()
        eng.set_profile(False)
        peaks = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks):
            peak, peak_src = float(json.load(open(peaks))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (burst)"
        else:
            peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
        m = prof["match"]
        full_ms = prof.get("match_first", {"ms": m["ms"] / max(m["launches"], 1)})["ms"]
        achieved = N / (full_ms * 1e-3) / 1e9
        # dram__bytes_read+write of one full k_match launch from the committed `ncu --set full` capture -- only if that capture
        # was made from THIS build of the kernels (sha256 of zb_kernels.cu recorded beside the number), else null
        traffic, traffic_note = None, None
        tp = os.path.join(ROOT, "profiles", "k_match_traffic.json")
        if os.path.exists(tp):
            import hashlib
            tj = json.load(open(tp))
            src_sha = hashlib.sha256(open(os.path.join(ROOT, "zlib_rs_b200", "csrc", "zb_kernels.cu"), "rb").read()).hexdigest()
            if tj.get("kernels_sha256") == src_sha:
                traffic, traffic_note = tj.get("dram_bytes_per_launch"), tj.get("capture")
            else:
                traffic_note = "profiles/k_match_traffic.json was captured from another build of zb_kernels.cu"
        roof = {"bound": "hbm", "kernel": "k_match", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_note, "peak_source": peak_src, "algorithmic_bytes_per_launch": N, "launch_ms": full_ms,
                "phases_ms": {k: round(v["ms"], 4) for k, v in prof.items()}, "iterations": int(res.iterations)}

    # One stream cut into `world` contiguous ranges (SURVEY.md 8e, BASELINE config 4): every rank compresses its range as a raw
    # segment (ZB_FLAG_NOT_LAST: closed by the sync marker, BFINAL only on the last), sizes and segment bytes are all-gathered,
    # rank 0 stitches zlib header + segments + combined adler32 and checks the stream with stock zlib.  Strong scaling: the total
    # work is fixed.  Valid stream, not the serial parser's bytes (the exact hand-off is described in DESIGN.md).
    sharded = {}

    def sharded_stream(name, data, level, reps=3):
        from zlib_rs_b200 import shard
        lo, hi = shard.plan_shards(len(data), world)[rank]
        part = torch.frombuffer(bytearray(data[lo:hi]), dtype=torch.uint8)
        part_d = torch.zeros(hi - lo + 4096, dtype=torch.uint8, device=dev)
        part_d[: hi - lo].copy_(part)
        pcap = (int(Z.lib().zb_deflate_bound(hi - lo)) + 64 + 255) & ~255
        seg_d = torch.zeros(pcap, dtype=torch.uint8, device=dev)
        flags = (0 if rank == world - 1 else Z.ZB_FLAG_NOT_LAST) | Z.ZB_FLAG_CHECK_ADLER
        best, keep = 1e9, None
        for r in range(reps):
            if dist:
                dist.barrier()
            torch.cuda.synchronize()
            _, rs = eng.deflate(part_d.data_ptr(), n=hi - lo, level=level, window_bits=-15, flags=flags, src_on_device=True,
                                dst=seg_d.data_ptr(), dst_cap=pcap, dst_on_device=True)
            ms = rs.gpu_ms
            if dist:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                g, sizes, mx = gather_segments(seg_d, int(rs.out_bytes))
                meta = torch.tensor([int(rs.check), hi - lo], dtype=torch.int64, device=dev)
                all_meta = torch.zeros(2 * world, dtype=torch.int64, device=dev)
                dist.all_gather_into_tensor(all_meta, meta)
                e1.record()
                torch.cuda.synchronize()
                ms += e0.elapsed_time(e1)
                t = torch.tensor([ms], device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t.item())
                keep = (g, sizes, mx, all_meta)
            else:
                keep = (seg_d, torch.tensor([int(rs.out_bytes)]), pcap, torch.tensor([int(rs.check), hi - lo]))
            best = min(best, ms)
        if rank != 0:
            return
        g, sizes, mx, all_meta = keep
        gh = g.cpu().numpy().tobytes()
        segs = [gh[i * mx: i * mx + int(sizes[i])] for i in range(world)]
        meta = [int(x) for x in all_meta.cpu()]
        stream = shard.stitch_zlib(segs, meta[0::2], meta[1::2], level)
        import zlib as _z
        ok = _z.decompress(stream) == data
        sharded[name] = {"ms": best, "GiBps": len(data) / (best * 1e-3) / GIB, "out_bytes": len(stream), "ranges": world,
                         "inflates_to_input_under_stock_zlib": bool(ok), "exact_parity": 1 if world == 1 else 0, "scaling": "strong",
                         "collective": "all_gather(sizes) + all_gather(segment bytes, padded to the largest) + all_gather(adler, length)" if world > 1 else "none",
                         "note": "device resident, CUDA events, max over ranks, best of %d" % reps}

    try:
        sharded_stream("sharded_deflate_level6_silesia_small_tar", tar, 6)
        from corpus import calgary_mix
        sharded_stream("sharded_deflate_level9_calgary_mix_64MiB", calgary_mix(), 9, reps=2)
    except Exception as ex:
        sharded["error"] = repr(ex)

    # the other BASELINE.json configs, measured once each on rank 0 at N=1 (device resident, CUDA events; reported, not the headline)
    other = None
    if rank == 0 and world == 1:
        try:
            from corpus import silesia_gz
            gz = silesia_gz()
            other = {}
            best = min(eng.inflate(gz, N)[2].gpu_ms for _ in range(3))
            rc, got, r3 = eng.inflate(gz, N)
            peak_i = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 6650.0
            alg = len(gz) + N  # SURVEY.md 8(d): compressed bytes in + raw bytes out
            other["inflate_silesia_small_tar_gz"] = {"ms": best, "out_GBps": N / best / 1e6, "bit_exact": bool(rc == 0 and got == tar),
                                                     "gpu_launches": int(r3.gpu_launches), "note": "config 3; host buffers, copies inside the timed region",
                                                     "roofline": {"bound": "hbm", "algorithmic_bytes": alg, "achieved": alg / best / 1e6, "peak": peak_i, "unit": "GB/s",
                                                                  "frac": alg / best / 1e6 / peak_i, "note": "whole call incl. H2D/D2H; the kernels are latency-bound (DESIGN.md 2c)"}}
            o9, r9 = eng.deflate(ins[0].data_ptr(), n=N, level=9, src_on_device=True, dst=out_t.data_ptr(), dst_cap=cap, dst_on_device=True)
            o9, r9 = eng.deflate(ins[1].data_ptr(), n=N, level=9, src_on_device=True, dst=out_t.data_ptr(), dst_cap=cap, dst_on_device=True)
            out9 = bytes(out_t[: int(r9.out_bytes)].cpu().numpy().tobytes())
            other["deflate_level9_silesia_small_tar"] = {"ms": r9.gpu_ms, "GiBps": N / (r9.gpu_ms * 1e-3) / GIB, "out_bytes": int(r9.out_bytes),
                                                         "equals_reference_file": out9 == gz, "exact_parity": int(r9.exact_parity)}
            for lv in (1, 2):  # deflate_quick / deflate_fast: the reference's serial parser on one warp (exact, latency-bound)
                olv, rlv = eng.deflate(ins[lv].data_ptr(), n=N, level=lv, src_on_device=True, dst=out_t.data_ptr(), dst_cap=cap, dst_on_device=True)
                other["deflate_level%d_silesia_small_tar" % lv] = {"ms": rlv.gpu_ms, "GiBps": N / (rlv.gpu_ms * 1e-3) / GIB, "out_bytes": int(rlv.out_bytes),
                                                                   "exact_parity": int(rlv.exact_parity), "note": "one warp per stream (zb_serial.h)"}
            try:
                from corpus import calgary_mix
                cm = calgary_mix()
                ocm, rcm = eng.deflate(cm, level=9)
                ocm, rcm = eng.deflate(cm, level=9)
                other["deflate_level9_calgary_mix_64MiB"] = {"ms": rcm.gpu_ms, "GiBps": len(cm) / (rcm.gpu_ms * 1e-3) / GIB, "out_bytes": int(rcm.out_bytes),
                                                            "exact_parity": int(rcm.exact_parity), "note": "config 4 as one stream; host buffers, copies inside the timed region"}
            except Exception as ex:
                other["calgary_mix_error"] = repr(ex)
            # several independent streams in flight on one GPU (one Engine = one CUDA stream + its own buffers per host thread):
            # the single-stream pipeline leaves most SMs idle in its latency-bound phases
            try:
                S = 4
                engs = [Z.Engine(local) for _ in range(S)]
                outs = [torch.zeros(cap, dtype=torch.uint8, device=dev) for _ in range(S)]
                bar = threading.Barrier(S + 1)
                reps = 6

                def worker(j):
                    e, o = engs[j], outs[j]
                    e.deflate(ins[j % ROT].data_ptr(), n=N, level=6, src_on_device=True, dst=o.data_ptr(), dst_cap=cap, dst_on_device=True)
                    bar.wait()
                    for r in range(reps):
                        e.deflate(ins[(j + r) % ROT].data_ptr(), n=N, level=6, src_on_device=True, dst=o.data_ptr(), dst_cap=cap, dst_on_device=True)
                    bar.wait()

                ths = [threading.Thread(target=worker, args=(j,)) for j in range(S)]
                for t_ in ths:
                    t_.start()
                bar.wait()
                t_a = time.perf_counter()
                bar.wait()
                t_b = time.perf_counter()
                for t_ in ths:
                    t_.join()
                other["deflate_level6_%d_concurrent_streams" % S] = {"GiBps_aggregate": S * reps * N / (t_b - t_a) / GIB, "ms_per_stream": (t_b - t_a) / reps * 1e3,
                                                                    "note": "wall clock; %d engines driven by %d host threads, same byte-identical output" % (S, S)}
                for e_ in engs:
                    e_.close()
            except Exception as ex:
                other["concurrent_streams_error"] = repr(ex)
            nck = 8 << 30
            pck = eng.alloc(nck)
            try:
                eng.fill_random(pck, nck, 42)
                a_ms = min(eng.adler32(pck, nck, on_device=True)[1] for _ in range(3))
                c_ms = min(eng.crc32(pck, nck, on_device=True)[1] for _ in range(3))
                other["checksums_8GiB"] = {"adler32_GBps": nck / a_ms / 1e6, "crc32_GBps": nck / c_ms / 1e6, "note": "config 5; splitmix64 buffer generated on the device"}
            finally:
                eng.free(pck)
        except Exception as ex:  # the headline must not depend on these
            other = {"error": repr(ex)}

    if rank == 0:
        value = world * N / (ms_per_step * 1e-3) / GIB
        e2e = world * N / (e2e_ms * 1e-3) / GIB
        line = {
            "metric": METRIC, "value": value, "unit": "GiB/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "silesia-small.tar (reference corpus, committed as data/silesia-small.tar.gz)",
            "config": {"workload": workload(world), "parity": "output byte-identical to the reference's compress2 (sha256 pinned in tests/)",
                       "l2": "inputs rotate over 10 device copies (157 MB > 126 MB L2); ~480 MB of intermediates per step",
                       "compressed_bytes": out_bytes, "wall_ms_per_step": wall_ms / K,
                       "parallelism": "1 stream per GPU" + (", NCCL all-gather of compressed segments" if world > 1 else "")},
            "clocks": clocks,
            "e2e": {"value": e2e, "unit": "GiB/s", "h2d_bytes_per_step": N, "d2h_bytes_per_step": out_bytes, "ms_per_step": e2e_ms,
                    "api": "compress2() of libz_b200.so, pinned host buffers"},
            "gpu_launches": launches,
            "roofline": roof,
        }
        if cpu_b:
            line["cpu_baseline"] = cpu_b
        if sharded:
            other = dict(other or {})
            other["chunk_sharded_single_stream"] = sharded
        if other:
            line["other_configs"] = other
        print(json.dumps(line))
    if dist:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
