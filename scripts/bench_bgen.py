"""BGEN ingest measurements on one GPU, written as JSON (--out; also printed).

Writes a synthetic BGEN 1.2 file (layout 2, B = 8, zlib; default 50 000 samples x 20 000 variants, about 3 GB of
inflated probability data: 80 % hard calls, the rest random probabilities, 1 % missing) into a temporary directory,
then times each stage of B200DenseLinAlg.from_bgen separately in one process:
  parse     BgenFile: header, sample block and the variant index (host)
  inflate   zlib.decompress of every block in ~64 MB batches on a thread pool (host)
  load      ihtb_geno_load_bgen_columns for all batches: pinned staging, H2D copies and the decode kernel (overlapped)
  decode    the k_bgen_decode kernel alone (torch.profiler CUDA activity, a separate load of the same batches)
  h2d       the host-to-device copies of that load (same trace)
  finalize  ihtb_geno_finalize (column statistics, missing-row index)
  end_to_end  from_bgen(path, standardize=True) as a user calls it (inflate overlapped with the device load)
and the decode kernel's bytes/s (inflated bytes read + code bytes written) against a device-to-device copy in the same
run (read + write bytes, torch, CUDA events, a buffer far larger than L2).  The card's name and power limit are read
in the same run.  The loaded handle is checked against the host twin (bgen.dosage_codes) on its first variants.

Selection cases ("selection" in the output; from_bgen(samples=, variants=)), each timed the same way -- inflate of the
kept variants, the decode kernel alone (torch.profiler), end-to-end from_bgen -- and checked against the host twin:
  samples_50_sorted     every variant, half of the samples in file order
  samples_50_shuffled   every variant, the same half in a random order (scattered reads inside each block)
  variants_10           every sample, a random 10 % of the variants (the others are never inflated)"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import mendeliht_jl_b200 as m  # noqa: E402
from mendeliht_jl_b200 import _lib, bgen  # noqa: E402
import bgen_writer as bw  # noqa: E402


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clk = [t.strip() for t in out.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clk}


def copy_bandwidth(nbytes: int, reps: int = 20) -> float:
    import torch
    a = torch.empty(nbytes // 4, dtype=torch.float32, device="cuda")
    b = torch.empty_like(a)
    a.fill_(1.0)
    for _ in range(3):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    e1.synchronize()
    s = e0.elapsed_time(e1) / 1e3
    del a, b
    torch.cuda.empty_cache()
    return 2.0 * nbytes * reps / s


def synth_block(seed: int, n: int) -> bytes:
    rng = np.random.default_rng(seed)
    return bw.random_block(rng, n, 8, phased=False, missing_rate=0.01)


def write_file(path: str, n: int, p: int, threads: int) -> None:
    """bw.write, with the blocks generated and compressed on a thread pool"""
    def one(j):
        blk = synth_block(j, n)
        return blk, zlib.compress(blk, 1)
    import struct
    header = struct.pack("<III", 20, p, n) + b"bgen" + struct.pack("<I", 1 | (2 << 2))
    with open(path, "wb") as f, ThreadPoolExecutor(threads) as pool:
        f.write(struct.pack("<I", len(header)) + header)
        for j, (blk, z) in enumerate(pool.map(one, range(p))):
            meta = bw._s16(f"v{j}") + bw._s16(f"rs{j + 1}") + bw._s16("1") + struct.pack("<IH", 1000 + j, 2)
            meta += struct.pack("<I", 1) + b"A" + struct.pack("<I", 1) + b"G"
            f.write(meta + struct.pack("<II", len(z) + 4, len(blk)) + z)


def selection_case(lib, path, f, rows, cols, threads):
    """inflate / decode-kernel / end-to-end seconds of from_bgen(path, samples=rows, variants=cols)"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    n = f.n if rows is None else rows.shape[0]
    out = {"n": n, "p": int(cols.shape[0])}
    batches = f.variant_batches(cols)
    out["inflated_bytes"] = int(f.inflated_len[cols].sum())
    t0 = time.perf_counter()
    with ThreadPoolExecutor(threads) as pool:
        data = [f.inflate_variants(idx, pool) for idx in batches]
    out["inflate_s"] = time.perf_counter() - t0
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        h = C.c_void_p()
        _lib.check(lib.ihtb_geno_create_dosage16_empty(n, out["p"], 255, 1, C.byref(h)))
        if rows is not None:
            _lib.check(lib.ihtb_geno_select_bgen_samples(h, _lib.ptr(rows, C.c_int64), f.n))
        j = 0
        for idx, (buf, offs) in zip(batches, data):
            _lib.check(lib.ihtb_geno_load_bgen_columns(h, _lib.ptr(buf, C.c_uint8), _lib.ptr(offs, C.c_int64), j,
                                                       idx.shape[0], 2))
            j += idx.shape[0]
        torch.cuda.synchronize()
    lib.ihtb_geno_destroy(h)
    del data
    out["decode_kernel_s"] = sum(ev.device_time for ev in prof.events() if "k_bgen_decode" in ev.name) / 1e6
    t0 = time.perf_counter()
    x = m.B200DenseLinAlg.from_bgen(path, standardize=True, samples=rows, variants=cols)
    out["end_to_end_s"] = time.perf_counter() - t0
    ref_cols = cols[:32]
    codes, miss, _ = bgen.dosage_codes(path, rows=rows, variants=ref_cols)
    ref = m.B200DenseLinAlg.from_array(np.asfortranarray(np.where(miss, np.nan, codes / 255.0)), standardize=True)
    out["matches_twin"] = bool(np.array_equal(x.decode(0, n, 0, ref_cols.shape[0]).view(np.uint64),
                                              ref.decode().view(np.uint64)))
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--n", type=int, default=50000)
    ap.add_argument("--p", type=int, default=20000)
    ap.add_argument("--threads", type=int, default=min(32, os.cpu_count() or 1))
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert m.device_count() > 0, "bench_bgen needs a CUDA device"
    import torch
    from torch.profiler import ProfilerActivity, profile
    res = {"card": card(), "n": a.n, "p": a.p, "B": 8, "compression": "zlib", "host_threads": a.threads,
           "host_cpus": os.cpu_count()}
    lib = m.load()
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "bench.bgen")
        t0 = time.perf_counter()
        write_file(path, a.n, a.p, a.threads)
        res["write_s"] = time.perf_counter() - t0
        res["file_bytes"] = os.path.getsize(path)

        t0 = time.perf_counter()
        f = bgen.BgenFile(path)
        res["parse_s"] = time.perf_counter() - t0
        res["inflated_bytes"] = int(f.inflated_len.sum())

        batches = f.batches()
        t0 = time.perf_counter()
        with ThreadPoolExecutor(a.threads) as pool:
            data = [f.inflate(c0, c1, pool) for c0, c1 in batches]
        res["inflate_s"] = time.perf_counter() - t0
        res["inflate_GBps"] = res["inflated_bytes"] / res["inflate_s"] / 1e9
        res["batches"] = len(batches)

        def load_all():
            h = C.c_void_p()
            _lib.check(lib.ihtb_geno_create_dosage16_empty(a.n, a.p, 255, 1, C.byref(h)))
            torch.cuda.synchronize()
            t = time.perf_counter()
            for (c0, c1), (buf, offs) in zip(batches, data):
                _lib.check(lib.ihtb_geno_load_bgen_columns(h, _lib.ptr(buf, C.c_uint8), _lib.ptr(offs, C.c_int64),
                                                           c0, c1 - c0, 2))
            return h, time.perf_counter() - t

        h, warm = load_all()                               # module load, first pinned allocations
        lib.ihtb_geno_destroy(h)
        h, res["load_s"] = load_all()
        t0 = time.perf_counter()
        _lib.check(lib.ihtb_geno_finalize(h))
        res["finalize_s"] = time.perf_counter() - t0
        res["load_GBps_inflated"] = res["inflated_bytes"] / res["load_s"] / 1e9
        lib.ihtb_geno_destroy(h)

        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            h, _ = load_all()
            torch.cuda.synchronize()
        lib.ihtb_geno_destroy(h)
        dec_us = h2d_us = 0.0
        h2d_bytes = 0
        for ev in prof.events():
            if "k_bgen_decode" in ev.name:
                dec_us += ev.device_time
            elif "Memcpy HtoD" in ev.name:
                h2d_us += ev.device_time
        res["decode_kernel_s"] = dec_us / 1e6
        res["h2d_s"] = h2d_us / 1e6
        ld = -(-a.n // 256) * 256
        dec_bytes = res["inflated_bytes"] + 2 * ld * a.p
        res["decode_kernel_bytes"] = dec_bytes
        res["decode_kernel_GBps"] = dec_bytes / res["decode_kernel_s"] / 1e9
        res["h2d_GBps"] = res["inflated_bytes"] / res["h2d_s"] / 1e9 if h2d_us else None
        res["d2d_copy_GBps"] = copy_bandwidth(4 << 30) / 1e9
        res["decode_vs_copy"] = res["decode_kernel_GBps"] / res["d2d_copy_GBps"]
        del data

        t0 = time.perf_counter()
        x = m.B200DenseLinAlg.from_bgen(path, standardize=True)
        res["end_to_end_s"] = time.perf_counter() - t0
        res["end_to_end_GBps_inflated"] = res["inflated_bytes"] / res["end_to_end_s"] / 1e9
        # correctness: the first 64 variants against the host twin (standardized through a Float64 handle)
        codes = np.zeros((a.n, 64), dtype=np.int64)
        miss = np.zeros((a.n, 64), dtype=bool)
        for c in range(64):
            codes[:, c], miss[:, c], _ = bgen.decode_block(f._block(c), a.n)
        want = np.where(miss, np.nan, codes / 255.0)
        ref = m.B200DenseLinAlg.from_array(np.asfortranarray(want), standardize=True)
        res["matches_twin"] = bool(np.array_equal(x.decode(0, a.n, 0, 64).view(np.uint64), ref.decode().view(np.uint64)))
        del x, ref
        rng = np.random.default_rng(0)
        half = np.sort(rng.choice(a.n, size=a.n // 2, replace=False))
        every = np.arange(a.p, dtype=np.int64)
        cases = {"samples_50_sorted": (half, every), "samples_50_shuffled": (rng.permutation(half), every),
                 "variants_10": (None, np.sort(rng.choice(a.p, size=max(1, a.p // 10), replace=False)))}
        res["selection"] = {name: selection_case(lib, path, f, rows, cols, a.threads)
                            for name, (rows, cols) in cases.items()}
        f.close()
    stages = {k: res[k] for k in ("parse_s", "inflate_s", "load_s", "finalize_s")}
    res["slowest_stage"] = max(stages, key=stages.get)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fo:
            fo.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
