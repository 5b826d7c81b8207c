"""Dense design-matrix measurements on one GPU, written as JSON to profiles/dense_sweep_<n>x<p>.json (or --out).

In one process: the card's name and power limit (read-only nvidia-smi query), the device-to-device copy bandwidth on a
buffer of >= 4 GB (torch, CUDA events), the dense X'v sweep alone (ihtb_sweep_bench, CUDA events, warmed up) for FP64 and
FP32 storage of an n x p matrix far larger than L2, its bytes/s as a fraction of that copy bandwidth, and the IHT
iterations per second of a device-resident Bernoulli k = 20 fit on the FP64 / FP32 matrices and on a PLINK handle of the
integer genotypes they blur.  The FP64 fit is checked against the dense oracle (support and iteration count).

`fix16`: the same matrix quantised to the PLINK 2 dosage grid 1/16384 and held as 16-bit codes (from_dosages): the code
sweep alone, its bytes/s against the same copy bandwidth, fit iterations/s, and whether the fit equals the Float64-handle
fit of the quantised values bit for bit.  `fix16_configs1` (--big-p > 0): BASELINE configs[1]'s shape (n x big_p, default
50 000 x 500 000) as D = 1 codes of synth's integer genotypes, loaded in column blocks through
ihtb_geno_create_dosage16_empty / ihtb_geno_load_dense_columns so host memory stays bounded (Float64 storage of this
matrix, 200 GB, does not fit on the card): sweep time, fit iterations/s, and whether the fit equals the PLINK handle's
fit of the same genotypes.

Copy bandwidth counts the bytes read plus the bytes written; the sweep counts the matrix bytes it reads (n p sizeof(T)),
which is what bounds it."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import mendeliht_jl_b200 as m  # noqa: E402
from mendeliht_jl_b200 import _lib, synth  # noqa: E402
from oracle import iht  # noqa: E402
from oracle.dense import DenseLinAlgOracle  # noqa: E402

_LUT = np.array([[((b >> (2 * s)) & 3) for s in range(4)] for b in range(256)])
_DOS = np.array([0.0, np.nan, 1.0, 2.0])[_LUT]            # byte -> 4 dosages
_CODES = np.array([0, _lib.DOSAGE16_MISSING, 1, 2], dtype=np.uint16)[_LUT]     # byte -> 4 dosage codes (D = 1)


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clk = [t.strip() for t in out.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clk}


def copy_bandwidth(nbytes: int, reps: int = 20):
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
    torch.cuda.synchronize()
    s = e0.elapsed_time(e1) / 1e3 / reps
    del a, b
    torch.cuda.empty_cache()
    return 2 * nbytes / s, s


def matrices(n: int, p: int, seed: int):
    """Packed integer genotypes (ihtb_synth_host), and the n x p float64 dosages (F order) they give with a small
    deterministic continuous perturbation (imputed-dosage-like, no NaN)."""
    nb = (n + 3) // 4
    bed = np.empty((p, nb), dtype=np.uint8)
    _lib.check(m.load().ihtb_synth_host(n, p, 0, seed, 0.0, _lib.ptr(bed, C.c_uint8)))
    xt = np.empty((p, n))                                   # x.T in C order = x in F order
    wig = 0.15 * np.sin(np.arange(4099) * 0.7)
    for j in range(0, p, 2048):
        blk = _DOS[bed[j:j + 2048]].reshape(-1, nb * 4)[:, :n]
        rows = np.arange(blk.shape[0])[:, None] + j
        xt[j:j + 2048] = np.clip(blk + wig[(np.arange(n)[None, :] + 7 * rows) % 4099], 0.0, 2.0)
    return bed, xt.T


def sweep(g, warmup: int, reps: int):
    k, t = C.c_double(), C.c_double()
    _lib.check(m.load().ihtb_sweep_bench(g._h, m.SWEEP_FAST, warmup, reps, C.byref(k), C.byref(t)))
    return k.value, t.value


def fit_rate(y, g, z, k):
    m.fit_iht(y, g, z, k=k, d="Bernoulli", l="LogitLink", max_iter=3)       # warm-up: workspace, modules
    res = m.fit_iht(y, g, z, k=k, d="Bernoulli", l="LogitLink")
    return res, {"iter": int(res.iter), "fit_seconds": res.time, "iters_per_second": res.iter / res.time,
                 "sweep_seconds": res.sweep_seconds}


def sweep_entry(g, nbytes, ms_k, ms_t, bw):
    return {"bytes": nbytes, "ms_kernel": ms_k, "ms_total": ms_t, "bytes_per_s_kernel": nbytes / (ms_k * 1e-3),
            "fraction_of_copy_bandwidth": nbytes / (ms_k * 1e-3) / bw,
            "fraction_of_copy_bandwidth_with_epilogue": nbytes / (ms_t * 1e-3) / bw}


def same_fit(a, b):
    """bit-for-bit equality of two fits: iterations, support, backtracks, beta, c, logl"""
    return bool(a.iter == b.iter and np.array_equal(np.flatnonzero(a.beta), np.flatnonzero(b.beta))
                and [t[1] for t in a.trace] == [t[1] for t in b.trace] and a.beta.tobytes() == b.beta.tobytes()
                and a.c.tobytes() == b.c.tobytes() and float(a.logl) == float(b.logl))


def fix16_configs1(n, p, k, seed, reps, bw, block=2048):
    """D = 1 codes of synth's integer genotypes (no missing, as configs[1]), uploaded block by block"""
    lib = m.load()
    nb = (n + 3) // 4
    h = C.c_void_p()
    t0 = time.time()
    _lib.check(lib.ihtb_geno_create_dosage16_empty(n, p, 1, 1, C.byref(h)))
    g = m.B200DenseLinAlg(h, n, p, np.uint16, True, 1)
    bed = np.empty((block, nb), dtype=np.uint8)
    for j in range(0, p, block):
        c = min(block, p - j)
        _lib.check(lib.ihtb_synth_host(n, c, j, seed, 0.0, _lib.ptr(bed, C.c_uint8)))
        codes = _CODES[bed[:c]].reshape(c, nb * 4)        # C order [c, 4 nb] = column-major with ld = 4 nb >= n
        _lib.check(lib.ihtb_geno_load_dense_columns(h, C.c_void_p(codes.ctypes.data), nb * 4, j, c))
    _lib.check(lib.ihtb_geno_finalize(h))
    out = {"n": n, "p": p, "denominator": 1, "load_seconds": time.time() - t0}
    ms_k, ms_t = sweep(g, 3, reps)
    out["sweep"] = sweep_entry(g, g.sweep_stream_bytes()[0], ms_k, ms_t, bw)
    y, z, *_ = synth.simulate_response(seed + 1, n, p, k, "Bernoulli", n_cov=1, geno_seed=seed)
    res, out["fit"] = fit_rate(y, g, z, k)
    g.close()
    gp = m.B200SnpLinAlg.synthetic(n, p, seed)
    ref, out["fit_plink"] = fit_rate(y, gp, z, k)
    gp.close()
    out["fit_equals_plink"] = {
        "iter_match": int(res.iter) == int(ref.iter),
        "support_match": bool(np.array_equal(np.flatnonzero(res.beta), np.flatnonzero(ref.beta))),
        "backtracks_match": [t[1] for t in res.trace] == [t[1] for t in ref.trace],
        "max_rel_beta_diff": float(np.max(np.abs(res.beta - ref.beta)) / np.max(np.abs(ref.beta))),
        "rel_logl_diff": float(abs(res.logl - ref.logl) / abs(ref.logl))}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=50000)
    ap.add_argument("--p", type=int, default=50000)
    ap.add_argument("--k", type=int, default=20)
    ap.add_argument("--copy-gb", type=float, default=4.0)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--no-oracle", action="store_true")
    ap.add_argument("--den", type=int, default=16384)
    ap.add_argument("--big-p", type=int, default=0, help="columns of the configs[1]-shape FIX16 run (0: skip)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if m.device_count() < 1:
        raise SystemExit("bench_dense.py needs a CUDA device")
    out = {"n": a.n, "p": a.p, "k": a.k, "card": card()}
    bw, s = copy_bandwidth(int(a.copy_gb * (1 << 30)))
    out["copy"] = {"bytes": int(a.copy_gb * (1 << 30)), "seconds": s, "bytes_per_s_read_plus_write": bw}
    t0 = time.time()
    bed, x = matrices(a.n, a.p, 99)
    y, z, *_ = synth.simulate_response(99, a.n, a.p, a.k, "Bernoulli", n_cov=1)
    out["host_setup_seconds"] = time.time() - t0
    fits = {}
    for name, dt in (("f64", np.float64), ("f32", np.float32)):
        xd = x if dt == np.float64 else x.astype(np.float32, order="F")
        g = m.B200DenseLinAlg.from_array(xd)
        ms_k, ms_t = sweep(g, 3, a.reps)
        nbytes = g.sweep_stream_bytes()[0]
        out[f"sweep_{name}"] = sweep_entry(g, nbytes, ms_k, ms_t, bw)
        res, out[f"fit_{name}"] = fit_rate(y, g, z, a.k)
        fits[name] = res
        g.close()
        del xd
    gp = m.B200SnpLinAlg.from_bed_columns(bed, a.n)
    _, out["fit_plink_integer_genotypes"] = fit_rate(y, gp, z, a.k)
    gp.close()
    if not a.no_oracle:
        ref = iht.fit_iht(y, DenseLinAlgOracle(x), z, k=a.k, d="Bernoulli", l="LogitLink")
        r = fits["f64"]
        out["oracle_f64"] = {"iter": int(ref.iter), "iter_match": int(ref.iter) == int(r.iter),
                             "support_match": bool(np.array_equal(np.flatnonzero(ref.beta), np.flatnonzero(r.beta))),
                             "max_rel_beta_diff": float(np.max(np.abs(r.beta - ref.beta)) / np.max(np.abs(ref.beta)))}
    # FIX16: the matrix quantised in place (column blocks) to the grid 1/den, as codes and as Float64 of the same values
    for j in range(0, a.p, 2048):
        x[:, j:j + 2048] = np.rint(x[:, j:j + 2048] * a.den) / a.den
    g16 = m.B200DenseLinAlg.from_dosages(x, a.den)
    ms_k, ms_t = sweep(g16, 3, a.reps)
    fx = {"denominator": a.den, "sweep": sweep_entry(g16, g16.sweep_stream_bytes()[0], ms_k, ms_t, bw)}
    r16, fx["fit"] = fit_rate(y, g16, z, a.k)
    g16.close()
    g64 = m.B200DenseLinAlg.from_array(x)
    r64, fx["fit_f64_same_values"] = fit_rate(y, g64, z, a.k)
    g64.close()
    fx["fit_equals_f64_handle"] = same_fit(r16, r64)
    out["fix16"] = fx
    if a.big_p > 0:
        del x
        out["fix16_configs1"] = fix16_configs1(a.n, a.big_p, a.k, 2024, a.reps, bw)
    path = a.out or os.path.join(ROOT, "profiles", f"dense_sweep_{a.n}x{a.p}.json")
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
