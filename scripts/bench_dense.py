"""Dense design-matrix measurements on one GPU, written as JSON to profiles/dense_sweep_<n>x<p>.json (or --out).

In one process: the card's name and power limit (read-only nvidia-smi query), the device-to-device copy bandwidth on a
buffer of >= 4 GB (torch, CUDA events), the dense X'v sweep alone (ihtb_sweep_bench, CUDA events, warmed up) for FP64 and
FP32 storage of an n x p matrix far larger than L2, its bytes/s as a fraction of that copy bandwidth, and the IHT
iterations per second of a device-resident Bernoulli k = 20 fit on the FP64 / FP32 matrices and on a PLINK handle of the
integer genotypes they blur.  The FP64 fit is checked against the dense oracle (support and iteration count).

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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=50000)
    ap.add_argument("--p", type=int, default=50000)
    ap.add_argument("--k", type=int, default=20)
    ap.add_argument("--copy-gb", type=float, default=4.0)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--no-oracle", action="store_true")
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
        out[f"sweep_{name}"] = {"bytes": nbytes, "ms_kernel": ms_k, "ms_total": ms_t,
                                "bytes_per_s_kernel": nbytes / (ms_k * 1e-3),
                                "fraction_of_copy_bandwidth": nbytes / (ms_k * 1e-3) / bw,
                                "fraction_of_copy_bandwidth_with_epilogue": nbytes / (ms_t * 1e-3) / bw}
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
    path = a.out or os.path.join(ROOT, "profiles", f"dense_sweep_{a.n}x{a.p}.json")
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
