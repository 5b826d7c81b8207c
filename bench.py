#!/usr/bin/env python
"""Benchmark of the IHT hot path (BASELINE.json metric: IHT iterations/s, with the X'r sweep against the HBM roofline).

Workload at N=1 = BASELINE.json configs[1]: synthetic PLINK n=50,000 x p=500,000, Bernoulli/LogitLink, k=20 `fit_iht`.
A "step" is one complete `fit_iht` (init_iht_indices! + the loop to convergence, reference defaults); the metric is
IHT iterations per second = (iterations summed over the K timed fits) / (device time of those fits).
  value : inputs (genotypes, y, z) resident in HBM, K x (ihtb_fit_init + ihtb_fit_run), CUDA events on the fit stream
  e2e   : K x the public `fit_iht(y, x, z)` call with HOST y / z and beta read back (the genotype operator `x` is
          constructed once from HOST .bed bytes before the timed region, like SnpLinAlg in the reference)
  roofline : the X'r sweep kernel timed alone with CUDA events (algorithmic bytes = p*ceil(n/4) + 8n + 24p)
  cpu_baseline : the CPU restatement of the reference (oracle/, C+OpenMP kernels) on the WHOLE workload, one fit; the
          same run is the parity check: `check.oracle_parity` = identical support / iterations / backtracks per
          iteration, beta and loglikelihood within 1e-6 relative of the oracle's (outside every timed region)
`--impl reference` times that CPU restatement as the reference arm (Julia is not installed in this image).
At N>1 the SNP columns are sharded over the ranks (weak scaling: p = 500,000 columns per GPU); at N=8 the line also
carries `north_star`: BASELINE configs[4] (n=500k x p=1M, Normal, k=100, 10 covariates) strong-sharded over the 8 GPUs.
`--dump-outputs DIR` writes the model of the last timed `value` fit (`--impl reference`: of its one fit) to
DIR/<name>.npy in float64: the inputs are seeded, so two builds run with the same arguments can be compared output for
output.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np

N_SAMPLES = int(os.environ.get("IHTB_BENCH_N", 50_000))      # overrides are for debugging only
P_PER_GPU = int(os.environ.get("IHTB_BENCH_P", 500_000))
K_SPARSITY = 20
SEED = 2024
DIST, LINK = "Bernoulli", "LogitLink"
CPU_SAMPLE_COLS = 500_000     # the reference arm at N>1 samples the first 500k columns of the N x 500k problem
DTYPE = "f64 (sweep: f32 LUT partials per slab of 640 samples (512 without the ternary copy), f64 across slabs; top-k candidates re-scored in f64)"
PARITY_RTOL = 1e-6
# One unit of work = one IHT iteration over one 50k x 500k shard.  At N=1 that is an IHT iteration of configs[1]; at N>1
# (weak scaling, one shard per GPU) the job performs N shard-iterations per global iteration.
UNIT = "iterations/s (x 500k-SNP shards)"
DUMP_BYTES = 64 << 20


def sweep_bytes(n, p):
    return p * ((n + 3) // 4) + 8 * n + 24 * p


def dump_outputs(out_dir, res, beta, c):
    """The model a caller of the timed fit receives: the dense beta, c, logl, iter and sigma_g, one float64 .npy each.
    A beta larger than half of DUMP_BYTES (only at IHTB_BENCH_P sizes) is stored at a fixed, seeded sample of positions
    joined with its support; beta_index.npy holds those positions."""
    beta = np.asarray(beta, dtype=np.float64)
    out = {"beta": beta, "c": c, "logl": [res.logl], "iter": [res.iter], "sigma_g": [res.sigma_g]}
    if beta.nbytes > DUMP_BYTES // 2:
        idx = np.random.default_rng(SEED).choice(beta.size, DUMP_BYTES // 32, replace=False)
        idx = np.union1d(idx, np.flatnonzero(beta))
        out["beta"], out["beta_index"] = beta[idx], idx
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = max([int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()] or [0])
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for i, nm in enumerate(names):
                if len(r) > 2 + i and r[2 + i].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_port_fit(n, p_full, k, bed=None, steps=1, warmup=0):
    """CPU restatement of the reference (oracle/) on this workload.  p_full <= CPU_SAMPLE_COLS: the whole problem;
    otherwise the first CPU_SAMPLE_COLS columns with their own simulated response, scaled by sample/p_full (an IHT
    iteration is dominated by the O(n p) sweep, reference test/fit_profile.ipynb: 77-87 %).
    Returns (iterations/s, threads, sample text, ms per fit, last oracle result)."""
    from oracle import cpu as ocpu
    from oracle import glm as oglm
    from oracle import iht as oiht
    from mendeliht_jl_b200 import synth
    ps = min(CPU_SAMPLE_COLS, p_full)
    if bed is None or bed.shape[0] != ps:
        bed = ocpu.synth_columns(SEED, n, 0, ps)
    x = ocpu.PackedSnpLinAlgCPU(bed, n)
    y, z, _, _, _ = synth.simulate_response(SEED + 1, n, ps, k, DIST, geno_seed=SEED)
    tot_it, tot_t, res = 0, 0.0, None
    for s in range(warmup + steps):
        t0 = time.perf_counter()
        res = oiht.fit_iht(y, x, z, k=k, d=oglm.BERNOULLI, l=oglm.LOGIT)
        dt = time.perf_counter() - t0
        if s >= warmup:
            tot_it += res.iter
            tot_t += dt
    v_sample = tot_it / tot_t
    v = v_sample * ps / p_full
    what = "the whole workload" if ps == p_full else f"the first {ps} of {p_full} columns (scaled by {ps}/{p_full})"
    sample = (f"fit_iht on n={n} x {what} ({DIST}, k={k}), {steps} fit(s), {tot_it} iterations in {tot_t:.2f}s "
              f"= {v_sample:.2f} it/s on {x.threads} threads")
    return v, x.threads, sample, tot_t / max(steps, 1) * 1e3, res


def parity_report(res, ref):
    """Our fit against the oracle's on the same inputs (SURVEY.md 8c bar: support / iterations exact, values 1e-6)."""
    nz, rz = np.flatnonzero(res.beta), np.flatnonzero(ref.beta)
    same_supp = bool(np.array_equal(nz, rz))
    bt, rbt = [t[1] for t in res.trace], list(ref.trace.backtracks)
    lg, rlg = np.array([t[0] for t in res.trace]), np.asarray(ref.trace.logl, dtype=np.float64)
    beta_err = None
    if same_supp and nz.size:
        beta_err = float(np.max(np.abs(res.beta[nz] - ref.beta[nz]) / np.abs(ref.beta[nz])))
    c_err = float(np.max(np.abs(res.c - ref.c) / np.maximum(np.abs(ref.c), 1e-12)))
    logl_err = float(abs(res.logl - ref.logl) / abs(ref.logl))
    trace_err = float(np.max(np.abs(lg - rlg) / np.abs(rlg))) if lg.shape == rlg.shape and lg.size else None
    ok = (same_supp and int(res.iter) == int(ref.iter) and bt == rbt and beta_err is not None
          and beta_err <= PARITY_RTOL and c_err <= PARITY_RTOL and logl_err <= PARITY_RTOL
          and trace_err is not None and trace_err <= PARITY_RTOL)
    return {"oracle_parity": bool(ok), "support_identical": same_supp, "iterations": int(res.iter),
            "oracle_iterations": int(ref.iter), "backtracks_identical": bt == rbt, "backtracks": int(sum(bt)),
            "max_rel_err_beta": beta_err, "max_rel_err_c": c_err, "rel_err_logl": logl_err,
            "max_rel_err_logl_trace": trace_err, "rtol": PARITY_RTOL,
            "oracle": "oracle.iht.fit_iht over oracle.cpu.PackedSnpLinAlgCPU (C+OpenMP) on the same host .bed bytes"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # one whole-workload fit at N=1 (about 40 s on 16 cores); at N>1 a 500k-column sample of the N x 500k problem
    v, threads, sample, ms, ref = cpu_port_fit(N_SAMPLES, P_PER_GPU * args.gpus, K_SPARSITY, steps=1, warmup=0)
    assert threads > 1 or (os.cpu_count() or 1) == 1, "the CPU reference arm must use all host cores"
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, ref, ref.beta, ref.c)
    line = {
        "impl": "reference", "metric": "iht_iterations_per_sec", "value": v * args.gpus, "unit": UNIT,
        "global_iterations_per_sec": v,
        "n_gpus": args.gpus, "steps": 1, "warmup": 0, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": v * args.gpus, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": v * args.gpus, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "Julia/SnpArrays.jl cannot run in this image; this is the C+OpenMP/numpy restatement of the reference "
                "algorithm (oracle/) on all host cores; one step = one whole fit_iht (requested steps/warmup are "
                "clamped to 1/0 so the run stays within minutes)",
    }
    print(json.dumps(line))


def workload_config(n_gpus):
    return {"workload": f"BASELINE configs[1]: synthetic PLINK n={N_SAMPLES} p={P_PER_GPU * n_gpus} "
                        f"{DIST}/{LINK} k={K_SPARSITY} fit_iht" + (f", SNP columns sharded over {n_gpus} GPUs"
                                                                   if n_gpus > 1 else ""),
            "n": N_SAMPLES, "p": P_PER_GPU * n_gpus, "k": K_SPARSITY, "dist": DIST, "link": LINK, "seed": SEED,
            "sweep_mode": "FAST (FP32 LUT partials, FP64 re-scoring of top-k candidates)",
            "l2_policy": "inputs larger than L2 (6.25 GB packed genotypes per sweep vs 126 MB L2)"}


def run_ours(args):
    import mendeliht_jl_b200 as m
    from mendeliht_jl_b200 import synth
    import ctypes as C

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        from mendeliht_jl_b200 import parallel
        return parallel.bench_sharded(args, rank, world, local_rank, globals())

    assert m.device_count() > 0, "bench.py needs a CUDA device (no CPU fallback)"
    lib = m.load()
    m._lib.check(lib.ihtb_set_device(0))
    n, p, k = N_SAMPLES, P_PER_GPU, K_SPARSITY

    # ---- inputs: HOST .bed bytes -> device genotype operator (constructed once, like SnpLinAlg) ----
    t0 = time.perf_counter()
    bed = np.empty((p, (n + 3) // 4), dtype=np.uint8)
    m._lib.check(lib.ihtb_synth_host(n, p, 0, SEED, 0.0, bed.ctypes.data_as(C.POINTER(C.c_uint8))))
    t_gen = time.perf_counter() - t0
    t0 = time.perf_counter()
    g = m.B200SnpLinAlg.from_bed_columns(bed, n)
    t_upload = time.perf_counter() - t0
    if args.no_cpu_baseline:
        del bed
    y, z, true_idx, true_beta, _ = synth.simulate_response(SEED + 1, n, p, k, DIST, geno_seed=SEED)

    launches0 = m.launch_count()
    clocks = ClockSampler(0)

    # ---- value: device-resident fits ----
    v = m.IHTVariable(g, z, y, k, DIST, LINK)
    for _ in range(args.warmup):
        v.init_iht_indices(None)
        v.fit(trace_cap=0)
    clocks.start()
    ms = C.c_double(0.0)
    m._lib.check(lib.ihtb_fit_timer(v._h, 0, None))
    l_before = m.launch_count()
    iters = sweeps = 0
    sweep_s = 0.0
    for _ in range(args.steps):
        v.init_iht_indices(None)
        res, _ = v.fit(trace_cap=0)
        iters += int(res.iter); sweeps += int(res.n_sweeps); sweep_s += res.sweep_seconds
    m._lib.check(lib.ihtb_fit_timer(v._h, 1, C.byref(ms)))
    l_timed = m.launch_count() - l_before
    t_value = ms.value * 1e-3
    ph = (C.c_double * 4)()
    m._lib.check(lib.ihtb_fit_phase_times(v._h, ph))
    phases = {k: ph[i] / max(iters + args.warmup * (iters // max(args.steps, 1)), 1) * 1e3
              for i, k in enumerate(["stepsize_ms", "gradstep_ms", "xb_glm_ms", "score_sweep_ms"])}
    if args.dump_outputs:
        beta_v, c_v, _, _ = v.get()
        dump_outputs(args.dump_outputs, res, beta_v, c_v)
    v.close()

    # ---- e2e: public API, host buffers in / out every step ----
    for _ in range(min(args.warmup, 1)):
        m.fit_iht(y, g, z, k=k, d=DIST, l=LINK)
    t0 = time.perf_counter()
    e_iters = 0
    for _ in range(args.steps):
        r = m.fit_iht(y, g, z, k=k, d=DIST, l=LINK)
        e_iters += r.iter
    t_e2e = time.perf_counter() - t0
    beta, c = r.beta, r.c
    clk = clocks.stop()

    # ---- roofline: the sweep kernel timed alone ----
    mk, mt = C.c_double(0.0), C.c_double(0.0)
    m._lib.check(lib.ihtb_sweep_bench(g._h, m.SWEEP_FAST, 3, 20, C.byref(mk), C.byref(mt)))
    peak, peak_src = measured_peak()
    abytes = sweep_bytes(n, p)
    achieved = abytes / (mk.value * 1e-3) / 1e9
    # what the kernel physically streams: the handle's ternary copy packs five dosages per byte (p * ceil(n/640) * 128 B)
    stream_b, ternary = g.sweep_stream_bytes()
    sbytes = stream_b + 8 * n + 24 * p
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "sweep_traffic.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            if bool(tj.get("ternary", False)) == ternary:       # an ncu capture of THIS kernel variant only
                traffic = tj.get("dram_bytes_per_launch")
                traffic_src = "static: " + tj.get("source", "profiles/sweep_traffic.json") + " (ncu cannot run inside a timed bench)"
        except Exception:
            traffic = None

    # ---- CPU baseline = the oracle on the whole workload, which is also the parity check (outside every timed region) ----
    cpu = None
    nz = np.flatnonzero(beta)
    check = {"support_size": int(nz.size), "true_positives": int(np.intersect1d(nz, true_idx).size),
             "iterations": iters // args.steps, "oracle_parity": None}
    if not args.no_cpu_baseline:
        cv, threads, sample, _, ref = cpu_port_fit(n, p, k, bed=bed, steps=1, warmup=0)
        del bed
        cpu = {"value": cv, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample}
        check.update(parity_report(r, ref))

    line = {
        "metric": "iht_iterations_per_sec", "value": iters / t_value, "unit": UNIT, "n_gpus": 1,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_value / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
        "config": workload_config(1),
        "iterations_per_fit": iters / args.steps, "sweeps_per_fit": sweeps / args.steps,
        "sweep_ms_in_fit": sweep_s / max(sweeps - args.steps, 1) * 1e3,
        "sweep_share_of_step": sweep_s / t_value, "host_phase_ms_per_iteration": phases,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "kernel": "k_sweep_lut",
                     "algorithmic_bytes_per_launch": abytes, "kernel_ms": mk.value,
                     "streamed_bytes_per_launch": sbytes, "streamed_gbs": sbytes / (mk.value * 1e-3) / 1e9,
                     "streamed_frac": sbytes / (mk.value * 1e-3) / 1e9 / peak,
                     "stream_encoding": ("ternary copy: 5 dosages per byte, lossless (missing -> CSR correction); `achieved` "
                                         "counts the PLINK 2-bit bytes of SURVEY 8d, `streamed_*` what the kernel reads")
                                        if ternary else "PLINK 2-bit tiles",
                     "sweep_with_epilogue_ms": mt.value, "sweep_with_epilogue_gbs": abytes / (mt.value * 1e-3) / 1e9},
        "e2e": {"value": e_iters / t_e2e, "unit": UNIT,
                "h2d_bytes_per_step": int(y.nbytes + z.nbytes), "d2h_bytes_per_step": int(16 * np.count_nonzero(beta) + c.nbytes + 8),
                "ms_per_step": t_e2e / args.steps * 1e3,
                "note": "fit_iht(y, x, z) with host y/z; the model comes back as k (index, value) pairs + c + logl (the "
                        "dense beta of IHTResult is built on first access); x (genotype operator) built once from "
                        "host .bed bytes before the timed region",
                "geno_host_generate_s": t_gen, "geno_create_from_host_s": t_upload,
                "geno_h2d_bytes": int(p * ((n + 3) // 4))},
        "gpu_launches": int(l_timed),
        "clocks": clk,
        "cpu_baseline": cpu,
        "check": check,
    }
    print(json.dumps(line))
    if check["oracle_parity"] is False:
        print("bench.py: the CUDA fit does not match the CPU oracle: " + json.dumps(check), file=sys.stderr)
        sys.exit(3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the model of the last timed fit to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
