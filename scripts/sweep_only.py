"""Runs the X'r sweep alone on a device-generated matrix (for ncu captures and quick kernel timing).
usage: sweep_only.py [n p reps mode]   mode 0 = FAST, 1 = EXACT, 2 = PAIR (two right-hand sides per pass)
env:   IHTB_TERN=0|1 (ternary copy of the tiles: default on when memory allows)"""
import ctypes as C
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mendeliht_jl_b200 as m

n = int(sys.argv[1]) if len(sys.argv) > 1 else 50000
p = int(sys.argv[2]) if len(sys.argv) > 2 else 500000
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 5
mode = int(sys.argv[4]) if len(sys.argv) > 4 else 0
g = m.B200SnpLinAlg.synthetic(n, p, 2024)
mk, mt = C.c_double(0), C.c_double(0)
m._lib.check(m.load().ihtb_sweep_bench(g._h, mode, 2, reps, C.byref(mk), C.byref(mt)))
b = p * ((n + 3) // 4) + 8 * n + 24 * p
rhs = 2 if mode == 2 else 1
print(json.dumps({"n": n, "p": p, "mode": ["FAST", "EXACT", "PAIR"][mode],
                  "ternary": g.sweep_stream_bytes()[1], "streamed_GBs": round((g.sweep_stream_bytes()[0] + 8 * n + 24 * p) / mk.value / 1e6, 1)
                  if mode != 1 else None, "rhs_per_pass": rhs,
                  "kernel_ms": round(mk.value, 4), "total_ms": round(mt.value, 4),
                  "kernel_GBs_matrix": round(b / mk.value / 1e6, 1), "total_GBs_matrix": round(b / mt.value / 1e6, 1),
                  "kernel_ms_per_rhs": round(mk.value / rhs, 4), "frac_of_6552": round(b / mk.value / 1e6 / 6552, 4)}))
