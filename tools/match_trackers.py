#!/usr/bin/env python
"""Whisk tracker matching through the C ABI (cdl_whisk_match_trackers): T trackers against V keys.

Per V: the device path the library took, the call time (host clock around the synchronous call:
decode, copies and kernels), the kernel time (CUDA events, cdl_engine_stats class 1: key preparation,
table builds and matching), pairs/s, and the field products per pair each kernel's schedule executes
beside the SURVEY.md §8d algorithmic figure (3 193 per scalar multiplication).  Every timed call's
owners are checked against the construction.  The CPU baseline is the repository's C port of the
group law (oracle/c, 6 x 64-bit Montgomery, one scalar multiplication per pair) on all host cores;
it is not gnark.

The table-path time is fitted as a + b V per tracker (a: building one tracker's tables, b: one
pair); with the shared-scalar path's time per pair c, the paths cost the same at V = a / (c - b), the
crossover from which kMatchTableMinKeys (csrc/capi_whisk_match.cu) is set."""
import argparse
import importlib
import os
import random
import statistics
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import bls12381 as b  # noqa: E402
from util import aff_enc, fr_enc  # noqa: E402


def crossover():
    import re
    src = open(os.path.join(ROOT, "go-curdleproofs_b200", "csrc", "capi_whisk_match.cu")).read()
    return int(re.search(r"kMatchTableMinKeys\s*=\s*(\d+)", src).group(1))


# ---- executed field products (multiplications + squarings), counted from the kernels' schedules (g1.cuh)
DBL_JAC, ADD_MIXED_JAC, ADD_MIXED_H = 7, 11, 11  # jac_dbl, jac_add_mixed, jac_add_mixed_h
ADD_MIXED_XYZZ, DBL_XYZZ = 10, 9                 # xyzz_add_mixed, xyzz_dbl
INV = 210                                        # fp_inv, in products (fields.cuh)


def products_shared():
    """k_match_shared: jac_scalar_mul_glv + jac_eq_affine, per pair"""
    table = DBL_JAC + 6 * ADD_MIXED_H + 7 * 5              # {1..8}P at a common Z
    dbls = 31 * 4 * DBL_JAC
    adds = 64 * 15 / 16 * ADD_MIXED_JAC + 32 * 15 / 16    # a signed 4-bit digit is 0 with probability 1/16; phi: 1
    return table + dbls + adds + 1 + 2                    # back from the isomorphic curve; compare (x mismatch)


def products_table_pair():
    """k_match_table: 32 windows of 8 bits, a digit is 0 with probability 1/128"""
    return 32 * 127 / 128 * ADD_MIXED_XYZZ + 1


def products_table_build():
    """per tracker: k_match_windows (2^(8w) P by doubling), their normalisation (k_jac_to_affine, one inversion per
    point at these sizes), and k_fixed_build<8>: 32 windows x 8 segments of 16 entries, one inversion per segment"""
    tot = 31 * 8 * DBL_JAC + 32 * (INV + 5)
    for w in range(32):
        for s in range(8):
            e = 16 * s
            tot += (e.bit_length() * DBL_XYZZ + bin(e).count("1") * ADD_MIXED_XYZZ) if e else 0
            tot += 16 * (ADD_MIXED_XYZZ + 1) + INV + 16 * 6
    return tot


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = f"unavailable ({e})"
    return out


def cpu_baseline(n=4096):
    from oracle.cbackend import CBackend

    cb = CBackend(accelerate_keccak=False)
    rnd = random.Random(3)
    pts = cb.mul_batch([b.G1_GEN] * 64, [rnd.randrange(1, b.R) for _ in range(64)])
    ks = [rnd.randrange(1, b.R) for _ in range(n)]
    thr = os.cpu_count() or 1
    allp = (pts * (n // 64 + 1))[:n]
    chunks = [allp[i::thr] for i in range(thr)]
    kch = [ks[i::thr] for i in range(thr)]
    t0 = time.perf_counter()
    with ThreadPoolExecutor(thr) as ex:  # ctypes drops the GIL for the C call
        list(ex.map(cb.mul_batch, chunks, kch))
    return n / (time.perf_counter() - t0), thr


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--T", type=int, default=8192)
    ap.add_argument("--V", default="")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    X = crossover()
    Vs = [int(v) for v in a.V.split(",")] if a.V else sorted({1, 16, 128, X - 1, X, 4096, 16384})
    pkg = importlib.import_module("go-curdleproofs_b200")
    ctx = pkg.Context(0)
    lines = []

    def emit(s=""):
        print(s, flush=True)
        lines.append(s)

    emit(f"# Whisk tracker matching, cdl_whisk_match_trackers, T = {a.T} trackers")
    emit(f"# card: {card()}   (name, power limit, max SM clock)")
    emit(f"# device: {ctx.device_info()}")
    emit(f"# kMatchTableMinKeys = {X}; {a.reps} timed calls per point after one warm-up call; "
         "median [min, max]; the table path works through tiles of 256 trackers (96 MiB of tables)")
    T = a.T
    NK = max(Vs) + 4096
    rnd = random.Random(1)
    keys = [rnd.randrange(1, b.R) for _ in range(NK)]
    j = [rnd.randrange(NK) for _ in range(T)]
    rs = b"".join(fr_enc(rnd.randrange(1, b.R)) for _ in range(T))
    rG = ctx.g1_scalar_mul_affine(aff_enc(b.G1_GEN) * T, rs, broadcast=False)
    krG = ctx.g1_scalar_mul_affine(rG, b"".join(fr_enc(keys[x]) for x in j), broadcast=False)
    e1, e2 = ctx.g1_compress(rG), ctx.g1_compress(krG)
    trackers = b"".join(e1[48 * t:48 * t + 48] + e2[48 * t:48 * t + 48] for t in range(T))
    ps, pf, pb = products_shared(), products_table_pair(), products_table_build()
    emit(f"# executed products per pair: shared {ps:.0f}; table {pf:.0f} + build {pb:.0f} per tracker / V; §8d: 3193")
    emit("")
    emit(f"{'V':>6} {'path':>6} {'call ms':>24} {'kernel ms':>24} {'Mpairs/s kern':>14} {'Mpairs/s call':>14} "
         f"{'prod/pair':>10} {'§8d':>5}")
    fit_s, fit_f = [], []
    for V in Vs:
        kb = b"".join(fr_enc(k) for k in keys[:V])
        want = [x if x < V else -1 for x in j]
        call, kern = [], []
        path = None
        for it in range(a.reps + 1):
            n0 = ctx.launch_count()
            ctx.engine_stats(reset=True)
            t0 = time.perf_counter()
            owner, status = ctx.whisk_match_trackers(trackers, kb)
            t1 = time.perf_counter()
            ms = ctx.engine_stats()["elem_scalar_mul"]["ms"]
            nl = ctx.launch_count() - n0
            assert owner == want and status == [0] * T, f"V={V}: wrong owners"
            path = "shared" if nl == 3 else "table"
            if it:
                call.append((t1 - t0) * 1e3)
                kern.append(ms)
        km, cm = statistics.median(kern), statistics.median(call)
        prod = ps if path == "shared" else pf + pb / V
        (fit_s if path == "shared" else fit_f).append((V, km))
        emit(f"{V:>6} {path:>6} {cm:>9.2f} [{min(call):.2f}, {max(call):.2f}] {km:>9.2f} [{min(kern):.2f}, {max(kern):.2f}] "
             f"{T * V / km / 1e3:>14.2f} {T * V / cm / 1e3:>14.2f} {prod:>10.0f} {3193:>5}")
    emit("")
    if fit_s:
        big = [p for p in fit_s if p[0] >= 16] or fit_s
        c = statistics.median(km / (T * V) for V, km in big)
        emit(f"# shared-scalar path: {c * 1e6:.3f} ns per pair (median over V >= 16)")
    if len(fit_f) >= 2 and fit_s:
        n = len(fit_f)
        mv = sum(V for V, _ in fit_f) / n
        mt = sum(t for _, t in fit_f) / n
        slope = sum((V - mv) * (t - mt) for V, t in fit_f) / sum((V - mv) ** 2 for V, _ in fit_f)
        icpt = mt - slope * mv
        bpp, apt = slope / T, icpt / T
        emit(f"# table path: {apt * 1e3:.2f} us per tracker (tables) + {bpp * 1e6:.3f} ns per pair "
             f"(least squares over V = {[V for V, _ in fit_f]})")
        if c > bpp:
            emit(f"# paths cost the same at V = {apt / (c - bpp):.0f} keys")
    cps, thr = cpu_baseline()
    emit(f"# CPU baseline: repository C port (oracle/c, not gnark), {thr} host threads: {cps / 1e3:.1f} kpairs/s")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
