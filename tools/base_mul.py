#!/usr/bin/env python
"""Batched fixed-base scalar multiplication through the C ABI (cdl_g1_batch_scalar_mul_base): n scalars times
one base of G1.

Per n, medians of `reps` calls after one warm-up call:
  * GLV today: what a caller does without the call, cdl_g1_scalar_mul_affine on n uploaded copies of the base
    (scalar_stride = 1), host clock around the synchronous call; "dev" is the same kernel on device-resident
    copies and scalars (cdl_g1_scalar_mul_affine_device: launch and kernel only);
  * fresh base: the call on a base it has not seen (every call a new base), i.e. what the library does when
    nothing is cached: its GLV path below kBaseTableMinScalars, the cold table path (check, table build,
    multiply) from there on; host clock, and device busy time (CUDA events, cdl_engine_busy_ms);
  * warm table: the same base again, its table cached.
Every result is compared with the GLV reference.  The table build on its own is the median over n >= the
crossover constant of (fresh-base busy time - warm busy time); below that constant the cold table path is
(build + warm), and the crossover is the smallest n at which it is no slower than the GLV path.  The CPU
baseline is the repository's C port of the group law (oracle/c, one scalar multiplication per scalar) on all
host cores; it is not gnark."""
import argparse
import importlib
import os
import random
import statistics
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import bls12381 as b  # noqa: E402
from util import aff_enc, fr_enc  # noqa: E402


def crossover():
    import re
    src = open(os.path.join(ROOT, "go-curdleproofs_b200", "csrc", "capi_base_mul.cu")).read()
    return int(re.search(r"kBaseTableMinScalars\s*=\s*(\d+)", src).group(1))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = f"unavailable ({e})"
    return out


def cpu_baseline(n=8192):
    from oracle.cbackend import CBackend
    cb = CBackend(accelerate_keccak=False)
    rnd = random.Random(3)
    base = b.g1_mul(b.G1_GEN, rnd.randrange(1, b.R))
    ks = [rnd.randrange(1, b.R) for _ in range(n)]
    thr = os.cpu_count() or 1
    kch = [ks[i::thr] for i in range(thr)]
    t0 = time.perf_counter()
    with ThreadPoolExecutor(thr) as ex:  # ctypes drops the GIL for the C call
        list(ex.map(lambda k: cb.mul_batch([base] * len(k), k), kch))
    return n / (time.perf_counter() - t0), thr


def med(v):
    return statistics.median(v)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--lg", default="4-22", help="log2 n range, e.g. 4-22")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    lo, hi = (int(x) for x in a.lg.split("-"))
    X = crossover()
    pkg = importlib.import_module("go-curdleproofs_b200")
    ctx = pkg.Context(0)
    lines = []

    def emit(s=""):
        print(s, flush=True)
        lines.append(s)

    emit("# Batched fixed-base scalar multiplication, cdl_g1_batch_scalar_mul_base, affine results")
    emit(f"# card: {card()}   (name, power limit, max SM clock)")
    emit(f"# device: {ctx.device_info()}")
    emit(f"# kBaseTableMinScalars = {X}; {a.reps} timed calls per point after one warm-up call, medians; "
         "n = 2^22 results and scalars (528 MB) exceed the 126 MB L2")
    rnd = random.Random(1)
    nb = (hi - lo + 1) * (a.reps + 1) + 1
    bases_aff = ctx.g1_scalar_mul_affine(aff_enc(b.G1_GEN) * nb, b"".join(fr_enc(rnd.randrange(1, b.R)) for _ in range(nb)),
                                         broadcast=False)
    bases = [bases_aff[96 * i:96 * i + 96] for i in range(nb)]
    nxt = iter(bases)
    emit("")
    emit(f"{'n':>8} | {'GLV today ms':>12} {'dev ms':>8} | {'fresh-base path':>15} {'ms':>8} {'busy ms':>8} | "
         f"{'warm table ms':>13} {'busy ms':>8} | {'M/s GLV dev':>11} {'M/s warm busy':>13}")
    rows = []
    for lg in range(lo, hi + 1):
        n = 1 << lg
        sc = np.random.default_rng(lg).integers(0, 256, size=32 * n, dtype=np.uint8).tobytes()
        base = bases[-1]
        # GLV today, host buffers and device buffers
        glv, glv_dev = [], []
        d_in, d_s, d_out = ctx.dev_buffer(96 * n), ctx.dev_buffer(32 * n), ctx.dev_buffer(96 * n)
        d_in.upload(base * n)
        d_s.upload(sc)
        for it in range(a.reps + 1):
            t0 = time.perf_counter()
            ctx.g1_scalar_mul_affine(base * n, sc, broadcast=False)
            t1 = time.perf_counter()
            ctx.g1_scalar_mul_affine_device(d_in, d_s, n, False, d_out)
            t2 = time.perf_counter()
            if it:
                glv.append((t1 - t0) * 1e3)
                glv_dev.append((t2 - t1) * 1e3)
        for d in (d_in, d_s, d_out):
            d.close()
        # a fresh base every call, then the same base warm
        fresh, fresh_busy, warm, warm_busy = [], [], [], []
        path = None
        for it in range(a.reps + 1):
            bs = next(nxt)
            n0 = ctx.launch_count()
            ctx.engine_stats(reset=True)
            t0 = time.perf_counter()
            got = ctx.g1_batch_scalar_mul_base(bs, sc)
            t1 = time.perf_counter()
            busy = ctx.engine_busy_ms()
            path = "GLV" if ctx.launch_count() - n0 == 3 else "cold table"
            if it == 0:
                assert got == ctx.g1_scalar_mul_affine(bs * n, sc, broadcast=False), f"n={n}: differs from GLV today"
            if path == "GLV":  # build the table of bs (untimed) so that the next call is a warm one
                ctx.g1_batch_scalar_mul_base(bs, bytes(32 * X))
            ctx.engine_stats(reset=True)
            t2 = time.perf_counter()
            got2 = ctx.g1_batch_scalar_mul_base(bs, sc)
            t3 = time.perf_counter()
            wbusy = ctx.engine_busy_ms()
            assert got2 == got, f"n={n}: warm table result differs"
            if it:
                fresh.append((t1 - t0) * 1e3)
                fresh_busy.append(busy)
                warm.append((t3 - t2) * 1e3)
                warm_busy.append(wbusy)
        r = dict(n=n, glv=med(glv), glv_dev=med(glv_dev), path=path, fresh=med(fresh), fresh_busy=med(fresh_busy),
                 warm=med(warm), warm_busy=med(warm_busy))
        rows.append(r)
        emit(f"{n:>8} | {r['glv']:>12.3f} {r['glv_dev']:>8.3f} | {path:>15} {r['fresh']:>8.3f} {r['fresh_busy']:>8.3f} | "
             f"{r['warm']:>13.3f} {r['warm_busy']:>8.3f} | {n / r['glv_dev'] / 1e3:>11.2f} {n / r['warm_busy'] / 1e3:>13.2f}")
    emit("")
    cold = [r for r in rows if r["path"] == "cold table"]
    if cold:
        build = med([r["fresh_busy"] - r["warm_busy"] for r in cold])
        build_wall = med([r["fresh"] - r["warm"] for r in cold])
        emit(f"# table build on its own (check + window bases + k_fixed_build, 4.3 MB): {build:.3f} ms busy, "
             f"{build_wall:.3f} ms wall (median of fresh - warm over n >= {X})")
        emit("# cold table path against the GLV path, wall ms (cold below the constant = build + warm; GLV = the "
             "call's own GLV path below it, GLV today from it on):")
        cross = None
        for r in rows:
            c = r["fresh"] if r["path"] == "cold table" else build_wall + r["warm"]
            g = r["fresh"] if r["path"] == "GLV" else r["glv"]
            emit(f"#   n = {r['n']:>8}: cold table {c:9.3f}  GLV {g:9.3f}  {'table' if c <= g else 'GLV'}")
            if cross is None and c <= g:
                cross = r["n"]
            elif c > g:
                cross = None
        emit(f"# crossover: the cold table path is no slower than the GLV path from n = {cross} on "
             f"(kBaseTableMinScalars = {X})")
        emit("# warm table faster than GLV today (device time) at every n >= kBaseTableMinScalars: "
             f"{all(r['warm_busy'] < r['glv_dev'] for r in rows if r['n'] >= X)}")
    big = rows[-1]
    emit(f"# rates at n = {big['n']}: warm table {big['n'] / big['warm_busy'] / 1e3:.1f} M/s busy, "
         f"{big['n'] / big['warm'] / 1e3:.1f} M/s wall; GLV {big['n'] / big['glv_dev'] / 1e3:.1f} M/s device, "
         f"{big['n'] / big['glv'] / 1e3:.1f} M/s wall")
    cps, thr = cpu_baseline()
    emit(f"# CPU baseline: repository C port (oracle/c, not gnark), {thr} host threads, n = 8192: "
         f"{cps / 1e3:.1f} k scalar multiplications/s")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
