#!/usr/bin/env python
"""Minimum block of the elementwise point calls that a multi-device context splits: one-GPU sweep.

For each of cdl_g1_decompress, cdl_g1_compress, cdl_g1_batch_to_affine, cdl_g1_scalar_mul_affine (per-point
scalars) and cdl_g1_fold on one device (Context(0)), at n = 1 and at powers of two:
  wall    median host-clock time of --reps calls after one warm-up call (uploads, launch, wait, download);
  kernel  the call's kernel time per call: torch.profiler's CUDA activity (kernels only, no copies) over --reps
          calls, in a run of its own.
The fixed cost of one more slot is taken as F = wall(1) - kernel(1): a lane's uploads, launch, wait and download
of a one-point call, without its kernel.  Cutting 2b points into two blocks of b on two GPUs takes
saved(b) = kernel(2b) - kernel(b) of kernel time off the call (the kernels are latency-bound up to several
thousand points, so a block's kernel time alone says nothing); the call's minimum block is the smallest b of the
sweep with saved(b) >= F.  Inputs: a set of 2^16 points a_i * G (Jacobian with random Z for batch_to_affine),
repeated.  The card's name and power limit are read in the same call."""
import argparse
import os
import random
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import bls12381 as b  # noqa: E402
from util import aff_enc  # noqa: E402

SET = 1 << 16
CALLS = ["decompress", "compress", "batch_to_affine", "scalar_mul_affine", "fold"]


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return f"unavailable ({e})"


def inputs(ctx):
    rnd = random.Random(12)
    sc = b"".join(rnd.randrange(1, b.R).to_bytes(32, "little") for _ in range(SET))
    pts = ctx.g1_scalar_mul_affine(aff_enc(b.G1_GEN) * SET, sc, broadcast=False)
    enc = ctx.g1_compress(pts)
    # (x z^2, y z^3, z) in Montgomery form: x_mont * z^2, y_mont * z^3, z * 2^384
    P, Rm = b.P, pow(2, 384, b.P)
    jac = bytearray()
    for i in range(SET):
        x = int.from_bytes(pts[96 * i:96 * i + 48], "little")
        y = int.from_bytes(pts[96 * i + 48:96 * i + 96], "little")
        z = rnd.randrange(1, P)
        z2 = z * z % P
        jac += (x * z2 % P).to_bytes(48, "little") + (y * z2 * z % P).to_bytes(48, "little") + \
            (z * Rm % P).to_bytes(48, "little")
    return pts, sc, enc, bytes(jac)


def rep(data, unit, n):
    return (data * -(-n // SET))[:unit * n]


def call_fn(ctx, name, base, n):
    pts, sc, enc, jac = base
    if name == "decompress":
        e = rep(enc, 48, n)
        return lambda: ctx.g1_decompress(e)
    if name == "compress":
        p = rep(pts, 96, n)
        return lambda: ctx.g1_compress(p)
    if name == "batch_to_affine":
        j = rep(jac, 144, n)
        return lambda: ctx.g1_batch_to_affine(j)
    if name == "scalar_mul_affine":
        p, s = rep(pts, 96, n), rep(sc, 32, n)
        return lambda: ctx.g1_scalar_mul_affine(p, s, broadcast=False)
    L, R = rep(pts, 96, n), rep(pts[96:] + pts[:96], 96, n)
    return lambda: ctx.g1_fold(L, R, sc[:32])


def kernel_us(fn, reps):
    """kernel time per call (µs): every CUDA kernel the profiler records over `reps` calls, copies excluded"""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
    tot = 0.0
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA and not e.name.startswith(("Memcpy", "Memset")):
            tot += e.device_time
    return tot / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--max-log2", type=int, default=22)
    ap.add_argument("--calls", nargs="+", choices=CALLS, default=CALLS)
    ap.add_argument("--out", default="", help="also write the report to this file")
    args = ap.parse_args()
    import importlib

    import torch

    if torch.cuda.device_count() < 1:
        raise SystemExit("no CUDA device")
    torch.zeros(1, device="cuda")
    pkg = importlib.import_module("go-curdleproofs_b200")
    ctx = pkg.Context(0)
    base = inputs(ctx)
    lines = [f"# tools/primitive_sweep.py --reps {args.reps} --calls {' '.join(args.calls)}  (host cores: {os.cpu_count()})",
             "# nvidia-smi index, name, power.limit, clocks.max.sm:", "# " + card().replace("\n", "\n# "),
             "# wall: median host-clock ms per call; kernel: profiler kernel ms per call;",
             "# saved(n) = kernel(2n) - kernel(n); F = wall(1) - kernel(1)"]
    out = open(args.out, "w") if args.out else None

    def emit(s):
        print(s, flush=True)
        if out:
            out.write(s + "\n")
            out.flush()

    for s in lines:
        emit(s)
    sizes = [1] + [1 << k for k in range(8, args.max_log2 + 1)]
    for name in args.calls:
        wall, kern = {}, {}
        for n in sizes:
            fn = call_fn(ctx, name, base, n)
            fn()
            ts = []
            for _ in range(args.reps):
                t0 = time.perf_counter()
                fn()
                ts.append(time.perf_counter() - t0)
            wall[n] = statistics.median(ts) * 1e3
            kern[n] = kernel_us(fn, args.reps) / 1e3
        F = wall[1] - kern[1]
        kmin = None
        for n in sizes:
            saved = kern[2 * n] - kern[n] if n > 1 and 2 * n in kern else None
            if kmin is None and saved is not None and saved >= F:
                kmin = n
            emit(f"  {name:18s} n={n:>9d}  wall {wall[n]:9.3f} ms  kernel {kern[n]:9.4f} ms  saved(n) " +
                 (f"{saved:9.4f} ms" if saved is not None else "        -"))
        emit(f"  {name:18s} F = {F:.4f} ms  minimum block = {kmin if kmin else 'beyond the sweep'}")
    ctx.close()


if __name__ == "__main__":
    main()
