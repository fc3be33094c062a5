#!/usr/bin/env python
"""Whisk registration through the C ABI: cdl_whisk_generate_registration_batch against the five-call composition
a caller makes without it, for B validators on one GPU.

  composition: draw r from every Rand (one cdl_rand_get_frs call per validator, not timed), rG = r*G with
  cdl_g1_batch_scalar_mul_base, krG = k*rG with cdl_g1_scalar_mul_affine and cdl_g1_compress, kG = k*G with
  cdl_g1_batch_scalar_mul_base, then cdl_whisk_generate_tracker_proof_batch;
  registration: the one call (r and the blinder drawn inside it, five multiples of G per validator).

Per B and per state of G's fixed-base table - warm (cached) or cold (evicted by four other bases just before the
call) - the median of `reps` timed calls after one warm-up call of each: wall time (host clock around the
synchronous calls) and device busy time from the library's CUDA events:
  registration: cdl_engine_busy_ms over the call, which times every kernel chain it launches (the launches per
  call are printed beside it);
  composition: cdl_engine_busy_ms over its three engine calls (both cdl_g1_batch_scalar_mul_base calls and
  cdl_whisk_generate_tracker_proof_batch) plus the GLV kernel of its k*rG step, timed as
  cdl_g1_scalar_mul_affine_device on device-resident copies of the same inputs (host clock around the
  synchronous call: one launch and the kernel).  The one k_compress launch of its cdl_g1_compress step is not
  counted, so the composition's busy time is short by that kernel and long by one launch latency.
The first call at every B checks that both give the same bytes, statuses and Rand positions."""
import argparse
import importlib
import os
import random
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import bls12381 as b  # noqa: E402
from util import aff_enc  # noqa: E402

GEN = aff_enc(b.G1_GEN)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = f"unavailable ({e})"
    return out


def table_min_scalars():
    import re
    src = open(os.path.join(ROOT, "go-curdleproofs_b200", "csrc", "capi_base_mul.cu")).read()
    return int(re.search(r"kBaseTableMinScalars\s*=\s*(\d+)", src).group(1))


def draw_r(rands):
    return b"".join(r.get_fr() for r in rands)


def compose(ctx, ks, rs, rands):
    B = len(rands)
    rG_aff, rG = ctx.g1_batch_scalar_mul_base(GEN, rs, affine=True, compressed=True)
    krG = ctx.g1_compress(ctx.g1_scalar_mul_affine(rG_aff, ks, broadcast=False))
    k_comms = ctx.g1_batch_scalar_mul_base(GEN, ks, affine=False, compressed=True)
    trackers = np.concatenate([np.frombuffer(rG, np.uint8).reshape(B, 48), np.frombuffer(krG, np.uint8).reshape(B, 48)],
                              axis=1).tobytes()
    proofs, status = ctx.whisk_generate_tracker_proof_batch(trackers, ks, rands)
    return trackers, k_comms, proofs, status


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--lg", default="10-20", help="log2 B range, e.g. 10-20")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    lo, hi = (int(x) for x in a.lg.split("-"))
    X = table_min_scalars()
    pkg = importlib.import_module("go-curdleproofs_b200")
    ctx = pkg.Context(0)
    lines = []

    def emit(s=""):
        print(s, flush=True)
        lines.append(s)

    gpu = card()
    tag = ", ".join(gpu.split(", ")[:2])  # name and power limit, on every result line
    emit("# Whisk registration: cdl_whisk_generate_registration_batch against the five-call composition "
         "(r*G, k*rG, k*G, cdl_whisk_generate_tracker_proof_batch)")
    emit(f"# card: {gpu}   (name, power limit, max SM clock)")
    emit(f"# device: {ctx.device_info()}")
    emit(f"# kBaseTableMinScalars = {X}; {a.reps} timed calls per point after one warm-up call, medians; wall = host "
         "clock around the synchronous calls (the composition's per-validator r draws excluded); busy = CUDA-event "
         "busy time (composition: its engine calls + its GLV k*rG kernel, k_compress not counted); launches = "
         "kernels per registration call; cold = G's table evicted by four other bases before each call")
    rnd = random.Random(1)
    others = [aff_enc(b.g1_mul(b.G1_GEN, rnd.randrange(1, b.R))) for _ in range(4)]
    zeros = bytes(32 * X)

    def set_state(state):
        if state == "warm":
            ctx.g1_batch_scalar_mul_base(GEN, zeros, affine=False, compressed=True)
        else:
            for o in others:
                ctx.g1_batch_scalar_mul_base(o, zeros, affine=False, compressed=True)

    emit("")
    emit(f"{'B':>8} {'G table':>7} | {'register ms':>11} {'busy ms':>8} {'launches':>8} | {'compose ms':>10} {'busy ms':>8} | "
         f"{'wall x':>6} {'busy x':>6} | {'register k/s':>12} {'compose k/s':>11} | card")
    med = statistics.median
    rows = []
    for lg in range(lo, hi + 1):
        B = 1 << lg
        ks = np.random.default_rng(lg).integers(0, 256, size=32 * B, dtype=np.uint8).tobytes()
        rands = [pkg.Rand(1_000_000 * lg + i) for i in range(B)]
        # the check: twin Rands, both ways
        twins = [pkg.Rand(1_000_000 * lg + i) for i in range(B)]
        got = ctx.whisk_generate_registration_batch(ks, rands)
        want = compose(ctx, ks, draw_r(twins), twins)
        assert got[3] == want[3] == [0] * B, f"B={B}: statuses"
        assert got[:3] == want[:3], f"B={B}: bytes differ from the composition"
        assert [r.get_fr() for r in rands[:64]] == [r.get_fr() for r in twins[:64]], f"B={B}: Rand positions"
        del twins
        # the composition's k*rG kernel on device-resident copies of its inputs
        rG_aff = ctx.g1_batch_scalar_mul_base(GEN, draw_r(rands))
        d_in, d_s, d_out = ctx.dev_buffer(96 * B), ctx.dev_buffer(32 * B), ctx.dev_buffer(96 * B)
        d_in.upload(rG_aff)
        d_s.upload(ks)
        glv = []
        for it in range(a.reps + 1):
            t0 = time.perf_counter()
            ctx.g1_scalar_mul_affine_device(d_in, d_s, B, False, d_out)
            if it:
                glv.append((time.perf_counter() - t0) * 1e3)
        assert d_out.download(96 * B) == ctx.g1_scalar_mul_affine(rG_aff, ks, broadcast=False), f"B={B}: k*rG"
        for d in (d_in, d_s, d_out):
            d.close()
        for state in ("warm", "cold"):
            reg, comp, reg_busy, comp_busy, launches = [], [], [], [], set()
            for it in range(a.reps + 1):
                set_state(state)
                ctx.engine_stats(reset=True)
                n0 = ctx.launch_count()
                t0 = time.perf_counter()
                ctx.whisk_generate_registration_batch(ks, rands)
                t1 = time.perf_counter()
                rb = ctx.engine_busy_ms()
                nl = ctx.launch_count() - n0
                set_state(state)
                rs = draw_r(rands)
                ctx.engine_stats(reset=True)
                t2 = time.perf_counter()
                compose(ctx, ks, rs, rands)
                t3 = time.perf_counter()
                cb = ctx.engine_busy_ms()
                if it:
                    reg.append((t1 - t0) * 1e3)
                    comp.append((t3 - t2) * 1e3)
                    reg_busy.append(rb)
                    comp_busy.append(cb)
                    launches.add(nl)
            r = dict(B=B, state=state, reg=med(reg), comp=med(comp), reg_busy=med(reg_busy),
                     comp_busy=med(comp_busy) + med(glv), launches="/".join(str(x) for x in sorted(launches)))
            rows.append(r)
            emit(f"{B:>8} {state:>7} | {r['reg']:>11.3f} {r['reg_busy']:>8.3f} {r['launches']:>8} | {r['comp']:>10.3f} "
                 f"{r['comp_busy']:>8.3f} | {r['comp'] / r['reg']:>6.2f} {r['comp_busy'] / r['reg_busy']:>6.2f} | "
                 f"{B / r['reg']:>12.1f} {B / r['comp']:>11.1f} | {tag}")
        del rands
    emit("")
    for state in ("warm", "cold"):
        big = [r for r in rows if r["state"] == state][-1]
        emit(f"# B = {big['B']}, G table {state}: registration {big['B'] / big['reg']:.1f} k validators/s wall, "
             f"composition {big['B'] / big['comp']:.1f} k/s; busy {big['reg_busy']:.2f} ms against "
             f"{big['comp_busy']:.2f} ms ({big['comp_busy'] / big['reg_busy']:.2f}x); {tag}")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
