#!/usr/bin/env python
"""Batched Whisk shuffle-proof verification (cdl_whisk_is_valid_shuffle_proof_batch) with the combined
check off (cdl_set_batch_verify_min 0: one small MSM per verifier equation) and forced on (1: one large
MSM over a random linear combination of a lane's equations, the per-proof MSMs only if it fails).

Part 1: B valid proofs (ell = 124, n = 128) at 1 lane and at the bench's lane count; the two modes
alternate, `--reps` timed calls each after one warm-up call per mode.  Per call: device busy time (union of
the kernel intervals of all lanes, cdl_engine_busy_ms), wall time, and the kernel-class split of
cdl_engine_stats (CUDA events on each lane's stream; with several lanes the classes overlap).
Part 2: one lane, sub-batches of 32 .. 1024 of the same proofs, both modes: the lane size from which the
combined check is cheaper in device time sets kBatchVerifyMinDefault (csrc/engine_verify.cu).
Every call's verdicts are checked (all valid)."""
import argparse
import importlib
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import bls12381 as b  # noqa: E402
from util import aff_enc  # noqa: E402

ELL, PROOF = 124, 4576


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = f"unavailable ({e})"
    return out


def make_batch(ctx, pkg, B):
    crs = ctx.generate_crs(ELL, pkg.Rand(0))
    r = pkg.Rand(1)
    pre = bytearray()
    gen = aff_enc(b.G1_GEN)
    for s in range(8):  # eight distinct tracker sets, reused round robin
        ks = b"".join(r.get_fr() for _ in range(ELL))
        rs = b"".join(r.get_fr() for _ in range(ELL))
        rG = ctx.g1_scalar_mul_affine(gen * ELL, rs, broadcast=False)
        krG = ctx.g1_scalar_mul_affine(rG, ks, broadcast=False)
        e1, e2 = ctx.g1_compress(rG), ctx.g1_compress(krG)
        pre += b"".join(e1[48 * j:48 * j + 48] + e2[48 * j:48 * j + 48] for j in range(ELL))
    tb = 96 * ELL
    pres = b"".join(bytes(pre[(i % 8) * tb:(i % 8 + 1) * tb]) for i in range(B))
    post, proofs, status = ctx.whisk_generate_shuffle_proof_batch(crs, pres, [pkg.Rand(100 + i) for i in range(B)],
                                                                  proof_size=PROOF)
    assert status == [0] * B
    return crs, pres, post, proofs


def timed_call(ctx, pkg, crs, pres, post, proofs, B):
    tb = 96 * ELL
    ctx.engine_stats(reset=True)
    n0 = ctx.launch_count()
    rands = [pkg.Rand(7000 + i) for i in range(B)]
    t0 = time.perf_counter()
    ok, st = ctx.whisk_is_valid_shuffle_proof_batch(crs, pres[:B * tb], post[:B * tb], proofs[:B * PROOF], rands,
                                                    proof_size=PROOF)
    wall = (time.perf_counter() - t0) * 1e3
    assert list(ok) == [1] * B and list(st) == [0] * B
    busy = ctx.engine_busy_ms()
    stats = ctx.engine_stats()
    for r in rands:
        r.close()
    return {"wall": wall, "busy": busy, "launches": ctx.launch_count() - n0,
            "cls": {k: v["ms"] for k, v in stats.items()}}


def fmt(xs):
    return f"{statistics.median(xs):8.2f} [{min(xs):.2f}, {max(xs):.2f}]"


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--B", type=int, default=4096)
    ap.add_argument("--lanes", type=int, default=0, help="the multi-lane point (default: bench.py's choice)")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--sizes", default="32,64,128,256,512,1024")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    lanes_hi = a.lanes or (6 if (os.cpu_count() or 1) >= 8 else 8)
    pkg = importlib.import_module("go-curdleproofs_b200")
    ctx = pkg.Context(0)
    lines = []

    def emit(s=""):
        print(s, flush=True)
        lines.append(s)

    emit("# Whisk shuffle-proof batch verification, ell = 124 (n = 128): combined check off (0) / forced on (1)")
    emit(f"# card: {card()}   (name, power limit, max SM clock)")
    emit(f"# device: {ctx.device_info()}; host cores: {os.cpu_count()}")
    emit(f"# {a.reps} timed calls per mode after one warm-up call each, modes alternating; median [min, max] ms")
    crs, pres, post, proofs = make_batch(ctx, pkg, max(a.B, max(int(s) for s in a.sizes.split(","))))
    emit("")
    emit(f"## B = {a.B}")
    emit(f"{'lanes':>5} {'mode':>4} {'busy ms':>26} {'wall ms':>26} {'launches':>9} "
         f"{'msm ms':>9} {'elem ms':>9} {'decomp ms':>9} {'comp ms':>9}")
    for lanes in (1, lanes_hi):
        ctx.set_lanes(lanes)
        res = {0: [], 1: []}
        for it in range(a.reps + 1):
            for mode in (0, 1):
                ctx.set_batch_verify_min(mode)
                r = timed_call(ctx, pkg, crs, pres, post, proofs, a.B)
                if it:
                    res[mode].append(r)
        for mode in (0, 1):
            rs = res[mode]
            cls = {k: statistics.median(r["cls"][k] for r in rs) for k in rs[0]["cls"]}
            emit(f"{lanes:>5} {mode:>4} {fmt([r['busy'] for r in rs]):>26} {fmt([r['wall'] for r in rs]):>26} "
                 f"{rs[0]['launches']:>9} {cls['msm_small']:>9.2f} {cls['elem_scalar_mul']:>9.2f} "
                 f"{cls['decompress']:>9.2f} {cls['compress']:>9.2f}")
        b0 = statistics.median(r["busy"] for r in res[0])
        b1 = statistics.median(r["busy"] for r in res[1])
        w0 = statistics.median(r["wall"] for r in res[0])
        w1 = statistics.median(r["wall"] for r in res[1])
        emit(f"#   {lanes} lane(s): combined check saves {b0 - b1:.2f} ms busy ({(b0 - b1) / b0 * 100:.1f} %), "
             f"{w0 - w1:.2f} ms wall ({(w0 - w1) / w0 * 100:.1f} %) per {a.B} verifications")
    emit("")
    emit("## one lane, sub-batch size (device busy ms per proof)")
    emit(f"{'proofs':>6} {'off us/proof':>13} {'on us/proof':>13} {'on/off':>7}")
    ctx.set_lanes(1)
    for B in [int(s) for s in a.sizes.split(",")]:
        res = {0: [], 1: []}
        for it in range(a.reps + 1):
            for mode in (0, 1):
                ctx.set_batch_verify_min(mode)
                r = timed_call(ctx, pkg, crs, pres, post, proofs, B)
                if it:
                    res[mode].append(r["busy"])
        m0, m1 = statistics.median(res[0]), statistics.median(res[1])
        emit(f"{B:>6} {m0 / B * 1e3:>13.1f} {m1 / B * 1e3:>13.1f} {m1 / m0:>7.3f}")
    ctx.set_batch_verify_min(-1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")
    crs.close()
    ctx.close()


if __name__ == "__main__":
    main()
