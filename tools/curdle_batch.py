#!/usr/bin/env python
"""Batched curdleproofs calls on caller-supplied instances (cdl_prove_batch / cdl_verify_batch) against the
single calls and against batched Whisk validation.

For each ell (default 124 and 508) and B (default 1, 64, 256, 1024), after one warm-up call per row:
  prove_batch         B proofs in one call;
  verify_batch        B verifications in one call, with the default combined check and with it off
                      (cdl_set_batch_verify_min 0);
  whisk_validate      cdl_whisk_is_valid_shuffle_proof_batch on B Whisk proofs of the same ell, which also
                      decompresses and subgroup-checks the 4 ell instance points per proof;
  prove / verify x B  a loop of B single calls (at --single-B only).
Each row gives the median of --reps timed calls: wall time (host clock around the call, which ends in a
device synchronise), device busy time (cdl_engine_busy_ms: union of the timed kernel intervals of all
lanes) and both as proofs per second.  Every verdict is checked (all valid).  The context's default lane
count (4) applies to the batched calls."""
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

SETS = 8  # distinct point / tracker sets, reused round robin


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = f"unavailable ({e})"
    return out


def whisk_proof_size(ell):
    m = (ell + 4).bit_length() - 1
    return 48 * (19 + 10 * m) + 7 * 32 + 10 * 4


def generic_batch(ctx, pkg, crs, B):
    """B instances with their commitments and proofs: lists of per-instance byte strings."""
    ell = crs.ell
    r = pkg.Rand(1)
    sets = [(ctx.rand_get_g1_affines(r, ell), ctx.rand_get_g1_affines(r, ell)) for _ in range(SETS)]
    Rs = [sets[i % SETS][0] for i in range(B)]
    Ss = [sets[i % SETS][1] for i in range(B)]
    perms, ks = [], []
    for i in range(B):
        ri = pkg.Rand(10_000 + i)
        perms.append(ri.generate_permutation(ell))
        ks.append(ri.get_fr())
    Ts, Us, M, rs_m, st = ctx.shuffle_permute_commit_batch(crs, Rs, Ss, perms, ks, [pkg.Rand(20_000 + i) for i in range(B)])
    assert st == [0] * B
    proofs, _, st = ctx.prove_batch(crs, Rs, Ss, Ts, Us, M, perms, ks, rs_m, [pkg.Rand(30_000 + i) for i in range(B)])
    assert st == [0] * B
    return dict(Rs=Rs, Ss=Ss, Ts=Ts, Us=Us, M=M, perms=perms, ks=ks, rs_m=rs_m, proofs=proofs)


def whisk_batch(ctx, pkg, crs, B):
    ell = crs.ell
    r = pkg.Rand(2)
    gen = aff_enc(b.G1_GEN)
    pres = []
    for _ in range(SETS):
        ks = b"".join(r.get_fr() for _ in range(ell))
        rs = b"".join(r.get_fr() for _ in range(ell))
        rG = ctx.g1_scalar_mul_affine(gen * ell, rs, broadcast=False)
        krG = ctx.g1_scalar_mul_affine(rG, ks, broadcast=False)
        e1, e2 = ctx.g1_compress(rG), ctx.g1_compress(krG)
        pres.append(b"".join(e1[48 * j:48 * j + 48] + e2[48 * j:48 * j + 48] for j in range(ell)))
    pre = b"".join(pres[i % SETS] for i in range(B))
    ps = whisk_proof_size(ell)
    post, proofs, st = ctx.whisk_generate_shuffle_proof_batch(crs, pre, [pkg.Rand(40_000 + i) for i in range(B)],
                                                              proof_size=ps)
    assert st == [0] * B
    return pre, bytes(post), bytes(proofs), ps


def timed(ctx, fn):
    ctx.engine_stats(reset=True)
    t0 = time.perf_counter()
    fn()
    wall = (time.perf_counter() - t0) * 1e3
    return wall, ctx.engine_busy_ms()


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--ells", default="124,508")
    ap.add_argument("--Bs", default="1,64,256,1024")
    ap.add_argument("--single-B", type=int, default=64)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    pkg = importlib.import_module("go-curdleproofs_b200")
    ctx = pkg.Context(0)
    lines = []

    def emit(s=""):
        print(s, flush=True)
        lines.append(s)

    emit("# curdleproofs Prove / Verify on caller-supplied instances: batched calls, single calls, Whisk validation")
    emit(f"# card: {card()}   (name, power limit, max SM clock)")
    emit(f"# device: {ctx.device_info()}; host cores: {os.cpu_count()}")
    emit(f"# median of {a.reps} timed calls after one warm-up; wall = host clock around the call, busy = device busy time")
    emit(f"{'ell':>4} {'B':>5} {'call':<28} {'wall ms':>10} {'busy ms':>10} {'proofs/s wall':>14} {'proofs/s busy':>14}")
    res = {}

    def row(ell, B, name, fn):
        fn()
        ws, bs = [], []
        for _ in range(a.reps):
            w, bz = timed(ctx, fn)
            ws.append(w)
            bs.append(bz)
        w, bz = statistics.median(ws), statistics.median(bs)
        res[(ell, B, name)] = (B / w * 1e3, B / bz * 1e3)
        emit(f"{ell:>4} {B:>5} {name:<28} {w:>10.2f} {bz:>10.2f} {B / w * 1e3:>14.1f} {B / bz * 1e3:>14.1f}")

    Bs = [int(x) for x in a.Bs.split(",")]
    for ell in [int(x) for x in a.ells.split(",")]:
        crs = ctx.generate_crs(ell, pkg.Rand(0))
        Bmax = max(Bs + [a.single_B])
        g = generic_batch(ctx, pkg, crs, Bmax)
        pre, post, wproofs, ps = whisk_batch(ctx, pkg, crs, Bmax)
        tb = 96 * ell
        for B in Bs:
            sl = {k: v[:B] for k, v in g.items()}

            def prove():
                _, _, st = ctx.prove_batch(crs, sl["Rs"], sl["Ss"], sl["Ts"], sl["Us"], sl["M"], sl["perms"], sl["ks"],
                                           sl["rs_m"], [pkg.Rand(50_000 + i) for i in range(B)])
                assert st == [0] * B

            def verify():
                ok, st = ctx.verify_batch(crs, sl["proofs"], sl["Rs"], sl["Ss"], sl["Ts"], sl["Us"], sl["M"],
                                          [pkg.Rand(60_000 + i) for i in range(B)])
                assert ok == [1] * B and st == [0] * B

            def whisk():
                ok, st = ctx.whisk_is_valid_shuffle_proof_batch(crs, pre[:B * tb], post[:B * tb], wproofs[:B * ps],
                                                                [pkg.Rand(70_000 + i) for i in range(B)], proof_size=ps)
                assert ok == [1] * B and st == [0] * B

            row(ell, B, "prove_batch", prove)
            row(ell, B, "verify_batch", verify)
            ctx.set_batch_verify_min(0)
            row(ell, B, "verify_batch, combined off", verify)
            ctx.set_batch_verify_min(-1)
            row(ell, B, "whisk_validate", whisk)
        B = a.single_B

        def prove_singles():
            for i in range(B):
                ctx.prove(crs, g["Rs"][i], g["Ss"][i], g["Ts"][i], g["Us"][i], g["M"][i], g["perms"][i], g["ks"][i],
                          g["rs_m"][i], pkg.Rand(50_000 + i))

        def verify_singles():
            for i in range(B):
                assert ctx.verify(crs, g["proofs"][i], g["Rs"][i], g["Ss"][i], g["Ts"][i], g["Us"][i], g["M"][i],
                                  pkg.Rand(60_000 + i))

        row(ell, B, f"prove x {B} single calls", prove_singles)
        row(ell, B, f"verify x {B} single calls", verify_singles)
        pb, vb = res[(ell, B, "prove_batch")], res[(ell, B, "verify_batch")]
        ps_, vs_ = res[(ell, B, f"prove x {B} single calls")], res[(ell, B, f"verify x {B} single calls")]
        emit(f"#   ell = {ell}, B = {B}: batch / single calls, proofs/s wall (busy): prove {pb[0] / ps_[0]:.1f}x "
             f"({pb[1] / ps_[1]:.1f}x), verify {vb[0] / vs_[0]:.1f}x ({vb[1] / vs_[1]:.1f}x)")
        for Bx in Bs:
            v, w = res[(ell, Bx, "verify_batch")], res[(ell, Bx, "whisk_validate")]
            emit(f"#   ell = {ell}, B = {Bx}: verify_batch / whisk_validate, proofs/s wall {v[0] / w[0]:.2f}x, "
                 f"busy {v[1] / w[1]:.2f}x")
        crs.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
