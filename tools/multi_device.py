#!/usr/bin/env python
"""One process, several GPUs: a multi-device context (cdl_create_devices) against bench.py's one process per
GPU.

For D = 1 .. --max-devices GPUs (default: every GPU of the box), on Context(devices=[0 .. D)), after one
warm-up call per row:
  whisk_round_trip  cdl_whisk_generate_shuffle_proof_batch + cdl_whisk_is_valid_shuffle_proof_batch at
                    ell = 124 (n = 128), B = 4 096 * D, end to end (host clock around the two calls);
  whisk_validate    the validation call alone;
  prove_batch       cdl_prove_batch at ell = 124, B = 1 024 * D caller-supplied instances;
  match             cdl_whisk_match_trackers, 8 192 trackers x 16 384 keys;
and, with --rows bulk (those rows alone) or --rows all (before the others), the two single calls that split by
size; the base_mul rows at 2^24 hold a 512 MB scalar vector and up to 1.6 GB of results per call:
  msm               cdl_g1_msm on host vectors at n = 2^16, 2^17, 2^18, 2^20 and 2^22 (a 2^20 set of points
                    repeated, its scalars rotated per repetition), wall time only (large MSMs are not in the
                    engine's accounting);
  base_mul          cdl_g1_batch_scalar_mul_base with a warm table at n = 2^16, 2^20, 2^22 and 2^24, affine and
                    compressed results.
Every row gives the median of --reps timed calls and the busy time of every device slot
(cdl_engine_busy_ms_device, union of that slot's kernel intervals) summed over the timed calls of the row.
Rows marked [0, 0] run two slots on GPU 0: what the split costs on one GPU (one PCIe link, one device), not a
speedup.  Lanes per slot and host cores follow bench.py's per-rank defaults.  With the protocol rows,
`bench.py --gpus D` (torchrun for D > 1, headline line only) then runs in the same process tree as the
multi-process comparison.  The card's name and power limit are read in the same call."""
import argparse
import importlib
import json
import os
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

ELL = 124
SETS = 8


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return f"unavailable ({e})"


def trackers(ctx, pkg, n, seed):
    r = pkg.Rand(seed)
    ks = b"".join(r.get_fr() for _ in range(n))
    rs = b"".join(r.get_fr() for _ in range(n))
    rG = ctx.g1_scalar_mul_affine(aff_enc(b.G1_GEN) * n, rs, broadcast=False)
    krG = ctx.g1_scalar_mul_affine(rG, ks, broadcast=False)
    e1, e2 = ctx.g1_compress(rG), ctx.g1_compress(krG)
    return b"".join(e1[48 * j:48 * j + 48] + e2[48 * j:48 * j + 48] for j in range(n))


def timed(ctx, D, reps, fn):
    """median wall seconds of `reps` calls of fn(rep) after one warm-up call, and per-slot busy ms summed
    over the timed calls"""
    fn(-1)
    ctx.engine_stats(reset=True)
    ts = []
    for i in range(reps):
        t0 = time.perf_counter()
        fn(i)
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts), [ctx.engine_busy_ms_device(s) for s in range(D)]


def measure(pkg, devices, reps, out):
    D = len(devices)
    ctx = pkg.Context(devices=devices)
    ctx.set_lanes(6 if (os.cpu_count() or 1) // len(set(devices)) >= 8 else 8)
    crs = ctx.generate_crs(ELL, pkg.Rand(0))
    rows = {}

    B = 4096 * D
    sets = [trackers(ctx, pkg, ELL, 1000 + i) for i in range(SETS)]
    pre = b"".join(sets[i % SETS] for i in range(B))
    res = {}

    def gen(i):
        res["g"] = ctx.whisk_generate_shuffle_proof_batch(crs, pre, [pkg.Rand(3000 + (i + 1) * B + j) for j in range(B)])

    def val(i):
        post, proofs, st = res["g"]
        ok, vst = ctx.whisk_is_valid_shuffle_proof_batch(crs, pre, post, proofs, [pkg.Rand(2000 + j) for j in range(B)])
        assert st == [0] * B and ok == [1] * B and vst == [0] * B

    def rt(i):
        gen(i)
        val(i)

    t, busy = timed(ctx, D, reps, rt)
    rows["whisk_round_trip"] = (B, B / t, t, busy)
    t, busy = timed(ctx, D, reps, val)
    rows["whisk_validate"] = (B, B / t, t, busy)

    Bp = 1024 * D
    r = pkg.Rand(1)
    psets = [(ctx.rand_get_g1_affines(r, ELL), ctx.rand_get_g1_affines(r, ELL)) for _ in range(SETS)]
    Rs = [psets[i % SETS][0] for i in range(Bp)]
    Ss = [psets[i % SETS][1] for i in range(Bp)]
    perms, ks = [], []
    for i in range(Bp):
        ri = pkg.Rand(10_000 + i)
        perms.append(ri.generate_permutation(ELL))
        ks.append(ri.get_fr())
    Ts, Us, M, rs_m, st = ctx.shuffle_permute_commit_batch(crs, Rs, Ss, perms, ks, [pkg.Rand(20_000 + i) for i in range(Bp)])
    assert st == [0] * Bp

    def prove(i):
        _, _, pst = ctx.prove_batch(crs, Rs, Ss, Ts, Us, M, perms, ks, rs_m, [pkg.Rand(30_000 + j) for j in range(Bp)])
        assert pst == [0] * Bp

    t, busy = timed(ctx, D, reps, prove)
    rows["prove_batch"] = (Bp, Bp / t, t, busy)

    T, V = 8192, 16384
    tr = b"".join(trackers(ctx, pkg, 1024, 5000 + i) for i in range(T // 1024))
    keys = pkg.Rand(6000).get_frs(V)

    def match(i):
        owner, status = ctx.whisk_match_trackers(tr, keys)
        assert status == [0] * T

    t, busy = timed(ctx, D, max(1, reps // 2), match)
    rows["match"] = (T * V, T * V / t, t, busy)
    crs.close()
    ctx.close()
    for k, (n, rate, t, busy) in rows.items():
        unit = "pairs/s" if k == "match" else ("round trips/s" if k == "whisk_round_trip" else "proofs/s")
        line = (f"  {str(devices):14s} {k:17s} n={n:>10d}  {rate:12.1f} {unit:14s} median {t * 1e3:9.1f} ms"
                f"   busy per slot ms: {' / '.join(f'{x:.1f}' for x in busy)}")
        print(line, file=out, flush=True)
    return rows


MSM_SIZES = [1 << 16, 1 << 17, 1 << 18, 1 << 20, 1 << 22]
BASE_SIZES = [1 << 16, 1 << 20, 1 << 22, 1 << 24]
SET = 1 << 20


def bulk_inputs(pkg):
    """a 2^20 set of points a_i * G and canonical scalars, made once on GPU 0; a fixed-base base"""
    ctx = pkg.Context(0)
    rng = np.random.default_rng(9)
    raw = rng.integers(0, 256, size=(SET, 32), dtype=np.uint8)
    raw[:, 31] &= 0x3F  # below 2^254 < r: canonical Montgomery limbs
    pts = ctx.g1_scalar_mul_affine(aff_enc(b.G1_GEN) * SET, raw.tobytes(), broadcast=False)
    raw2 = rng.integers(0, 256, size=(SET, 32), dtype=np.uint8)
    raw2[:, 31] &= 0x3F
    base = aff_enc(b.g1_mul(b.G1_GEN, 0x1234567890ABCDEF))
    ctx.close()
    return pts, raw2.tobytes(), base


def scalars(inputs, n):
    """n scalars: the 2^20 set repeated, rotated by one term per repetition"""
    sc = inputs[1]
    return b"".join(sc[32 * r:] + sc[:32 * r] for r in range(-(-n // SET)))[:32 * n]


def points(inputs, n):
    """n points: the 2^20 set repeated"""
    return (inputs[0] * -(-n // SET))[:96 * n]


def measure_bulk(pkg, devices, reps, inputs, out):
    D = len(devices)
    ctx = pkg.Context(devices=devices)
    ctx.set_lanes(6 if (os.cpu_count() or 1) // len(set(devices)) >= 8 else 8)
    rows = []
    for n in MSM_SIZES:
        P, S = points(inputs, n), scalars(inputs, n)
        t, _ = timed(ctx, D, reps, lambda i: ctx.g1_msm(P, S))
        rows.append(f"  {str(devices):14s} msm               n={n:>10d}  {n / t / 1e6:10.2f} M terms/s  median "
                    f"{t * 1e3:9.2f} ms")
    base = inputs[2]
    for n in BASE_SIZES:
        S = scalars(inputs, n)
        for kind, kw in (("affine", {}), ("compressed", {"affine": False, "compressed": True})):
            t, busy = timed(ctx, D, reps, lambda i: ctx.g1_batch_scalar_mul_base(base, S, **kw))
            rows.append(f"  {str(devices):14s} base_mul {kind:10s} n={n:>10d}  {n / t / 1e6:10.2f} M/s        median "
                        f"{t * 1e3:9.2f} ms   busy per slot ms: {' / '.join(f'{x:.1f}' for x in busy)}")
    ctx.close()
    for line in rows:
        print(line, file=out, flush=True)


def bench(D, steps, warmup):
    args = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", str(D), "--steps", str(steps), "--warmup",
            str(warmup), "--no-cpu-baseline", "--no-msm", "--no-latency", "--no-config4", "--no-n512"]
    if D > 1:
        args = [sys.executable, "-m", "torch.distributed.run", "--standalone", f"--nproc_per_node={D}"] + args[1:]
    p = subprocess.run(args, capture_output=True, text=True, cwd=ROOT)
    for ln in reversed(p.stdout.splitlines()):
        if ln.startswith("{"):
            return json.loads(ln)
    raise RuntimeError(f"bench.py --gpus {D} failed:\n{p.stdout[-2000:]}\n{p.stderr[-4000:]}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--max-devices", type=int, default=0, help="largest D (default: every GPU of the box)")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--bench-steps", type=int, default=3)
    ap.add_argument("--bench-warmup", type=int, default=2)
    ap.add_argument("--out", default="", help="also write the report to this file")
    ap.add_argument("--rows", choices=["protocol", "bulk", "all"], default="protocol",
                    help="protocol (default): the batched calls and the bench.py comparison; bulk: msm and base_mul; "
                         "all: both")
    args = ap.parse_args()
    import torch

    n = torch.cuda.device_count()
    if n < 1:
        raise SystemExit("no CUDA device")
    Dmax = min(n, args.max_devices) if args.max_devices else n
    pkg = importlib.import_module("go-curdleproofs_b200")

    class Tee:
        def __init__(self, path):
            self.f = open(path, "w") if path else None

        def write(self, s):
            sys.stdout.write(s)
            if self.f:
                self.f.write(s)

        def flush(self):
            sys.stdout.flush()
            if self.f:
                self.f.flush()

    out = Tee(args.out)
    print(f"# tools/multi_device.py  (host cores: {os.cpu_count()}, GPUs: {n})", file=out)
    print(f"# nvidia-smi index, name, power.limit, clocks.max.sm:\n# " + card().replace("\n", "\n# "), file=out)
    lists = [list(range(D)) for D in range(1, Dmax + 1)] + [[0, 0]]
    if args.rows != "protocol":
        print(f"# in-process, bulk rows: median wall time of {args.reps} calls after one warm-up call; [0, 0] = two "
              "slots on GPU 0 (the split's cost on one GPU, not a speedup)", file=out)
        inputs = bulk_inputs(pkg)
        for devs in lists:
            measure_bulk(pkg, devs, args.reps, inputs, out)
        del inputs
    if args.rows == "bulk":
        return
    print("# in-process: one context over the device list", file=out)
    inproc = {}
    for D in range(1, Dmax + 1):
        inproc[D] = measure(pkg, list(range(D)), args.reps, out)
    measure(pkg, [0, 0], args.reps, out)
    print("# multi-process: bench.py --gpus D (headline line; e2e = round trips/s wall clock, device = busy time)",
          file=out)
    for D in range(1, Dmax + 1):
        line = bench(D, args.bench_steps, args.bench_warmup)
        e2e = line["e2e"]["value"]
        mine = inproc[D]["whisk_round_trip"][1]
        print(f"  D={D}  bench.py e2e {e2e:10.1f} round trips/s  device {line['value']:10.1f}   in-process "
              f"{mine:10.1f} round trips/s  ratio in-process / bench {mine / e2e:.3f}", file=out, flush=True)


if __name__ == "__main__":
    main()
