#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native G1 hot path.

Workload (BASELINE.json configs[1]): Whisk shape, shuffled_elements = 124 (n = 128):
GenerateWhiskShuffleProof + IsValidWhiskShuffleProof round trips.  One *step* = one batch of B
independent round trips (synthetic trackers) driven through the C ABI (cdl_whisk_*_batch) with HOST
buffers.

  e2e.value  THE HEADLINE: proofs/s wall clock through the C ABI, host<->device copies and the host-side
             Fiat-Shamir work inside the timed region
  value      proofs/s counting only device time: B*K / device busy time (union of the CUDA-event
             intervals of every kernel the step launched on any lane's stream); explains e2e, and is the
             number `roofline` is built on
  roofline   the dominant kernel class against the nominal integer-pipe peak (64 IMAD lanes / clk / SM
             at the measured clock / 300 multiply-adds per 381-bit Montgomery product, SURVEY.md §8d),
             HBM GB/s secondary
  cpu_baseline  the CPU oracle ("port": C 6x64 Montgomery restatement driven by the Python protocol
             restatement; the reference's gnark-crypto cannot be built: no Go toolchain here or on the
             GPU box) on the host cores — persistent workers, set-up outside the timed region

Further keys of the GPU line (all through the C ABI):
  config4       BASELINE.json configs[3]: 4 096 independent n = 128 verifications SHARDED over the N
                ranks (strong scaling), every 8th proof mutated (five kinds, SURVEY.md §8d), verdicts
                gathered across ranks and compared with the expected list and, for the first 64, with the
                CPU oracle's verdicts
  n512          batched round trips at shuffled_elements = 508 (n = 512; BASELINE `metric` names n = 512)
  single_proof  configs[0] and [2] (+ n = 128): one proof at a time, with the CPU port beside it
  msm           configs[4]: standalone G1 MSM sweep 2^10 .. 2^22 (device-resident inputs; at N > 1 the
                window-partitioned form with one NCCL all-gather inside libcurdle_b200.so), adversarial
                inputs at 2^16, the CPU port's bucket MSM beside it

`--impl reference` times the CPU path alone on all host cores (same `config`, bounded sample per step).
Multi-GPU: one process per GPU (torchrun); the headline shards independent proofs across ranks with no
data-path collective (weak scaling); NCCL carries the barrier, the max-over-ranks time, the verdict
gather of config 4 and the partial sums of the sharded MSM.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ELL = 124
METRIC = "whisk_shuffle_proof_roundtrips_per_s (GenerateWhiskShuffleProof + IsValidWhiskShuffleProof, n=128)"
UNIT = "proofs/s"
MODMUL_IMADS = 300.0  # 2*12^2 + 12 wide multiply-adds per 381-bit Montgomery product (SURVEY.md §8d)
IMAD_LANES_PER_SM_CLK = 64.0  # nominal 32-bit IMAD issue rate (measured: profiles/r2_probe2.txt)
VERIFY_TOTAL = 4096
KINDS = 5


def config_dict(batch: int, world: int, lanes, info=None):
    """The same dict in both arms (the reference arm times a bounded sample of this workload)."""
    d = {"workload": "whisk_n128_roundtrip", "shuffled_elements": ELL, "proofs_per_gpu_per_step": batch,
         "parallelism": f"proof-parallel x{world}, no data-path collective"}
    if info is not None:
        d.update({"l2": "flushed between steps (256 MiB write); the step's own working set (about 120 kB of points "
                        "per instance) exceeds the 126 MB L2 as well",
                  "value_definition": "proofs / device busy time = union of CUDA-event kernel intervals over all lanes "
                                      "(host Fiat-Shamir excluded); e2e is the wall-clock headline",
                  "lanes": lanes, "host_threads_cap": int(os.environ.get("CDL_HOST_THREADS", "0")),
                  "device": info["name"], "sm_count": info["sm_count"]})
    return d


# ----------------------------------------------------------------------------- CPU workers (oracle port)
_W = {}


def _w_init(ells, ready=None):
    """Worker set-up (outside every timed region): backend, CRS and one tracker set per shape."""
    sys.path.insert(0, ROOT)
    from oracle import protocol as P, whisk as W
    from oracle.cbackend import CBackend
    from oracle.rand import Rand

    cb = CBackend(threads=1)
    P.set_backend(cb)
    _W.update(P=P, W=W, Rand=Rand, cb=cb, crs={}, pre={})
    for ell in ells:
        _W["crs"][ell] = P.generate_crs(ell, Rand(0, backend=cb))
        _W["pre"][ell] = W.generate_shuffle_trackers(Rand(1000, backend=cb), ell)
    if ready is not None:
        with ready.get_lock():
            ready.value += 1


def _w_roundtrips(args):
    """`count` Whisk round trips; returns the seconds spent in the proof loop only."""
    ell, seed, count = args
    P, W, Rand, cb = _W["P"], _W["W"], _W["Rand"], _W["cb"]
    crs, pre = _W["crs"][ell], _W["pre"][ell]
    size = 4576 if ell <= 124 else 48 * (19 + 10 * (ell + 4).bit_length()) + 7 * 32 + 40
    t0 = time.perf_counter()
    for i in range(count):
        r = Rand(3000 + seed * 1000 + i, backend=cb)
        post, proof = W.generate_whisk_shuffle_proof(crs, pre, r, ell=ell, proof_size=size)
        assert W.is_valid_whisk_shuffle_proof(crs, pre, post, proof, r)
    return time.perf_counter() - t0


def _w_single(ell):
    """curdleproof_test.go:184-237 shapes on the CPU port: (prove s, verify s) for one proof."""
    P, Rand, cb = _W["P"], _W["Rand"], _W["cb"]
    rand = Rand(0, backend=cb)
    crs = P.generate_crs(ell, rand)
    perm = Rand(42).generate_permutation(ell)
    k = rand.get_fr()
    Rs, Ss = rand.get_g1_affines(ell), rand.get_g1_affines(ell)
    Ts, Us, M, rs_m = P.shuffle_permute_commit(crs.Gs, crs.Hs, Rs, Ss, perm, k, rand)
    t0 = time.perf_counter()
    proof = P.prove(crs, Rs, Ss, Ts, Us, M, perm, k, rs_m, Rand(42, backend=cb))
    t1 = time.perf_counter()
    assert P.verify(proof, crs, Rs, Ss, Ts, Us, M, Rand(43, backend=cb))
    return t1 - t0, time.perf_counter() - t1


def _w_verdict(args):
    """Oracle verdict of one Whisk validation: (ok, error?)."""
    ell, pre, post, proof, seed = args
    P, W, Rand, cb = _W["P"], _W["W"], _W["Rand"], _W["cb"]
    split = lambda t: [(t[96 * j:96 * j + 48], t[96 * j + 48:96 * j + 96]) for j in range(ell)]  # noqa: E731
    try:
        return bool(W.is_valid_whisk_shuffle_proof(_W["crs"][ell], split(pre), split(post), proof, Rand(seed, backend=cb))), False
    except (W.WhiskError, P.ProofError):
        return False, True


_POOL = None


def cpu_pool():
    """Persistent worker pool (one process per host core), set up once."""
    global _POOL
    if _POOL is None:
        import multiprocessing as mp
        from oracle.cbackend import build as build_oracle

        build_oracle()
        cores = os.cpu_count() or 1
        mpc = mp.get_context("spawn")
        ready = mpc.Value("i", 0)
        _POOL = (mpc.Pool(cores, initializer=_w_init, initargs=((ELL,), ready)), cores)
        t0 = time.time()
        while ready.value < cores and time.time() - t0 < 300:  # every worker finished its set-up
            time.sleep(0.05)
    return _POOL


def cpu_roundtrip_sample(per_worker: int):
    """One bounded sample: every worker does `per_worker` round trips; wall clock of the whole map."""
    pool, cores = cpu_pool()
    t0 = time.perf_counter()
    pool.map(_w_roundtrips, [(ELL, w, per_worker) for w in range(cores)], chunksize=1)
    return cores * per_worker, time.perf_counter() - t0


def reference_main(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    pool, cores = cpu_pool()
    per_worker = 4
    for _ in range(args.warmup):
        cpu_roundtrip_sample(1)
    proofs, total = 0, 0.0
    for _ in range(args.steps):
        n, dt = cpu_roundtrip_sample(per_worker)
        proofs += n
        total += dt
    value = proofs / total
    sample = (f"{cores} persistent worker processes x {per_worker} Whisk n=128 round trips per step (workers, CRS and "
              f"trackers set up before the timed region); {args.steps} steps, {total:.1f} s")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / max(1, args.steps),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64 (6x64-bit Montgomery limbs)",
        "data": "synthetic", "config": config_dict(args.batch, args.gpus, args.lanes),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "proofs_per_step": cores * per_worker,
                         "note": "CPU oracle port (C 6x64 Montgomery + Python orchestration), not gnark-crypto: no Go "
                                 "toolchain in the image or on the GPU box"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    pool.close()


# ----------------------------------------------------------------------------- GPU arm
class ClockSampler(threading.Thread):
    """SM clock and throttle reasons of one GPU DURING the timed region.  Sampled in-process through NVML
    (nvidia_ml_py); spawning `nvidia-smi` five times a second from every rank takes the driver's global lock
    often enough to slow the other ranks' launches (measured at 4 GPUs), so the subprocess form is only the
    fallback and runs at 1 Hz."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.sm, self.mx, self.reasons, self.n = [], [], set(), 0
        self.stop_flag = threading.Event()
        self.nvml = None
        try:
            import pynvml

            pynvml.nvmlInit()
            # NVML enumerates physical devices: honour CUDA_VISIBLE_DEVICES when it is a plain index list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            phys = index
            if vis and all(x.strip().isdigit() for x in vis.split(",")):
                phys = int(vis.split(",")[index])
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml = pynvml
            self.source = "nvml"
        except Exception:
            self.source = "nvidia-smi"

    def sample(self):
        if self.nvml is not None:
            nv = self.nvml
            self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
            self.mx.append(float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)))
            try:
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            except Exception:
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            for name, bit in (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20),
                              ("sw_power_cap", 0x4)):
                if r & bit:
                    self.reasons.add(name)
        else:
            out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                  str(self.index)], capture_output=True, text=True, timeout=10).stdout.strip()
            s = [x.strip() for x in out.split(",")]
            if len(s) > 8:
                self.sm.append(float(s[1]))
                self.mx.append(float(s[2]))
                for k, nm in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]):
                    if s[5 + k].lower().startswith("active"):
                        self.reasons.add(nm)
        self.n += 1

    def run(self):
        while not self.stop_flag.is_set():
            try:
                self.sample()
            except Exception:
                pass
            self.stop_flag.wait(0.2 if self.nvml is not None else 1.0)

    def summary(self):
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                "reasons": sorted(self.reasons), "samples": self.n, "source": self.source}


def make_trackers(ctx, pkg, ell: int, seeds):
    """Synthetic pre-shuffle trackers (whisk_test.go generateShuffleTrackers): (r*G, k*r*G) compressed."""
    enc = importlib.import_module("go-curdleproofs_b200.encoding")
    gen = enc.aff_enc(enc.G1_GEN)
    out = []
    for s in seeds:
        r = pkg.Rand(s)
        ks, rs = [], []
        for _ in range(ell):
            ks.append(r.get_fr())
            rs.append(r.get_fr())
        rG = ctx.g1_scalar_mul_affine(gen * ell, b"".join(rs), broadcast=False)
        krG = ctx.g1_scalar_mul_affine(rG, b"".join(ks), broadcast=False)
        e1, e2 = ctx.g1_compress(rG), ctx.g1_compress(krG)
        out.append(b"".join(e1[48 * j:48 * j + 48] + e2[48 * j:48 * j + 48] for j in range(ell)))
    return out


def msm_alg_modmul(n: int) -> int:
    """SURVEY.md §8d: min_c [6 n W + 28 2^(c-1) W + 9 c (W-1) + 14 W], W = ceil(256 / c)."""
    best = None
    for c in range(1, 25):
        W = -(-256 // c)
        v = 6 * n * W + 28 * (1 << (c - 1)) * W + 9 * c * (W - 1) + 14 * W
        best = v if best is None or v < best else best
    return best


def proof_size_for(ell: int) -> int:
    if ell <= ELL:
        return 4576  # whisk/types.go:21
    m = (ell + 4).bit_length() - 1
    return 48 * (19 + 10 * m) + 7 * 32 + 10 * 4 + 8


def msm_sweep(ctx, pkg, log2_sizes, reps, world, rank, peak_modmul, barrier, cpu_sizes):
    """Config 5: points P_i = a_i*G (a_i = Rand(5).GetFr), scalars Rand(6).GetFr, both replicated on every
    rank; every result is checked against (sum a_i*s_i)*G computed with host integer arithmetic and one
    1-point scalar multiplication on the GPU.  Adversarial inputs at 2^16 (SURVEY.md §8d) are timed and
    checked the same way."""
    enc = importlib.import_module("go-curdleproofs_b200.encoding")
    R, RR, RR_INV, aff_enc, fr_enc = enc.R, pow(2, 256, enc.R), enc.RR_INV, enc.aff_enc, enc.fr_enc
    gen = aff_enc(enc.G1_GEN)

    nmax = 1 << max(log2_sizes)
    r5, r6 = pkg.Rand(5), pkg.Rand(6)
    dp, da, ds = ctx.dev_buffer(96 * nmax), ctx.dev_buffer(32 * nmax), ctx.dev_buffer(32 * nmax)
    chunk = min(nmax, 1 << 16)
    acc = {}
    marks = sorted(1 << lg for lg in log2_sizes)
    run, done = 0, 0
    for o in range(0, nmax, chunk):
        m = min(chunk, nmax - o)
        A, S = r5.get_frs(m), r6.get_frs(m)
        dp.upload(gen * m, 96 * o)
        da.upload(A, 32 * o)
        ds.upload(S, 32 * o)
        if rank == 0:  # host-side check value: prefix sums of a_i * s_i (Montgomery decode folded into one factor)
            cuts = [x - done for x in marks if done < x <= done + m]
            lo = 0
            for cut in cuts + ([m] if not cuts or cuts[-1] != m else []):
                for i in range(lo, cut):
                    run += int.from_bytes(A[32 * i:32 * i + 32], "little") * int.from_bytes(S[32 * i:32 * i + 32], "little")
                lo = cut
                if done + cut in marks:
                    acc[(done + cut).bit_length() - 1] = run
        done += m
    if rank != 0:
        acc = {lg: 0 for lg in log2_sizes}
    ctx.g1_scalar_mul_affine_device(dp, da, nmax, False, dp)

    def check(res, k):
        want = ctx.g1_scalar_mul_affine(gen, fr_enc(k % R), broadcast=True)
        if k % R == 0:
            return res[96:144] == bytes(48)
        return res[:96] == want and res[96:144] != bytes(48)

    def timed(d_points, d_scalars, n):
        best, res = None, None
        for _ in range(reps + 1):
            barrier()
            res, ms = ctx.g1_msm_sharded_device(d_points, d_scalars, n)
            best = ms if best is None or ms < best else best
        return res, best

    out = []
    for lg in log2_sizes:
        n = 1 << lg
        res, best = timed(dp, ds, n)
        mm = msm_alg_modmul(n)
        out.append({"log2n": lg, "ms": best, "mpoints_per_s": n / best / 1e3, "gmodmul_per_s": mm / best / 1e6,
                    "frac_of_int_peak": mm / (best * 1e-3) / (peak_modmul * world),
                    "check": ("ok" if check(res, acc[lg] * RR_INV * RR_INV) else "MISMATCH") if rank == 0 else "rank 0 checks",
                    "windows_per_rank": pkg.comm_partition(n, world, rank)[3]})

    # adversarial inputs at 2^16: same check with the modified (a, s) vectors
    adv = []
    lgA = 16 if nmax >= (1 << 16) else min(log2_sizes)
    nA = 1 << lgA
    fa, fs = pkg.Rand(7).get_frs(nA), pkg.Rand(8).get_frs(nA)
    A0 = [int.from_bytes(fa[32 * i:32 * i + 32], "little") * RR_INV % R for i in range(nA)]
    S0 = [int.from_bytes(fs[32 * i:32 * i + 32], "little") * RR_INV % R for i in range(nA)]
    if True:
        dpa, daa, dsa = ctx.dev_buffer(96 * nA), ctx.dev_buffer(32 * nA), ctx.dev_buffer(32 * nA)
        variants = {
            "all_equal_scalars": (A0, [S0[0]] * nA),
            "scalars_below_2^9": (A0, [s & 511 for s in S0]),
            "1pct_infinity_bases": ([0 if i % 100 == 0 else a for i, a in enumerate(A0)], S0),
            "duplicated_points": ([A0[0]] * nA, S0),
            "plus_minus_pairs": ([A0[i - 1] * (R - 1) % R if i & 1 else A0[i] for i in range(nA)], S0),
        }
        for name, (av, sv) in variants.items():
            daa.upload(b"".join((a * RR % R).to_bytes(32, "little") for a in av))
            dsa.upload(b"".join((s * RR % R).to_bytes(32, "little") for s in sv))
            dpa.upload(gen * nA)
            ctx.g1_scalar_mul_affine_device(dpa, daa, nA, False, dpa)
            res, best = timed(dpa, dsa, nA)
            k = sum(a * s for a, s in zip(av, sv))
            adv.append({"input": name, "log2n": lgA, "ms": best, "mpoints_per_s": nA / best / 1e3,
                        "check": ("ok" if check(res, k) else "MISMATCH") if rank == 0 else "rank 0 checks"})
        for d in (dpa, daa, dsa):
            d.close()

    cpu = None
    if rank == 0 and cpu_sizes:
        # the same MSM on the host cores with the CPU oracle port (bucket method, windows spread over threads;
        # the reference's gnark-crypto MultiExp cannot be built here)
        try:
            from oracle.cbackend import CBackend  # CPU baseline leg: the one place the GPU arm runs the oracle

            RP_INV, FP_P = enc.RP_INV, enc.P
            cb = CBackend(accelerate_keccak=False)
            cores = os.cpu_count() or 1
            nc = 1 << max(cpu_sizes)
            raw_p = dp.download(96 * nc)
            raw_s = ds.download(32 * nc)
            cp = b"".join((int.from_bytes(raw_p[48 * i:48 * i + 48], "little") * RP_INV % FP_P).to_bytes(48, "little")
                          for i in range(2 * nc))
            cs = b"".join((int.from_bytes(raw_s[32 * i:32 * i + 32], "little") * RR_INV % R).to_bytes(32, "little")
                          for i in range(nc))
            cpu = []
            for lg in cpu_sizes:
                n = 1 << lg
                t0 = time.perf_counter()
                res_cpu = cb.msm_raw(cp[:96 * n], cs[:32 * n], n, cores)
                dt = time.perf_counter() - t0
                gpu_res, _ = ctx.g1_msm_device(dp, ds, n)  # local (non-collective): only rank 0 is here
                same = all((int.from_bytes(gpu_res[48 * k:48 * k + 48], "little") * RP_INV % FP_P) ==
                           int.from_bytes(res_cpu[48 * k:48 * k + 48], "little") for k in range(2))
                cpu.append({"log2n": lg, "ms": dt * 1e3, "mpoints_per_s": n / dt / 1e6, "cores": cores, "kind": "port",
                            "check": "equal to the GPU result" if same else "MISMATCH"})
        except Exception as e:  # reported baseline, never required
            cpu = {"failed": str(e)}
    for d in (dp, da, ds):
        d.close()
    return out, adv, cpu


def single_proof_latency(ctx, pkg, ells=(60, 124, 508)):
    """BASELINE.json configs 1-3: curdleproof.Prove / Verify for one proof at a time through the C ABI
    (setup of curdleproof_test.go:239-274 with perm = Rand(42).GeneratePermutation), best of 3, wall clock."""
    out = []
    for ell in ells:
        r = pkg.Rand(0)
        crs = ctx.generate_crs(ell, r)
        k = r.get_fr()
        Rs = ctx.rand_get_g1_affines(r, ell)
        Ss = ctx.rand_get_g1_affines(r, ell)
        perm = pkg.Rand(42).generate_permutation(ell)
        Ts, Us, M, rs_m = ctx.shuffle_permute_commit(crs, Rs, Ss, perm, k, r)
        bp = bv = None
        for it in range(4):
            t0 = time.perf_counter()
            proof = ctx.prove(crs, Rs, Ss, Ts, Us, M, perm, k, rs_m, pkg.Rand(42))
            t1 = time.perf_counter()
            ok = ctx.verify(crs, proof, Rs, Ss, Ts, Us, M, pkg.Rand(43))
            t2 = time.perf_counter()
            assert ok
            if it:
                bp = t1 - t0 if bp is None else min(bp, t1 - t0)
                bv = t2 - t1 if bv is None else min(bv, t2 - t1)
        out.append({"shuffled_elements": ell, "prove_ms": bp * 1e3, "verify_ms": bv * 1e3, "proof_bytes": len(proof)})
        crs.close()
    return out


def mutate_batch(ctx, pkg, ell, pre, post, proofs, proof_size, first_index, every=8):
    """Config-4 mutations on a contiguous block of instances (global indices first_index ..): every
    `every`-th GLOBAL index is mutated, cycling through the five kinds of SURVEY.md §8d.  Returns the
    three mutated buffers and the expected (ok, status) lists."""
    B = len(pre) // (96 * ell)
    tb = 96 * ell
    pre_m, post_m, proofs_m = bytearray(pre), bytearray(post), bytearray(proofs)
    want_ok, want_st = [1] * B, [0] * B
    used = 48 * (19 + 10 * ((ell + 4).bit_length() - 1)) + 7 * 32 + 40
    p2 = pkg.Rand(5).generate_permutation(ell)
    km_idx = []
    for b in range(B):
        g = first_index + b
        if g % every:
            continue
        kind = (g // every) % KINDS
        want_ok[b] = 0
        if kind == 0:    # Rs / Ss swapped: the two halves of every pre-tracker
            blk = pre_m[b * tb:(b + 1) * tb]
            pre_m[b * tb:(b + 1) * tb] = b"".join(bytes(blk[96 * j + 48:96 * j + 96]) + bytes(blk[96 * j:96 * j + 48]) for j in range(ell))
        elif kind == 1:  # post-trackers re-permuted
            blk = bytes(post_m[b * tb:(b + 1) * tb])
            post_m[b * tb:(b + 1) * tb] = b"".join(blk[96 * j:96 * j + 96] for j in p2)
        elif kind == 2:  # M -> k*M (done for all such instances at once below)
            km_idx.append(b)
        elif kind == 3:  # one bit of the proof's last scalar x flipped
            proofs_m[b * proof_size + used - 1] ^= 1
        else:            # Ts[0] replaced by the infinity encoding: "randomizer is zero" (an error)
            post_m[b * tb:b * tb + 48] = bytes([0xC0]) + bytes(47)
            want_st[b] = -5
    if km_idx:
        M_enc = b"".join(bytes(proofs_m[b * proof_size:b * proof_size + 48]) for b in km_idx)
        M_aff, st = ctx.g1_decompress(M_enc)
        assert not any(st)
        kM = ctx.g1_compress(ctx.g1_scalar_mul_affine(M_aff, pkg.Rand(9).get_fr(), broadcast=True))
        for j, b in enumerate(km_idx):
            proofs_m[b * proof_size:b * proof_size + 48] = kM[48 * j:48 * j + 48]
    return pre_m, post_m, proofs_m, want_ok, want_st


DUMP_SAMPLE = 256  # instances whose post-trackers and proofs are written: about 17 MB as float32 at n = 128


def dump_outputs(out_dir: str, B: int, post, proofs, status, ok, st, ell: int = ELL, proof_size: int = 4576):
    """What the round trips of one step return to their caller, as float32 .npy files, so that two builds
    can be compared output for output: post-trackers and proofs (one byte per element) of a fixed, seeded
    sample of the batch, the sampled indices, and every instance's generation status, verdict and
    validation status."""
    import numpy as np

    idx = np.arange(B)
    if B > DUMP_SAMPLE:
        idx = np.sort(np.random.default_rng(0).choice(B, DUMP_SAMPLE, replace=False))
    arrays = {
        "sample_index": idx,
        "post_trackers": np.frombuffer(post, np.uint8).reshape(B, ell * 96)[idx],
        "proofs": np.frombuffer(proofs, np.uint8).reshape(B, proof_size)[idx],
        "generate_status": status,
        "valid": ok,
        "validate_status": st,
    }
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float32))


def gpu_main(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    # ranks of one box share its host cores (Fiat-Shamir work between launches)
    os.environ.setdefault("CDL_HOST_THREADS", str(max(2, (os.cpu_count() or 1) // max(1, world))))
    pkg = importlib.import_module("go-curdleproofs_b200")
    sharding = importlib.import_module("go-curdleproofs_b200.sharding")
    ctx = pkg.Context(local)  # raises without a GPU / without the built library: no fallback
    if args.lanes:
        ctx.set_lanes(args.lanes)
    if world > 1:  # the library's own NCCL communicator (window-partitioned MSM)
        uid = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            uid = torch.tensor(list(pkg.comm_unique_id()), dtype=torch.uint8, device=dev)
        dist.broadcast(uid, 0)
        ctx.comm_init(bytes(uid.cpu().tolist()), rank, world)
    info = ctx.device_info()
    B = args.batch
    crs = ctx.generate_crs(ELL, pkg.Rand(0))
    # a few distinct tracker sets, cycled over the batch (every instance still gets its own RNG stream);
    # set 0 is the one the CPU workers use (Rand(1000)), so config 4's oracle sample sees the same bytes
    base_sets = make_trackers(ctx, pkg, ELL, [1000 + i for i in range(8)])
    pre = b"".join(base_sets[(rank * B + i) % len(base_sets)] for i in range(B))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    # nominal integer-pipe peak at the clock measured live: a dependent IMAD chain times the clock, the
    # roofline denominator is 64 IMAD lanes / clk / SM (SURVEY.md §8d) / 300 per modmul
    imad_per_s, _ = ctx.int_peak(0, 4000)
    peak_modmul = imad_per_s / MODMUL_IMADS

    step_no = [0]
    # the caller's common.Rand objects (one per instance and step) are inputs: created before the timed region
    n_steps_total = args.warmup + args.steps + 2
    all_rands = [[pkg.Rand((rank << 40) | (s << 20) | i) for i in range(B)] for s in range(n_steps_total)]

    def step():
        flush.zero_()  # L2 flush between iterations
        s = step_no[0]
        step_no[0] += 1
        rands = all_rands[s]
        post, proofs, status = ctx.whisk_generate_shuffle_proof_batch(crs, pre, rands)
        ok, st = ctx.whisk_is_valid_shuffle_proof_batch(crs, pre, post, proofs, rands)
        return post, proofs, status, ok, st

    for _ in range(args.warmup):
        _, _, status, ok, st = step()
        assert status == [0] * B and ok == [1] * B and st == [0] * B, "warm-up round trip failed"

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def max_over_ranks(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    ctx.engine_stats(reset=True)
    l0 = ctx.launch_count()
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        post, proofs, status, ok, st = step()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    barrier()
    sampler.stop_flag.set()
    sampler.join(timeout=2)
    assert status == [0] * B and ok == [1] * B and st == [0] * B, "timed round trip failed"
    stats_timed = ctx.engine_stats()
    launches = ctx.launch_count() - l0
    busy_ms = ctx.engine_busy_ms()
    wall_max, dev_max = max_over_ranks(wall), max_over_ranks(busy_ms / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, B, post, proofs, status, ok, st)

    # roofline pass: the same step with ONE lane, so that the CUDA-event interval of a kernel is its own
    # duration (with several lanes the streams share the GPU and every interval also contains the other
    # lanes' kernels); one untimed warm-up, then one measured step
    ctx.set_lanes(1)
    step()
    ctx.engine_stats(reset=True)
    _, _, status, ok, st = step()
    torch.cuda.synchronize()
    assert status == [0] * B and ok == [1] * B and st == [0] * B, "roofline-pass round trip failed"
    stats = ctx.engine_stats()
    ctx.set_lanes(args.lanes or 4)
    dev_ms = sum(v["ms"] for v in stats.values())

    # ---- config 4: VERIFY_TOTAL proofs sharded over the ranks (strong scaling), five mutation kinds
    config4 = None
    if not args.no_config4:
        total = args.verify_total
        lo, hi = sharding.shard_bounds(total, world, rank)
        Bv = hi - lo
        pre_v = b"".join(base_sets[i % len(base_sets)] for i in range(lo, hi))
        post_v, proofs_v, status = ctx.whisk_generate_shuffle_proof_batch(crs, pre_v, [pkg.Rand((77 << 24) | i) for i in range(lo, hi)])
        assert status == [0] * Bv
        pre_m, post_m, proofs_m, want_ok, want_st = mutate_batch(ctx, pkg, ELL, pre_v, post_v, proofs_v, 4576, lo)
        vt, busy = [], []
        vok = vst = None
        for it in range(3):  # first pass is the warm-up
            flush.zero_()
            ctx.engine_stats(reset=True)
            vrands = [pkg.Rand((78 << 24) | i) for i in range(lo, hi)]  # the verifier's RNG per proof: an input
            barrier()
            t1 = time.perf_counter()
            vok, vst = ctx.whisk_is_valid_shuffle_proof_batch(crs, pre_m, post_m, proofs_m, vrands)
            torch.cuda.synchronize()
            vt.append(time.perf_counter() - t1)
            busy.append(ctx.engine_busy_ms() / 1e3)
        t_wall, t_busy = max_over_ranks(sum(vt[1:])), max_over_ranks(sum(busy[1:]))
        all_ok = sharding.gather_verdicts(vok, total, world, rank, device=dev)
        all_st = sharding.gather_verdicts(vst, total, world, rank, device=dev)
        exp_ok = sharding.gather_verdicts(want_ok, total, world, rank, device=dev)
        exp_st = sharding.gather_verdicts(want_st, total, world, rank, device=dev)
        config4 = {"workload": f"{total} independent n=128 IsValidWhiskShuffleProof calls sharded over {world} GPU(s) "
                               "(contiguous blocks), every 8th proof mutated: Rs/Ss swapped, post-trackers re-permuted, "
                               "M -> k*M, one scalar bit flipped, Ts[0] = infinity, in turn",
                   "value": total * 2 / t_wall, "unit": "verifications/s", "scaling": "strong",
                   "device_busy_value": total * 2 / t_busy if t_busy else None, "proofs_per_gpu": Bv,
                   "timing": "wall clock through the C ABI with host buffers, 2 passes after 1 warm-up, max over ranks",
                   "verdicts_gathered": len(all_ok),
                   "verdicts": "as expected" if all_ok == exp_ok and all_st == exp_st else "MISMATCH",
                   "rejected": all_ok.count(0), "errors": sum(1 for s in all_st if s != 0)}
        if rank == 0 and not args.no_cpu_baseline:  # the CPU oracle's verdicts for the first 64 proofs
            try:
                ns = min(64, Bv)
                tb = 96 * ELL
                pool, cores = cpu_pool()
                t1 = time.perf_counter()
                got = pool.map(_w_verdict, [(ELL, bytes(pre_m[i * tb:(i + 1) * tb]), bytes(post_m[i * tb:(i + 1) * tb]),
                                             bytes(proofs_m[i * 4576:(i + 1) * 4576]), (78 << 24) | i) for i in range(ns)])
                dt = time.perf_counter() - t1
                same = all(bool(vok[i]) == g[0] and (vst[i] != 0) == g[1] for i, g in enumerate(got))
                config4["oracle_sample"] = {"proofs": ns, "mutated": sum(1 for i in range(ns) if i % 8 == 0),
                                            "check": "identical verdicts and errors" if same else "MISMATCH",
                                            "cpu_verifications_per_s": ns / dt, "cores": cores, "kind": "port"}
            except Exception as e:
                config4["oracle_sample"] = {"failed": str(e)}

    # ---- n = 512 (BASELINE metric: "proofs/s at n=128,512"): batched round trips at shuffled_elements = 508
    n512 = None
    if not args.no_n512:
        ell5, B5 = 508, args.batch512
        crs5 = ctx.generate_crs(ell5, pkg.Rand(0))
        sets5 = make_trackers(ctx, pkg, ell5, [1000 + i for i in range(2)])
        pre5 = b"".join(sets5[i % 2] for i in range(B5))
        size5 = proof_size_for(ell5)
        t_w, t_b = [], []
        for it in range(3):
            flush.zero_()
            ctx.engine_stats(reset=True)
            rands = [pkg.Rand((rank << 40) | ((90 + it) << 20) | i) for i in range(B5)]
            barrier()
            t1 = time.perf_counter()
            post5, proofs5, st5 = ctx.whisk_generate_shuffle_proof_batch(crs5, pre5, rands, proof_size=size5)
            ok5, vs5 = ctx.whisk_is_valid_shuffle_proof_batch(crs5, pre5, post5, proofs5, rands, proof_size=size5)
            torch.cuda.synchronize()
            t_w.append(time.perf_counter() - t1)
            t_b.append(ctx.engine_busy_ms() / 1e3)
            assert st5 == [0] * B5 and ok5 == [1] * B5 and vs5 == [0] * B5, "n=512 round trip failed"
        tw, tbz = max_over_ranks(sum(t_w[1:])), max_over_ranks(sum(t_b[1:]))
        n512 = {"workload": "whisk-style round trips at shuffled_elements=508 (n=512), proof buffer %d B" % size5,
                "proofs_per_gpu_per_step": B5, "e2e_value": world * B5 * 2 / tw, "value": world * B5 * 2 / tbz, "unit": UNIT,
                "timing": "2 batches after 1 warm-up; e2e = wall clock through the C ABI, value = device busy time"}
        crs5.close()

    msm = adv = msm_cpu = None
    if not args.no_msm:
        sizes = [int(x) for x in args.msm_sizes.split(",")] if args.msm_sizes else list(range(10, 23))
        cpu_sizes = [] if args.no_cpu_baseline else [s for s in (10, 14, 16, 20) if s <= max(sizes)]
        msm, adv, msm_cpu = msm_sweep(ctx, pkg, sizes, 2, world, rank, peak_modmul, barrier, cpu_sizes)

    total_proofs = world * B * args.steps
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        top = max(stats, key=lambda k: stats[k]["ms"])
        tk = stats[top]
        n_launch = max(1, tk["launches"])
        achieved = tk["modmul"] / (tk["ms"] * 1e-3) if tk["ms"] else 0.0
        traffic, traffic_src = None, None
        try:  # dram bytes per launch of the dominant kernel class: CACHED figure from an ncu capture of this command
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            if tj.get("batch") == B:
                traffic, traffic_src = tj.get(top), tj.get("source", "profiles/traffic.json")
        except Exception:
            pass
        timed = stats_timed[top]
        roofline = {
            "bound": "int_alu", "kernel": top + (" (k_msm_recode + k_msm_warp_gmem + k_msm_chunk_sum + k_msm_combine_tp)"
                                                 if top == "msm_small" else ""),
            "achieved": achieved / 1e9, "peak": peak_modmul / 1e9,
            "unit": "Gmodmul/s", "frac": achieved / peak_modmul if peak_modmul else None, "traffic": traffic,
            "traffic_source": (f"cached: {traffic_src} (ncu dram__bytes of this command, not measured in this run)"
                               if traffic is not None else None),
            "measured_in": "one extra step of the same batch with 1 lane, CUDA events on the launching stream "
                           "(kernel intervals of concurrent lanes overlap and would count each other's time)",
            "timed_region": {"lanes": args.lanes or 4, "launches": timed["launches"],
                             "avg_launch_ms_overlapped": timed["ms"] / max(1, timed["launches"])},
            "pipe_ceiling": "a wide multiply (IMAD.WIDE / IMAD.HI, with or without carry) issues at 32 lanes/clk/SM on "
                            "sm_100a, half the nominal 64 (profiles/r2_probe2.txt): no 32-bit-limb product can exceed "
                            "frac 0.5; DFMA and reduced-radix forms were built and measured (profiles/r2_fieldmul_variants.txt)",
            "peak_source": "64 IMAD lanes/clk/SM x SM count x SM clock measured live (dependent IMAD chain, cdl_int_peak "
                           "kind 0) / 300 per modmul",
            "avg_launch_ms": tk["ms"] / n_launch, "launches": tk["launches"],
            "algorithmic_modmul_per_launch": tk["modmul"] / n_launch,
            "work_definition": "SURVEY.md 8d modmul(N) per MSM task at the REFERENCE's term count N (a base the prover "
                               "writes as several CRS-point terms counts once), summed over the tasks of a launch",
            "hbm": {"achieved_gbs": tk["bytes"] / (tk["ms"] * 1e-3) / 1e9 if tk["ms"] else 0.0, "peak_gbs": hbm_peak,
                    "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"},
            "per_kernel": {k: {"ms": v["ms"], "launches": v["launches"],
                               "gmodmul_per_s": (v["modmul"] / (v["ms"] * 1e-3) / 1e9) if v["ms"] else 0.0,
                               "share_of_device_time": v["ms"] / dev_ms if dev_ms else 0.0} for k, v in stats.items()},
        }
        h2d = B * (ELL * 96) + B * (2 * ELL * 96 + 4576)   # generate: pre ; validate: pre + post + proof
        d2h = B * (ELL * 96 + 4576) + B * 8                # generate: post + proof ; validate: verdict + status
        line = {
            "metric": METRIC, "value": total_proofs / dev_max, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * wall_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32 (12x32-bit Montgomery limbs, IMAD.WIDE)",
            "data": "synthetic", "config": config_dict(B, world, args.lanes or 4, info),
            "e2e": {"value": total_proofs / wall_max, "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h,
                    "note": "C ABI with host buffers; stage descriptors/scalars (about 36 B per MSM term) are extra H2D"},
            "gpu_launches": int(launches),
            "roofline": roofline,
            "clocks": sampler.summary(),
        }
        if config4 is not None:
            line["config4"] = config4
        if n512 is not None:
            line["n512"] = n512
        pool_cores = None
        if world == 1 and not args.no_latency:
            sp = {"what": "curdleproof.Prove / Verify, one proof at a time (configs 1-3), wall clock through the C ABI",
                  "reference_published_ms": {"prove": [96.4, 150.2, 412.5], "verify": [12.0, 12.3, 20.8],
                                             "hardware": "Ryzen 7 3800XT, README.md:19-26"},
                  "sizes": single_proof_latency(ctx, pkg)}
            if not args.no_cpu_baseline:
                try:  # the same shapes on the CPU port, one proof on one core (BASELINE.md §2.3)
                    pool, pool_cores = cpu_pool()
                    res = pool.map(_w_single, [60, 124, 508])
                    sp["cpu_port_ms"] = [{"shuffled_elements": e, "prove_ms": r[0] * 1e3, "verify_ms": r[1] * 1e3, "cores": 1}
                                         for e, r in zip((60, 124, 508), res)]
                except Exception as e:
                    sp["cpu_port_ms"] = {"failed": str(e)}
            line["single_proof"] = sp
        if msm is not None:
            line["msm"] = {"workload": "standalone G1 MSM, random points/scalars, device resident"
                                       + (f", windows dealt to {world} ranks + NCCL all-gather" if world > 1 else ""),
                           "sizes": msm, "adversarial": adv, "cpu_baseline": msm_cpu}
        if world == 1 and not args.no_cpu_baseline:
            try:
                pool, cores = cpu_pool()
                per_worker = 3
                n, dt = cpu_roundtrip_sample(per_worker)
                line["cpu_baseline"] = {
                    "value": n / dt, "unit": UNIT, "cores": cores, "kind": "port",
                    "sample": f"{cores} persistent worker processes x {per_worker} Whisk n=128 round trips on the CPU oracle "
                              f"(C 6x64 Montgomery port + Python orchestration), {dt:.1f} s; workers, CRS and trackers set up "
                              f"before the timed region",
                    "published_reference": "README.md:20,24 — Prove 150.2 ms + Verify 12.3 ms on a Ryzen 7 3800XT "
                                           "(16 threads) = 6.2 proofs/s excl. ShufflePermuteCommit and decompression",
                }
            except Exception as e:  # the baseline is reported, never required for the GPU number
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"failed: {e}"}
        print(json.dumps(line), flush=True)
        if _POOL is not None:
            _POOL[0].close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=4096, help="independent Whisk round trips per GPU per step")
    ap.add_argument("--batch512", type=int, default=384, help="round trips per GPU per step of the n=512 line")
    ap.add_argument("--verify-total", type=int, default=VERIFY_TOTAL, help="proofs of config 4, sharded over the ranks")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--lanes", type=int, default=-1,
                    help="concurrent sub-batches per GPU (0 = library default; -1 = 6, or 8 when a rank has fewer than "
                         "8 host cores: measured best on 16 / 4 cores per GPU)")
    ap.add_argument("--no-msm", action="store_true", help="skip the standalone MSM sweep")
    ap.add_argument("--no-latency", action="store_true", help="skip the single-proof latency lines")
    ap.add_argument("--no-config4", action="store_true", help="skip the sharded batched-verification pass")
    ap.add_argument("--no-n512", action="store_true", help="skip the n=512 throughput line")
    ap.add_argument("--msm-sizes", default="", help="comma separated log2 sizes for the MSM sweep")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the last timed step's post-trackers, proofs and verdicts (rank 0's batch) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    if args.lanes < 0:
        world_ = max(1, int(os.environ.get("WORLD_SIZE", "1")))
        args.lanes = 6 if (os.cpu_count() or 1) // world_ >= 8 else 8
    if args.impl == "reference":
        reference_main(args)
    else:
        gpu_main(args)


if __name__ == "__main__":
    main()
