"""The launch-size crossovers of the kernel launchers, read from the CUDA sources, and a restatement of the MSM
window-combine schedules and of the Pippenger bucket fill on discrete logarithms, so that a test can show that a
crafted MSM task makes a combine step add two equal or two opposite points, or fills a bucket with a known multiset.
Shared by test_crossovers_cpu.py (no GPU), test_gpu_crossovers.py and test_gpu_msm_repeated_bases.py.

Every point of a crafted task is a multiple a * G of the generator, so a point is its discrete log a mod r (0 is
the point at infinity) and phi(P) = lambda * P is lambda * a."""
from __future__ import annotations

import os
import re

from oracle import bls12381 as b

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "go-curdleproofs_b200", "csrc")
R = b.R
LAMBDA = 0xAC45A4010001A40200000000FFFFFFFF  # glv.cuh LAM: z^2 - 1, phi(P) = lambda * P on G1

# (file, regex with one integer group) for every threshold a test derives its sizes from
SOURCES = {
    "kQuadMaxOps": ("k_elem.cu", r"constexpr int kQuadMaxOps\s*=\s*(\d+);"),
    "kEB": ("k_elem.cu", r"constexpr int kEB\s*=\s*(\d+);"),
    "kCombineQuadMaxTasks": ("k_msm_tp.cu", r"constexpr int kCombineQuadMaxTasks\s*=\s*(\d+);"),
    "kMsmChunk": ("launch.h", r"constexpr uint32_t kMsmChunk\s*=\s*(\d+);"),
    "kMsmSplitThreshold": ("launch.h", r"constexpr int kMsmSplitThreshold\s*=\s*(\d+);"),
    "kMsmSplitTerms": ("launch.h", r"constexpr size_t kMsmSplitTerms\s*=\s*(\d+);"),
    "kBigMsmThreshold": ("launch.h", r"constexpr size_t kBigMsmThreshold\s*=\s*(\d+);"),
    "kBigQuadMaxOutputs": ("k_msm_big.cu", r"constexpr int kBigQuadMaxOutputs\s*=\s*(\d+);"),
    "kMsmC": ("k_msm.cu", r"constexpr int kMsmC\s*=\s*(\d+);"),
    "kBigLargeBucket": ("k_msm_big.cu", r"constexpr uint32_t kBigLargeBucket\s*=\s*(\d+);"),
    "kBigMaxBaRounds": ("launch.h", r"constexpr int kBigMaxBaRounds\s*=\s*(\d+);"),
}


def _src(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def const(name):
    fname, pat = SOURCES[name]
    m = re.search(pat, _src(fname))
    if m is None:
        raise LookupError(f"{name} not found in {fname}")
    return int(m.group(1))


def jac_to_affine_bounds():
    """[(E, n_min)] of launch_jac_to_affine, largest E first: k_jac_to_affine<E> from n_min points (k_elem.cu)"""
    body = re.search(r"void launch_jac_to_affine\(.*?\n}\n", _src("k_elem.cu"), re.S).group(0)
    found = re.findall(r"if \(n >= (\d+) \* (\d+) \* (\d+)\)\s*{\s*const int threads = \(n \+ (\d+)\) / (\d+);\s*"
                       r"k_jac_to_affine<(\d+)>", body)
    if not found:
        raise LookupError("launch_jac_to_affine bounds not found")
    out = []
    for e, sms, tpb, _, div, tmpl in found:
        assert e == div == tmpl, (e, div, tmpl)
        out.append((int(e), int(e) * int(sms) * int(tpb)))
    return out


def jac_to_affine_e(n):
    for e, lo in jac_to_affine_bounds():
        if n >= lo:
            return e
    return 1


def jac_to_affine_threads(n):
    """grid threads T of the launch: thread t takes points t, t + T, .., t + (E - 1) T"""
    e = jac_to_affine_e(n)
    return e, (-(-n // e) + 63) // 64 * 64


def big_c_table():
    m = re.search(r"int big_msm_pick_c\(size_t n\) {.*?static const int table\[\] = {([\d,\s]+)};\s*"
                  r"return lg <= (\d+) \? table\[lg\] : (\d+);", _src("k_msm_big.cu"), re.S)
    if m is None:
        raise LookupError("big_msm_pick_c table not found")
    return [int(x) for x in m.group(1).split(",")], int(m.group(2)), int(m.group(3))


def big_pick_c(n):
    """restatement of big_msm_pick_c"""
    table, top, last = big_c_table()
    lg = n.bit_length() - 1
    return table[lg] if lg <= top else last


def big_reduce1_outputs(n):
    """outputs of the first bucket reduction of a one-device Pippenger MSM of n terms (launch_big_msm)"""
    c = big_pick_c(n)
    W, M = (128 + c - 1) // c, 1 << (c - 1)
    return W * (M // min(M, 8))


def big_large(n, c, rounds):
    """restatement of BigMsmDims::large (big_msm_dims): a bucket of more entries than this after the batch-affine
    rounds is summed by k_big_slice / k_big_large_finish instead of one k_big_accum thread"""
    mean = 2 * n // (1 << (c - 1)) + 1
    return min(max(8 * ((mean >> rounds) + 1), 64), const("kBigLargeBucket"))


def pick_chunk(nterm, sm_count):
    """restatement of msm_tp_pick_chunk"""
    return 32 if nterm // const("kMsmChunk") < 2 * sm_count else const("kMsmChunk")


def msm_batch_path(lengths):
    """'small' (k_msm_small) or 'tp' (throughput kernels) for one cdl_g1_msm_batch launch (Engine::run_msm)"""
    tp = len(lengths) >= const("kMsmSplitThreshold") or max(lengths, default=0) > const("kMsmSplitTerms")
    return "tp" if tp else "small"


# ------------------------------------------------------------------------------------------------- schedules
def glv_split(hc, scalars):
    """(|k1|, k2, neg1, neg2) of every canonical scalar, from the product's glv_decompose (hostcheck build)"""
    import ctypes

    n = len(scalars)
    k = b"".join(s.to_bytes(32, "little") for s in scalars)
    k1, k2 = ctypes.create_string_buffer(16 * n), ctypes.create_string_buffer(16 * n)
    n1, n2 = (ctypes.c_int * n)(), (ctypes.c_int * n)()
    hc.hc_glv_decompose(k, k1, k2, n1, n2, n)
    return [(int.from_bytes(k1.raw[16 * i:16 * i + 16], "little"), int.from_bytes(k2.raw[16 * i:16 * i + 16], "little"),
             bool(n1[i]), bool(n2[i])) for i in range(n)]


def halves(hc, task):
    """the (magnitude, discrete log) of both GLV halves of every term (a, s) of a task"""
    out = []
    for (a, _), (k1, k2, n1, n2) in zip(task, glv_split(hc, [s % R for _, s in task])):
        out.append((k1, (-a if n1 else a) % R))
        out.append((k2, (-(LAMBDA * a) if n2 else LAMBDA * a) % R))
    return out


def biased_digits(k):
    """digits of a GLV half as the 4-bit kernels read them: glv_bias, then glv_digit"""
    kp = k + int("0" + "8" * 31, 16)
    return [((kp >> (4 * w)) & 15) - (8 if w != 31 else 0) for w in range(32)]


def signed_digits(k, c):
    """restatement of k_big_digits (test_msm_partition_cpu.signed_digits)"""
    from test_msm_partition_cpu import signed_digits as sd

    return sd(k, c)


def window_sums(hs, digits):
    W = len(digits(0))
    S = [0] * W
    for k, a in hs:
        for w, d in enumerate(digits(k)):
            S[w] = (S[w] + d * a) % R
    return S


def _meet(x, y):
    """'equal' / 'opposite' when an addition x + y of two finite points is an exceptional case"""
    if x == 0 or y == 0:
        return None
    return "equal" if x == y else "opposite" if (x + y) % R == 0 else None


def horner(S, c):
    """acc = sum_w 2^(c w) S_w walked from the top window (k_msm_combine_tp / _quad, k_big_horner):
    (result, [(window, kind)] of the exceptional additions)"""
    acc, hits = 0, []
    for w in range(len(S) - 1, -1, -1):
        acc = acc * (1 << c) % R
        kind = _meet(acc, S[w])
        if kind:
            hits.append((w, kind))
        acc = (acc + S[w]) % R
    return acc, hits


def tree(S, c):
    """k_msm_small's binary tree: level L adds win[2g] and 2^(c 2^L) win[2g + 1]:
    (result, [(level, pair, kind)] of the exceptional additions)"""
    win, hits, level = list(S), [], 0
    while len(win) > 1:
        nxt = []
        for g in range(len(win) // 2):
            lo, hi = win[2 * g], win[2 * g + 1] * pow(2, (c << level), R) % R
            kind = _meet(lo, hi)
            if kind:
                hits.append((level, g, kind))
            nxt.append((lo + hi) % R)
        win, level = nxt, level + 1
    return win[0], hits


def small_schedule(hc, task):
    hs = halves(hc, task)
    S = window_sums(hs, biased_digits)
    return {"horner": horner(S, const("kMsmC")), "tree": tree(S, const("kMsmC"))}


def big_schedule(hc, task, c):
    hs = halves(hc, task)
    return horner(window_sums(hs, lambda k: signed_digits(k, c)), c)


# ------------------------------------------------------------------------------------------------- crafted tasks
def collision_tasks():
    """Tasks of (discrete log, scalar) terms for the 4-bit window kernels: for L = 0 .. 4, [G, 2^(4 2^L) G] times
    [2^(4 2^L), 1] puts G in window 2^L and 2^(4 2^L) G in window 0, so k_msm_small's tree adds two equal points
    at level L and the Horner walks add them at window 0 (L = 0: the last step adds 16G to 16G); with -2^(4 2^L) G
    the two are opposite and the task sums to infinity.  {name: (task, expected tree level)}"""
    out = {}
    c = const("kMsmC")
    for L in range(5):
        e = 1 << (c << L)
        out[f"equal-L{L}"] = ([(1, e), (e, 1)], L)
        out[f"opposite-L{L}"] = ([(1, e), (R - e, 1)], L)
    return out


def padded_collision_task(n, kind):
    """the L = 0 task of collision_tasks padded to n terms with zero scalars on the bases 2 G, 3 G, .."""
    task = collision_tasks()[f"{kind}-L0"][0]
    return task + [(2 + i, 0) for i in range(n - len(task))]


def big_collision_task(n, kind):
    """one Pippenger MSM of n terms (n > kBigMsmThreshold): [G, +-2^c G] times [2^c, 1] with c = big_pick_c(n),
    padded with zero scalars on the bases 2 G, 3 G, ..: the last Horner step adds two equal / opposite points"""
    e = 1 << big_pick_c(n)
    task = [(1, e), (e if kind == "equal" else R - e, 1)]
    return task + [(2 + i, 0) for i in range(n - 2)]


# ------------------------------------------------------------------------------------------------- bucket contents
def big_buckets(hc, task, c):
    """restatement of k_big_digits' bucket fill for a one-device Pippenger MSM: {(window, |digit|): sorted discrete
    logs of the bucket's entries}.  Entry = the half's base (P or phi(P)), negated when the digit's sign and the
    half's GLV sign differ; the order the scatter leaves inside a bucket is not modelled (it varies)."""
    out = {}
    for k, a in halves(hc, task):
        for w, d in enumerate(signed_digits(k, c)):
            if d:
                out.setdefault((w, abs(d)), []).append(a if d > 0 else (R - a) % R)
    return {key: sorted(v) for key, v in out.items()}


KNOWN_WINDOWS = 3  # windows 0 .. 2 carry the digit of a known-bucket scalar, the others are zero


def known_bucket_task(c, rounds):
    """Terms (discrete log, scalar) on the bases P = G (log 1) and -P whose Pippenger buckets hold known multisets
    at window width c: a scalar d * (1 + 2^c + 2^(2c)) with d in [1, 2^(c-1)] is far below lambda / 2, so the GLV
    split leaves it whole (k2 = 0, no negation), and its c-bit digits are d, d, d and zeros: no carry, so it puts
    exactly one +P into bucket (w, d) of windows 0 .. 2.  For every count m in {1, 2, 3, 2^R - 1, 2^R, 2^R + 1}
    (R = rounds) m terms share a digit d_m (d = 2^(c-1), the largest digit, first), and one more digit holds one
    term on P and one on -P.  Returns (task, {bucket: intended sorted multiset}).  Whatever order the scatter
    leaves, the first batch-affine round then adds (P, P), (P, inf), (inf, inf) and (P, -P) pairs, and round j
    adds (2^(j-1) P, 2^(j-1) P) in the buckets of 2^R entries."""
    M = 1 << (c - 1)
    spread = sum(1 << (c * w) for w in range(KNOWN_WINDOWS))
    counts = sorted({1, 2, 3, (1 << rounds) - 1, 1 << rounds, (1 << rounds) + 1} - {0})
    task, want, d = [], {}, M
    for m in counts:
        task += [(1, d * spread)] * m
        want.update({(w, d): [1] * m for w in range(KNOWN_WINDOWS)})
        d -= 1
    task += [(1, d * spread), (R - 1, d * spread)]
    want.update({(w, d): [1, R - 1] for w in range(KNOWN_WINDOWS)})
    return task, want
