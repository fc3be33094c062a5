"""The kernels that only large launches take, against the CPU oracle or closed-form (sum a_i s_i) * G, on both
sides of every launch-size crossover.  Sizes come from the thresholds in the CUDA sources (crossovers.py) and the
device's SM count; every case also checks, with torch.profiler, which kernel the launch ran.

Inputs repeat a set of SET distinct (point, scalar) pairs, so the oracle computes SET products however long the
call; the set holds the point at infinity, +-P pairs, zero scalars, scalars with limbs >= r up to 2^256 - 1 and
(MSMs) tasks crafted so that a window-combine addition meets two equal or two opposite points (test_crossovers_cpu
shows that they do under the kernels' digit schedules)."""
import os
import random
import re
from concurrent.futures import ThreadPoolExecutor

import pytest

import crossovers as X
from oracle import bls12381 as b
from util import R, affs_enc, fr_dec, fr_enc, jac_dec, jac_enc

pytestmark = pytest.mark.gpu

SET = 4096
G = b.G1_GEN


# ------------------------------------------------------------------------------------------------- helpers
def launched(fn):
    """(fn(), the set of kernel names fn launched) from a torch.profiler capture with CUDA activities"""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
    return out, {e.key for e in prof.key_averages()}


def ran(names, kernel):
    """kernel (a template with its arguments, e.g. k_jac_to_affine<2>) is among the demangled names"""
    pat = re.compile(r"(^|[\s:])" + re.escape(kernel) + r"\(")
    return any(pat.search(n) for n in names)


def expect_kernels(names, yes, no):
    print("kernels:", sorted({m.group(0) for n in names for m in [re.search(r"\bk_\w+(<\w+>)?", n)] if m}))
    assert all(ran(names, k) for k in yes) and not any(ran(names, k) for k in no), (
        yes, no, sorted(n for n in names if "k_" in n))


_CB = None


def _cb():
    global _CB
    if _CB is None:
        from oracle.cbackend import CBackend

        _CB = CBackend(accelerate_keccak=False)
    return _CB


def _split(fn, *cols):
    """fn over chunks of the columns on host threads (the oracle's ctypes calls drop the GIL)"""
    n = len(cols[0])
    step = max(64, -(-n // (4 * (os.cpu_count() or 1))))
    with ThreadPoolExecutor(os.cpu_count() or 1) as ex:
        parts = ex.map(lambda i: fn(*[c[i:i + step] for c in cols]), range(0, n, step))
        return [p for part in parts for p in part]


def omul(pts, ks):
    return _split(_cb().mul_batch, pts, ks)


def ofold(L, R_, x):
    return _split(lambda l, r: _cb().fold(l, r, x), L, R_)


def rep(data, unit, n, shift=0):
    """n units of `unit` bytes: the units of data rotated by `shift`, repeated"""
    k = len(data) // unit
    d = data[unit * shift:] + data[:unit * shift]
    return (d * -(-n // k))[:unit * n]


def first_diff(got, want, unit):
    for i in range(0, max(len(got), len(want)), unit):
        if got[i:i + unit] != want[i:i + unit]:
            return f"first difference at item {i // unit} of {len(want) // unit}"
    return "equal"


@pytest.fixture(scope="module")
def sm_count(ctx):
    return ctx.device_info()["sm_count"]


@pytest.fixture(scope="module")
def base():
    """SET points a_i G (every 97th at infinity, +-P pairs) and SET raw 32-byte scalars with their values"""
    rnd = random.Random(29)
    a = [rnd.randrange(1, R) for _ in range(SET)]
    for i in range(0, SET, 97):
        a[i] = 0
    for i in range(3, SET, 89):
        a[i] = (R - a[i - 1]) % R
    pts = omul([G] * SET, a)
    raw = bytearray(rnd.randbytes(32 * SET))  # raw limbs: about half of them >= r
    special = [bytes(32), fr_enc(1), fr_enc(R - 1), b"\xff" * 32, R.to_bytes(32, "little"),
               (R + 5).to_bytes(32, "little"), ((1 << 256) - R).to_bytes(32, "little")]
    for i, s in enumerate(special):
        raw[32 * i:32 * i + 32] = s
    for i in range(9, SET, 61):
        raw[32 * i:32 * i + 32] = bytes(32)
    raw = bytes(raw)
    vals = [fr_dec(raw[32 * i:32 * i + 32]) for i in range(SET)]
    return {"a": a, "pts": pts, "enc": affs_enc(pts), "raw": raw, "vals": vals}


def elem_sizes():
    """both sides of kQuadMaxOps, and a size that gives every thread of a persistent k_scalar_mul grid (at most
    4 CTAs of 64 threads per SM on 148 SMs) more than kEB items: a second pass of its item loop"""
    q = X.const("kQuadMaxOps")
    big = (1 << 19) + 3
    assert big > X.const("kEB") * 148 * 4 * 64
    return (q, q + 1, big)


def elem_kernels(n):
    q = X.const("kQuadMaxOps")
    return (["k_scalar_mul_quad"], ["k_scalar_mul"]) if n <= q else (["k_scalar_mul"], ["k_scalar_mul_quad"])


# ------------------------------------------------------------------------------------------------- elementwise
@pytest.mark.parametrize("n", elem_sizes())
def test_scalar_mul_per_element(ctx, base, n):
    want = affs_enc(omul(base["pts"], base["vals"]))
    got, names = launched(lambda: ctx.g1_scalar_mul_affine(rep(base["enc"], 96, n), rep(base["raw"], 32, n), broadcast=False))
    assert got == rep(want, 96, n), first_diff(got, rep(want, 96, n), 96)
    expect_kernels(names, *elem_kernels(n))


@pytest.mark.parametrize("n", elem_sizes())
def test_scalar_mul_broadcast(ctx, base, n):
    """one scalar for every point: zero (every result at infinity), r - 1, 2^256 - 1 and a random one"""
    for s in (bytes(32), fr_enc(R - 1), b"\xff" * 32, base["raw"][32 * 100:32 * 101]):
        want = affs_enc(omul(base["pts"], [fr_dec(s)] * SET))
        if s == bytes(32):
            assert want == bytes(96 * SET)
        got, names = launched(lambda: ctx.g1_scalar_mul_affine(rep(base["enc"], 96, n, 5), s, broadcast=True))
        assert got == rep(want, 96, n, 5), (s.hex(), first_diff(got, rep(want, 96, n, 5), 96))
        expect_kernels(names, *elem_kernels(n))


@pytest.mark.parametrize("n", elem_sizes())
def test_fold(ctx, base, n):
    """L + x R with L = -x R (infinity), L = x R (a doubling), L or R at infinity among random pairs; then a
    call whose results are all at infinity (L at infinity, x = 0)"""
    pts = base["pts"]
    for x in (fr_enc(random.Random(n).randrange(R)), b"\xff" * 32):
        xv = fr_dec(x)
        Rr = pts[1:] + pts[:1]
        L = list(pts)
        sel = [i for i in range(SET) if i % 50 in (5, 6)]
        xr = dict(zip(sel, omul([Rr[i] for i in sel], [xv] * len(sel))))
        for i in range(SET):
            if i % 50 == 5:
                L[i] = b.g1_neg(xr[i])
            elif i % 50 == 6:
                L[i] = xr[i]
            elif i % 50 == 7:
                L[i] = None
            elif i % 50 == 8:
                Rr[i] = None
        want = ofold(L, Rr, xv)
        assert want[5] is None and want[6] is not None
        want = affs_enc(want)
        got, names = launched(lambda: ctx.g1_fold(rep(affs_enc(L), 96, n), rep(affs_enc(Rr), 96, n), x))
        assert got == rep(want, 96, n), (x.hex(), first_diff(got, rep(want, 96, n), 96))
        expect_kernels(names, *elem_kernels(n))
    got, names = launched(lambda: ctx.g1_fold(bytes(96 * n), rep(base["enc"], 96, n), bytes(32)))
    assert got == bytes(96 * n)
    expect_kernels(names, *elem_kernels(n))


# ------------------------------------------------------------------------------------------------- to affine
def affine_sizes():
    (e8, n8), (e2, n2) = X.jac_to_affine_bounds()
    return (n2 - 1, n2, n2 + 1, n8 - 1, n8, n8 + 5)


@pytest.mark.parametrize("n", affine_sizes())
def test_batch_to_affine(ctx, base, n):
    """Z != 1 everywhere; Z = 0 (gnark's (1, 1, 0)) at the first and last point of a few threads and at every
    point of one thread.  The reference inverts Z with pow(Z, -1, p)."""
    rnd = random.Random(n)
    jac = b"".join(jac_enc(p, rnd.randrange(2, b.P)) for p in base["pts"])
    want = affs_enc([jac_dec(jac[144 * i:144 * i + 144]) for i in range(SET)])
    E, T = X.jac_to_affine_threads(n)
    J, W = bytearray(rep(jac, 144, n, 7)), bytearray(rep(want, 96, n, 7))
    inf = set()
    for t in (0, 1, T // 2, min(T, n) - 1, (n - 1) % T):
        items = [t + e * T for e in range(E) if t + e * T < n]
        inf.update((items[0], items[-1]))
    inf.update(t for t in range(5, n, T))  # every point of thread 5
    for i in inf:
        J[144 * i:144 * i + 144] = jac_enc(None)
        W[96 * i:96 * i + 96] = bytes(96)
    got, names = launched(lambda: ctx.g1_batch_to_affine(bytes(J)))
    assert got == bytes(W), first_diff(got, bytes(W), 96)
    others = [f"k_jac_to_affine<{e}>" for e in (1, 2, 8) if e != E]
    expect_kernels(names, [f"k_jac_to_affine<{E}>"], others)


# ------------------------------------------------------------------------------------------------- MSM batches
@pytest.fixture(scope="module")
def crafted():
    """the collision tasks as (point, discrete log, scalar) terms"""
    tasks = [t for t, _ in X.collision_tasks().values()]
    logs = sorted({a for t in tasks for a, _ in t})
    pt = dict(zip(logs, omul([G] * len(logs), logs)))
    return [[(pt[a], a, s) for a, s in t] for t in tasks]


def msm_batch_case(ctx, base, crafted, lengths, seed):
    """one cdl_g1_msm_batch call: the crafted tasks first, then tasks of the given lengths drawn from the set
    (with an empty and a one-term task), and a crafted task at the last index; checked against
    (sum a_i s_i mod r) G.  Returns the kernel names and the task lengths."""
    rnd = random.Random(seed)
    tasks = list(crafted)
    for n in lengths:
        idx = [rnd.randrange(SET) for _ in range(n)]
        tasks.append([(base["pts"][i], base["a"][i], base["raw"][32 * j:32 * j + 32])
                      for i, j in zip(idx, (rnd.randrange(SET) for _ in range(n)))])
    tasks.append(crafted[0])
    offs, pts, sc, ks = [0], [], [], []
    for t in tasks:
        offs.append(offs[-1] + len(t))
        k = 0
        for p, a, s in t:
            pts.append(p)
            s = s if isinstance(s, bytes) else fr_enc(s)
            sc.append(s)
            k += a * fr_dec(s)
        ks.append(k % R)
    want = affs_enc(omul([G] * len(ks), ks))
    got, names = launched(lambda: ctx.g1_msm_batch(affs_enc(pts), b"".join(sc), offs))
    assert got == want, first_diff(got, want, 96)
    assert got[96 * 1:96 * 2] == bytes(96)  # the first opposite task
    return names, [len(t) for t in tasks]


def _lengths(rnd, count, choices):
    out = [rnd.choice(choices) for _ in range(count)]
    out[:2] = [0, 1]
    return out


@pytest.mark.parametrize("side", [-1, 0])
def test_msm_batch_task_count(ctx, base, crafted, side):
    n = X.const("kMsmSplitThreshold") + side
    ls = _lengths(random.Random(1), n - len(crafted) - 1, [0, 1, 2, 7, 16, 33, 64])
    names, lens = msm_batch_case(ctx, base, crafted, ls, 10 + side)
    assert len(lens) == n
    if X.msm_batch_path(lens) == "small":
        assert side == -1
        expect_kernels(names, ["k_msm_small"], ["k_msm_warp_gmem"])
    else:
        assert side == 0
        expect_kernels(names, ["k_msm_warp_gmem", "k_msm_combine_quad"], ["k_msm_small"])


@pytest.mark.parametrize("side", [0, 1])
def test_msm_batch_longest_task(ctx, base, crafted, side):
    t = X.const("kMsmSplitTerms") + side
    ls = _lengths(random.Random(2), 20, [3, 9, 40, 200]) + [t]
    names, lens = msm_batch_case(ctx, base, crafted, ls, 20 + side)
    assert max(lens) == t and X.msm_batch_path(lens) == ("tp" if side else "small")
    if side:
        expect_kernels(names, ["k_msm_warp_gmem", "k_msm_combine_quad"], ["k_msm_small"])
    else:
        expect_kernels(names, ["k_msm_small"], ["k_msm_warp_gmem"])


@pytest.mark.parametrize("side", [-1, 0])
def test_msm_batch_total_terms(ctx, base, crafted, sm_count, side):
    """32-term chunks below 2 sm_count kMsmChunk terms, kMsmChunk-term chunks from there (one bucket kernel:
    the chunk length is checked through the restatement of msm_tp_pick_chunk)"""
    total = 2 * sm_count * X.const("kMsmChunk") + side
    rnd = random.Random(3)
    fixed = sum(len(t) for t in crafted) + len(crafted[0])
    ls = [0, 1]
    while sum(ls) + fixed < total:
        ls.append(min(rnd.choice([5, 64, 127, 128, 129, 300, 384]), total - fixed - sum(ls)))
    names, lens = msm_batch_case(ctx, base, crafted, ls, 30 + side)
    assert sum(lens) == total and len(lens) <= X.const("kCombineQuadMaxTasks")
    assert X.pick_chunk(total, sm_count) == (32 if side else X.const("kMsmChunk"))
    expect_kernels(names, ["k_msm_warp_gmem", "k_msm_combine_quad"], ["k_msm_small", "k_msm_combine_tp"])


@pytest.mark.parametrize("side", [0, 1])
def test_msm_batch_combine_kernel(ctx, base, crafted, side):
    n = X.const("kCombineQuadMaxTasks") + side
    ls = _lengths(random.Random(4), n - len(crafted) - 1, [0, 1, 2, 3, 5, 8])
    names, lens = msm_batch_case(ctx, base, crafted, ls, 40 + side)
    assert len(lens) == n
    if side:
        expect_kernels(names, ["k_msm_warp_gmem", "k_msm_combine_tp"], ["k_msm_combine_quad"])
    else:
        expect_kernels(names, ["k_msm_warp_gmem", "k_msm_combine_quad"], ["k_msm_combine_tp"])


# ------------------------------------------------------------------------------------------------- single MSMs
@pytest.mark.parametrize("kind", ["equal", "opposite"])
@pytest.mark.parametrize("side", [0, 1])
def test_msm_collision_at_pippenger_threshold(ctx, side, kind):
    """cdl_g1_msm at kBigMsmThreshold terms (throughput path, 4-bit Horner) and one more (Pippenger, c-bit
    Horner): a task whose last Horner step adds two equal / opposite points, padded with zero scalars"""
    n = X.const("kBigMsmThreshold") + side
    task = X.big_collision_task(n, kind) if side else X.padded_collision_task(n, kind)
    pts = omul([G] * n, [a for a, _ in task])
    want = b.g1_mul(G, sum(a * s for a, s in task) % R)
    got, names = launched(lambda: ctx.g1_msm(affs_enc(pts), b"".join(fr_enc(s) for _, s in task)))
    assert jac_dec(got) == want
    assert (want is None) == (kind == "opposite")
    if side:
        expect_kernels(names, ["k_big_horner"], ["k_msm_warp_gmem", "k_msm_small"])
    else:
        expect_kernels(names, ["k_msm_warp_gmem"], ["k_big_horner"])


@pytest.mark.parametrize("n", [(1 << 15) - 1, 1 << 15])
def test_msm_pippenger_reduction_kernels(ctx, base, n):
    """quad bucket reductions up to kBigQuadMaxOutputs outputs, thread-per-output ones above (the window width
    changes at the same size); closed-form result"""
    want = b.g1_mul(G, sum(base["a"][i % SET] * base["vals"][(i + 11) % SET] for i in range(n)) % R)
    got, names = launched(lambda: ctx.g1_msm(rep(base["enc"], 96, n), rep(base["raw"], 32, n, 11)))
    assert jac_dec(got) == want
    if X.big_reduce1_outputs(n) <= X.const("kBigQuadMaxOutputs"):
        expect_kernels(names, ["k_big_reduce1_quad"], ["k_big_reduce1"])
    else:
        expect_kernels(names, ["k_big_reduce1"], ["k_big_reduce1_quad"])


# ------------------------------------------------------------------------------------------------- Whisk batch
def test_whisk_batch_past_every_protocol_threshold(pkg, sm_count):
    """One lane, ell = 124, B = 320 proofs in one call: step 3's 14 MSMs per proof give 4 480 tasks
    (k_msm_combine_tp), the lazy first-round passes 64 elementwise ops per proof (k_elem_ops on the fixed-base
    tables), B_c 259 terms per proof (kMsmChunk-term chunks and k_msm_fixed).  Proofs and post-trackers of
    instances on both sides of the combine crossover (task 4 096 is in proof 292) against the oracle's prover;
    five mutation kinds, some past it, against the oracle's verifier."""
    from oracle import protocol as P, whisk as W
    from oracle.cbackend import CBackend
    from oracle.rand import Rand as ORand
    from test_gpu_parity_batch import KINDS, make_trackers, mutate, oracle_crs

    ell, B, size = 124, 320, 4576
    assert 14 * B > X.const("kCombineQuadMaxTasks") and 64 * B > X.const("kQuadMaxOps")
    assert X.pick_chunk(259 * B, sm_count) == X.const("kMsmChunk") and B >= 64
    c = pkg.Context(0)
    try:
        c.set_lanes(1)
        crs = c.generate_crs(ell, pkg.Rand(0))
        sets = [make_trackers(c, pkg, ell, 1000 + i) for i in range(3)]
        pres = [sets[i % 3] for i in range(B)]
        (post, proofs, status), names = launched(lambda: c.whisk_generate_shuffle_proof_batch(
            crs, b"".join(pres), [pkg.Rand(3000 + i) for i in range(B)]))
        assert status == [0] * B
        expect_kernels(names, ["k_msm_combine_tp", "k_elem_ops", "k_msm_fixed"], [])
        tb = 96 * ell
        posts = [bytes(post[i * tb:(i + 1) * tb]) for i in range(B)]
        prfs = [bytes(proofs[i * size:(i + 1) * size]) for i in range(B)]
        checked = [0, 1, 292, 293, B - 1]
        kinds = {7: 0, 150: 1, 291: 2, 294: 3, 310: 4, 318: 0}
        assert set(kinds.values()) == set(range(KINDS))
        for i, k in kinds.items():
            pres[i], posts[i], prfs[i] = mutate(c, pkg, k, ell, pres[i], posts[i], prfs[i])
        ok, st = c.whisk_is_valid_shuffle_proof_batch(crs, b"".join(pres), b"".join(posts), b"".join(prfs),
                                                      [pkg.Rand(2000 + i) for i in range(B)])
        for i in range(B):
            if i not in kinds:
                assert ok[i] == 1 and st[i] == 0, i
        P.set_backend(CBackend())
        try:
            ocrs = oracle_crs(c, crs, ell)
            split = lambda t: [(t[96 * j:96 * j + 48], t[96 * j + 48:96 * j + 96]) for j in range(ell)]  # noqa: E731
            for i in checked:
                want_post, want_proof = W.generate_whisk_shuffle_proof(ocrs, split(sets[i % 3]), ORand(3000 + i), ell=ell,
                                                                       proof_size=size)
                assert b"".join(x + y for x, y in want_post) == bytes(post[i * tb:(i + 1) * tb]), i
                assert want_proof == bytes(proofs[i * size:(i + 1) * size]), i
            for i in sorted(set(checked) | set(kinds)):
                try:
                    want, err = W.is_valid_whisk_shuffle_proof(ocrs, split(pres[i]), split(posts[i]), prfs[i],
                                                               ORand(2000 + i)), False
                except (W.WhiskError, P.ProofError):
                    want, err = False, True
                assert bool(ok[i]) == want and (st[i] != 0) == err, (i, kinds.get(i), ok[i], st[i])
                assert want == (i not in kinds)
        finally:
            P.set_backend(P.PyBackend())
        crs.close()
    finally:
        c.close()
