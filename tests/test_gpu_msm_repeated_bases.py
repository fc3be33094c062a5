"""MSMs whose bases repeat: one point P many times, P next to -P, one pool index used twice within a task.  The
bucket stages (k_msm_small's and the throughput kernels' bucket warps, the batch-affine pair rounds k_ba_fwd /
k_ba_bwd, k_big_accum, k_big_slice / k_big_large_finish) then add equal and opposite points on purpose rather than
by chance.  Every expected value is in closed form: (sum of the scalars mod r) * P.

The known-bucket cases use the tasks of crossovers.known_bucket_task, whose bucket contents test_crossovers_cpu
checks under a restatement of k_big_digits: whatever order the scatter leaves, every forced batch-affine round
count meets (P, P), (P, inf), (inf, inf), (P, -P) and, in later rounds, (2^j P, 2^j P)."""
import random

import pytest

import crossovers as X
from oracle import bls12381 as b
from test_gpu_crossovers import expect_kernels, launched
from util import R, aff_enc, fr_enc, jac_dec

pytestmark = pytest.mark.gpu

A = 0x1D5F3A7C00E4B6D2  # P = A * G
P = b.g1_mul(b.G1_GEN, A)
P_ENC, NP_ENC = aff_enc(P), aff_enc(b.g1_neg(P))


@pytest.fixture(scope="module")
def mctx(pkg):
    """a context of its own: the forced window widths and round counts, and the large scratch of c = 16 with
    8 rounds, stay with it"""
    c = pkg.Context(0)
    yield c
    c.close()


def times_p(k):
    return b.g1_mul(P, k % R)


def rand_scalars(seed, n):
    rnd = random.Random(seed)
    return [rnd.randrange(R) for _ in range(n)]


def msm_one_base(ctx, ks, signs=None):
    """cdl_g1_msm over P (or -P where signs[i] < 0) with the scalars ks -> affine result"""
    pts = P_ENC * len(ks) if signs is None else b"".join(P_ENC if s > 0 else NP_ENC for s in signs)
    return jac_dec(ctx.g1_msm(pts, b"".join(fr_enc(k) for k in ks)))


# ------------------------------------------------------------------------------------------------- one base
@pytest.mark.parametrize("n", [2, 33, 300, 1024])
def test_one_base_small_and_throughput_paths(mctx, n):
    ks = rand_scalars(n, n)
    path = X.msm_batch_path([n])
    got, names = launched(lambda: msm_one_base(mctx, ks))
    assert got == times_p(sum(ks))
    expect_kernels(names, ["k_msm_small"] if path == "small" else ["k_msm_warp_gmem"],
                   ["k_msm_warp_gmem"] if path == "small" else ["k_msm_small"])
    # all scalars equal, and P / -P pairs with equal scalars (the sum is the point at infinity)
    assert msm_one_base(mctx, [ks[0]] * n) == times_p(n * ks[0])
    half = ks[:n // 2]
    assert msm_one_base(mctx, half + half, [1] * len(half) + [-1] * len(half)) is None


@pytest.mark.parametrize("n", [1025, 4099, 1 << 14, 1 << 16])
def test_one_base_pippenger_every_round_count(mctx, n):
    ks = rand_scalars(n, n)
    want = times_p(sum(ks))
    pts, sc = P_ENC * n, b"".join(fr_enc(k) for k in ks)
    try:
        for c in (8, 11, 16):
            mctx.set_msm_window(c)
            for rounds in range(X.const("kBigMaxBaRounds") + 1):
                mctx.set_msm_batch_affine(rounds)
                assert jac_dec(mctx.g1_msm(pts, sc)) == want, (n, c, rounds)
    finally:
        mctx.set_msm_window(0)
        mctx.set_msm_batch_affine(-1)


@pytest.mark.parametrize("c", [8, 11, 16])
def test_known_bucket_contents(mctx, c):
    """the crafted tasks padded to 1025 terms with zero scalars (Pippenger path), every forced round count"""
    n = 1025
    try:
        mctx.set_msm_window(c)
        for rounds in range(X.const("kBigMaxBaRounds") + 1):
            task, _ = X.known_bucket_task(c, rounds)
            task += [(1, 0)] * (n - len(task))
            want = times_p(sum(s if a == 1 else -s for a, s in task))
            pts = b"".join(P_ENC if a == 1 else NP_ENC for a, _ in task)
            mctx.set_msm_batch_affine(rounds)
            got, names = launched(lambda: jac_dec(mctx.g1_msm(pts, b"".join(fr_enc(s) for _, s in task))))
            assert got == want, (c, rounds)
            if rounds:
                expect_kernels(names, ["k_ba_fwd<false>", "k_ba_bwd<false>", "k_big_accum<true>"], [])
            else:
                expect_kernels(names, ["k_big_accum<false>"], ["k_ba_fwd<false>"])
    finally:
        mctx.set_msm_window(0)
        mctx.set_msm_batch_affine(-1)


@pytest.mark.parametrize("rounds", [0, 3])
def test_slice_path(mctx, rounds):
    """8192 copies of P with one scalar: one bucket per window and GLV half holds all 8192 entries, more than
    BigMsmDims::large after the rounds (test_crossovers_cpu.test_slice_path_sizes), so the CTA-per-slice path sums
    it.  The slice kernels are launched for every Pippenger MSM; the size check is what puts work on them."""
    n = 8192
    k = rand_scalars(77, 1)[0]
    assert n >> rounds > X.big_large(n, X.big_pick_c(n), rounds)
    try:
        mctx.set_msm_batch_affine(rounds)
        got, names = launched(lambda: msm_one_base(mctx, [k] * n))
        assert got == times_p(n * k)
        expect_kernels(names, ["k_big_slice<%s>" % ("true" if rounds else "false"), "k_big_large_finish"], [])
        # half of them on -P: every large bucket sums to infinity
        assert msm_one_base(mctx, [k] * n, [1, -1] * (n // 2)) is None
    finally:
        mctx.set_msm_batch_affine(-1)


# ------------------------------------------------------------------------------------------------- batched MSMs
def batch_tasks(seed, lengths):
    """tasks alternating between copies of P with random scalars and P / -P pairs with equal scalars:
    [(points, scalars, expected affine)]"""
    rnd = random.Random(seed)
    out = []
    for j, n in enumerate(lengths):
        if j % 2 == 0:
            ks = [rnd.randrange(R) for _ in range(n)]
            out.append((P_ENC * n, ks, times_p(sum(ks))))
        else:
            ks = [rnd.randrange(R) for _ in range(n // 2)]
            out.append(((P_ENC + NP_ENC) * (n // 2), [k for k in ks for _ in (0, 1)], None))
    return out


@pytest.mark.parametrize("shape", ["small", "tp-chunk32", "tp-chunk128"])
def test_msm_batch(mctx, shape):
    sm = mctx.device_info()["sm_count"]
    if shape == "small":
        lengths = [2, 3, 32, 33, 128, 200, 384] * 5
    elif shape == "tp-chunk32":
        lengths = [2, 40, 128, 130, 384] * 20
    else:
        lengths = [384] * 100
    tasks = batch_tasks(len(lengths), lengths)
    lens = [len(ks) for _, ks, _ in tasks]  # a P / -P task of odd length drops one term
    offs = [0]
    for n in lens:
        offs.append(offs[-1] + n)
    path = X.msm_batch_path(lens)
    assert path == ("small" if shape == "small" else "tp")
    if path == "tp":
        assert X.pick_chunk(offs[-1], sm) == (32 if shape == "tp-chunk32" else X.const("kMsmChunk"))
    got, names = launched(lambda: mctx.g1_msm_batch(b"".join(p for p, _, _ in tasks),
                                                    b"".join(fr_enc(k) for _, ks, _ in tasks for k in ks), offs))
    want = b"".join(aff_enc(w) for _, _, w in tasks)
    assert got == want
    expect_kernels(names, ["k_msm_small"] if path == "small" else ["k_msm_warp_gmem"],
                   ["k_msm_warp_gmem"] if path == "small" else ["k_msm_small"])


@pytest.mark.parametrize("ntask", [8, 100])
def test_msm_batch_device_repeated_pool_index(pkg, mctx, ntask):
    """one pool index used by every term of a task; bit 31 negates, so a term and its negated twin cancel"""
    Q = b.g1_mul(b.G1_GEN, 0xBEEF)
    pool = mctx.dev_buffer(3 * 96)
    pool.upload(P_ENC + aff_enc(Q) + bytes(96))  # slot 2: the point at infinity
    rnd = random.Random(ntask)
    idx, sc, offs, want = [], [], [0], []
    for t in range(ntask):
        n = [1, 2, 17, 64, 200][t % 5]
        ks = [rnd.randrange(R) for _ in range(n)]
        kind = t % 4
        if kind == 0:  # P n times
            idx += [0] * n
            sc += ks
            want.append(times_p(sum(ks)))
        elif kind == 1:  # P and its negated twin, equal scalars: infinity
            idx += [0, 0x80000000] * n
            sc += [k for k in ks for _ in (0, 1)]
            want.append(None)
        elif kind == 2:  # P n times, -P n - 1 times with the same scalars, Q once
            idx += [0] * n + [0x80000000] * (n - 1) + [1, 2]
            sc += ks + ks[:n - 1] + [ks[0], ks[-1]]
            want.append(b.g1_add(times_p(ks[-1]), b.g1_mul(Q, ks[0])))
        else:  # -P n times
            idx += [0x80000000] * n
            sc += ks
            want.append(times_p(-sum(ks)))
        offs.append(len(idx))
    aff, enc = mctx.g1_msm_batch_device(pool, idx, b"".join(fr_enc(k) for k in sc), offs)
    assert aff == b"".join(aff_enc(w) for w in want)
    assert enc == mctx.g1_compress(aff)
    pool.close()


# ------------------------------------------------------------------------------------------------- two slots
def test_msm_split_over_two_slots(pkg, mctx):
    n = (1 << 17) + 5
    ks = rand_scalars(17, n)
    pts, sc = P_ENC * n, b"".join(fr_enc(k) for k in ks)
    want = times_p(sum(ks))
    assert jac_dec(mctx.g1_msm(pts, sc)) == want
    two = pkg.Context(devices=[0, 0])
    try:
        assert jac_dec(two.g1_msm(pts, sc)) == want
    finally:
        two.close()
