"""cdl_g1_msm above 2 * kMsmSlotTerms terms and cdl_g1_batch_scalar_mul_base from 2 * kBaseSlotScalars scalars
on a multi-device context: the call is dealt to the device slots in contiguous blocks (lane 0 of each slot), and
the bytes must equal those of the one-device context `ctx` for every input - the normalised representative, the
point at infinity, rejected bases and all.  [0, 0] and [0, 0, 0] run two and three slots on one GPU (three slots
give unequal blocks); the real-device tests use [0 .. min(device_count, 4)) and skip below 2 GPUs."""
import ctypes as C
import os
import random
import re

import pytest

from oracle import bls12381 as b
from util import R, aff_enc, affs_enc, affs_dec, fr_enc, frs_enc, jac_dec

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "go-curdleproofs_b200", "csrc")
INVALID, TOO_LARGE = -3, -6
GEN = aff_enc(b.G1_GEN)
ONE_MONT = pow(2, 384, b.P).to_bytes(48, "little")


def _const(fname, name):
    src = open(os.path.join(CSRC, fname)).read()
    return int(re.search(name + r"\s*=\s*(\d+)", src).group(1))


T = _const("capi_msm.cu", "kMsmSlotTerms")  # terms per slot of a split MSM
S = _const("capi_base_mul.cu", "kBaseSlotScalars")  # scalars per slot of a split fixed-base call
X = _const("capi_base_mul.cu", "kBaseTableMinScalars")


def _device_count():
    import torch

    return torch.cuda.device_count()


def shard_lo(n, D, s):
    """first unit of block s of n units dealt to D slots (sharding.shard_bounds)"""
    return s * (n // D) + min(s, n % D)


def slots(n, D, per):
    return max(1, min(D, n // per))


def blocks(n, D, per):
    d = slots(n, D, per)
    return [(shard_lo(n, d, s), shard_lo(n, d, s + 1)) for s in range(d)]


@pytest.fixture(scope="module")
def m2(pkg):
    c = pkg.Context(devices=[0, 0])
    yield c
    c.close()


@pytest.fixture(scope="module")
def m3(pkg):
    c = pkg.Context(devices=[0, 0, 0])
    yield c
    c.close()


@pytest.fixture(scope="module")
def vec(ctx):
    """a_i, s_i and P_i = a_i * G for 3 * kMsmSlotTerms + 5 terms"""
    n = 3 * T + 5
    rnd = random.Random(41)
    a = [rnd.randrange(1, R) for _ in range(n)]
    s = [rnd.randrange(R) for _ in range(n)]
    pts = ctx.g1_scalar_mul_affine(GEN * n, frs_enc(a), broadcast=False)
    return a, s, pts


def expected(a, s):
    return b.g1_mul(b.G1_GEN, sum(x * y for x, y in zip(a, s)) % R)


def _same_msm(ctx, ms, pts, sc):
    """the one-device bytes, after checking that every multi-device context gives them"""
    want = ctx.g1_msm(pts, sc)
    for m in ms:
        assert m.g1_msm(pts, sc) == want
    return want


# ------------------------------------------------------------------------------------------------- MSM
def test_msm_sizes(ctx, m2, m3, vec):
    """one slot (2T - 1), two equal blocks (2T), three unequal blocks (3T + 5) and an odd size: all 144 bytes
    equal the one-device result, which is (sum a_i s_i) * G with Z = 1"""
    a, s, pts = vec
    for n in (2 * T - 1, 2 * T, 2 * T + 777, 3 * T + 5):
        got = _same_msm(ctx, (m2, m3), pts[:96 * n], frs_enc(s[:n]))
        assert jac_dec(got) == expected(a[:n], s[:n]) and got[96:] == ONE_MONT, n


def test_msm_adversarial(ctx, m2, m3, vec):
    a, s, pts = vec
    rnd = random.Random(5)
    n = 3 * T
    P, A, Sc = pts[:96 * n], a[:n], s[:n]
    # the last slot's whole block of zero scalars (its partial sum is infinity)
    for m, D in ((m2, 2), (m3, 3)):
        lo = blocks(n, D, T)[-1][0]
        z = Sc[:lo] + [0] * (n - lo)
        want = ctx.g1_msm(P, frs_enc(z))
        assert m.g1_msm(P, frs_enc(z)) == want and jac_dec(want) == expected(A, z)
    # all scalars zero: infinity, gnark's (1, 1, 0)
    got = _same_msm(ctx, (m2, m3), P, bytes(32 * n))
    assert jac_dec(got) is None and got[96:] == bytes(48)
    # P in block 0, -P in block 1 with equal scalars: the partials cancel across blocks
    h = T
    neg = affs_enc([b.g1_neg(p) for p in affs_dec(pts[:96 * h])])
    got = _same_msm(ctx, (m2, m3), pts[:96 * h] + neg, frs_enc(s[:h] * 2))
    assert jac_dec(got) is None and got[96:] == bytes(48)
    # ... and on three blocks: P, -P, Q
    got = _same_msm(ctx, (m3,), pts[:96 * h] + neg + pts[96 * h:96 * 2 * h], frs_enc(s[:h] * 2 + s[h:2 * h]))
    assert jac_dec(got) == expected(a[h:2 * h], s[h:2 * h])
    # 1 % infinity bases
    n = 3 * T + 5
    Pb, A2 = bytearray(pts), list(a)
    for i in rnd.sample(range(n), n // 100):
        Pb[96 * i:96 * i + 96] = bytes(96)
        A2[i] = 0
    got = _same_msm(ctx, (m2, m3), bytes(Pb), frs_enc(s))
    assert jac_dec(got) == expected(A2, s)
    # all-equal scalars
    k = rnd.randrange(R)
    got = _same_msm(ctx, (m2, m3), pts, fr_enc(k) * n)
    assert jac_dec(got) == expected(a, [k] * n)


def test_msm_settings_reach_the_slots(ctx, m2, m3, vec):
    """window width and batch-affine rounds set after the lanes exist: the bytes never depend on them (that the
    settings do reach the lanes is checked by test_msm_settings_size_the_lane_scratch)"""
    a, s, pts = vec
    n = 3 * T + 5
    sc = frs_enc(s)
    want = ctx.g1_msm(pts, sc)
    for m in (m2, m3):
        assert m.g1_msm(pts, sc) == want  # the lanes exist from here on
        try:
            for c, r in ((9, 0), (12, 2), (16, -1), (0, 3), (5, 1)):
                m.set_msm_window(c)
                m.set_msm_batch_affine(r)
                assert m.g1_msm(pts, sc) == want, (c, r)
        finally:
            m.set_msm_window(0)
            m.set_msm_batch_affine(-1)
    assert jac_dec(want) == expected(a, s)


def test_msm_settings_size_the_lane_scratch(pkg, ctx, vec):
    """Observable evidence that the settings reach the lanes: a wider window (more buckets) and batch-affine
    rounds (padded pair buffers) make every lane's MSM scratch grow, which shows in the GPU's free memory.
    Set on the root after a first split call, they must grow both lanes' scratch of a [0, 0] context."""
    import torch

    a, s, pts = vec
    sc = frs_enc(s)
    want = ctx.g1_msm(pts, sc)
    m = pkg.Context(devices=[0, 0])
    try:
        torch.cuda.mem_get_info(0)  # torch's own context first
        assert m.g1_msm(pts, sc) == want  # blocks of ~98 k terms: c = 16, no rounds; the lanes exist from here on
        free = [torch.cuda.mem_get_info(0)[0]]
        # c = 18: 2^20 buckets per lane instead of 2^18 (192 B each, plus the reduction buffers), ~ +300 MB per lane
        m.set_msm_window(18)
        assert m.g1_msm(pts, sc) == want
        free.append(torch.cuda.mem_get_info(0)[0])
        # c = 16 with 6 rounds: every bucket padded to 64 slots, ~ 1 GB of pair buffers per lane
        m.set_msm_window(0)
        m.set_msm_batch_affine(6)
        assert m.g1_msm(pts, sc) == want
        free.append(torch.cuda.mem_get_info(0)[0])
        assert free[0] - free[1] >= 2 * (256 << 20), free
        assert free[1] - free[2] >= 2 * (512 << 20), free
    finally:
        m.close()


def test_sum_affine(ctx, m2, m3, vec):
    a, s, pts = vec
    want = ctx.g1_sum_affine(pts)
    assert m2.g1_sum_affine(pts) == want and m3.g1_sum_affine(pts) == want
    assert affs_dec(want)[0] == b.g1_mul(b.G1_GEN, sum(a) % R)


def test_msm_whole_call_limit(m2, m3):
    """2^30 terms are refused before any input is read (the buffers hold one term)"""
    out = C.create_string_buffer(144)
    for m in (m2, m3):
        assert m.lib.cdl_g1_msm(m.h, bytes(96), bytes(32), 1 << 30, out) == TOO_LARGE
        assert b"2^30" in m.lib.cdl_last_error(m.h)
        assert out.raw == bytes(144)


# ------------------------------------------------------------------------------------ fixed-base multiplication
def _fresh_base(seed):
    return aff_enc(b.g1_mul(b.G1_GEN, random.Random(seed).randrange(1, R)))


def _scalars(n, seed):
    """n raw 32-byte values (any limbs: the library reduces them)"""
    return random.Random(seed).randbytes(32 * n)


def _mul(c, base, sc, **kw):
    n0 = c.launch_count()
    r = c.g1_batch_scalar_mul_base(base, sc, **kw)
    return r, c.launch_count() - n0


def test_base_mul_sizes(ctx, m2, m3):
    base = _fresh_base(1)
    for n in (2 * S - 1, 2 * S + 3, 3 * S + 7):
        sc = _scalars(n, n)
        want = ctx.g1_batch_scalar_mul_base(base, sc, affine=True, compressed=True)
        for m in (m2, m3):
            assert m.g1_batch_scalar_mul_base(base, sc, affine=True, compressed=True) == want, n
            assert m.g1_batch_scalar_mul_base(base, sc, affine=False, compressed=True) == want[1], n
            assert m.g1_batch_scalar_mul_base(base, sc) == want[0], n


def test_base_mul_mixed_cache_states(pkg, ctx):
    """A one-slot call warms the root engine only; a two-slot call builds the tables of slots 0 and 1; a
    three-slot call finds them and builds slot 2's.  Bytes equal the one-device results throughout."""
    base = _fresh_base(2)
    m = pkg.Context(devices=[0, 0, 0])
    try:
        cold, warm = 4, 1  # kernels of a call of one chunk, affine results: check + jac_to_affine + build + multiply
        for n, launches in ((X + 5, cold), (2 * S + 3, 2 * cold), (3 * S + 7, 2 * warm + cold), (3 * S + 7, 3 * warm)):
            sc = _scalars(n, 7 * n)
            got, k = _mul(m, base, sc)
            assert got == ctx.g1_batch_scalar_mul_base(base, sc), n
            assert k == launches, n
    finally:
        m.close()


def _bad_bases():
    gx, gy = b.G1_GEN
    off = aff_enc((gx, (gy + 1) % b.P))
    x = 1
    while True:  # on the curve, outside G1
        y = b.fp_sqrt((x ** 3 + 4) % b.P)
        if y is not None and not b.g1_in_subgroup((x, y)):
            break
        x += 1
    noncanon = (b.P + gx).to_bytes(48, "little") + GEN[48:]
    return {"not on the curve": off, "not in G1": aff_enc((x, y)), "canonical": noncanon}


def test_base_mul_rejected_bases(ctx, m2, m3):
    """every piece refuses the base alike: CDL_ERR_INVALID_ARG with the one-device message, outputs untouched"""
    for why, bad in _bad_bases().items():
        for m in (m2, m3):
            for n in (2 * S + 3, 3 * S + 7):
                sc = _scalars(n, 3)
                out = C.create_string_buffer(b"\xa5" * (96 * n), 96 * n)
                out48 = C.create_string_buffer(b"\x5a" * (48 * n), 48 * n)
                rc = m.lib.cdl_g1_batch_scalar_mul_base(m.h, bad, sc, n, out, out48)
                assert rc == INVALID, (why, n)
                msg = m.lib.cdl_last_error(m.h).decode()
                assert "base rejected" in msg and why in msg, msg
                assert out.raw == b"\xa5" * (96 * n) and out48.raw == b"\x5a" * (48 * n)
    sc = _scalars(2 * S + 3, 4)
    want = ctx.g1_batch_scalar_mul_base(GEN, sc)
    assert m2.g1_batch_scalar_mul_base(GEN, sc) == want and m3.g1_batch_scalar_mul_base(GEN, sc) == want


def test_base_mul_accounting(pkg, ctx):
    base = _fresh_base(3)
    m = pkg.Context(devices=[0, 0, 0])
    try:
        m.engine_stats(reset=True)
        sc = _scalars(2 * S - 1, 8)
        assert m.g1_batch_scalar_mul_base(base, sc) == ctx.g1_batch_scalar_mul_base(base, sc)
        assert m.engine_busy_ms_device(0) > 0 and m.engine_busy_ms_device(1) == 0
        n = 3 * S + 7
        sc = _scalars(n, 9)
        m.g1_batch_scalar_mul_base(base, sc)  # warms the three slots' tables
        ctx.g1_batch_scalar_mul_base(base, sc)  # and ctx's
        m.engine_stats(reset=True)
        got, k = _mul(m, base, sc)
        assert all(m.engine_busy_ms_device(s) > 0 for s in range(3))
        n0 = ctx.launch_count()
        parts = [ctx.g1_batch_scalar_mul_base(base, sc[32 * lo:32 * hi]) for lo, hi in blocks(n, 3, S)]
        assert got == b"".join(parts)
        assert k == ctx.launch_count() - n0 == 3
        st = m.engine_stats()["elem_scalar_mul"]
        assert st["launches"] == 3 and st["modmul"] == pytest.approx(3193.0 * n)
    finally:
        m.close()


# ------------------------------------------------------------------------------------------- real devices
def test_real_devices(pkg, ctx, vec):
    """MSM and fixed-base multiplication at 2^20 over the box's GPUs (at most 4); every GPU's free memory drops
    by at least its block of MSM inputs (the lane buffers persist until the context is destroyed)."""
    import torch

    D = min(_device_count(), 4)
    if D < 2:
        pytest.skip("needs >= 2 GPUs")
    a, s, pts = vec
    n = 1 << 20
    reps = -(-n // T)
    P = (pts[:96 * T] * reps)[:96 * n]
    sc = frs_enc((s[i % T] * (1 + i // T)) % R for i in range(n))
    want = ctx.g1_msm(P, sc)
    m = pkg.Context(devices=list(range(D)))
    try:
        for d in range(D):
            torch.cuda.mem_get_info(d)  # torch's own context on every GPU first
        free0 = [torch.cuda.mem_get_info(d)[0] for d in range(D)]
        assert m.g1_msm(P, sc) == want
        free1 = [torch.cuda.mem_get_info(d)[0] for d in range(D)]
        for d, (lo, hi) in enumerate(blocks(n, D, T)):
            assert free0[d] - free1[d] >= 128 * (hi - lo), (d, free0[d], free1[d])
        base = _fresh_base(4)
        bsc = _scalars(n, 10)
        m.engine_stats(reset=True)
        assert m.g1_batch_scalar_mul_base(base, bsc, affine=True, compressed=True) == \
            ctx.g1_batch_scalar_mul_base(base, bsc, affine=True, compressed=True)
        assert all(m.engine_busy_ms_device(d) > 0 for d in range(D))
    finally:
        m.close()
