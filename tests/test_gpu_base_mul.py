"""cdl_g1_batch_scalar_mul_base: many scalars times one base through the C ABI, on both device paths (GLV
scalar multiplication below kBaseTableMinScalars scalars with an uncached base, the base's width-12
fixed-base table otherwise)."""
import ctypes as C
import os
import random
import re

import numpy as np
import pytest

from oracle import bls12381 as b
from util import aff_enc, affs_dec, fr_enc, frs_enc

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INF48 = bytes([0xC0]) + bytes(47)
INVALID, TOO_LARGE = -3, -6
GEN = aff_enc(b.G1_GEN)
KAT = [  # eth2 public keys of sk = 1..5: the compressed k * G
    "97f1d3a73197d7942695638c4fa9ac0fc3688c4f9774b905a14e3a3f171bac586c55e83ff97a1aeffb3af00adb22c6bb",
    "a572cbea904d67468808c8eb50a9450c9721db309128012543902d0ac358a62ae28f75bb8f1c7c42c39a8c5529bf0f4e",
    "89ece308f9d1f0131765212deca99697b112d61f9be9a5f1f3780a51335b3ff981747a0b2ca2179b96d2c0c9024e5224",
    "ac9b60d5afcbd5663a8a44b7c5a02f19e9a77ab0a35bd65809bb5c67ec582c897feb04decc694b13e08587f3ff9b5b60",
    "b0e7791fb972fe014159aa33a98622da3cdc98ff707965e536d8636b5fcc5ac7a91a8c46e59a00dca575af0f18fb13dc",
]


def _crossover():
    src = open(os.path.join(ROOT, "go-curdleproofs_b200", "csrc", "capi_base_mul.cu")).read()
    return int(re.search(r"kBaseTableMinScalars\s*=\s*(\d+)", src).group(1))


X = _crossover()
MAX = 1 << 24


def _fresh_base(seed):
    """a random point of G1 (affine bytes)"""
    return aff_enc(b.g1_mul(b.G1_GEN, random.Random(seed).randrange(1, b.R)))


def _mul(ctx, base, sc, affine=True, compressed=False):
    """(result, launches of the call)"""
    n0 = ctx.launch_count()
    res = ctx.g1_batch_scalar_mul_base(base, sc, affine=affine, compressed=compressed)
    return res, ctx.launch_count() - n0


# kernels per call, affine results only: GLV = check + fill + scalar mul; cold table = check + jac_to_affine +
# table build + multiply; warm table = multiply
GLV, COLD, WARM = 3, 4, 1


def _edge_scalars():
    """raw 32-byte scalar encodings (gnark Montgomery limbs) of the edge cases"""
    R = b.R
    canon = [0, 1, 2, R - 1, R - 2, (R - 1) // 2]
    canon += [1 << j for j in range(255) if (1 << j) < R]
    canon += [sum(0x800 << (12 * w) for w in range(21)), sum(0xFFF << (12 * w) for w in range(21))]
    canon += [sum(0x800 << (12 * w) for w in range(21)) + (3 << 252), sum(0x7FF << (12 * w) for w in range(21))]
    for w in (19, 20, 21):
        for d in (1, 2, 0x7FF, 0x800, 0x801, 0xFFF):
            for e in (-2, -1, 0, 1, 2):
                k = d * (1 << (12 * w)) + e
                if 0 <= k < R:
                    canon.append(k)
                    canon.append(R - k if k else 0)
    for e in range(1, 40):
        canon.append(R - e)
        canon.append((R - 1) // 2 + e)
    raw = [fr_enc(k) for k in canon]
    # non-canonical Montgomery limbs: r and above, all ones
    raw += [(R + i).to_bytes(32, "little") for i in range(4)]
    raw += [(2 * R + 5).to_bytes(32, "little"), bytes([0xFF]) * 32, (1 << 255).to_bytes(32, "little")]
    return raw


def _random_scalars(n, seed):
    """n raw 32-byte values (any limbs: the library reduces them as cdl_g1_scalar_mul_affine does)"""
    return np.random.default_rng(seed).integers(0, 256, size=32 * n, dtype=np.uint8).tobytes()


def _glv_reference(ctx, base, sc):
    """what callers do without this call: cdl_g1_scalar_mul_affine on n copies of the base, stride 1"""
    n = len(sc) // 32
    return ctx.g1_scalar_mul_affine(base * n, sc, broadcast=False)


def test_known_answers_both_paths(pkg):
    """k * G for k = 1..5 gives the eth2 public keys, on the GLV path (fresh context, 5 scalars) and on the
    table path (the table of G built by a large call first), as points and byte for byte as encodings."""
    ctx = pkg.Context(0)
    sc = frs_enc([1, 2, 3, 4, 5])
    (aff, enc), launches = _mul(ctx, GEN, sc, compressed=True)
    assert launches == GLV + 1  # + compress
    assert enc.hex() == "".join(KAT)
    assert ctx.g1_compress(aff) == enc
    _, launches = _mul(ctx, GEN, frs_enc(range(X)))
    assert launches == COLD
    (aff2, enc2), launches = _mul(ctx, GEN, sc, compressed=True)
    assert launches == WARM
    assert aff2 == aff and enc2 == enc
    ctx.close()


@pytest.mark.parametrize("n", [300, None])
def test_oracle_parity(pkg, n):
    """A random base of G1 and random scalars against the oracle's C port, below the crossover (GLV path) and
    at it (cold table path), on a fresh context each."""
    from oracle.cbackend import CBackend

    rnd = random.Random(7 if n else 8)
    n = n or X
    base_pt = b.g1_mul(b.G1_GEN, rnd.randrange(1, b.R))
    ks = [rnd.randrange(b.R) for _ in range(n)]
    ks[:3] = [0, 1, b.R - 1]
    ctx = pkg.Context(0)
    got, launches = _mul(ctx, aff_enc(base_pt), frs_enc(ks))
    assert launches == (GLV if n < X else COLD)
    sample = list(range(0, n, max(1, n // 300)))
    want = CBackend().mul_batch([base_pt] * len(sample), [ks[i] for i in sample])
    got_pts = affs_dec(got)
    assert [got_pts[i] for i in sample] == want
    ctx.close()


@pytest.mark.parametrize("n", [1 << 16, 1 << 20])
def test_equals_scalar_mul_affine(pkg, n):
    """Byte-for-byte equality with cdl_g1_scalar_mul_affine on n copies of the base, for random scalars and
    every edge scalar (zero, r - 1, powers of two, carries through every window, sums meeting table entries
    near r and near multiples of 2^(12 w), non-canonical limbs), on the cold and then the warm table path."""
    ctx = pkg.Context(0)
    base = _fresh_base(n)
    edge = b"".join(_edge_scalars())
    sc = edge + _random_scalars(n - len(edge) // 32, n)
    want = _glv_reference(ctx, base, sc)
    want48 = ctx.g1_compress(want)
    (aff, enc), launches = _mul(ctx, base, sc, compressed=True)
    assert launches == COLD
    assert aff == want
    assert enc == want48
    (aff, enc), launches = _mul(ctx, base, sc, compressed=True)
    assert launches == WARM
    assert aff == want and enc == want48
    # the GLV path on the edge scalars (a fresh base, fewer scalars than the crossover)
    base2 = _fresh_base(n + 1)
    got, launches = _mul(ctx, base2, edge)
    assert launches == GLV
    assert got == _glv_reference(ctx, base2, edge)
    ctx.close()


def test_infinity_and_bad_bases(ctx, pkg):
    """The point at infinity as base gives infinity everywhere; a point off the curve and a point on the curve
    outside G1 are refused on either path."""
    sc = _random_scalars(X + 5, 1)
    aff, enc = ctx.g1_batch_scalar_mul_base(bytes(96), sc, affine=True, compressed=True)
    assert aff == bytes(96 * (X + 5)) and enc == INF48 * (X + 5)
    gx, gy = b.G1_GEN
    off = aff_enc((gx, (gy + 1) % b.P))
    x = 1
    while True:  # on the curve, outside G1
        y = b.fp_sqrt((x ** 3 + 4) % b.P)
        if y is not None and not b.g1_in_subgroup((x, y)):
            break
        x += 1
    outside = aff_enc((x, y))
    noncanon = (b.P + gx).to_bytes(48, "little") + aff_enc(b.G1_GEN)[48:]
    for bad in (off, outside, noncanon):
        for n in (7, X):
            with pytest.raises(pkg.CdlError) as ei:
                ctx.g1_batch_scalar_mul_base(bad, sc[:32 * n])
            assert ei.value.code == INVALID
    # a refused base leaves nothing cached: a good base still works on both paths
    assert ctx.g1_batch_scalar_mul_base(GEN, frs_enc([1]), affine=False, compressed=True).hex() == KAT[0]


def test_cache_lru_and_isolation(pkg):
    """Five distinct bases then G again: equal to a fresh context's results, warm calls launch no build,
    and the least recently used table is the one rebuilt.  Whisk round trips on the same context stay
    byte-identical to those of a context that never made the call."""
    bases = [GEN] + [_fresh_base(100 + i) for i in range(4)]
    sc = _random_scalars(X, 5)
    small = sc[:32 * 9]
    ref = pkg.Context(0)
    want = [ref.g1_batch_scalar_mul_base(bs, sc) for bs in bases]
    want_small = [w[:96 * 9] for w in want]
    ell, B = 12, 32

    pre = b"".join(b.g1_compress(b.g1_mul(b.G1_GEN, i + 2)) * 2 for i in range(ell)) * B  # trackers (rG, 1 rG)

    def round_trip(c):
        crs = c.generate_crs(ell, pkg.Rand(0))
        post, proofs, status = c.whisk_generate_shuffle_proof_batch(crs, pre, [pkg.Rand(3000 + i) for i in range(B)])
        ok, st = c.whisk_is_valid_shuffle_proof_batch(crs, pre, post, proofs, [pkg.Rand(2000 + i) for i in range(B)])
        assert status == [0] * B and st == [0] * B and ok == [1] * B
        return bytes(post), bytes(proofs)

    clean = pkg.Context(0)
    first = round_trip(clean)
    clean.close()
    ctx = pkg.Context(0)
    assert round_trip(ctx) == first
    for i, bs in enumerate(bases):
        got, launches = _mul(ctx, bs, sc)
        assert got == want[i] and launches == COLD
        assert round_trip(ctx) == first
    # bases 1..4 are cached (warm, also below the crossover), G was replaced
    for i in (4, 1, 3, 2):
        got, launches = _mul(ctx, bases[i], small)
        assert got == want_small[i] and launches == WARM
    got, launches = _mul(ctx, GEN, small)
    assert got == want_small[0] and launches == GLV
    got, launches = _mul(ctx, GEN, sc)
    assert got == want[0] and launches == COLD  # replaces base 4, used least recently
    got, launches = _mul(ctx, bases[4], small)
    assert got == want_small[4] and launches == GLV
    got, launches = _mul(ctx, bases[1], small)
    assert got == want_small[1] and launches == WARM
    assert round_trip(ctx) == first
    ctx.close()
    ref.close()


def test_outputs_and_arguments(ctx, pkg):
    """out only, out48 only, both (out48 == cdl_g1_compress(out)); null pointers, n = 0 and the size limit."""
    sc = _random_scalars(333, 9)
    base = _fresh_base(9)
    aff = ctx.g1_batch_scalar_mul_base(base, sc)
    enc = ctx.g1_batch_scalar_mul_base(base, sc, affine=False, compressed=True)
    a2, e2 = ctx.g1_batch_scalar_mul_base(base, sc, affine=True, compressed=True)
    assert a2 == aff and e2 == enc and ctx.g1_compress(aff) == enc
    lib, h = ctx.lib, ctx.h
    out = C.create_string_buffer(96 * 4)
    out48 = C.create_string_buffer(48 * 4)
    f = lib.cdl_g1_batch_scalar_mul_base
    assert f(None, base, sc, 4, out, out48) == INVALID
    assert f(h, None, sc, 4, out, out48) == INVALID
    assert f(h, base, None, 4, out, out48) == INVALID
    assert f(h, base, sc, 4, None, None) == INVALID
    assert f(h, base, sc, 0, out, out48) == 0
    assert f(h, None, None, 0, None, None) == 0
    assert f(h, base, sc, MAX + 1, out, out48) == TOO_LARGE  # refused before any input is read
    assert b"2^24" in lib.cdl_last_error(h)
    assert f(h, base, sc, 4, None, out48) == 0 and out48.raw == enc[:48 * 4]


def test_multi_device_and_accounting(pkg):
    """A two-slot context gives what a one-slot context gives; class 1 of engine_stats grows by one launch per
    chunk and 3 193 modmul per scalar."""
    sc = _random_scalars(X + 17, 3)
    base = _fresh_base(3)
    one = pkg.Context(0)
    two = pkg.Context(devices=[0, 0])
    for c in (one, two):
        c.engine_stats(reset=True)
    small = sc[:32 * 40]
    r1 = [one.g1_batch_scalar_mul_base(base, s, compressed=True) for s in (small, sc, small)]
    r2 = [two.g1_batch_scalar_mul_base(base, s, compressed=True) for s in (small, sc, small)]
    assert r1 == r2
    for c in (one, two):
        st = c.engine_stats()["elem_scalar_mul"]
        assert st["launches"] == 3
        assert st["modmul"] == pytest.approx(3193.0 * (40 + X + 17 + 40))
        assert c.engine_busy_ms() > 0
    assert two.engine_busy_ms_device(1) == 0
    one.close()
    two.close()
