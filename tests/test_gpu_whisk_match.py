"""cdl_whisk_match_trackers: which of V secrets own which of T Whisk trackers, through the C ABI, on both
device paths (shared-scalar scalar multiplications below kMatchTableMinKeys keys, per-tracker fixed-base
tables from there on)."""
import os
import random
import re

import pytest

from oracle import bls12381 as b
from util import aff_enc, fr_dec, fr_enc

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INF48 = bytes([0xC0]) + bytes(47)
DECODE, PROTOCOL, INVALID, TOO_LARGE = -4, -5, -3, -6


def _crossover():
    src = open(os.path.join(ROOT, "go-curdleproofs_b200", "csrc", "capi_whisk_match.cu")).read()
    return int(re.search(r"kMatchTableMinKeys\s*=\s*(\d+)", src).group(1))


X = _crossover()


def _gpu_trackers(ctx, rs, ks):
    """trackers (r_t G, k_t r_t G) built on the device, rs / ks: fr encodings"""
    n = len(rs) // 32
    rG = ctx.g1_scalar_mul_affine(aff_enc(b.G1_GEN) * n, rs, broadcast=False)
    krG = ctx.g1_scalar_mul_affine(rG, ks, broadcast=False)
    e1, e2 = ctx.g1_compress(rG), ctx.g1_compress(krG)
    return b"".join(e1[48 * j:48 * j + 48] + e2[48 * j:48 * j + 48] for j in range(n))


def _match(ctx, trackers, keys):
    """(owner, status, launches of the call) with keys a list of ints"""
    n0 = ctx.launch_count()
    owner, status = ctx.whisk_match_trackers(trackers, b"".join(fr_enc(k) for k in keys))
    return owner, status, ctx.launch_count() - n0


def _path_ok(V, launches):
    # decompress + prep + one shared-scalar kernel, or + a table build and a table kernel per tile of trackers
    return launches == 3 if V < X else launches > 3 and launches % 2 == 0


def test_owner_matches_oracle(ctx):
    """48 trackers in random order, some owned by the 12 listed keys, some by unlisted ones: owner equals a
    brute-force k * rG == krG over the oracle's C backend, and the call is accounted as class-1 work."""
    from oracle.cbackend import CBackend

    cb = CBackend()
    rnd = random.Random(7)
    ks = [rnd.randrange(1, b.R) for _ in range(12)]
    unlisted = [rnd.randrange(1, b.R) for _ in range(6)]
    owners = [rnd.choice(ks) for _ in range(30)] + [rnd.choice(unlisted) for _ in range(18)]
    rnd.shuffle(owners)
    rG = cb.mul_batch([b.G1_GEN] * 48, [rnd.randrange(1, b.R) for _ in range(48)])
    krG = cb.mul_batch(rG, owners)
    trackers = b"".join(b.g1_compress(p) + b.g1_compress(q) for p, q in zip(rG, krG))
    prod = cb.mul_batch([p for p in rG for _ in ks], ks * 48)
    want = []
    for t in range(48):
        hits = [v for v in range(12) if prod[12 * t + v] == krG[t]]
        want.append(hits[0] if hits else -1)
    assert sum(w >= 0 for w in want) == 30
    ctx.engine_stats(reset=True)
    owner, status, launches = _match(ctx, trackers, ks)
    assert status == [0] * 48
    assert owner == want
    assert _path_ok(12, launches)
    st = ctx.engine_stats()["elem_scalar_mul"]
    assert st["launches"] == 1 and st["modmul"] == 3193.0 * 48 * 12 and st["ms"] > 0  # one timed kernel chain


@pytest.fixture(scope="module")
def big_set(ctx, pkg):
    """8192 trackers; tracker t is owned by key j_t of a 6000-key list (so by no key of the first V when
    j_t >= V)."""
    T, NK = 8192, 6000
    kb = pkg.Rand(77).get_frs(NK)
    keys = [fr_dec(kb[32 * i:32 * i + 32]) for i in range(NK)]
    assert len(set(keys)) == NK
    j = [(t * 7919 + 13) % NK for t in range(T)]
    rs = pkg.Rand(78).get_frs(T)
    trackers = _gpu_trackers(ctx, rs, b"".join(fr_enc(keys[j[t]]) for t in range(T)))
    return trackers, keys, j


@pytest.mark.parametrize("V", [1, 2, X - 1, X, 4096])
def test_both_paths_at_real_sizes(ctx, big_set, V):
    """Exact owners for 8192 trackers on either side of the crossover; the same key list extended with
    decoy keys (to at least the crossover, so the table path then runs) gives identical owners."""
    trackers, keys, j = big_set
    T = len(j)
    want = [j[t] if j[t] < V else -1 for t in range(T)]
    owner, status, launches = _match(ctx, trackers, keys[:V])
    assert status == [0] * T
    assert owner == want
    assert _path_ok(V, launches)
    rnd = random.Random(V)
    decoys = [rnd.randrange(1, b.R) for _ in range(max(37, X - V))]
    owner2, status2, launches2 = _match(ctx, trackers, keys[:V] + decoys)
    assert status2 == [0] * T and owner2 == want
    assert _path_ok(V + len(decoys), launches2)


def test_edge_cases(ctx, pkg):
    """Duplicate keys, k = 0, rG at infinity, malformed encodings, counts off every tile size: identical
    results on both paths."""
    rnd = random.Random(11)
    T = 300  # not a multiple of 32 or of the table tile
    a, c, d = (rnd.randrange(1, b.R) for _ in range(3))
    keys = [a, c, a, 0, d, c]  # V = 6; a at 0 and 2, c at 1 and 5
    own = [rnd.choice([a, c, d, rnd.randrange(1, b.R)]) for _ in range(T)]
    rs = b"".join(fr_enc(rnd.randrange(1, b.R)) for _ in range(T))
    tr = bytearray(_gpu_trackers(ctx, rs, b"".join(fr_enc(k) for k in own)))
    first = {a: 0, c: 1, d: 4}
    want = [first.get(k, -1) for k in own]
    wst = [0] * T

    def put(t, rg, krg, owner, status):
        tr[96 * t:96 * t + 48] = rg
        tr[96 * t + 48:96 * t + 96] = krg
        want[t], wst[t] = owner, status

    g = b.g1_compress(b.G1_GEN)
    put(5, g, INF48, 3, 0)                      # k = 0: krG at infinity, rG finite
    put(6, INF48, INF48, -1, PROTOCOL)          # rG at infinity identifies nobody, though k * rG == krG
    put(7, INF48, g, -1, PROTOCOL)
    bad_flags = bytes([g[0] | 0x60]) + g[1:]
    x_ge_p = bytes([0x9F]) + b"\xff" * 47
    x = 1
    while True:
        y = b.fp_sqrt((x**3 + 4) % b.P)
        if y is not None and not b.g1_in_subgroup((x, y)):
            break
        x += 1
    not_sub = b.g1_compress((x, y))
    put(8, bad_flags, g, -1, DECODE)
    put(9, g, x_ge_p, -1, DECODE)
    put(10, not_sub, g, -1, DECODE)
    put(11, g, not_sub, -1, DECODE)
    assert want[4] >= -1 and want[12] >= -1  # neighbours keep their owners
    owner, status, launches = _match(ctx, bytes(tr), keys)
    assert status == wst
    assert owner == want
    assert _path_ok(len(keys), launches)
    decoys = [rnd.randrange(1, b.R) for _ in range(X + 5)]
    owner2, status2, launches2 = _match(ctx, bytes(tr), keys + decoys)
    assert status2 == wst and owner2 == want
    assert _path_ok(len(keys) + len(decoys), launches2)
    # T = 1, V = 1
    assert _match(ctx, bytes(tr[:96]), [own[0]])[:2] == ([0], [0])


def test_invalid_arguments(ctx, pkg):
    import ctypes as C

    lib, h = ctx.lib, ctx.h
    tr = b.g1_compress(b.G1_GEN) * 2
    k = fr_enc(1)
    o, s = (C.c_int32 * 1)(), (C.c_int32 * 1)()
    assert lib.cdl_whisk_match_trackers(h, 0, tr, 1, k, o, s) == INVALID
    assert lib.cdl_whisk_match_trackers(h, 1, tr, 0, k, o, s) == INVALID
    assert lib.cdl_whisk_match_trackers(None, 1, tr, 1, k, o, s) == INVALID
    assert lib.cdl_whisk_match_trackers(h, 1, None, 1, k, o, s) == INVALID
    assert lib.cdl_whisk_match_trackers(h, 1, tr, 1, None, o, s) == INVALID
    assert lib.cdl_whisk_match_trackers(h, 1, tr, 1, k, None, s) == INVALID
    assert lib.cdl_whisk_match_trackers(h, 1, tr, 1, k, o, None) == INVALID
    # sizes are checked before any input is read
    assert lib.cdl_whisk_match_trackers(h, (1 << 24) + 1, tr, 1, k, o, s) == TOO_LARGE
    assert lib.cdl_whisk_match_trackers(h, 1, tr, (1 << 24) + 1, k, o, s) == TOO_LARGE
    with pytest.raises(pkg.CdlError) as ei:
        ctx.whisk_match_trackers(b"", k)
    assert ei.value.code == INVALID
    # the context is still usable
    assert ctx.whisk_match_trackers(tr, k) == ([0], [0])


def test_match_through_a_shuffle(ctx, pkg):
    """124 pre-trackers of 3 keys (and some of nobody's), shuffled by a Whisk shuffle proof: the
    post-trackers give every key as many trackers as it had before."""
    ell = 124
    rnd = random.Random(5)
    keys = [rnd.randrange(1, b.R) for _ in range(3)]
    own = [keys[i % 3] if i % 10 else rnd.randrange(1, b.R) for i in range(ell)]
    rs = b"".join(fr_enc(rnd.randrange(1, b.R)) for _ in range(ell))
    pre = _gpu_trackers(ctx, rs, b"".join(fr_enc(k) for k in own))
    want = [keys.index(k) if k in keys else -1 for k in own]
    owner, status, _ = _match(ctx, pre, keys)
    assert status == [0] * ell and owner == want
    crs = ctx.generate_crs(ell, pkg.Rand(0))
    post, proofs, st = ctx.whisk_generate_shuffle_proof_batch(crs, pre, [pkg.Rand(42)])
    assert st == [0]
    post = bytes(post)
    assert post != pre
    owner2, status2, _ = _match(ctx, post, keys)
    assert status2 == [0] * ell
    assert sorted(owner2) == sorted(want)


def test_match_shares_the_engine_pool_with_protocol_calls(ctx, pkg, big_set):
    """The match call overwrites the start of the engine's point pool.  Whisk round trips before and after
    it, with the same seeds, must be byte-identical."""
    ell, B = 12, 32
    crs = ctx.generate_crs(ell, pkg.Rand(0))
    r = pkg.Rand(1000)
    rs, ks = r.get_frs(ell), r.get_frs(ell)
    pre = _gpu_trackers(ctx, rs, ks) * B

    def round_trip():
        post, proofs, status = ctx.whisk_generate_shuffle_proof_batch(crs, pre, [pkg.Rand(3000 + i) for i in range(B)])
        ok, st = ctx.whisk_is_valid_shuffle_proof_batch(crs, pre, post, proofs, [pkg.Rand(2000 + i) for i in range(B)])
        assert status == [0] * B and st == [0] * B and ok == [1] * B
        return bytes(post), bytes(proofs)

    first = round_trip()
    trackers, keys, j = big_set
    owner, status, _ = _match(ctx, trackers, keys[:X])
    assert owner == [v if v < X else -1 for v in j]
    assert round_trip() == first
