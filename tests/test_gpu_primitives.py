"""GPU parity tests, through the C ABI, against the CPU oracle: bit-exact."""
import random

import pytest

from oracle import bls12381 as b
from oracle.rand import Rand
from util import (P, R, RP, aff_dec, aff_enc, affs_dec, affs_enc, fp_dec, fp_enc, fr_enc, frs_enc, jac_dec, jac_enc)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pts():
    return Rand(101).get_g1_affines(64)


def test_device_is_b200(ctx):
    info = ctx.device_info()
    assert info["sm_count"] > 0


def test_fp_mul(ctx):
    random.seed(1)
    edge = [0, 1, P - 1, P - 2, RP, RP * RP % P, 2**380, P - 3, (P - 1) // 2]
    vals = edge + [random.randrange(P) for _ in range(500)]
    A = [random.choice(vals) for _ in range(5000)]
    B = [random.choice(vals) for _ in range(5000)]
    out = ctx.fp_mul(b"".join(fp_enc(a) for a in A), b"".join(fp_enc(x) for x in B))
    got = [fp_dec(out[i:i + 48]) for i in range(0, len(out), 48)]
    assert got == [a * x % P for a, x in zip(A, B)]


def test_scalar_mul_per_element_and_broadcast(ctx, pts):
    random.seed(2)
    ks = [0, 1, 2, R - 1, R - 2, 16, 15] + [random.randrange(R) for _ in range(40)]
    ps = [pts[i % len(pts)] for i in range(len(ks))]
    ps[5] = None
    out = affs_dec(ctx.g1_scalar_mul_affine(affs_enc(ps), frs_enc(ks), broadcast=False))
    assert out == [b.g1_mul(p, k) for p, k in zip(ps, ks)]
    k = random.randrange(R)
    out = affs_dec(ctx.g1_scalar_mul_affine(affs_enc(pts[:33]), fr_enc(k), broadcast=True))
    assert out == b.g1_mul_batch(pts[:33], [k] * 33)


def test_fold(ctx, pts):
    random.seed(3)
    x = random.randrange(R)
    L = pts[:16] + [None, pts[3]]
    Rr = pts[16:32] + [pts[1], None]
    # exceptional: L = -x*R (sum is infinity), L = x*R (doubling)
    xr = b.g1_mul(pts[40], x)
    L += [b.g1_neg(xr), xr]
    Rr += [pts[40], pts[40]]
    got = affs_dec(ctx.g1_fold(affs_enc(L), affs_enc(Rr), fr_enc(x)))
    want = [b.g1_add(l, b.g1_mul(r, x)) for l, r in zip(L, Rr)]
    assert got == want
    assert want[-2] is None


@pytest.mark.parametrize("n", [1, 2, 7, 8, 9, 64, 128, 300, 628])
def test_msm_sizes(ctx, n):
    r = Rand(1000 + n)
    base = r.get_g1_affines(min(n, 48))
    ps = [base[i % len(base)] for i in range(n)]
    ks = r.get_frs(n)
    got = jac_dec(ctx.g1_msm(affs_enc(ps), frs_enc(ks)))
    assert got == b.g1_msm(ps, ks)


def test_msm_degenerate_inputs(ctx, pts):
    random.seed(5)
    n = 60
    ps = list(pts[:n])
    beta = random.randrange(R)
    # all-equal scalars (samepermutationargument.go:62-67)
    assert jac_dec(ctx.g1_msm(affs_enc(ps), frs_enc([beta] * n))) == b.g1_mul(b.g1_sum(ps), beta)
    # tiny scalars 0..n-1 permuted (common/util.go:68-75)
    sc = list(range(n))
    random.shuffle(sc)
    assert jac_dec(ctx.g1_msm(affs_enc(ps), frs_enc(sc))) == b.g1_msm(ps, sc)
    # zero scalars, infinity bases with non-zero scalars, repeated bases, P and -P
    ps2 = ps[:20] + [None, None, ps[0], ps[0], b.g1_neg(ps[1])]
    sc2 = [random.randrange(R) for _ in range(20)] + [random.randrange(R), 7, 3, R - 3, 0]
    sc2[1] = 0
    sc2[2] = 0
    assert jac_dec(ctx.g1_msm(affs_enc(ps2), frs_enc(sc2))) == b.g1_msm_naive(ps2, sc2)
    # P and -P with the same scalar cancel to infinity
    k = random.randrange(R)
    out = ctx.g1_msm(affs_enc([ps[4], b.g1_neg(ps[4])]), frs_enc([k, k]))
    assert jac_dec(out) is None
    assert out[96:144] == bytes(48)  # gnark infinity: Z == 0
    # empty MSM is infinity
    assert jac_dec(ctx.g1_msm(b"", b"")) is None


def test_msm_batch(ctx, pts):
    r = Rand(77)
    sizes = [4, 1, 64, 32, 16, 8, 2, 0, 5]
    offs = [0]
    for s in sizes:
        offs.append(offs[-1] + s)
    ps = [pts[i % len(pts)] for i in range(offs[-1])]
    ks = r.get_frs(offs[-1])
    got = affs_dec(ctx.g1_msm_batch(affs_enc(ps), frs_enc(ks), offs))
    want = [b.g1_msm_naive(ps[offs[i]:offs[i + 1]], ks[offs[i]:offs[i + 1]]) for i in range(len(sizes))]
    assert got == want


def test_msm_length_mismatch_is_error(ctx, pkg, pts):
    with pytest.raises(pkg.CdlError) as ei:
        ctx.g1_msm(affs_enc(pts[:3]), frs_enc([1, 2]))
    assert ei.value.code == -3


def test_batch_to_affine_and_sum(ctx, pts):
    random.seed(6)
    zs = [random.randrange(1, P) for _ in range(10)]
    jac = b"".join(jac_enc(p, z) for p, z in zip(pts[:10], zs)) + jac_enc(None)
    assert affs_dec(ctx.g1_batch_to_affine(jac)) == pts[:10] + [None]
    assert aff_dec(ctx.g1_sum_affine(affs_enc(pts[:31]))) == b.g1_sum(pts[:31])


def test_compress_decompress(ctx, pkg, pts):
    ps = pts[:20] + [None, b.g1_neg(pts[0])]
    enc = ctx.g1_compress(affs_enc(ps))
    assert enc == b"".join(b.g1_compress(p) for p in ps)
    dec, st = ctx.g1_decompress(enc)
    assert affs_dec(dec) == ps and not any(st)
    # rejects: bad flags, x >= p, non-residue, not in subgroup, dirty infinity, uncompressed flag
    good = b.g1_compress(pts[0])
    bad_flags = bytes([good[0] | 0x60]) + good[1:]
    x_ge_p = bytes([0x9F]) + b"\xff" * 47
    x = 1
    while b.fp_sqrt((x**3 + 4) % P) is not None:
        x += 1
    non_res = bytearray(x.to_bytes(48, "big"))
    non_res[0] |= 0x80
    x = 1
    while True:
        y = b.fp_sqrt((x**3 + 4) % P)
        if y is not None and not b.g1_in_subgroup((x, y)):
            break
        x += 1
    not_sub = b.g1_compress((x, y))
    dirty_inf = bytes([0xC0]) + bytes(46) + b"\x01"
    uncompressed = bytes([good[0] & 0x1F]) + good[1:]
    enc = b"".join([good, bad_flags, x_ge_p, bytes(non_res), not_sub, dirty_inf, uncompressed])
    dec, st = ctx.g1_decompress(enc, check=False)
    assert st == [0, 1, 2, 3, 4, 5, 1]
    for e, s in zip([enc[i:i + 48] for i in range(0, len(enc), 48)], st):
        try:
            b.g1_decompress(e)
            ok = True
        except b.DecodeError:
            ok = False
        assert ok == (s == 0)
    with pytest.raises(pkg.CdlError) as ei:
        ctx.g1_decompress(enc)
    assert ei.value.code == -4


def test_int_peak_runs(ctx):
    for kind in (0, 1, 2):
        ops, ms = ctx.int_peak(kind, 200)
        assert ops > 0 and ms > 0


def test_msm_batch_throughput_path(ctx, pts):
    """>= 96 MSMs in one call take the two-kernel path (bucket kernel + per-MSM
    Horner combine); results must match the oracle exactly, incl. empty /
    degenerate tasks."""
    import random
    random.seed(11)
    r = Rand(78)
    sizes = [random.choice([0, 1, 2, 3, 7, 16, 33, 64]) for _ in range(130)]
    offs = [0]
    for s in sizes:
        offs.append(offs[-1] + s)
    ps = [pts[random.randrange(len(pts))] for _ in range(offs[-1])]
    ks = r.get_frs(offs[-1])
    # degenerate content: infinity bases, zero scalars, P and -P
    for i in range(0, len(ps), 17):
        ps[i] = None
    for i in range(5, len(ks), 23):
        ks[i] = 0
    got = affs_dec(ctx.g1_msm_batch(affs_enc(ps), frs_enc(ks), offs))
    from oracle.cbackend import CBackend
    cb = CBackend(accelerate_keccak=False)
    want = [cb.msm(ps[offs[i]:offs[i + 1]], ks[offs[i]:offs[i + 1]]) for i in range(len(sizes))]
    assert got == want


def test_public_known_answers(ctx):
    """Independent of the oracle: eth2 public keys for sk = 1..5 are the compressed k*G."""
    kat = [
        "97f1d3a73197d7942695638c4fa9ac0fc3688c4f9774b905a14e3a3f171bac586c55e83ff97a1aeffb3af00adb22c6bb",
        "a572cbea904d67468808c8eb50a9450c9721db309128012543902d0ac358a62ae28f75bb8f1c7c42c39a8c5529bf0f4e",
        "89ece308f9d1f0131765212deca99697b112d61f9be9a5f1f3780a51335b3ff981747a0b2ca2179b96d2c0c9024e5224",
        "ac9b60d5afcbd5663a8a44b7c5a02f19e9a77ab0a35bd65809bb5c67ec582c897feb04decc694b13e08587f3ff9b5b60",
        "b0e7791fb972fe014159aa33a98622da3cdc98ff707965e536d8636b5fcc5ac7a91a8c46e59a00dca575af0f18fb13dc",
    ]
    gen = aff_enc(b.G1_GEN)
    pts = ctx.g1_scalar_mul_affine(gen * 5, frs_enc([1, 2, 3, 4, 5]), broadcast=False)
    assert ctx.g1_compress(pts).hex() == "".join(kat)
    dec, st = ctx.g1_decompress(bytes.fromhex("".join(kat)))
    assert dec == pts and not any(st)
    # 1*G + 2*G + ... as one MSM: 15*G = 5*G + 10*G
    s15 = ctx.g1_msm(pts, frs_enc([1, 1, 1, 1, 1]))
    assert jac_dec(s15) == jac_dec(ctx.g1_msm(gen, fr_enc(15)))


def test_msm_batch_multi_chunk_tasks(ctx, pts):
    """Throughput path with tasks longer than one bucket-warp chunk (128 terms): the chunk partials
    are summed per (task, window) before the Horner combine; also a single long MSM (> 384 terms,
    chunked chain with 32-term chunks) next to short ones."""
    import random
    random.seed(12)
    r = Rand(79)
    from oracle.cbackend import CBackend
    cb = CBackend(accelerate_keccak=False)
    for sizes in ([random.choice([1, 5, 127, 128, 129, 300, 700]) for _ in range(100)], [3, 500, 0, 9]):
        offs = [0]
        for s in sizes:
            offs.append(offs[-1] + s)
        ps = [pts[random.randrange(len(pts))] for _ in range(offs[-1])]
        ks = r.get_frs(offs[-1])
        for i in range(0, len(ps), 41):
            ps[i] = None
        got = affs_dec(ctx.g1_msm_batch(affs_enc(ps), frs_enc(ks), offs))
        want = [cb.msm(ps[offs[i]:offs[i + 1]], ks[offs[i]:offs[i + 1]]) for i in range(len(sizes))]
        assert got == want


def test_msm_batch_over_device_resident_pool(ctx, pkg):
    """cdl_g1_msm_batch_device: the Go-hosted form of an IPA round (innerproductargument.go:100-172) —
    bases stay in HBM, indices / scalars come from the host, results land in pool slots, are returned
    affine and as the 48-byte encodings the transcript hashes; then the bases are folded on the device
    and used again.  Everything is compared with the host-pointer entry points and the oracle."""
    import random

    random.seed(21)
    n = 16
    pts = [b.g1_mul(b.G1_GEN, random.randrange(1, b.R)) for _ in range(n)]
    pool = ctx.dev_buffer(96 * (n + 4))
    pool.upload(affs_enc(pts) + bytes(96 * 4))
    half = n // 2
    cL = [random.randrange(b.R) for _ in range(half)]
    cR = [random.randrange(b.R) for _ in range(half)]
    # two MSMs of one round: <c_L, G_R> and <c_R, -G_L> (bit 31 negates), results into slots n, n+1
    idx = [half + i for i in range(half)] + [(1 << 31) | i for i in range(half)]
    sc = b"".join(fr_enc(x) for x in cL + cR)
    aff, enc = ctx.g1_msm_batch_device(pool, idx, sc, [0, half, n], out_slot=[n, n + 1])
    want0 = b.g1_msm(pts[half:], cL)
    want1 = b.g1_neg(b.g1_msm(pts[:half], cR))
    assert affs_dec(aff) == [want0, want1]
    assert enc == b.g1_compress(want0) + b.g1_compress(want1)
    assert affs_dec(pool.download(96 * 2, 96 * n)) == [want0, want1]
    # fold the resident bases: G_L[i] += x * G_R[i], then an MSM over the folded half plus a result slot
    x = random.randrange(1, b.R)
    dx = ctx.dev_buffer(32)
    dx.upload(fr_enc(x))
    L, Rr = ctx.dev_buffer(96 * half), ctx.dev_buffer(96 * half)
    L.upload(affs_enc(pts[:half]))
    Rr.upload(affs_enc(pts[half:]))
    ctx.g1_fold_device(L, Rr, dx, half)
    folded = [b.g1_add(pts[i], b.g1_mul(pts[half + i], x)) for i in range(half)]
    assert affs_dec(L.download(96 * half)) == folded
    pool.upload(L.download(96 * half))  # folded bases back into the pool's first half
    s2 = [random.randrange(b.R) for _ in range(half + 1)]
    aff2, enc2 = ctx.g1_msm_batch_device(pool, list(range(half)) + [n], b"".join(fr_enc(v) for v in s2), [0, half + 1])
    want2 = b.g1_add(b.g1_msm(folded, s2[:half]), b.g1_mul(want0, s2[half]))
    assert affs_dec(aff2) == [want2] and enc2 == b.g1_compress(want2)
    # degenerate: an empty MSM and zero scalars give infinity
    aff3, enc3 = ctx.g1_msm_batch_device(pool, [0, 1], fr_enc(0) * 2, [0, 0, 2])
    assert affs_dec(aff3) == [None, None] and enc3 == (bytes([0xC0]) + bytes(47)) * 2
    for d in (pool, dx, L, Rr):
        d.close()


def test_msm_calls_share_the_engine_pool_with_protocol_calls(ctx, pkg, pts):
    """The batched-MSM entry points run on the context's engine and overwrite the start of the point pool
    that the protocol calls keep their CRS image and instances in.  A batch of 32 Whisk round trips runs on
    that same (root) engine; MSM calls between two runs with the same seeds must give the oracle's results
    and leave the second run byte-identical to the first."""
    ell, B = 12, 32
    crs = ctx.generate_crs(ell, pkg.Rand(0))
    r = pkg.Rand(1000)
    rs, ks = r.get_frs(ell), r.get_frs(ell)
    rG = ctx.g1_scalar_mul_affine(aff_enc(b.G1_GEN) * ell, rs, broadcast=False)
    e1, e2 = ctx.g1_compress(rG), ctx.g1_compress(ctx.g1_scalar_mul_affine(rG, ks, broadcast=False))
    pre = b"".join(e1[48 * j:48 * j + 48] + e2[48 * j:48 * j + 48] for j in range(ell)) * B

    def round_trip():
        post, proofs, status = ctx.whisk_generate_shuffle_proof_batch(crs, pre, [pkg.Rand(3000 + i) for i in range(B)])
        ok, st = ctx.whisk_is_valid_shuffle_proof_batch(crs, pre, post, proofs, [pkg.Rand(2000 + i) for i in range(B)])
        assert status == [0] * B and st == [0] * B and ok == [1] * B
        return bytes(post), bytes(proofs)

    first = round_trip()
    random.seed(31)
    offs = [0, 5, 5, 45, 46]
    ps = [pts[random.randrange(len(pts))] for _ in range(offs[-1])]
    sc = [random.randrange(R) for _ in range(offs[-1])]
    got = affs_dec(ctx.g1_msm_batch(affs_enc(ps), frs_enc(sc), offs))
    assert got == [b.g1_msm_naive(ps[offs[i]:offs[i + 1]], sc[offs[i]:offs[i + 1]]) for i in range(len(offs) - 1)]
    pool = ctx.dev_buffer(96 * 10)
    pool.upload(affs_enc(pts[:8]) + bytes(96 * 2))
    sc = [random.randrange(R) for _ in range(8)]
    aff, enc = ctx.g1_msm_batch_device(pool, list(range(8)), frs_enc(sc), [0, 3, 8], out_slot=[9, 8])
    want = [b.g1_msm(pts[:3], sc[:3]), b.g1_msm(pts[3:8], sc[3:])]
    assert affs_dec(aff) == want and enc == b"".join(b.g1_compress(p) for p in want)
    assert affs_dec(pool.download(96 * 2, 96 * 8)) == want[::-1]
    pool.close()
    assert round_trip() == first
