"""CRSes built from the caller's points (cdl_crs_from_points, how a node wraps the CRS it already holds) against
generated ones and the CPU oracle.

The prover and verifier use Gsum and Hsum in place of the vectors Gs and Hs (B = A + alpha M + beta Gsum,
D = B - beta^-1 Gsum + alpha Hsum), so a CRS whose sums are not the sums of its points would give proofs that differ
from the reference's; the reference's own verifier rejects its proofs under such a CRS.  cdl_crs_from_points
refuses it.  Consistent but degenerate CRSes (one point everywhere, opposite and infinite points) make the
protocol MSMs add equal and opposite bases; their proofs and verdicts must still be the oracle's."""
import pytest

from oracle import bls12381 as b
from test_gpu_parity_batch import KINDS, make_trackers, mutate, used_len
from util import aff_enc, affs_dec, affs_enc, fr_dec, jac_dec

pytestmark = pytest.mark.gpu

INVALID_ARG = -3
SIZE = 4576
G = b.G1_GEN
P = b.g1_mul(G, 0x5EED0F1234567)


def oracle_crs(pts_aff, ell):
    from oracle import protocol as OP

    p = affs_dec(pts_aff)
    return OP.CRS(p[:ell], p[ell:ell + 4], p[ell + 4], p[ell + 5], p[ell + 6], p[ell + 7], p[ell + 8])


def split(t, ell):
    return [(t[96 * j:96 * j + 48], t[96 * j + 48:96 * j + 96]) for j in range(ell)]


def with_sums(drawn, ell):
    """the ell + 7 drawn points followed by their Gsum and Hsum, as the C ABI's affine image"""
    return affs_enc(drawn + [b.g1_sum(drawn[:ell]), b.g1_sum(drawn[ell:ell + 4])])


_TRACKERS = {}


def trackers(ctx, pkg, ell, i):
    key = (ell, i % 3)
    if key not in _TRACKERS:
        _TRACKERS[key] = make_trackers(ctx, pkg, ell, 1000 + i % 3)
    return _TRACKERS[key]


def protocol_calls(c, pkg, crs, ell, B):
    """shuffle-permute-commit, prove, verify (3 instances) and Whisk generation / validation (B instances, one
    of them with a flipped proof bit) on one CRS: every output byte, verdict and status"""
    n = 3
    Rs = [c.rand_get_g1_affines(pkg.Rand(100 + i), ell) for i in range(n)]
    Ss = [c.rand_get_g1_affines(pkg.Rand(200 + i), ell) for i in range(n)]
    perms = [pkg.Rand(300 + i).generate_permutation(ell) for i in range(n)]
    ks = [pkg.Rand(400 + i).get_fr() for i in range(n)]
    Ts, Us, Ms, rs_ms, st = c.shuffle_permute_commit_batch(crs, Rs, Ss, perms, ks, [pkg.Rand(500 + i) for i in range(n)])
    proofs, lens, pst = c.prove_batch(crs, Rs, Ss, Ts, Us, Ms, perms, ks, rs_ms, [pkg.Rand(600 + i) for i in range(n)])
    ok, vst = c.verify_batch(crs, proofs, Rs, Ss, Ts, Us, Ms, [pkg.Rand(700 + i) for i in range(n)])
    assert st == pst == vst == [0] * n and ok == [1] * n
    pre = b"".join(trackers(c, pkg, ell, i) for i in range(B))
    post, wproofs, wst = c.whisk_generate_shuffle_proof_batch(crs, pre, [pkg.Rand(3000 + i) for i in range(B)])
    wproofs = bytearray(wproofs)
    wproofs[SIZE + used_len(ell) - 1] ^= 1  # instance 1's last scalar: a valid encoding that must fail
    wok, wvst = c.whisk_is_valid_shuffle_proof_batch(crs, pre, post, wproofs, [pkg.Rand(2000 + i) for i in range(B)])
    assert wst == wvst == [0] * B and wok == [1] + [0] + [1] * (B - 2)
    return Ts, Us, Ms, rs_ms, proofs, ok, bytes(post), bytes(wproofs), wok


# ------------------------------------------------------------------------------------------------- round trip
@pytest.mark.parametrize("ell", [4, 12, 124])
def test_round_trip_matches_generated_crs(ctx, pkg, ell):
    gen = ctx.generate_crs(ell, pkg.Rand(0))
    pts = gen.export()
    own = ctx.crs_from_points(ell, pts)
    assert own.ell == ell and len(pts) == 96 * (ell + 9)
    assert own.export() == pts
    runs = []
    try:
        for tables in (1, 0):
            ctx.set_fixed_base_min_batch(tables)
            want = protocol_calls(ctx, pkg, gen, ell, 64)
            assert protocol_calls(ctx, pkg, own, ell, 64) == want, tables
            runs.append(want)
    finally:
        ctx.set_fixed_base_min_batch(-1)
    assert runs[0] == runs[1]
    own.close()
    gen.close()


def test_round_trip_on_two_slots(ctx, pkg):
    """Context(devices=[0, 0]): slot 1 uploads its replica of the CRS from the host image on first use; 64 Whisk
    instances split over both slots.  Same bytes as the one-device context; a CRS of one context is refused by the
    other."""
    ell = 12
    pts = ctx.generate_crs(ell, pkg.Rand(0)).export()
    want = protocol_calls(ctx, pkg, ctx.crs_from_points(ell, pts), ell, 64)
    two = pkg.Context(devices=[0, 0])
    try:
        own = two.crs_from_points(ell, pts)
        assert own.export() == pts
        for tables in (1, 0):
            two.set_fixed_base_min_batch(tables)
            assert protocol_calls(two, pkg, own, ell, 64) == want, tables
        pre = trackers(ctx, pkg, ell, 0)
        with pytest.raises(pkg.CdlError) as ei:
            ctx.whisk_generate_shuffle_proof_batch(own, pre, [pkg.Rand(1)])
        assert ei.value.code == INVALID_ARG and "another context" in ei.value.msg
        own.close()
    finally:
        two.close()


# ------------------------------------------------------------------------------------------------- wrong sums
@pytest.mark.parametrize("which", ["Gsum", "Hsum"])
def test_inconsistent_sums_are_refused(ctx, pkg, which):
    """Gsum + G in place of Gsum (or Hsum + G for Hsum) is refused with the sum named.  The oracle's prover does
    not read the sums, its verifier does: its own proof under the bad CRS is rejected, the same proof under the
    consistent CRS accepted, which is why such a CRS is refused rather than used."""
    from oracle import protocol as OP, whisk as W
    from oracle.cbackend import CBackend
    from oracle.rand import Rand as ORand

    ell = 12
    pts = ctx.generate_crs(ell, pkg.Rand(0)).export()
    slot = ell + 7 if which == "Gsum" else ell + 8
    bad = bytearray(pts)
    bad[96 * slot:96 * slot + 96] = aff_enc(b.g1_add(affs_dec(pts[96 * slot:96 * slot + 96])[0], G))
    bad = bytes(bad)
    with pytest.raises(pkg.CdlError) as ei:
        ctx.crs_from_points(ell, bad)
    assert ei.value.code == INVALID_ARG and which in ei.value.msg, ei.value.msg
    assert ctx.crs_from_points(ell, pts).export() == pts  # the context is still usable
    OP.set_backend(CBackend())
    try:
        pre = split(trackers(ctx, pkg, ell, 0), ell)
        post, proof = W.generate_whisk_shuffle_proof(oracle_crs(bad, ell), pre, ORand(3000), ell=ell, proof_size=SIZE)
        assert W.is_valid_whisk_shuffle_proof(oracle_crs(pts, ell), pre, post, proof, ORand(2000)) is True
        try:
            verdict = W.is_valid_whisk_shuffle_proof(oracle_crs(bad, ell), pre, post, proof, ORand(2000))
        except (W.WhiskError, OP.ProofError):
            verdict = False
        assert verdict is False
    finally:
        OP.set_backend(OP.PyBackend())


# ------------------------------------------------------------------------------------------------- degenerate
def degenerate_points(ctx, pkg, case, ell):
    if case == "one-point":  # every drawn point is P
        drawn = [P] * (ell + 7)
    elif case == "multiples":  # Gs[i] = (i + 1) P, Hs[j] = -Gs[j], H = Gt = Gu = P
        gs = [P]
        for _ in range(ell - 1):
            gs.append(b.g1_add(gs[-1], P))
        drawn = gs + [b.g1_neg(gs[j]) for j in range(4)] + [P, P, P]
    else:  # a random CRS with Gs[1] = -Gs[0] and Hs[2] at infinity
        drawn = affs_dec(ctx.generate_crs(ell, pkg.Rand(5)).export())[:ell + 7]
        drawn[1] = b.g1_neg(drawn[0])
        drawn[ell + 2] = None
    return with_sums(drawn, ell)


def oracle_outcome(fn):
    """fn()'s value, or "error" where the reference returns an error"""
    from oracle import protocol as OP, whisk as W

    try:
        return fn()
    except (W.WhiskError, OP.ProofError, b.DecodeError):
        return "error"


@pytest.mark.parametrize("ell", [12, 124])
@pytest.mark.parametrize("case", ["one-point", "multiples", "opposite-and-infinity"])
def test_degenerate_consistent_crs_matches_oracle(ctx, pkg, case, ell):
    from oracle import protocol as OP, whisk as W
    from oracle.cbackend import CBackend
    from oracle.rand import Rand as ORand

    B, checked = 64, 3
    pts = degenerate_points(ctx, pkg, case, ell)
    crs = ctx.crs_from_points(ell, pts)
    assert crs.export() == pts
    ocrs = oracle_crs(pts, ell)
    sets = [trackers(ctx, pkg, ell, i) for i in range(3)]
    pres = [sets[i % 3] for i in range(B)]
    outs = []
    try:
        for tables in (1, 0):
            ctx.set_fixed_base_min_batch(tables)
            outs.append(ctx.whisk_generate_shuffle_proof_batch(crs, b"".join(pres), [pkg.Rand(3000 + i) for i in range(B)]))
    finally:
        ctx.set_fixed_base_min_batch(-1)
    assert outs[0] == outs[1]
    post, proofs, status = outs[0]
    tb = 96 * ell
    posts = [bytes(post[i * tb:(i + 1) * tb]) for i in range(B)]
    prfs = [bytes(proofs[i * SIZE:(i + 1) * SIZE]) for i in range(B)]
    OP.set_backend(CBackend())
    try:
        # the first instances' post-trackers and proofs against the oracle's prover
        for i in range(checked):
            want = oracle_outcome(lambda: W.generate_whisk_shuffle_proof(ocrs, split(sets[i % 3], ell), ORand(3000 + i),
                                                                          ell=ell, proof_size=SIZE))
            if want == "error":
                assert status[i] != 0, i
                continue
            assert status[i] == 0 and b"".join(x + y for x, y in want[0]) == posts[i] and want[1] == prfs[i], i
        # verdicts: the checked instances and one of every mutation kind against the oracle's verifier
        kinds = {8 * (j + 1): j for j in range(KINDS)}
        for i, k in kinds.items():
            pres[i], posts[i], prfs[i] = mutate(ctx, pkg, k, ell, pres[i], posts[i], prfs[i])
        ok, st = ctx.whisk_is_valid_shuffle_proof_batch(crs, b"".join(pres), b"".join(posts), b"".join(prfs),
                                                        [pkg.Rand(2000 + i) for i in range(B)])
        for i in sorted(set(range(checked)) | set(kinds)):
            if status[i] != 0:
                continue
            want = oracle_outcome(lambda: W.is_valid_whisk_shuffle_proof(ocrs, split(pres[i], ell), split(posts[i], ell),
                                                                          prfs[i], ORand(2000 + i)))
            assert (st[i] != 0) == (want == "error") and bool(ok[i]) == (want is True), (i, kinds.get(i), ok[i], st[i], want)
        for i in range(B):  # the instances left alone verify as the first one does
            if i not in kinds and status[i] == status[0] == 0:
                assert (ok[i], st[i]) == (ok[0], st[0]), i

        # one prove / verify pair of the curdleproof API
        Rs_b, Ss_b = ctx.rand_get_g1_affines(pkg.Rand(11), ell), ctx.rand_get_g1_affines(pkg.Rand(12), ell)
        perm, k = pkg.Rand(13).generate_permutation(ell), pkg.Rand(14).get_fr()
        Rs, Ss, kv = affs_dec(Rs_b), affs_dec(Ss_b), fr_dec(k)
        oTs, oUs, oM, ors_m = OP.shuffle_permute_commit(ocrs.Gs, ocrs.Hs, Rs, Ss, perm, kv, ORand(15))
        Ts, Us, M, rs_m = ctx.shuffle_permute_commit(crs, Rs_b, Ss_b, perm, k, pkg.Rand(15))
        assert Ts == affs_enc(oTs) and Us == affs_enc(oUs) and jac_dec(M) == oM
        want = oracle_outcome(lambda: OP.prove(ocrs, Rs, Ss, oTs, oUs, oM, perm, kv, ors_m, ORand(16)).serialize())
        if want == "error":
            with pytest.raises(pkg.CdlError):
                ctx.prove(crs, Rs_b, Ss_b, Ts, Us, M, perm, k, rs_m, pkg.Rand(16))
        else:
            proof = ctx.prove(crs, Rs_b, Ss_b, Ts, Us, M, perm, k, rs_m, pkg.Rand(16))
            assert proof == want
            verdict = oracle_outcome(lambda: OP.verify(OP.Proof.deserialize(proof), ocrs, Rs, Ss, oTs, oUs, oM, ORand(17)))
            if verdict == "error":
                with pytest.raises(pkg.CdlError):
                    ctx.verify(crs, proof, Rs_b, Ss_b, Ts, Us, M, pkg.Rand(17))
            else:
                assert ctx.verify(crs, proof, Rs_b, Ss_b, Ts, Us, M, pkg.Rand(17)) is verdict
    finally:
        OP.set_backend(OP.PyBackend())
    crs.close()
