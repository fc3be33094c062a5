"""Batched parity at the reference's own shapes (VERDICT r1 item 1a): cdl_whisk_*_batch against the
CPU oracle, instance by instance, at ell = 124 (Whisk, n = 128; BASELINE.json configs 2 and 4) and
ell = 252 (n = 256, a reference benchmark shape, curdleproof_test.go:184-237), with all five mutation
kinds of SURVEY.md §8d config 4 mixed into the batch:

  0  Rs / Ss swapped (the two components of every pre-tracker)      curdleproof_test.go:48-75
  1  post-trackers re-permuted                                      curdleproof_test.go:77-107
  2  M -> k*M                                                       curdleproof_test.go:109-137
  3  one bit of the proof's last scalar x flipped
  4  Ts[0] replaced by the infinity encoding ("randomizer is zero", an error, curdleproof.go:208-211)

The expected verdict / error of every instance is what oracle.whisk.is_valid_whisk_shuffle_proof
returns for the same bytes and the same verifier RNG seed.  Proof bytes of the first instances are
also compared with the oracle's prover (byte identical)."""
import pytest

from oracle import bls12381 as b
from util import aff_enc

pytestmark = pytest.mark.gpu

KINDS = 5


def make_trackers(ctx, pkg, ell, seed):
    """whisk_test.go generateShuffleTrackers: per tracker k then r; (r*G, k*r*G) compressed."""
    r = pkg.Rand(seed)
    ks, rs = [], []
    for _ in range(ell):
        ks.append(r.get_fr())
        rs.append(r.get_fr())
    gen = aff_enc(b.G1_GEN)
    rG = ctx.g1_scalar_mul_affine(gen * ell, b"".join(rs), broadcast=False)
    krG = ctx.g1_scalar_mul_affine(rG, b"".join(ks), broadcast=False)
    e1, e2 = ctx.g1_compress(rG), ctx.g1_compress(krG)
    return b"".join(e1[48 * j:48 * j + 48] + e2[48 * j:48 * j + 48] for j in range(ell))


def oracle_crs(ctx, crs, ell):
    from oracle import protocol as P

    enc = bytes(ctx.g1_compress(crs.export()))
    pts = [b.g1_decompress(enc[48 * j:48 * j + 48]) for j in range(ell + 9)]
    return P.CRS(pts[:ell], pts[ell:ell + 4], pts[ell + 4], pts[ell + 5], pts[ell + 6], pts[ell + 7], pts[ell + 8])


def used_len(ell):
    n = ell + 4
    m = n.bit_length() - 1
    return 48 * (19 + 10 * m) + 7 * 32 + 10 * 4


def mutate(ctx, pkg, kind, ell, pre, post, proof):
    """Returns (pre, post, proof) of one instance after mutation `kind`."""
    pre, post, proof = bytearray(pre), bytearray(post), bytearray(proof)
    if kind == 0:
        for j in range(ell):
            pre[96 * j:96 * j + 48], pre[96 * j + 48:96 * j + 96] = pre[96 * j + 48:96 * j + 96], pre[96 * j:96 * j + 48]
    elif kind == 1:
        p2 = pkg.Rand(5).generate_permutation(ell)
        post = bytearray(b"".join(bytes(post[96 * j:96 * j + 96]) for j in p2))
    elif kind == 2:
        M_aff, st = ctx.g1_decompress(bytes(proof[:48]))
        assert list(st) == [0]
        kM = ctx.g1_scalar_mul_affine(M_aff, pkg.Rand(9).get_fr(), broadcast=True)
        proof[:48] = ctx.g1_compress(kM)
    elif kind == 3:
        proof[used_len(ell) - 1] ^= 1
    elif kind == 4:
        post[0:48] = bytes([0xC0]) + bytes(47)
    return bytes(pre), bytes(post), bytes(proof)


def run_batch(ctx, pkg, ell, B, proof_size, every, n_byte_checks):
    from oracle import protocol as P, whisk as W
    from oracle.cbackend import CBackend
    from oracle.rand import Rand as ORand

    crs = ctx.generate_crs(ell, pkg.Rand(0))
    sets = [make_trackers(ctx, pkg, ell, 1000 + i) for i in range(3)]
    pres = [sets[i % 3] for i in range(B)]
    post, proofs, status = ctx.whisk_generate_shuffle_proof_batch(crs, b"".join(pres), [pkg.Rand(3000 + i) for i in range(B)],
                                                                  proof_size=proof_size)
    assert status == [0] * B
    tb = 96 * ell
    posts = [bytes(post[i * tb:(i + 1) * tb]) for i in range(B)]
    prfs = [bytes(proofs[i * proof_size:(i + 1) * proof_size]) for i in range(B)]
    kinds = {}
    for i in range(0, B, every):
        kinds[i] = (i // every) % KINDS
        pres[i], posts[i], prfs[i] = mutate(ctx, pkg, kinds[i], ell, pres[i], posts[i], prfs[i])
    assert set(kinds.values()) == set(range(KINDS))
    ok, st = ctx.whisk_is_valid_shuffle_proof_batch(crs, b"".join(pres), b"".join(posts), b"".join(prfs),
                                                    [pkg.Rand(2000 + i) for i in range(B)], proof_size=proof_size)
    P.set_backend(CBackend())
    try:
        ocrs = oracle_crs(ctx, crs, ell)
        split = lambda t: [(t[96 * j:96 * j + 48], t[96 * j + 48:96 * j + 96]) for j in range(ell)]  # noqa: E731
        # byte-identical proofs and post-trackers against the oracle's prover for the first instances
        for i in range(n_byte_checks):
            want_post, want_proof = W.generate_whisk_shuffle_proof(ocrs, split(sets[i % 3]), ORand(3000 + i), ell=ell,
                                                                   proof_size=proof_size)
            assert b"".join(x + y for x, y in want_post) == bytes(post[i * tb:(i + 1) * tb]), i
            assert want_proof == bytes(proofs[i * proof_size:(i + 1) * proof_size]), i
        # verdict / error of every instance
        for i in range(B):
            try:
                want, err = W.is_valid_whisk_shuffle_proof(ocrs, split(pres[i]), split(posts[i]), prfs[i], ORand(2000 + i)), False
            except (W.WhiskError, P.ProofError):
                want, err = False, True
            assert bool(ok[i]) == want and (st[i] != 0) == err, (i, kinds.get(i), ok[i], st[i], want, err)
            if i not in kinds:
                assert ok[i] == 1 and st[i] == 0, i
            else:
                assert ok[i] == 0, (i, kinds[i])
                assert (st[i] == -5) == (kinds[i] == 4), (i, kinds[i], st[i])
    finally:
        P.set_backend(P.PyBackend())
    crs.close()


def test_batched_generation_matches_single_calls_and_oracle(ctx, pkg):
    """B >= 8 takes the two-launch form of the prover's step 3 (R, S first, then T_2/U_2/A_2/B_2 as
    two-term MSMs); one proof at a time takes the fused form: both must give the oracle's bytes."""
    ell, B = 12, 9
    crs = ctx.generate_crs(ell, pkg.Rand(0))
    pres = [make_trackers(ctx, pkg, ell, 1000 + i) for i in range(B)]
    single = [ctx.whisk_generate_shuffle_proof(crs, pres[i], pkg.Rand(3000 + i)) for i in range(B)]
    post, proofs, status = ctx.whisk_generate_shuffle_proof_batch(crs, b"".join(pres), [pkg.Rand(3000 + i) for i in range(B)])
    assert status == [0] * B
    for i in range(B):
        assert bytes(post[i * ell * 96:(i + 1) * ell * 96]) == single[i][0]
        assert bytes(proofs[i * 4576:(i + 1) * 4576]) == single[i][1]
    crs.close()
    run_batch(ctx, pkg, ell, 20, 4576, 2, 3)


def test_whisk_n128_batch64_five_mutation_kinds_match_oracle(ctx, pkg):
    run_batch(ctx, pkg, 124, 64, 4576, 4, 2)


def test_fixed_base_tables_give_the_same_bytes_and_verdicts(ctx, pkg):
    """CRS fixed-base tables (cdl_set_fixed_base_min_batch; csrc/fixed_base.cuh) forced on for every call, with
    them the lazy schedule of Engine::prove (second-round MSMs on pairs of CRS points, the twice-folded G, G', Gm
    built straight from the CRS), against the oracle's proofs and verdicts with all five mutation kinds, at
    n = 128 and (small, so that short windows, tiny tasks and the Gt / Gu slots of the first fold are hit) n = 16;
    then the same batch with the tables off: identical bytes.  These batches of at most 32 instances per lane
    read the tables in the MSMs only (k_msm_fixed, the commitments, B_c / B_a and the verifier's merged CRS
    terms): their elementwise stages stay within kQuadMaxOps ops, and the quad kernel that runs them has no
    tables.  The folds and Gs' on the tables are checked in test_gpu_crossovers.py."""
    try:
        ctx.set_fixed_base_min_batch(1)
        run_batch(ctx, pkg, 124, 64, 4576, 4, 2)
        run_batch(ctx, pkg, 12, 20, 4576, 2, 3)
        ell, B = 124, 40
        crs = ctx.generate_crs(ell, pkg.Rand(0))
        pre = b"".join(make_trackers(ctx, pkg, ell, 1000 + i % 3) for i in range(B))
        on = ctx.whisk_generate_shuffle_proof_batch(crs, pre, [pkg.Rand(3000 + i) for i in range(B)])
        ctx.set_fixed_base_min_batch(0)
        off = ctx.whisk_generate_shuffle_proof_batch(crs, pre, [pkg.Rand(3000 + i) for i in range(B)])
        assert bytes(on[0]) == bytes(off[0]) and bytes(on[1]) == bytes(off[1]) and on[2] == off[2] == [0] * B
        crs.close()
    finally:
        ctx.set_fixed_base_min_batch(-1)


def test_n256_batch_five_mutation_kinds_match_oracle(ctx, pkg):
    run_batch(ctx, pkg, 252, 20, 5056, 2, 1)


def test_verifier_scalars_device_and_host_paths_agree(ctx, pkg):
    """The verifier's merged-base scalars come from k_verify_scalars (device) by default; CDL_VERIFY_SCALARS=host
    keeps the host computation.  Both must return the verdicts of this process (which the tests above pin to
    the oracle) on a batch with every mutation kind."""
    import json
    import os
    import subprocess
    import sys

    ell, B = 12, 20
    crs = ctx.generate_crs(ell, pkg.Rand(0))
    sets = [make_trackers(ctx, pkg, ell, 1000 + i) for i in range(3)]
    pres = [sets[i % 3] for i in range(B)]
    post, proofs, status = ctx.whisk_generate_shuffle_proof_batch(crs, b"".join(pres), [pkg.Rand(3000 + i) for i in range(B)])
    assert status == [0] * B
    tb = 96 * ell
    posts = [bytes(post[i * tb:(i + 1) * tb]) for i in range(B)]
    prfs = [bytes(proofs[i * 4576:(i + 1) * 4576]) for i in range(B)]
    for i in range(0, B, 2):
        pres[i], posts[i], prfs[i] = mutate(ctx, pkg, (i // 2) % KINDS, ell, pres[i], posts[i], prfs[i])
    ok, st = ctx.whisk_is_valid_shuffle_proof_batch(crs, b"".join(pres), b"".join(posts), b"".join(prfs),
                                                    [pkg.Rand(2000 + i) for i in range(B)])
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = (
        "import importlib, json, sys; sys.path.insert(0, %r); pkg = importlib.import_module('go-curdleproofs_b200'); "
        "ctx = pkg.Context(0); crs = ctx.generate_crs(%d, pkg.Rand(0)); d = json.load(sys.stdin); "
        "ok, st = ctx.whisk_is_valid_shuffle_proof_batch(crs, bytes.fromhex(d['pre']), bytes.fromhex(d['post']), "
        "bytes.fromhex(d['proofs']), [pkg.Rand(2000 + i) for i in range(%d)]); print(json.dumps([ok, st]))" % (root, ell, B))
    payload = json.dumps({"pre": b"".join(pres).hex(), "post": b"".join(posts).hex(), "proofs": b"".join(prfs).hex()})
    out = subprocess.run([sys.executable, "-c", code], input=payload, capture_output=True, text=True,
                         env=dict(os.environ, CDL_VERIFY_SCALARS="host"), check=True).stdout
    assert json.loads(out.strip().splitlines()[-1]) == [ok, st]
    assert ok.count(1) == B - len(range(0, B, 2))
    crs.close()


def test_n512_batch_five_mutation_kinds_match_oracle(ctx, pkg):
    """BASELINE.json names n = 512: the batched entry points at shuffled_elements = 508 (bench.py's n512 line)."""
    run_batch(ctx, pkg, 508, 10, 5504, 2, 1)
