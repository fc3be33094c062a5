"""The combined verifier check of batched Whisk shuffle-proof verification (cdl_set_batch_verify_min): forced on
(1) it must give exactly what forced off (0) gives on the same inputs: verdicts, statuses (which separate a
false verdict from an error), and the
position of every caller Rand afterwards (the reference restores its snapshot when the same-scalar check
fails).  Mutation kinds are those of test_gpu_parity_batch."""
import pytest

from test_gpu_parity_batch import make_trackers, mutate, oracle_crs

pytestmark = pytest.mark.gpu


@pytest.fixture
def knob(ctx):
    yield
    ctx.set_batch_verify_min(-1)


def gen(ctx, pkg, ell, B, proof_size=None):
    crs = ctx.generate_crs(ell, pkg.Rand(0))
    sets = [make_trackers(ctx, pkg, ell, 1000 + i) for i in range(3)]
    pres = [sets[i % 3] for i in range(B)]
    ps = proof_size or wire_len(ell)
    post, proofs, status = ctx.whisk_generate_shuffle_proof_batch(crs, b"".join(pres), [pkg.Rand(3000 + i) for i in range(B)],
                                                                  proof_size=ps)
    assert status == [0] * B
    tb = 96 * ell
    return (crs, pres, [bytes(post[i * tb:(i + 1) * tb]) for i in range(B)],
            [bytes(proofs[i * ps:(i + 1) * ps]) for i in range(B)], ps)


def wire_len(ell):
    m = (ell + 4).bit_length() - 1
    return 48 * (19 + 10 * m) + 7 * 32 + 10 * 4


def verify(ctx, pkg, crs, pres, posts, prfs, ps, mode):
    ctx.set_batch_verify_min(mode)
    B = len(pres)
    rands = [pkg.Rand(2000 + i) for i in range(B)]
    n0 = ctx.launch_count()
    ok, st = ctx.whisk_is_valid_shuffle_proof_batch(crs, b"".join(pres), b"".join(posts), b"".join(prfs), rands,
                                                    proof_size=ps)
    nl = ctx.launch_count() - n0
    nxt = [r.get_fr() for r in rands]
    for r in rands:
        r.close()
    return list(ok), list(st), None, nxt, nl


def same_both_ways(ctx, pkg, crs, pres, posts, prfs, ps):
    off = verify(ctx, pkg, crs, pres, posts, prfs, ps, 0)
    on = verify(ctx, pkg, crs, pres, posts, prfs, ps, 1)
    assert on[0] == off[0]
    assert on[1] == off[1]
    assert on[3] == off[3], "caller Rand positions differ"
    return on, off


# offsets inside a Whisk proof (M first, then curdleproof.go:358-387) of ell = 124 fields
def layout(ell):
    m = (ell + 4).bit_length() - 1
    sl = 4 + 48 * m
    zk = 48 * 12 + 32 + 4 * sl + 64 + 4 * 48  # M, A..S, B, C, Rp, B_c, B_d, 4 IPA slices, c0, d0, A_1..B_2
    la = zk + 3 * 32 + 3 * 48                 # Z_k, Z_t, Z_u, B_a, B_t, B_u
    return m, zk, la


def flip_zk(ell, proof):
    """Z_k's lowest bit: only the same-scalar equalities change (Z_k is never hashed)."""
    _, zk, _ = layout(ell)
    p = bytearray(proof)
    p[zk + 31] ^= 1
    return bytes(p)


def short_la(ell, proof):
    """L_A one point shorter and L_T one longer: the proof parses and decodes, the same-scalar check still
    holds, and the verifier fails later with "must by log2(L_a)" (an error, not a false verdict)."""
    m, _, la = layout(ell)
    p = bytes(proof)
    pts_a = p[la + 4:la + 4 + 48 * m]
    lt = la + 4 + 48 * m
    pts_t = p[lt + 4:lt + 4 + 48 * m]
    new = (m - 1).to_bytes(4, "big") + pts_a[:-48] + (m + 1).to_bytes(4, "big") + pts_a[-48:] + pts_t
    return p[:la] + new + p[lt + 4 + 48 * m:]


@pytest.mark.parametrize("ell,B", [(124, 64), (12, 96)])
def test_all_valid(ctx, pkg, knob, ell, B):
    crs, pres, posts, prfs, ps = gen(ctx, pkg, ell, B)
    on, off = same_both_ways(ctx, pkg, crs, pres, posts, prfs, ps)
    assert on[0] == [1] * B and on[1] == [0] * B
    assert on[4] != off[4], "the combined check did not run"
    crs.close()


def test_mutation_kinds_match_oracle(ctx, pkg, knob):
    from oracle import protocol as P, whisk as W
    from oracle.cbackend import CBackend
    from oracle.rand import Rand as ORand

    ell, B, every = 124, 48, 8
    crs, pres, posts, prfs, ps = gen(ctx, pkg, ell, B)
    kinds = {}
    for i in range(0, B - every, every):
        kinds[i] = (i // every) % 5
        pres[i], posts[i], prfs[i] = mutate(ctx, pkg, kinds[i], ell, pres[i], posts[i], prfs[i])
    on, _ = same_both_ways(ctx, pkg, crs, pres, posts, prfs, ps)
    ok, st = on[0], on[1]
    for i in range(B):
        if i in kinds:
            assert ok[i] == 0 and (st[i] == -5) == (kinds[i] == 4), (i, kinds[i], ok[i], st[i])
        else:
            assert ok[i] == 1 and st[i] == 0, i
    P.set_backend(CBackend())
    try:
        ocrs = oracle_crs(ctx, crs, ell)
        split = lambda t: [(t[96 * j:96 * j + 48], t[96 * j + 48:96 * j + 96]) for j in range(ell)]  # noqa: E731
        for i in sorted(kinds)[:5] + [1, B - 1]:
            try:
                want, err = W.is_valid_whisk_shuffle_proof(ocrs, split(pres[i]), split(posts[i]), prfs[i], ORand(2000 + i)), False
            except (W.WhiskError, P.ProofError):
                want, err = False, True
            assert bool(ok[i]) == want and (st[i] != 0) == err, (i, ok[i], st[i], want, err)
    finally:
        P.set_backend(P.PyBackend())
    crs.close()


@pytest.mark.parametrize("where", ["first", "middle", "last"])
def test_one_invalid_proof(ctx, pkg, knob, where):
    ell, B = 124, 64
    crs, pres, posts, prfs, ps = gen(ctx, pkg, ell, B)
    i = {"first": 0, "middle": B // 2 + 3, "last": B - 1}[where]
    pres[i], posts[i], prfs[i] = mutate(ctx, pkg, 3, ell, pres[i], posts[i], prfs[i])
    on, _ = same_both_ways(ctx, pkg, crs, pres, posts, prfs, ps)
    assert on[0] == [0 if j == i else 1 for j in range(B)]
    assert on[1] == [0] * B
    crs.close()


def test_same_scalar_and_late_failures(ctx, pkg, knob):
    ell, B = 124, 64
    crs, pres, posts, prfs, ps = gen(ctx, pkg, ell, B)
    prfs[5] = flip_zk(ell, prfs[5])                    # same-scalar check fails: (false, nil)
    prfs[20] = short_la(ell, prfs[20])                 # late error: (false, err)
    prfs[40] = flip_zk(ell, short_la(ell, prfs[40]))   # both: the same-scalar check decides first, (false, nil)
    on, _ = same_both_ways(ctx, pkg, crs, pres, posts, prfs, ps)
    ok, st = on[0], on[1]
    assert [ok[j] for j in (5, 20, 40)] == [0, 0, 0]
    assert st[5] == 0 and st[20] != 0 and st[40] == 0, (st[5], st[20], st[40])
    assert all(ok[j] == 1 and st[j] == 0 for j in range(B) if j not in (5, 20, 40))
    crs.close()


def test_lanes(ctx, pkg, knob):
    ell, B = 124, 256
    crs, pres, posts, prfs, ps = gen(ctx, pkg, ell, B)
    for i in (7, 130, 255):
        pres[i], posts[i], prfs[i] = mutate(ctx, pkg, 3, ell, pres[i], posts[i], prfs[i])
    ctx.set_lanes(4)
    on, _ = same_both_ways(ctx, pkg, crs, pres, posts, prfs, ps)
    assert on[0] == [0 if j in (7, 130, 255) else 1 for j in range(B)]
    crs.close()
