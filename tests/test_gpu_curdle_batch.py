"""Batched ShufflePermuteCommit / Prove / Verify on caller-supplied instances (cdl_*_batch).  The single calls
are the reference (they are pinned to the golden fixtures and the oracle): per instance, a batch must give
the same outputs, the same status as the single call's return code, and leave the caller's Rand at the same
position."""
import ctypes as C
import json
import os

import numpy as np
import pytest

from test_gpu_parity_batch import make_trackers
from util import aff_dec, fr_dec, jac_enc

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
INVALID_ARG, DECODE, PROTOCOL, TOO_LARGE = -3, -4, -5, -6


@pytest.fixture
def knobs(ctx):
    yield
    ctx.set_lanes(4)
    ctx.set_batch_verify_min(-1)


def nxt(rand):
    return fr_dec(rand.get_fr())


def instances(ctx, pkg, ell, B, seed, point_sets=None):
    """B instances (Rs, Ss, perm, k), each with its own permutation and k; the points come from
    `point_sets` seeds (all distinct when None)."""
    sets = {}
    out = []
    for i in range(B):
        s = seed + (i if point_sets is None else i % point_sets)
        if s not in sets:
            r = pkg.Rand(s)
            sets[s] = (ctx.rand_get_g1_affines(r, ell), ctx.rand_get_g1_affines(r, ell))
        r = pkg.Rand(seed + 10_000 + i)
        out.append(sets[s] + (r.generate_permutation(ell), r.get_fr()))
    return out


def golden_instance(ctx, pkg, ell):
    """curdleproof_test.go:239-274 as test_gpu_protocol._setup builds it; returns the instance and the
    continuing Rand(0) that ShufflePermuteCommit draws from."""
    rand = pkg.Rand(0)
    rand.get_frs(ell + 7)  # GenerateCRS's draws
    k = rand.get_fr()
    Rs = ctx.rand_get_g1_affines(rand, ell)
    Ss = ctx.rand_get_g1_affines(rand, ell)
    return (Rs, Ss, pkg.Rand(42).generate_permutation(ell), k), rand


def single_commit(ctx, crs, inst, rand):
    Rs, Ss, perm, k = inst
    try:
        return ctx.shuffle_permute_commit(crs, Rs, Ss, perm, k, rand) + (0,)
    except Exception as e:  # CdlError
        return (None, None, None, None, e.code)


def single_prove(ctx, crs, inst, com, rand):
    Rs, Ss, perm, k = inst
    Ts, Us, M, rs_m = com
    try:
        return ctx.prove(crs, Rs, Ss, Ts, Us, M, perm, k, rs_m, rand), 0
    except Exception as e:
        return b"", e.code


def single_verify(ctx, crs, case, rand):
    proof, Rs, Ss, Ts, Us, M = case
    try:
        return int(ctx.verify(crs, proof, Rs, Ss, Ts, Us, M, rand)), 0
    except Exception as e:
        return 0, e.code


def commit_batch(ctx, pkg, crs, insts, seeds):
    rands = [pkg.Rand(s) for s in seeds]
    Ts, Us, M, rs_m, st = ctx.shuffle_permute_commit_batch(crs, [i[0] for i in insts], [i[1] for i in insts],
                                                           [i[2] for i in insts], [i[3] for i in insts], rands)
    return Ts, Us, M, rs_m, st, [nxt(r) for r in rands]


def prove_batch(ctx, pkg, crs, insts, coms, seeds, **kw):
    rands = [pkg.Rand(s) for s in seeds]
    proofs, lens, st = ctx.prove_batch(crs, [i[0] for i in insts], [i[1] for i in insts], [c[0] for c in coms],
                                       [c[1] for c in coms], [c[2] for c in coms], [i[2] for i in insts],
                                       [i[3] for i in insts], [c[3] for c in coms], rands, **kw)
    return proofs, lens, st, [nxt(r) for r in rands]


def verify_batch(ctx, pkg, crs, cases, seeds):
    rands = [pkg.Rand(s) for s in seeds]
    ok, st = ctx.verify_batch(crs, *[[c[j] for c in cases] for j in range(6)], rands)
    return ok, st, [nxt(r) for r in rands]


@pytest.mark.parametrize("ell,B", [(12, 8), (12, 70), (124, 8), (124, 70)])
def test_commit_and_prove_equal_single_calls(ctx, pkg, ell, B):
    crs = ctx.generate_crs(ell, pkg.Rand(0))
    insts = instances(ctx, pkg, ell, B, 100)
    golden = None
    if ell == 12:  # instance 3 is the golden one, with its continuing Rand(0) for the commitment
        insts[3], _ = golden_instance(ctx, pkg, ell)
        golden = json.load(open(os.path.join(GOLD, "prove_ell12.json")))
    cseeds = [5000 + i for i in range(B)]
    pseeds = [42 if golden and i == 3 else 6000 + i for i in range(B)]  # the golden proof uses Rand(42)

    def crand(i):
        return golden_instance(ctx, pkg, ell)[1] if golden and i == 3 else pkg.Rand(cseeds[i])

    singles = []
    for i in range(B):
        r = crand(i)
        singles.append(single_commit(ctx, crs, insts[i], r) + (nxt(r),))
    rands = [crand(i) for i in range(B)]
    Ts, Us, M, rs_m, st = ctx.shuffle_permute_commit_batch(crs, [x[0] for x in insts], [x[1] for x in insts],
                                                           [x[2] for x in insts], [x[3] for x in insts], rands)
    assert st == [0] * B
    for i in range(B):
        assert (Ts[i], Us[i], M[i], rs_m[i]) == singles[i][:4], i
        assert nxt(rands[i]) == singles[i][5], i
    coms = [s[:4] for s in singles]

    sp = []
    for i in range(B):
        r = pkg.Rand(pseeds[i])
        sp.append(single_prove(ctx, crs, insts[i], coms[i], r) + (nxt(r),))
    proofs, lens, pst, pnext = prove_batch(ctx, pkg, crs, insts, coms, pseeds)
    assert pst == [0] * B
    for i in range(B):
        assert proofs[i] == sp[i][0] and lens[i] == len(sp[i][0]) and pnext[i] == sp[i][2], i
    if golden:
        assert proofs[3].hex() == golden["proof"]


def mutated_cases(ctx, pkg, crs, insts, coms, proofs):
    """Valid instances interleaved with every mutation of test_gpu_protocol's golden and malformed-input tests."""
    ell = crs.ell
    cases = [(proof, inst[0], inst[1]) + com[:3] for inst, com, proof in zip(insts, coms, proofs)]
    p0, Rs, Ss, Ts, Us, M = cases[0]
    k = insts[0][3]
    p2 = pkg.Rand(5).generate_permutation(ell)
    perm_pts = lambda pts: b"".join(pts[96 * j:96 * j + 96] for j in p2)  # noqa: E731
    kM = ctx.g1_scalar_mul_affine(ctx.g1_batch_to_affine(M), k, broadcast=True)
    k2 = pkg.Rand(9).get_fr()
    flags, noncanon, flip = bytearray(p0), bytearray(p0), bytearray(p0)
    flags[0] |= 0xE0
    noncanon[-32:] = b"\xff" * 32
    flip[-1] ^= 1
    off = 48 * 9 + 32 + 48 * 2
    m = (ell + 4).bit_length() - 1
    assert int.from_bytes(p0[off:off + 4], "big") == m
    rounds = p0[:off] + (m - 1).to_bytes(4, "big") + p0[off + 4 + 48:]
    mutations = [
        (p0, Ss, Rs, Ts, Us, M),                                      # swap Rs / Ss
        (p0, Rs, Ss, perm_pts(Ts), perm_pts(Us), M),                  # re-permute Ts / Us
        (p0, Rs, Ss, Ts, Us, jac_enc(aff_dec(kM))),                   # M * k
        (p0, Rs, Ss, ctx.g1_scalar_mul_affine(Ts, k2, broadcast=True),
         ctx.g1_scalar_mul_affine(Us, k2, broadcast=True), M),        # rescale Ts / Us
        (p0, Rs, Ss, bytes(96) + Ts[96:], Us, M),                     # Ts[0] at infinity
        (p0[:-1], Rs, Ss, Ts, Us, M),                                 # truncated proof
        (bytes(flags), Rs, Ss, Ts, Us, M),                            # bad flag bits
        (bytes(noncanon), Rs, Ss, Ts, Us, M),                         # non-canonical scalar
        (bytes(flip), Rs, Ss, Ts, Us, M),                             # flipped scalar bit
        (rounds, Rs, Ss, Ts, Us, M),                                  # wrong round count
    ]
    out = []
    for i, c in enumerate(cases):
        out.append(c)
        if i < len(mutations):
            out.append(mutations[i])
    return out + mutations[len(cases):]


@pytest.mark.parametrize("mode", [1, 0])
def test_verify_equals_single_calls_on_a_mixed_batch(ctx, pkg, knobs, mode):
    ell, B = 12, 6
    crs = ctx.generate_crs(ell, pkg.Rand(0))
    insts = instances(ctx, pkg, ell, B, 200)
    coms = [single_commit(ctx, crs, insts[i], pkg.Rand(300 + i))[:4] for i in range(B)]
    proofs = [single_prove(ctx, crs, insts[i], coms[i], pkg.Rand(400 + i))[0] for i in range(B)]
    cases = mutated_cases(ctx, pkg, crs, insts, coms, proofs)
    seeds = [700 + i for i in range(len(cases))]
    want = []
    for c, s in zip(cases, seeds):
        r = pkg.Rand(s)
        want.append(single_verify(ctx, crs, c, r) + (nxt(r),))
    # every kind of outcome is present: valid, false, decode error, protocol error
    assert {w[:2] for w in want} >= {(1, 0), (0, 0), (0, DECODE), (0, PROTOCOL)}
    ctx.set_batch_verify_min(mode)
    ok, st, after = verify_batch(ctx, pkg, crs, cases, seeds)
    assert ok == [w[0] for w in want]
    assert st == [w[1] for w in want]
    assert after == [w[2] for w in want], "caller Rand positions differ"


def test_per_instance_failures(ctx, pkg):
    ell, B = 12, 5
    crs = ctx.generate_crs(ell, pkg.Rand(0))
    insts = instances(ctx, pkg, ell, B, 500)
    bad = list(insts)
    bad[1] = insts[1][:2] + ([ell] + insts[1][2][1:], insts[1][3])  # permutation entry out of range
    cseeds = [5100 + i for i in range(B)]
    Ts, Us, M, rs_m, st, after = commit_batch(ctx, pkg, crs, bad, cseeds)
    assert st == [0, INVALID_ARG, 0, 0, 0]
    assert after[1] == nxt(pkg.Rand(cseeds[1])), "a refused instance must not draw"
    assert Ts[1] == Us[1] == bytes(96 * ell) and M[1] == bytes(144) and rs_m[1] == bytes(128)
    good = commit_batch(ctx, pkg, crs, insts, cseeds)
    for i in (0, 2, 3, 4):
        assert (Ts[i], Us[i], M[i], rs_m[i], after[i]) == tuple(good[j][i] for j in (0, 1, 2, 3, 5))
    coms = [tuple(good[j][i] for j in range(4)) for i in range(B)]

    pseeds = [6100 + i for i in range(B)]
    ref, ref_lens, ref_st, ref_after = prove_batch(ctx, pkg, crs, insts, coms, pseeds)
    assert ref_st == [0] * B
    proofs, lens, pst, pafter = prove_batch(ctx, pkg, crs, bad, coms, pseeds)
    assert pst == [0, INVALID_ARG, 0, 0, 0]
    assert pafter[1] == nxt(pkg.Rand(pseeds[1]))
    for i in (0, 2, 3, 4):
        assert (proofs[i], pafter[i]) == (ref[i], ref_after[i])
    # a wrong rs_m breaks the witness: msm(G', d) != D, as the single call reports it
    wrong = list(coms)
    wrong[2] = coms[2][:3] + (coms[3][3],)
    proofs, lens, pst, pafter = prove_batch(ctx, pkg, crs, insts, wrong, pseeds)
    assert pst == [0, 0, PROTOCOL, 0, 0]
    assert "msm(G', d) != D" in ctx.lib.cdl_last_error(ctx.h).decode()
    r = pkg.Rand(pseeds[2])
    assert single_prove(ctx, crs, insts[2], wrong[2], r)[1] == PROTOCOL and nxt(r) == pafter[2]
    for i in (0, 1, 3, 4):
        assert proofs[i] == ref[i]
    # a proof buffer that is too small: the instance's error, with the length it needs
    proofs, lens, pst, pafter = prove_batch(ctx, pkg, crs, insts, coms, pseeds, proof_cap=100)
    assert pst == [INVALID_ARG] * B and lens == ref_lens and pafter == ref_after


def test_argument_errors(ctx, pkg):
    ell = 12
    crs = ctx.generate_crs(ell, pkg.Rand(0))
    insts = instances(ctx, pkg, ell, 2, 800)
    coms = [single_commit(ctx, crs, x, pkg.Rand(1))[:4] for x in insts]
    proofs = [single_prove(ctx, crs, x, c, pkg.Rand(2))[0] for x, c in zip(insts, coms)]
    for f, args in ((ctx.shuffle_permute_commit_batch, lambda rs: ([x[0] for x in insts], [x[1] for x in insts],
                                                                   [x[2] for x in insts], [x[3] for x in insts], rs)),
                    (ctx.prove_batch, lambda rs: ([x[0] for x in insts], [x[1] for x in insts], [c[0] for c in coms],
                                                  [c[1] for c in coms], [c[2] for c in coms], [x[2] for x in insts],
                                                  [x[3] for x in insts], [c[3] for c in coms], rs)),
                    (ctx.verify_batch, lambda rs: (proofs, [x[0] for x in insts], [x[1] for x in insts],
                                                   [c[0] for c in coms], [c[1] for c in coms], [c[2] for c in coms], rs))):
        with pytest.raises(pkg.CdlError) as ei:  # B == 0
            f(crs, *[[] for _ in args([])])
        assert ei.value.code == INVALID_ARG
    other = pkg.Context(0)
    try:
        ocrs = other.generate_crs(ell, pkg.Rand(0))
        with pytest.raises(pkg.CdlError) as ei:
            ctx.prove_batch(ocrs, [x[0] for x in insts], [x[1] for x in insts], [c[0] for c in coms], [c[1] for c in coms],
                            [c[2] for c in coms], [x[2] for x in insts], [x[3] for x in insts], [c[3] for c in coms],
                            [pkg.Rand(1), pkg.Rand(2)])
        assert ei.value.code == INVALID_ARG and "another context" in ei.value.msg
        with pytest.raises(pkg.CdlError) as ei:
            ctx.verify_batch(ocrs, proofs, [x[0] for x in insts], [x[1] for x in insts], [c[0] for c in coms],
                             [c[1] for c in coms], [c[2] for c in coms], [pkg.Rand(1), pkg.Rand(2)])
        assert ei.value.code == INVALID_ARG
        ocrs.close()
    finally:
        other.close()
    # null pointers, straight through the C ABI
    lib = ctx.lib
    r = pkg.Rand(3)
    rh = (C.c_void_p * 2)(r.h, r.h)
    perms = (C.c_uint32 * (2 * ell))()
    buf = C.create_string_buffer(2 * ell * 144 + 4096)
    st = (C.c_int32 * 2)()
    assert lib.cdl_shuffle_permute_commit_batch(ctx.h, crs.h, 2, None, buf, perms, buf, rh, buf, buf, buf, buf, st) == INVALID_ARG
    assert lib.cdl_shuffle_permute_commit_batch(ctx.h, crs.h, 2, buf, buf, perms, buf, (C.c_void_p * 2)(r.h, None), buf,
                                                buf, buf, buf, st) == INVALID_ARG
    lens = (C.c_size_t * 2)()
    assert lib.cdl_prove_batch(ctx.h, crs.h, 2, buf, buf, buf, buf, buf, perms, buf, buf, rh, None, 4096, lens, st) == INVALID_ARG
    ok = (C.c_int32 * 2)()
    assert lib.cdl_verify_batch(ctx.h, None, 2, buf, 16, lens, buf, buf, buf, buf, buf, rh, ok, st) == INVALID_ARG
    lens[0] = 17  # longer than the stride
    assert lib.cdl_verify_batch(ctx.h, crs.h, 2, buf, 16, lens, buf, buf, buf, buf, buf, rh, ok, st) == INVALID_ARG


def test_pool_index_bound(ctx, pkg, knobs):
    """A lane whose instances would need pool indices of 2^30 or more is refused before any instance is read."""
    ell = 12
    crs = ctx.generate_crs(ell, pkg.Rand(0))
    ctx.set_lanes(1)
    B = 1 << 22  # about 2^31 pool points at ell = 12
    r = pkg.Rand(1)
    rands = np.full(B, r.h.value, dtype=np.uint64)
    tiny = C.create_string_buffer(4096)
    perms = (C.c_uint32 * ell)()
    st = (C.c_int32 * 1)()
    rc = ctx.lib.cdl_shuffle_permute_commit_batch(ctx.h, crs.h, B, tiny, tiny, perms, tiny,
                                                  rands.ctypes.data_as(C.POINTER(C.c_void_p)), tiny, tiny, tiny, tiny, st)
    assert rc == TOO_LARGE
    assert "2^30" in ctx.lib.cdl_last_error(ctx.h).decode()


def test_lanes_give_the_same_results(ctx, pkg, knobs):
    ell, B = 124, 256
    crs = ctx.generate_crs(ell, pkg.Rand(0))
    insts = instances(ctx, pkg, ell, B, 900, point_sets=4)
    insts[17] = insts[17][:2] + ([ell] * ell, insts[17][3])  # one refused instance per run
    out = {}
    for lanes in (4, 1):
        ctx.set_lanes(lanes)
        c = commit_batch(ctx, pkg, crs, insts, [5200 + i for i in range(B)])
        coms = [tuple(c[j][i] for j in range(4)) for i in range(B)]
        p = prove_batch(ctx, pkg, crs, insts, coms, [6200 + i for i in range(B)])
        cases = [(p[0][i], insts[i][0], insts[i][1], coms[i][0], coms[i][1], coms[i][2]) for i in range(B)]
        cases[5] = (cases[5][0], cases[5][2], cases[5][1]) + cases[5][3:]  # a false verdict
        cases[17] = cases[16]
        v = verify_batch(ctx, pkg, crs, cases, [7200 + i for i in range(B)])
        out[lanes] = (c, p, v)
    c, p, v = out[1]
    assert c[4] == [0] * 17 + [INVALID_ARG] + [0] * (B - 18)
    assert v[0] == [0 if i == 5 else 1 for i in range(B)] and v[1] == [0] * B
    assert out[4] == out[1]


def test_shared_engine_keeps_whisk_results(ctx, pkg):
    ell, B = 12, 8
    crs = ctx.generate_crs(ell, pkg.Rand(0))
    pre = b"".join(make_trackers(ctx, pkg, ell, 1000 + i % 3) for i in range(B))

    def whisk():
        post, proofs, st = ctx.whisk_generate_shuffle_proof_batch(crs, pre, [pkg.Rand(3000 + i) for i in range(B)])
        ok, vst = ctx.whisk_is_valid_shuffle_proof_batch(crs, pre, bytes(post), bytes(proofs),
                                                         [pkg.Rand(2000 + i) for i in range(B)])
        return bytes(post), bytes(proofs), st, ok, vst

    first = whisk()
    assert first[2] == [0] * B and first[3] == [1] * B
    insts = instances(ctx, pkg, ell, B, 1100)
    c = commit_batch(ctx, pkg, crs, insts, [5300 + i for i in range(B)])
    coms = [tuple(c[j][i] for j in range(4)) for i in range(B)]
    p = prove_batch(ctx, pkg, crs, insts, coms, [6300 + i for i in range(B)])
    v = verify_batch(ctx, pkg, crs, [(p[0][i], insts[i][0], insts[i][1]) + coms[i][:3] for i in range(B)],
                     [7300 + i for i in range(B)])
    assert c[4] == p[2] == v[1] == [0] * B and v[0] == [1] * B
    assert whisk() == first
