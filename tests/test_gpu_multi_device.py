"""Multi-device contexts (cdl_create_devices): the batched calls of a context over several device slots are
dealt to the slots in contiguous blocks, and every instance must come out as on a plain Context(0) with the
same seeds and the same lanes setting - the same post-trackers and proof bytes, verdicts, per-instance
statuses and the same next draw from every caller Rand.  The device list [0, 0] runs on one GPU with two
slots; the real-device tests use [0 .. min(device_count, 4)) and skip below 2 GPUs."""
import ctypes as C

import pytest

from oracle import bls12381 as b
from test_gpu_curdle_batch import commit_batch, instances, nxt, prove_batch, verify_batch
from test_gpu_parity_batch import KINDS, make_trackers, mutate
from test_gpu_whisk_match import _gpu_trackers
from util import aff_enc

pytestmark = pytest.mark.gpu

INVALID_ARG, DECODE = -3, -4


def _device_count():
    import torch

    return torch.cuda.device_count()


@pytest.fixture(scope="module")
def mctx(pkg):
    c = pkg.Context(devices=[0, 0])
    yield c
    c.close()


@pytest.fixture(params=["plain", "forced"])
def mode(request, ctx, mctx):
    """'forced': fixed-base tables and the combined verifier check on for every call, so that every slot
    builds its own CRS replica and tables."""
    on = request.param == "forced"
    for c in (ctx, mctx):
        c.set_fixed_base_min_batch(1 if on else -1)
        c.set_batch_verify_min(1 if on else -1)
    yield request.param
    for c in (ctx, mctx):
        c.set_fixed_base_min_batch(-1)
        c.set_batch_verify_min(-1)
        c.set_lanes(4)


def whisk_round_trip(c, pkg, crs, pre, B, ell, every=4):
    """Batched generate, then validate with every `every`-th instance mutated (all five kinds): every output,
    and the next draw of every caller Rand."""
    gr = [pkg.Rand(3000 + i) for i in range(B)]
    post, proofs, st = c.whisk_generate_shuffle_proof_batch(crs, pre, gr)
    tb = 96 * ell
    pres = [pre[i * tb:(i + 1) * tb] for i in range(B)]
    posts = [bytes(post[i * tb:(i + 1) * tb]) for i in range(B)]
    prfs = [bytes(proofs[i * 4576:(i + 1) * 4576]) for i in range(B)]
    for i in range(0, B, every):
        pres[i], posts[i], prfs[i] = mutate(c, pkg, (i // every) % KINDS, ell, pres[i], posts[i], prfs[i])
    vr = [pkg.Rand(2000 + i) for i in range(B)]
    ok, vst = c.whisk_is_valid_shuffle_proof_batch(crs, b"".join(pres), b"".join(posts), b"".join(prfs), vr)
    return bytes(post), bytes(proofs), st, ok, vst, [nxt(r) for r in gr], [nxt(r) for r in vr]


def curdle_batches(c, pkg, crs, insts, B):
    """commit / prove / verify batches with a permutation entry >= ell (instance 40), a proof that does not
    decode (instance 45) and a false verdict (instance 50)."""
    ell = crs.ell
    insts = list(insts)
    insts[40] = insts[40][:2] + ([ell] + insts[40][2][1:], insts[40][3])
    com = commit_batch(c, pkg, crs, insts, [5200 + i for i in range(B)])
    coms = [tuple(com[j][i] for j in range(4)) for i in range(B)]
    prv = prove_batch(c, pkg, crs, insts, coms, [6200 + i for i in range(B)])
    cases = [(prv[0][i], insts[i][0], insts[i][1], coms[i][0], coms[i][1], coms[i][2]) for i in range(B)]
    cases[40] = cases[39]
    cases[45] = (cases[45][0][:-1],) + cases[45][1:]
    cases[50] = (cases[50][0], cases[50][2], cases[50][1]) + cases[50][3:]
    ver = verify_batch(c, pkg, crs, cases, [7200 + i for i in range(B)])
    return com, prv, ver


def tracker_proofs(c, pkg, trackers, ks, B):
    gr = [pkg.Rand(8000 + i) for i in range(B)]
    proofs, st = c.whisk_generate_tracker_proof_batch(trackers, ks, gr)
    k_comms = c.g1_compress(c.g1_scalar_mul_affine(aff_enc(b.G1_GEN) * B, ks, broadcast=False))
    bad = bytearray(proofs)
    bad[128 * 3 + 127] ^= 1  # a wrong s: a false verdict
    ok, vst = c.whisk_is_valid_tracker_proof_batch(trackers, k_comms, bytes(bad))
    return proofs, st, [nxt(r) for r in gr], ok, vst


def tracker_set(c, pkg, B, malformed=70):
    r = pkg.Rand(77)
    rs, ks = r.get_frs(B), r.get_frs(B)
    tr = bytearray(_gpu_trackers(c, rs, ks))
    if malformed is not None:
        tr[96 * malformed] |= 0x40  # infinity flag on a finite point: does not decode
    return bytes(tr), ks


def match_set(c, pkg, T, V):
    kb = pkg.Rand(90).get_frs(V + 40)
    owners = [kb[32 * ((t * 7 + 3) % (V + 40)):][:32] for t in range(T)]
    tr = bytearray(_gpu_trackers(c, pkg.Rand(91).get_frs(T), b"".join(owners)))
    tr[96 * (T - 2)] |= 0x40
    return bytes(tr), kb[:32 * V]


def compare_all(pkg, a, m, ell, B):
    """Whisk round trips, curdleproof batches, tracker proofs and matching on contexts a and m."""
    crs_a, crs_m = a.generate_crs(ell, pkg.Rand(0)), m.generate_crs(ell, pkg.Rand(0))
    assert crs_a.export() == crs_m.export()
    pre = b"".join(make_trackers(a, pkg, ell, 1000 + i % 3) for i in range(B))
    wa, wm = whisk_round_trip(a, pkg, crs_a, pre, B, ell), whisk_round_trip(m, pkg, crs_m, pre, B, ell)
    assert wa[2] == [0] * B and 0 < sum(wa[3]) < B and set(wa[4]) >= {0, -5}
    assert wm == wa
    insts = instances(a, pkg, ell, B, 900, point_sets=4)
    ca, cm = curdle_batches(a, pkg, crs_a, insts, B), curdle_batches(m, pkg, crs_m, insts, B)
    assert ca[0][4][40] == INVALID_ARG and ca[2][1][45] == DECODE and ca[2][0][50] == 0 and ca[2][0][0] == 1
    assert cm == ca
    crs_a.close()
    crs_m.close()


def test_whisk_equals_one_device(pkg, ctx, mctx, mode):
    for ell, B in ((124, 130), (12, 70)):
        crs_a, crs_m = ctx.generate_crs(ell, pkg.Rand(0)), mctx.generate_crs(ell, pkg.Rand(0))
        pre = b"".join(make_trackers(ctx, pkg, ell, 1000 + i % 3) for i in range(B))
        want = whisk_round_trip(ctx, pkg, crs_a, pre, B, ell)
        assert want[2] == [0] * B and 0 < sum(want[3]) < B
        assert set(want[4]) >= {0, -5}
        assert whisk_round_trip(mctx, pkg, crs_m, pre, B, ell) == want, (ell, B)
        crs_a.close()
        crs_m.close()


def test_curdle_batches_equal_one_device(pkg, ctx, mctx, mode):
    ell, B = 12, 70
    crs_a, crs_m = ctx.generate_crs(ell, pkg.Rand(0)), mctx.generate_crs(ell, pkg.Rand(0))
    insts = instances(ctx, pkg, ell, B, 900, point_sets=4)
    want = curdle_batches(ctx, pkg, crs_a, insts, B)
    com, prv, ver = want
    assert com[4] == [0] * 40 + [INVALID_ARG] + [0] * (B - 41)
    assert prv[2][40] == INVALID_ARG and ver[1][45] == DECODE and ver[0][50] == 0
    assert ver[0].count(1) == B - 2
    assert curdle_batches(mctx, pkg, crs_m, insts, B) == want


def test_tracker_proofs_equal_one_device(pkg, ctx, mctx, mode):
    B = 100
    trackers, ks = tracker_set(ctx, pkg, B)
    want = tracker_proofs(ctx, pkg, trackers, ks, B)
    assert want[1] == [0] * 70 + [DECODE] + [0] * 29
    assert want[3] == [0 if i in (3, 70) else 1 for i in range(B)] and want[4][70] == DECODE
    assert tracker_proofs(mctx, pkg, trackers, ks, B) == want


@pytest.mark.parametrize("T", [300, 1000])
@pytest.mark.parametrize("V", [6, 300])
def test_matching_equals_one_device(pkg, ctx, mctx, mode, T, V):
    """T = 300: slots take [0, 256) and [256, 300); T = 1000: [0, 512) and [512, 1000).  V = 300 takes the
    table path, V = 6 the shared-scalar one."""
    trackers, ks = match_set(ctx, pkg, T, V)
    want = ctx.whisk_match_trackers(trackers, ks)
    assert want[1][T - 2] == DECODE and 0 < sum(o >= 0 for o in want[0]) < T
    mctx.engine_stats(reset=True)
    assert mctx.whisk_match_trackers(trackers, ks) == want
    assert mctx.engine_busy_ms_device(0) > 0 and mctx.engine_busy_ms_device(1) > 0


def test_small_batches_stay_on_slot_0(pkg, ctx, mctx):
    """B < 32 * D and B = 1 run on slot 0 alone, with the same results."""
    ell = 12
    crs_a, crs_m = ctx.generate_crs(ell, pkg.Rand(0)), mctx.generate_crs(ell, pkg.Rand(0))
    for B in (40, 1):
        pre = b"".join(make_trackers(ctx, pkg, ell, 1000 + i % 3) for i in range(B))
        want = whisk_round_trip(ctx, pkg, crs_a, pre, B, ell)
        mctx.engine_stats(reset=True)
        assert whisk_round_trip(mctx, pkg, crs_m, pre, B, ell) == want, B
        assert mctx.engine_busy_ms_device(0) > 0 and mctx.engine_busy_ms_device(1) == 0, B
    single = ctx.whisk_generate_shuffle_proof(crs_a, pre, pkg.Rand(5))
    assert mctx.whisk_generate_shuffle_proof(crs_m, pre, pkg.Rand(5)) == single


def test_crs_ownership(pkg, ctx, mctx):
    """One CRS of the multi-device context serves all of its slots (the tests above); a CRS of another
    context is refused on the split path too."""
    ell, B = 12, 70
    crs_a, crs_m = ctx.generate_crs(ell, pkg.Rand(0)), mctx.generate_crs(ell, pkg.Rand(0))
    pre = make_trackers(ctx, pkg, ell, 1000) * B
    for c, crs in ((mctx, crs_a), (ctx, crs_m)):
        for n in (B, 1):
            with pytest.raises(pkg.CdlError) as ei:
                c.whisk_generate_shuffle_proof_batch(crs, pre[:96 * ell * n], [pkg.Rand(i) for i in range(n)])
            assert ei.value.code == INVALID_ARG and "another context" in ei.value.msg
    crs_a.close()
    crs_m.close()


def test_round_trips_around_a_match_call(pkg, mctx):
    """Matching overwrites the start of every slot's engine pool; Whisk round trips before and after it stay
    byte-identical."""
    ell, B = 12, 96
    crs = mctx.generate_crs(ell, pkg.Rand(0))
    pre = b"".join(make_trackers(mctx, pkg, ell, 1000 + i % 3) for i in range(B))
    first = whisk_round_trip(mctx, pkg, crs, pre, B, ell)
    trackers, ks = match_set(mctx, pkg, 1000, 300)
    mctx.whisk_match_trackers(trackers, ks)
    assert whisk_round_trip(mctx, pkg, crs, pre, B, ell) == first
    crs.close()


def test_accounting(pkg, ctx, mctx):
    """cdl_launch_count sums over slots: a split call launches what its two blocks launch as calls of their
    own on one device; every slot that received work reports busy time; the device list reads back."""
    assert mctx.devices() == [0, 0] and ctx.devices() == [0]
    ell, B = 12, 70
    crs_a, crs_m = ctx.generate_crs(ell, pkg.Rand(0)), mctx.generate_crs(ell, pkg.Rand(0))
    tb = 96 * ell
    pre = b"".join(make_trackers(ctx, pkg, ell, 1000 + i % 3) for i in range(B))
    n0 = ctx.launch_count()
    for lo, hi in ((0, 35), (35, 70)):
        ctx.whisk_generate_shuffle_proof_batch(crs_a, pre[lo * tb:hi * tb], [pkg.Rand(3000 + i) for i in range(lo, hi)])
    per_block = ctx.launch_count() - n0
    mctx.engine_stats(reset=True)
    n0 = mctx.launch_count()
    mctx.whisk_generate_shuffle_proof_batch(crs_m, pre, [pkg.Rand(3000 + i) for i in range(B)])
    assert mctx.launch_count() - n0 == per_block
    busy = [mctx.engine_busy_ms_device(s) for s in range(2)]
    assert all(x > 0 for x in busy)
    assert mctx.engine_busy_ms() == max(busy)
    assert sum(v["launches"] for v in mctx.engine_stats().values()) > 0
    crs_a.close()
    crs_m.close()


def test_argument_errors(pkg, ctx, mctx):
    lib = ctx.lib
    h = C.c_void_p()

    def create(devs):
        return lib.cdl_create_devices((C.c_int32 * max(1, len(devs)))(*devs), len(devs), C.byref(h))

    assert create([]) == INVALID_ARG
    assert create([0] * 17) == INVALID_ARG
    assert create([0, _device_count()]) == INVALID_ARG
    assert create([-1]) == INVALID_ARG
    assert lib.cdl_create_devices(None, 1, C.byref(h)) == INVALID_ARG
    with pytest.raises(pkg.CdlError) as ei:
        pkg.Context(devices=[])
    assert ei.value.code == INVALID_ARG
    rc = lib.cdl_comm_init(mctx.h, bytes(128), 0, 1)
    assert rc == INVALID_ARG and "slots" in lib.cdl_last_error(mctx.h).decode()
    with pytest.raises(pkg.CdlError) as ei:
        mctx.engine_busy_ms_device(2)
    assert ei.value.code == INVALID_ARG
    n = C.c_size_t()
    assert lib.cdl_context_devices(mctx.h, None, 1, C.byref(n)) == INVALID_ARG
    assert lib.cdl_context_devices(mctx.h, None, 0, C.byref(n)) == 0 and n.value == 2
    # a full-size list of 16 slots is accepted
    c16 = pkg.Context(devices=[0] * 16)
    assert c16.devices() == [0] * 16
    c16.close()


def test_real_devices(pkg, ctx):
    """Whisk, curdleproof and matching comparisons on the GPUs of the box (at most 4)."""
    D = min(_device_count(), 4)
    if D < 2:
        pytest.skip("needs >= 2 GPUs")
    m = pkg.Context(devices=list(range(D)))
    try:
        assert m.devices() == list(range(D))
        compare_all(pkg, ctx, m, 12, 32 * D + 10)
        compare_all(pkg, ctx, m, 124, 64 * D)
        trackers, ks = tracker_set(ctx, pkg, 40 * D)
        assert tracker_proofs(m, pkg, trackers, ks, 40 * D) == tracker_proofs(ctx, pkg, trackers, ks, 40 * D)
        trackers, ks = match_set(ctx, pkg, 300 * D + 7, 300)
        m.engine_stats(reset=True)
        assert m.whisk_match_trackers(trackers, ks) == ctx.whisk_match_trackers(trackers, ks)
        assert all(m.engine_busy_ms_device(s) > 0 for s in range(D))
    finally:
        m.close()
