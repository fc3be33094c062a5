"""The elementwise point calls and cdl_g1_msm_batch on a multi-device context.  From 2 * kMin units (each call's own
minimum block, read from capi.cu) a call is dealt to the device slots in contiguous blocks, each run on lane 0 of
its slot; below that it runs unsplit.  Return code, output bytes, status bytes and the cdl_last_error text must
equal those of the one-device context `ctx` for every input.  [0, 0] and [0, 0, 0] run two and three slots on one
GPU (three slots give unequal blocks); the real-device context uses [0 .. min(device_count, 4)) and skips below 2
GPUs."""
import ctypes as C
import os
import random
import re

import pytest

from oracle import bls12381 as b
from util import R, aff_enc, frs_enc

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "go-curdleproofs_b200", "csrc")
INVALID, DECODE = -3, -4
GEN = aff_enc(b.G1_GEN)
SET = 4096  # distinct points of the inputs, repeated to size


def _const(name):
    src = open(os.path.join(CSRC, "capi.cu")).read()
    return int(re.search(name + r"\s*=\s*(\d+)", src).group(1))


K_DEC = _const("kDecompressSlotPoints")
K_CMP = _const("kCompressSlotPoints")
K_AFF = _const("kToAffineSlotPoints")
K_MUL = _const("kScalarMulSlotPoints")
K_FOLD = _const("kFoldSlotPoints")
K_MSM = _const("kMsmBatchSlotTerms")


def sizes(k):
    """just below two blocks, two equal blocks, and an odd size that gives [0, 0, 0] three unequal blocks"""
    return (2 * k - 1, 2 * k, 3 * k + 7)


def shard_lo(n, D, s):
    return s * (n // D) + min(s, n % D)


def _device_count():
    import torch

    return torch.cuda.device_count()


@pytest.fixture(scope="module", params=["0,0", "0,0,0", "real"])
def multi(request, pkg):
    if request.param == "real":
        D = min(_device_count(), 4)
        if D < 2:
            pytest.skip("needs >= 2 GPUs")
        devs = list(range(D))
    else:
        devs = [int(d) for d in request.param.split(",")]
    c = pkg.Context(devices=devs)
    c.n_slots = len(devs)
    yield c
    c.close()


@pytest.fixture(scope="module")
def base(ctx):
    """SET points a_i * G with every 97th the point at infinity, their encodings, Jacobian forms with Z != 1
    (infinity as gnark's (1, 1, 0)) and scalars: zero, one, r - 1, limbs >= r and random"""
    rnd = random.Random(17)
    a = [rnd.randrange(1, R) for _ in range(SET)]
    pts = bytearray(ctx.g1_scalar_mul_affine(GEN * SET, frs_enc(a), broadcast=False))
    for i in range(0, SET, 97):
        pts[96 * i:96 * i + 96] = bytes(96)
    pts = bytes(pts)
    enc = ctx.g1_compress(pts)
    P, Rm = b.P, pow(2, 384, b.P)
    jac = bytearray()
    for i in range(SET):
        x = int.from_bytes(pts[96 * i:96 * i + 48], "little")
        y = int.from_bytes(pts[96 * i + 48:96 * i + 96], "little")
        if x == 0 and y == 0:
            jac += Rm.to_bytes(48, "little") * 2 + bytes(48)
            continue
        z = rnd.randrange(1, P)
        z2 = z * z % P
        jac += (x * z2 % P).to_bytes(48, "little") + (y * z2 * z % P).to_bytes(48, "little") + \
            (z * Rm % P).to_bytes(48, "little")
    sc = bytearray(rnd.randbytes(32 * SET))  # raw limbs: many above r
    sc[0:32] = bytes(32)
    sc[32:64] = frs_enc([1])
    sc[64:96] = frs_enc([R - 1])
    sc[96:128] = b"\xff" * 32
    for i in range(5, SET, 61):
        sc[32 * i:32 * i + 32] = bytes(32)
    return pts, enc, bytes(jac), bytes(sc)


def rep(data, unit, n, shift=0):
    """n units of `unit` bytes: the SET units of data rotated by `shift`, repeated"""
    d = data[unit * shift:] + data[:unit * shift]
    return (d * -(-n // SET))[:unit * n]


def _err(c, rc):
    return c.lib.cdl_last_error(c.h) if rc else None


def decompress(c, enc):
    n = len(enc) // 48
    out = C.create_string_buffer(b"\xa5" * (96 * n), 96 * n)
    st = C.create_string_buffer(b"\x5a" * n, n)
    rc = c.lib.cdl_g1_decompress(c.h, enc, n, out, st)
    return rc, _err(c, rc), out.raw, st.raw


def compress(c, pts):
    n = len(pts) // 96
    out = C.create_string_buffer(b"\xa5" * (48 * n), 48 * n)
    rc = c.lib.cdl_g1_compress(c.h, pts, n, out)
    return rc, _err(c, rc), out.raw


def to_affine(c, jac):
    n = len(jac) // 144
    out = C.create_string_buffer(b"\xa5" * (96 * n), 96 * n)
    rc = c.lib.cdl_g1_batch_to_affine(c.h, jac, n, out)
    return rc, _err(c, rc), out.raw


def scalar_mul(c, pts, sc, stride):
    n = len(pts) // 96
    out = C.create_string_buffer(b"\xa5" * (96 * n), 96 * n)
    rc = c.lib.cdl_g1_scalar_mul_affine(c.h, pts, sc, n, stride, out)
    return rc, _err(c, rc), out.raw


def fold(c, L, R_, x):
    n = len(L) // 96
    buf = C.create_string_buffer(L, len(L))
    rc = c.lib.cdl_g1_fold(c.h, buf, R_, x, n)
    return rc, _err(c, rc), buf.raw


def msm_batch(c, pts, sc, offsets):
    k = len(offsets) - 1
    offs = (C.c_uint32 * (k + 1))(*offsets)
    out = C.create_string_buffer(b"\xa5" * (96 * k), 96 * k)
    rc = c.lib.cdl_g1_msm_batch(c.h, pts, sc, offs, k, out)
    return rc, _err(c, rc), out.raw


# ------------------------------------------------------------------------------------------------- codecs
def test_compress(ctx, multi, base):
    pts = base[0]
    for n in sizes(K_CMP):
        p = rep(pts, 96, n, n % SET)
        want = compress(ctx, p)
        assert want[0] == 0
        assert compress(multi, p) == want, n


def test_batch_to_affine(ctx, multi, base):
    pts, jac = base[0], base[2]
    for n in sizes(K_AFF):
        want = to_affine(ctx, rep(jac, 144, n, 3))
        assert want[0] == 0 and want[2] == rep(pts, 96, n, 3)
        assert to_affine(multi, rep(jac, 144, n, 3)) == want, n


def _rejects():
    """one encoding per reason code 1 .. 5"""
    good = b.g1_compress(b.G1_GEN)
    bad_flags = bytes([good[0] | 0x60]) + good[1:]
    x_ge_p = bytes([0x9F]) + b"\xff" * 47
    x = 1
    while b.fp_sqrt((x ** 3 + 4) % b.P) is not None:
        x += 1
    non_res = bytearray(x.to_bytes(48, "big"))
    non_res[0] |= 0x80
    x = 1
    while True:
        y = b.fp_sqrt((x ** 3 + 4) % b.P)
        if y is not None and not b.g1_in_subgroup((x, y)):
            break
        x += 1
    not_sub = b.g1_compress((x, y))
    dirty_inf = bytes([0xC0]) + bytes(46) + b"\x01"
    return {1: bad_flags, 2: x_ge_p, 3: bytes(non_res), 4: not_sub, 5: dirty_inf}


def test_decompress_valid(ctx, multi, base):
    pts, enc = base[0], base[1]
    for n in sizes(K_DEC):
        e = rep(enc, 48, n, 5)
        want = decompress(ctx, e)
        assert want[0] == 0 and want[2] == rep(pts, 96, n, 5) and want[3] == bytes(n)
        assert decompress(multi, e) == want, n


def test_decompress_rejects(ctx, multi, base):
    """rejects of every reason in the first, a middle and the last block and on block boundaries: every block
    writes all of its points and statuses, and the message names the call's first rejected point"""
    enc = base[1]
    bad = _rejects()
    for n in sizes(K_DEC):
        D = max(1, min(multi.n_slots, n // K_DEC))
        starts = [shard_lo(n, D, s) for s in range(D)]
        e0 = bytearray(rep(enc, 48, n, 11))
        places = {
            "first block": [7],
            "middle block": [starts[D // 2] + 3],
            "last block": [n - 1],
            "block boundaries": [s for s in starts[1:]] + [s - 1 for s in starts[1:]] or [n // 2],
            "every block": [s + 1 for s in starts] + [n - 2],
        }
        for where, idx in places.items():
            for why, enc_bad in bad.items():
                e = bytearray(e0)
                for i in idx:
                    e[48 * i:48 * i + 48] = enc_bad
                want = decompress(ctx, bytes(e))
                assert want[0] == DECODE and f"point {min(idx)} rejected (reason {why})".encode() in want[1]
                assert decompress(multi, bytes(e)) == want, (n, where, why)
        # five different reasons in five places: the first one is reported
        e = bytearray(e0)
        for why, i in zip(sorted(bad), (n - 1, starts[-1], n // 2, 1, 0)):
            e[48 * i:48 * i + 48] = bad[why]
        want = decompress(ctx, bytes(e))
        assert b"point 0 rejected (reason 5)" in want[1]
        assert decompress(multi, bytes(e)) == want, n


# ------------------------------------------------------------------------------------------------- elementwise
def test_scalar_mul_per_point(ctx, multi, base):
    pts, sc = base[0], base[3]
    for n in sizes(K_MUL):
        p, s = rep(pts, 96, n, 1), rep(sc, 32, n, n % SET)
        want = scalar_mul(ctx, p, s, 1)
        assert want[0] == 0
        assert scalar_mul(multi, p, s, 1) == want, n


def test_scalar_mul_broadcast(ctx, multi, base):
    """one scalar for every block: random, zero, and limbs >= r"""
    pts, sc = base[0], base[3]
    for n in sizes(K_MUL):
        p = rep(pts, 96, n, 2)
        for s in (sc[32 * 200:32 * 201], bytes(32), b"\xff" * 32):
            want = scalar_mul(ctx, p, s, 0)
            assert want[0] == 0
            assert scalar_mul(multi, p, s, 0) == want, n


def test_fold(ctx, multi, base):
    pts, sc = base[0], base[3]
    for n in sizes(K_FOLD):
        L, R_ = rep(pts, 96, n, 4), rep(pts, 96, n, 9)
        for x in (sc[32 * 300:32 * 301], bytes(32), b"\xff" * 32):
            want = fold(ctx, L, R_, x)
            assert want[0] == 0
            assert fold(multi, L, R_, x) == want, n
        # L and R with the same contents: L + x L
        want = fold(ctx, L, L, sc[32 * 301:32 * 302])
        assert fold(multi, L, L, sc[32 * 301:32 * 302]) == want, n


def test_split_uses_lane_buffers(pkg):
    """Evidence that a call of N >= 2 * kMin units splits on [0, 0]: after cdl_fp_mul has grown the root context's
    input and output buffers beyond what the call needs, the call still takes at least N units' worth of new device
    memory, because both blocks run on lane buffers of their own (which persist until the context is destroyed).
    Unsplit, it would grow at most the root's status (decompress) or addend (fold) buffer."""
    import torch

    pts = GEN * SET
    jac = (GEN + pow(2, 384, b.P).to_bytes(48, "little")) * SET
    enc = b.g1_compress(b.G1_GEN) * SET
    cases = [("compress", K_CMP, 96 + 48, lambda c, n: compress(c, rep(pts, 96, n))),
             ("batch_to_affine", K_AFF, 144 + 96, lambda c, n: to_affine(c, rep(jac, 144, n))),
             ("decompress", K_DEC, 48 + 96 + 1, lambda c, n: decompress(c, rep(enc, 48, n))),
             ("scalar_mul", K_MUL, 96 + 32 + 96, lambda c, n: scalar_mul(c, rep(pts, 96, n), bytes(32 * n), 1)),
             ("fold", K_FOLD, 96 + 96 + 96, lambda c, n: fold(c, rep(pts, 96, n), rep(pts, 96, n), bytes(32)))]
    torch.cuda.mem_get_info(0)
    for name, k, per, fn in cases:
        n = max(2 * k, 1 << 18)
        fp = pow(2, 384, b.P).to_bytes(48, "little") * (3 * n)  # 144 bytes per unit in each root buffer
        m = pkg.Context(devices=[0, 0])
        try:
            m.fp_mul(fp, fp)
            free0 = torch.cuda.mem_get_info(0)[0]
            assert fn(m, n)[0] == 0
            free1 = torch.cuda.mem_get_info(0)[0]
            assert free0 - free1 >= n * per, (name, free0, free1)
        finally:
            m.close()


# ------------------------------------------------------------------------------------------------- MSM batch
@pytest.fixture(scope="module")
def msm_vec(ctx):
    """3 * kMsmBatchSlotTerms + 64 points a_i * G (a few at infinity) and scalars (zeros and limbs >= r)"""
    n = 3 * K_MSM + 64
    rnd = random.Random(23)
    a = [rnd.randrange(1, R) for _ in range(SET)]
    pts = bytearray(ctx.g1_scalar_mul_affine(GEN * SET, frs_enc(a), broadcast=False))
    for i in range(0, SET, 101):
        pts[96 * i:96 * i + 96] = bytes(96)
    sc = bytearray(rnd.randbytes(32 * n))
    for i in range(0, n, 53):
        sc[32 * i:32 * i + 32] = bytes(32)
    return rep(bytes(pts), 96, n, 0), bytes(sc)


def msm_cuts(offsets, D):
    """the MSM blocks capi.cu's msm_batch_cuts gives, or None when the call does not split"""
    k = len(offsets) - 1
    first, terms = offsets[0], offsets[k] - offsets[0]
    Dp = max(1, min(D, terms // K_MSM))
    cut = [0]
    for s in range(1, Dp):
        t = first + shard_lo(terms, Dp, s)
        j = next(j for j in range(k + 1) if offsets[j] >= t)
        v = offsets[j - 1] if j > 0 and t - offsets[j - 1] < offsets[j] - t else offsets[j]
        cut.append(k if v == offsets[k] else offsets.index(v))
    cut.append(k)
    busy = sum(offsets[cut[s]] > offsets[cut[s - 1]] for s in range(1, len(cut)))
    return cut if busy >= 2 else None


def _offsets(sizes_):
    offs = [0]
    for s in sizes_:
        offs.append(offs[-1] + s)
    return offs


def _msm_shapes(total):
    """MSM size lists of `total` terms: many mixed sizes with empty MSMs, one large MSM among small ones,
    leading and trailing empty MSMs"""
    rnd = random.Random(total)
    mixed = []
    left = total
    while left:
        s = min(left, rnd.choice([0, 0, 1, 2, 7, 64, 300, 1000, 5000, 20000]))
        mixed.append(s)
        left -= s
    big = [3, 0, 5] + [total - 8 - 40 * 9] + [9] * 40
    edges = [0, 0] + [total // 3, 0, total // 3, total - 2 * (total // 3)] + [0, 0, 0]
    return {"mixed": mixed, "one large": big, "empty ends": edges}


def test_msm_batch_sizes(ctx, multi, msm_vec):
    pts, sc = msm_vec
    for total in sizes(K_MSM):
        for shape, ss in _msm_shapes(total).items():
            offs = _offsets(ss)
            assert offs[-1] == total
            want = msm_batch(ctx, pts[:96 * total], sc[:32 * total], offs)
            assert want[0] == 0
            assert msm_batch(multi, pts[:96 * total], sc[:32 * total], offs) == want, (total, shape)


def test_msm_batch_offset_base(ctx, multi, msm_vec):
    """offsets[0] > 0: the terms before it belong to no MSM, in both forms"""
    pts, sc = msm_vec
    n = 3 * K_MSM + 7
    offs = [50, 60, 60 + K_MSM, 60 + 2 * K_MSM, n]
    want = msm_batch(ctx, pts[:96 * n], sc[:32 * n], offs)
    assert want[0] == 0
    assert msm_batch(multi, pts[:96 * n], sc[:32 * n], offs) == want


def test_msm_batch_single_msm_does_not_split(pkg, ctx, msm_vec):
    """every term in one MSM (alone or among empty ones): only slot 0 works, as on a one-device context"""
    pts, sc = msm_vec
    n = 3 * K_MSM
    m = pkg.Context(devices=[0, 0, 0])
    try:
        for offs in ([0, n], [0, 0, n, n, n], [0, 0, 0, n]):
            m.engine_stats(reset=True)
            n0, c0 = m.launch_count(), ctx.launch_count()
            want = msm_batch(ctx, pts[:96 * n], sc[:32 * n], offs)
            assert msm_batch(m, pts[:96 * n], sc[:32 * n], offs) == want
            assert m.launch_count() - n0 == ctx.launch_count() - c0
            assert m.engine_busy_ms_device(0) > 0
            assert m.engine_busy_ms_device(1) == 0 and m.engine_busy_ms_device(2) == 0
            assert msm_cuts(offs, 3) is None
    finally:
        m.close()


def test_msm_batch_accounting(pkg, ctx, msm_vec):
    """launches and class statistics of a split call are the sum over its blocks run alone"""
    pts, sc = msm_vec
    total = 3 * K_MSM + 7
    offs = _offsets(_msm_shapes(total)["mixed"])
    cut = msm_cuts(offs, 3)
    assert cut is not None and len(cut) == 4
    m = pkg.Context(devices=[0, 0, 0])
    try:
        msm_batch(m, pts[:96 * total], sc[:32 * total], offs)  # the lanes exist from here on
        m.engine_stats(reset=True)
        n0 = m.launch_count()
        got = msm_batch(m, pts[:96 * total], sc[:32 * total], offs)
        k = m.launch_count() - n0
        st = m.engine_stats()
        assert all(m.engine_busy_ms_device(s) > 0 for s in range(3))
        ctx.engine_stats(reset=True)
        c0 = ctx.launch_count()
        parts = []
        for j0, j1 in zip(cut, cut[1:]):
            o = [x - offs[j0] for x in offs[j0:j1 + 1]]
            r = msm_batch(ctx, pts[96 * offs[j0]:96 * offs[j1]], sc[32 * offs[j0]:32 * offs[j1]], o)
            assert r[0] == 0
            parts.append(r[2])
        assert got[0] == 0 and got[2] == b"".join(parts)
        assert k == ctx.launch_count() - c0
        want = ctx.engine_stats()
        for cls, v in st.items():
            assert v["launches"] == want[cls]["launches"], cls
            assert v["modmul"] == pytest.approx(want[cls]["modmul"]), cls
    finally:
        m.close()


def test_msm_batch_refusals(ctx, multi):
    """non-monotone offsets and a call over the 2^30-point pool: the one-device status and message, nothing
    written (the offsets claim terms the buffers do not hold: the checks run before any input is read)"""
    pts, sc = bytes(96), bytes(32)
    n = 3 * K_MSM
    for offs in ([0, n, K_MSM, n], [0, 2 * K_MSM, K_MSM, 3 * K_MSM + 1],
                 [0, 1 << 29, (1 << 29) + (1 << 28), 1 << 30], [0, K_MSM, (1 << 30) - 2]):
        want = msm_batch(ctx, pts, sc, offs)
        assert want[0] == INVALID and want[2] == b"\xa5" * (96 * (len(offs) - 1))
        assert msm_batch(multi, pts, sc, offs) == want, offs
