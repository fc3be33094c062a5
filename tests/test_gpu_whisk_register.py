"""cdl_whisk_generate_registration_batch: a fresh tracker (rG, krG), the k-commitment kG and the tracker opening
proof for many validators in one call.  Its bytes, statuses and Rand positions must be those of the composition
through the existing entry points (draw r; r*G and k*G with cdl_g1_batch_scalar_mul_base; k*rG with
cdl_g1_scalar_mul_affine; cdl_whisk_generate_tracker_proof_batch), on either path of G's fixed-base
multiplication, whatever G's cache state and the context's device list."""
import ctypes as C
import os
import random
import re

import pytest

from oracle import bls12381 as b
from util import aff_enc, fr_dec, fr_enc, frs_enc

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INVALID, TOO_LARGE = -3, -6
GEN = aff_enc(b.G1_GEN)
MAX = 1 << 21  # CDL_WHISK_REGISTER_MAX
PER = 5  # scalars per validator: r, k r, k, blinder, blinder r


def _const(name):
    src = open(os.path.join(ROOT, "go-curdleproofs_b200", "csrc", "capi_base_mul.cu")).read()
    return int(re.search(name + r"\s*=\s*(\d+)", src).group(1))


X = _const("kBaseTableMinScalars")  # scalars from which a cold base_mul builds G's table
S = -(-_const("kBaseSlotScalars") // PER)  # validators per device slot of a split call


@pytest.fixture(scope="module")
def ref(pkg):
    """the one-device context the composition and the reference runs use"""
    c = pkg.Context(0)
    yield c
    c.close()


def _rands(pkg, B, seed):
    return [pkg.Rand(seed + i) for i in range(B)]


def _ks(B, seed):
    rnd = random.Random(seed)
    return frs_enc(rnd.randrange(b.R) for _ in range(B))


def _next(rands):
    return [r.get_fr() for r in rands]


def _diff(a, b_, size):
    """index of the first record of `size` bytes where a and b_ differ, or None"""
    if a == b_:
        return None
    if len(a) != len(b_):
        return "length"
    return next(i // size for i in range(0, len(a), size) if a[i:i + size] != b_[i:i + size])


def composition(c, ks, rands):
    """what a caller does without the call"""
    B = len(rands)
    rs = b"".join(r.get_fr() for r in rands)
    rG_aff, rG = c.g1_batch_scalar_mul_base(GEN, rs, affine=True, compressed=True)
    krG = c.g1_compress(c.g1_scalar_mul_affine(rG_aff, ks, broadcast=False))
    k_comms = c.g1_batch_scalar_mul_base(GEN, ks, affine=False, compressed=True)
    trackers = b"".join(rG[48 * i:48 * i + 48] + krG[48 * i:48 * i + 48] for i in range(B))
    proofs, status = c.whisk_generate_tracker_proof_batch(trackers, ks, rands)
    return trackers, k_comms, proofs, status


def assert_same(got, want):
    for name, size, g, w in zip(("trackers", "k_comms", "proofs"), (96, 48, 128), got[:3], want[:3]):
        assert _diff(g, w, size) is None, (name, _diff(g, w, size))
    assert got[3] == want[3]


def check_composition(pkg, c, ref, ks, seed):
    """c's registration of ks against ref's composition, with twin Rands; then the next draw of every Rand"""
    B = len(ks) // 32
    ra, rb = _rands(pkg, B, seed), _rands(pkg, B, seed)
    got = c.whisk_generate_registration_batch(ks, ra)
    assert got[3] == [0] * B
    assert_same(got, composition(ref, ks, rb))
    assert _next(ra) == _next(rb)
    return got


def _launches(c, fn):
    n0 = c.launch_count()
    out = fn()
    return out, c.launch_count() - n0


@pytest.mark.parametrize("B", [1, 5, 33, 6553, 6554, 20000])
def test_equals_composition(pkg, ref, B):
    """Byte equality with the five-call composition on a context that has no table of G: up to 6 553
    validators (32 765 scalars) the call runs G's multiplication on the GLV path, from 6 554 on it builds and
    uses G's table, which a following one-validator call then finds (1 launch instead of 4)."""
    c = pkg.Context(0)
    check_composition(pkg, c, ref, _ks(B, B), 100_000 + 30 * B)
    _, n = _launches(c, lambda: c.whisk_generate_registration_batch(_ks(1, 0), [pkg.Rand(1)]))
    assert n == (1 if PER * B >= X else 4)
    c.close()


def test_matches_oracle(pkg, ref):
    """The first 8 validators against the oracle's new_tracker and generate_whisk_tracker_proof (with an
    oracle Rand advanced past r); every validator of a 1 000-validator call is accepted by the oracle's
    is_valid_whisk_tracker_proof and by cdl_whisk_is_valid_tracker_proof_batch."""
    from oracle import protocol as P, whisk as W
    from oracle.cbackend import CBackend
    from oracle.rand import Rand as ORand

    B = 1000
    rnd = random.Random(77)
    kv = [rnd.randrange(b.R) for _ in range(B)]
    seeds = [5000 + i for i in range(B)]
    trackers, k_comms, proofs, status = ref.whisk_generate_registration_batch(frs_enc(kv), [pkg.Rand(s) for s in seeds])
    assert status == [0] * B
    P.set_backend(CBackend())
    try:
        for i in range(8):
            o = ORand(seeds[i])
            rG = b.g1_mul(b.G1_GEN, o.get_fr())
            tr = W.new_tracker(rG, b.g1_mul(rG, kv[i]))
            assert trackers[96 * i:96 * i + 96] == tr[0] + tr[1], i
            assert k_comms[48 * i:48 * i + 48] == b.g1_compress(b.g1_mul(b.G1_GEN, kv[i])), i
            assert proofs[128 * i:128 * i + 128] == W.generate_whisk_tracker_proof(tr, kv[i], o), i
        for i in range(B):
            tr = (trackers[96 * i:96 * i + 48], trackers[96 * i + 48:96 * i + 96])
            assert W.is_valid_whisk_tracker_proof(tr, k_comms[48 * i:48 * i + 48], proofs[128 * i:128 * i + 128]), i
    finally:
        P.set_backend(P.PyBackend())
    ok, st = ref.whisk_is_valid_tracker_proof_batch(trackers, k_comms, proofs)
    assert ok == [1] * B and st == [0] * B


def _edge_ks():
    """raw 32-byte secrets (gnark Montgomery limbs): k = 0, 1, q - 1, limbs >= q, duplicates"""
    R = b.R
    raw = [fr_enc(k) for k in (0, 1, R - 1, 2, (R - 1) // 2)]
    raw += [(R + i).to_bytes(32, "little") for i in (0, 1, 5)]
    raw += [(2 * R + 5).to_bytes(32, "little"), bytes([0xFF]) * 32, (1 << 255).to_bytes(32, "little")]
    raw += [raw[0], raw[1], raw[9], raw[9], raw[3]]
    return raw


@pytest.mark.parametrize("B", [16, 7000])
def test_scalar_edges(pkg, ref, B):
    """Edge secrets among B validators (GLV path at 16, table path at 7 000) equal the composition; the
    non-reduced limbs give the bytes of their reduced forms."""
    edge = _edge_ks()
    ks = b"".join(edge) + _ks(B - len(edge), 11)
    c = pkg.Context(0)
    got = check_composition(pkg, c, ref, ks, 200_000)
    reduced = b"".join(fr_enc(fr_dec(k)) for k in edge) + ks[32 * len(edge):]
    assert reduced != ks
    again = c.whisk_generate_registration_batch(reduced, _rands(pkg, B, 200_000))
    assert_same(again, got)
    c.close()


@pytest.mark.parametrize("B", [100, 7000])
def test_cache_states(pkg, ref, B):
    """The same bytes with G's table cold, warm, and evicted by four other bases in between."""
    c = pkg.Context(0)
    ks = _ks(B, 21)
    want = composition(ref, ks, _rands(pkg, B, 300_000))

    def run():
        rands = _rands(pkg, B, 300_000)
        got, n = _launches(c, lambda: c.whisk_generate_registration_batch(ks, rands))
        assert_same(got, want)
        return n

    assert run() == 4  # cold: GLV + compress at 100; check, window bases, table build and multiply at 7 000
    c.g1_batch_scalar_mul_base(GEN, bytes(32 * X), affine=False, compressed=True)
    assert run() == 1  # warm
    rnd = random.Random(B)
    for _ in range(4):
        c.g1_batch_scalar_mul_base(aff_enc(b.g1_mul(b.G1_GEN, rnd.randrange(1, b.R))), bytes(32 * X),
                                   affine=False, compressed=True)
    assert run() == 4  # evicted
    c.close()


def _device_count():
    import torch

    return torch.cuda.device_count()


@pytest.mark.parametrize("devices", [[0, 0], [0, 0, 0], "real"])
def test_multi_device(pkg, ref, devices):
    """A context over several device slots gives a one-device context's bytes, statuses and Rand positions
    around the split bounds (2 S and 3 S validators, S = ceil(kBaseSlotScalars / 5)), and the same class-1
    accounting (3 193 modmul per scalar)."""
    if devices == "real":
        n = _device_count()
        if n < 2:
            pytest.skip("one GPU")
        devices = list(range(min(n, 4)))
    m = pkg.Context(devices=devices)
    sizes = [2 * S - 1, 2 * S, 3 * S - 1, 3 * S + 1]
    m.engine_stats(reset=True)
    for B in sizes:
        ks = _ks(B, B + 1)
        ra, rb = _rands(pkg, B, 400_000), _rands(pkg, B, 400_000)
        got = m.whisk_generate_registration_batch(ks, ra)
        assert got[3] == [0] * B
        assert_same(got, ref.whisk_generate_registration_batch(ks, rb))
        assert _next(ra) == _next(rb)
    st = m.engine_stats()["elem_scalar_mul"]
    assert st["modmul"] == pytest.approx(3193.0 * PER * sum(sizes))
    for s in range(min(len(devices), 3)):
        assert m.engine_busy_ms_device(s) > 0, s  # 3 S + 1 validators use three slots
    m.close()


def test_arguments(pkg, ref):
    """Null pointers (also a null Rand) and B == 0 give CDL_ERR_INVALID_ARG, B > CDL_WHISK_REGISTER_MAX gives
    CDL_ERR_TOO_LARGE on a one- and a two-slot context; none of them draws from any Rand."""
    B = 3
    ks = _ks(B, 6)
    rands = _rands(pkg, B, 600)
    rh = (C.c_void_p * B)(*[r.h for r in rands])
    tr, kc, pr = C.create_string_buffer(96 * B), C.create_string_buffer(48 * B), C.create_string_buffer(128 * B)
    st = (C.c_int32 * B)()
    two = pkg.Context(devices=[0, 0])
    f = ref.lib.cdl_whisk_generate_registration_batch
    args = [ref.h, B, ks, rh, tr, kc, pr, st]
    for i in (0, 2, 3, 4, 5, 6, 7):
        bad = list(args)
        bad[i] = None
        assert f(*bad) == INVALID, i
    assert f(ref.h, 0, ks, rh, tr, kc, pr, st) == INVALID
    holes = (C.c_void_p * B)(rands[0].h, None, rands[2].h)
    assert f(ref.h, B, ks, holes, tr, kc, pr, st) == INVALID
    for c in (ref, two):
        assert f(c.h, MAX + 1, ks, rh, tr, kc, pr, st) == TOO_LARGE
        assert b"2^21" in ref.lib.cdl_last_error(c.h)
    assert tr.raw == bytes(96 * B) and list(st) == [0] * B
    assert _next(rands) == _next(_rands(pkg, B, 600))
    two.close()
