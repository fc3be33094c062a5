"""The library's scratch buffers: a refused allocation leaves no error behind for the next call, and the
buffers of the host-pointer calls and of the protocol engine grow and are then reused with correct results."""
import random

import pytest

from oracle import bls12381 as b
from oracle import protocol as P, whisk as W
from oracle.cbackend import CBackend
from oracle.rand import Rand
from util import P as FP, R, affs_dec, affs_enc, fp_dec, fp_enc, fr_enc, frs_enc, jac_enc

pytestmark = pytest.mark.gpu


@pytest.fixture
def fresh(pkg):
    """A context of its own: its buffers start empty."""
    c = pkg.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def cb():
    return CBackend(accelerate_keccak=False)


def test_refused_allocation_does_not_fail_the_next_call(fresh, pkg):
    import torch

    too_big = 2 * torch.cuda.get_device_properties(0).total_memory
    with pytest.raises(pkg.CdlError):
        fresh.dev_buffer(too_big)
    # same context, same thread: the refused cudaMalloc must not surface as this call's error
    pts = Rand(7).get_g1_affines(3) + [None]
    assert fresh.g1_compress(affs_enc(pts)) == b"".join(b.g1_compress(p) for p in pts)
    ks = [5, R - 1, 123456789, 2]
    got = affs_dec(fresh.g1_scalar_mul_affine(affs_enc(pts), frs_enc(ks), broadcast=False))
    assert got == [b.g1_mul(p, k) for p, k in zip(pts, ks)]


def test_host_pointer_calls_grow_then_reuse_their_buffers(fresh, cb):
    rnd = random.Random(11)
    base = Rand(12, cb).get_g1_affines(64)
    for n in (4, 5000, 4):
        ps = [base[rnd.randrange(64)] for _ in range(n)]
        ps[n // 2] = None
        qs = [base[rnd.randrange(64)] for _ in range(n)]
        ks = [rnd.randrange(R) for _ in range(n)]
        x = rnd.randrange(R)

        A = [rnd.randrange(FP) for _ in range(n)]
        B = [rnd.randrange(FP) for _ in range(n)]
        out = fresh.fp_mul(b"".join(fp_enc(a) for a in A), b"".join(fp_enc(v) for v in B))
        assert [fp_dec(out[i:i + 48]) for i in range(0, len(out), 48)] == [a * v % FP for a, v in zip(A, B)], n

        got = affs_dec(fresh.g1_scalar_mul_affine(affs_enc(ps), frs_enc(ks), broadcast=False))
        assert got == cb.mul_batch(ps, ks), n

        assert affs_dec(fresh.g1_fold(affs_enc(ps), affs_enc(qs), fr_enc(x))) == cb.fold(ps, qs, x), n

        jac = b"".join(jac_enc(p, rnd.randrange(1, FP)) for p in ps)
        assert affs_dec(fresh.g1_batch_to_affine(jac)) == ps, n

        enc = fresh.g1_compress(affs_enc(ps))
        assert enc == cb.compress(ps), n
        dec, status = fresh.g1_decompress(enc)
        assert affs_dec(dec) == ps and status == [0] * n, n


def test_protocol_calls_grow_then_reuse_the_engine_buffers(fresh, pkg, cb):
    """Whisk tracker proofs (whisk/whisk.go:116-176) at B = 1, 64, 1 on one engine: byte-identical to the
    oracle's proofs, and every one of them accepted."""
    B = 64
    P.set_backend(cb)
    try:
        ks, trackers, kcomms, oproofs = [], [], [], []
        for i in range(B):
            r = Rand(700 + i)
            k, rr = r.get_fr(), r.get_fr()
            rG = cb.mul(b.G1_GEN, rr)
            tr = W.new_tracker(rG, cb.mul(rG, k))
            ks.append(k)
            trackers.append(tr[0] + tr[1])
            kcomms.append(b.g1_compress(cb.mul(b.G1_GEN, k)))
            oproofs.append(W.generate_whisk_tracker_proof(tr, k, Rand(900 + i)))
    finally:
        P.set_backend(P.PyBackend())
    for n in (1, B, 1):
        proofs, status = fresh.whisk_generate_tracker_proof_batch(b"".join(trackers[:n]), b"".join(fr_enc(k) for k in ks[:n]),
                                                                  [pkg.Rand(900 + i) for i in range(n)])
        assert status == [0] * n
        assert [proofs[128 * i:128 * i + 128] for i in range(n)] == oproofs[:n]
        ok, st = fresh.whisk_is_valid_tracker_proof_batch(b"".join(trackers[:n]), b"".join(kcomms[:n]), proofs)
        assert ok == [1] * n and st == [0] * n
