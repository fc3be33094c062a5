"""No GPU: the thresholds test_gpu_crossovers.py derives its sizes from are still found in the CUDA sources, and
the MSM tasks it crafts to hit the exceptional cases of the window-combine additions really do so under a
restatement of the kernels' digit schedules (digits from the product's own glv_decompose, built for the host), and
the tasks test_gpu_msm_repeated_bases crafts fill the Pippenger buckets with the multisets it intends."""
import ctypes
import os
import subprocess

import pytest

import crossovers as X
from oracle import bls12381 as b

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def hc(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("hc") / "libhostcheck.so")
    src = os.path.join(HERE, "hostcheck", "hostcheck.cpp")
    subprocess.run(["g++", "-O2", "-std=c++17", "-x", "c++", "-shared", "-fPIC", "-o", out, src], check=True)
    return ctypes.CDLL(out)


def test_every_threshold_is_found():
    got = {name: X.const(name) for name in X.SOURCES}
    assert all(v > 0 for v in got.values()), got
    assert X.jac_to_affine_bounds() == [(8, 8 * 148 * 64), (2, 2 * 148 * 64)]
    table, top, last = X.big_c_table()
    assert len(table) == top + 1 and last > 0
    # the sizes the GPU tests use sit on both sides of each crossover
    assert X.jac_to_affine_e(18943) == 1 and X.jac_to_affine_e(18944) == 2
    assert X.jac_to_affine_e(75775) == 2 and X.jac_to_affine_e(75776) == 8
    assert X.pick_chunk(2 * 148 * X.const("kMsmChunk") - 1, 148) == 32
    assert X.pick_chunk(2 * 148 * X.const("kMsmChunk"), 148) == X.const("kMsmChunk")
    n = X.const("kMsmSplitThreshold")
    assert X.msm_batch_path([1] * (n - 1)) == "small" and X.msm_batch_path([1] * n) == "tp"
    t = X.const("kMsmSplitTerms")
    assert X.msm_batch_path([t, 1]) == "small" and X.msm_batch_path([t + 1, 1]) == "tp"
    q = X.const("kBigQuadMaxOutputs")
    assert X.big_reduce1_outputs((1 << 15) - 1) <= q < X.big_reduce1_outputs(1 << 15)


def test_threshold_lookup_fails_loudly(monkeypatch):
    monkeypatch.setitem(X.SOURCES, "kQuadMaxOps", ("k_elem.cu", r"constexpr int kNoSuchConstant\s*=\s*(\d+);"))
    with pytest.raises(LookupError):
        X.const("kQuadMaxOps")


def test_glv_split_reconstructs(hc):
    ks = [0, 1, 16, 1 << 64, b.R - 1, b.R - 16, (b.R - 1) // 2, (b.R + 1) // 2, 0xFFFFFFFF << 100]
    for s, (k1, k2, n1, n2) in zip(ks, X.glv_split(hc, ks)):
        assert k1 < 1 << 127 and k2 < 1 << 127
        assert ((-k1 if n1 else k1) + (-k2 if n2 else k2) * X.LAMBDA) % b.R == s
    for k in (0, 1, 16, (1 << 127) - 1, 0x123456789ABCDEF << 60):
        assert sum(d << (4 * w) for w, d in enumerate(X.biased_digits(k))) == k


@pytest.mark.parametrize("name", sorted(X.collision_tasks()))
def test_crafted_tasks_collide_in_the_4bit_combines(hc, name):
    """k_msm_small's tree at level L, and both Horner walks (k_msm_combine_quad / _tp) at window 0"""
    task, level = X.collision_tasks()[name]
    kind = name.split("-")[0]
    want = sum(a * s for a, s in task) % b.R
    sch = X.small_schedule(hc, task)
    res, hits = sch["tree"]
    assert res == want and hits == [(level, 0, kind)]
    res, hits = sch["horner"]
    assert res == want and hits == [(0, kind)]
    assert (want == 0) == (kind == "opposite")


@pytest.mark.parametrize("kind", ["equal", "opposite"])
def test_crafted_tasks_collide_in_the_pippenger_horner(hc, kind):
    n = X.const("kBigMsmThreshold") + 1
    c = X.big_pick_c(n)
    task = X.big_collision_task(n, kind)
    assert len(task) == n
    res, hits = X.big_schedule(hc, task, c)
    assert res == sum(a * s for a, s in task) % b.R
    assert hits == [(0, kind)]
    # the 4-bit Horner of the throughput path (cdl_g1_msm at kBigMsmThreshold terms) with the 4-bit task
    small = X.padded_collision_task(n - 1, kind)
    assert len(small) == n - 1 and X.small_schedule(hc, small)["horner"][1] == [(0, kind)]


def test_a_changed_task_no_longer_collides(hc):
    """the checks above have teeth: one scalar off and no combine step meets an exceptional case"""
    for name, (task, _) in X.collision_tasks().items():
        (a0, s0), (a1, s1) = task
        sch = X.small_schedule(hc, [(a0, s0 + 1), (a1, s1)])
        assert sch["tree"][1] == [] and sch["horner"][1] == [], name
    n = X.const("kBigMsmThreshold") + 1
    task = X.big_collision_task(n, "equal")
    task[0] = (1, task[0][1] * 2)
    assert X.big_schedule(hc, task, X.big_pick_c(n))[1] == []


def test_slice_path_sizes():
    """test_gpu_msm_repeated_bases' slice case: 8192 copies of one base with one scalar put 8192 entries into one
    bucket per window and GLV half, above BigMsmDims::large at 0 and 3 batch-affine rounds"""
    n = 8192
    c = X.big_pick_c(n)
    for rounds in (0, 3):
        assert n >> rounds > X.big_large(n, c, rounds), rounds
    assert X.big_large(1 << 22, 16, 0) <= X.const("kBigLargeBucket")


@pytest.mark.parametrize("c", [8, 11, 16])
def test_known_buckets_hold_their_multisets(hc, c):
    """For every forced round count the crafted task fills each targeted bucket with exactly the intended multiset
    (counts 1, 2, 3, 2^R - 1, 2^R, 2^R + 1 of +P, and {P, -P}) and no other bucket, its scalars take no GLV split or
    negation, and a task with one scalar changed no longer does."""
    assert X.const("kBigMaxBaRounds") == 8
    for rounds in range(X.const("kBigMaxBaRounds") + 1):
        task, want = X.known_bucket_task(c, rounds)
        scalars = sorted({s for _, s in task})
        assert all(k2 == 0 and not n1 and not n2 for _, k2, n1, n2 in X.glv_split(hc, scalars))
        got = X.big_buckets(hc, task, c)
        for key, v in want.items():
            assert got.get(key) == v, (c, rounds, key, got.get(key), v)
        assert set(got) == set(want)  # no bucket outside the targeted ones
        assert {len(v) for v in want.values()} == {1, 2, 3, (1 << rounds) - 1, 1 << rounds, (1 << rounds) + 1} - {0}
        for i in (0, len(task) - 1):
            changed = list(task)
            changed[i] = (changed[i][0], changed[i][1] + 1)
            got = X.big_buckets(hc, changed, c)
            assert any(got.get(key) != v for key, v in want.items()), (c, rounds, i)
