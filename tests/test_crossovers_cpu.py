"""No GPU: the thresholds test_gpu_crossovers.py derives its sizes from are still found in the CUDA sources, and
the MSM tasks it crafts to hit the exceptional cases of the window-combine additions really do so under a
restatement of the kernels' digit schedules (digits from the product's own glv_decompose, built for the host)."""
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
