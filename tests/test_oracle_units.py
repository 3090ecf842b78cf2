"""CPU: the oracle's building blocks against CPython / numpy themselves (third-party arithmetic the reference leans on:
set iteration order, tuple and float hashes, lstsq) and against records of the reference's convex_hull.py."""
import ctypes as C
import os
import random

import numpy as np
import pytest

import pct_oracle

L = pct_oracle.lib()


def test_set_order_matches_cpython():
    rng = random.Random(5)
    for trial in range(400):
        n = rng.choice([1, 3, 7, 20, 60, 200, 700, 1300])
        hi = rng.choice([3, 10, 11, 40])
        keys = [tuple(rng.randrange(0, hi) for _ in range(6)) for _ in range(n)]
        s = set()
        for k in keys:
            s.add(k)
        want = list(s)
        uniq, seen = [], set()
        for k in keys:
            if k not in seen:
                seen.add(k); uniq.append(k)
        arr = np.array(keys, dtype=np.int64)
        order = np.zeros(len(keys) + 1, dtype=np.int32)
        m = L.pcto_set_order6(arr.ctypes.data_as(C.POINTER(C.c_int64)), len(keys), order.ctypes.data_as(C.POINTER(C.c_int)))
        got = [uniq[i] for i in order[:m]]
        assert got == want, "trial %d n=%d" % (trial, n)


def test_float_hash_matches_cpython():
    rng = np.random.RandomState(1)
    vals = list(rng.uniform(-3, 3, 2000)) + [0.0, 0.1, 0.5, 1.0, 0.123456, 1e-6, 123456.789, 2.0 ** 70, -0.3]
    vals += [round(v, 3) for v in rng.uniform(0.1, 0.5, 500)] + [round(a + b, 6) for a, b in rng.uniform(0, 1, (300, 2))]
    for v in vals:
        assert L.pcto_hash_double(float(v)) == (hash(float(v)) & ((1 << 64) - 1)), v


def test_lstsq_close_to_numpy():
    rng = np.random.RandomState(2)
    for k in (3, 4, 5, 8, 16):
        for trial in range(40):
            M = k * (k - 1) // 2 + 1
            A = np.zeros((M, k))
            c = 0
            for i in range(k - 1):
                for j in range(i + 1, k):
                    if rng.rand() > 0.15:
                        A[c, i] = 1; A[c, j] = -abs(rng.randn()) * rng.choice([1, 1, 1, -1])
                    c += 1
            A[-1] = 1
            b = np.zeros(M); b[-1] = 1
            x = np.zeros(k)
            Ac = np.ascontiguousarray(A)
            L.pcto_lstsq(Ac.ctypes.data_as(C.POINTER(C.c_double)), M, k, b.ctypes.data_as(C.POINTER(C.c_double)),
                         x.ctypes.data_as(C.POINTER(C.c_double)))
            want = np.linalg.lstsq(A, b[:, None], rcond=None)[0][:, 0]
            assert np.allclose(x, want, rtol=1e-9, atol=1e-11), (k, trial)


def test_lstsq_rank_deficient_minimum_norm():
    A = np.zeros((4, 3)); A[-1] = 1          # all pair rows zero: x = 1/3 each
    b = np.array([0, 0, 0, 1.0]); x = np.zeros(3)
    L.pcto_lstsq(A.ctypes.data_as(C.POINTER(C.c_double)), 4, 3, b.ctypes.data_as(C.POINTER(C.c_double)), x.ctypes.data_as(C.POINTER(C.c_double)))
    assert np.allclose(x, 1 / 3, atol=1e-14)
    A = np.array([[1, -1e16, 0], [0, 0, 0], [0, 1, -2.0], [1, 1, 1]])  # huge ratio: truncated singular value like gelsd
    want = np.linalg.lstsq(A, b[:, None], rcond=None)[0][:, 0]
    L.pcto_lstsq(np.ascontiguousarray(A).ctypes.data_as(C.POINTER(C.c_double)), 4, 3, b.ctypes.data_as(C.POINTER(C.c_double)),
                 x.ctypes.data_as(C.POINTER(C.c_double)))
    assert np.allclose(x, want, rtol=1e-6, atol=1e-9)


def test_hull_and_pip_match_reference_module():
    """oracle hull / point-in-polygon against the reference's ConvexHull + Space.scale_down and point_in_polygen on the same random draws
    (records of tests/golden/make_reference_records.py)"""
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "hull_pip.npz"))
    off = np.concatenate([[0], np.cumsum(g["hull_len"])])
    rng = np.random.RandomState(3)
    n_pip = 0
    for trial in range(600):
        k = rng.choice([1, 1, 2, 2, 3, 4, 6])
        pts = []
        for _ in range(k):
            x1, y1 = rng.randint(0, 8, 2); x2, y2 = x1 + rng.randint(1, 4), y1 + rng.randint(1, 4)
            pts += [[x1, y1], [x1, y2], [x2, y1], [x2, y2]]
        want = g["hull_flat"][off[trial]:off[trial + 1]]
        p = np.array(pts, dtype=np.float64)
        out = np.zeros((2 * len(pts), 2))
        m = L.pcto_hull_shrunk(p.ctypes.data_as(C.POINTER(C.c_double)), len(pts), out.ctypes.data_as(C.POINTER(C.c_double)))
        assert m == len(want) and np.array_equal(out[:m], want), trial
        for _ in range(6):
            q = np.array([rng.randint(0, 20) / 2.0, rng.randint(0, 20) / 2.0]) if rng.rand() < 0.5 else rng.uniform(0, 10, 2)
            got = L.pcto_pip(q[0], q[1], np.ascontiguousarray(want).ctypes.data_as(C.POINTER(C.c_double)), m)
            assert bool(got) == bool(g["pip"][n_pip])
            n_pip += 1
    assert n_pip == len(g["pip"])


def test_around6_commutes_with_min():
    """The identity behind the opt-in pre-rounded resting-height loop of the continuous feasibility kernel
    (csrc/pct_continuous.cu rest_height_pre): around6(v) = rint(v * 1e6) / 1e6 is monotone, hence
    around6(min(a, b)) == min(around6(a), around6(b)) bit for bit — checked on random, nearly equal and half-way operands."""
    rng = np.random.default_rng(5)
    r6 = lambda v: np.rint(v * 1e6) / 1e6
    a = rng.uniform(-3, 3, 400000)
    pairs = [(a, rng.uniform(-3, 3, a.size)), (a, a + rng.uniform(-2e-6, 2e-6, a.size)), (a, np.nextafter(a, 9.0)), (a, np.nextafter(a, -9.0))]
    k = rng.integers(-3000000, 3000000, a.size).astype(np.float64)
    half = (k + 0.5) / 1e6  # operands around the rounding boundaries
    pairs += [(half, np.nextafter(half, 9.0)), (half, np.nextafter(half, -9.0)), (half, half + rng.uniform(-1e-9, 1e-9, a.size)), (-half, half)]
    for x, y in pairs:
        lhs, rhs = r6(np.minimum(x, y)), np.minimum(r6(x), r6(y))
        assert np.array_equal(lhs, rhs)
        assert np.all(np.diff(r6(np.sort(x))) >= 0)  # monotone


@pytest.mark.parametrize("setting", [1, 2, 3])
def test_threaded_continuous_batch_equals_single_env_oracle(setting):
    """oracle/pct_oracle_batch_continuous.c (in-oracle sample_from_distribution draws, synthetic policy, auto-reset, pthreads) against the
    Python-driven single-env oracle on make_continuous_stream: same final observations, reward sums and episode counts"""
    from pct_oracle import OracleBatchContinuous, OracleContinuous, make_continuous_stream, policy_pick
    n, steps, iseed, pseed = 6, 60, 1234, 4321
    b = OracleBatchContinuous(n, setting, iseed, pseed, threads=3)
    b.run(25)
    b.run(steps - 25)  # the step counter of the policy continues across calls
    obs, rew, nd = b.get()
    for e in range(n):
        env = OracleContinuous(setting, stream=make_continuous_stream(iseed, e, 400, setting))
        o, rs, dn = env.reset(), 0.0, 0
        for t in range(steps):
            _, row = policy_pick(o, 80, 50, pseed, e, t)
            o, r, d, _ = env.step(row)
            rs += r
            if d:
                dn += 1
                o = env.reset()
        assert np.array_equal(o, obs[e]) and dn == nd[e] and abs(rs - rew[e]) < 1e-9, e
    b.close()
