"""CPU: lock-step of the C oracle against records of the unmodified Python reference (every observation including terminal ones,
reward, done, info) on fresh seeds, recorded by tests/golden/make_reference_records.py."""
import os

import numpy as np
import pytest

from harness import make_stream, obs_digest, obs_digests, policy_pick
from pct_oracle import OracleDiscrete

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _ref_info(g, t):
    """the reference's info dict of step t, rebuilt from the record"""
    keys = str(g["info_keys"][t]).split(",")
    full = {"counter": int(g["counter"][t]), "ratio": float(g["ratio"][t]), "reward": float(g["info_reward"][t])}
    return {k: full[k] for k in keys}


@pytest.mark.parametrize("setting", [1, 2, 3])
def test_lockstep_with_reference(setting):
    g = np.load(os.path.join(G, "lockstep_s%d.npz" % setting))
    seed, env_id, steps = 900 + setting, 3, 260
    stream = make_stream(seed, env_id, steps + 64, setting)
    orc = OracleDiscrete(setting, stream=stream)
    o2 = orc.reset()
    for t in range(steps):
        assert np.array_equal(g["pre_obs"][t], obs_digest(o2)), t
        _, row = policy_pick(o2, 80, 50, seed, env_id, t)
        o2, r2, d2, i2 = orc.step(row)
        d1 = bool(g["done"][t])
        assert np.array_equal(g["post_obs"][t], obs_digest(o2)), "observation after step %d (done=%s)" % (t, d1)
        assert (float(g["reward"][t]), d1) == (r2, d2) and _ref_info(g, t) == i2
        if d1:
            o2 = orc.reset()


# ---- other configurations (fresh seeds; the records of the same configurations that the GPU tests use are tests/golden/case_*.npz) ----
from harness import CASES, CONT_CASES  # noqa: E402


def _equal_records(a, b):
    for k in ("obs", "reward", "done", "counter", "ratio"):
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("name", sorted(CASES))
def test_cases_lockstep_with_reference(name):
    """the recorder of tests/golden/make_golden_cases.py on the reference vs the same loop on the oracle, new seed"""
    from harness import case_stream
    c = dict(CASES[name], steps=60)
    ref = np.load(os.path.join(G, "lockstep_case_%s.npz" % name))

    orc = OracleDiscrete(c["setting"], container_size=c["container"], internal_node_holder=c["nb"], leaf_node_holder=c["nl"],
                         size_minimum=min(min(i) for i in c["items"]), stream=case_stream(c, 8800, 4, c["steps"] + 64), lnes=c["lnes"])
    o = orc.reset()
    obs, rew, done, counter, ratio = [o.copy()], [], [], [], []
    for t in range(c["steps"]):
        o, r, d, info = orc.step(ref["rows"][t])
        obs.append(o.copy()); rew.append(r); done.append(d); counter.append(info["counter"]); ratio.append(info.get("ratio", -1.0))
        if d:
            o = orc.reset()
            obs.append(o.copy())
    _equal_records(ref, dict(obs=obs_digests(obs), reward=np.array(rew), done=np.array(done), counter=np.array(counter), ratio=np.array(ratio)))


@pytest.mark.parametrize("name", sorted(CONT_CASES))
def test_continuous_cases_lockstep_with_reference(name):
    from harness import cont_case_stream
    from pct_oracle import OracleContinuous
    c = dict(CONT_CASES[name], steps=70)
    ref = np.load(os.path.join(G, "lockstep_ccase_%s.npz" % name))
    orc = OracleContinuous(c["setting"], container_size=c["container"], internal_node_holder=c["nb"], leaf_node_holder=c["nl"],
                           size_minimum=c["low"], stream=cont_case_stream(c, 8801, 5, c["steps"] + 64))
    o = orc.reset()
    obs, rew, done, counter, ratio = [o.copy()], [], [], [], []
    for t in range(c["steps"]):
        o, r, d, info = orc.step(ref["rows"][t])
        obs.append(o.copy()); rew.append(r); done.append(d); counter.append(info["counter"]); ratio.append(info.get("ratio", -1.0))
        if d:
            o = orc.reset()
            obs.append(o.copy())
    _equal_records(ref, dict(obs=obs_digests(obs), reward=np.array(rew), done=np.array(done), counter=np.array(counter), ratio=np.array(ratio)))


def test_the_known_divergence_is_lapack_rounding_at_a_geometric_tie():
    """The one disagreement a 130k-env-step fresh-seed soak found (scratch/soak_oracle_vs_reference.py; setting 1, seed 135409): a 4x2x1
    item resting on three boxes whose common edge passes exactly under its centre of mass -> no direct edge -> np.linalg.lstsq (LAPACK
    gelsd) splits the load.  The oracle's solver agrees with gelsd to 4e-16, but the next box's centre of mass then lies exactly ON the
    border between two of ITS supports, and the strict `centre > area` tests (D:space.py:186-187) are decided by that last bit.
    Demonstrated on the reference's own code: feed it the oracle solver's solution instead of LAPACK's and ITS verdict flips too.
    (gelsd's last bits depend on the BLAS build, so this tie is not reproducible across machines even by the reference itself.)
    The record holds the reference's observations up to the tie, the least-squares system there, LAPACK's solution on the recording machine
    and the reference's verdict with LAPACK's solution (infeasible) and with the oracle solver's (feasible)."""
    from harness import case_stream
    from pct_oracle import _dp, lib
    g = np.load(os.path.join(G, "lapack_tie.npz"))
    assert not g["verdict_lapack"] and g["verdict_oracle_solver"]
    c, seed, env_id = CASES["holders_s1"], 135409, 0
    stream = case_stream(c, seed, env_id, 200)
    orc = OracleDiscrete(1, internal_node_holder=c["nb"], leaf_node_holder=c["nl"], stream=stream)
    o2 = orc.reset()
    for t in range(47):
        assert np.array_equal(g["obs"][t], obs_digest(o2)), t
        _, row = policy_pick(o2, c["nb"], c["nl"], seed, env_id, t)
        o2, _, d2, _ = orc.step(row)
        if d2:
            o2 = orc.reset()
    A, b, x = g["A"], g["b"], np.zeros(g["A"].shape[1])
    lib().pcto_lstsq(_dp(np.ascontiguousarray(A)), A.shape[0], A.shape[1], _dp(np.ascontiguousarray(b)), _dp(x))
    if not np.array_equal(g["obs"][47], obs_digest(o2)):  # on the recording machine's BLAS the tie falls the other way for the oracle: the documented divergence
        assert 0 < np.abs(g["x_lapack"] - x).max() < 1e-15
