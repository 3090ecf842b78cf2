"""Shared helpers for the parity tests (test infrastructure)."""
import hashlib

import numpy as np

from pct_oracle import OracleDiscrete, policy_pick, rnd_u64  # noqa: F401  (oracle/ is on sys.path via conftest)

ITEM_SET = [(i, j, k) for i in range(1, 6) for j in range(1, 6) for k in range(1, 6)]  # givenData.py:7-14
# the same 125 sizes scaled to the unit container of the continuous domain (givenData.py:4 `container_size = [1,1,1]`)
CONT_ITEM_SET = [(round(0.1 * i, 1), round(0.1 * j, 1), round(0.1 * k, 1)) for i in range(1, 6) for j in range(1, 6) for k in range(1, 6)]


def make_stream(seed, env, n, setting):
    """Deterministic per-env draw sequence (x,y,z,density) over the 125-item set."""
    s = np.zeros((n, 4))
    for d in range(n):
        s[d, :3] = ITEM_SET[rnd_u64(seed, env, d) % 125]
        s[d, 3] = max((rnd_u64(seed ^ 0xABCDEF, env, d) >> 11), 1) / float(1 << 53) if setting == 3 else 1.0
    return s


def obs_digest(obs):
    """SHA-256 of the float64 values of an observation (-0.0 counted as 0.0) as 32 uint8: the reference records of
    tests/golden/make_reference_records.py keep observations in this form, so that equal digests mean np.array_equal observations"""
    a = np.ascontiguousarray(obs, dtype=np.float64) + 0.0
    return np.frombuffer(hashlib.sha256(a.tobytes()).digest(), dtype=np.uint8)


def obs_digests(obs_seq):
    return np.stack([obs_digest(o) for o in obs_seq])


# ---- non-default configurations (tests/golden/make_golden_cases.py records them from the reference; the GPU cases of
# tests/test_gpu_discrete_cases.py use the same containers / item sets) ----------------------------------------------------
def _case(setting, container, items, nb=80, nl=50, steps=90, lnes="EMS"):
    return dict(setting=setting, container=tuple(container), items=[tuple(i) for i in items], nb=nb, nl=nl, steps=steps, lnes=lnes)


_BIG = [(i, j, k) for i in (4, 6, 9) for j in (5, 8) for k in (3, 7, 10)]
_SMALL = [(2, 2, 2), (3, 3, 2), (2, 3, 3), (4, 2, 2), (3, 4, 3)]
CASES = {
    "big_s1": _case(1, (20, 18, 24), _BIG), "big_s2": _case(2, (20, 18, 24), _BIG), "big_s3": _case(3, (20, 18, 24), _BIG),
    "holders_s1": _case(1, (10, 10, 10), ITEM_SET, nb=60, nl=30), "holders_s2": _case(2, (10, 10, 10), ITEM_SET, nb=80, nl=64),
    "dense16_s1": _case(1, (16, 16, 16), _SMALL, steps=70), "dense16_s2": _case(2, (16, 16, 16), _SMALL, steps=70),
    "flat_s1": _case(1, (12, 7, 9), [(i, j, k) for i in (1, 2, 4) for j in (1, 3) for k in (2, 3)], nb=70, nl=40),
    "cp_big_s1": _case(1, (14, 12, 10), ITEM_SET, steps=70, lnes="CP"), "ep_big_s2": _case(2, (14, 12, 10), ITEM_SET, steps=70, lnes="EP"),
    # found by scratch/soak_oracle_vs_reference.py: in extreme2D the dict newEps received key 2 before key 0 and the two points collide in
    # the 8-slot set table, so list(set(newEps.values())) lists them in the other order (D:PctTools.py:113-133)
    "ep_dictorder_s2": dict(_case(2, (14, 12, 10), ITEM_SET, steps=70, lnes="EP"), seed=134366, env=3),
    # the BASELINE-stream trajectories (items seed 1234, policy seed 4321) on which the object-alias semantics of the reference's real placement and
    # the snapshot semantics of round 1 part (scratch/alias_rate.py; DESIGN.md section 3 (b)) — recorded from the reference through and 30 steps past
    # the parting step; only the alias semantics (default since round 2) replays them
    "alias_d1_e126": dict(_case(1, (10, 10, 10), ITEM_SET, steps=69), seed=1234, pseed=4321, env=126),
    "alias_d1_e835": dict(_case(1, (10, 10, 10), ITEM_SET, steps=197), seed=1234, pseed=4321, env=835),
    "alias_d3_e92": dict(_case(3, (10, 10, 10), ITEM_SET, steps=133), seed=1234, pseed=4321, env=92),
}
NEEDS_ALIAS_D = ("alias_d1_e126", "alias_d1_e835", "alias_d3_e92")


def case_stream(c, seed, env, n):
    """draw sequence (x, y, z, density) over the case's item set"""
    s = np.zeros((n, 4))
    for d in range(n):
        s[d, :3] = c["items"][rnd_u64(seed, env, d) % len(c["items"])]
        s[d, 3] = max((rnd_u64(seed ^ 0xABCDEF, env, d) >> 11), 1) / float(1 << 53) if c["setting"] == 3 else 1.0
    return s


def _ccase(setting, container, lo, hi, nb=80, nl=50, steps=110):
    return dict(setting=setting, container=tuple(container), lo=lo, hi=hi, low=lo, nb=nb, nl=nl, steps=steps)


# continuous: a non-unit container (bounds scale like tools.py:178-181: U(0.1, 0.5) x min side) and other holder sizes
CONT_CASES = {"box2_s1": _ccase(1, (2.0, 1.5, 2.5), 0.15, 0.75), "box2_s2": _ccase(2, (2.0, 1.5, 2.5), 0.15, 0.75),
              "box2_s3": _ccase(3, (2.0, 1.5, 2.5), 0.15, 0.75), "holders_s1": _ccase(1, (1.0, 1.0, 1.0), 0.1, 0.5, nb=60, nl=25),
              # found by scratch/soak_oracle_vs_reference.py: a real placement whose verdict depends on Python object aliasing in the reference
              # (`up_edges[self] = self.thisStack` stores the live Stack object; DESIGN.md section 3).  Replayed exactly only under the object-alias semantics (default since round 2).
              "alias_s1": dict(_ccase(1, (2.0, 1.5, 2.5), 0.15, 0.75, steps=95), seed=136818, env=2)}
NEEDS_ALIAS = ("alias_s1",)  # records only the object-alias semantics (the default of the oracle AND of the kernels since round 2) reproduces; the
#                              snapshot mode (PCT_ORACLE_ALIAS=0 / PCT_B200_ALIAS=0) must NOT: tests/test_oracle_golden.py


def cont_case_stream(c, seed, env, n):
    """x, y = round(U(lo, hi), 3); z likewise (setting 2) or one of five levels (C:bin3D.py:103-115 scaled to the container)"""
    s = np.zeros((n, 4))
    lo, hi = c["lo"], c["hi"]
    u = lambda salt, d: ((rnd_u64(seed ^ salt, env, d) >> 11) / float(1 << 53))
    levels = [round(lo * k, 3) for k in (1, 2, 3, 4, 5)]
    for d in range(n):
        s[d, 0] = round(lo + (hi - lo) * u(0x11, d), 3)
        s[d, 1] = round(lo + (hi - lo) * u(0x22, d), 3)
        s[d, 2] = round(lo + (hi - lo) * u(0x33, d), 3) if c["setting"] == 2 else levels[rnd_u64(seed ^ 0x44, env, d) % 5]
        s[d, 3] = max((rnd_u64(seed ^ 0xABCDEF, env, d) >> 11), 1) / float(1 << 53) if c["setting"] == 3 else 1.0
    return s


class OracleVec(object):
    """N independent oracle envs with the ShmemVecEnv worker semantics (auto-reset on done,
    wrapper/shmem_vec_env.py:139-143) and the shared deterministic policy."""

    def __init__(self, n, setting, streams, nb=80, nl=50, container=(10, 10, 10)):
        self.envs = [OracleDiscrete(setting, container_size=container, internal_node_holder=nb, leaf_node_holder=nl, stream=streams[i])
                     for i in range(n)]
        self.n, self.nb, self.nl = n, nb, nl

    def reset(self):
        return np.stack([e.reset() for e in self.envs])

    def step(self, actions):
        obs, rew, done, infos = [], [], [], []
        for e, a in zip(self.envs, actions):
            o, r, d, i = e.step(a)
            if d:
                o = e.reset()
            obs.append(o); rew.append(r); done.append(d); infos.append(i)
        return np.stack(obs), np.array(rew), np.array(done), infos

    def pick(self, obs, seed, t, env_id_base=0):
        idx, rows = [], []
        for e in range(self.n):
            k, row = policy_pick(obs[e], self.nb, self.nl, seed, env_id_base + e, t)
            idx.append(k); rows.append(row)
        return np.array(idx, dtype=np.int32), np.stack(rows)


# ---- batched-evaluation parity helpers (evaluation_tools.py:7-52 restated as a plain loop) -------------------------------
def eval_policy_np(obs, nb=80, nl=50):
    """deterministic test policy: a fixed function of (#valid leaves, #valid internal rows)"""
    o = obs.reshape(nb + nl + 1, 9)
    nv, nbx = int((o[nb:nb + nl, 8] == 1).sum()), int((o[:nb, 8] == 1).sum())
    return (7 * nv + 3 * nbx) % max(nv, 1)


def eval_policy_torch(obs, batch):
    import torch
    o = obs.reshape(obs.shape[0], batch.nb + batch.nl + 1, 9)
    nv, nbx = (o[:, batch.nb:batch.nb + batch.nl, 8] == 1).sum(1), (o[:, :batch.nb, 8] == 1).sum(1)
    return ((7 * nv + 3 * nbx) % torch.clamp(nv, min=1)).to(torch.int32)


def sequential_eval(make_env, episodes, nb=80, nl=50):
    """the reference's evaluation loop on any single env with its call surface (reference env or oracle):
    per episode -> (ratio, counter, packed)"""
    out = []
    for ep in range(episodes):
        env, obs = make_env(ep)
        while True:
            k = eval_policy_np(obs, nb, nl)
            row = obs.reshape(nb + nl + 1, 9)[nb + k].copy()
            items = env.packed
            obs, _, done, info = env.step(row)
            if done:
                out.append((float(info["ratio"]), int(info["counter"]), [list(p) for p in items]))
                break
    return out
