"""CPU: copy.deepcopy of the single-env facades and the argument checks of PctBatch.load_envs, on an oracle-backed stand-in for PctBatch.

The stand-in's records are "configuration + item source + event history" and a load replays that history on a fresh oracle env, so what is
checked here is the host logic (the facades' __deepcopy__, record_arguments); the device records themselves are checked by
tests/test_zzz_gpu_snapshot.py.  One `reference`-marked test deep-copies the unmodified reference's envs next to the facades."""
import copy
import os
import pickle

import numpy as np
import pytest

torch = pytest.importorskip("torch")
from fake_batch import FakeBatch  # noqa: E402
from harness import ITEM_SET  # noqa: E402
import ref_shim  # noqa: E402

G = os.path.join(os.path.dirname(__file__), "golden")


class RecordingFakeBatch(FakeBatch):
    """FakeBatch with save_envs / load_envs: a record is (constructor arguments, index of the env whose item source it follows, the events
    since creation, episode sums, LSAH state, last observation); a load rebuilds that env on the oracle and replays the events."""
    RECORD_BYTES = 1 << 16

    def __init__(self, *args, **kw):
        super().__init__(*args, **kw)
        self._args = (args, kw)
        self._traj = 0
        self._src = list(range(self.n_envs))
        self._hist = [[] for _ in range(self.n_envs)]

    @property
    def record_bytes(self):
        return self.RECORD_BYTES

    def set_trajectory_length(self, n):
        super().set_trajectory_length(n)
        self._traj = n

    def reset(self, out=None):
        for h in self._hist:
            h.append(None)
        return super().reset(out)

    def step(self, actions=None, leaf_idx=None, out=None):
        for i in range(self.n_envs):
            if leaf_idx is not None:
                k = int(leaf_idx[i])
                leaf = self._obs64[i].reshape(-1, 9)[self.nb:self.nb + self.nl]
                row = leaf[k].copy() if 0 <= k < int((leaf[:, 8] == 1).sum()) else np.zeros(9)
            else:
                row = np.asarray(actions[i], dtype=np.float64).copy()
            self._hist[i].append(row)
        return super().step(actions=actions, leaf_idx=leaf_idx, out=out)

    def save_envs(self, env_ids=None, out=None):
        ids = list(range(self.n_envs)) if env_ids is None else [int(i) for i in env_ids]
        rec = torch.zeros((len(ids), self.RECORD_BYTES), dtype=torch.uint8)
        for r, i in enumerate(ids):
            blob = pickle.dumps((repr(self._args), self._traj, self._src[i], list(self._hist[i]), self._ep[i].copy(), copy.deepcopy(self._hstate[i]),
                                 self._obs64[i].copy()))
            assert len(blob) + 4 <= self.RECORD_BYTES
            rec[r, :4] = torch.from_numpy(np.array([len(blob)], dtype=np.int32).view(np.uint8))
            rec[r, 4:4 + len(blob)] = torch.frombuffer(bytearray(blob), dtype=torch.uint8)
        return rec

    def load_envs(self, records, env_ids=None, obs=None, check=True):
        from pct_b200.batch import PctError, record_arguments
        records, ids, n = record_arguments(records, env_ids, self.n_envs, self.RECORD_BYTES, torch.device("cpu"))
        for r in range(n):
            d = r if ids is None else int(ids[r])
            a = records[r].numpy()
            blob = a[4:4 + int(a[:4].view(np.int32)[0])].tobytes()
            args, traj, src, hist, ep, hstate, obs64 = pickle.loads(blob)
            if args != repr(self._args) or traj != self._traj:
                raise PctError("record of another configuration")
            fresh = FakeBatch(*self._args[0], **self._args[1])
            if traj:
                fresh.set_trajectory_length(traj)
            e = fresh.envs[src]
            for ev in hist:  # replay
                if ev is None:
                    e.reset()
                else:
                    _, _, done, _ = e.step(ev)
                    if done and self.auto_reset:
                        e.reset()
            self.envs[d], self._src[d], self._hist[d] = e, src, list(hist)
            self._ep[d], self._hstate[d], self._obs64[d] = ep, hstate, obs64
        return None


@pytest.fixture
def fake(monkeypatch):
    import importlib
    monkeypatch.setattr(importlib.import_module("pct_b200.envs"), "PctBatch", RecordingFakeBatch)
    return RecordingFakeBatch


def _pick(obs, nb, nl, rng):
    leaves = np.asarray(obs, dtype=np.float64).reshape(-1, 9)[nb:nb + nl]
    valid = np.nonzero(leaves[:, 8] == 1)[0]
    return leaves[valid[rng.randint(len(valid))]].copy() if len(valid) else np.zeros(9)


def _run(env, obs, rng, steps, nb=80, nl=50):
    """steps of a seeded random-leaf policy; resets after an episode; -> (observations, rewards, dones), last observation"""
    out = []
    for _ in range(steps):
        row = _pick(obs, nb, nl, rng)
        obs, r, d, _ = env.step(row)
        out.append((np.asarray(obs, dtype=np.float64).copy(), float(r), bool(d)))
        if d:
            obs = env.reset()
            out.append((np.asarray(obs, dtype=np.float64).copy(), 0.0, False))
    return out, obs


def _same(a, b):
    assert len(a) == len(b)
    for (oa, ra, da), (ob, rb, db) in zip(a, b):
        assert np.array_equal(oa, ob) and ra == rb and da == db


def _dataset(tmp_path, name):
    g = np.load(os.path.join(G, name))
    ds = os.path.join(str(tmp_path), "set.pt")
    torch.save([t.tolist() for t in g["data"]], ds)
    return int(g["setting"]), ds


def _facades(tmp_path):
    import pct_b200
    s, ds = _dataset(tmp_path, "eval_s1.npz")
    return [
        lambda: pct_b200.PackingDiscrete(setting=1, container_size=[10, 10, 10], item_set=ITEM_SET, seed=5),
        lambda: pct_b200.PackingDiscrete(setting=2, container_size=[10, 10, 10], item_set=ITEM_SET, seed=6, shuffle=True),
        lambda: pct_b200.PackingDiscrete(setting=s, container_size=[10, 10, 10], item_set=ITEM_SET, data_name=ds, load_test_data=True),
        lambda: pct_b200.PackingContinuous(setting=1, container_size=[1, 1, 1], seed=3),
    ]


@pytest.mark.parametrize("case", range(4))
def test_deepcopy_continues_like_the_original(fake, case, tmp_path):
    make = _facades(tmp_path)[case]
    a = make()
    rng = np.random.RandomState(case)
    _, oa = _run(a, a.reset(), rng, 23)
    b = copy.deepcopy(a)
    assert type(b) is type(a) and b._batch is not a._batch
    s = rng.get_state()
    ra, _ = _run(a, oa, rng, 40)
    rng.set_state(s)
    rb, _ = _run(b, oa, rng, 40)
    _same(ra, rb)


@pytest.mark.parametrize("case", range(4))
def test_stepping_the_copy_leaves_the_original_unchanged(fake, case, tmp_path):
    make = _facades(tmp_path)[case]
    a = make()
    rng = np.random.RandomState(10 + case)
    _, oa = _run(a, a.reset(), rng, 17)
    twin, c = copy.deepcopy(a), copy.deepcopy(a)
    _run(c, oa, np.random.RandomState(99), 25)  # the copy goes its own way
    s = rng.get_state()
    ra, _ = _run(a, oa, rng, 30)
    rng.set_state(s)
    rt, _ = _run(twin, oa, rng, 30)
    _same(ra, rt)


def test_deepcopy_keeps_the_next_box_override(fake):
    import pct_b200
    a = pct_b200.PackingDiscrete(setting=1, container_size=[10, 10, 10], item_set=ITEM_SET, seed=1)
    a.reset()
    nb = a.next_box
    a.next_box = [nb[1], nb[0], nb[2]]
    b = copy.deepcopy(a)
    assert b.next_box == [nb[1], nb[0], nb[2]]
    b.next_box = nb
    assert a.next_box == [nb[1], nb[0], nb[2]]


def test_load_arguments_are_checked(fake):
    from pct_b200.batch import PctError, record_arguments
    fb = RecordingFakeBatch(4, 1, item_set=ITEM_SET)
    fb.reset()
    rec = fb.save_envs([0, 0, 2])
    assert rec.shape == (3, fb.record_bytes)
    fb.load_envs(rec, [1, 3, 0])
    with pytest.raises(PctError, match="duplicate"):
        fb.load_envs(rec, [1, 1, 0])
    with pytest.raises(PctError, match="uint8"):
        fb.load_envs(rec.to(torch.int16), [1, 3, 0])
    with pytest.raises(PctError, match="uint8"):
        fb.load_envs(rec[:, :100], [1, 3, 0])
    with pytest.raises(PctError, match="uint8"):
        fb.load_envs(rec[0], [1])
    with pytest.raises(PctError, match="records for"):
        fb.load_envs(rec, [1, 3])
    with pytest.raises(PctError, match="all 4 envs"):
        fb.load_envs(rec)
    with pytest.raises(PctError, match=r"\[0, 4\)"):
        fb.load_envs(rec, [1, 4, 0])
    with pytest.raises(PctError, match="integers"):
        fb.load_envs(rec, torch.tensor([1.0, 3.0, 0.0]))
    with pytest.raises(PctError, match="tensor"):
        record_arguments(rec.numpy(), [1, 3, 0], 4, fb.record_bytes, torch.device("cpu"))
    out, ids, n = record_arguments(rec, np.array([3, 2, 1]), 4, fb.record_bytes, torch.device("cpu"))
    assert n == 3 and ids.dtype == torch.int32 and ids.tolist() == [3, 2, 1]


# ---- against the unmodified reference ----------------------------------------------------------------------------------------------
@pytest.mark.reference
@pytest.mark.skipif(not ref_shim.reference_available(), reason="reference not mounted")
@pytest.mark.parametrize("continuous", [False, True])
def test_deepcopy_matches_the_reference_with_load_test_data(fake, continuous, tmp_path):
    """copy.deepcopy of the reference's PackingDiscrete / PackingContinuous(load_test_data=True) (LoadBoxCreator: the copy replays the same
    trajectory) next to copy.deepcopy of the facade: the originals and the copies continue identically."""
    import pct_b200
    D, Cm = ref_shim.load_reference()
    if continuous:
        setting, ds = _dataset(tmp_path, "eval_cont_s1.npz")
        kw = dict(setting=setting, container_size=[1, 1, 1], item_set=None, data_name=ds, load_test_data=True, sample_from_distribution=True,
                  sample_left_bound=0.1, sample_right_bound=0.5)
        ref, fac = Cm.PackingContinuous(**kw), pct_b200.PackingContinuous(**kw)
    else:
        setting, ds = _dataset(tmp_path, "eval_s1.npz")
        kw = dict(setting=setting, container_size=[10, 10, 10], item_set=ITEM_SET, data_name=ds, load_test_data=True)
        ref, fac = D.PackingDiscrete(**kw), pct_b200.PackingDiscrete(**kw)
    ro, fo = ref.reset(), fac.reset()
    assert np.array_equal(np.asarray(ro, dtype=np.float64), fo)
    rr, ro = _run(ref, ro, np.random.RandomState(4), 12)
    rf, fo = _run(fac, fo, np.random.RandomState(4), 12)
    _same(rr, rf)
    ref2, fac2 = copy.deepcopy(ref), copy.deepcopy(fac)
    for env_r, env_f in ((ref2, fac2), (ref, fac)):  # the copies first, then the originals: both continue from the copied state
        a, _ = _run(env_r, ro, np.random.RandomState(8), 30)
        b, _ = _run(env_f, fo, np.random.RandomState(8), 30)
        _same(a, b)
