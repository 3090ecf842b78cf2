"""CPU: the HOST logic of the product (pct_b200.evaluation.evaluate_batched, pct_b200.heuristics.run_heuristic, the single-env facades'
dataset handling) on an oracle-backed stand-in for PctBatch (tests/fake_batch.py), against the records of the unmodified reference.
What is exercised here is Python only — stream layout, per-env quotas, episode bookkeeping, the 3-decimal rounding of continuous datasets,
packed-list extraction — ; the kernels behind the real PctBatch are checked by the `-m gpu` tests."""
import glob
import importlib
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")
from fake_batch import FakeBatch  # noqa: E402
from harness import CONT_ITEM_SET, ITEM_SET, eval_policy_torch, sequential_eval  # noqa: E402

G = os.path.join(os.path.dirname(__file__), "golden")


def _eval_golden(path):
    g = np.load(path)
    off = np.concatenate([[0], np.cumsum(g["packed_len"])])
    packed = [g["packed_flat"][off[i]:off[i + 1]].tolist() for i in range(len(g["ratio"]))]
    return int(g["setting"]), g["data"], g["ratio"], g["counter"], packed


def _heur_golden(path, name, key):
    g = np.load(path)
    off = np.concatenate([[0], np.cumsum(g["len_" + name])])
    return int(g["setting"]), g[key], [g["flat_" + name][off[i]:off[i + 1]].tolist() for i in range(len(off) - 1)]


@pytest.fixture
def fake(monkeypatch):
    for mod in ("pct_b200.evaluation", "pct_b200.heuristics", "pct_b200.envs"):
        monkeypatch.setattr(importlib.import_module(mod), "PctBatch", FakeBatch)
    return FakeBatch


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(G, "eval_s*.npz"))))
@pytest.mark.parametrize("n_envs", [1, 7])
def test_evaluate_batched_host_logic_discrete(fake, path, n_envs, tmp_path):
    from pct_b200.evaluation import evaluate_batched
    setting, data, ratio, counter, packed = _eval_golden(path)
    out = evaluate_batched(list(data), setting, policy=eval_policy_torch, item_set=ITEM_SET, n_envs=n_envs, out_dir=str(tmp_path))
    assert out["length"].tolist() == counter.tolist() and out["packed"] == packed
    assert np.allclose(out["ratio"], ratio, rtol=0, atol=1e-15)
    saved = np.load(os.path.join(str(tmp_path), "trajs.npy"), allow_pickle=True)
    assert [list(map(list, ep)) for ep in saved] == packed


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(G, "eval_cont_s*.npz"))))
@pytest.mark.parametrize("n_envs", [1, 5])
def test_evaluate_batched_host_logic_continuous(fake, path, n_envs):
    from pct_b200.evaluation import evaluate_batched
    setting, data, ratio, counter, packed = _eval_golden(path)
    out = evaluate_batched(list(data), setting, policy=eval_policy_torch, container_size=(1.0, 1.0, 1.0), continuous=True, sample_left_bound=0.1,
                           n_envs=n_envs)
    assert out["length"].tolist() == counter.tolist()
    assert out["packed"] == packed
    assert out["ratio"].tolist() == ratio.tolist()


@pytest.mark.parametrize("name", ["LSAH", "OnlineBPH", "BR", "DBL"])
def test_run_heuristic_host_logic_discrete(fake, name):
    from pct_b200.heuristics import run_heuristic
    setting, data, packed = _heur_golden(os.path.join(G, "heur_s1.npz"), name, "data")
    (mean, var, length), rec = run_heuristic(name, setting, len(packed), item_set=ITEM_SET, data=list(data), n_envs=3, return_episodes=True)
    assert rec["packed"] == packed
    ratios = [sum(p[0] * p[1] * p[2] for p in ep) / 1000.0 for ep in packed]
    assert abs(mean - np.mean(ratios)) < 1e-12 and abs(var - np.var(ratios)) < 1e-12 and length == np.mean([len(ep) for ep in packed])


@pytest.mark.parametrize("name", ["LSAH", "OnlineBPH", "BR"])
@pytest.mark.parametrize("setting", [1, 2])
def test_run_heuristic_host_logic_continuous(fake, name, setting):
    from pct_b200.heuristics import run_heuristic
    _, stream, packed = _heur_golden(os.path.join(G, "heur_cont_s%d.npz" % setting), name, "stream")
    (mean, var, length), rec = run_heuristic(name, setting, len(packed), container_size=(1.0, 1.0, 1.0), item_set=CONT_ITEM_SET, continuous=True,
                                             item_stream=stream[None], n_envs=1, return_episodes=True)
    assert rec["packed"] == packed
    with pytest.raises(ValueError):
        run_heuristic("DBL", setting, 1, continuous=True)


def test_facade_dataset_handling_discrete(fake, tmp_path):
    import pct_b200
    setting, data, ratio, counter, packed = _eval_golden(os.path.join(G, "eval_s1.npz"))
    ds = os.path.join(str(tmp_path), "set.pt")
    torch.save([t.tolist() for t in data], ds)
    env = pct_b200.PackingDiscrete(setting=setting, container_size=[10, 10, 10], item_set=ITEM_SET, data_name=ds, load_test_data=True)
    rec = sequential_eval(lambda ep: (env, env.reset()), 6)
    assert [r[1] for r in rec] == counter[:6].tolist() and [r[2] for r in rec] == packed[:6]
    assert np.allclose([r[0] for r in rec], ratio[:6], rtol=0, atol=1e-15)


def test_facade_dataset_handling_continuous(fake, tmp_path):
    import pct_b200
    setting, data, ratio, counter, packed = _eval_golden(os.path.join(G, "eval_cont_s1.npz"))
    ds = os.path.join(str(tmp_path), "set.pt")
    torch.save([t.tolist() for t in data], ds)
    env = pct_b200.PackingContinuous(setting=setting, container_size=[1, 1, 1], item_set=None, data_name=ds, load_test_data=True,
                                     sample_from_distribution=True, sample_left_bound=0.1, sample_right_bound=0.5)
    rec = sequential_eval(lambda ep: (env, env.reset()), 5)
    assert [r[1] for r in rec] == counter[:5].tolist() and [r[2] for r in rec] == packed[:5]
    assert np.allclose([r[0] for r in rec], ratio[:5], rtol=0, atol=1e-12)


# ---- the vector surface against the reference's OWN wrappers ---------------------------------------------------------------------
import ref_shim  # noqa: E402


@pytest.mark.parametrize("setting", [1, 2])
def test_vec_env_equals_reference_shmem_vecpytorch_monitor(fake, setting, monkeypatch):
    """VecPyTorch(ShmemVecEnv([Monitor(PackingDiscrete)] * N, context='fork')) of the unmodified reference (envs.py:75-116,159-182,
    wrapper/shmem_vec_env.py, wrapper/monitor.py), recorded by tests/golden/make_reference_records.py, next to PctVecEnv: observation
    tensors, reward shape / values, done array, info dicts (terminal ones with Monitor's 'episode' entry, the auto-reset observation) over
    70 vector steps."""
    from harness import make_stream, obs_digests, policy_pick
    monkeypatch.setattr(importlib.import_module("pct_b200.vec_env"), "PctBatch", FakeBatch)
    import pct_b200
    g = np.load(os.path.join(G, "vecenv_s%d.npz" % setting))
    n, seed = 5, 50 + setting
    streams = np.stack([make_stream(seed, e, 300, setting) for e in range(n)])
    ours = pct_b200.PctVecEnv(n, setting, item_set=ITEM_SET, item_stream=streams)
    try:
        o = ours.reset()
        assert o.dtype == torch.float32 and tuple(o.shape) == (n, 1179)  # the reference's VecPyTorch observations: float32, (n, 1179)
        dones = 0
        for t in range(70):
            assert np.array_equal(g["obs"][t], obs_digests(o.cpu().numpy())), "observations before step %d" % t
            rows = np.stack([policy_pick(o[e].cpu().numpy().astype(np.float64), 80, 50, seed, e, t)[1] for e in range(n)]).astype(np.float32)
            o, r, d, i = ours.step(rows)  # float32 numpy leaf rows, as train_tools.py:66-67 passes them
            r_ref, d_ref = torch.from_numpy(g["reward"][t]), g["done"][t]
            assert tuple(r.shape) == tuple(r_ref.shape) == (n, 1) and r.dtype == r_ref.dtype and torch.equal(r, r_ref)
            assert d.dtype == d_ref.dtype == np.bool_ and np.array_equal(d, d_ref)
            for e in range(n):
                keys_ref = set(str(g["info_keys"][t, e]).split(","))
                assert i[e]["counter"] == g["counter"][t, e]
                if d_ref[e]:
                    dones += 1
                    assert keys_ref == set(i[e]) == {"counter", "ratio", "reward", "episode"}
                    assert abs(i[e]["ratio"] - g["ratio"][t, e]) < 1e-6 and abs(i[e]["reward"] - g["info_reward"][t, e]) < 1e-5
                    assert i[e]["episode"]["l"] == g["ep_l"][t, e] and abs(i[e]["episode"]["r"] - g["ep_r"][t, e]) < 1e-4
                else:
                    assert set(i[e]) == keys_ref == {"counter"}
        assert np.array_equal(g["obs"][70], obs_digests(o.cpu().numpy()))
        assert dones >= 8
    finally:
        ours.close()


@pytest.mark.reference
@pytest.mark.skipif(not ref_shim.reference_available(), reason="reference not mounted")
@pytest.mark.parametrize("name,fn", [("LSAH", "LASH"), ("OnlineBPH", "OnlineBPH"), ("BR", "BR"), ("DBL", "DBL"), ("HM", "heightmap_min"), ("MACS", "MACS")])
def test_unmodified_heuristic_functions_run_on_the_facade(fake, name, fn, tmp_path):
    """heuristic.py's own LASH / OnlineBPH / BR / DBL / heightmap_min (unmodified) driving the drop-in PackingDiscrete: every attribute
    they touch (space.EMS, space.boxes, space.get_ratio, space.drop_box_virtual(returnH / returnMap), next_box get + set, next_den,
    orientation, bin_size, item_set, step([0, lx, ly]), reset) — episodes equal the records of the same functions on the reference env."""
    import contextlib
    import io
    import sys
    import pct_b200
    ref_shim.load_reference()
    argv, sys.argv = sys.argv, sys.argv[:1]
    try:
        H = importlib.import_module("heuristic")
    finally:
        sys.argv = argv
    setting, data, packed = _heur_golden(os.path.join(G, "heur_s1.npz"), name, "data")
    ds = os.path.join(str(tmp_path), "set.pt")
    torch.save([t.tolist() for t in data], ds)

    class Recording(pct_b200.PackingDiscrete):
        def reset(self):
            if getattr(self, "_played", False):
                self.log.append([list(p) for p in self.packed])
            self._played = True
            return super().reset()

    env = Recording(setting=setting, container_size=[10, 10, 10], item_set=ITEM_SET, data_name=ds, load_test_data=True)
    env.log = []
    episodes = 1 if name == "MACS" else 3
    with contextlib.redirect_stdout(io.StringIO()):
        getattr(H, fn)(env, episodes)
    assert env.log[:episodes] == packed[:episodes]


@pytest.mark.reference
@pytest.mark.skipif(not ref_shim.reference_available(), reason="reference not mounted")
@pytest.mark.parametrize("name,fn", [("LSAH", "LASH"), ("OnlineBPH", "OnlineBPH"), ("BR", "BR")])
def test_unmodified_heuristic_functions_run_on_the_continuous_facade(fake, name, fn):
    import contextlib
    import io
    import sys
    import pct_b200
    ref_shim.load_reference()
    argv, sys.argv = sys.argv, sys.argv[:1]
    try:
        H = importlib.import_module("heuristic")
    finally:
        sys.argv = argv
    setting, stream, packed = _heur_golden(os.path.join(G, "heur_cont_s1.npz"), name, "stream")

    class Recording(pct_b200.PackingContinuous):
        def reset(self):
            if getattr(self, "_played", False):
                self.log.append([list(map(float, p)) for p in self.packed])
            self._played = True
            return super().reset()

    env = Recording(setting=setting, container_size=[1, 1, 1], item_set=CONT_ITEM_SET, sample_from_distribution=False, item_stream=stream[None],
                    size_minimum=0.1)
    env.log = []
    with contextlib.redirect_stdout(io.StringIO()):
        getattr(H, fn)(env, 3)
    assert env.log[:3] == packed[:3]


@pytest.mark.parametrize("argv,continuous", [(["--setting", "1", "--num-processes", "6", "--seed", "9"], False),
                                              (["--setting", "2", "--continuous", "--sample-from-distribution", "--num-processes", "4"], True)])
def test_make_vec_envs_takes_the_reference_args(fake, argv, continuous, monkeypatch):
    """envs.make_vec_envs(args, log_dir, allow_early_resets) (envs.py:75-116) with the namespace tools.get_args() builds from `argv`
    (recorded from the reference by tests/golden/make_reference_records.py)"""
    import argparse
    import json
    import pct_b200
    monkeypatch.setattr(importlib.import_module("pct_b200.vec_env"), "PctBatch", FakeBatch)
    with open(os.path.join(G, "reference_args.json")) as f:
        rec = json.load(f)["continuous" if continuous else "discrete"]
    assert rec["argv"] == argv
    args = argparse.Namespace(**rec["args"])
    if continuous:
        args.container_size = [1, 1, 1]  # givenData.py:5 (the commented alternative)
        args.sample_left_bound, args.sample_right_bound = 0.1, 0.5
    envs = pct_b200.make_vec_envs(args, "./logs/runinfo", True)
    assert envs.num_envs == args.num_processes and envs.observation_space.shape == (1179,)
    obs = envs.reset()
    assert tuple(obs.shape) == (args.num_processes, 1179) and obs.dtype == torch.float32
    for t in range(30):
        leaf = obs.view(args.num_processes, 131, 9)[:, 80:130]
        nvalid = (leaf[:, :, 8] == 1).sum(1)
        rows = torch.stack([leaf[e, t % max(int(nvalid[e]), 1)] if nvalid[e] else torch.zeros(9) for e in range(args.num_processes)])
        obs, rew, done, infos = envs.step(rows.numpy())
        assert tuple(rew.shape) == (args.num_processes, 1) and len(infos) == args.num_processes
    nxt = obs.view(args.num_processes, 131, 9)[:, 130, 3:6]
    assert (nxt.min() >= 0.0999 and nxt.max() <= 0.5001) if continuous else (nxt.min() >= 1 and nxt.max() <= 5)
    envs.close()


@pytest.fixture
def one_torch_thread():
    n = torch.get_num_threads()
    torch.set_num_threads(1)  # main.py:28 does the same; the network is tiny
    yield
    torch.set_num_threads(n)


class _Stop(Exception):
    pass


class _Counting(object):
    """ends the reference's endless train loop after `limit` vector steps and logs what the trainer received"""

    def __init__(self, venv, limit):
        self.venv, self.limit, self.log = venv, limit, []

    def __getattr__(self, name):
        return getattr(self.venv, name)

    def reset(self):
        obs = self.venv.reset()
        self.log.append(obs.clone())
        return obs

    def step(self, actions):
        if len(self.log) > self.limit:
            raise _Stop()
        obs, rew, done, infos = self.venv.step(actions)
        self.log.append(obs.clone())
        return obs, rew, done, infos


@pytest.mark.reference
@pytest.mark.skipif(not ref_shim.reference_available(), reason="reference not mounted")
@pytest.mark.parametrize("acktr", [True, False])
def test_reference_trainer_runs_on_the_vector_surface(fake, acktr, tmp_path, monkeypatch, one_torch_thread):
    """train_tools.train_n_steps (train_tools.py:32-150: rollouts through envs.step(leaf rows), PCTRolloutStorage, ACKTR / A2C updates) —
    unmodified — on PctVecEnv and on the reference's own VecPyTorch(ShmemVecEnv(Monitor(env))) stack: same seeds, same item streams ->
    the trainer sees the same observations step after step and ends with the same network parameters."""
    from harness import make_stream
    monkeypatch.setattr(importlib.import_module("pct_b200.vec_env"), "PctBatch", FakeBatch)
    import pct_b200
    compat = importlib.import_module("pct_b200.compat")
    D, _ = ref_shim.load_reference()
    model, _ = compat.load_policy_modules(ref_shim.REFERENCE_ROOT)
    tt = importlib.import_module("train_tools")
    renvs = importlib.import_module("envs")
    ShmemVecEnv = importlib.import_module("wrapper.shmem_vec_env").ShmemVecEnv
    Monitor = importlib.import_module("wrapper.monitor").Monitor
    n, setting, limit = 4, 1, 16  # 3 updates of num_steps = 5, then one more step
    args = compat.reference_args(ref_shim.REFERENCE_ROOT, ["--setting", str(setting), "--num-processes", str(n), "--no-cuda", "--seed", "3"])
    args.use_acktr = acktr  # tools.py:121 `type=bool`: not settable to False from the command line
    args.model_save_path = str(tmp_path)
    streams = np.stack([make_stream(77, e, 400, setting) for e in range(n)])

    def thunk(rank):
        def _t():
            env = D.PackingDiscrete(setting=setting, container_size=[10, 10, 10], item_set=ITEM_SET, internal_node_holder=80, leaf_node_holder=50,
                                    shuffle=False, LNES="EMS")
            env.box_creator = ref_shim.make_stream_creator(D, [tuple(int(v) for v in r[:3]) for r in streams[rank]])
            env.test = True
            return Monitor(env, os.path.join(str(tmp_path), str(rank)), allow_early_resets=True)
        return _t

    probe = D.PackingDiscrete(setting=setting, container_size=[10, 10, 10], item_set=ITEM_SET)
    results = []
    for which in ("reference", "ours"):
        if which == "reference":
            venv = renvs.VecPyTorch(ShmemVecEnv([thunk(r) for r in range(n)], [probe.observation_space, probe.action_space], context="fork"), "cpu")
        else:
            venv = pct_b200.PctVecEnv(n, setting, item_set=ITEM_SET, item_stream=streams)
        counting = _Counting(venv, limit)
        torch.manual_seed(11)
        policy = model.DRL_GAT(args)
        trainer = tt.train_tools(None, "t", policy, args)
        try:
            with pytest.raises(_Stop):
                trainer.train_n_steps(counting, args, torch.device("cpu"))
        finally:
            venv.close()
        results.append((torch.stack(counting.log), [p.detach().clone() for p in policy.parameters()], trainer.step_counter))
    assert results[0][2] == results[1][2] == 4
    assert torch.equal(results[0][0], results[1][0])
    assert all(torch.equal(a, b) for a, b in zip(results[0][1], results[1][1]))


# ---- reference-default kwargs (ADVICE round 1): PackingContinuous' class defaults are sample_from_distribution=True, U(0.1, 0.5) (C:bin3D.py:14-16),
# so Space.low_bound is 0.1 even when a dataset supplies the items (heuristic.py:585-591 builds the env exactly like that) -----------------------
class _Recorder(FakeBatch):
    seen = None

    def __init__(self, *a, **kw):
        _Recorder.seen = dict(kw)
        super().__init__(*a, **kw)


def test_continuous_facade_has_the_reference_defaults(monkeypatch, tmp_path):
    import pct_b200.envs as E
    monkeypatch.setattr(E, "PctBatch", _Recorder)
    g = np.load(sorted(glob.glob(os.path.join(G, "eval_cont_s*.npz")))[0])
    path = os.path.join(str(tmp_path), "data.pt")
    torch.save([np.asarray(t) for t in g["data"]], path)
    env = E.PackingContinuous(setting=int(g["setting"]), container_size=[1.0, 1.0, 1.0], item_set=CONT_ITEM_SET, data_name=path, load_test_data=True,
                              internal_node_holder=80, leaf_node_holder=50)
    kw = _Recorder.seen
    assert kw["sample_from_distribution"] is True and kw["sample_left_bound"] == 0.1 and kw["sample_right_bound"] == 0.5
    assert kw["item_stream"] is not None  # the dataset supplies the items
    assert env._batch.size_minimum == 0.1
    o = env.reset()
    assert o.shape == (131 * 9,)


def test_run_heuristic_continuous_dataset_uses_reference_bounds_and_rounding(monkeypatch):
    import pct_b200.heuristics as Hm
    monkeypatch.setattr(Hm, "PctBatch", _Recorder)
    data = [np.array([[0.30004, 0.2, 0.1], [0.25, 0.25, 0.25]]) for _ in range(3)]
    Hm.run_heuristic("LSAH", 2, 2, container_size=(1.0, 1.0, 1.0), data=data, n_envs=2, continuous=True, sample_from_distribution=True,
                     sample_left_bound=0.1, sample_right_bound=0.5)
    kw = _Recorder.seen
    assert kw["sample_from_distribution"] is True and kw["sample_left_bound"] == 0.1
    assert kw["item_stream"][0, 0, 0] == 0.3  # round3 (C:bin3D.py:84-87) applied to the dataset
