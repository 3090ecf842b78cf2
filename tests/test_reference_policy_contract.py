"""CPU: the reference's OWN policy network and evaluation loop on the drop-in env surface.

`model.DRL_GAT` (attention_model.AttentionModel + graph encoder) driven with the calls of evaluation_tools.evaluate (:9-24:
tools.get_leaf_nodes_with_factor on the observation, PCT_policy(all_nodes, True, normFactor), `leaf_nodes[batchX, idx]`, `env.step(row[0:6])`,
`env.packed`) on the reference env is recorded by tests/golden/make_reference_records.py: every observation, the leaf index the network
chose and each episode's (ratio, counter, packed).  The same choices are replayed on an env with the facade's call surface.  The CPU
oracle stands in for the CUDA path here — the GPU parity tests assert the two produce bit-identical observations, which is all the policy
ever sees, and equal observations mean the network would choose the same leaves.  Equal trajectories = the observation layout, the mask
column, the 6-float action rows and `packed` are what the unmodified consumers expect.  test_compat_runs_the_unmodified_evaluate runs the
reference's own code and is skipped without the reference checkout."""
import os
import sys

import numpy as np
import pytest

import ref_shim
from harness import make_stream, obs_digests
from pct_oracle import OracleDiscrete

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
sys.path.insert(0, G)
torch = pytest.importorskip("torch")


@pytest.fixture(autouse=True)
def _one_torch_thread():
    """evaluation.py:22 / main.py:28 do the same; the network is tiny and 8 BLAS threads only fight over it"""
    n = torch.get_num_threads()
    torch.set_num_threads(1)
    yield
    torch.set_num_threads(n)


def _replay(env, leaf_idx, n_episodes):
    """the body of evaluation_tools.evaluate (:9-41) for one env, with the leaf indices the reference's network chose"""
    out, traj = [], []
    obs = env.reset()
    for idx in leaf_idx:
        row = np.asarray(obs, dtype=np.float32).reshape(-1, 9)[80 + idx][0:6]  # torch.FloatTensor(obs) -> leaf_nodes[0, idx][0:6]
        items = env.packed
        traj.append(np.asarray(obs).copy())
        obs, reward, done, infos = env.step(row)
        if done:
            out.append((infos["ratio"], infos["counter"], [list(map(float, p)) for p in items]))
            obs = env.reset()
    assert len(out) == n_episodes
    return out, np.array(traj)


@pytest.mark.parametrize("setting", [1, 2, 3])
def test_reference_policy_and_eval_loop_on_the_drop_in_surface(setting):
    g = np.load(os.path.join(G, "policy_eval_s%d.npz" % setting))
    off = np.concatenate([[0], np.cumsum(g["packed_len"])])
    a = [(float(g["ratio"][e]), int(g["counter"][e]), g["packed_flat"][off[e]:off[e + 1]].tolist()) for e in range(len(g["ratio"]))]
    stream = make_stream(600 + setting, 0, 500, setting)
    b, tb = _replay(OracleDiscrete(setting, stream=stream), g["leaf_idx"], 4)
    assert np.array_equal(g["traj"], obs_digests(tb))
    assert [(x[0], x[1]) for x in a] == [(x[0], x[1]) for x in b] and [x[2] for x in a] == [x[2] for x in b]
    assert min(x[1] for x in a) >= 5  # the argmax policy of a random-init network still packs several items per episode


@pytest.mark.reference
@pytest.mark.skipif(not ref_shim.reference_available(), reason="reference not mounted")
def test_compat_runs_the_unmodified_evaluate(tmp_path):
    """pct_b200.compat: evaluation.py:10-56 around the UNMODIFIED evaluation_tools.evaluate (policy forward, env.step(row[0:6]), env.packed,
    trajs.npy, result.txt) — once on the reference env, once on an env with the facade's surface (oracle-backed here) — same files."""
    import os
    from importlib import import_module
    from make_eval_golden import dataset  # tests/golden (on sys.path through the lock-step module above or inserted here)
    compat = import_module("pct_b200.compat")
    D, _ = ref_shim.load_reference()
    data = dataset(1)[:7]
    ds = os.path.join(str(tmp_path), "set.pt")
    torch.save([t.tolist() for t in data], ds)
    args = compat.reference_args(ref_shim.REFERENCE_ROOT, ["--setting", "1", "--evaluate", "--no-cuda", "--load-dataset", "--dataset-path", ds,
                                                           "--evaluation-episodes", "5"])
    assert args.id == "PctDiscrete-v0" and args.num_processes == 1 and args.normFactor == 0.1
    model, _ = compat.load_policy_modules(ref_shim.REFERENCE_ROOT)
    torch.manual_seed(7)
    policy = model.DRL_GAT(args)
    ref_env = D.PackingDiscrete(setting=1, container_size=args.container_size, item_set=args.item_size_set, data_name=ds, load_test_data=True,
                                internal_node_holder=80, leaf_node_holder=50, LNES="EMS", shuffle=False)
    rows = []
    for t in data[1:]:
        rows += [np.concatenate([t, np.ones((len(t), 1))], 1), [[100, 100, 100, 1.0]]]
    ours = OracleDiscrete(1, stream=np.concatenate(rows))
    ours.set_trajectory_length(data.shape[1] + 1)
    outs = []
    for name, env in (("ref", ref_env), ("ours", ours)):
        work = os.path.join(str(tmp_path), name)
        os.makedirs(work)
        d = compat.reference_evaluate(ref_shim.REFERENCE_ROOT, args, env=env, policy=policy, custom=name, work_dir=work)
        trajs = np.load(os.path.join(d, "trajs.npy"), allow_pickle=True)
        outs.append(([[list(map(float, p)) for p in ep] for ep in trajs], open(os.path.join(d, "result.txt")).read()))
    assert outs[0] == outs[1] and len(outs[0][0]) == 5 and outs[0][1].startswith("Evaluation using 5 episodes")
    # env=None: compat builds the drop-in facade itself from `args` (evaluation.py:27-40); its batch is the oracle-backed stand-in here
    import importlib
    from fake_batch import FakeBatch
    envs_mod = importlib.import_module("pct_b200.envs")
    real = envs_mod.PctBatch
    envs_mod.PctBatch = FakeBatch
    try:
        work = os.path.join(str(tmp_path), "facade")
        os.makedirs(work)
        with pytest.warns(UserWarning, match="shuffle"):
            d = compat.reference_evaluate(ref_shim.REFERENCE_ROOT, args, policy=policy, custom="facade", work_dir=work)
    finally:
        envs_mod.PctBatch = real
    trajs = np.load(os.path.join(d, "trajs.npy"), allow_pickle=True)
    assert ([[list(map(float, p)) for p in ep] for ep in trajs], open(os.path.join(d, "result.txt")).read()) == outs[0]
