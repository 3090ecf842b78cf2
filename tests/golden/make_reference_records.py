"""Records of the UNMODIFIED reference that the reference-comparison tests replay (needs the reference checkout, see oracle/ref_shim.py):

    lockstep_s{1,2,3}.npz              tests/test_oracle_vs_reference.py::test_lockstep_with_reference
    lockstep_case_*.npz / _ccase_*.npz    ::test_cases_lockstep_with_reference / ::test_continuous_cases_lockstep_with_reference
    lapack_tie.npz                        ::test_the_known_divergence_is_lapack_rounding_at_a_geometric_tie
    hull_pip.npz                       tests/test_oracle_units.py::test_hull_and_pip_match_reference_module
    policy_eval_s{1,2,3}.npz           tests/test_reference_policy_contract.py::test_reference_policy_and_eval_loop_on_the_drop_in_surface
    vecenv_s{1,2}.npz                  tests/test_host_logic.py::test_vec_env_equals_reference_shmem_vecpytorch_monitor
    reference_args.json                tests/test_host_logic.py::test_make_vec_envs_takes_the_reference_args

Each record holds what the test used to take from the live reference: its observations (as SHA-256 digests, tests/harness.py obs_digest),
rewards, done flags and infos on the test's item streams and policy, and for the policy-facing test the leaf indices the reference's network
chose.

    python tests/golden/make_reference_records.py
"""
import importlib
import json
import os
import sys
import tempfile
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests"), HERE]
import ref_shim  # noqa: E402
from harness import CASES, CONT_CASES, ITEM_SET, case_stream, make_stream, obs_digests, policy_pick  # noqa: E402


def _save(name, **arrays):
    path = os.path.join(HERE, name)
    np.savez_compressed(path, **arrays)
    print(path, os.path.getsize(path) // 1024, "KiB", flush=True)


def _info_arrays(infos):
    """info dicts -> counter, ratio and reward arrays (-1 / nan where the key is absent)"""
    return dict(counter=np.array([i["counter"] for i in infos]), ratio=np.array([i.get("ratio", -1.0) for i in infos]),
                info_reward=np.array([i.get("reward", np.nan) for i in infos]), info_keys=np.array([",".join(sorted(i)) for i in infos]))


def record_lockstep(D, setting):
    seed, env_id, steps = 900 + setting, 3, 260
    stream = make_stream(seed, env_id, steps + 64, setting)
    ref = D.PackingDiscrete(setting=setting, container_size=[10, 10, 10], item_set=ITEM_SET, internal_node_holder=80,
                            leaf_node_holder=50, shuffle=False, LNES="EMS")
    ref.box_creator = ref_shim.make_stream_creator(D, [tuple(r) if setting == 3 else tuple(int(v) for v in r[:3]) for r in stream])
    ref.test = True
    o = ref.reset()
    pre, post, rew, done, infos = [], [], [], [], []
    for t in range(steps):
        pre.append(o.copy())
        _, row = policy_pick(o, 80, 50, seed, env_id, t)
        o, r, d, i = ref.step(row)
        post.append(o.copy()); rew.append(r); done.append(d); infos.append(i)
        if d:
            o = ref.reset()
    _save("lockstep_s%d.npz" % setting, pre_obs=obs_digests(pre), post_obs=obs_digests(post), reward=np.array(rew), done=np.array(done),
          **_info_arrays(infos))


def record_cases(D, Cm):
    import make_golden_cases as M
    def slim(rec):  # the tests draw the stream themselves
        rec.pop("stream")
        return dict(rec, obs=obs_digests(rec["obs"]))

    for name in sorted(CASES):
        _save("lockstep_case_%s.npz" % name, **slim(M.record_case(D, dict(CASES[name], steps=60), 8800, 4)))
    for name in sorted(CONT_CASES):
        _save("lockstep_ccase_%s.npz" % name, **slim(M.record_cont_case(Cm, dict(CONT_CASES[name], steps=70), 8801, 5)))


def record_lapack_tie(D):
    """the 47 steps before the tie, the least-squares system of the tie and the reference's verdicts with LAPACK's and the oracle's solution"""
    from pct_oracle import _dp, lib
    import pct_envs.PctDiscrete0.space as SP
    c, seed, env_id = CASES["holders_s1"], 135409, 0
    stream = case_stream(c, seed, env_id, 200)
    ref = D.PackingDiscrete(setting=1, container_size=[10, 10, 10], item_set=c["items"], internal_node_holder=c["nb"], leaf_node_holder=c["nl"],
                            shuffle=False, LNES="EMS")
    ref.box_creator = ref_shim.make_stream_creator(D, [tuple(int(v) for v in r[:3]) for r in stream])
    ref.test = True
    o = ref.reset()
    obs = [o.copy()]
    for t in range(47):
        _, row = policy_pick(o, c["nb"], c["nl"], seed, env_id, t)
        o, _, d, _ = ref.step(row)
        if d:
            o = ref.reset()
        obs.append(o.copy())
    lapack, L = np.linalg.lstsq, lib()
    systems = []

    def recording(A, b, rcond=None):
        r = lapack(A, b, rcond=rcond)
        systems.append((np.array(A, dtype=float), np.array(b, dtype=float).reshape(-1), r[0].reshape(-1).copy()))
        return r

    def with_oracle_solver(A, b, rcond=None):
        r = lapack(A, b, rcond=rcond)
        x = np.zeros(A.shape[1])
        L.pcto_lstsq(_dp(np.ascontiguousarray(A, dtype=float)), A.shape[0], A.shape[1], _dp(np.ascontiguousarray(np.array(b, dtype=float).reshape(-1))), _dp(x))
        return (x.reshape(-1, 1),) + tuple(r[1:])

    args = ([4, 2, 1], (5, 0), False, ref.next_den, 1)
    verdicts = []
    for solver in (recording, with_oracle_solver):
        SP.np.linalg.lstsq = solver
        try:
            verdicts.append(bool(ref.space.drop_box_virtual(*args)))
        finally:
            SP.np.linalg.lstsq = lapack
    assert len(systems) == 1
    A, b, x = systems[0]
    _save("lapack_tie.npz", obs=obs_digests(obs), A=A, b=b, x_lapack=x, verdict_lapack=verdicts[0], verdict_oracle_solver=verdicts[1])


def record_hull_pip(D):
    from pct_envs.PctDiscrete0.convex_hull import ConvexHull, point_in_polygen
    from pct_envs.PctDiscrete0.space import Space
    sp = Space(10, 10, 10, 1, 80)
    rng = np.random.RandomState(3)
    hulls, lens, pip = [], [], []
    for trial in range(600):  # the draw order of tests/test_oracle_units.py::test_hull_and_pip_match_reference_module
        k = rng.choice([1, 1, 2, 2, 3, 4, 6])
        pts = []
        for _ in range(k):
            x1, y1 = rng.randint(0, 8, 2); x2, y2 = x1 + rng.randint(1, 4), y1 + rng.randint(1, 4)
            pts += [[x1, y1], [x1, y2], [x2, y1], [x2, y2]]
        want = np.array(sp.scale_down(ConvexHull([list(p) for p in pts])), dtype=np.float64).reshape(-1, 2)
        hulls.append(want); lens.append(len(want))
        for _ in range(6):
            q = np.array([rng.randint(0, 20) / 2.0, rng.randint(0, 20) / 2.0]) if rng.rand() < 0.5 else rng.uniform(0, 10, 2)
            pip.append(bool(point_in_polygen(q, want.tolist())))
    _save("hull_pip.npz", hull_len=np.array(lens), hull_flat=np.concatenate(hulls), pip=np.array(pip))


def record_policy_eval(D, setting):
    """the reference's DRL_GAT (seed 1234 + setting) in the body of evaluation_tools.evaluate on the reference env: observations, chosen leaf
    indices, per-episode (ratio, counter, packed)"""
    import torch
    torch.set_num_threads(1)
    model, tools = ref_shim.load_policy_module()
    a = types.SimpleNamespace(embedding_size=64, hidden_size=128, gat_layer_num=1, internal_node_holder=80,
                              internal_node_length=7 if setting == 3 else 6, leaf_node_holder=50)
    torch.manual_seed(1234 + setting)
    policy = model.DRL_GAT(a).eval()
    stream = make_stream(600 + setting, 0, 500, setting)
    env = D.PackingDiscrete(setting=setting, container_size=[10, 10, 10], item_set=ITEM_SET, internal_node_holder=80, leaf_node_holder=50,
                            shuffle=False, LNES="EMS")
    env.box_creator = ref_shim.make_stream_creator(D, [tuple(r) if setting == 3 else tuple(int(v) for v in r[:3]) for r in stream])
    env.test = True
    out, traj, leaf_idx = [], [], []
    obs = env.reset()
    while len(out) < 4:
        obs_t = torch.FloatTensor(obs).unsqueeze(dim=0)
        all_nodes, leaf_nodes = tools.get_leaf_nodes_with_factor(obs_t, 1, 80, 50)
        with torch.no_grad():
            _, idx, _, _ = policy(all_nodes, True, normFactor=0.1)
        row = leaf_nodes[torch.arange(1), idx.squeeze()].cpu().numpy()[0][0:6]
        items = env.packed
        traj.append(np.asarray(obs).copy()); leaf_idx.append(int(idx.squeeze()))
        obs, reward, done, infos = env.step(row)
        if done:
            out.append((infos["ratio"], infos["counter"], [list(map(float, p)) for p in items]))
            obs = env.reset()
    _save("policy_eval_s%d.npz" % setting, traj=obs_digests(traj), leaf_idx=np.array(leaf_idx), ratio=np.array([x[0] for x in out]),
          counter=np.array([x[1] for x in out]), packed_len=np.array([len(x[2]) for x in out]),
          packed_flat=np.array([p for x in out for p in x[2]], dtype=np.float64))


def record_vec_env(D, setting):
    """VecPyTorch(ShmemVecEnv([Monitor(PackingDiscrete)] * 5, context='fork')) of the reference over 70 vector steps"""
    import torch
    renvs = importlib.import_module("envs")
    ShmemVecEnv = importlib.import_module("wrapper.shmem_vec_env").ShmemVecEnv
    Monitor = importlib.import_module("wrapper.monitor").Monitor
    n, seed = 5, 50 + setting
    streams = np.stack([make_stream(seed, e, 300, setting) for e in range(n)])
    tmp = tempfile.TemporaryDirectory()  # Monitor's csv files

    def thunk(rank):
        def _t():
            env = D.PackingDiscrete(setting=setting, container_size=[10, 10, 10], item_set=ITEM_SET, internal_node_holder=80, leaf_node_holder=50,
                                    shuffle=False, LNES="EMS")
            env.box_creator = ref_shim.make_stream_creator(D, [tuple(int(v) for v in r[:3]) for r in streams[rank]])
            env.test = True
            return Monitor(env, os.path.join(tmp.name, str(rank)), allow_early_resets=True)
        return _t

    probe = D.PackingDiscrete(setting=setting, container_size=[10, 10, 10], item_set=ITEM_SET)
    ref = renvs.VecPyTorch(ShmemVecEnv([thunk(r) for r in range(n)], [probe.observation_space, probe.action_space], context="fork"), "cpu")
    obs, rew, done, infos = [], [], [], []
    try:
        o = ref.reset()
        assert o.dtype == torch.float32
        obs.append(o.numpy().copy())
        for t in range(70):
            rows = np.stack([policy_pick(o[e].numpy().astype(np.float64), 80, 50, seed, e, t)[1] for e in range(n)]).astype(np.float32)
            o, r, d, i = ref.step(rows)
            assert r.dtype == torch.float32 and d.dtype == np.bool_
            obs.append(o.numpy().copy()); rew.append(r.numpy().copy()); done.append(d.copy()); infos.append(i)
    finally:
        ref.close()
        tmp.cleanup()
    flat = [i for step in infos for i in step]
    ep = [i.get("episode", {}) for i in flat]
    arr = _info_arrays(flat)
    arr = {k: v.reshape(70, n) for k, v in arr.items()}
    _save("vecenv_s%d.npz" % setting, obs=np.stack([obs_digests(o) for o in obs]), reward=np.array(rew), done=np.array(done),
          ep_l=np.array([e.get("l", -1) for e in ep]).reshape(70, n), ep_r=np.array([e.get("r", np.nan) for e in ep]).reshape(70, n), **arr)


ARGVS = {"discrete": ["--setting", "1", "--num-processes", "6", "--seed", "9"],
         "continuous": ["--setting", "2", "--continuous", "--sample-from-distribution", "--num-processes", "4"]}


def record_reference_args():
    """tools.get_args() of the reference on the argument lists of test_make_vec_envs_takes_the_reference_args"""
    compat = importlib.import_module("pct_b200.compat")
    out = {}
    for key, argv in ARGVS.items():
        ns = vars(compat.reference_args(ref_shim.REFERENCE_ROOT, argv))
        out[key] = {"argv": argv, "args": ns}
    path = os.path.join(HERE, "reference_args.json")
    with open(path, "w") as f:
        json.dump(out, f, sort_keys=True)
        f.write("\n")
    print(path, flush=True)


def main():
    D, Cm = ref_shim.load_reference()
    for s in (1, 2, 3):
        record_lockstep(D, s)
    record_cases(D, Cm)
    record_lapack_tie(D)
    record_hull_pip(D)
    for s in (1, 2, 3):
        record_policy_eval(D, s)
    for s in (1, 2):
        record_vec_env(D, s)
    record_reference_args()


if __name__ == "__main__":
    main()
