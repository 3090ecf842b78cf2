"""GPU: saved env records (pct_save_envs / pct_load_envs, PctBatch.save_envs / load_envs, the facades' __deepcopy__).  Every comparison is
bit-exact: a loaded env must continue exactly like its source — observation rows, reward, done, all eight pct_step_info fields — through
auto-resets, across handles, inside a captured graph, for the LSAH footprint and for a checkpoint restored into a fresh batch."""
import copy
import os

import numpy as np
import pytest
import torch

from harness import ITEM_SET

pytestmark = pytest.mark.gpu
CONT_STREAM_LEN = 160


def _stream(n, length, continuous, base=0, seed=11, rows=1024):
    """rows [base, base + n) of one global item stream (so that shards of it hold the same rows)"""
    rs = np.random.RandomState(seed)
    if continuous:
        g = np.round(rs.uniform(0.1, 0.5, size=(rows, length, 3)), 3)
    else:
        g = np.array(ITEM_SET, dtype=np.float64)[rs.randint(len(ITEM_SET), size=(rows, length))]
    d = np.round(rs.uniform(0.1, 1.0, size=(rows, length, 1)), 3)
    return np.concatenate([g, d], axis=2)[base:base + n]


def _batch(n, cfg, env_id_base=0, stream_base=0):
    import pct_b200
    kw = dict(cfg)
    traj = kw.pop("traj_len", 0)
    stream = kw.pop("stream", False)
    cont = kw.get("continuous", False)
    if stream:
        kw["item_stream"] = _stream(n, 120 if not cont else CONT_STREAM_LEN, cont, base=stream_base)
    elif not cont:
        kw.setdefault("item_set", ITEM_SET)
    if cont:
        kw.setdefault("container_size", (1.0, 1.0, 1.0))
        if not stream:
            kw["sample_from_distribution"] = True
    b = pct_b200.PctBatch(n, kw.pop("setting", 1), env_id_base=env_id_base, **kw)
    if traj:
        b.set_trajectory_length(traj)
    return b


def _rows(b, obs, idx, f64):
    """the leaf rows idx selects in obs, as (N, 9) action rows"""
    o = obs.view(b.n_envs, -1, 9)
    r = o[torch.arange(b.n_envs, device=o.device), b.nb + idx.long()]
    return r.to(torch.float64 if f64 else torch.float32).contiguous()


def _step(b, obs, idx, action):
    if action == "idx":
        return b.step(leaf_idx=idx)
    return b.step(actions=_rows(b, obs, idx, action == "f64"))


def _snap(res):
    return [x.clone() for x in res]


def _eq_rows(ra, da, rb, sb):
    for x, y in zip(ra, rb):
        assert torch.equal(x[da], y[sb])


def _state_eq(a, d, b, s):
    x, y = a.state(d), b.state(s)
    for k in x:
        assert np.array_equal(np.asarray(x[k]), np.asarray(y[k])), k


CASES = {
    "s1": dict(setting=1), "s2": dict(setting=2), "s3": dict(setting=3),
    "EP": dict(setting=1, LNES="EP"), "CP": dict(setting=1, LNES="CP"), "FC": dict(setting=1, LNES="FC"), "EV": dict(setting=1, LNES="EV"),
    "shuffle": dict(setting=1, shuffle=True), "stream_traj": dict(setting=1, stream=True, traj_len=40), "f64obs": dict(setting=1, obs_dtype=torch.float64),
    "rows_f32": dict(setting=1, action="f32"), "rows_f64": dict(setting=3, action="f64"),
    "c1": dict(setting=1, continuous=True), "c2": dict(setting=2, continuous=True), "c1_stream": dict(setting=1, continuous=True, stream=True),
}


@pytest.mark.parametrize("case", list(CASES))
def test_loaded_env_continues_like_its_source(case):
    cfg = dict(CASES[case])
    action = cfg.pop("action", "idx")
    n = 512
    a, t = _batch(n, cfg), _batch(n, cfg)  # t: twin of a that sees no load
    oa, ot = a.reset(), t.reset()
    for k in range(37):
        oa = _step(a, oa, a.random_policy(5, k), action)[0]
        ot = _step(t, ot, t.random_policy(5, k), action)[0]
    g = torch.Generator().manual_seed(3)
    perm = torch.randperm(n, generator=g)
    D = perm[:150].to(a.device)
    S = perm[150:][torch.randint(0, 60, (150,), generator=g)].to(a.device)  # repeats; disjoint from D
    rec = a.save_envs(S)
    for k in range(37, 37 + 20):  # the destinations get longer, different histories before the load
        oa = _step(a, oa, a.random_policy(9, k), action)[0]
    a.load_envs(rec, D, obs=oa)
    torch.cuda.synchronize()
    for d, s in zip(D.tolist()[:20], S.tolist()[:20]):
        _state_eq(a, d, t, s)
    for k in range(120):
        it = t.random_policy(7, k).clone()
        ia = a.random_policy(8, k).clone()
        ia[D] = it[S]
        rt = _snap(_step(t, ot, it, action))
        ra = _snap(_step(a, oa, ia, action))
        ot, oa = t._obs, a._obs
        _eq_rows(ra, D, rt, S)
        assert (ra[3][D, 1] == 0).all()  # no capacity / hand-over flags
    assert int(t.decode_info(rt[3])["ep_len"].max()) > 0


@pytest.mark.parametrize("stream", [False, True])
def test_records_move_between_handles(stream):
    cfg = dict(setting=1, stream=stream)
    src = _batch(64, cfg, env_id_base=0)
    base = 30 if stream else 1000
    dst, twin = _batch(300, cfg, env_id_base=base, stream_base=base), _batch(300, cfg, env_id_base=base, stream_base=base)
    os_, od, ow = src.reset(), dst.reset(), twin.reset()
    for k in range(25):
        os_ = src.step(leaf_idx=src.random_policy(1, k))[0]
        od = dst.step(leaf_idx=dst.random_policy(2, k))[0]
        ow = twin.step(leaf_idx=twin.random_policy(2, k))[0]
    D = torch.randperm(300, generator=torch.Generator().manual_seed(1))[:64].to(dst.device)
    status = torch.full((64,), -1, dtype=torch.int32, device=dst.device)
    dst.load_envs(src.save_envs(), D, check=False, status=status)
    st = status.cpu().numpy()
    ok = st == 0
    if stream:  # source envs 0..29 draw from rows that dst (rows 30..329) does not hold
        assert (st[:30] == 2).all() and ok[30:].all()
    else:
        assert ok.all()
    Dok, Sok = D[torch.from_numpy(ok).to(D.device)], torch.arange(64, device=D.device)[torch.from_numpy(ok).to(D.device)]
    Dno = D[torch.from_numpy(~ok).to(D.device)]
    for k in range(100):
        i_s = src.random_policy(3, k).clone()
        i_w = twin.random_policy(4, k).clone()
        i_d = i_w.clone()
        i_d[Dok] = i_s[Sok]
        rs, rd, rw = _snap(src.step(leaf_idx=i_s)), _snap(dst.step(leaf_idx=i_d)), _snap(twin.step(leaf_idx=i_w))
        _eq_rows(rd, Dok, rs, Sok)
        _eq_rows(rd, Dno, rw, Dno)  # rejected records left their envs untouched


@pytest.mark.parametrize("variant", ["setting", "container", "holders", "item_set", "seed", "alias"])
def test_incompatible_records_are_rejected(variant, monkeypatch):
    from pct_b200 import PctError
    base = dict(setting=1)
    other = dict(base)
    if variant == "setting":
        other["setting"] = 3
    elif variant == "container":
        other["container_size"] = (10, 10, 12)
    elif variant == "holders":
        other["internal_node_holder"] = 60
    elif variant == "item_set":
        other["item_set"] = ITEM_SET[:-1]
    elif variant == "seed":
        other["seed"] = 1
    src = _batch(32, other if variant != "alias" else base)
    if variant == "alias":
        monkeypatch.setenv("PCT_B200_ALIAS", "0")
    dst, twin = _batch(32, base), _batch(32, base)
    src.reset(), dst.reset(), twin.reset()
    for k in range(10):
        src.step(leaf_idx=src.random_policy(1, k))
        dst.step(leaf_idx=dst.random_policy(2, k))
        twin.step(leaf_idx=twin.random_policy(2, k))
    rec = src.save_envs()
    status = torch.full((32,), -1, dtype=torch.int32, device=dst.device)
    dst.load_envs(rec, check=False, status=status)
    assert (status.cpu() == 1).all()
    with pytest.raises(PctError, match="rejected 32 of 32"):
        dst.load_envs(rec)
    for k in range(40):
        rd, rw = _snap(dst.step(leaf_idx=dst.random_policy(5, k))), _snap(twin.step(leaf_idx=twin.random_policy(5, k)))
        for x, y in zip(rd, rw):
            assert torch.equal(x, y)


@pytest.mark.parametrize("continuous", [False, True])
def test_observation_on_load_and_delta_rows(continuous, monkeypatch):
    cfg = dict(setting=1, continuous=continuous, auto_reset=False)
    monkeypatch.setenv("PCT_B200_OBS_DELTA", "1")
    a = _batch(96, cfg)
    monkeypatch.setenv("PCT_B200_OBS_DELTA", "0")
    full = _batch(96, cfg)
    oa, of = a.reset(), full.reset()
    done_seen = torch.zeros(96, dtype=torch.bool, device=a.device)
    for k in range(60):  # no auto-reset: finished envs keep returning their terminal observation
        oa, _, da, _ = a.step(leaf_idx=a.random_policy(1, k))
        of = full.step(leaf_idx=full.random_policy(1, k))[0]
        done_seen |= da.bool()
    assert done_seen.any()
    last = oa.clone()
    S = torch.arange(96, device=a.device).flip(0)  # every env takes its mirror's state (terminal ones included)
    rec = a.save_envs(S)
    buf = torch.zeros_like(oa)
    b2 = _batch(96, cfg)
    b2.reset()
    b2.load_envs(rec, obs=buf)
    assert torch.equal(buf, last[S])
    # delta rows: load into the tracked buffer of `a`, the next step equals the full-rewrite twin loaded the same way
    a.load_envs(rec, obs=oa)
    full.load_envs(full.save_envs(S))
    for k in range(30):
        ra, rf = _snap(a.step(leaf_idx=a.random_policy(2, k))), _snap(full.step(leaf_idx=full.random_policy(2, k)))
        for x, y in zip(ra, rf):
            assert torch.equal(x, y)


def test_graph_capture_of_save_load_step():
    n = 256
    a, b = _batch(n, dict(setting=1)), _batch(n, dict(setting=1))
    a.reset(), b.reset()
    for k in range(20):
        a.step(leaf_idx=a.random_policy(1, k))
        b.step(leaf_idx=b.random_policy(1, k))
    S = torch.randint(0, n // 2, (n // 2,), device=a.device, generator=torch.Generator(device=a.device).manual_seed(2))
    D = torch.arange(n // 2, n, device=a.device)
    idx = torch.randint(0, 4, (n,), dtype=torch.int32, device=a.device)
    rec = torch.empty((n // 2, a.record_bytes), dtype=torch.uint8, device=a.device)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        a.step(leaf_idx=idx)  # warm-up outside the capture
        b.step(leaf_idx=idx)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            a.save_envs(S, out=rec)
            a.load_envs(rec, D, check=False)
            out_a = a.step(leaf_idx=idx)
    torch.cuda.current_stream().wait_stream(s)
    for r in range(3):
        g.replay()
        b.load_envs(b.save_envs(S), D)
        out_b = b.step(leaf_idx=idx)
        torch.cuda.synchronize()
        for x, y in zip(out_a, out_b):
            assert torch.equal(x, y)


@pytest.mark.parametrize("continuous", [False, True])
def test_lsah_footprint_carries_over(continuous):
    n = 128
    a = _batch(n, dict(setting=1, continuous=continuous))
    a.reset()
    for k in range(6):
        a.step(actions=a.heuristic_actions("LSAH").clone())
    S, D = torch.arange(0, 32, device=a.device), torch.arange(64, 96, device=a.device)
    a.load_envs(a.save_envs(S), D)
    ended = torch.zeros(32, dtype=torch.bool, device=a.device)
    for k in range(40):
        rows = a.heuristic_actions("LSAH").clone()
        live = ~ended
        assert torch.equal(rows[D][live], rows[S][live])
        done = a.step(actions=rows)[2].bool()
        ended |= done[S]
    assert ended.any()


def test_checkpoint_and_resume():
    cfg = dict(setting=1)
    a = _batch(200, cfg)
    a.reset()
    for k in range(30):
        a.step(leaf_idx=a.random_policy(1, k))
    rec = a.save_envs().cpu()  # e.g. written to disk
    b = _batch(200, cfg)
    b.reset()
    b.load_envs(rec)
    for k in range(200):
        ra, rb = _snap(a.step(leaf_idx=a.random_policy(2, k))), _snap(b.step(leaf_idx=b.random_policy(2, k)))
        for x, y in zip(ra, rb):
            assert torch.equal(x, y)


@pytest.mark.parametrize("kind", ["discrete", "continuous", "discrete_dataset", "continuous_dataset"])
def test_facade_deepcopy(kind, tmp_path):
    import pct_b200
    if kind.endswith("dataset"):
        g = np.load(os.path.join(os.path.dirname(__file__), "golden", "eval_cont_s1.npz" if kind.startswith("cont") else "eval_s1.npz"))
        ds = os.path.join(str(tmp_path), "set.pt")
        torch.save([t.tolist() for t in g["data"]], ds)
        kw = dict(data_name=ds, load_test_data=True)
    else:
        kw = dict(seed=4)
    if kind.startswith("cont"):
        env = pct_b200.PackingContinuous(setting=1, container_size=[1, 1, 1], **kw)
    else:
        env = pct_b200.PackingDiscrete(setting=1, container_size=[10, 10, 10], item_set=ITEM_SET, **kw)
    rs = np.random.RandomState(0)

    def run(e, obs, rng, steps):
        out = []
        for _ in range(steps):
            leaves = obs.reshape(-1, 9)[80:130]
            v = np.nonzero(leaves[:, 8] == 1)[0]
            obs, r, d, _ = e.step(leaves[v[rng.randint(len(v))]] if len(v) else np.zeros(9))
            out.append((obs.copy(), r, d))
            if d:
                obs = e.reset()
        return out, obs

    _, obs = run(env, env.reset(), rs, 9)
    twin, other = copy.deepcopy(env), copy.deepcopy(env)
    run(other, obs, np.random.RandomState(5), 20)  # stepping one copy leaves the others unchanged
    a, _ = run(env, obs, np.random.RandomState(1), 40)
    b, _ = run(twin, obs, np.random.RandomState(1), 40)
    for (x, r, d), (y, q, e) in zip(a, b):
        assert np.array_equal(x, y) and r == q and d == e
