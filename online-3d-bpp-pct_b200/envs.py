"""Single-environment facades and factories with the reference's names and kwargs.

    PackingDiscrete / PackingContinuous   <->  pct_envs/PctDiscrete0/bin3D.py:8-188, pct_envs/PctContinuous0/bin3D.py:8-207
    make_vec_envs(args, log_dir, allow_early_resets)   <->  envs.py:75-116
    registration_envs()                                 <->  tools.py:232-240

The facades are a batch of ONE environment on the GPU in plain gym.Env mode (no auto-reset, float64
observations as the reference returns them), so `evaluation_tools.evaluate` (evaluation_tools.py:7-52) and the
heuristics' read-only attribute accesses work unchanged.  They exist for drop-in compatibility; throughput comes
from PctVecEnv / PctBatch.
"""
import copy

import numpy as np
import torch

from .batch import PctBatch
from .vec_env import PctVecEnv, _make_box


class _SpaceView(object):
    """The few `env.space.*` members external code reads (evaluation / heuristics): boxes, EMS, get_ratio()."""

    def __init__(self, env):
        self._env = env

    @property
    def boxes(self):
        return [tuple(b) for b in self._env._state()["boxes"]]

    @property
    def EMS(self):
        # integer rows in the discrete env (D:space.py:298: np.array([0, 0, 0, W, L, H])) — heuristic.py:50,115 slices arrays with them
        ems = self._env._state()["ems"]
        return [np.array(e) for e in ems] if self._env._continuous else [np.array(e).astype(np.int64) for e in ems]

    @property
    def plain_size(self):
        return np.array(self._env.bin_size)

    @property
    def plain(self):  # the height map (D:space.py:316-326)
        W, L = int(self._env.bin_size[0]), int(self._env.bin_size[1])
        return self._env._batch.query_placement(0, (1, 1, 0), 0, 0, want_map=True)[2][:W, :L]

    def drop_box_virtual(self, box_size, idx, flag, density, setting, returnH=False, returnMap=False):
        """D:space.py:393-433 — what heuristic.py asks for every placement it considers"""
        x, y, z = box_size if not flag else (box_size[1], box_size[0], box_size[2])
        res = self._env._batch.query_placement(0, (x, y, z), idx[0], idx[1], density=density, want_map=returnMap and not returnH)
        if returnH:
            return res[0], res[1]
        if returnMap:
            return res[0], res[2]
        return res[0]

    def get_ratio(self):  # D:space.py:334-339
        st = self._env._state()
        b = st["boxes"]
        vol = float(np.sum((b[:, 3] - b[:, 0]) * (b[:, 4] - b[:, 1]) * (b[:, 5] - b[:, 2]))) if len(b) else 0.0
        return vol / float(np.prod(self._env.bin_size))


class _PackingBase(object):
    _continuous = False
    metadata = {}
    spec = None
    action_space = None
    reward_range = (-float("inf"), float("inf"))

    def __init__(self, setting, container_size=(10, 10, 10), item_set=None, data_name=None, load_test_data=False,
                 internal_node_holder=80, leaf_node_holder=50, next_holder=1, shuffle=False, LNES="EMS",
                 sample_from_distribution=False, sample_left_bound=None, sample_right_bound=None, device=0, seed=0,
                 item_stream=None, size_minimum=None, **kwags):
        if next_holder != 1:
            raise NotImplementedError("next_holder must be 1 (reference default)")
        self._init_args = (setting, dict(container_size=container_size, item_set=item_set, data_name=data_name, load_test_data=load_test_data,
                                         internal_node_holder=internal_node_holder, leaf_node_holder=leaf_node_holder, next_holder=next_holder,
                                         shuffle=shuffle, LNES=LNES, sample_from_distribution=sample_from_distribution,
                                         sample_left_bound=sample_left_bound, sample_right_bound=sample_right_bound, device=device, seed=seed,
                                         item_stream=item_stream, size_minimum=size_minimum, **kwags))  # __deepcopy__ builds its twin from them
        self.internal_node_holder, self.leaf_node_holder, self.next_holder = internal_node_holder, leaf_node_holder, next_holder
        self.bin_size = container_size
        self.setting = setting
        self.item_set = item_set
        self.orientation = 6 if setting == 2 else 2
        self.test = load_test_data
        self.LNES = LNES
        self.shuffle = shuffle
        stream, traj_len = item_stream, 0
        if load_test_data:
            # LoadBoxCreator (binCreator.py:41-72): one trajectory per episode (reset() pre-increments the index, so
            # trajectory 0 is never used), each followed by the [100,100,100] sentinel that ends the episode.
            from .evaluation import load_trajectories, round3
            trajs = load_trajectories(data_name)[1:]  # torch.load(..., weights_only=False): the datasets are pickled lists (binCreator.py:48-49)
            if self._continuous:  # test mode rounds the item sizes to 3 decimals (C:bin3D.py:84-87)
                trajs = round3(trajs)
            traj_len = max(len(t) for t in trajs) + 1
            seq = np.full((len(trajs), traj_len, 4), 100.0)
            seq[:, :, 3] = 1.0
            for i, t in enumerate(trajs):
                seq[i, :len(t), :t.shape[1]] = t
            stream = seq.reshape(1, -1, 4)
        self._batch = PctBatch(1, setting, container_size=container_size, item_set=item_set, internal_node_holder=internal_node_holder,
                               leaf_node_holder=leaf_node_holder, continuous=self._continuous, obs_dtype=torch.float64, seed=seed,
                               device=device, sample_from_distribution=sample_from_distribution and self._continuous,
                               sample_left_bound=sample_left_bound, sample_right_bound=sample_right_bound, item_stream=stream,
                               size_minimum=size_minimum, auto_reset=False, LNES=LNES, shuffle=shuffle)
        if traj_len:
            self._batch.set_trajectory_length(traj_len)
        self.observation_space = _make_box(0.0, float(container_size[2]), (self._batch.obs_len,))
        self.space = _SpaceView(self)
        self.SEED = seed
        self._next_box_override = None

    # ---- gym.Env API ----
    def seed(self, seed=None):  # D:bin3D.py:47-54 (the item generator is counter-based: the seed is fixed at construction)
        return [seed]

    def reset(self):
        self._next_box_override = None
        return self._batch.reset().cpu().numpy()[0].copy()

    def step(self, action):
        a = np.asarray(action, dtype=np.float64).reshape(-1)
        if len(a) == 3:  # (rot, lx, ly) triples of the heuristics (heuristic.py:127,221,289): expand to a leaf row
            nb = self.next_box
            x, y = (nb[1], nb[0]) if a[0] else (nb[0], nb[1])
            a = np.array([a[1], a[2], 0, a[1] + x, a[2] + y, 0, 0, 0, 0], dtype=np.float64)
        row = np.zeros(9)
        row[:min(9, len(a))] = a[:9]
        nb = self.next_box  # reward in float64 like the reference: vol(item) / vol(bin) * 10 (D:bin3D.py:180-183)
        obs, rew, done, info = self._batch.step(actions=torch.from_numpy(row[None]).to(self._batch.device))
        self._next_box_override = None
        rec = PctBatch.decode_info(info)
        d = bool(done.cpu().numpy()[0])
        reward = 0.0 if d else (nb[0] * nb[1] * nb[2]) / (self.bin_size[0] * self.bin_size[1] * self.bin_size[2]) * 10  # C:bin3D.py:199-202 too
        out = {"counter": int(rec["counter"][0])}
        if d:
            ratio = self.space.get_ratio()
            out.update(ratio=ratio, reward=ratio * 10)
        if rec["flags"][0]:
            out["flags"] = int(rec["flags"][0])
        return obs.cpu().numpy()[0].copy(), reward, d, out

    def close(self):
        self._batch.close()

    def __deepcopy__(self, memo):
        """copy.deepcopy(env), as search / lookahead code does with the reference's plain-Python env: an independent env in the same state that
        continues exactly like this one under the same actions (a new batch of one with the same constructor arguments, reset, then loaded with
        this env's saved record).  The items drawn after the copy are the original's too (DESIGN.md 3(d): the copy follows the original's item
        sequence); with RandomBoxCreator the reference's copies share numpy's global RNG instead and do not replay."""
        setting, kw = self._init_args
        new = type(self).__new__(type(self))
        memo[id(self)] = new
        _PackingBase.__init__(new, setting, **kw)
        new._batch.reset()
        new._batch.load_envs(self._batch.save_envs())
        new._next_box_override = copy.deepcopy(self._next_box_override, memo)
        return new

    @property
    def unwrapped(self):
        return self

    # ---- attributes read by evaluation_tools.py:23 and heuristic.py ----
    def _state(self):
        return self._batch.state(0)

    @property
    def packed(self):
        b = self._state()["boxes"]
        if self._continuous:  # the state dump holds lo / hi corners; item sizes carry <= 6 decimals, so rounding the differences returns them
            return [[float(np.round(r[3] - r[0], 6)), float(np.round(r[4] - r[1], 6)), float(np.round(r[5] - r[2], 6)), r[0], r[1], r[2], 0] for r in b]
        return [[int(r[3] - r[0]), int(r[4] - r[1]), int(r[5] - r[2]), int(r[0]), int(r[1]), int(r[2]), 0] for r in b]

    @property
    def next_box(self):
        if self._next_box_override is not None:
            return list(self._next_box_override)
        nb = self._state()["next_box"]
        return list(nb) if self._continuous else [int(v) for v in nb]

    @next_box.setter
    def next_box(self, dims):  # heuristic.py:120 etc.: `env.next_box = [x, y, z]` (the chosen orientation) before env.step([0, lx, ly])
        self._next_box_override = list(dims)

    @property
    def next_den(self):
        return self._state()["next_den"]


class PackingDiscrete(_PackingBase):
    """Drop-in for pct_envs.PctDiscrete0.PackingDiscrete."""
    _continuous = False


class PackingContinuous(_PackingBase):
    """Drop-in for pct_envs.PctContinuous0.PackingContinuous — including its class defaults sample_from_distribution=True, U(0.1, 0.5)
    (C:bin3D.py:14-16), which set Space.low_bound = 0.1 even when a dataset supplies the items (heuristic.py:585-591 relies on them)."""
    _continuous = True

    def __init__(self, setting, container_size=(10, 10, 10), item_set=None, data_name=None, load_test_data=False,
                 internal_node_holder=80, leaf_node_holder=50, next_holder=1, shuffle=False,
                 sample_from_distribution=True, sample_left_bound=0.1, sample_right_bound=0.5, **kwags):
        super().__init__(setting, container_size=container_size, item_set=item_set, data_name=data_name, load_test_data=load_test_data,
                         internal_node_holder=internal_node_holder, leaf_node_holder=leaf_node_holder, next_holder=next_holder,
                         shuffle=shuffle, sample_from_distribution=sample_from_distribution, sample_left_bound=sample_left_bound,
                         sample_right_bound=sample_right_bound, **kwags)


def make_vec_envs(args, log_dir=None, allow_early_resets=True):
    """envs.make_vec_envs (envs.py:75-116) on the GPU: `args` is the namespace of tools.get_args()."""
    dev = getattr(args, "device", 0)
    dev = 0 if isinstance(dev, str) else int(dev)
    return PctVecEnv(args.num_processes, args.setting, container_size=args.container_size, item_set=args.item_size_set,
                     internal_node_holder=args.internal_node_holder, leaf_node_holder=args.leaf_node_holder,
                     continuous=getattr(args, "continuous", False) or str(getattr(args, "id", "")).startswith("PctContinuous"),
                     device=dev, seed=args.seed, sample_from_distribution=getattr(args, "sample_from_distribution", False),
                     sample_left_bound=getattr(args, "sample_left_bound", None), sample_right_bound=getattr(args, "sample_right_bound", None),
                     LNES=getattr(args, "lnes", "EMS"), shuffle=bool(getattr(args, "shuffle", False)))  # tools.py:136: --shuffle defaults to True


def registration_envs():
    """tools.registration_envs (tools.py:232-240): same ids, our entry points (no-op without gym)."""
    try:
        from gym.envs.registration import register
    except Exception:
        return False
    register(id="PctDiscrete-v0", entry_point="pct_b200.envs:PackingDiscrete")
    register(id="PctContinuous-v0", entry_point="pct_b200.envs:PackingContinuous")
    return True
