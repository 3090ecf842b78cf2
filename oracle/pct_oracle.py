"""TEST INFRASTRUCTURE — ctypes binding of the CPU oracle (oracle/_build/libpct_oracle.so).

Only tests/, __graft_entry__.smoke() and bench.py (cpu_baseline / --impl reference) may import this.
The product path (pct_b200) never does.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "_build", "libpct_oracle.so")


def build(force=False):
    srcs = [os.path.join(_HERE, f) for f in os.listdir(_HERE) if f.endswith((".c", ".h"))]
    if force or not os.path.exists(_LIB) or any(os.path.getmtime(s) > os.path.getmtime(_LIB) for s in srcs):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return _LIB


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB)
        dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int)
        L.pcto_create.restype = C.c_void_p
        L.pcto_create.argtypes = [C.c_int] * 6 + [C.c_double]
        L.pcto_destroy.argtypes = [C.c_void_p]
        L.pcto_set_stream.argtypes = [C.c_void_p, dp, C.c_int]
        L.pcto_obs_len.argtypes = [C.c_void_p]
        L.pcto_reset.argtypes = [C.c_void_p, dp]
        L.pcto_step.argtypes = [C.c_void_p, dp, C.c_int, dp, dp, ip, dp]
        L.pcto_get_ems.argtypes = [C.c_void_p, ip, C.c_int]
        L.pcto_get_candidates.argtypes = [C.c_void_p, ip, ip, C.c_int]
        L.pcto_get_packed.argtypes = [C.c_void_p, ip, C.c_int]
        for f in ("pcto_n_lstsq", "pcto_n_boxes", "pcto_stream_pos"):
            getattr(L, f).argtypes = [C.c_void_p]
        L.pcto_set_order6.argtypes = [C.POINTER(C.c_int64), C.c_int, ip]
        L.pcto_hull_shrunk.argtypes = [dp, C.c_int, dp]
        L.pcto_pip.argtypes = [C.c_double, C.c_double, dp, C.c_int]
        L.pcto_lstsq.argtypes = [dp, C.c_int, C.c_int, dp, dp]
        L.pcto_hash_double.argtypes = [C.c_double]
        L.pcto_hash_double.restype = C.c_uint64
        _lib = L
    return _lib


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int))


class OracleDiscrete(object):
    """Single discrete env, same call surface as the reference's PackingDiscrete
    (pct_envs/PctDiscrete0/bin3D.py:8-188) restricted to LNES='EMS', shuffle=False and an injected
    item stream (array (n,4): x, y, z, density)."""

    def __init__(self, setting, container_size=(10, 10, 10), internal_node_holder=80, leaf_node_holder=50,
                 size_minimum=1, stream=None, lnes="EMS"):
        self.L = lib()
        self.h = self.L.pcto_create(setting, *[int(c) for c in container_size], internal_node_holder,
                                    leaf_node_holder, float(size_minimum))
        self.L.pcto_set_lnes.argtypes = [C.c_void_p, C.c_int]
        self.L.pcto_set_lnes(self.h, {"EMS": 0, "EV": 1, "EP": 2, "CP": 3, "FC": 4}[lnes])
        self.nb, self.nl = internal_node_holder, leaf_node_holder
        self.obs_len = self.L.pcto_obs_len(self.h)
        self.container, self.setting = tuple(int(c) for c in container_size), int(setting)
        self._stream = None
        if stream is not None:
            self.set_stream(stream)

    def set_stream(self, stream):
        s = np.ascontiguousarray(stream, dtype=np.float64)
        if s.shape[1] == 3:
            s = np.concatenate([s, np.ones((len(s), 1))], axis=1)
        self._stream = np.ascontiguousarray(s)
        self.L.pcto_set_stream(self.h, _dp(self._stream), len(self._stream))

    def set_alias_mode(self, on=True):
        """read the up_edges values that ARE the upper box's own Stack object live, like the reference's Python objects (DESIGN.md section 3)"""
        self.L.pcto_set_alias_mode.argtypes = [C.c_void_p, C.c_int]
        self.L.pcto_set_alias_mode(self.h, int(on))

    def set_shuffle(self, seed, gid, on=True):
        """shuffle=True (D:bin3D.py:114-115) with the product's keyed permutation: stable argsort of rnd_u64(seed ^ SALT, gid, draws << 16 | i)"""
        self.L.pcto_set_shuffle.argtypes = [C.c_void_p, C.c_int, C.c_uint64, C.c_uint64]
        self.L.pcto_set_shuffle(self.h, int(on), int(seed) & ((1 << 64) - 1), int(gid))

    def set_random_items(self, item_set, seed, gid):
        """RandomBoxCreator draws from the counter-based generator the device uses (item_set[rnd(seed, gid, d) % n], density for setting 3)"""
        self._items = np.ascontiguousarray(np.array(item_set, dtype=np.float64).reshape(-1, 3))
        self.L.pcto_set_random_items.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.c_int, C.c_uint64, C.c_uint64]
        self.L.pcto_set_random_items(self.h, _dp(self._items), len(self._items), int(seed), int(gid))

    def set_trajectory_length(self, n):
        self.L.pcto_set_trajectory_length.argtypes = [C.c_void_p, C.c_int]
        self.L.pcto_set_trajectory_length(self.h, int(n))

    def reset(self):
        obs = np.zeros(self.obs_len)
        self.L.pcto_reset(self.h, _dp(obs))
        return obs

    def step(self, action):
        a = np.ascontiguousarray(action, dtype=np.float64)
        obs = np.zeros(self.obs_len)
        rew = C.c_double()
        done = C.c_int()
        info = np.zeros(3)
        err = self.L.pcto_step(self.h, _dp(a), len(a), _dp(obs), C.byref(rew), C.byref(done), _dp(info))
        d = {"counter": int(info[0])}
        if done.value:
            d.update(ratio=float(info[1]), reward=float(info[2]))
        if err:
            d["error"] = err
        return obs, rew.value, bool(done.value), d

    def ems(self):
        buf = np.zeros((4096, 6), dtype=np.int32)
        n = self.L.pcto_get_ems(self.h, _ip(buf), 4096)
        return buf[:n].copy()

    def candidates(self):
        buf = np.zeros((8192, 6), dtype=np.int32)
        feas = np.zeros(8192, dtype=np.int32)
        n = self.L.pcto_get_candidates(self.h, _ip(buf), _ip(feas), 8192)
        return buf[:n].copy(), feas[:n].copy()

    @property
    def packed(self):
        buf = np.zeros((256, 7), dtype=np.int32)
        n = self.L.pcto_get_packed(self.h, _ip(buf), 256)
        return buf[:n].tolist()

    # -- what the heuristic baselines read from the env (heuristic.py): space.drop_box_virtual(returnH), space.plain, next_box/den
    def drop_box_virtual(self, dims, lx, ly):
        mh = C.c_int()
        self.L.pcto_drop_box_virtual.argtypes = [C.c_void_p] + [C.c_int] * 5 + [C.c_double, C.POINTER(C.c_int)]
        ok = self.L.pcto_drop_box_virtual(self.h, int(dims[0]), int(dims[1]), int(dims[2]), int(lx), int(ly), self.next_den, C.byref(mh))
        return bool(ok), mh.value

    def plain(self):
        buf = np.zeros((self.container[0], self.container[1]), dtype=np.int32)
        self.L.pcto_get_plain.argtypes = [C.c_void_p, C.POINTER(C.c_int)]
        self.L.pcto_get_plain(self.h, _ip(buf))
        return buf

    def _next(self):
        out = np.zeros(4)
        self.L.pcto_get_next.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
        self.L.pcto_get_next(self.h, _dp(out))
        return out

    @property
    def next_box(self):
        return [int(v) for v in self._next()[:3]]

    @property
    def next_den(self):
        return float(self._next()[3])

    @property
    def n_lstsq(self):
        return self.L.pcto_n_lstsq(self.h)

    @property
    def stream_pos(self):
        return self.L.pcto_stream_pos(self.h)

    def __del__(self):
        try:
            self.L.pcto_destroy(self.h)
        except Exception:
            pass


# ---- shared deterministic test policy / item streams -------------------------------------------
M64 = (1 << 64) - 1


def splitmix64(x):
    x = (x + 0x9E3779B97F4A7C15) & M64
    z = x
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def rnd_u64(seed, a, b):
    """Counter-based generator shared by host tests, the oracle harness and the device code
    (csrc/pct_rng.cuh): splitmix64(splitmix64(seed ^ a*GOLD) + b)."""
    return splitmix64((splitmix64((seed ^ (a * 0x9E3779B97F4A7C15)) & M64) + b) & M64)


def policy_pick(obs, nb, nl, seed, env, t):
    """Uniform choice among valid leaf rows (all-zero leaf row if none): returns (index, row)."""
    leaf = obs.reshape(-1, 9)[nb:nb + nl]
    nvalid = int((leaf[:, 8] == 1).sum())
    if nvalid == 0:
        return 0, np.zeros(9)
    k = rnd_u64(seed, env, t) % nvalid
    return int(k), leaf[k].copy()


class OracleBatch(object):
    """N oracle envs stepped by host threads with the synthetic policy (oracle/pct_oracle_batch.c)."""

    def __init__(self, n_envs, setting, item_set, item_seed, policy_seed, container_size=(10, 10, 10), nb=80, nl=50,
                 size_minimum=1, gid_base=0, threads=None):
        L = lib()
        L.pcto_batch_create.restype = C.c_void_p
        L.pcto_batch_create.argtypes = [C.c_int] * 6 + [C.c_double, C.POINTER(C.c_double), C.c_int, C.c_uint64, C.c_uint64,
                                                          C.c_int64, C.c_int, C.c_int]
        L.pcto_batch_run.restype = C.c_double
        L.pcto_batch_run.argtypes = [C.c_void_p, C.c_int]
        L.pcto_batch_get.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int)]
        L.pcto_batch_destroy.argtypes = [C.c_void_p]
        self.L = L
        self.n, self.obs_len = n_envs, (nb + nl + 1) * 9
        self.threads = threads or os.cpu_count() or 1
        its = np.ascontiguousarray(np.array(item_set, dtype=np.float64).reshape(-1, 3))
        self.h = L.pcto_batch_create(setting, int(container_size[0]), int(container_size[1]), int(container_size[2]), nb, nl,
                                     float(size_minimum), _dp(its), len(its), item_seed, policy_seed, gid_base, n_envs, self.threads)

    def run(self, steps):
        """returns elapsed seconds for `steps` vector steps"""
        return self.L.pcto_batch_run(self.h, steps)

    def get(self):
        obs = np.zeros((self.n, self.obs_len))
        rew = np.zeros(self.n)
        nd = np.zeros(self.n, dtype=np.int32)
        self.L.pcto_batch_get(self.h, _dp(obs), _dp(rew), _ip(nd))
        return obs, rew, nd

    def close(self):
        if self.h:
            self.L.pcto_batch_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class OracleBatchContinuous(object):
    """N continuous oracle envs (sample_from_distribution items, C:bin3D.py:103-115) stepped by host threads with the synthetic
    policy (oracle/pct_oracle_batch_continuous.c): BASELINE config 4 on the host cores."""

    def __init__(self, n_envs, setting, item_seed, policy_seed, container_size=(1.0, 1.0, 1.0), nb=80, nl=50, lo=0.1, hi=0.5, gid_base=0,
                 threads=None):
        L = lib()
        L.pctc_batch_create.restype = C.c_void_p
        L.pctc_batch_create.argtypes = [C.c_int, C.c_double, C.c_double, C.c_double, C.c_int, C.c_int, C.c_double, C.c_double, C.c_uint64,
                                        C.c_uint64, C.c_int64, C.c_int, C.c_int]
        L.pctc_batch_run.restype = C.c_double
        L.pctc_batch_run.argtypes = [C.c_void_p, C.c_int]
        L.pctc_batch_get.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int)]
        L.pctc_batch_destroy.argtypes = [C.c_void_p]
        self.L = L
        self.n, self.obs_len = n_envs, (nb + nl + 1) * 9
        self.threads = threads or os.cpu_count() or 1
        self.h = L.pctc_batch_create(setting, float(container_size[0]), float(container_size[1]), float(container_size[2]), nb, nl, float(lo),
                                     float(hi), item_seed, policy_seed, gid_base, n_envs, self.threads)

    def run(self, steps):
        """returns elapsed seconds for `steps` vector steps"""
        return self.L.pctc_batch_run(self.h, steps)

    def get(self):
        obs = np.zeros((self.n, self.obs_len))
        rew = np.zeros(self.n)
        nd = np.zeros(self.n, dtype=np.int32)
        self.L.pctc_batch_get(self.h, _dp(obs), _dp(rew), _ip(nd))
        return obs, rew, nd

    def close(self):
        if self.h:
            self.L.pctc_batch_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class OracleContinuous(object):
    """Single continuous env (pct_envs/PctContinuous0/bin3D.py:8-207), float64 actions, injected item stream."""

    def __init__(self, setting, container_size=(1.0, 1.0, 1.0), internal_node_holder=80, leaf_node_holder=50,
                 size_minimum=0.1, stream=None):
        L = lib()
        dp = C.POINTER(C.c_double)
        L.pctc_create.restype = C.c_void_p
        L.pctc_create.argtypes = [C.c_int, C.c_double, C.c_double, C.c_double, C.c_int, C.c_int, C.c_double]
        L.pctc_destroy.argtypes = [C.c_void_p]
        L.pctc_set_stream.argtypes = [C.c_void_p, dp, C.c_int]
        L.pctc_obs_len.argtypes = [C.c_void_p]
        L.pctc_reset.argtypes = [C.c_void_p, dp]
        L.pctc_step.argtypes = [C.c_void_p, dp, C.c_int, dp, dp, C.POINTER(C.c_int), dp]
        L.pctc_get_ems.argtypes = [C.c_void_p, dp, C.c_int]
        L.pctc_get_candidates.argtypes = [C.c_void_p, dp, C.POINTER(C.c_int), C.c_int]
        L.pctc_get_packed.argtypes = [C.c_void_p, dp, C.c_int]
        L.pctc_n_lstsq.argtypes = [C.c_void_p]
        L.pctc_drop_box_virtual.argtypes = [C.c_void_p] + [C.c_double] * 6 + [dp]
        L.pctc_get_next.argtypes = [C.c_void_p, dp]
        self.L = L
        self.h = L.pctc_create(setting, float(container_size[0]), float(container_size[1]), float(container_size[2]),
                               internal_node_holder, leaf_node_holder, float(size_minimum))
        self.nb, self.nl = internal_node_holder, leaf_node_holder
        self.obs_len = L.pctc_obs_len(self.h)
        self.container, self.setting = tuple(float(c) for c in container_size), int(setting)
        if stream is not None:
            self.set_stream(stream)

    def set_stream(self, stream):
        s = np.ascontiguousarray(stream, dtype=np.float64)
        if s.shape[1] == 3:
            s = np.concatenate([s, np.ones((len(s), 1))], axis=1)
        self._stream = np.ascontiguousarray(s)
        self.L.pctc_set_stream(self.h, _dp(self._stream), len(self._stream))

    def set_alias_mode(self, on=True):
        self.L.pctc_set_alias_mode.argtypes = [C.c_void_p, C.c_int]
        self.L.pctc_set_alias_mode(self.h, int(on))

    def set_shuffle(self, seed, gid, on=True):
        """shuffle=True (C:bin3D.py:126-127) with the product's keyed permutation (see OracleDiscrete.set_shuffle)"""
        self.L.pctc_set_shuffle.argtypes = [C.c_void_p, C.c_int, C.c_uint64, C.c_uint64]
        self.L.pctc_set_shuffle(self.h, int(on), int(seed) & ((1 << 64) - 1), int(gid))

    def set_random_sample(self, seed, gid, lo, hi):
        """sample_from_distribution draws (C:bin3D.py:103-115) from the counter-based generator the device uses"""
        self.L.pctc_set_random_sample.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_double, C.c_double]
        self.L.pctc_set_random_sample(self.h, int(seed), int(gid), float(lo), float(hi))

    def set_trajectory_length(self, n):
        self.L.pctc_set_trajectory_length.argtypes = [C.c_void_p, C.c_int]
        self.L.pctc_set_trajectory_length(self.h, int(n))

    def reset(self):
        obs = np.zeros(self.obs_len)
        self.L.pctc_reset(self.h, _dp(obs))
        return obs

    def step(self, action):
        a = np.ascontiguousarray(action, dtype=np.float64)
        obs = np.zeros(self.obs_len)
        rew, done, info = C.c_double(), C.c_int(), np.zeros(3)
        err = self.L.pctc_step(self.h, _dp(a), len(a), _dp(obs), C.byref(rew), C.byref(done), _dp(info))
        d = {"counter": int(info[0])}
        if done.value:
            d.update(ratio=float(info[1]), reward=float(info[2]))
        if err:
            d["error"] = err
        return obs, rew.value, bool(done.value), d

    def ems(self):
        buf = np.zeros((1000, 6))
        n = self.L.pctc_get_ems(self.h, _dp(buf), 1000)
        return buf[:n].copy()

    def candidates(self):
        buf = np.zeros((8192, 6))
        feas = np.zeros(8192, dtype=np.int32)
        n = self.L.pctc_get_candidates(self.h, _dp(buf), _ip(feas), 8192)
        return buf[:n].copy(), feas[:n].copy()

    @property
    def packed(self):
        buf = np.zeros((128, 7))
        n = self.L.pctc_get_packed(self.h, _dp(buf), 128)
        return buf[:n].tolist()

    # -- what the heuristic baselines read from the env (heuristic.py): space.drop_box_virtual(returnH), next_box / next_den
    def drop_box_virtual(self, dims, lx, ly):
        mh = C.c_double()
        ok = self.L.pctc_drop_box_virtual(self.h, float(dims[0]), float(dims[1]), float(dims[2]), float(lx), float(ly), self.next_den, C.byref(mh))
        return bool(ok), mh.value

    def _next(self):
        out = np.zeros(4)
        self.L.pctc_get_next(self.h, _dp(out))
        return out

    @property
    def next_box(self):
        return [float(v) for v in self._next()[:3]]

    @property
    def next_den(self):
        return float(self._next()[3])

    @property
    def n_lstsq(self):
        return self.L.pctc_n_lstsq(self.h)

    def __del__(self):
        try:
            self.L.pctc_destroy(self.h)
        except Exception:
            pass


def make_continuous_stream(seed, env, n, setting):
    """Per-env draw sequence with the distribution of C:bin3D.py:103-115 (values rounded to 3 decimals)."""
    s = np.zeros((n, 4))
    u = lambda salt, d: ((rnd_u64(seed ^ salt, env, d) >> 11) / float(1 << 53))
    for d in range(n):
        s[d, 0] = round(0.1 + 0.4 * u(0x11, d), 3)
        s[d, 1] = round(0.1 + 0.4 * u(0x22, d), 3)
        s[d, 2] = round(0.1 + 0.4 * u(0x33, d), 3) if setting == 2 else [0.1, 0.2, 0.3, 0.4, 0.5][rnd_u64(seed ^ 0x44, env, d) % 5]
        s[d, 3] = max((rnd_u64(seed ^ 0xABCDEF, env, d) >> 11), 1) / float(1 << 53) if setting == 3 else 1.0
    return s
