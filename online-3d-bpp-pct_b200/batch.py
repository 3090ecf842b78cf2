"""PctBatch — N PCT environments living on one B200, stepped by the CUDA kernels behind the C ABI.

PyTorch is used for device buffers and streams only (observation / action / reward tensors); every
environment computation happens inside libpct_b200.so.  Mirrors the constructor kwargs of the reference's
PackingDiscrete / PackingContinuous (pct_envs/PctDiscrete0/bin3D.py:9-15, pct_envs/PctContinuous0/bin3D.py:9-17).
"""
import ctypes as C

import numpy as np
import torch

from . import _lib


class PctError(RuntimeError):
    pass


def record_arguments(records, env_ids, n_envs, record_bytes, device):
    """Checks and normalises the arguments of PctBatch.load_envs: -> (records, env ids or None, n).  records: (n, record_bytes) uint8, moved to
    `device` when they live elsewhere; env_ids: None (n == n_envs, record i -> env i) or n distinct ids in [0, n_envs) as a contiguous int32
    tensor on `device`.  Raises PctError."""
    if not isinstance(records, torch.Tensor):
        raise PctError("records must be a tensor (the output of save_envs)")
    if records.dtype != torch.uint8 or records.dim() != 2 or records.shape[1] != record_bytes:
        raise PctError("records must be a (n, %d) uint8 tensor, got %s %s" % (record_bytes, tuple(records.shape), records.dtype))
    if records.device != device:
        records = records.to(device)
    records = records.contiguous()
    n = int(records.shape[0])
    ids = env_id_tensor(env_ids, n_envs, device)
    if ids is None:
        if n != n_envs:
            raise PctError("records for all %d envs expected without env_ids, got %d" % (n_envs, n))
    else:
        if ids.numel() != n:
            raise PctError("%d records for %d env ids" % (n, ids.numel()))
        if n and (int(ids.min()) < 0 or int(ids.max()) >= n_envs):
            raise PctError("env ids must lie in [0, %d)" % n_envs)
        if torch.unique(ids).numel() != n:
            raise PctError("duplicate destination env ids in one load")
    return records, ids, n


def env_id_tensor(env_ids, n_envs, device):
    """None, or env ids (tensor / sequence of integers) as a contiguous 1-D int32 tensor on `device`"""
    if env_ids is None:
        return None
    if isinstance(env_ids, torch.Tensor):
        if env_ids.dtype.is_floating_point or env_ids.dtype == torch.bool:
            raise PctError("env ids must be integers, got %s" % env_ids.dtype)
        ids = env_ids
    else:
        ids = torch.as_tensor(np.asarray(env_ids, dtype=np.int64))
    if ids.dim() != 1:
        raise PctError("env ids must be a 1-D sequence")
    return ids.to(device=device, dtype=torch.int32).contiguous()


class PctBatch(object):
    def __init__(self, n_envs, setting, container_size=(10, 10, 10), item_set=None, internal_node_holder=80,
                 leaf_node_holder=50, continuous=False, obs_dtype=torch.float32, seed=0, env_id_base=0, device=0,
                 sample_from_distribution=False, sample_left_bound=None, sample_right_bound=None, item_stream=None,
                 size_minimum=None, auto_reset=True, LNES="EMS", shuffle=False):
        """shuffle: the reference's `shuffle` kwarg (D:bin3D.py:114-115; tools.py:136 defaults --shuffle to True for training): the ordered candidate list
        is permuted before the feasibility tests and the leaf cap, by a keyed counter-based permutation (include/pct_b200.h, pct_config::shuffle)."""
        if not torch.cuda.is_available():
            raise PctError("pct_b200 needs a CUDA device (sm_100a kernels; there is no CPU fallback)")
        self.L = _lib.lib()
        self.n_envs = int(n_envs)
        self.device = torch.device("cuda", device)
        self.nb, self.nl = int(internal_node_holder), int(leaf_node_holder)
        self.obs_dtype = obs_dtype
        self.container_size = tuple(container_size)
        self.setting = int(setting)
        self.continuous = bool(continuous)
        cfg = _lib.Config()
        cfg.domain = _lib.PCT_CONTINUOUS if continuous else _lib.PCT_DISCRETE
        cfg.setting = self.setting
        for i in range(3):
            cfg.container_size[i] = float(container_size[i])
        cfg.internal_node_holder, cfg.leaf_node_holder = self.nb, self.nl
        cfg.obs_dtype = _lib.PCT_F64 if obs_dtype == torch.float64 else _lib.PCT_F32
        cfg.item_mode = _lib.PCT_ITEMS_RANDOM
        cfg.sample_from_distribution = int(bool(sample_from_distribution))
        if sample_from_distribution:
            # tools.get_args :178-181
            if sample_left_bound is None:
                sample_left_bound = 0.1 * min(container_size)
            if sample_right_bound is None:
                sample_right_bound = 0.5 * min(container_size)
            cfg.sample_left_bound, cfg.sample_right_bound = float(sample_left_bound), float(sample_right_bound)
        if size_minimum is None:
            # D:bin3D.py:23 / C:bin3D.py:25-29
            if continuous and sample_from_distribution:
                size_minimum = sample_left_bound
            else:
                size_minimum = float(np.min(np.array(item_set))) if item_set is not None else 1.0
        cfg.size_minimum = float(size_minimum)
        cfg.seed = int(seed) & ((1 << 64) - 1)
        cfg.env_id_base = int(env_id_base)
        cfg.no_auto_reset = 0 if auto_reset else 1
        cfg.lnes = _lib.LNES_CODES[LNES]
        cfg.shuffle = int(bool(shuffle))
        self.cfg = cfg
        h = C.c_void_p()
        rc = self.L.pct_create(C.byref(cfg), self.n_envs, int(device), C.byref(h))
        if rc != 0:
            raise PctError("pct_create failed (%d): %s" % (rc, self.L.pct_last_error(None).decode()))
        self.h = h
        self.obs_len = self.L.pct_obs_len(self.h)
        if item_set is not None:
            self.set_item_set(item_set)
        if item_stream is not None:
            self.set_item_stream(item_stream)
        with torch.cuda.device(self.device):
            self._obs = torch.empty((self.n_envs, self.obs_len), dtype=obs_dtype, device=self.device)
            # reward (N f32) | info (N x 8 i32) | done (N u8) live in ONE allocation, so that a host-facing caller fetches all three with one copy
            n = self.n_envs
            self._pack = torch.zeros((n * 4 + n * 32 + n,), dtype=torch.uint8, device=self.device)
            self._rew = self._pack[:4 * n].view(torch.float32)
            self._info = self._pack[4 * n:36 * n].view(torch.int32).view(n, 8)
            self._done = self._pack[36 * n:]
            self._idx = torch.zeros((self.n_envs,), dtype=torch.int32, device=self.device)

    # -- plumbing ------------------------------------------------------------------------------------------
    def _check(self, rc, what):
        if rc != 0:
            raise PctError("%s failed (%d): %s" % (what, rc, self.L.pct_last_error(self.h).decode()))

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def set_item_set(self, item_set):
        a = np.ascontiguousarray(np.array(item_set, dtype=np.float64).reshape(-1, 3))
        self._check(self.L.pct_set_item_set(self.h, a.ctypes.data_as(C.POINTER(C.c_double)), len(a)), "pct_set_item_set")

    def set_item_stream(self, stream):
        """stream: array (n_envs, len, 3|4) of per-env draws (x, y, z[, density])."""
        a = np.array(stream, dtype=np.float64)
        if a.ndim != 3 or a.shape[0] != self.n_envs:
            raise PctError("item stream must have shape (n_envs, len, 3|4)")
        if a.shape[2] == 3:
            a = np.concatenate([a, np.ones(a.shape[:2] + (1,))], axis=2)
        a = np.ascontiguousarray(a)
        self._check(self.L.pct_set_item_stream(self.h, a.ctypes.data_as(C.POINTER(C.c_double)), a.shape[1]), "pct_set_item_stream")

    def set_trajectory_length(self, traj_len):
        self._check(self.L.pct_set_trajectory_length(self.h, int(traj_len)), "pct_set_trajectory_length")

    # -- device-resident API -------------------------------------------------------------------------------
    def reset(self, out=None):
        obs = self._obs if out is None else out
        self._check(self.L.pct_reset(self.h, C.c_void_p(obs.data_ptr()), self._stream()), "pct_reset")
        return obs

    def step(self, actions=None, leaf_idx=None, out=None):
        """actions: (N,9) float32/float64 CUDA tensor of leaf rows, or leaf_idx: (N,) int32 CUDA tensor.
        Returns (obs, reward(N,), done(N,) uint8, info(N,8) int32 raw pct_step_info records) — all on the GPU.
        NOTE: without `out`, the four tensors are the library-owned buffers, rewritten IN PLACE by the next reset / step (zero-copy; and with the
        delta observation rows, include/pct_b200.h, the observation buffer must not be modified by the caller).  Keep a result across steps with
        .clone(), or pass your own `out` buffers (e.g. a rollout storage, GraphedRollout); PctVecEnv hands out fresh observation tensors."""
        obs = self._obs if out is None else out
        a_ptr, i_ptr, f64 = None, None, 0
        if actions is not None:
            if actions.dtype not in (torch.float32, torch.float64):
                actions = actions.float()
            actions = actions.contiguous()
            if actions.shape != (self.n_envs, 9):
                raise PctError("actions must have shape (n_envs, 9)")
            a_ptr, f64 = C.c_void_p(actions.data_ptr()), int(actions.dtype == torch.float64)
        else:
            leaf_idx = leaf_idx.to(torch.int32).contiguous()
            i_ptr = C.c_void_p(leaf_idx.data_ptr())
        self._check(self.L.pct_step(self.h, a_ptr, f64, i_ptr, C.c_void_p(obs.data_ptr()), C.c_void_p(self._rew.data_ptr()),
                                    C.c_void_p(self._done.data_ptr()), C.c_void_p(self._info.data_ptr()), self._stream()), "pct_step")
        return obs, self._rew, self._done, self._info

    def random_policy(self, seed, t, out=None):
        idx = self._idx if out is None else out
        self._check(self.L.pct_policy_random(self.h, C.c_void_p(idx.data_ptr()), int(seed) & ((1 << 64) - 1), int(t), self._stream()),
                    "pct_policy_random")
        return idx

    def random_policy_dev(self, seed, t_dev, out=None):
        """random_policy with the step counter read from a device int64 tensor at execution time (graph-capturable)"""
        idx = self._idx if out is None else out
        self._check(self.L.pct_policy_random_dev(self.h, C.c_void_p(idx.data_ptr()), int(seed) & ((1 << 64) - 1), C.c_void_p(t_dev.data_ptr()),
                                                 self._stream()), "pct_policy_random_dev")
        return idx

    # -- saved env records (include/pct_b200.h, pct_save_envs / pct_load_envs) ----------------------------------------
    @property
    def record_bytes(self):
        """size of one saved env record (fixed per domain)"""
        return int(self.L.pct_env_record_bytes(self.h))

    def save_envs(self, env_ids=None, out=None):
        """The state of the envs `env_ids` (repeats allowed: repeat_interleave(src, K) gives K copies of each source; None = every env in order)
        as a (n, record_bytes) uint8 CUDA tensor (or into `out`).  The records are opaque; load_envs puts them into this or any handle with the
        same configuration (another env_id_base, GPU or observation dtype included).  Enqueued on the current stream, no synchronisation."""
        ids = env_id_tensor(env_ids, self.n_envs, self.device)
        n = self.n_envs if ids is None else int(ids.numel())
        rb = self.record_bytes
        if out is None:
            out = torch.empty((n, rb), dtype=torch.uint8, device=self.device)
        if out.dtype != torch.uint8 or tuple(out.shape) != (n, rb) or not out.is_contiguous() or out.device != self.device:
            raise PctError("out must be a contiguous (%d, %d) uint8 tensor on %s" % (n, rb, self.device))
        self._check(self.L.pct_save_envs(self.h, C.c_void_p(ids.data_ptr()) if ids is not None else None, n, C.c_void_p(out.data_ptr()),
                                         self._stream()), "pct_save_envs")
        return out

    def load_envs(self, records, env_ids=None, obs=None, check=True, status=None):
        """Env env_ids[i] takes the state saved in records[i] (None: record i -> env i) and continues exactly like its source, items drawn after the
        load included.  obs: an (n_envs, obs_len) tensor of the handle's observation dtype that receives the loaded envs' observation rows.
        check=True synchronises and raises PctError when a record does not belong to this configuration (or, in item-stream mode, draws from a
        stream row this handle does not hold), and rejects duplicate destination ids.  check=False does not synchronise (CUDA-graph capture):
        pass `status` (n int32 on the device) to get the per-record codes (0 loaded, 1 other configuration, 2 stream row not here, 3 bad env
        id); a rejected record leaves its env untouched.  Returns the status tensor (None with check=False and no `status`)."""
        if check:
            records, ids, n = record_arguments(records, env_ids, self.n_envs, self.record_bytes, self.device)
        else:  # no host synchronisation: shape checks only
            if records.device != self.device:
                records = records.to(self.device)
            records = records.contiguous()
            n = int(records.shape[0])
            if records.dtype != torch.uint8 or records.dim() != 2 or records.shape[1] != self.record_bytes:
                raise PctError("records must be a (n, %d) uint8 tensor" % self.record_bytes)
            ids = env_id_tensor(env_ids, self.n_envs, self.device)
            if ids is not None and ids.numel() != n:
                raise PctError("%d records for %d env ids" % (n, ids.numel()))
        if obs is not None and (obs.dtype != self.obs_dtype or tuple(obs.shape) != (self.n_envs, self.obs_len) or not obs.is_contiguous()
                                or obs.device != self.device):
            raise PctError("obs must be a contiguous (%d, %d) %s tensor on %s" % (self.n_envs, self.obs_len, self.obs_dtype, self.device))
        if status is None and check:
            status = torch.empty((n,), dtype=torch.int32, device=self.device)
        if status is not None and (status.dtype != torch.int32 or status.numel() < n or not status.is_contiguous() or status.device != self.device):
            raise PctError("status must be a contiguous int32 tensor of >= %d elements on %s" % (n, self.device))
        self._check(self.L.pct_load_envs(self.h, C.c_void_p(ids.data_ptr()) if ids is not None else None, n, C.c_void_p(records.data_ptr()),
                                         C.c_void_p(obs.data_ptr()) if obs is not None else None,
                                         C.c_void_p(status.data_ptr()) if status is not None else None, self._stream()), "pct_load_envs")
        if check:
            st = status[:n].cpu().numpy()
            if st.any():
                bad = np.nonzero(st)[0]
                raise PctError("pct_load_envs rejected %d of %d record(s) (first: record %d, status %d = %s); rejected records left their envs untouched"
                               % (len(bad), n, int(bad[0]), int(st[bad[0]]), _lib.RECORD_STATUS.get(int(st[bad[0]]), "?")))
        return status

    # -- heuristic baselines (heuristic.py) ------------------------------------------------------------------
    def heuristic_actions(self, name, seed=0, t=0, out=None):
        """(N, 9) float32 CUDA tensor of action rows: the placement the baseline `name` (LSAH, OnlineBPH, BR, MACS, DBL, HM,
        RANDOM) selects for every env's current item; feed to step(actions=...).
        Continuous domain: LSAH / OnlineBPH / BR (tools.py:217-218), float64 rows."""
        if name not in _lib.HEURISTIC_CODES:
            raise PctError("unknown heuristic %r" % (name,))
        if self.continuous:
            if out is None:
                if getattr(self, "_hrows", None) is None:
                    self._hrows = torch.zeros((self.n_envs, 9), dtype=torch.float64, device=self.device)
                out = self._hrows
            if out.dtype != torch.float64 or not out.is_contiguous() or out.shape != (self.n_envs, 9):
                raise PctError("continuous heuristic rows must be a contiguous (n_envs, 9) float64 tensor")
            self._check(self.L.pct_heuristic_actions_f64(self.h, _lib.HEURISTIC_CODES[name], C.c_void_p(out.data_ptr()), self._stream()),
                        "pct_heuristic_actions_f64")
            return out
        if out is None:
            if getattr(self, "_hrows", None) is None:
                self._hrows = torch.zeros((self.n_envs, 9), dtype=torch.float32, device=self.device)
            out = self._hrows
        self._check(self.L.pct_heuristic_actions(self.h, _lib.HEURISTIC_CODES[name], C.c_void_p(out.data_ptr()), int(seed) & ((1 << 64) - 1),
                                                 int(t), self._stream()), "pct_heuristic_actions")
        return out

    def query_placement(self, env, dims, lx, ly, density=1.0, want_map=False):
        """Space.drop_box_virtual for one env (D:space.py:393-433): -> (feasible, rest_height[, height map after])"""
        if self.continuous:  # C:space.py:380-425 has no returnMap
            d, feas, mh = (C.c_double * 3)(float(dims[0]), float(dims[1]), float(dims[2])), C.c_int32(), C.c_double()
            self._check(self.L.pct_query_placement_f64(self.h, int(env), d, float(lx), float(ly), float(density), C.byref(feas), C.byref(mh)),
                        "pct_query_placement_f64")
            return (bool(feas.value), mh.value, None) if want_map else (bool(feas.value), mh.value)
        d = (C.c_int32 * 3)(int(dims[0]), int(dims[1]), int(dims[2]))
        feas, mh = C.c_int32(), C.c_int32()
        W, L = int(self.container_size[0]), int(self.container_size[1])
        hm = np.zeros((W, L), dtype=np.int32) if want_map else None
        self._check(self.L.pct_query_placement(self.h, int(env), d, int(lx), int(ly), float(density), C.byref(feas), C.byref(mh),
                                               hm.ctypes.data_as(C.POINTER(C.c_int32)) if want_map else None), "pct_query_placement")
        return (bool(feas.value), mh.value, hm) if want_map else (bool(feas.value), mh.value)

    # -- host-buffer API (what the reference's VecEnv exchanges over its pipes) --------------------------------
    def reset_host(self, obs_out):
        self._check(self.L.pct_reset_host(self.h, C.c_void_p(obs_out.ctypes.data)), "pct_reset_host")
        return obs_out

    def step_host(self, obs_out, rew_out, done_out, info_out=None, actions=None, leaf_idx=None):
        a_ptr, i_ptr, f64 = None, None, 0
        if actions is not None:
            a_ptr, f64 = C.c_void_p(actions.ctypes.data), int(actions.dtype == np.float64)
        else:
            i_ptr = C.c_void_p(leaf_idx.ctypes.data)
        self._check(self.L.pct_step_host(self.h, a_ptr, f64, i_ptr, C.c_void_p(obs_out.ctypes.data), C.c_void_p(rew_out.ctypes.data),
                                         C.c_void_p(done_out.ctypes.data), C.c_void_p(info_out.ctypes.data) if info_out is not None else None),
                    "pct_step_host")

    # -- introspection -------------------------------------------------------------------------------------
    @staticmethod
    def check_flags(flags, ignore=0, what="pct_step"):
        """Raise PctError when any env's step record carries a capacity / hand-over flag (pct_step_info.flags) outside `ignore`: a flagged env's
        results are not the reference's (which would have raised IndexError / ValueError, or has no such limit).  Used by PctVecEnv,
        evaluate_batched and run_heuristic; low-level PctBatch.step callers check `decode_info(info)['flags']` themselves."""
        f = np.asarray(flags).astype(np.int64) & ~int(ignore)
        if f.any():
            bad = np.nonzero(f)[0]
            names = sorted({nm for v in f[bad] for bit, nm in _lib.FLAG_NAMES.items() if v & bit})
            raise PctError("%s flagged %d env(s) (first: env %d, flags %d = %s) — results of flagged envs are not the reference's"
                           % (what, len(bad), int(bad[0]), int(f[bad[0]]), "|".join(names)))

    @staticmethod
    def decode_info(info_cpu):
        """(N,8) int32 tensor/array of pct_step_info records -> dict of numpy arrays."""
        a = info_cpu.cpu().numpy() if hasattr(info_cpu, "cpu") else np.asarray(info_cpu)
        f = a.view(np.float32)
        return dict(counter=a[:, 0], flags=a[:, 1], ratio=f[:, 2], ep_reward=f[:, 3], ep_len=a[:, 4], n_leaf=a[:, 5], n_cand=a[:, 6],
                    n_ems=a[:, 7])

    def state(self, env):
        d = _lib.StateDump()
        self._check(self.L.pct_get_state(self.h, int(env), C.byref(d)), "pct_get_state")
        boxes = np.array([list(d.boxes[i]) for i in range(d.n_boxes)]).reshape(-1, 7)
        ems = np.array([list(d.ems[i]) for i in range(min(d.n_ems, 256))]).reshape(-1, 6)
        return dict(n_boxes=d.n_boxes, n_ems=d.n_ems, n_leaf=d.n_leaf, flags=d.flags, draw_pos=d.draw_pos,
                    next_box=list(d.next_box), next_den=d.next_den, boxes=boxes, ems=ems)

    def profile(self, on=True):
        self._check(self.L.pct_profile_enable(self.h, int(on)), "pct_profile_enable")

    def profile_read(self):
        """-> ({'apply': ms, 'candidates': ms, 'feas_emit': ms} summed over the recorded steps, n_steps)"""
        ms = (C.c_double * 3)()
        n = C.c_int32()
        self._check(self.L.pct_profile_read(self.h, ms, C.byref(n)), "pct_profile_read")
        return dict(apply=ms[0], candidates=ms[1], feas_emit=ms[2]), n.value

    @property
    def kernel_launches(self):
        return int(self.L.pct_kernel_launches(self.h))

    @property
    def state_bytes_per_env(self):
        return int(self.L.pct_state_bytes_per_env(self.h))

    def close(self):
        if getattr(self, "h", None):
            self.L.pct_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
