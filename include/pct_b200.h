/* pct_b200 — C ABI of the B200-native batched PCT environment (drop-in boundary).
 *
 * The reference (alexfrom0815/Online-3D-BPP-PCT @ 5e088f2) has no native interface: its
 * environment is a Python gym.Env (pct_envs/PctDiscrete0/bin3D.py:8-188,
 * pct_envs/PctContinuous0/bin3D.py:8-207) fanned out over forked workers by
 * wrapper/shmem_vec_env.py:20-156.  This header is what a ctypes binding of that path binds
 * instead (see INTEGRATION.md): every entry point names the reference interface it replaces.
 *
 * Conventions
 *   - plain C types only; device pointers are raw CUDA device addresses (e.g. tensor.data_ptr()),
 *     `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *   - every function returns 0 on success or a negative pct_status; pct_last_error() gives text.
 *   - the library owns the per-environment state; the caller owns action / observation / reward /
 *     done / info buffers.  No host synchronisation happens inside pct_reset / pct_step /
 *     pct_policy_random: they only enqueue work on `stream` (CUDA-graph capturable).
 *   - one host thread per handle.
 *
 * Observation layout (identical to D:bin3D.py:86-93 after the float32 cast of envs.py:168,180):
 *   row-major (internal_node_holder + leaf_node_holder + 1, 9)
 *   rows [0, NB)        placed boxes  [x1,y1,z1,x2,y2,z2,density,0,valid]   (row 0 col 8 is always 1)
 *   rows [NB, NB+NL)    leaf nodes    [x1,y1,z1,x2,y2,BIN_H,0,0,valid]
 *   row  NB+NL          next item     [density,0,0,d0<=d1<=d2,0,0,1]
 */
#ifndef PCT_B200_H
#define PCT_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pct_env_batch *pct_handle;

enum pct_status {
    PCT_OK = 0,
    PCT_ERR_INVALID = -1,   /* bad argument / unsupported configuration            */
    PCT_ERR_CUDA = -2,      /* CUDA runtime error (text in pct_last_error)          */
    PCT_ERR_NO_DEVICE = -3, /* no usable sm_100 device: the library has NO CPU fallback */
    PCT_ERR_STATE = -4      /* call sequence error (e.g. step before reset)         */
};

enum pct_domain { PCT_DISCRETE = 0, PCT_CONTINUOUS = 1 };
enum pct_obs_dtype { PCT_F32 = 0, PCT_F64 = 1 };
enum pct_lnes { PCT_LNES_EMS = 0, PCT_LNES_EV = 1, PCT_LNES_EP = 2, PCT_LNES_CP = 3, PCT_LNES_FC = 4 };
/* heuristic baselines of the reference (heuristic.py): LASH :138-226, OnlineBPH :364-424, BR :500-577, MACS :11-131,
 * DBL :431-493, heightmap_min :232-293, random :300-357 */
enum pct_heuristic {
    PCT_H_LSAH = 0, PCT_H_ONLINEBPH = 1, PCT_H_BR = 2, PCT_H_MACS = 3, /* placements taken from the EMS list   */
    PCT_H_DBL = 4, PCT_H_HM = 5, PCT_H_RANDOM = 6                      /* placements taken from the (lx, ly) grid */
};
enum pct_item_mode {
    PCT_ITEMS_RANDOM = 0, /* uniform over item_set with the counter-based generator (RandomBoxCreator, */
                          /*   D:binCreator.py:24-39); continuous + sample_from_distribution: C:bin3D.py:103-115 */
    PCT_ITEMS_STREAM = 1  /* caller-supplied per-env draw sequence (pct_set_item_stream)              */
};

/* Per-environment flag bits reported in pct_step_info.flags (sticky until the env resets). */
enum pct_env_flags {
    PCT_FLAG_BOX_OVERFLOW = 1,      /* more than internal_node_holder boxes (IndexError in D:space.py:385) */
    PCT_FLAG_BAD_ACTION = 2,        /* leaf row does not match the item (ValueError in D:bin3D.py:144-145) */
    PCT_FLAG_EMS_OVERFLOW = 4,      /* EMS list exceeded the fixed capacity                                */
    PCT_FLAG_CAND_OVERFLOW = 8,     /* candidate set exceeded the fixed capacity                           */
    PCT_FLAG_EDGE_OVERFLOW = 16,    /* support-edge pool exceeded the fixed capacity                       */
    PCT_FLAG_SUPPORT_OVERFLOW = 32, /* more supports under one box than the stability routine handles      */
    PCT_FLAG_SYNC_TIMEOUT = 64      /* internal: a kernel gave up waiting for the previous stage of this env */
};

/* Constructor arguments = the kwargs of PackingDiscrete / PackingContinuous.__init__
 * (D:bin3D.py:9-15, C:bin3D.py:9-17) forwarded by envs.make_env (envs.py:33-47). */
typedef struct pct_config {
    int32_t domain;               /* pct_domain                                                   */
    int32_t setting;              /* 1, 2 or 3                                                    */
    double container_size[3];     /* W, L, H (integers for the discrete domain)                   */
    int32_t internal_node_holder; /* <= 80 in this build                                          */
    int32_t leaf_node_holder;     /* <= 64 in this build                                          */
    int32_t obs_dtype;            /* pct_obs_dtype: float32 (VecPyTorch contract) or float64      */
    int32_t item_mode;            /* pct_item_mode                                                */
    double size_minimum;          /* np.min(item_set) (D:bin3D.py:23) / sample_left_bound (C:bin3D.py:26) */
    int32_t sample_from_distribution; /* continuous only (C:bin3D.py:14)                          */
    double sample_left_bound, sample_right_bound;
    uint64_t seed;                /* item generator seed (PCT_ITEMS_RANDOM)                       */
    int64_t env_id_base;          /* global index of env 0 of this handle (multi-GPU sharding:    */
                                  /*   per-env streams depend on the GLOBAL index only)           */
    int32_t no_auto_reset;        /* 0: ShmemVecEnv worker semantics (finished envs are reset inside the step,   */
                                  /*    wrapper/shmem_vec_env.py:141-142); 1: plain gym.Env semantics (the       */
                                  /*    terminal observation is returned, the caller resets; D:bin3D.py:160-165) */
    int32_t lnes;                 /* leaf-node expansion scheme (D:bin3D.py:101-112): pct_lnes, 0 = EMS (reference default) */
    int32_t shuffle;              /* `shuffle` kwarg (D:bin3D.py:114-115, C:bin3D.py:126-127; tools.py:136 defaults it to True for training): the   */
                                  /*   ordered candidate list is permuted before the feasibility tests and the leaf cap.  The reference draws from  */
                                  /*   the global numpy RNG (no parity definition); here the permutation is the stable argsort of counter-based     */
                                  /*   keys rnd_u64(seed ^ 0x5AFE5EED, global env id, draws << 16 | i) — uniform, reproducible, independent of the  */
                                  /*   sharding — and the oracle (test infrastructure) implements the same definition.                              */
} pct_config;

/* Terminal-step info (the dict built at D:bin3D.py:163-164 plus what Monitor adds, wrapper/monitor.py:58-77) */
typedef struct pct_step_info {
    int32_t counter;    /* len(space.boxes)                                      */
    int32_t flags;      /* pct_env_flags                                         */
    float ratio;        /* space.get_ratio()  (valid when done)                  */
    float ep_reward;    /* sum of rewards of the finished episode (Monitor 'r')  */
    int32_t ep_len;     /* number of steps of the finished episode (Monitor 'l') */
    int32_t n_leaf;     /* number of valid leaf rows in the new observation      */
    int32_t n_cand;     /* number of candidate placements generated (before the feasibility test) */
    int32_t n_ems;      /* EMS count after the step                              */
} pct_step_info;

/* Host-side dump of one environment (parity tests; replaces poking at env.space.* in Python). */
typedef struct pct_state_dump {
    int32_t n_boxes, n_ems, n_leaf, flags;
    int64_t draw_pos;
    double next_box[3];
    double next_den;
    double boxes[80][7]; /* lx,ly,lz,hx,hy,hz,density */
    double ems[256][6];
} pct_state_dump;

/* gym.make('PctDiscrete-v0' | 'PctContinuous-v0', **kwargs) x n_envs   (envs.py:84-108, tools.py:232-240) */
int pct_create(const pct_config *cfg, int32_t n_envs, int32_t device, pct_handle *out);
/* VecEnv.close()  (wrapper/vec_env.py:93-99) */
void pct_destroy(pct_handle h);
/* text of the last error on this handle (NULL handle: last pct_create error) */
const char *pct_last_error(pct_handle h);

/* item_set kwarg (givenData.py:4-14): host array (n,3) of item sizes used by PCT_ITEMS_RANDOM */
int pct_set_item_set(pct_handle h, const double *items_xyz, int32_t n_items);
/* replaces box_creator (D:binCreator.py): host array (n_envs, len, 4) of (x,y,z,density) draws per env,
 * consumed one per reset and one per successful placement, cyclically. Switches the handle to PCT_ITEMS_STREAM. */
int pct_set_item_stream(pct_handle h, const double *items_xyzd, int32_t len);
/* LoadBoxCreator episodes (D:binCreator.py:41-72): the stream is a sequence of fixed-length trajectories and every
 * reset jumps to the start of the next one (0 = plain continuous stream, the RandomBoxCreator discipline). */
int pct_set_trajectory_length(pct_handle h, int32_t traj_len);

/* VecEnv.reset()  (wrapper/shmem_vec_env.py:61-68 -> D:bin3D.py:61-67): resets every env, writes d_obs
 * (n_envs x obs_len elements of cfg.obs_dtype). */
int pct_reset(pct_handle h, void *d_obs, void *stream);

/* VecEnv.step_async + step_wait  (wrapper/shmem_vec_env.py:70-81,139-143 -> D:bin3D.py:151-188):
 * applies one action per env, auto-resets finished envs (the returned observation of a finished env is
 * its reset observation; reward/done/info are the terminal ones).
 *   d_actions  : n_envs x 9 leaf rows (float32 if action_f64==0 else float64), or NULL
 *   d_leaf_idx : n_envs int32 indices into the previous observation's leaf rows (fast path), or NULL;
 *                an index >= the env's n_leaf selects the all-zero row.  Exactly one of the two is non-NULL.
 *   d_reward   : n_envs float32;  d_done: n_envs uint8;  d_info: n_envs pct_step_info (may be NULL)
 * Observation buffer contract (delta rows, default; PCT_B200_OBS_DELTA=0 restores full rewrites): 75 % of the (internal + leaf + 1) x 9
 * observation is zero padding and the internal-node rows are append-only within an episode, so when a call receives the SAME d_obs pointer
 * as the previous reset / step of this handle, only the rows that can have changed are rewritten (the rows below max(rows now, rows the
 * buffer may hold non-zero) and the item row).  A caller that hands the same buffer to consecutive calls must therefore not modify it in
 * between (reading is fine); a caller that alternates buffers, or passes a fresh one, always gets every row written.  Both domains. */
int pct_step(pct_handle h, const void *d_actions, int32_t action_f64, const int32_t *d_leaf_idx, void *d_obs,
             float *d_reward, uint8_t *d_done, pct_step_info *d_info, void *stream);

/* Same call with HOST buffers (what the reference's VecEnv.step exchanges over its pipes): copies actions host->device, steps, delivers
 * obs / reward / done / info to the host, synchronises.  When h_obs is pinned (cudaHostAlloc / cudaHostRegister, i.e. mapped under UVA) the
 * emit kernel writes the observation rows STRAIGHT into it over PCIe (zero-copy, default; PCT_B200_HOST_ZEROCOPY=0 or an unpinned buffer:
 * staged device buffer + pipelined copies); the buffer contract of pct_step applies to h_obs in that mode. */
int pct_step_host(pct_handle h, const void *h_actions, int32_t action_f64, const int32_t *h_leaf_idx, void *h_obs,
                  float *h_reward, uint8_t *h_done, pct_step_info *h_info);
int pct_reset_host(pct_handle h, void *h_obs);

/* Uniform-random choice among the valid leaf rows of each env (the synthetic policy of SURVEY.md §8(d)):
 * d_leaf_idx[e] = rnd(seed, env_id_base+e, t) % n_leaf[e]  (0 when there is no valid leaf). */
int pct_policy_random(pct_handle h, int32_t *d_leaf_idx, uint64_t seed, int64_t t, void *stream);
/* same, with the step counter read from device memory (*d_t) at execution time: lets a captured CUDA graph of
 * policy -> step draw fresh actions on every replay (the caller increments *d_t inside the graph) */
int pct_policy_random_dev(pct_handle h, int32_t *d_leaf_idx, uint64_t seed, const int64_t *d_t, void *stream);

/* Heuristic baselines, batched (discrete domain).  For every env: the placement the baseline `heuristic` (enum
 * pct_heuristic) selects for the env's current item, written as an action row d_rows[e] = [lx, ly, 0, lx+x, ly+y, 0, 0, 0, 1]
 * (float32, N x 9) that pct_step(d_actions = d_rows, action_f64 = 0) applies; where the baseline finds no feasible
 * placement (the reference then ends the episode without stepping, e.g. heuristic.py:223-225) the row is
 * [1,0,0,1,0,0,0,0,1], which no item matches, so pct_step ends the episode (PCT_FLAG_BAD_ACTION is set in its info).
 * Replaces the per-env Python loops over Space.drop_box_virtual (D:space.py:393-433).  LSAH keeps its running footprint
 * per env inside the handle.  PCT_H_RANDOM draws with rnd(seed, env_id_base+e, t).  PCT_H_BR needs pct_set_item_set;
 * PCT_H_HM / PCT_H_MACS / PCT_H_RANDOM need container sides <= 32. */
int pct_heuristic_actions(pct_handle h, int32_t heuristic, float *d_rows, uint64_t seed, int64_t t, void *stream);
/* Same for the CONTINUOUS domain, where tools.py:217-218 allows PCT_H_LSAH, PCT_H_ONLINEBPH and PCT_H_BR only (heuristic.py
 * LASH :138-226, OnlineBPH :364-424, BR :500-577 over pct_envs.PctContinuous0): float64 rows (N x 9) for
 * pct_step(d_actions = d_rows, action_f64 = 1).  "No feasible placement" is the row [W+1,0,0,W+1,0,0,0,0,1]: the continuous
 * LeafNode2Action (C:bin3D.py:151-167) never raises, Space.drop_box rejects the position (C:space.py:336) and the episode ends.
 * Item sizes must carry <= 6 decimals (the reference's generators round to 3, C:bin3D.py:106-111), so that the
 * round(xe - xs, 6) of LeafNode2Action returns the chosen orientation's sizes exactly. */
int pct_heuristic_actions_f64(pct_handle h, int32_t heuristic, double *d_rows, void *stream);
/* Space.drop_box_virtual(dims, (lx, ly), False, density, setting, returnH / returnMap) for ONE env (D:space.py:393-433): what
 * the reference's heuristic.py calls on `env.space`; synchronous.  height_map: W*L int32 (row-major, after the virtual
 * placement — Space.update_height_graph on a copy) or NULL. */
int pct_query_placement(pct_handle h, int32_t env, const int32_t dims[3], int32_t lx, int32_t ly, double density,
                        int32_t *feasible, int32_t *rest_height, int32_t *height_map);

/* Space.drop_box_virtual(dims, (lx, ly), False, density, setting, returnH=True) of the CONTINUOUS env (C:space.py:380-425) for
 * ONE env; synchronous.  rest_height is interSect2D's max_h (C:space.py:391). */
int pct_query_placement_f64(pct_handle h, int32_t env, const double dims[3], double lx, double ly, double density,
                            int32_t *feasible, double *rest_height);

/* Saved env records: copy the state of environments, within a handle or between handles (search / lookahead from a branch point,
 * checkpoint and resume, moving envs between shards or GPUs).  What a copy continues with is defined by item_env: every env draws its items
 * from the sequence of ONE global env id — its own (cfg.env_id_base + e) until a record is loaded into it, then the source's, kept across
 * resets.  So "load the source's record into env d, then apply the same actions" gives exactly what the source gets, items drawn after the
 * load included.  The random policy and PCT_H_RANDOM keep drawing with the env's own id: they are policy randomness, not env state.
 *
 * A record is an opaque, fixed-size (pct_env_record_bytes), 16-byte-aligned device slot per env.  It holds the env's live state (boxes, EMS,
 * leaves of the last observation, item source position, episode sums, flags, load edges, the LSAH footprint) and a header with a 64-bit
 * fingerprint of the configuration: domain, setting, container, holders, lnes, shuffle, seed, item mode, size_minimum, sample bounds,
 * trajectory length, no_auto_reset, the item set contents, the stream length and the alias mode.  It leaves out env_id_base and obs_dtype,
 * so records move between shards, GPUs and observation dtypes.  In stream mode the record also carries the content hash of the stream row it
 * draws from.
 *
 * Both calls only enqueue stream-ordered work on `stream`: no host synchronisation, no allocation (CUDA-graph capturable). */
int64_t pct_env_record_bytes(pct_handle h);
/* d_records[i] = record of env d_env_ids[i], i < n.  Ids may repeat (saving repeat_interleave(src, K) gives K copies of each source);
 * d_env_ids == NULL: n == n_envs, record i = env i.  An id outside [0, n_envs) writes a record with an invalid header (it loads nowhere). */
int pct_save_envs(pct_handle h, const int32_t *d_env_ids, int32_t n, void *d_records, void *stream);
/* env d_env_ids[i] = the state in d_records[i], i < n (d_env_ids == NULL: n == n_envs, env i).  Each record is checked against the handle
 * before anything is written; d_status (n int32, may be NULL) receives per record
 *   0  loaded
 *   1  not a record of this configuration (header, version, domain or fingerprint differ; stream mode: the stream row differs)
 *   2  stream mode: the item row the record draws from (item_env - cfg.env_id_base) is not one of this handle's rows
 *   3  destination env id outside [0, n_envs)
 * and a rejected record leaves its destination untouched.  Destination ids must be distinct within one call (duplicates: undefined).
 * d_obs (n_envs x obs_len of cfg.obs_dtype, may be NULL) receives the full observation rows of the loaded envs (their source's last
 * observation, terminal ones of a no_auto_reset handle included); whatever buffer the next pct_step gets, it rewrites every row of the
 * loaded envs, so the delta-row contract of pct_step holds.  Needs a handle that has been reset (else PCT_ERR_STATE). */
int pct_load_envs(pct_handle h, const int32_t *d_env_ids, int32_t n, const void *d_records, void *d_obs, int32_t *d_status, void *stream);

/* introspection */
int pct_get_state(pct_handle h, int32_t env, pct_state_dump *out);
int32_t pct_obs_len(pct_handle h);       /* (NB + NL + 1) * 9 */
int32_t pct_num_envs(pct_handle h);
int64_t pct_state_bytes_per_env(pct_handle h); /* HBM bytes of library-owned state per env (roofline accounting) */
int64_t pct_kernel_launches(pct_handle h);     /* kernels launched by this handle so far */
/* Per-kernel device timing for roofline accounting: while enabled, every pct_step records CUDA events around its three
 * kernels on the launching stream; pct_profile_read synchronises and returns the summed milliseconds of
 * {apply, candidates, feas_emit} and the number of steps recorded since pct_profile_enable(h, 1). */
int pct_profile_enable(pct_handle h, int32_t on);
int pct_profile_read(pct_handle h, double ms_out[3], int32_t *n_steps);
const char *pct_version(void);

#ifdef __cplusplus
}
#endif
#endif
