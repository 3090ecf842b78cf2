// C-ABI layer (include/pct_b200.h): owns the per-environment device state, validates arguments, enqueues
// the kernels on the caller's stream.  No torch types, no exceptions across the boundary, no CPU fallback.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "pct_common.cuh"  // splitmix64
#include "pct_kernels.h"
#include "pct_handle.h"

using namespace pct;

static thread_local std::string g_create_err;
static_assert(sizeof(pct_config) == 112 && sizeof(pct_step_info) == 32, "C ABI layout (tests/test_cabi.py checks the ctypes mirror against the same numbers)");

#define CK(h, call)                                                                                        \
    do {                                                                                                   \
        cudaError_t e_ = (call);                                                                           \
        if (e_ != cudaSuccess) {                                                                           \
            (h)->err = std::string(#call) + ": " + cudaGetErrorString(e_);                                 \
            return PCT_ERR_CUDA;                                                                           \
        }                                                                                                  \
    } while (0)

namespace pct {
// continuous domain (pct_continuous.cu)
int continuous_create(pct_env_batch *h);
void continuous_destroy(pct_env_batch *h);
int continuous_launch(pct_env_batch *h, int mode, const void *actions, int action_f64, const int32_t *leaf_idx, void *obs, float *rew,
                      uint8_t *done, pct_step_info *info, cudaStream_t st);
int continuous_policy_random(pct_env_batch *h, int32_t *leaf_idx, uint64_t seed, int64_t t, cudaStream_t st);
int continuous_get_state(pct_env_batch *h, int env, pct_state_dump *out);
int64_t continuous_state_bytes();
int continuous_heuristic(pct_env_batch *h, int code, double *rows, double *hstate, cudaStream_t st);
int continuous_query(pct_env_batch *h, int env, const double q[5], double density, double *d_out, cudaStream_t st);
int64_t continuous_record_bytes();
int continuous_records(pct_env_batch *h, const RecArgs &s, int load, void *obs, cudaStream_t st);
}  // namespace pct

// 64-bit FNV-1a over byte ranges, finished with splitmix64 (host side: configuration fingerprint, item set / stream row hashes)
static uint64_t fnv1a(uint64_t hash, const void *data, size_t n) {
    const unsigned char *b = (const unsigned char *)data;
    for (size_t i = 0; i < n; i++) { hash ^= b[i]; hash *= 0x100000001B3ull; }
    return hash;
}
constexpr uint64_t FNV_SEED = 0xCBF29CE484222325ull;

// Everything that gives a saved env record its meaning: a record loads only into a handle with the same fingerprint.  Leaves out
// env_id_base (records move between shards: item_env keeps the item sequence) and obs_dtype (the record holds no observation).
static uint64_t config_fingerprint(pct_handle h) {
    const pct_config &c = h->cfg;
    uint64_t f = FNV_SEED;
    auto mix = [&](const auto &v) { f = fnv1a(f, &v, sizeof v); };
    mix(c.domain); mix(c.setting); mix(c.container_size); mix(c.internal_node_holder); mix(c.leaf_node_holder); mix(c.lnes); mix(c.shuffle);
    mix(c.seed); mix(h->item_mode); mix(c.size_minimum); mix(c.sample_from_distribution); mix(c.sample_left_bound); mix(c.sample_right_bound);
    mix(h->traj_len); mix(c.no_auto_reset);
    mix(h->n_items); mix(h->item_set_hash);  // item set contents
    mix(h->stream_len);                      // item stream: its rows are checked one by one (RecHdr::row_hash)
    const int32_t alias = h->alias_mode ? 1 : 0;  // PCT_B200_ALIAS=0 handles do not maintain DEnvAux::box_st
    mix(alias);
    return splitmix64(f);
}

extern "C" {

const char *pct_version(void) { return "pct_b200 0.1 (sm_100a)"; }

const char *pct_last_error(pct_handle h) { return h ? h->err.c_str() : g_create_err.c_str(); }

int pct_create(const pct_config *cfg, int32_t n_envs, int32_t device, pct_handle *out) {
    if (!cfg || !out || n_envs <= 0) { g_create_err = "pct_create: bad arguments"; return PCT_ERR_INVALID; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        g_create_err = "pct_create: no CUDA device — this library has no CPU fallback";
        return PCT_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= ndev) { g_create_err = "pct_create: bad device index"; return PCT_ERR_INVALID; }
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    if (prop.major != 10) {
        g_create_err = std::string("pct_create: device '") + prop.name + "' is not sm_100 (kernels are built for sm_100a only)";
        return PCT_ERR_NO_DEVICE;
    }
    if (cfg->setting < 1 || cfg->setting > 3) { g_create_err = "pct_create: setting must be 1, 2 or 3"; return PCT_ERR_INVALID; }
    if (cfg->internal_node_holder < 1 || cfg->internal_node_holder > NB_MAX || cfg->leaf_node_holder < 1 || cfg->leaf_node_holder > NL_MAX) {
        g_create_err = "pct_create: holder sizes out of range (internal <= 80, leaf <= 64)";
        return PCT_ERR_INVALID;
    }
    if (cfg->lnes < 0 || cfg->lnes > 4 || (cfg->lnes != 0 && cfg->domain != PCT_DISCRETE)) {
        g_create_err = "pct_create: lnes must be 0 (EMS) .. 4 (FC); the continuous domain builds EMS only";
        return PCT_ERR_INVALID;
    }
    if (cfg->domain == PCT_DISCRETE) {
        for (int i = 0; i < 3; i++)
            if (cfg->container_size[i] < 1 || cfg->container_size[i] > 255 || cfg->container_size[i] != (int)cfg->container_size[i]) {
                g_create_err = "pct_create: discrete container sizes must be integers in [1,255]";
                return PCT_ERR_INVALID;
            }
    } else if (cfg->domain != PCT_CONTINUOUS) {
        g_create_err = "pct_create: unknown domain";
        return PCT_ERR_INVALID;
    }
    pct_env_batch *h = new pct_env_batch();
    h->cfg = *cfg;
    h->n_envs = n_envs;
    h->device = device;
    h->obs_len = (cfg->internal_node_holder + cfg->leaf_node_holder + 1) * 9;
    h->item_mode = cfg->item_mode;
    cudaError_t e = cudaSetDevice(device);
    // pct_step_host pipelines env ranges over these streams; earlier ranges get a higher priority so that their kernels
    // finish (and their device->host copies start) while later ranges still compute.  PCT_B200_HOST_PRIO=0 disables.
    int prio_least = 0, prio_greatest = 0;
    bool use_prio = true;
    if (const char *pv = getenv("PCT_B200_HOST_PRIO")) use_prio = atoi(pv) != 0;
    if (e == cudaSuccess && use_prio) e = cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest);
    auto prio_of = [&](int gi) { int p = prio_greatest + gi; return p > prio_least ? prio_least : p; };
    if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&h->own_stream, cudaStreamNonBlocking, prio_of(0));
    if (const char *ov = getenv("PCT_B200_OVERLAP")) h->overlap = atoi(ov) != 0;
    if (const char *ov = getenv("PCT_B200_OVERLAP_CONT")) h->overlap_cont = atoi(ov) != 0;
    if (const char *pv = getenv("PCT_B200_CONT_PRE")) h->cont_pre = atoi(pv) != 0;
    if (const char *zv = getenv("PCT_B200_HOST_ZEROCOPY")) h->host_zero_copy = atoi(zv) != 0;
    if (const char *dv = getenv("PCT_B200_OBS_DELTA")) h->obs_delta = atoi(dv) != 0;
    if (const char *av = getenv("PCT_B200_ALIAS")) h->alias_mode = atoi(av) != 0;
    if (const char *kv = getenv("PCT_B200_K3")) h->k3_block = strcmp(kv, "block") == 0;
    if (const char *wv = getenv("PCT_B200_WALK_LANES_TALL")) { h->walk_lanes_tall = atoi(wv); if (h->walk_lanes_tall < 1) h->walk_lanes_tall = 1; if (h->walk_lanes_tall > 32) h->walk_lanes_tall = 32; }
    if (const char *ev = getenv("PCT_B200_EMIT_PDL")) h->no_emit_pdl = atoi(ev) == 0;
    if (const char *wv = getenv("PCT_B200_WALK")) h->walk_fork = strcmp(wv, "fork") == 0;  // fork: the fork-join continuation kernel (A/B; default: sequential walks)
    if (const char *wv = getenv("PCT_B200_WALK_KEEP")) { h->walk_keep = atoi(wv); if (h->walk_keep < 1) h->walk_keep = 1; }
    if (const char *wv = getenv("PCT_B200_WALK_BLOCKS")) { h->walk_blocks = atoi(wv); if (h->walk_blocks < 1) h->walk_blocks = 1; if (h->walk_blocks > 8) h->walk_blocks = 8; }
    if (const char *wv = getenv("PCT_B200_WALK_LANES")) { h->walk_lanes = atoi(wv); if (h->walk_lanes < 1) h->walk_lanes = 1; if (h->walk_lanes > 32) h->walk_lanes = 32; }
    if (cfg->setting == 2) h->alias_mode = false;  // no stability check, no load entries
    // LSAH footprint state: per-env state that saved records carry, allocated here so that a load never allocates
    const size_t hs_bytes = (cfg->domain == PCT_CONTINUOUS ? sizeof(double) : sizeof(int32_t)) * 4 * (size_t)n_envs;
    if (e == cudaSuccess) e = cudaMalloc(cfg->domain == PCT_CONTINUOUS ? (void **)&h->d_hstate_c : (void **)&h->d_hstate, hs_bytes);
    if (e == cudaSuccess) e = cudaMemset(cfg->domain == PCT_CONTINUOUS ? (void *)h->d_hstate_c : (void *)h->d_hstate, 0, hs_bytes);
    if ((h->obs_delta || h->alias_mode) && e == cudaSuccess) {
        e = cudaMalloc(&h->d_aux, sizeof(DEnvAux) * (size_t)n_envs);
        if (e == cudaSuccess) e = cudaMemset(h->d_aux, 0, sizeof(DEnvAux) * (size_t)n_envs);
    }
    h->groups = 1;  // PCT_B200_GROUPS > 1 splits the batch over internal streams (measured: no gain, see DESIGN.md)
    if (const char *gv = getenv("PCT_B200_GROUPS")) h->groups = atoi(gv);
    h->host_groups = 4;
    if (const char *gv = getenv("PCT_B200_HOST_GROUPS")) h->host_groups = atoi(gv);
    if (h->host_groups < 1) h->host_groups = 1;
    if (h->host_groups > 8) h->host_groups = 8;
    if (h->groups < 1) h->groups = 1;
    if (h->groups > 8) h->groups = 8;
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming);
    for (int gi = 1; gi < 8 && e == cudaSuccess; gi++) {
        e = cudaStreamCreateWithPriority(&h->sub[gi], cudaStreamNonBlocking, prio_of(gi));
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_join[gi], cudaEventDisableTiming);
    }
    if (e == cudaSuccess) {
        if (cfg->domain == PCT_DISCRETE) {
            e = cudaMalloc(&h->d_hot, sizeof(DEnvHot) * (size_t)n_envs);
            if (e == cudaSuccess) e = cudaMalloc(&h->d_cold, sizeof(DEnvCold) * (size_t)n_envs);
            if (e == cudaSuccess) e = cudaMemset(h->d_hot, 0, sizeof(DEnvHot) * (size_t)n_envs);
            if (e == cudaSuccess) {  // item_env = the env's own global id (DHdr::item_env)
                std::vector<int64_t> id((size_t)n_envs);
                for (int i = 0; i < n_envs; i++) id[i] = cfg->env_id_base + i;
                e = cudaMemcpy2D((char *)h->d_hot + offsetof(DEnvHot, h) + offsetof(DHdr, item_env), sizeof(DEnvHot), id.data(), sizeof(int64_t),
                                 sizeof(int64_t), (size_t)n_envs, cudaMemcpyHostToDevice);
            }
            if (e == cudaSuccess) e = cudaMalloc(&h->d_ready, sizeof(int32_t) * 2 * (size_t)n_envs);
            if (e == cudaSuccess) e = cudaMemset(h->d_ready, 0, sizeof(int32_t) * 2 * (size_t)n_envs);
            if (e == cudaSuccess) e = cudaMemset(h->d_cold, 0, sizeof(DEnvCold) * (size_t)n_envs);
            if (e == cudaSuccess && !h->k3_block) {  // the step's pool of stability walks: worst-case capacity, only the used prefix is ever touched
                e = cudaMalloc(&h->d_walkq, sizeof(WalkItem) * (size_t)CAND_MAX * (size_t)n_envs);
                if (e == cudaSuccess) e = cudaMalloc(&h->d_walk_ctr, sizeof(int32_t) * (size_t)n_envs);
                if (e == cudaSuccess) e = cudaMemset(h->d_walk_ctr, 0, sizeof(int32_t) * (size_t)n_envs);
                // continuation pool: WalkCont entries for the sequential kernel, the (larger) piece queue + its flags and per-walk counters only with PCT_B200_WALK=fork
                h->contq_env_bytes = h->walk_fork ? sizeof(WalkPiece) * (size_t)WALK_PIECES_PER_ENV : sizeof(WalkCont) * (size_t)WALK_CONT_PER_ENV;
                if (e == cudaSuccess) e = cudaMalloc((void **)&h->d_contq, h->contq_env_bytes * (size_t)n_envs);
                if (e == cudaSuccess) e = cudaMalloc(&h->d_cont_ctr, sizeof(int32_t) * 8 * ((size_t)n_envs + 1));  // eight counters per (possible) env range
                if (e == cudaSuccess) e = cudaMemset(h->d_cont_ctr, 0, sizeof(int32_t) * 8 * ((size_t)n_envs + 1));
                if (e == cudaSuccess && h->walk_fork) e = cudaMalloc(&h->d_piece_ready, sizeof(int32_t) * (size_t)WALK_PIECES_PER_ENV * (size_t)n_envs);
                if (e == cudaSuccess && h->walk_fork) e = cudaMemset(h->d_piece_ready, 0, sizeof(int32_t) * (size_t)WALK_PIECES_PER_ENV * (size_t)n_envs);
                if (e == cudaSuccess && h->walk_fork) e = cudaMalloc(&h->d_walk_pend, sizeof(int32_t) * (size_t)CAND_MAX * (size_t)n_envs);
            }
            h->lpt = !h->k3_block;   // heaviest-env-first block order (pct_discrete.cu, order_lookup / order_file); PCT_B200_LPT=0 disables
            if (const char *lv = getenv("PCT_B200_LPT")) h->lpt = atoi(lv) != 0 && !h->k3_block;
            if (e == cudaSuccess && h->lpt) {
                // parity + two 64-bucket histograms + two sets of per-bucket env lists; starts as "every env in the lightest bucket, in env order"
                const size_t words = 2 + 2 * 64 + 2 * 64 * (size_t)n_envs;
                e = cudaMalloc(&h->d_order, sizeof(int32_t) * words);
                if (e == cudaSuccess) e = cudaMemset(h->d_order, 0, sizeof(int32_t) * words);
                if (e == cudaSuccess) {
                    std::vector<int32_t> id((size_t)n_envs);
                    for (int i = 0; i < n_envs; i++) id[i] = i;
                    const int32_t n32 = n_envs;
                    e = cudaMemcpy(h->d_order + 2 + 63, &n32, sizeof n32, cudaMemcpyHostToDevice);
                    if (e == cudaSuccess) e = cudaMemcpy(h->d_order + 2 + 128 + 63 * (size_t)n_envs, id.data(), sizeof(int32_t) * id.size(), cudaMemcpyHostToDevice);
                }
            }
        } else {
            int rc = continuous_create(h);
            if (rc != PCT_OK) { g_create_err = h->err; delete h; return rc; }
        }
    }
    if (e != cudaSuccess) {
        g_create_err = std::string("pct_create: ") + cudaGetErrorString(e);
        pct_destroy(h);
        return PCT_ERR_CUDA;
    }
    *out = h;
    return PCT_OK;
}

void pct_destroy(pct_handle h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->cfg.domain == PCT_CONTINUOUS) continuous_destroy(h);
    cudaFree(h->d_order);
    cudaFree(h->d_walkq); cudaFree(h->d_walk_ctr); cudaFree(h->d_contq); cudaFree(h->d_cont_ctr); cudaFree(h->d_piece_ready); cudaFree(h->d_walk_pend);
    cudaFree(h->d_hstate); cudaFree(h->d_hstate_c); cudaFree(h->d_query_c); cudaFree(h->d_query); cudaFree(h->d_aux);
    cudaFree(h->d_ready);
    cudaFree(h->d_hot); cudaFree(h->d_cold); cudaFree(h->d_item_set); cudaFree(h->d_stream); cudaFree(h->d_row_hash);
    cudaFree(h->d_obs); cudaFree(h->d_act); cudaFree(h->d_idx); cudaFree(h->d_rew); cudaFree(h->d_done); cudaFree(h->d_info);
    for (cudaEvent_t ev : h->prof_ev) if (ev) cudaEventDestroy(ev);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    for (int gi = 1; gi < 8; gi++) {
        if (h->sub[gi]) cudaStreamDestroy(h->sub[gi]);
        if (h->ev_join[gi]) cudaEventDestroy(h->ev_join[gi]);
    }
    delete h;
}

int pct_set_item_set(pct_handle h, const double *items_xyz, int32_t n_items) {
    if (!h || !items_xyz || n_items <= 0) return PCT_ERR_INVALID;
    CK(h, cudaSetDevice(h->device));
    cudaFree(h->d_item_set);
    h->d_item_set = nullptr;
    CK(h, cudaMalloc(&h->d_item_set, sizeof(double) * 3 * (size_t)n_items));
    CK(h, cudaMemcpy(h->d_item_set, items_xyz, sizeof(double) * 3 * (size_t)n_items, cudaMemcpyHostToDevice));
    h->n_items = n_items;
    h->item_set_hash = splitmix64(fnv1a(FNV_SEED, items_xyz, sizeof(double) * 3 * (size_t)n_items));
    return PCT_OK;
}

int pct_set_item_stream(pct_handle h, const double *items_xyzd, int32_t len) {
    if (!h || !items_xyzd || len <= 0) return PCT_ERR_INVALID;
    CK(h, cudaSetDevice(h->device));
    cudaFree(h->d_stream);
    h->d_stream = nullptr;
    const size_t bytes = sizeof(double) * 4 * (size_t)len * (size_t)h->n_envs;
    CK(h, cudaMalloc(&h->d_stream, bytes));
    CK(h, cudaMemcpy(h->d_stream, items_xyzd, bytes, cudaMemcpyHostToDevice));
    std::vector<uint64_t> rows((size_t)h->n_envs);
    const size_t row_bytes = sizeof(double) * 4 * (size_t)len;
    for (int i = 0; i < h->n_envs; i++) rows[i] = splitmix64(fnv1a(FNV_SEED, (const char *)items_xyzd + row_bytes * i, row_bytes));
    if (!h->d_row_hash) CK(h, cudaMalloc(&h->d_row_hash, sizeof(uint64_t) * (size_t)h->n_envs));
    CK(h, cudaMemcpy(h->d_row_hash, rows.data(), sizeof(uint64_t) * rows.size(), cudaMemcpyHostToDevice));
    h->stream_len = len;
    h->item_mode = PCT_ITEMS_STREAM;
    return PCT_OK;
}

int pct_set_trajectory_length(pct_handle h, int32_t traj_len) {
    if (!h || traj_len < 0) return PCT_ERR_INVALID;
    h->traj_len = traj_len;
    return PCT_OK;
}

// enqueue reset / step of the env range [off, off + cnt) on stream `gs`; all buffer pointers are BASE pointers
// Delta observation writes: called once per reset / step with the caller's observation buffer.  A buffer other than the one the
// previous call wrote may hold anything, so its row counts are reset to "all rows" (by the launches of this step, on their streams).
static void begin_obs(pct_handle h, const void *obs) {
    if (!h->obs_delta) return;
    h->fill_pending = obs != h->tracked_obs;
    h->tracked_obs = obs;
}

static int launch_range(pct_handle h, int mode, int off, int cnt, const void *actions, int action_f64, const int32_t *leaf_idx, void *obs,
                        float *rew, uint8_t *done, pct_step_info *info, cudaStream_t gs, bool whole_batch) {
    const size_t osz = h->cfg.obs_dtype == PCT_F64 ? 8 : 4, asz = action_f64 ? 8 : 4;
    DParams p{};
    p.hot = h->d_hot + off; p.cold = h->d_cold + off; p.n_envs = cnt;
    p.W = (int)h->cfg.container_size[0]; p.L = (int)h->cfg.container_size[1]; p.H = (int)h->cfg.container_size[2];
    p.nb = h->cfg.internal_node_holder; p.nl = h->cfg.leaf_node_holder; p.setting = h->cfg.setting;
    p.low_bound = h->cfg.size_minimum; p.lnes = h->cfg.lnes; p.shuffle = h->cfg.shuffle;
    p.item_mode = h->item_mode; p.item_set = h->d_item_set; p.n_items = h->n_items;
    p.stream = h->d_stream ? h->d_stream + (size_t)off * h->stream_len * 4 : nullptr; p.stream_len = h->stream_len; p.traj_len = h->traj_len;
    p.seed = h->cfg.seed; p.env_id_base = h->cfg.env_id_base + off; p.env_id_base0 = h->cfg.env_id_base;
    p.actions = actions ? (const char *)actions + (size_t)off * 9 * asz : nullptr; p.action_f64 = action_f64;
    p.leaf_idx = leaf_idx ? leaf_idx + off : nullptr;
    p.obs = (char *)obs + (size_t)off * h->obs_len * osz; p.obs_f64 = h->cfg.obs_dtype == PCT_F64;
    p.reward = rew ? rew + off : nullptr; p.done = done ? done + off : nullptr; p.info = info ? info + off : nullptr; p.mode = mode;
    p.dbg = (long long *)h->dbg;
    p.order = (h->lpt && whole_batch) ? h->d_order : nullptr;
    p.keep_draw = h->did_reset ? 1 : 0; p.no_auto_reset = h->cfg.no_auto_reset;
    // overlapped launch mode: not while a CUDA graph is being captured (the epoch would be frozen into the graph and a replay
    // would find the flags of the previous replay already set), not under the per-kernel profiler, not with the LPT permutation
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(gs, &cap);
    if (h->overlap && !h->prof_on && cap == cudaStreamCaptureStatusNone) {
        p.ready = h->d_ready + 2 * (size_t)off;
        p.epoch = ++h->epoch;
    }
    if (h->d_aux) {
        if (h->obs_delta && h->fill_pending) launch_fill_prev(h->d_aux + off, cnt, p.nb, p.nl, gs);
        p.aux = h->d_aux + off;
        p.opt = (h->obs_delta ? PCT_OPT_DELTA : 0) | (h->alias_mode ? PCT_OPT_ALIAS : 0);
    }
    if (h->k3_block) p.opt |= PCT_OPT_K3_BLOCK;
    if (h->no_emit_pdl) p.opt |= PCT_OPT_NO_EMIT_PDL;
    cudaEvent_t *prof = nullptr;
    if (h->prof_on && mode == 1 && whole_batch) {
        if ((size_t)(h->prof_steps + 1) * 4 > h->prof_ev.size()) {
            const size_t old = h->prof_ev.size();
            h->prof_ev.resize(old + 4096, nullptr);
            for (size_t i = old; i < h->prof_ev.size(); i++) CK(h, cudaEventCreate(&h->prof_ev[i]));
        }
        prof = &h->prof_ev[(size_t)h->prof_steps * 4];
        h->prof_steps++;
    }
    p.walkq = h->d_walkq ? h->d_walkq + (size_t)off * CAND_MAX : nullptr;  // env ranges stepped concurrently (pct_step_host's staged path) own disjoint slices
    p.walk_ctr = h->d_walk_ctr ? h->d_walk_ctr + off : nullptr;
    p.contq = h->d_contq ? (WalkCont *)((char *)h->d_contq + (size_t)off * h->contq_env_bytes) : nullptr;  // an env range's slice of the pool
    p.cont_ctr = h->d_cont_ctr ? h->d_cont_ctr + 8 * (size_t)off : nullptr;
    p.walk_lanes = h->walk_lanes; p.walk_lanes_tall = h->walk_lanes_tall;
    p.walk_fork = h->walk_fork ? 1 : 0; p.walk_blocks = h->walk_blocks; p.walk_keep = h->walk_keep; p.piece_cap = cnt * WALK_PIECES_PER_ENV;
    p.piece_ready = h->d_piece_ready ? h->d_piece_ready + (size_t)off * WALK_PIECES_PER_ENV : nullptr;
    p.walk_pend = h->d_walk_pend ? h->d_walk_pend + (size_t)off * CAND_MAX : nullptr;
    CK(h, launch_discrete(p, gs, prof));
    h->launches += discrete_kernels_per_step(p);
    return PCT_OK;
}

static int check_item_source(pct_handle h) {
    if (h->item_mode == PCT_ITEMS_RANDOM && !(h->cfg.domain == PCT_CONTINUOUS && h->cfg.sample_from_distribution) && !h->d_item_set) {
        h->err = "no item source: call pct_set_item_set or pct_set_item_stream first";
        return PCT_ERR_STATE;
    }
    if (h->item_mode == PCT_ITEMS_STREAM && !h->d_stream) { h->err = "item stream not set"; return PCT_ERR_STATE; }
    return PCT_OK;
}

static int launch(pct_handle h, int mode, const void *actions, int action_f64, const int32_t *leaf_idx, void *obs, float *rew, uint8_t *done,
                  pct_step_info *info, cudaStream_t st) {
    int rc = check_item_source(h);
    if (rc) return rc;
    CK(h, cudaSetDevice(h->device));
    begin_obs(h, obs);
    if (h->cfg.domain == PCT_CONTINUOUS) {
        rc = continuous_launch(h, mode, actions, action_f64, leaf_idx, obs, rew, done, info, st);
        if (rc == PCT_OK) h->launches++;
        return rc;
    }
    // PCT_B200_GROUPS > 1: the batch is cut into contiguous env ranges, each enqueued on its own internal stream between a
    // fork and a join event on the caller's stream (measured: no gain for the device-resident path, see DESIGN.md).
    const int G = h->groups;
    if (G > 1) CK(h, cudaEventRecord(h->ev_fork, st));
    for (int gi = 0; gi < G; gi++) {
        const int off = (int)((int64_t)h->n_envs * gi / G), cnt = (int)((int64_t)h->n_envs * (gi + 1) / G) - off;
        if (cnt <= 0) continue;
        cudaStream_t gs = gi == 0 ? st : h->sub[gi];
        if (gi > 0) CK(h, cudaStreamWaitEvent(gs, h->ev_fork, 0));
        rc = launch_range(h, mode, off, cnt, actions, action_f64, leaf_idx, obs, rew, done, info, gs, G == 1);
        if (rc) return rc;
        if (gi > 0) {
            CK(h, cudaEventRecord(h->ev_join[gi], gs));
            CK(h, cudaStreamWaitEvent(st, h->ev_join[gi], 0));
        }
    }
    h->fill_pending = false;
    return PCT_OK;
}

int pct_reset(pct_handle h, void *d_obs, void *stream) {
    if (!h || !d_obs) return PCT_ERR_INVALID;
    int rc = launch(h, 0, nullptr, 0, nullptr, d_obs, nullptr, nullptr, nullptr, (cudaStream_t)stream);
    if (rc == PCT_OK) h->did_reset = true;
    return rc;
}

int pct_step(pct_handle h, const void *d_actions, int32_t action_f64, const int32_t *d_leaf_idx, void *d_obs, float *d_reward,
             uint8_t *d_done, pct_step_info *d_info, void *stream) {
    if (!h || !d_obs || !d_reward || !d_done) return PCT_ERR_INVALID;
    if ((d_actions == nullptr) == (d_leaf_idx == nullptr)) { h->err = "pct_step: pass exactly one of d_actions / d_leaf_idx"; return PCT_ERR_INVALID; }
    if (!h->did_reset) { h->err = "pct_step before pct_reset"; return PCT_ERR_STATE; }
    return launch(h, 1, d_actions, action_f64, d_leaf_idx, d_obs, d_reward, d_done, d_info, (cudaStream_t)stream);
}

static int ensure_staging(pct_handle h) {
    if (h->d_obs) return PCT_OK;
    const size_t n = (size_t)h->n_envs;
    CK(h, cudaMalloc(&h->d_obs, n * h->obs_len * (h->cfg.obs_dtype == PCT_F64 ? 8 : 4)));
    CK(h, cudaMalloc(&h->d_act, n * 9 * 8));
    CK(h, cudaMalloc(&h->d_idx, n * 4));
    CK(h, cudaMalloc(&h->d_rew, n * 4));
    CK(h, cudaMalloc(&h->d_done, n));
    CK(h, cudaMalloc(&h->d_info, n * sizeof(pct_step_info)));
    return PCT_OK;
}

int pct_reset_host(pct_handle h, void *h_obs) {
    if (!h || !h_obs) return PCT_ERR_INVALID;
    CK(h, cudaSetDevice(h->device));
    int rc = ensure_staging(h);
    if (rc) return rc;
    rc = pct_reset(h, h->d_obs, h->own_stream);
    if (rc) return rc;
    const size_t ob = (size_t)h->n_envs * h->obs_len * (h->cfg.obs_dtype == PCT_F64 ? 8 : 4);
    CK(h, cudaMemcpyAsync(h_obs, h->d_obs, ob, cudaMemcpyDeviceToHost, h->own_stream));
    CK(h, cudaStreamSynchronize(h->own_stream));
    return PCT_OK;
}

int pct_step_host(pct_handle h, const void *h_actions, int32_t action_f64, const int32_t *h_leaf_idx, void *h_obs, float *h_reward,
                  uint8_t *h_done, pct_step_info *h_info) {
    if (!h || !h_obs || !h_reward || !h_done) return PCT_ERR_INVALID;
    if ((h_actions == nullptr) == (h_leaf_idx == nullptr)) { h->err = "pct_step_host: pass exactly one of actions / leaf_idx"; return PCT_ERR_INVALID; }
    if (!h->did_reset) { h->err = "pct_step_host before pct_reset"; return PCT_ERR_STATE; }
    CK(h, cudaSetDevice(h->device));
    int rc = ensure_staging(h);
    if (rc) return rc;
    rc = check_item_source(h);
    if (rc) return rc;
    const size_t osz = h->cfg.obs_dtype == PCT_F64 ? 8 : 4, asz = action_f64 ? 8 : 4;
    if (h->host_zero_copy) {
        // Zero-copy observation delivery (the default; PCT_B200_HOST_ZEROCOPY=0 disables): when h_obs is pinned (mapped under UVA) the feasibility
        // kernel writes every env's observation straight into it over PCIe as that env finishes — no staging copy after the kernels
        // and no env-range pipeline; the whole batch runs as ONE launch sequence (overlapped mode, heaviest-env-first order).  The
        // observation is write-only for the kernels.  Actions and the small reward / done / info records keep their staged copies
        // (info is read back by the kernels).  Unpinned h_obs: the staged path below.
        void *obs_alias = nullptr;
        if (cudaHostGetDevicePointer(&obs_alias, h_obs, 0) == cudaSuccess && obs_alias) {
            cudaStream_t st = h->own_stream;
            const size_t n = (size_t)h->n_envs;
            // reward / done are write-only for the kernels too: when their buffers are pinned the apply kernel writes them straight into the mapped
            // host buffers (posted PCIe writes), saving two of the four staging copies.  Actions / leaf indices (READ by the apply kernel) and info
            // (read-modify-write by the emit kernel) keep their staged copies: measured (round 2, call 14), device-side READS of mapped host memory
            // put a PCIe round trip on every env's critical path — pct_step_host went from 426 to 661 us per step with everything mapped.
            auto alias = [](const void *hp) -> void * {
                void *d = nullptr;
                if (hp && cudaHostGetDevicePointer(&d, const_cast<void *>(hp), 0) == cudaSuccess && d) return d;
                (void)cudaGetLastError();
                return nullptr;
            };
            void *a_act = nullptr, *a_rew = alias(h_reward), *a_done = alias(h_done), *a_info = nullptr;
            if (!a_act) {
                if (h_actions) CK(h, cudaMemcpyAsync(h->d_act, h_actions, n * 9 * asz, cudaMemcpyHostToDevice, st));
                else CK(h, cudaMemcpyAsync(h->d_idx, h_leaf_idx, n * 4, cudaMemcpyHostToDevice, st));
            }
            const void *k_act = h_actions ? (a_act ? a_act : h->d_act) : nullptr;
            const int32_t *k_idx = h_actions ? nullptr : (a_act ? (const int32_t *)a_act : h->d_idx);
            pct_step_info *k_info = h_info ? (a_info ? (pct_step_info *)a_info : h->d_info) : h->d_info;
            rc = launch(h, 1, k_act, action_f64, k_idx, obs_alias, a_rew ? (float *)a_rew : h->d_rew, a_done ? (uint8_t *)a_done : h->d_done, k_info, st);
            if (rc) return rc;
            if (!a_rew) CK(h, cudaMemcpyAsync(h_reward, h->d_rew, n * 4, cudaMemcpyDeviceToHost, st));
            if (!a_done) CK(h, cudaMemcpyAsync(h_done, h->d_done, n, cudaMemcpyDeviceToHost, st));
            if (h_info && !a_info) CK(h, cudaMemcpyAsync(h_info, h->d_info, n * sizeof(pct_step_info), cudaMemcpyDeviceToHost, st));
            CK(h, cudaStreamSynchronize(st));
            return PCT_OK;
        }
        (void)cudaGetLastError();  // not a mapped host pointer
    }
    // Software pipeline over env ranges: range g's device->host copies overlap the kernels of range g+1 (envs are
    // independent, so the ranges need no ordering between them).  Host buffers should be pinned.
    const int G = (h->cfg.domain == PCT_DISCRETE && h->n_envs >= 1024) ? h->host_groups : 1;
    if (G > 1) begin_obs(h, h->d_obs);  // G == 1 goes through launch(), which does it
    for (int gi = 0; gi < G; gi++) {
        const int off = (int)((int64_t)h->n_envs * gi / G), cnt = (int)((int64_t)h->n_envs * (gi + 1) / G) - off;
        if (cnt <= 0) continue;
        cudaStream_t st = gi == 0 ? h->own_stream : h->sub[gi];
        if (h_actions) CK(h, cudaMemcpyAsync((char *)h->d_act + (size_t)off * 9 * asz, (const char *)h_actions + (size_t)off * 9 * asz, (size_t)cnt * 9 * asz, cudaMemcpyHostToDevice, st));
        else CK(h, cudaMemcpyAsync(h->d_idx + off, h_leaf_idx + off, (size_t)cnt * 4, cudaMemcpyHostToDevice, st));
        if (G == 1) rc = launch(h, 1, h_actions ? h->d_act : nullptr, action_f64, h_actions ? nullptr : h->d_idx, h->d_obs, h->d_rew, h->d_done, h->d_info, st);
        else rc = launch_range(h, 1, off, cnt, h_actions ? h->d_act : nullptr, action_f64, h_actions ? nullptr : h->d_idx, h->d_obs, h->d_rew, h->d_done, h->d_info, st, false);
        if (rc) return rc;
        CK(h, cudaMemcpyAsync((char *)h_obs + (size_t)off * h->obs_len * osz, (char *)h->d_obs + (size_t)off * h->obs_len * osz, (size_t)cnt * h->obs_len * osz, cudaMemcpyDeviceToHost, st));
        CK(h, cudaMemcpyAsync(h_reward + off, h->d_rew + off, (size_t)cnt * 4, cudaMemcpyDeviceToHost, st));
        CK(h, cudaMemcpyAsync(h_done + off, h->d_done + off, (size_t)cnt, cudaMemcpyDeviceToHost, st));
        if (h_info) CK(h, cudaMemcpyAsync(h_info + off, h->d_info + off, (size_t)cnt * sizeof(pct_step_info), cudaMemcpyDeviceToHost, st));
    }
    h->fill_pending = false;
    for (int gi = 0; gi < G; gi++) CK(h, cudaStreamSynchronize(gi == 0 ? h->own_stream : h->sub[gi]));
    return PCT_OK;
}

int pct_policy_random(pct_handle h, int32_t *d_leaf_idx, uint64_t seed, int64_t t, void *stream) {
    if (!h || !d_leaf_idx) return PCT_ERR_INVALID;
    if (!h->did_reset) { h->err = "pct_policy_random before pct_reset"; return PCT_ERR_STATE; }
    CK(h, cudaSetDevice(h->device));
    if (h->cfg.domain == PCT_CONTINUOUS) {
        int rc = continuous_policy_random(h, d_leaf_idx, seed, t, (cudaStream_t)stream);
        if (rc == PCT_OK) h->launches++;
        return rc;
    }
    CK(h, launch_policy_random_discrete(h->d_hot, h->n_envs, h->cfg.env_id_base, seed, t, d_leaf_idx, (cudaStream_t)stream));
    h->launches++;
    return PCT_OK;
}

int pct_policy_random_dev(pct_handle h, int32_t *d_leaf_idx, uint64_t seed, const int64_t *d_t, void *stream) {
    if (!h || !d_leaf_idx || !d_t) return PCT_ERR_INVALID;
    if (!h->did_reset) { h->err = "pct_policy_random_dev before pct_reset"; return PCT_ERR_STATE; }
    if (h->cfg.domain != PCT_DISCRETE) { h->err = "pct_policy_random_dev: discrete domain only"; return PCT_ERR_INVALID; }
    CK(h, cudaSetDevice(h->device));
    CK(h, launch_policy_random_discrete(h->d_hot, h->n_envs, h->cfg.env_id_base, seed, 0, d_leaf_idx, (cudaStream_t)stream, d_t));
    h->launches++;
    return PCT_OK;
}

// DParams of the whole batch for the read-only selection kernels (no action / observation buffers)
static DParams state_params(pct_handle h) {
    DParams p{};
    p.hot = h->d_hot; p.cold = h->d_cold; p.n_envs = h->n_envs;
    p.W = (int)h->cfg.container_size[0]; p.L = (int)h->cfg.container_size[1]; p.H = (int)h->cfg.container_size[2];
    p.nb = h->cfg.internal_node_holder; p.nl = h->cfg.leaf_node_holder; p.setting = h->cfg.setting;
    p.low_bound = h->cfg.size_minimum; p.lnes = h->cfg.lnes;
    p.item_mode = h->item_mode; p.item_set = h->d_item_set; p.n_items = h->n_items;
    p.seed = h->cfg.seed; p.env_id_base = h->cfg.env_id_base; p.env_id_base0 = h->cfg.env_id_base;
    return p;
}

int pct_heuristic_actions(pct_handle h, int32_t heuristic, float *d_rows, uint64_t seed, int64_t t, void *stream) {
    if (!h || !d_rows) return PCT_ERR_INVALID;
    if (heuristic < PCT_H_LSAH || heuristic > PCT_H_RANDOM) { h->err = "pct_heuristic_actions: unknown heuristic"; return PCT_ERR_INVALID; }
    if (h->cfg.domain != PCT_DISCRETE) { h->err = "pct_heuristic_actions: discrete domain only"; return PCT_ERR_INVALID; }
    if (!h->did_reset) { h->err = "pct_heuristic_actions before pct_reset"; return PCT_ERR_STATE; }
    CK(h, cudaSetDevice(h->device));
    DParams p = state_params(h);
    if (heuristic == PCT_H_BR && !h->d_item_set) { h->err = "PCT_H_BR scores an EMS by the item types that fit: call pct_set_item_set"; return PCT_ERR_STATE; }
    if ((heuristic == PCT_H_HM || heuristic == PCT_H_MACS || heuristic == PCT_H_RANDOM) && (p.W > HEUR_SIDE_MAX || p.L > HEUR_SIDE_MAX)) {
        h->err = "PCT_H_HM / PCT_H_MACS / PCT_H_RANDOM need container sides <= 32";
        return PCT_ERR_INVALID;
    }
    HParams hp{};
    hp.code = heuristic; hp.rows = d_rows; hp.hstate = h->d_hstate; hp.seed = seed; hp.t = t;
    CK(h, launch_heuristic_discrete(p, hp, (cudaStream_t)stream));
    h->launches++;
    return PCT_OK;
}

int pct_heuristic_actions_f64(pct_handle h, int32_t heuristic, double *d_rows, void *stream) {
    if (!h || !d_rows) return PCT_ERR_INVALID;
    if (h->cfg.domain != PCT_CONTINUOUS) { h->err = "pct_heuristic_actions_f64: continuous domain only (discrete: pct_heuristic_actions)"; return PCT_ERR_INVALID; }
    if (heuristic != PCT_H_LSAH && heuristic != PCT_H_ONLINEBPH && heuristic != PCT_H_BR) {  // tools.py:217-218
        h->err = "only LSAH, OnlineBPH, and BR allowed for continuous environment";
        return PCT_ERR_INVALID;
    }
    if (!h->did_reset) { h->err = "pct_heuristic_actions_f64 before pct_reset"; return PCT_ERR_STATE; }
    if (heuristic == PCT_H_BR && !h->d_item_set) { h->err = "PCT_H_BR scores an EMS by the item types that fit: call pct_set_item_set"; return PCT_ERR_STATE; }
    CK(h, cudaSetDevice(h->device));
    int rc = continuous_heuristic(h, heuristic, d_rows, h->d_hstate_c, (cudaStream_t)stream);
    if (rc != PCT_OK) return rc;
    h->launches++;
    return PCT_OK;
}

int pct_query_placement_f64(pct_handle h, int32_t env, const double dims[3], double lx, double ly, double density, int32_t *feasible,
                            double *rest_height) {
    if (!h || !dims || !feasible || !rest_height || env < 0 || env >= h->n_envs) return PCT_ERR_INVALID;
    if (h->cfg.domain != PCT_CONTINUOUS) { h->err = "pct_query_placement_f64: continuous domain only (discrete: pct_query_placement)"; return PCT_ERR_INVALID; }
    if (!h->did_reset) { h->err = "pct_query_placement_f64 before pct_reset"; return PCT_ERR_STATE; }
    CK(h, cudaSetDevice(h->device));
    if (!h->d_query_c) CK(h, cudaMalloc(&h->d_query_c, sizeof(double) * 2));
    const double q[5] = {dims[0], dims[1], dims[2], lx, ly};
    CK(h, cudaDeviceSynchronize());
    int rc = continuous_query(h, env, q, density, h->d_query_c, h->own_stream);
    if (rc != PCT_OK) return rc;
    h->launches++;
    double out[2];
    CK(h, cudaMemcpyAsync(out, h->d_query_c, sizeof out, cudaMemcpyDeviceToHost, h->own_stream));
    CK(h, cudaStreamSynchronize(h->own_stream));
    *feasible = out[0] != 0.0;
    *rest_height = out[1];
    return PCT_OK;
}

int pct_query_placement(pct_handle h, int32_t env, const int32_t dims[3], int32_t lx, int32_t ly, double density, int32_t *feasible,
                        int32_t *rest_height, int32_t *height_map) {
    if (!h || !dims || !feasible || !rest_height || env < 0 || env >= h->n_envs) return PCT_ERR_INVALID;
    if (h->cfg.domain != PCT_DISCRETE) { h->err = "pct_query_placement: discrete domain only"; return PCT_ERR_INVALID; }
    if (!h->did_reset) { h->err = "pct_query_placement before pct_reset"; return PCT_ERR_STATE; }
    CK(h, cudaSetDevice(h->device));
    DParams p = state_params(h);
    if (p.W > HEUR_SIDE_MAX || p.L > HEUR_SIDE_MAX) { h->err = "pct_query_placement needs container sides <= 32"; return PCT_ERR_INVALID; }
    const size_t cells = (size_t)p.W * p.L;
    if (!h->d_query) CK(h, cudaMalloc(&h->d_query, sizeof(int32_t) * (2 + HEUR_SIDE_MAX * HEUR_SIDE_MAX)));
    HParams hp{};
    hp.code = PCT_H_QUERY_; hp.q_env = env; hp.q_den = density; hp.q_out = h->d_query;
    hp.q[0] = dims[0]; hp.q[1] = dims[1]; hp.q[2] = dims[2]; hp.q[3] = lx; hp.q[4] = ly;
    CK(h, cudaDeviceSynchronize());
    CK(h, launch_heuristic_discrete(p, hp, h->own_stream));
    h->launches++;
    std::vector<int32_t> out(2 + cells);
    CK(h, cudaMemcpyAsync(out.data(), h->d_query, sizeof(int32_t) * out.size(), cudaMemcpyDeviceToHost, h->own_stream));
    CK(h, cudaStreamSynchronize(h->own_stream));
    *feasible = out[0];
    *rest_height = out[1];
    if (height_map) memcpy(height_map, out.data() + 2, sizeof(int32_t) * cells);
    return PCT_OK;
}

int pct_get_state(pct_handle h, int32_t env, pct_state_dump *out) {
    if (!h || !out || env < 0 || env >= h->n_envs) return PCT_ERR_INVALID;
    CK(h, cudaSetDevice(h->device));
    CK(h, cudaDeviceSynchronize());
    if (h->cfg.domain == PCT_CONTINUOUS) return continuous_get_state(h, env, out);
    DEnvHot hot;
    std::vector<double> den(NB_MAX);
    CK(h, cudaMemcpy(&hot, h->d_hot + env, sizeof(hot), cudaMemcpyDeviceToHost));
    CK(h, cudaMemcpy(den.data(), (const char *)(h->d_cold + env) + offsetof(DEnvCold, density), sizeof(double) * NB_MAX, cudaMemcpyDeviceToHost));
    memset(out, 0, sizeof(*out));
    out->n_boxes = hot.h.n_box; out->n_ems = hot.h.n_ems; out->n_leaf = hot.h.n_leaf; out->flags = hot.h.flags;
    out->draw_pos = hot.h.draw_pos;
    for (int i = 0; i < 3; i++) out->next_box[i] = hot.h.next_box[i];
    out->next_den = hot.h.next_den;
    for (int i = 0; i < hot.h.n_box && i < 80; i++) {
        for (int t = 0; t < 6; t++) out->boxes[i][t] = hot.box[i][t];
        out->boxes[i][6] = h->cfg.setting == 3 ? den[i] : 1.0;
    }
    for (int i = 0; i < hot.h.n_ems && i < 256 && i < E_MAX; i++)
        for (int t = 0; t < 6; t++) out->ems[i][t] = hot.ems[i][t];
    return PCT_OK;
}

int64_t pct_env_record_bytes(pct_handle h) {
    if (!h) return 0;
    return h->cfg.domain == PCT_CONTINUOUS ? continuous_record_bytes() : discrete_record_bytes();
}

// save (load == 0) / load (load == 1): argument checks, then one stream-ordered kernel; no host synchronisation, no allocation
static int env_records(pct_handle h, const int32_t *d_env_ids, int32_t n, const void *d_records, void *d_obs, int32_t *d_status, void *stream,
                       int load) {
    const char *what = load ? "pct_load_envs" : "pct_save_envs";
    if (!h) return PCT_ERR_INVALID;
    if (n < 0 || (n > 0 && !d_records) || (!d_env_ids && n != h->n_envs && n != 0)) {
        h->err = std::string(what) + ": bad arguments (d_env_ids == NULL means all n_envs envs in order)";
        return PCT_ERR_INVALID;
    }
    if (((uintptr_t)d_records & 15) != 0) { h->err = std::string(what) + ": records must be 16-byte aligned"; return PCT_ERR_INVALID; }
    if (load && !h->did_reset) { h->err = "pct_load_envs before pct_reset"; return PCT_ERR_STATE; }
    CK(h, cudaSetDevice(h->device));
    RecArgs s{};
    s.ids = d_env_ids; s.n = n; s.rec = (unsigned char *)const_cast<void *>(d_records); s.rec_bytes = pct_env_record_bytes(h);
    s.fingerprint = config_fingerprint(h);
    s.row_hash = h->item_mode == PCT_ITEMS_STREAM ? h->d_row_hash : nullptr;
    s.alias = h->alias_mode && h->d_aux && h->cfg.setting != 2;
    s.status = d_status;
    const cudaStream_t st = (cudaStream_t)stream;
    if (h->cfg.domain == PCT_CONTINUOUS) {
        s.hstate = h->d_hstate_c;
        const int rc = continuous_records(h, s, load, load ? d_obs : nullptr, st);
        if (rc == PCT_OK && n > 0) h->launches++;
        return rc;
    }
    s.hstate = h->d_hstate;
    DParams p = state_params(h);
    p.aux = h->d_aux;
    p.obs = load ? d_obs : nullptr;
    p.obs_f64 = h->cfg.obs_dtype == PCT_F64;
    CK(h, launch_records_discrete(p, s, load, st));
    if (n > 0) h->launches++;
    return PCT_OK;
}

int pct_save_envs(pct_handle h, const int32_t *d_env_ids, int32_t n, void *d_records, void *stream) {
    return env_records(h, d_env_ids, n, d_records, nullptr, nullptr, stream, 0);
}

int pct_load_envs(pct_handle h, const int32_t *d_env_ids, int32_t n, const void *d_records, void *d_obs, int32_t *d_status, void *stream) {
    return env_records(h, d_env_ids, n, d_records, d_obs, d_status, stream, 1);
}

int32_t pct_obs_len(pct_handle h) { return h ? h->obs_len : 0; }
int32_t pct_num_envs(pct_handle h) { return h ? h->n_envs : 0; }
int64_t pct_state_bytes_per_env(pct_handle h) {
    if (!h) return 0;
    if (h->cfg.domain == PCT_CONTINUOUS) return continuous_state_bytes();
    return (int64_t)(sizeof(DEnvHot) + sizeof(DEnvCold));
}
int64_t pct_kernel_launches(pct_handle h) { return h ? h->launches : 0; }
int pct_profile_enable(pct_handle h, int32_t on) {
    if (!h) return PCT_ERR_INVALID;
    h->prof_on = on ? 1 : 0;
    h->prof_steps = 0;
    return PCT_OK;
}
int pct_profile_read(pct_handle h, double ms_out[3], int32_t *n_steps) {
    if (!h || !ms_out || !n_steps) return PCT_ERR_INVALID;
    CK(h, cudaSetDevice(h->device));
    CK(h, cudaDeviceSynchronize());
    ms_out[0] = ms_out[1] = ms_out[2] = 0;
    for (int s = 0; s < h->prof_steps; s++)
        for (int k = 0; k < 3; k++) {
            float ms = 0;
            CK(h, cudaEventElapsedTime(&ms, h->prof_ev[(size_t)s * 4 + k], h->prof_ev[(size_t)s * 4 + k + 1]));
            ms_out[k] += ms;
        }
    *n_steps = h->prof_steps;
    return PCT_OK;
}
/* debug: device buffer of n_envs x 8 int64 phase timers (library built with -DPCT_PHASE_TIMERS) */
void pct_debug_set_timer_buffer(pct_handle h, void *d_buf) { if (h) h->dbg = d_buf; }

}  // extern "C"
