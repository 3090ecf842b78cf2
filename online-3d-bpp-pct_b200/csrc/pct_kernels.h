// Internal: device record layouts and kernel launch parameters shared by the kernels and the C-ABI layer.
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>
#include "pct_b200.h"

namespace pct {

constexpr int NB_MAX = 80;    // internal_node_holder capacity
constexpr int NL_MAX = 64;    // leaf_node_holder capacity
constexpr int EMS_TMP_MAX = 256;  // intermediate EMS list inside GENEMS (before EliminateInscribedEMS)
constexpr int E_MAX = 128;    // EMS list capacity (reference: unbounded python list; max observed 51)
constexpr int TAB_A = 2048;   // CPython-set emulation: largest table (<= 1228 distinct candidates)
constexpr int TAB_B = 512;
constexpr int WARPS_PER_BLOCK = 2;
constexpr int CAND_MAX = 1232;    // ordered candidate list capacity (K2 emits <= 1228 distinct candidates)
constexpr int FBITS_WORDS = 40;   // feasibility bits of <= 1280 candidates

constexpr int PCT_FLAG_BOX_OVERFLOW_ = PCT_FLAG_BOX_OVERFLOW;
constexpr int PCT_FLAG_BAD_ACTION_ = PCT_FLAG_BAD_ACTION;
constexpr int PCT_FLAG_EMS_OVERFLOW_ = PCT_FLAG_EMS_OVERFLOW;
constexpr int PCT_FLAG_CAND_OVERFLOW_ = PCT_FLAG_CAND_OVERFLOW;
typedef pct_step_info pct_step_info_;

constexpr int KSUP_SMALL = 8;    // supports handled with lane-local scratch
constexpr int KSUP_MAX = 32;     // supports handled with the per-env scratch in HBM (serialised by a lock)
constexpr int STAB_DEPTH = 14;   // DFS depth (levels of boxes on top of each other)
constexpr int STAB_SUP_POOL = 48;
constexpr int EDGE_MAX = 255;    // load edges per env; positions are uint8, 255 = NIL
constexpr int EDGE_NIL = 255;
// Staging areas of the apply kernel.  Small on purpose: its descent runs on ONE lane per warp, so every hot word of that lane's local-memory stack
// costs a whole 128-byte L1 line; 64 loads + 96 vertices per warp put the kernel at the 164 KB shared-memory carve-out (92 KB of L1), 16 + 32 at
// the 132 KB one (124 KB of L1): apply kernel 0.1126 -> 0.1075 ms (B200, 4096 envs; r2_c25).  Entries beyond the staged ones are read from L1 / L2.
#ifndef PCT_EDGE_STAGE
#define PCT_EDGE_STAGE 16
#endif
#ifndef PCT_POLY_STAGE
#define PCT_POLY_STAGE 32
#endif
constexpr int EDGE_STAGE = PCT_EDGE_STAGE;    // loads staged in shared memory by the apply kernel (serial descent reads would otherwise be HBM-latency bound)
constexpr int POLY_MAX = 256;                 // stored support-polygon vertices per env (boxes with >= 2 supports)
constexpr int POLY_STAGE = PCT_POLY_STAGE;    // vertices staged in shared memory

struct Stack4 { double cx, cy, cz, m; };

// Load-edge pool of one env.  Edges are appended when a box is placed (one per support, in support order), so the
// pool is a CSR by upper box: the supports of placed box u are lower[off[u] .. off[u+1]).  The loads resting on a
// box t (the reference's insertion-ordered `up_edges` dict of t) are the linked list first_in[t] -> next[..], which
// is in pool (= placement) order.  Index arrays live in the staged record (shared memory), the loads in HBM.
struct EdgePool {
    uint8_t *lower;        // [EDGE_MAX] supporting box of edge e
    uint8_t *next;         // [EDGE_MAX] next edge with the same lower box, EDGE_NIL at the end
    uint16_t *off;         // [NB_MAX + 1] CSR offsets by upper box
    uint8_t *first_in;     // [NB_MAX] first / last incoming edge of a box (EDGE_NIL if none)
    uint8_t *last_in;
    Stack4 *st;            // [EDGE_MAX] load centre xyz + mass (global memory)
    Stack4 *st_sm;         // the first EDGE_STAGE loads, staged in shared memory by a TMA bulk copy
    int n;                 // current count (lane-local copy; the REAL path writes it back)
    // support polygons (hull vertices already scaled down, x/y interleaved) of the placed boxes with >= 2 supports: the
    // reference stores bottom_whole_contact_area per box at placement (D:space.py:378-379); CSR by box.  A box with exactly two
    // supports has one more entry behind its vertices: the split direction of its load (split2_dir).
    uint16_t *poly_off;    // [NB_MAX + 2]
    double *poly;          // [POLY_MAX][2] global
    double *poly_sm;       // first POLY_STAGE vertices staged in shared memory
    int n_poly;
    __device__ __forceinline__ Stack4 &load(int q) const { return q < EDGE_STAGE ? st_sm[q] : st[q]; }
    __device__ __forceinline__ double *poly_at(int v) const { return v < POLY_STAGE ? poly_sm + 2 * v : poly + 2 * v; }
};

// Extra state of the ALIAS variant of the stability routine (the reference's Python object aliasing, DESIGN.md section 3 (b)): the
// reference keeps every box's stack in an object (`thisStack`) that `calculate_new_com` rewrites in place at every SET_EDGE, and the
// `up_edges` entries of a single support / of the direct support ARE that object.  Passed as the EdgePool& of stability_check<.., ALIAS = true>.
struct EdgePoolA : EdgePool {
    Stack4 *box_st;        // [NB_MAX + 1] thisStack of every placed box and of the box being placed
    uint8_t *e_upper;      // [EDGE_MAX] upper box of edge q
    uint32_t *e_alias;     // [(EDGE_MAX + 32) / 32] bit q: the entry is the upper box's own Stack object
};

// Per-env state of the opt-in kernel variants (one allocation, reached through DParams::aux):
//   PCT_OPT_ALIAS  K1: the three arrays of EdgePoolA
//   PCT_OPT_DELTA  K3: obs_prev = how many internal / leaf rows of the caller's observation buffer may be non-zero
struct DEnvAux {
    Stack4 box_st[NB_MAX + 1];
    uint8_t e_upper[EDGE_MAX + 1];
    uint32_t e_alias[(EDGE_MAX + 32) / 32];
    int32_t obs_prev[2];
};

// per-env HBM scratch for the rare big cases (k > KSUP_SMALL)
struct BigScratch {
    double rect[KSUP_MAX][4];
    double px[4 * KSUP_MAX], py[4 * KSUP_MAX];
    double hx[8 * KSUP_MAX], hy[8 * KSUP_MAX];
    double R[KSUP_MAX * KSUP_MAX], V[KSUP_MAX * KSUP_MAX], y[KSUP_MAX], row[KSUP_MAX], x[KSUP_MAX];
};


// ---- discrete domain -----------------------------------------------------------------------------------
// "Hot" record: everything a step reads and rewrites, one contiguous 16-byte-aligned blob per env so that a
// single TMA bulk copy stages it into shared memory and another one writes it back.
struct alignas(16) DHdr {  // 64 bytes
    int32_t n_box, n_ems, n_leaf, flags;
    int64_t draw_pos;      // draws consumed from the item source (one per reset + one per placed box)
    double ep_reward;      // Monitor: sum of rewards of the running episode
    int32_t next_box[3];
    int32_t n_edge;        // load edges in the pool (stability settings)
    double next_den;
    int32_t vol_sum;       // sum of packed volumes (get_ratio numerator)
    int32_t ep_len;
    int32_t n_cand;
    int32_t n_poly;        // vertices in the polygon pool
    int64_t item_env;      // global env id whose item sequence this env follows (its own id unless a saved record was loaded into it)
};
struct alignas(16) DEnvHot {
    DHdr h;
    int16_t box[NB_MAX][6];  // lx,ly,lz,hx,hy,hz  (placement order)
    int16_t ems[E_MAX][6];   // x1,y1,z1,x2,y2,z2  (reference list order)
    // --- everything above is what the candidate kernel needs (HOT_PREFIX bytes) ---
    uint16_t e_off[NB_MAX + 2];
    uint8_t e_lower[EDGE_MAX + 1], e_next[EDGE_MAX + 1];
    uint8_t first_in[NB_MAX], last_in[NB_MAX];
    uint16_t poly_off[NB_MAX + 2];
    uint8_t pad_[8];
};
constexpr int HOT_PREFIX = sizeof(DHdr) + NB_MAX * 12 + E_MAX * 12;
static_assert(HOT_PREFIX % 16 == 0, "prefix is a TMA bulk copy");
static_assert(sizeof(DHdr) == 72 || sizeof(DHdr) == 80 || sizeof(DHdr) == 64, "header size");
static_assert(offsetof(DHdr, item_env) == 72 && sizeof(DHdr) == 80, "item_env sits in the header's former padding");
static_assert(sizeof(DEnvHot) % 16 == 0, "TMA bulk copies move multiples of 16 bytes");

// "Cold" record: touched only by the paths that need it (leaf-index actions, setting-3 densities, the
// stability load edges, the rare >8-support scratch).  Lives in HBM / L2, never staged.
struct alignas(16) DEnvCold {
    int16_t leaf[NL_MAX][6];  // leaves emitted with the last observation (xs,ys,zs,xe,ye,ze)
    double density[NB_MAX];   // per placed box (setting 3)
    Stack4 e_st[EDGE_MAX + 1];
    double poly[POLY_MAX][2];
    uint32_t cand[CAND_MAX];  // ordered candidate keys written by K2, read by K3 (<= 1228 distinct candidates)
    uint32_t raw[2048];       // insertion sequence produced by the EV / EP / CP / FC generators
    uint32_t tab_big[TAB_A];  // 2048-slot stage of the set emulation when it does not live in shared memory
    BigScratch big;
    // feasibility of the candidates of the CURRENT observation, one bit per candidate in candidate order: written per 32-candidate chunk by
    // the classification at the end of K2 (bounds / resting height / floor), completed by the pooled stability walks (atomicOr), read by the emit kernel
    uint32_t fbits[FBITS_WORDS];
    int32_t n_fw;             // chunks classified (classification stops once `leaf_node_holder` candidates are known feasible)
    int32_t lock;             // serialises the rare > KSUP_SMALL-support visits of this env on `big` (walk lanes of one env sit in different warps)
    int32_t n_pending;        // stability walks of this env still running (set by the classification, decremented by the walk kernels, polled by the emit kernel)
    int32_t pad_;
};

// One stability walk (calculated_impact_virtual of one candidate placement) of the step's global pool: produced by the classification at
// the end of K2 for every candidate that is in bounds, fits under the lid and rests on boxes (not on the floor), consumed by pct_walk_kernel.
struct WalkItem {
    uint32_t env;             // launch-local env index
    uint32_t pack;            // the first four supports of the placement (8 bits each, scan order)
    uint16_t c;               // candidate index (bit position in DEnvCold::fbits)
    uint8_t xs, ys, mh, sx, sy, sz, k, pad_;  // footprint corner, resting height, oriented dims, number of supports
};
static_assert(sizeof(WalkItem) == 20, "queue entry");
// A walk that the light-prefix kernel could not finish: it stands in front of placed box / the placement itself (`node`, NODE_NEW = 255) with
// the stack `st`; pct_walk_kernel continues it (stab_virtual's continuation entry).
struct WalkCont {
    uint32_t item;            // index of its WalkItem in the pool
    uint32_t node;
    Stack4 st;
};
static_assert(sizeof(WalkCont) == 40, "queue entry");
// A piece of a walk in the fork-join form (stab_piece, pct_stability.cuh): "enter `node` with the stack (a, b, c) = (cx, cy, mass)" (kind 0) or "the load
// (a, b, c) = (x, y, mass) arrives on `node` in place of the stored edge `skip`: combine, then enter" (kind 1)
struct WalkPiece {
    uint32_t item;           // index of the WalkItem (the candidate placement this piece belongs to)
    uint8_t node, skip, kind, pad_;
    double a, b, c;
};
static_assert(sizeof(WalkPiece) == 32, "queue entry");
constexpr int WALK_FAILED = 1 << 30;
constexpr int WALK_PIECES_PER_ENV = 1024;  // capacity of the fork-join piece queue = n_envs x this (32 B entries; mean use ~5 per env); overflow -> PCT_FLAG_CAND_OVERFLOW
constexpr int WALK_CONT_PER_ENV = 256;  // capacity of the continuation pool = n_envs x this (mean use: 3 per env); overflow -> PCT_FLAG_CAND_OVERFLOW

struct DParams {
    DEnvHot *hot;
    DEnvCold *cold;
    int n_envs;
    int W, L, H, nb, nl, setting;
    double low_bound;
    int item_mode;
    const double *item_set;
    int n_items;
    const double *stream;
    int stream_len;
    int traj_len;  // > 0: resets jump to the next multiple of traj_len in the stream
    uint64_t seed;
    int64_t env_id_base;
    int64_t env_id_base0;  // env_id_base of env 0 of the handle (debug timers index by handle-local env)
    const void *actions;
    int action_f64;
    const int32_t *leaf_idx;
    void *obs;
    int obs_f64;
    float *reward;
    uint8_t *done;
    pct_step_info *info;
    int lnes;  // leaf-node expansion scheme: 0 EMS, 1 EV, 2 EP, 3 CP, 4 FC
    int shuffle;  // pct_config::shuffle: keyed permutation of the ordered candidate list (shuffle_candidates)
    int mode;  // 0 = reset all, 1 = step
    int keep_draw;      // mode 0: continue the item source instead of rewinding it (env.reset() after an episode)
    int no_auto_reset;  // mode 1: leave a finished env untouched (gym.Env semantics)
    // One pointer slot, two exclusive users (keeps sizeof(DParams), and with it the code of the default kernels, unchanged):
    //   dbg      phase timers (only in -DPCT_PHASE_TIMERS builds)
    //   aux      per-env state of the opt-in variants (production builds; nullptr unless `opt` is non-zero), see DEnvAux
    union {
        long long *dbg;
        struct DEnvAux *aux;
    };
    int32_t *order;  // heaviest-first scheduling order of the apply / candidates kernels: parity, bucket counts, per-bucket env lists (pct_discrete.cu, order_lookup); nullptr = env order
    int32_t *ready;  // [2 * n_envs] per-env hand-over flags (apply -> candidates, candidates -> feas_emit); nullptr = kernels run back to back
    int32_t epoch;   // value published in `ready` by this launch
    WalkItem *walkq;    // [n_envs * CAND_MAX] the step's pool of stability walks (worst-case capacity; only the used prefix is touched)
    int32_t *walk_ctr;  // its fill counter; reset by the emit kernel (sequential walks) / the last warp of the fork-join kernel
    WalkCont *contq;    // [n_envs * WALK_CONT_PER_ENV] walks the light-prefix kernel hands to the continuation kernel
    int32_t *cont_ctr;  // [2]: continuations pooled from the front (ordinary) / from the end (tall walks) of contq
    int32_t walk_lanes, walk_lanes_tall; // continuations per warp of pct_walk_kernel (1..32): ordinary / tall (resting height >= 0.6 H) walks
    // fork-join walks (pct_walk_fork_kernel, opt-in with PCT_B200_WALK=fork; the default is the sequential continuation kernel): contq holds WalkPiece entries,
    // cont_ctr = the queue's counters (pct_walkq.cuh); piece_ready[slot] = 1 once the slot's piece is written (cleared by its consumer);
    // walk_pend[item] = pieces of the walk still running (+ WALK_FAILED once one of them failed)
    int32_t walk_fork;
    int32_t walk_blocks;   // blocks per SM of the fork-join kernel (1..8)
    int32_t walk_keep;     // its warps that stay as helpers for forked pieces until the step's walks are done (the others leave when the fork queue is empty)
    int32_t piece_cap;     // entries of contq / piece_ready in this launch (WALK_PIECES_PER_ENV per env)
    int32_t *piece_ready;
    int32_t *walk_pend;
    int32_t opt;     // opt-in variants served by `aux`: PCT_OPT_DELTA (K3 delta observation writes), PCT_OPT_ALIAS (K1 object semantics of the loads)
};
constexpr int PCT_OPT_DELTA = 1, PCT_OPT_ALIAS = 2, PCT_OPT_K3_BLOCK = 4, PCT_OPT_NO_EMIT_PDL = 8;  // K3_BLOCK: round 1's block-per-env feasibility kernel (A/B)

// heuristic baselines (pct_heuristics.cuh)
struct HParams {
    int code;                // enum pct_heuristic; PCT_H_QUERY_ = single placement query
    float *rows;             // (n_envs, 9) action rows
    int32_t *hstate;         // (n_envs, 4) LSAH footprint of the packed items: maxX, maxY, minX, minY (heuristic.py:146-147)
    uint64_t seed;           // RANDOM
    int64_t t;
    int q_env, q[5];         // query: handle-local env, oriented dims, lx, ly
    double q_den;
    int32_t *q_out;          // [feasible, rest height, W*L height map after the placement]
};
// continuous domain (pct_heuristics_continuous.cuh): LSAH / OnlineBPH / BR, float64 rows and footprint state
struct HParamsC {
    int code;
    double *rows;            // (n_envs, 9) float64 action rows
    double *hstate;          // (n_envs, 4) LSAH footprint: maxX, maxY, minX, minY
    int q_env;               // PCT_H_QUERY_: handle-local env, oriented sizes + position, density, result [feasible, rest height]
    double q[5], q_den;
    double *q_out;
};
constexpr int PCT_H_QUERY_ = 7;
constexpr int HEUR_SIDE_MAX = 32;  // height-map based codes (HM, MACS, RANDOM's bitmap, queries): W, L <= 32
cudaError_t launch_heuristic_discrete(const DParams &p, const HParams &hp, cudaStream_t st);

// delta observation writes: aux[i].obs_prev = {nb, nl} for n envs ("every row of the buffer may be non-zero")
void launch_fill_prev(DEnvAux *aux, int n_envs, int nb, int nl, cudaStream_t st);

int discrete_kernels_per_step(const DParams &p);
cudaError_t launch_discrete(const DParams &p, cudaStream_t st, cudaEvent_t *prof = nullptr);
cudaError_t launch_policy_random_discrete(const DEnvHot *hot, int n_envs, int64_t env_id_base, uint64_t seed, int64_t t, int32_t *leaf_idx,
                                          cudaStream_t st, const int64_t *t_dev = nullptr);

// ---- saved env records (pct_save_envs / pct_load_envs) -------------------------------------------------------
// A record is a fixed-size, 16-byte-aligned slot: this header, then the domain's layout (DRec in pct_discrete.cu, CRec in pct_continuous.cu).
constexpr uint32_t REC_MAGIC = 0x52544350u;  // "PCTR"
constexpr uint32_t REC_VERSION = 1;
constexpr int REC_BAD_RECORD = 1, REC_ROW_OUTSIDE = 2, REC_BAD_ENV = 3;  // pct_load_envs status codes (0 = loaded)
struct alignas(16) RecHdr {
    uint32_t magic, version, domain, valid;  // valid = 0: written for an env id outside the saving handle
    uint64_t fingerprint;  // configuration fingerprint of the saving handle (pct_api.cu, config_fingerprint)
    uint64_t row_hash;     // item-stream mode: content hash of the stream row the env draws from (its item_env); 0 otherwise
    uint64_t pad_[4];
};
static_assert(sizeof(RecHdr) == 64, "record header");
struct RecArgs {
    const int32_t *ids;       // [n] env ids (nullptr: record i <-> env i)
    int n;
    unsigned char *rec;       // n records of rec_bytes each (read-only for a load)
    int64_t rec_bytes;
    uint64_t fingerprint;
    const uint64_t *row_hash; // item-stream mode: content hash of every stream row of this handle [n_envs]; nullptr otherwise
    int alias;                // DEnvAux::box_st / e_upper / e_alias are live (ALIAS apply kernels)
    void *hstate;             // LSAH footprint, 4 words per env (int32 discrete, double continuous)
    int32_t *status;          // load: [n] per-record codes, may be nullptr
};
int64_t discrete_record_bytes();
// save (load == 0) or load (load == 1) of the records in `s`; p: state_params of the handle + obs / obs_f64 / aux
cudaError_t launch_records_discrete(const DParams &p, const RecArgs &s, int load, cudaStream_t st);

}  // namespace pct
