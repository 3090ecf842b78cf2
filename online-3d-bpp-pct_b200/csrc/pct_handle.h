// Internal: the object behind pct_handle.
#pragma once
#include <string>
#include <vector>
#include "pct_kernels.h"

struct pct_env_batch {
    pct_config cfg;
    int n_envs = 0, device = 0;
    int obs_len = 0;
    bool did_reset = false;
    int64_t launches = 0;
    std::string err;
    // device state
    pct::DEnvHot *d_hot = nullptr;
    pct::DEnvCold *d_cold = nullptr;
    void *c_state = nullptr;  // continuous-domain state (pct_continuous.cu)
    void *c_walkq = nullptr;  // continuous-domain pool of stability walks (WalkItemC, pct_continuous.cu)
    double *d_item_set = nullptr;
    int n_items = 0;
    double *d_stream = nullptr;
    int stream_len = 0;
    uint64_t item_set_hash = 0;   // content hash of the item set (part of the record fingerprint, pct_api.cu config_fingerprint)
    uint64_t *d_row_hash = nullptr;  // [n_envs] content hash of every item-stream row: a loaded record must find the row it draws from unchanged
    int traj_len = 0;
    int32_t *d_ready = nullptr;   // [2 * n_envs] per-env hand-over flags of the overlapped launch mode
    int32_t epoch = 0;
    bool overlap = true;          // PCT_B200_OVERLAP=0: plain back-to-back kernels
    bool overlap_cont = false;    // continuous domain: measured slower overlapped (5.35 M -> 3.97 M env-steps/s), off unless PCT_B200_OVERLAP_CONT=1
    // delta observation writes (default ON since round 2: +3 % device path, and with zero-copy 5.2 -> 9.1 M env-steps/s through pct_step_host;
    // PCT_B200_OBS_DELTA=0 disables): the feasibility kernel writes only the rows that can differ from what the SAME caller buffer already holds
    // (DEnvAux::obs_prev = per env the internal / leaf rows of the tracked buffer that may be non-zero).  Contract (include/pct_b200.h): a caller
    // that hands the same observation pointer to consecutive calls must not have modified the buffer in between.
    bool obs_delta = true;
    // object semantics of the load entries in the real placement = what the reference's Python objects do (DESIGN.md section 3 (b)):
    // pct_apply_kernel<STAB, ALIAS = true> / pctc_apply_kernel<true, true>.  Default ON since round 2 (green on hardware, oracle default flipped with it);
    // PCT_B200_ALIAS=0 selects the snapshot semantics of round 1 (kept for the sensitivity tests).
    bool alias_mode = true;
    bool no_emit_pdl = false;     // PCT_B200_EMIT_PDL=0: launch the emit kernel in plain stream order (A/B measurement of the emit / walk-tail overlap)
    bool k3_block = false;        // PCT_B200_K3=block: round 1's block-per-env feasibility kernel instead of the warp-per-env one (A/B measurements)
    pct::DEnvAux *d_aux = nullptr;  // per-env state of the opt-in variants (allocated when one of them is on)
    const void *tracked_obs = nullptr;
    bool fill_pending = false;
    bool host_zero_copy = true;   // pct_step_host: kernels write the observation straight into the pinned (mapped) host buffer; PCT_B200_HOST_ZEROCOPY=0: staged copies
    bool cont_pre = true;         // continuous feas_emit: resting heights from pre-rounded rectangles (exact, +2 %; PCT_B200_CONT_PRE=0 disables)
    int32_t *d_hstate = nullptr;  // (n_envs, 4) LSAH footprint state (pct_heuristic_actions); allocated at pct_create (per-env state: saved records carry it)
    double *d_hstate_c = nullptr; // same for the continuous domain (pct_heuristic_actions_f64)
    double *d_query_c = nullptr;  // 2 doubles: result of pct_query_placement_f64
    int32_t *d_query = nullptr;   // 2 + W*L ints: result of pct_query_placement
    int item_mode = 0;
    // staging for the host-buffer entry points
    void *d_obs = nullptr, *d_act = nullptr;
    int32_t *d_idx = nullptr;
    float *d_rew = nullptr;
    uint8_t *d_done = nullptr;
    pct_step_info *d_info = nullptr;
    cudaStream_t own_stream = nullptr;
    void *dbg = nullptr;
    int32_t *d_order = nullptr;   // heaviest-first scheduling order: parity, bucket counts, per-bucket env lists (pct_discrete.cu order_lookup)
    pct::WalkItem *d_walkq = nullptr;  // [n_envs * CAND_MAX] pool of stability walks of the current step (pct_walk_kernel)
    int32_t *d_walk_ctr = nullptr;     // [n_envs] fill counters (index = first env of the launched range)
    pct::WalkCont *d_contq = nullptr;  // [n_envs * WALK_CONT_PER_ENV] continuations: light-prefix kernel -> pct_walk_kernel
    int32_t *d_cont_ctr = nullptr;
    size_t contq_env_bytes = 0;        // bytes of d_contq per env (WalkCont pool / WalkPiece queue)
    int32_t *d_piece_ready = nullptr, *d_walk_pend = nullptr;  // fork-join walks: per-slot publication flags, per-walk piece counters
    bool walk_fork = false;            // PCT_B200_WALK=fork: fork-join continuation kernel (pct_walkq.cuh) instead of the sequential one — measured equal-to-slower (DESIGN.md 5d), kept as an opt-in
    int walk_blocks = 6;               // its blocks per SM (PCT_B200_WALK_BLOCKS)
    int walk_keep = 296;               // its warps that stay as helpers for forked pieces (PCT_B200_WALK_KEEP)
    int walk_lanes_tall = 4;           // ... of the tall walks (resting height >= 0.6 H: the longest chains), PCT_B200_WALK_LANES_TALL
    int walk_lanes = 16;               // continuations per warp of pct_walk_kernel (PCT_B200_WALK_LANES; few long serial chains: more warps beat fuller warps)
    bool lpt = false;
    int prof_on = 0;
    std::vector<cudaEvent_t> prof_ev;   // 4 events per recorded step
    int prof_steps = 0;
    int host_groups = 4;          // env ranges pipelined by pct_step_host (kernels of one range overlap the D2H of another)
    int groups = 1;               // env ranges stepped concurrently on internal streams
    cudaStream_t sub[8] = {};
    cudaEvent_t ev_fork = nullptr, ev_join[8] = {};
};

