// Continuous PCT environment (pct_envs/PctContinuous0 in the reference, "C:" below): batched reset / step for sm_100a.
//
// Same three-kernel pipeline as the discrete domain (apply / candidates / feasibility+emit) and the same stability
// routine (pct_stability.cuh) instantiated with a float64 geometry policy that carries the reference's 1e-6
// tolerances and 6-decimal roundings.  This first version keeps the per-env record in HBM (no TMA staging): it is the
// correctness path for BASELINE config 4; the discrete kernels are the tuned ones.
//
// Reference behaviour restated:
//   PackingContinuous.step / reset / cur_observation / get_possible_position / LeafNode2Action   C:bin3D.py:69-207
//   Space.interSect2D / drop_box / drop_box_virtual / check_box                                   C:space.py:305-439
//   Space.interSectEMS3D / GENEMS / Difference / EliminateInscribedEMS / EMSPoint                 C:space.py:441-568
// Parity contract (see oracle/pct_oracle_continuous.c): float64 leaf rows as actions; float32 rows are widened.
#include "pct_common.cuh"
#include "pct_stability.cuh"
#include "pct_kernels.h"
#include "pct_handle.h"
#include "pct_geom_continuous.cuh"
#include "pct_walkq.cuh"
#include "pct_records.cuh"

namespace pct {

constexpr int CE_MAX = 256;     // EMS capacity (reference preallocates 1000, C:space.py:276)
constexpr int CE_TMP = 512;     // intermediate list inside GENEMS
constexpr int CC_TAB = 2048;    // set-emulation table (<= 1228 distinct candidates)

struct CHdr {
    int32_t n_box, n_ems, n_leaf, flags;
    int64_t draw_pos;
    double ep_reward;
    double next_box[3];
    double next_den;
    double vol_sum;
    int32_t ep_len, n_cand, n_edge, n_poly;
    int64_t item_env;   // global env id whose item sequence this env follows (its own id unless a saved record was loaded into it)
};
struct alignas(16) CEnv {
    CHdr h;
    double box[NB_MAX][6];      // lx,ly,lz,x,y,z
    double den[NB_MAX];
    double ems[CE_MAX][6];
    double ems_tmp[CE_TMP][6];
    uint16_t e_off[NB_MAX + 2], poly_off[NB_MAX + 2];
    uint8_t e_lower[EDGE_MAX + 1], e_next[EDGE_MAX + 1], first_in[NB_MAX], last_in[NB_MAX];
    uint8_t pad_topo_[8];         // keeps e_st / poly / leaf 16-byte aligned (saved records copy them in 16-byte units)
    Stack4 e_st[EDGE_MAX + 1];
    double poly[POLY_MAX][2];
    double leaf[NL_MAX][6];
    uint16_t cand[1232];
    BigScratch big;
    uint32_t fbits[FBITS_WORDS];  // feasibility bits of the current observation's candidates (classification at the end of K2, pooled walks, emit kernel)
    int32_t n_fw, lock, n_pending, pad_;  // n_pending: stability walks still running (classification sets, walk kernels decrement, emit kernel polls)
};

// one pooled stability walk of the continuous domain (cf. WalkItem): the candidate's tuple is rebuilt from `code` (cand_tuple)
struct WalkItemC {
    uint32_t env, pack;
    uint16_t c, code;
    int32_t k;
    double mh;
};
static_assert(sizeof(WalkItemC) == 24, "queue entry");

struct CParams {
    CEnv *env;
    int n_envs;
    double W, L, H, low_bound;
    int nb, nl, setting;
    int item_mode, sample_dist;
    double sample_a, sample_b;
    const double *item_set;
    int n_items;
    const double *stream;
    int stream_len, traj_len;
    uint64_t seed;
    int64_t env_id_base;
    const void *actions;
    int action_f64;
    const int32_t *leaf_idx;
    void *obs;
    int obs_f64;
    float *reward;
    uint8_t *done;
    pct_step_info *info;
    int mode, keep_draw, no_auto_reset;
    int32_t *ready;  // overlapped launch mode: per-env hand-over flags [2 * n_envs] (see pct_common.cuh), nullptr = off
    int32_t epoch;
    int shuffle;     // pct_config::shuffle: keyed permutation of the ordered candidate list (shuffle_candidates)
    WalkItemC *walkq;   // pooled stability walks (round 2, see pct_discrete.cu "K3 (round 2)"); nullptr: round 1's block kernel does everything
    int32_t *walk_ctr;
    WalkCont *contq;
    int32_t *cont_ctr;
    int32_t walk_lanes, walk_lanes_tall;
    int32_t walk_fork, walk_blocks, walk_keep, piece_cap;   // fork-join continuation kernel (see DParams)
    int32_t *piece_ready, *walk_pend;
    int32_t delta;   // delta observation rows (DEnvAux::obs_prev), emit kernel only
    DEnvAux *aux;    // per-env state of the ALIAS apply kernel (EdgePoolA arrays), nullptr with PCT_B200_ALIAS=0 / setting 2
};

// around6, NodeC / GeomC (geometry policy of the stability routine), rest_height_c, rest_height_pre: pct_geom_continuous.cuh

__device__ __forceinline__ bool rot_dims_c(const double nb[3], int rot, double &sx, double &sy, double &sz) {  // C:space.py:537-559
    switch (rot) {
    case 0: sx = nb[0]; sy = nb[1]; sz = nb[2]; return true;
    case 1: sx = nb[1]; sy = nb[0]; sz = nb[2]; return !(fabs(sx - sy) < 1e-6);
    case 2: sx = nb[0]; sy = nb[2]; sz = nb[1]; return !(fabs(sx - sy) < 1e-6 && fabs(sy - sz) < 1e-6);
    case 3: sx = nb[1]; sy = nb[2]; sz = nb[0]; return !(fabs(sx - sy) < 1e-6 && fabs(sy - sz) < 1e-6);
    case 4: sx = nb[2]; sy = nb[0]; sz = nb[1]; return !(fabs(sx - sy) < 1e-6);
    default: sx = nb[2]; sy = nb[1]; sz = nb[0]; return !(fabs(sx - sy) < 1e-6);
    }
}
// candidate code = ems_idx << 5 | rot << 2 | corner  ->  the 6-tuple the reference adds to its set (C:space.py:563-566)
__device__ __forceinline__ void cand_tuple(uint16_t code, const double (*ems)[6], const double nb[3], double t[6]) {
    const double *m = ems[code >> 5];
    double sx, sy, sz;
    rot_dims_c(nb, (code >> 2) & 7, sx, sy, sz);
    const int q = code & 3;
    if (q & 1) { t[0] = m[3] - sx; t[3] = m[3]; } else { t[0] = m[0]; t[3] = m[0] + sx; }
    if (q & 2) { t[1] = m[4] - sy; t[4] = m[4]; } else { t[1] = m[1]; t[4] = m[1] + sy; }
    t[2] = m[2]; t[5] = m[2] + sz;
}
__device__ __noinline__ uint64_t hash_double_call(double v) { return hash_double(v); }  // one copy of the routine for the three call sites of the candidates kernel
__device__ __noinline__ uint64_t cand_hash_c(const double t[6]) {
    uint64_t l[6];
#pragma unroll 1
    for (int i = 0; i < 6; i++) l[i] = hash_double(t[i]);
    return tuple_hash6(l);
}

__device__ __noinline__ void draw_item_c(const CParams &p, int e, CHdr &h) {
    const uint64_t gid = (uint64_t)h.item_env, d = (uint64_t)h.draw_pos;  // item_env: the env's own global id unless a saved record was loaded
    if (p.item_mode == 0 && p.sample_dist) {  // C:bin3D.py:103-112
        auto u01 = [&](uint64_t salt) { return (double)(rnd_u64(p.seed ^ salt, gid, d) >> 11) * (1.0 / 9007199254740992.0); };
        auto r3 = [&](double v) { return ddiv(rint(v * 1000.0), 1000.0); };
        h.next_box[0] = r3(p.sample_a + (p.sample_b - p.sample_a) * u01(0x11));
        h.next_box[1] = r3(p.sample_a + (p.sample_b - p.sample_a) * u01(0x22));
        if (p.setting == 2) h.next_box[2] = r3(p.sample_a + (p.sample_b - p.sample_a) * u01(0x33));
        else {
            const double ch[5] = {0.1, 0.2, 0.3, 0.4, 0.5};
            h.next_box[2] = ch[rnd_u64(p.seed ^ 0x44, gid, d) % 5];
        }
        h.next_den = p.setting == 3 ? rnd_density(p.seed, gid, d) : 1.0;
    } else {
        const double *it = p.item_mode == 0 ? p.item_set + (rnd_u64(p.seed, gid, d) % (uint64_t)p.n_items) * 3
                                            : p.stream + ((size_t)(h.item_env - p.env_id_base) * p.stream_len + (size_t)(d % (uint64_t)p.stream_len)) * 4;
        h.next_box[0] = it[0]; h.next_box[1] = it[1]; h.next_box[2] = it[2];
        h.next_den = p.setting == 3 ? (p.item_mode == 0 ? rnd_density(p.seed, gid, d) : it[3]) : 1.0;
    }
    h.draw_pos++;
}

__device__ __noinline__ void reset_space_c(CEnv *ev, const CParams &p, int e, int lane) {
    if (lane == 0) {
        CHdr &h = ev->h;
        h.n_box = 0; h.n_ems = 1; h.n_leaf = 0; h.flags = 0; h.n_edge = 0; h.n_poly = 0; h.vol_sum = 0; h.ep_len = 0; h.ep_reward = 0;
        ev->ems[0][0] = 0; ev->ems[0][1] = 0; ev->ems[0][2] = 0; ev->ems[0][3] = p.W; ev->ems[0][4] = p.L; ev->ems[0][5] = p.H;
        if (p.traj_len > 0 && h.draw_pos % p.traj_len) h.draw_pos += p.traj_len - h.draw_pos % p.traj_len;
        draw_item_c(p, e, h);
    }
    __syncwarp();
}

// GENEMS (C:space.py:441-528): same ballot / scan compaction as the discrete kernel, float64 with rounded intersections
constexpr int CE_STAGE = 128;  // intermediate EMS entries staged in shared memory for the inscribed-EMS purge (6 KB per warp)
__device__ __noinline__ int genems_warp_c(CEnv *ev, const int n0, const double loc[6], double lb, int lane, int &flags, double (*stage)[6]) {
    double (*ems)[6] = ev->ems, (*tmp)[6] = ev->ems_tmp;
    const int nch = (n0 + 31) >> 5;
    const double itn[6] = {-loc[0], -loc[1], -loc[2], loc[3], loc[4], loc[5]};
    int off = 0;
#pragma unroll 1
    for (int pass = 0; pass < 2; pass++) {
#pragma unroll 1
        for (int c = 0; c < nch; c++) {
            const int i = c * 32 + lane;
            bool inter = false;
            double it[6], m[6];
            if (i < n0) {
#pragma unroll
                for (int t = 0; t < 6; t++) m[t] = ems[i][t];
#pragma unroll
                for (int t = 0; t < 6; t++) it[t] = around6(fmin(itn[t], t < 3 ? -m[t] : m[t]));
                inter = (it[0] + it[3] > 0) && (it[1] + it[4] > 0) && (it[2] + it[5] > 0);
            }
            if (pass == 0) {  // survivors keep their order
                const bool keep = i < n0 && !inter;
                const uint32_t bm = __ballot_sync(FULL, keep);
                if (keep) {
                    const int p = off + __popc(bm & ((1u << lane) - 1));
#pragma unroll
                    for (int t = 0; t < 6; t++) tmp[p][t] = m[t];
                }
                off += __popc(bm);
            } else {  // children: left, right, front, back, top (Difference, :490-502)
                uint32_t cm = 0;
                const double x3 = -it[0], y3 = -it[1], x4 = it[3], y4 = it[4], z4 = it[5];
                if (inter) {
                    const bool ux = m[3] - m[0] + 1e-6 >= lb, uy = m[4] - m[1] + 1e-6 >= lb, uz = m[5] - m[2] + 1e-6 >= lb;
                    if (x3 - m[0] + 1e-6 >= lb && uy && uz) cm |= 1;
                    if (m[3] - x4 + 1e-6 >= lb && uy && uz) cm |= 2;
                    if (ux && y3 - m[1] + 1e-6 >= lb && uz) cm |= 4;
                    if (ux && m[4] - y4 + 1e-6 >= lb && uz) cm |= 8;
                    if (ux && uy && m[5] - z4 + 1e-6 >= lb) cm |= 16;
                }
                const int cnt = __popc(cm);
                const int incl = warp_incl_scan(cnt, lane);
                int p = off + incl - cnt;
#pragma unroll 1
                for (int ch = 0; ch < 5 && cm; ch++) {
                    if (!(cm & (1u << ch))) continue;
                    double q[6] = {m[0], m[1], m[2], m[3], m[4], m[5]};
                    if (ch == 0) q[3] = x3; else if (ch == 1) q[0] = x4; else if (ch == 2) q[4] = y3; else if (ch == 3) q[1] = y4; else q[2] = z4;
                    if (p < CE_TMP) {
#pragma unroll
                        for (int t = 0; t < 6; t++) tmp[p][t] = q[t];
                    } else flags |= PCT_FLAG_EMS_OVERFLOW;
                    p++;
                }
                off += __shfl_sync(FULL, incl, 31);
            }
        }
    }
    flags = __reduce_or_sync(FULL, flags);
    const int n = off < CE_TMP ? off : CE_TMP;
    __syncwarp();
    // EliminateInscribedEMS (C:space.py:505-528): the O(n^2) containment test read every candidate container b from the env record in global memory
    // (ncu r2, profiles/r2_cont_head.txt: 30 % of this kernel's stall samples on that line); the intermediate list is staged in shared memory first
    // (lists longer than CE_STAGE entries — not seen on the BASELINE streams — keep reading the record).
    const bool staged = n <= CE_STAGE;
    // Every EMS coordinate is a 6-decimal value (the container's corners or an np.around(.., 6) result), so v -> rint(v * 1e6) is an order-preserving
    // bijection onto integers; for bins up to 1.048575 they fit 20 bits and the six comparisons of a containment test become two 64-bit subtractions on
    // packed fields with guard bits (the discrete kernel's trick; ncu r2: this loop was 21 % of the kernel's instructions).  Any coordinate that is not
    // exactly such a value (checked per entry) sends the whole list through the float64 comparisons.
    constexpr uint64_t GUARD = (1ull << 20) | (1ull << 41) | (1ull << 62);
    uint64_t *pk = (uint64_t *)&stage[0][0];
    bool packed = staged;
    if (packed) {
        bool good = true;
#pragma unroll 1
        for (int i = lane; i < n; i += 32) {
            uint64_t w2[2] = {0, 0};
#pragma unroll
            for (int t = 0; t < 6; t++) {
                const double v = tmp[i][t], k = rint(v * 1e6);
                good = good && k >= 0.0 && k < 1048576.0 && around6(v) == v;
                w2[t / 3] |= (uint64_t)(long long)k << (21 * (t % 3));
            }
            pk[2 * i] = w2[0]; pk[2 * i + 1] = w2[1];
        }
        packed = __all_sync(FULL, good);
        __syncwarp();
    }
    if (staged && !packed)
        for (int t = lane; t < n * 6; t += 32) (&stage[0][0])[t] = (&tmp[0][0])[t];
    __syncwarp();
    const double (*src)[6] = (staged && !packed) ? stage : tmp;
    int w = 0;
    const int nch2 = (n + 31) >> 5;
#pragma unroll 1
    for (int c = 0; c < nch2; c++) {
        const int i = c * 32 + lane;
        bool keep = false;
        double a[6];
        if (i < n) {
#pragma unroll
            for (int t = 0; t < 6; t++) a[t] = src[i][t];
            int hit = 0;
            if (packed) {
                const uint64_t alo = pk[2 * i] | GUARD, ahi = pk[2 * i + 1];
#pragma unroll 4
                for (int j = 0; j < n; j++) {
                    const ulonglong2 b = *(const ulonglong2 *)(pk + 2 * j);
                    hit |= (int)(j != i && (((alo - b.x) & ((b.y | GUARD) - ahi) & GUARD) == GUARD));
                }
            } else {
#pragma unroll 2
                for (int j = 0; j < n; j++) {
                    const double *b = src[j];
                    hit |= (int)(j != i && a[0] >= b[0] && a[1] >= b[1] && a[2] >= b[2] && a[3] <= b[3] && a[4] <= b[4] && a[5] <= b[5]);
                }
            }
            keep = !hit;
        }
        const uint32_t bm = __ballot_sync(FULL, keep);
        if (keep) {
            const int p = w + __popc(bm & ((1u << lane) - 1));
            if (p < CE_MAX) {
#pragma unroll
                for (int t = 0; t < 6; t++) ems[p][t] = a[t];
            }
        }
        w += __popc(bm);
    }
    if (w > CE_MAX) { flags |= PCT_FLAG_EMS_OVERFLOW; w = CE_MAX; }
    __syncwarp();
    return w;
}

// ================= K1: apply =================
// ALIAS variant (the default; PCT_B200_ALIAS=0 selects the snapshot kernels): the reference's object semantics of the load entries (EdgePoolA,
// DESIGN.md section 3 (b)); per-env state through CParams::aux.

template <bool STAB, bool ALIAS = false>
__global__ void __launch_bounds__(64) pctc_apply_kernel(const CParams p) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int e = blockIdx.x * 2 + warp;
    if (e >= p.n_envs) return;
    __shared__ int lock_s[2];
    __shared__ __align__(16) double ems_stage[2][CE_STAGE][6];
    int *lock = &lock_s[warp];
    static_assert(sizeof(StabScratch) <= sizeof(double) * CE_STAGE * 6, "the descent's scratch fits the EMS stage");
    StabScratch *scr = (StabScratch *)&ems_stage[warp][0][0];  // the descent's working arrays: aliased onto the EMS stage, which only GENEMS (after the descent) uses
    CEnv *ev = p.env + e;
    CHdr &h = ev->h;
    if (p.ready) pdl_launch_dependents();
    if (lane == 0) *lock = 0;
    float reward = 0.f;
    int done = 0;
    pct_step_info info{};
    if (p.mode == 0) {
        const int64_t dp = p.keep_draw ? h.draw_pos : 0;
        const int64_t ie = p.keep_draw ? h.item_env : p.env_id_base + e;
        __syncwarp();
        if (lane == 0) { h.draw_pos = dp; h.item_env = ie; }
        reset_space_c(ev, p, e, lane);
    } else {
        const double nb0 = h.next_box[0], nb1 = h.next_box[1], nb2 = h.next_box[2], den0 = h.next_den;
        const int n_box0 = h.n_box, n_leaf0 = h.n_leaf, flags0 = h.flags, n_ems0 = h.n_ems;
        __syncwarp();
        // ---- LeafNode2Action (C:bin3D.py:151-167) ----
        double lx = 0, ly = 0, x = nb0, y = nb1, z = nb2;
        {
            double a[6] = {0, 0, 0, 0, 0, 0}, s = 0;
            bool zero = true;
            if (p.leaf_idx) {
                const int k = p.leaf_idx[e];
                if (k >= 0 && k < n_leaf0) {
                    zero = false;
                    for (int t = 0; t < 6; t++) a[t] = ev->leaf[k][t];
                }
            } else {
                for (int t = 0; t < 6; t++) {
                    a[t] = p.action_f64 ? ((const double *)p.actions)[(size_t)e * 9 + t] : (double)((const float *)p.actions)[(size_t)e * 9 + t];
                    s += a[t];
                }
                zero = (s == 0);
            }
            if (!zero) {
                x = around6(a[3] - a[0]);
                y = around6(a[4] - a[1]);
                const double nb[3] = {nb0, nb1, nb2};
                int rec[3] = {0, 1, 2}, n = 3;
                for (int i = 0; i < n; i++)
                    if (fabs(x - nb[rec[i]]) < 1e-6) { for (int u = i; u < n - 1; u++) rec[u] = rec[u + 1]; n--; break; }
                for (int i = 0; i < n; i++)
                    if (fabs(y - nb[rec[i]]) < 1e-6) { for (int u = i; u < n - 1; u++) rec[u] = rec[u + 1]; n--; break; }
                z = nb[rec[0]];
                lx = a[0]; ly = a[1];
            }
        }
        lx = around6(lx); ly = around6(ly);  // C:bin3D.py:173
        // ---- Space.drop_box (C:space.py:329-376) ----
        bool ok = !(lx + x - 1e-6 > p.W || ly + y - 1e-6 > p.L) && !(lx + 1e-6 < 0 || ly + 1e-6 < 0);
        double max_h = 0;
        if (lane == 0) { ev->e_off[n_box0] = (uint16_t)h.n_edge; ev->poly_off[n_box0] = (uint16_t)h.n_poly; ev->first_in[n_box0 < NB_MAX ? n_box0 : 0] = EDGE_NIL; }
        __syncwarp();
        if (ok) {
            double mh = rest_height_c(ev->box, lane, n_box0, 32, lx, ly, lx + x, ly + y);
#pragma unroll
            for (int d = 16; d; d >>= 1) mh = fmax(mh, __shfl_xor_sync(FULL, mh, d));
            max_h = mh < 0 ? 0.0 : mh;
            if (max_h + z - 1e-6 > p.H) ok = false;
            else if (STAB && !(fabs(max_h) < 1e-6)) {
                int res = 0;
                if (lane == 0) {
                    int fl = 0;
                    GeomC g{ev->box, ev->den, n_box0};
                    NodeC root{lx, ly, max_h, x, y, z, x * y * z * den0};
                    if constexpr (ALIAS) {
                        EdgePoolA pool;
                        static_cast<EdgePool &>(pool) = EdgePool{ev->e_lower, ev->e_next, ev->e_off, ev->first_in, ev->last_in, ev->e_st, ev->e_st, h.n_edge,
                                                                 ev->poly_off, &ev->poly[0][0], &ev->poly[0][0], h.n_poly};
                        DEnvAux *ax = p.aux + e;
                        pool.box_st = ax->box_st; pool.e_upper = ax->e_upper; pool.e_alias = ax->e_alias;
                        res = stability_check<true, GeomC, true>(g, root, pool, &ev->big, lock, n_box0, fl, nullptr, scr);
                        if (!res) alias_sync_loads(pool);
                        h.n_edge = pool.n; h.n_poly = pool.n_poly;
                    } else {
                    EdgePool pool{ev->e_lower, ev->e_next, ev->e_off, ev->first_in, ev->last_in, ev->e_st, ev->e_st, h.n_edge,
                                  ev->poly_off, &ev->poly[0][0], &ev->poly[0][0], h.n_poly};
                    res = stability_check<true, GeomC>(g, root, pool, &ev->big, lock, n_box0, fl, nullptr, scr);
                    h.n_edge = pool.n; h.n_poly = pool.n_poly;
                    }
                    h.flags |= fl;
                }
                __syncwarp();
                ok = __shfl_sync(FULL, res, 0) != 0;
            }
            if (ok && n_box0 >= p.nb) { ok = false; if (lane == 0) h.flags |= PCT_FLAG_BOX_OVERFLOW; }
        }
        __syncwarp();
        const double binvol = p.W * p.L * p.H;
        if (ok) {
            if (lane == 0) {
                double *b = ev->box[n_box0];
                b[0] = lx; b[1] = ly; b[2] = max_h; b[3] = x; b[4] = y; b[5] = z;
                ev->den[n_box0] = den0;
                h.n_box = n_box0 + 1;
                h.vol_sum += x * y * z;
                ev->e_off[n_box0 + 1] = (uint16_t)h.n_edge; ev->poly_off[n_box0 + 1] = (uint16_t)h.n_poly;
            }
            __syncwarp();
            int fl = 0;
            const double loc[6] = {lx, ly, max_h, around6(lx + x), around6(ly + y), around6(max_h + z)};  // C:bin3D.py:191-194
            const int n_ems = genems_warp_c(ev, n_ems0, loc, p.low_bound, lane, fl, ems_stage[warp]);
            const double rw = (nb0 * nb1 * nb2) / binvol * 10;
            reward = (float)rw;
            info.counter = n_box0 + 1;
            info.flags = flags0 | fl;
            if (lane == 0) {
                h.n_ems = n_ems; h.flags |= fl; h.ep_len++; h.ep_reward += rw;
                draw_item_c(p, e, h);
            }
            __syncwarp();
        } else {
            done = 1;
            info.counter = n_box0;
            info.flags = h.flags;
            info.ratio = (float)(h.vol_sum / binvol);
            info.ep_reward = (float)h.ep_reward;
            info.ep_len = h.ep_len + 1;
            __syncwarp();
            if (!p.no_auto_reset) reset_space_c(ev, p, e, lane);
        }
    }
    __syncwarp();
    if (lane == 0) {
        if (p.reward) p.reward[e] = reward;
        if (p.done) p.done[e] = (uint8_t)done;
        if (p.info) p.info[e] = info;
        if (p.ready) env_publish(p.ready + e, p.epoch);
    }
}

// ================= K2: candidates in CPython-set order (C:space.py:531-568) =================
// Table slots are 32 bits: candidate code | 16-bit tag (the top bits of the tuple hash — CPython compares the stored hash before the keys, setobject.c).
// A probe rejects a non-matching slot on the tag alone; the exact 6-double comparison (tuples rebuilt from the two codes) runs only on a tag match,
// i.e. practically only for true duplicates.  Round 1 rebuilt and compared the tuple of EVERY probed slot and broadcast the six doubles of every
// inserted key through shuffles (ncu r2, profiles/r2_cont_head.txt: 25 % of this kernel in _Py_HashDouble's frexp loop — now an integer rotation,
// pct_pyhash.cuh —, 15 % in shuffles).
__device__ __forceinline__ bool cand_equal(uint16_t a, uint16_t b, const double (*ems)[6], const double nb[3]) {
    double u[6], v[6];
    cand_tuple(a, ems, nb, u);
    cand_tuple(b, ems, nb, v);
    return u[0] == v[0] && u[1] == v[1] && u[2] == v[2] && u[3] == v[3] && u[4] == v[4] && u[5] == v[5];
}

__global__ void __launch_bounds__(32) pctc_candidates_kernel(const CParams p) {
    __shared__ uint32_t tabA[CC_TAB], tabB[512];
    __shared__ uint64_t stg_h[32], rs_h[32];  // staged (hash, code) of the chunk's new keys / of the slots being re-inserted by a resize
    __shared__ uint32_t rs_c[32];
    __shared__ uint16_t stg_c[32];
    const int lane = threadIdx.x, e = blockIdx.x;
    CEnv *ev = p.env + e;
    int fl = 0;
    if (p.ready) {  // overlapped mode: wait for the apply kernel's hand-over of THIS env
        pdl_launch_dependents();
        if (lane == 0 && !env_wait(p.ready + e, p.epoch)) fl = PCT_FLAG_SYNC_TIMEOUT;
        fl = __shfl_sync(FULL, fl, 0);
    }
    const CHdr &h = ev->h;
    const double nb[3] = {h.next_box[0], h.next_box[1], h.next_box[2]};
    const int R = p.setting == 2 ? 6 : 2, n_ems = h.n_ems;
    constexpr uint32_t EMPTY = 0xFFFFFFFFu;
    uint32_t *tab = tabA;
    uint32_t mask = 7;
    int fill = 0;
    if (lane < 8) tab[lane] = EMPTY;
    __syncwarp();
    const int raw = n_ems * R * 4;
    bool stop = false;
#pragma unroll 1
    for (int base = 0; base < raw && !stop; base += 32) {
        const int r = base + lane;
        bool valid = false;
        uint64_t hash = 0;
        uint16_t code = 0;
        // The four corners of one (EMS, orientation) are four adjacent lanes and their 6-tuples draw on ten distinct coordinates (x: m0, m0 + sx, m3 - sx,
        // m3; y alike; z: m2, m2 + sz): every lane hashes two or three of them (_Py_HashDouble, the expensive part) and the group exchanges the results,
        // instead of six hashes per lane (ncu r2: 17 % of this kernel's instructions).  Same expressions as cand_tuple, so the same bits.
        uint64_t h0 = 0, h1 = 0, h2 = 0;
        const int q = r & 3;
        if (r < raw) {
            const int er = r >> 2, rot = er % R, ei = er / R;
            double sx, sy, sz;
            if (rot_dims_c(nb, rot, sx, sy, sz)) {
                const double *m = ev->ems[ei];
                if (m[3] - m[0] + 1e-6 >= sx && m[4] - m[1] + 1e-6 >= sy && m[5] - m[2] + 1e-6 >= sz) {
                    valid = true;
                    code = (uint16_t)((ei << 5) | (rot << 2) | q);
                    double v0, v1, v2 = 0;
                    if (q == 0) { v0 = m[0]; v1 = m[0] + sx; v2 = m[2]; }
                    else if (q == 1) { v0 = m[3] - sx; v1 = m[3]; v2 = m[2] + sz; }
                    else if (q == 2) { v0 = m[1]; v1 = m[1] + sy; }
                    else { v0 = m[4] - sy; v1 = m[4]; }
                    h0 = hash_double_call(v0);
                    h1 = hash_double_call(v1);
                    if (q < 2) h2 = hash_double_call(v2);
                }
            }
        }
        {
            const int gb = lane & ~3, lx = gb + (q & 1), ly = gb + 2 + (q >> 1);
            uint64_t l6[6];
            l6[0] = __shfl_sync(FULL, h0, lx); l6[3] = __shfl_sync(FULL, h1, lx);
            l6[1] = __shfl_sync(FULL, h0, ly); l6[4] = __shfl_sync(FULL, h1, ly);
            l6[2] = __shfl_sync(FULL, h2, gb); l6[5] = __shfl_sync(FULL, h2, gb + 1);
            if (valid) hash = tuple_hash6(l6);
        }
        // already present? (read-only probe; present keys sit on their own probe sequence)
        if (valid) {
            const uint32_t tag = (uint32_t)(hash >> 48);
            uint64_t perturb = hash;
            uint32_t i = (uint32_t)hash & mask;
            bool open = true;
            while (open) {
                const int probes = (i + 9 <= mask) ? 9 : 0;
                for (int j = 0; j <= probes; j++) {
                    const uint32_t s = tab[i + j];
                    if (s == EMPTY) { open = false; break; }
                    if ((s >> 16) == tag && cand_equal((uint16_t)s, code, ev->ems, nb)) { open = false; valid = false; break; }
                }
                perturb >>= 5;
                i = (uint32_t)((uint64_t)i * 5 + 1 + perturb) & mask;
            }
        }
        // the new keys of this chunk go through the order-defining insertion in lane (= reference) order: staged in shared memory and inserted by
        // lane 0 with a scalar set_add_entry (3x fewer warp instructions than a warp-uniform probe with shuffles, as in the discrete kernel);
        // an equal tuple staged by an earlier lane of the same chunk is found by the tag + exact comparison like any other present key
        const uint32_t vm = __ballot_sync(FULL, valid);
        const int n_new = __popc(vm);
        if (valid) {
            const int pos = __popc(vm & ((1u << lane) - 1));
            stg_h[pos] = hash;
            stg_c[pos] = code;
        }
        __syncwarp();
        int done = 0;
#pragma unroll 1
        while (done < n_new && !stop) {
            int upto = n_new;
            if (lane == 0) {
#pragma unroll 1
                for (int t = done; t < n_new; t++) {
                    const uint64_t hk = stg_h[t];
                    const uint16_t ck = stg_c[t];
                    const uint32_t tagk = (uint32_t)(hk >> 48);
                    uint64_t perturb = hk;
                    uint32_t i = (uint32_t)hk & mask;
                    int state = 0;
#pragma unroll 1
                    while (!state) {
                        const int probes = (i + 9 <= mask) ? 9 : 0;
#pragma unroll 1
                        for (int j = 0; j <= probes; j++) {
                            const uint32_t sl = tab[i + j];
                            if (sl == EMPTY) { tab[i + j] = (tagk << 16) | ck; state = 1; break; }
                            if ((sl >> 16) == tagk && cand_equal((uint16_t)sl, ck, ev->ems, nb)) { state = 2; break; }
                        }
                        perturb >>= 5;
                        i = (uint32_t)((uint64_t)i * 5 + 1 + perturb) & mask;
                    }
                    if (state == 1 && (uint32_t)(++fill) * 5 >= mask * 3) { upto = t + 1; break; }
                }
            }
            upto = __shfl_sync(FULL, upto, 0);
            fill = __shfl_sync(FULL, fill, 0);
            done = upto;
            __syncwarp();
            if ((uint32_t)fill * 5 >= mask * 3) {
                uint32_t newsize = 8;
                while (newsize <= (uint32_t)fill * 4) newsize <<= 1;
                if (newsize > CC_TAB) { fl |= PCT_FLAG_CAND_OVERFLOW; stop = true; break; }
                uint32_t *nt = (tab == tabA) ? tabB : tabA;
                for (uint32_t t = lane; t < newsize; t += 32) nt[t] = EMPTY;
                __syncwarp();
#pragma unroll 1
                for (uint32_t b2 = 0; b2 <= mask; b2 += 32) {  // set_table_resize: re-insert in slot order (set_insert_clean: no comparisons)
                    const uint32_t sidx = b2 + lane;
                    const uint32_t c2 = sidx <= mask ? tab[sidx] : EMPTY;
                    const uint32_t em = __ballot_sync(FULL, c2 != EMPTY);
                    if (c2 != EMPTY) {
                        double u[6];
                        cand_tuple((uint16_t)c2, ev->ems, nb, u);
                        const int pos = __popc(em & ((1u << lane) - 1));
                        rs_h[pos] = cand_hash_c(u);
                        rs_c[pos] = c2;
                    }
                    __syncwarp();
                    if (lane == 0) {
                        const int m2 = __popc(em);
#pragma unroll 1
                        for (int t = 0; t < m2; t++) {
                            uint64_t pt = rs_h[t];
                            uint32_t ii = (uint32_t)pt & (newsize - 1);
                            bool placed = false;
#pragma unroll 1
                            while (!placed) {
                                const int pr = (ii + 9 <= newsize - 1) ? 9 : 0;
                                for (int j = 0; j <= pr; j++)
                                    if (nt[ii + j] == EMPTY) { nt[ii + j] = rs_c[t]; placed = true; break; }
                                pt >>= 5;
                                ii = (uint32_t)((uint64_t)ii * 5 + 1 + pt) & (newsize - 1);
                            }
                        }
                    }
                    __syncwarp();
                }
                tab = nt;
                mask = newsize - 1;
            }
        }
        __syncwarp();
    }
    __syncwarp();
    int cnt = 0;
#pragma unroll 1
    for (uint32_t b2 = 0; b2 <= mask; b2 += 32) {
        const uint32_t s = b2 + lane;
        const uint32_t c2 = s <= mask ? tab[s] : EMPTY;
        const uint32_t em = __ballot_sync(FULL, c2 != EMPTY);
        if (c2 != EMPTY) ev->cand[cnt + __popc(em & ((1u << lane) - 1))] = (uint16_t)c2;
        cnt += __popc(em);
    }
    __syncwarp();
    if (p.shuffle) {  // scratch: the GENEMS temp list (24 KB, idle between apply kernels): keys at 0, permuted codes at 10 KB
        static_assert(sizeof(ev->ems_tmp) >= 10240 + sizeof(ev->cand), "shuffle scratch fits");
        shuffle_candidates<uint16_t>(ev->cand, cnt, (uint64_t *)ev->ems_tmp, (uint16_t *)((char *)ev->ems_tmp + 10240), p.seed, (uint64_t)h.item_env,
                                     (uint64_t)h.draw_pos, lane);
    }
    if (p.walkq) {
        // ---- classify (round 2): drop_box_virtual's bounds / resting height (C:space.py:380-398) on pre-rounded box rectangles, supports + exact
        // quick reject for the placements that rest on boxes; the stability walks of all envs go to one pool (pctc_walk_light / pctc_walk kernels) ----
        __shared__ double rb[NB_MAX][5];
        const int n_box = h.n_box, nl = p.nl;
        const bool stab = p.setting != 2;
        for (int t = lane; t < n_box; t += 32) {
            const double *b = ev->box[t];
            rb[t][0] = around6(-b[0]); rb[t][1] = around6(-b[1]); rb[t][2] = around6(b[0] + b[3]); rb[t][3] = around6(b[1] + b[4]);
            rb[t][4] = b[2] + b[5];
        }
        __syncwarp();
        const uint32_t lt = (1u << lane) - 1;
        const double margin = 2e-6 * (1.0 + fmax(p.W, p.L));  // the support polygon lies inside the contact rectangles' bounding box up to the 1e-6 * y perturbation
        int pos = 0, nf = 0, n_walk = 0;
#pragma unroll 1
        while (pos < cnt && nf < nl) {
            const int c = pos + lane;
            bool feas = false, pend = false;
            int k = 0;
            uint32_t pack = 0;
            uint16_t code = 0;
            double mh = 0;
            if (c < cnt) {
                code = ev->cand[c];
                double t6[6];
                cand_tuple(code, ev->ems, nb, t6);
                const double x = t6[3] - t6[0], y = t6[4] - t6[1], z = t6[5] - t6[2], lx = t6[0], ly = t6[1];
                bool chk = !(lx + x - 1e-6 > p.W || ly + y - 1e-6 > p.L) && !(lx + 1e-6 < 0 || ly + 1e-6 < 0);
                const double c0 = around6(-lx), c1 = around6(-ly), c2 = around6(lx + x), c3 = around6(ly + y);
                mh = rest_height_pre(rb, n_box, c0, c1, c2, c3);
                if (mh < 0) mh = 0.0;
                if (mh + z - 1e-6 > p.H) chk = false;
                if (!chk) feas = false;
                else if (!stab || fabs(mh) < 1e-6) feas = true;
                else {
                    // supports = GeomC::support(root, t): top within 1e-6 of the resting height and a positive rounded intersection (C:space.py:350-359)
                    double X1 = 0, Y1 = 0, X2 = 0, Y2 = 0;
#pragma unroll 1
                    for (int t = 0; t < n_box; t++) {
                        const double *b = rb[t];
                        if (!(fabs(b[4] - mh) < 1e-6)) continue;
                        const double i0 = fmin(c0, b[0]), i1 = fmin(c1, b[1]), i2 = fmin(c2, b[2]), i3 = fmin(c3, b[3]);
                        if (!((i0 + i2 > 0) && (i1 + i3 > 0))) continue;
                        if (k == 0) { X1 = -i0; Y1 = -i1; X2 = i2; Y2 = i3; }
                        else { X1 = fmin(X1, -i0); Y1 = fmin(Y1, -i1); X2 = fmax(X2, i2); Y2 = fmax(Y2, i3); }
                        if (k < 4) pack |= (uint32_t)t << (8 * k);
                        k++;
                    }
                    const double cx = lx + x * 0.5, cy = ly + y * 0.5;
                    const bool far_out = k > 0 && (cx < X1 - margin || cx > X2 + margin || cy < Y1 - margin || cy > Y2 + margin);
                    pend = !far_out;  // centre outside the supports' bounding box: the root test fails (cf. rest_height_supports, pct_geom.cuh)
                }
            }
            const uint32_t fm = __ballot_sync(FULL, feas), pm = __ballot_sync(FULL, pend);
            if (lane == 0) ev->fbits[pos >> 5] = fm;
            nf += __popc(fm);
            n_walk += __popc(pm);
            if (pm) {
                int qb = 0;
                if (lane == 0) qb = atomicAdd(p.walk_ctr, __popc(pm));
                qb = __shfl_sync(FULL, qb, 0);
                if (pend) p.walkq[qb + __popc(pm & lt)] = WalkItemC{(uint32_t)e, pack, (uint16_t)c, code, k, mh};
            }
            pos += 32;
        }
        if (lane == 0) { ev->n_fw = pos >> 5; ev->n_pending = n_walk; }
    }
    if (lane == 0) {
        ev->h.n_cand = cnt;
        if (fl) ev->h.flags |= fl;
        if (p.ready) env_publish(p.ready + p.n_envs + e, p.epoch);
    }
}

// ---- pooled walks (round 2): see pct_discrete.cu — light prefix for every walk, continuation kernel for the walks that reach a node with >= 2 supports ----
struct WalkViewC {
    GeomC g;
    EdgePool pool;
    NodeC root;
    CEnv *ev;
};
__device__ __forceinline__ WalkViewC walk_view_c(const CParams &p, const WalkItemC &it, bool has) {
    CEnv *ev = p.env + it.env;
    const CHdr &h = ev->h;
    double t6[6] = {0, 0, 0, 0, 0, 0};
    if (has) {
        const double nb[3] = {h.next_box[0], h.next_box[1], h.next_box[2]};
        cand_tuple(it.code, ev->ems, nb, t6);
    }
    const double x = t6[3] - t6[0], y = t6[4] - t6[1], z = t6[5] - t6[2];
    return WalkViewC{GeomC{ev->box, ev->den, has ? h.n_box : 0},
                     EdgePool{ev->e_lower, ev->e_next, ev->e_off, ev->first_in, ev->last_in, ev->e_st, ev->e_st, has ? h.n_edge : 0, ev->poly_off,
                              &ev->poly[0][0], &ev->poly[0][0], has ? h.n_poly : 0},
                     NodeC{t6[0], t6[1], it.mh, x, y, z, x * y * z * (has ? h.next_den : 1.0)}, ev};
}

__global__ void __launch_bounds__(128, 4) pctc_walk_light_kernel(const CParams p) {
    const int lane = threadIdx.x & 31;
    const int total = *(volatile const int32_t *)p.walk_ctr;
    const int nwarps = gridDim.x * 4;
    const int cap = p.n_envs * WALK_CONT_PER_ENV;
#pragma unroll 1
    for (int base = (blockIdx.x * 4 + (threadIdx.x >> 5)) * 32; base < total; base += nwarps * 32) {
        const int i = base + lane;
        const bool has = i < total;
        WalkItemC it{};
        if (has) it = p.walkq[i];
        const WalkViewC v = walk_view_c(p, it, has);
        int node = NODE_NEW, res = 0;
        Stack4 st{};
        if (has) res = stab_light<GeomC>(v.g, v.root, it.k, it.pack, v.pool, node, st);
        if (res == 1) atomicOr(&v.ev->fbits[it.c >> 5], 1u << (it.c & 31));
        if (has && res != 2) { __threadfence(); atomicSub(&v.ev->n_pending, 1); }
        if (p.walk_fork) {  // fork-join continuation kernel: one queue of pieces (pct_walkq.cuh)
            const uint32_t pm = __ballot_sync(FULL, res == 2);
            if (pm) {
                const PieceQueue pq{(WalkPiece *)p.contq, p.piece_ready, p.cont_ctr, p.piece_cap};
                int qb = 0;
                if (lane == 0) qb = pq_reserve_initial(pq, __popc(pm));
                qb = __shfl_sync(FULL, qb, 0);
                if (res == 2) {
                    const int idx = qb + __popc(pm & ((1u << lane) - 1));
                    if (idx < pq.cap) {
                        p.walk_pend[i] = 1;
                        pq.q[idx] = WalkPiece{(uint32_t)i, (uint8_t)node, (uint8_t)EDGE_NIL, 0, 0, st.cx, st.cy, st.m};
                    } else {
                        atomicOr(&v.ev->h.flags, PCT_FLAG_CAND_OVERFLOW);
                        __threadfence();
                        atomicSub(&v.ev->n_pending, 1);
                        pq_piece_done(pq);
                    }
                }
            }
            continue;
        }
        const bool tall = it.mh >= 0.6 * p.H;  // the longest chains: pooled from the end, fewer lanes per warp (see pct_discrete.cu)
        const uint32_t ps = __ballot_sync(FULL, res == 2 && !tall), pt = __ballot_sync(FULL, res == 2 && tall);
        if (ps | pt) {
            int qs = 0, qt = 0;
            if (lane == 0) {
                if (ps) qs = atomicAdd(p.cont_ctr, __popc(ps));
                if (pt) qt = atomicAdd(p.cont_ctr + 1, __popc(pt));
            }
            qs = __shfl_sync(FULL, qs, 0);
            qt = __shfl_sync(FULL, qt, 0);
            if (res == 2) {
                const uint32_t lt = (1u << lane) - 1;
                const int idx = tall ? qt + __popc(pt & lt) : qs + __popc(ps & lt);
                if (idx < cap / 2) p.contq[tall ? cap - 1 - idx : idx] = WalkCont{(uint32_t)i, (uint32_t)node, st};
                else { atomicOr(&v.ev->h.flags, PCT_FLAG_CAND_OVERFLOW); __threadfence(); atomicSub(&v.ev->n_pending, 1); }
            }
        }
    }
}

__global__ void __launch_bounds__(64, 8) pctc_walk_kernel(const CParams p) {
    const int lane = threadIdx.x & 31;
    const int cap = p.n_envs * WALK_CONT_PER_ENV;
    const int n_short = min(*(volatile const int32_t *)p.cont_ctr, cap / 2), n_tall = min(*(volatile const int32_t *)(p.cont_ctr + 1), cap / 2);
    __syncthreads();
    pdl_launch_dependents();  // the emit kernel may follow: its blocks wait for their env's last walk (CEnv::n_pending)
    const int nwarps = gridDim.x * 2, Ls = p.walk_lanes, Lt = p.walk_lanes_tall;
    const int w_tall = (n_tall + Lt - 1) / Lt, w_all = w_tall + (n_short + Ls - 1) / Ls;
#pragma unroll 1
    for (int w = blockIdx.x * 2 + (threadIdx.x >> 5); w < w_all; w += nwarps) {
        const bool tw = w < w_tall;
        const int L = tw ? Lt : Ls;
        const unsigned mask = L >= 32 ? FULL : ((1u << L) - 1u);
        if (lane >= L) continue;
        const int i = tw ? w * Lt + lane : (w - w_tall) * Ls + lane;
        const bool has = i < (tw ? n_tall : n_short);
        WalkCont ct{};
        WalkItemC it{};
        if (has) { ct = p.contq[tw ? cap - 1 - i : i]; it = p.walkq[ct.item]; }
        const WalkViewC v = walk_view_c(p, it, has);
        int fl = 0;
        const bool ok = stab_virtual<GeomC>(v.g, v.root, it.k, it.pack, v.pool, &v.ev->big, &v.ev->lock, fl, has, mask, has ? (int)ct.node : NODE_NEW, &ct.st) != 0;
        if (has && ok) atomicOr(&v.ev->fbits[it.c >> 5], 1u << (it.c & 31));
        if (has && fl) atomicOr(&v.ev->h.flags, fl);
        if (has) { __threadfence(); atomicSub(&v.ev->n_pending, 1); }
    }
}

// fork-join form of the continuation kernel: see pct_walk_fork_kernel (pct_discrete.cu) and pct_walkq.cuh — same protocol, continuous geometry
struct PieceForkC {
    PieceQueue pq;
    int32_t *pend;
    uint32_t item;
    int n_init;
    bool overflow;
    __device__ __forceinline__ void operator()(int child, int skip, double vx, double vy, double vm) {
        if (!pq_fork(pq, n_init, pend, WalkPiece{item, (uint8_t)child, (uint8_t)skip, 1, 0, vx, vy, vm})) overflow = true;
    }
};
__device__ __forceinline__ void run_piece_c(const CParams &p, const PieceQueue &pq, int n_init, int slot) {
    const WalkPiece pc = pq.q[slot];
    if (slot >= n_init) pq.ready[slot] = 0;
    const WalkItemC it = p.walkq[pc.item];
    const WalkViewC v = walk_view_c(p, it, true);
    int32_t *pend = p.walk_pend + pc.item;
    int fl = 0, ok = 0;
    if (!(*(volatile const int32_t *)pend & WALK_FAILED)) {
        PieceForkC fork{pq, pend, pc.item, n_init, false};
        ok = stab_piece<GeomC>(v.g, v.root, it.k, it.pack, v.pool, &v.ev->big, &v.ev->lock, fl, (int)pc.node, (int)pc.kind, (int)pc.skip, pc.a, pc.b, pc.c, fork);
        if (fork.overflow) { fl |= PCT_FLAG_CAND_OVERFLOW; ok = 0; }
    }
    if (fl) atomicOr(&v.ev->h.flags, fl);
    if (!ok) atomicOr(pend, WALK_FAILED);
    __threadfence();
    const int r = atomicSub(pend, 1);
    if ((r & (WALK_FAILED - 1)) == 1) {
        if (!(r & WALK_FAILED)) atomicOr(&v.ev->fbits[it.c >> 5], 1u << (it.c & 31));
        __threadfence();
        atomicSub(&v.ev->n_pending, 1);
    }
    pq_piece_done(pq);
}
__global__ void __launch_bounds__(64, 8) pctc_walk_fork_kernel(const CParams p) {
    const int lane = threadIdx.x & 31;
    const int wid = blockIdx.x * 2 + (threadIdx.x >> 5), n_warps = gridDim.x * 2;
    const PieceQueue pq{(WalkPiece *)p.contq, p.piece_ready, p.cont_ctr, p.piece_cap};
    const int n_init = min(*(volatile const int32_t *)(pq.ctr + PQ_NINIT), pq.cap);
    const int L = p.walk_lanes;
    pdl_launch_dependents();
    if (n_init > 0) {
#pragma unroll 1
        for (int b = wid * L; b < n_init; b += n_warps * L) {
            if (lane < L && b + lane < n_init) run_piece_c(p, pq, n_init, b + lane);
            __syncwarp();
        }
        const bool keep = wid < p.walk_keep;
#pragma unroll 1
        for (;;) {
            int t0 = -1;
            if (lane == 0 && (keep || *(volatile const int32_t *)(pq.ctr + PQ_ALLOC) - *(volatile const int32_t *)(pq.ctr + PQ_HEAD) > 0))
                t0 = atomicAdd(pq.ctr + PQ_HEAD, L);
            t0 = __shfl_sync(FULL, t0, 0);
            if (t0 < 0) break;
            bool fin = false;
            if (lane < L) {
                const int slot = n_init + t0 + lane;
                if (pq_wait(pq, slot)) run_piece_c(p, pq, n_init, slot);
                else fin = true;
            }
            __syncwarp();
            if (__any_sync(FULL, fin)) break;
        }
    }
    if (lane == 0) pq_warp_exit(pq, n_warps, p.walk_ctr);
}

template <typename OT> __device__ __noinline__ void write_obs_c(const CParams &p, int e, const CEnv *ev, const double (*leaf)[6], int n_leaf, int tid, int nthreads);
template <typename OT> __device__ __noinline__ void write_obs_c_delta(const CParams &p, int e, const CEnv *ev, const double (*leaf)[6], int n_leaf, int tid, int nthreads);

// emit (round 2): the first `nl` set feasibility bits in candidate order -> leaf rows, observation; 64 threads per env
template <typename OT>
__global__ void __launch_bounds__(64) pctc_emit_kernel(const CParams p) {
    __shared__ double leaf[NL_MAX][6];
    __shared__ int s_nleaf;
    const int tid = threadIdx.x, lane = tid & 31, e = blockIdx.x;
    CEnv *ev = p.env + e;
    const CHdr &h = ev->h;
    const double nb[3] = {h.next_box[0], h.next_box[1], h.next_box[2]};
    if (e == 0 && tid == 0 && !p.walk_fork) { *p.walk_ctr = 0; p.cont_ctr[0] = 0; p.cont_ctr[1] = 0; }  // every walk-kernel block has read them (programmatic dependency): empty the pools for the next step
    if (tid == 0) {  // may run while this env's walks are still in flight (programmatic dependent of the continuation kernel)
        int spins = 0;
        while (*(volatile const int32_t *)&ev->n_pending > 0) {
            __nanosleep(spins < 16 ? 100 : 1000);
            if (++spins > (1 << 22)) { atomicOr(&ev->h.flags, PCT_FLAG_SYNC_TIMEOUT); break; }
        }
        __threadfence();
    }
    __syncthreads();
    if (tid < 32) {
        const int nl = p.nl, nw = ev->n_fw;
        const uint32_t lt = (1u << lane) - 1;
        int base = 0;
#pragma unroll 1
        for (int w = 0; w < nw && base < nl; w++) {
            const uint32_t bits = ev->fbits[w];
            if ((bits >> lane) & 1u) {
                const int kk = base + __popc(bits & lt);
                if (kk < nl) {
                    double t6[6];
                    cand_tuple(ev->cand[w * 32 + lane], ev->ems, nb, t6);
                    for (int t = 0; t < 6; t++) leaf[kk][t] = t6[t];
                }
            }
            base += __popc(bits);
        }
        if (lane == 0) s_nleaf = min(base, nl);
    }
    __syncthreads();
    const int n_leaf = s_nleaf;
    for (int t = tid; t < n_leaf * 6; t += 64) ((double *)ev->leaf)[t] = ((double *)leaf)[t];
    if (tid == 0) {
        ev->h.n_leaf = n_leaf;
        if (p.info) {
            p.info[e].n_leaf = n_leaf; p.info[e].n_cand = h.n_cand; p.info[e].n_ems = h.n_ems; p.info[e].flags |= h.flags;
        }
    }
    if (p.delta) write_obs_c_delta<OT>(p, e, ev, leaf, n_leaf, tid, 64);
    else write_obs_c<OT>(p, e, ev, leaf, n_leaf, tid, 64);
}


// ================= K3: feasibility per candidate + leaf compaction + observation =================
template <typename OT>
__device__ __noinline__ void write_obs_c(const CParams &p, int e, const CEnv *ev, const double (*leaf)[6], int n_leaf, int tid, int nthreads) {
    OT *obs = (OT *)p.obs + (size_t)e * (size_t)((p.nb + p.nl + 1) * 9);
    const int n_box = ev->h.n_box, total = (p.nb + p.nl + 1) * 9;
    double s0 = ev->h.next_box[0], s1 = ev->h.next_box[1], s2 = ev->h.next_box[2];
    if (s1 < s0) { double t = s0; s0 = s1; s1 = t; }
    if (s2 < s1) { double t = s1; s1 = s2; s2 = t; }
    if (s1 < s0) { double t = s0; s0 = s1; s1 = t; }
#pragma unroll 1
    for (int f = tid; f < total; f += nthreads) {
        const int row = f / 9, col = f - row * 9;
        double v = 0;
        if (row < p.nb) {
            if (row < n_box) {  // C:space.py:372-373  [lx,ly,lz,lx+x,ly+y,lz+z,0,0,1]
                const double *b = ev->box[row];
                if (col < 3) v = b[col];
                else if (col < 6) v = b[col - 3] + b[col];
                else if (col == 8) v = 1;
            } else if (row == 0 && col == 8) v = 1;
        } else if (row < p.nb + p.nl) {
            const int k = row - p.nb;
            if (k < n_leaf) {
                if (col < 5) v = leaf[k][col];
                else if (col == 5) v = p.H;
                else if (col == 8) v = 1;
            }
        } else {
            if (col == 0) v = ev->h.next_den;
            else if (col == 3) v = s0;
            else if (col == 4) v = s1;
            else if (col == 5) v = s2;
            else if (col == 8) v = 1;
        }
        obs[f] = (OT)v;
    }
}

// Delta variant of write_obs_c (cf. write_obs_delta, pct_discrete.cu): the caller hands back the same observation buffer, obs_prev[0] / [1] say how
// many internal / leaf rows of it may be non-zero; only the rows below max(now, prev) and the item row are written.  Same values as write_obs_c.
template <typename OT>
__device__ __noinline__ void write_obs_c_delta(const CParams &p, int e, const CEnv *ev, const double (*leaf)[6], int n_leaf, int tid, int nthreads) {
    OT *obs = (OT *)p.obs + (size_t)e * (size_t)((p.nb + p.nl + 1) * 9);
    int32_t *prev = p.aux[e].obs_prev;
    const int n_box = ev->h.n_box;
    const int pb = min(prev[0], p.nb), pl = min(prev[1], p.nl);
    __syncthreads();  // every thread of the block (= env) has read prev before thread 0 replaces it
    const int wb = max(max(n_box, pb), 1), wl = max(n_leaf, pl);
    double s0 = ev->h.next_box[0], s1 = ev->h.next_box[1], s2 = ev->h.next_box[2];
    if (s1 < s0) { double t = s0; s0 = s1; s1 = t; }
    if (s2 < s1) { double t = s1; s1 = s2; s2 = t; }
    if (s1 < s0) { double t = s0; s0 = s1; s1 = t; }
    const int total = (wb + wl + 1) * 9;
#pragma unroll 1
    for (int f = tid; f < total; f += nthreads) {
        const int r = f / 9, col = f - r * 9;
        double v = 0;
        int row;
        if (r < wb) {
            row = r;
            if (row < n_box) {
                const double *b = ev->box[row];
                if (col < 3) v = b[col];
                else if (col < 6) v = b[col - 3] + b[col];
                else if (col == 8) v = 1;
            } else if (row == 0 && col == 8) v = 1;
        } else if (r < wb + wl) {
            const int k = r - wb;
            row = p.nb + k;
            if (k < n_leaf) {
                if (col < 5) v = leaf[k][col];
                else if (col == 5) v = p.H;
                else if (col == 8) v = 1;
            }
        } else {
            row = p.nb + p.nl;
            if (col == 0) v = ev->h.next_den;
            else if (col == 3) v = s0;
            else if (col == 4) v = s1;
            else if (col == 5) v = s2;
            else if (col == 8) v = 1;
        }
        obs[row * 9 + col] = (OT)v;
    }
    if (tid == 0) { prev[0] = max(n_box, 1); prev[1] = n_leaf; }
}

template <bool PRE>
__device__ __forceinline__ double (*rb_store())[5] {  // the default instantiation owns no such array
    if constexpr (PRE) { __shared__ double rb_s[NB_MAX][5]; return rb_s; }
    else return nullptr;
}

// PRE: resting heights from pre-rounded box rectangles staged in shared memory (rest_height_pre; opt-in, PCT_B200_CONT_PRE=1)
template <typename OT, bool STAB, bool PRE>
__global__ void __launch_bounds__(64) pctc_feas_emit_kernel(const CParams p) {
    __shared__ double leaf[NL_MAX][6];
    double (*rb)[5] = rb_store<PRE>();
    __shared__ uint32_t wb[2];
    __shared__ int lock;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, e = blockIdx.x;
    CEnv *ev = p.env + e;
    const CHdr &h = ev->h;
    if (tid == 0) {
        lock = 0;
        if (p.ready && !env_wait(p.ready + p.n_envs + e, p.epoch)) atomicOr(&ev->h.flags, PCT_FLAG_SYNC_TIMEOUT);
    }
    __syncthreads();
    const double nb[3] = {h.next_box[0], h.next_box[1], h.next_box[2]};
    const int n_cand = h.n_cand, n_box = h.n_box;
    const double den = h.next_den;
    GeomC g{ev->box, ev->den, n_box};
    EdgePool pool{ev->e_lower, ev->e_next, ev->e_off, ev->first_in, ev->last_in, ev->e_st, ev->e_st, h.n_edge,
                  ev->poly_off, &ev->poly[0][0], &ev->poly[0][0], h.n_poly};
    int n_leaf = 0, fl = 0;
    if (PRE) {
        for (int t = tid; t < n_box; t += 64) {
            const double *b = ev->box[t];
            rb[t][0] = around6(-b[0]); rb[t][1] = around6(-b[1]); rb[t][2] = around6(b[0] + b[3]); rb[t][3] = around6(b[1] + b[4]);
            rb[t][4] = b[2] + b[5];
        }
        __syncthreads();
    }
#pragma unroll 1
    for (int base = 0; base < n_cand && n_leaf < p.nl; base += 64) {
        const int c = base + tid;
        bool feas = false;
        double t6[6] = {0, 0, 0, 0, 0, 0};
        if (c < n_cand) {
            cand_tuple(ev->cand[c], ev->ems, nb, t6);
            // get_possible_position: x = xe - xs ... (C:bin3D.py:134-137); drop_box_virtual (C:space.py:380-425)
            const double x = t6[3] - t6[0], y = t6[4] - t6[1], z = t6[5] - t6[2], lx = t6[0], ly = t6[1];
            bool chk = !(lx + x - 1e-6 > p.W || ly + y - 1e-6 > p.L) && !(lx + 1e-6 < 0 || ly + 1e-6 < 0);
            double mh = PRE ? rest_height_pre(rb, n_box, around6(-lx), around6(-ly), around6(lx + x), around6(ly + y))
                            : rest_height_c(ev->box, 0, n_box, 1, lx, ly, lx + x, ly + y);
            if (mh < 0) mh = 0.0;
            if (mh + z - 1e-6 > p.H) chk = false;
            if (!chk) feas = false;
            else if (!STAB || fabs(mh) < 1e-6) feas = true;
            else {
                NodeC root{lx, ly, mh, x, y, z, x * y * z * den};
                feas = stability_check<false, GeomC>(g, root, pool, &ev->big, &lock, 0, fl) != 0;
            }
        }
        const uint32_t fm = __ballot_sync(FULL, feas);
        if (lane == 0) wb[warp] = fm;
        __syncthreads();
        const int before = warp == 1 ? __popc(wb[0]) : 0, total = __popc(wb[0]) + __popc(wb[1]);
        if (feas) {
            const int k = n_leaf + before + __popc(fm & ((1u << lane) - 1));
            if (k < p.nl)
                for (int t = 0; t < 6; t++) leaf[k][t] = t6[t];
        }
        n_leaf += total;
        __syncthreads();
    }
    if (n_leaf > p.nl) n_leaf = p.nl;
    fl = __reduce_or_sync(FULL, fl);
    if (fl && lane == 0) atomicOr(&ev->h.flags, fl);
    __syncthreads();
    for (int t = tid; t < n_leaf * 6; t += 64) ((double *)ev->leaf)[t] = ((double *)leaf)[t];
    if (tid == 0) {
        ev->h.n_leaf = n_leaf;
        if (p.info) {
            p.info[e].n_leaf = n_leaf; p.info[e].n_cand = n_cand; p.info[e].n_ems = h.n_ems; p.info[e].flags |= h.flags;
        }
    }
    write_obs_c<OT>(p, e, ev, leaf, n_leaf, tid, 64);
}

__global__ void pctc_policy_random_kernel(const CEnv *env, int n_envs, int64_t env_id_base, uint64_t seed, int64_t t, int32_t *leaf_idx) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_envs) return;
    const int n = env[e].h.n_leaf;
    leaf_idx[e] = n > 0 ? (int32_t)(rnd_u64(seed, (uint64_t)(env_id_base + e), (uint64_t)t) % (uint64_t)n) : 0;
}

// ================= saved env records (pct_save_envs / pct_load_envs) =================
// Live between calls (cf. the discrete list next to DRec, pct_discrete.cu): the header, box / den [0, n_box), ems [0, n_ems), the load-edge
// topology (e_off .. last_in, copied whole), e_st [0, n_edge), poly [0, n_poly), leaf [0, n_leaf), on ALIAS handles DEnvAux::box_st [0, n_box]
// / e_upper [0, n_edge) / e_alias, and the LSAH footprint (4 doubles).  Not saved: ems_tmp (GENEMS / shuffle scratch), cand, big, fbits / n_fw
// (per-step), lock / n_pending (zeroed on load).
struct alignas(16) CRec {
    RecHdr s;
    CHdr h;
    double box[NB_MAX][6];
    double den[NB_MAX];
    double ems[CE_MAX][6];
    unsigned char topo[offsetof(CEnv, e_st) - offsetof(CEnv, e_off)];
    Stack4 e_st[EDGE_MAX + 1];
    double poly[POLY_MAX][2];
    double leaf[NL_MAX][6];
    Stack4 box_st[NB_MAX + 1];
    uint8_t e_upper[EDGE_MAX + 1];
    uint32_t e_alias[(EDGE_MAX + 32) / 32];
    double hstate[4];
};
static_assert(sizeof(CHdr) % 16 == 0 && offsetof(CEnv, box) % 16 == 0 && offsetof(CEnv, den) % 16 == 0 && offsetof(CEnv, ems) % 16 == 0 &&
              offsetof(CEnv, e_off) % 16 == 0 && offsetof(CEnv, e_st) % 16 == 0 && offsetof(CEnv, poly) % 16 == 0 && offsetof(CEnv, leaf) % 16 == 0,
              "record parts are copied in 16-byte units");
static_assert(offsetof(CRec, h) % 16 == 0 && offsetof(CRec, box) % 16 == 0 && offsetof(CRec, den) % 16 == 0 && offsetof(CRec, ems) % 16 == 0 &&
              offsetof(CRec, topo) % 16 == 0 && offsetof(CRec, e_st) % 16 == 0 && offsetof(CRec, poly) % 16 == 0 && offsetof(CRec, leaf) % 16 == 0 &&
              offsetof(CRec, box_st) % 16 == 0 && offsetof(CRec, e_upper) % 16 == 0 && offsetof(CRec, hstate) % 16 == 0, "record layout");

// one warp per record; counts from the source's header, clamped to the capacities
template <bool LOAD, typename OT>
__global__ void __launch_bounds__(128, 4) pctc_env_record_kernel(const CParams p, const RecArgs s) {
    const int lane = threadIdx.x & 31, i = blockIdx.x * 4 + (threadIdx.x >> 5);
    if (i >= s.n) return;
    const int e = s.ids ? s.ids[i] : i;
    CRec *r = (CRec *)(s.rec + (size_t)i * (size_t)s.rec_bytes);
    if (e < 0 || e >= p.n_envs) {
        if (LOAD) { if (lane == 0 && s.status) s.status[i] = REC_BAD_ENV; }
        else if (lane == 0) { RecHdr z{}; z.magic = REC_MAGIC; z.version = REC_VERSION; r->s = z; }  // valid = 0
        return;
    }
    CEnv *ev = p.env + e;
    DEnvAux *aux = p.aux ? p.aux + e : nullptr;
    const CHdr &src = LOAD ? r->h : ev->h;
    if (LOAD) {
        int st = 0;
        if (lane == 0) st = rec_check(r->s, PCT_CONTINUOUS, src.item_env, s, p.env_id_base, p.n_envs);
        st = __shfl_sync(FULL, st, 0);
        if (lane == 0 && s.status) s.status[i] = st;
        if (st) return;  // a rejected record leaves its env untouched
    } else if (lane == 0) {
        RecHdr z{};
        z.magic = REC_MAGIC; z.version = REC_VERSION; z.domain = PCT_CONTINUOUS; z.valid = 1; z.fingerprint = s.fingerprint;
        const int64_t row = src.item_env - p.env_id_base;
        z.row_hash = (s.row_hash && row >= 0 && row < p.n_envs) ? s.row_hash[row] : 0;
        r->s = z;
    }
    const int n_box = min(max(src.n_box, 0), NB_MAX), n_ems = min(max(src.n_ems, 0), CE_MAX), n_leaf = min(max(src.n_leaf, 0), NL_MAX);
    const int n_edge = min(max(src.n_edge, 0), EDGE_MAX + 1), n_poly = min(max(src.n_poly, 0), POLY_MAX);
    __syncwarp();
    auto cp = [&](void *rec_part, void *env_part, int bytes) {
        if (LOAD) warp_copy16(env_part, rec_part, bytes, lane);
        else warp_copy16(rec_part, env_part, bytes, lane);
    };
    auto cp8 = [&](void *rec_part, void *env_part, int bytes) {
        if (LOAD) warp_copy8(env_part, rec_part, bytes, lane);
        else warp_copy8(rec_part, env_part, bytes, lane);
    };
    cp(&r->h, &ev->h, (int)sizeof(CHdr));
    cp(r->box, ev->box, n_box * 48);
    cp(r->den, ev->den, n_box * 8);
    cp(r->ems, ev->ems, n_ems * 48);
    cp(r->topo, ev->e_off, (int)sizeof(r->topo));
    cp(r->e_st, ev->e_st, n_edge * (int)sizeof(Stack4));
    cp(r->poly, ev->poly, n_poly * 16);
    cp(r->leaf, ev->leaf, n_leaf * 48);
    if (s.alias) {
        cp8(r->box_st, aux->box_st, min(n_box + 1, NB_MAX + 1) * (int)sizeof(Stack4));
        cp8(r->e_upper, aux->e_upper, n_edge);
        if (lane < (EDGE_MAX + 32) / 32) { if (LOAD) aux->e_alias[lane] = r->e_alias[lane]; else r->e_alias[lane] = aux->e_alias[lane]; }
    }
    if (lane < 2) {
        uint4 *hs = (uint4 *)((double *)s.hstate + (size_t)e * 4) + lane;
        if (LOAD) *hs = ((const uint4 *)r->hstate)[lane]; else ((uint4 *)r->hstate)[lane] = *hs;
    }
    if (LOAD) {
        if (lane == 0) { ev->lock = 0; ev->n_pending = 0; }
        if (aux && lane == 0) { aux->obs_prev[0] = p.nb; aux->obs_prev[1] = p.nl; }  // the next step rewrites every row of whichever buffer it gets
        if (p.obs) {
            __syncwarp();
            write_obs_c<OT>(p, e, ev, ev->leaf, n_leaf, lane, 32);
        }
    }
}

int64_t continuous_record_bytes() { return (int64_t)sizeof(CRec); }

// plain stream-ordered launches, see launch_records_discrete
int continuous_records(pct_env_batch *h, const RecArgs &s, int load, void *obs, cudaStream_t st) {
    if (s.n <= 0) return PCT_OK;
    CParams p{};
    p.env = (CEnv *)h->c_state; p.n_envs = h->n_envs;
    p.H = h->cfg.container_size[2]; p.nb = h->cfg.internal_node_holder; p.nl = h->cfg.leaf_node_holder;
    p.env_id_base = h->cfg.env_id_base; p.aux = h->d_aux; p.obs = obs;
    const int blocks = (s.n + 3) / 4;
    if (!load) pctc_env_record_kernel<false, float><<<blocks, 128, 0, st>>>(p, s);
    else if (h->cfg.obs_dtype == PCT_F64) pctc_env_record_kernel<true, double><<<blocks, 128, 0, st>>>(p, s);
    else pctc_env_record_kernel<true, float><<<blocks, 128, 0, st>>>(p, s);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { h->err = std::string("env records: ") + cudaGetErrorString(e); return PCT_ERR_CUDA; }
    return PCT_OK;
}

// ================= host side =================
int continuous_create(pct_env_batch *h) {
    cudaError_t e = cudaMalloc(&h->c_state, sizeof(CEnv) * (size_t)h->n_envs);
    if (e == cudaSuccess) e = cudaMemset(h->c_state, 0, sizeof(CEnv) * (size_t)h->n_envs);
    if (e == cudaSuccess) e = cudaMalloc(&h->d_ready, sizeof(int32_t) * 2 * (size_t)h->n_envs);
    if (e == cudaSuccess) e = cudaMemset(h->d_ready, 0, sizeof(int32_t) * 2 * (size_t)h->n_envs);
    if (e == cudaSuccess && !h->k3_block) {  // pools of the round-2 walk kernels (worst-case capacity for the walks; only the used prefix is touched)
        e = cudaMalloc(&h->c_walkq, sizeof(WalkItemC) * (size_t)CAND_MAX * (size_t)h->n_envs);
        if (e == cudaSuccess) e = cudaMalloc(&h->d_walk_ctr, sizeof(int32_t) * 16);  // [0] walk pool, [1..] continuation pool counters (sequential kernel: ordinary / tall; fork-join: pct_walkq.cuh)
        if (e == cudaSuccess) e = cudaMemset(h->d_walk_ctr, 0, sizeof(int32_t) * 16);
        if (e == cudaSuccess && h->walk_fork) e = cudaMalloc(&h->d_piece_ready, sizeof(int32_t) * (size_t)WALK_PIECES_PER_ENV * (size_t)h->n_envs);
        if (e == cudaSuccess && h->walk_fork) e = cudaMemset(h->d_piece_ready, 0, sizeof(int32_t) * (size_t)WALK_PIECES_PER_ENV * (size_t)h->n_envs);
        if (e == cudaSuccess && h->walk_fork) e = cudaMalloc(&h->d_walk_pend, sizeof(int32_t) * (size_t)CAND_MAX * (size_t)h->n_envs);
        h->contq_env_bytes = h->walk_fork ? sizeof(WalkPiece) * (size_t)WALK_PIECES_PER_ENV : sizeof(WalkCont) * (size_t)WALK_CONT_PER_ENV;
        if (e == cudaSuccess) e = cudaMalloc((void **)&h->d_contq, h->contq_env_bytes * (size_t)h->n_envs);
    }
    if (e == cudaSuccess) {  // item_env = the env's own global id (CHdr::item_env)
        std::vector<int64_t> id((size_t)h->n_envs);
        for (int i = 0; i < h->n_envs; i++) id[i] = h->cfg.env_id_base + i;
        e = cudaMemcpy2D((char *)h->c_state + offsetof(CEnv, h) + offsetof(CHdr, item_env), sizeof(CEnv), id.data(), sizeof(int64_t), sizeof(int64_t),
                         (size_t)h->n_envs, cudaMemcpyHostToDevice);
    }
    if (e != cudaSuccess) { h->err = std::string("continuous_create: ") + cudaGetErrorString(e); return PCT_ERR_CUDA; }
    return PCT_OK;
}
void continuous_destroy(pct_env_batch *h) { cudaFree(h->c_state); h->c_state = nullptr; cudaFree(h->c_walkq); h->c_walkq = nullptr; }
int64_t continuous_state_bytes() { return (int64_t)sizeof(CEnv); }

int continuous_launch(pct_env_batch *h, int mode, const void *actions, int action_f64, const int32_t *leaf_idx, void *obs, float *rew,
                      uint8_t *done, pct_step_info *info, cudaStream_t st) {
    CParams p{};
    p.env = (CEnv *)h->c_state; p.n_envs = h->n_envs;
    p.W = h->cfg.container_size[0]; p.L = h->cfg.container_size[1]; p.H = h->cfg.container_size[2];
    p.low_bound = h->cfg.size_minimum;
    p.nb = h->cfg.internal_node_holder; p.nl = h->cfg.leaf_node_holder; p.setting = h->cfg.setting;
    p.item_mode = h->item_mode; p.sample_dist = h->cfg.sample_from_distribution;
    p.sample_a = h->cfg.sample_left_bound; p.sample_b = h->cfg.sample_right_bound;
    p.item_set = h->d_item_set; p.n_items = h->n_items; p.stream = h->d_stream; p.stream_len = h->stream_len; p.traj_len = h->traj_len;
    p.seed = h->cfg.seed; p.env_id_base = h->cfg.env_id_base; p.shuffle = h->cfg.shuffle;
    p.actions = actions; p.action_f64 = action_f64; p.leaf_idx = leaf_idx;
    p.obs = obs; p.obs_f64 = h->cfg.obs_dtype == PCT_F64; p.reward = rew; p.done = done; p.info = info;
    p.mode = mode; p.keep_draw = h->did_reset ? 1 : 0; p.no_auto_reset = h->cfg.no_auto_reset;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(st, &cap);
    if (h->overlap_cont && h->d_ready && cap == cudaStreamCaptureStatusNone) { p.ready = h->d_ready; p.epoch = ++h->epoch; }
    const bool stab = p.setting != 2;
    const int b2 = (p.n_envs + 1) / 2;
    if (stab && h->alias_mode && h->d_aux) {
        p.aux = h->d_aux;
        pctc_apply_kernel<true, true><<<b2, 64, 0, st>>>(p);
    } else if (stab) pctc_apply_kernel<true><<<b2, 64, 0, st>>>(p);
    else pctc_apply_kernel<false><<<b2, 64, 0, st>>>(p);
    // candidates / feas_emit: with p.ready as programmatic dependent launches (their blocks become resident during the previous
    // kernel's tail and wait per env on the hand-over flags), else plain back-to-back launches
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg{};
    cfg.stream = st; cfg.attrs = at; cfg.numAttrs = p.ready ? 1 : 0;
    const bool pooled = h->c_walkq != nullptr && !h->k3_block;
    if (pooled && h->obs_delta && h->d_aux) {  // delta observation rows (emit kernel): a buffer other than the tracked one may hold anything -> "all rows"
        if (h->fill_pending) launch_fill_prev(h->d_aux, p.n_envs, p.nb, p.nl, st);
        p.aux = h->d_aux;
        p.delta = 1;
    }
    h->fill_pending = false;
    if (pooled) {
        p.walkq = (WalkItemC *)h->c_walkq; p.walk_ctr = h->d_walk_ctr; p.contq = h->d_contq; p.cont_ctr = h->d_walk_ctr + 1; p.walk_lanes = h->walk_lanes; p.walk_lanes_tall = h->walk_lanes_tall;
        p.walk_fork = h->walk_fork ? 1 : 0; p.walk_blocks = h->walk_blocks; p.walk_keep = h->walk_keep; p.piece_cap = p.n_envs * WALK_PIECES_PER_ENV;
        p.piece_ready = h->d_piece_ready; p.walk_pend = h->d_walk_pend;
    }
    cfg.gridDim = dim3(p.n_envs); cfg.blockDim = dim3(32);
    cudaLaunchKernelEx(&cfg, pctc_candidates_kernel, p);
    if (pooled) {
        static int n_sm = 0;
        if (!n_sm) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev); }
        if (stab) {
            pctc_walk_light_kernel<<<n_sm * 4, 128, 0, st>>>(p);
            if (p.walk_fork) pctc_walk_fork_kernel<<<n_sm * max(1, min(p.walk_blocks, 8)), 64, 0, st>>>(p);  // one resident wave
            else pctc_walk_kernel<<<n_sm * 8, 64, 0, st>>>(p);  // one resident wave
        }
        {
            cudaLaunchAttribute at2[1];
            at2[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            at2[0].val.programmaticStreamSerializationAllowed = 1;
            cudaLaunchConfig_t c2{};
            c2.stream = st; c2.attrs = at2; c2.numAttrs = (stab && cap == cudaStreamCaptureStatusNone) ? 1 : 0;
            c2.gridDim = dim3(p.n_envs); c2.blockDim = dim3(64);
            if (p.obs_f64) cudaLaunchKernelEx(&c2, pctc_emit_kernel<double>, p);
            else cudaLaunchKernelEx(&c2, pctc_emit_kernel<float>, p);
        }
        cudaError_t e2 = cudaGetLastError();
        if (e2 != cudaSuccess) { h->err = std::string("continuous launch: ") + cudaGetErrorString(e2); return PCT_ERR_CUDA; }
        h->launches += stab ? 4 : 2;  // apply, candidates, [light, walk], emit; the caller counts one
        return PCT_OK;
    }
    cfg.blockDim = dim3(64);
    if (h->cont_pre) {
        if (p.obs_f64) { if (stab) cudaLaunchKernelEx(&cfg, pctc_feas_emit_kernel<double, true, true>, p); else cudaLaunchKernelEx(&cfg, pctc_feas_emit_kernel<double, false, true>, p); }
        else { if (stab) cudaLaunchKernelEx(&cfg, pctc_feas_emit_kernel<float, true, true>, p); else cudaLaunchKernelEx(&cfg, pctc_feas_emit_kernel<float, false, true>, p); }
    } else {
        if (p.obs_f64) { if (stab) cudaLaunchKernelEx(&cfg, pctc_feas_emit_kernel<double, true, false>, p); else cudaLaunchKernelEx(&cfg, pctc_feas_emit_kernel<double, false, false>, p); }
        else { if (stab) cudaLaunchKernelEx(&cfg, pctc_feas_emit_kernel<float, true, false>, p); else cudaLaunchKernelEx(&cfg, pctc_feas_emit_kernel<float, false, false>, p); }
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { h->err = std::string("continuous launch: ") + cudaGetErrorString(e); return PCT_ERR_CUDA; }
    h->launches += 2;  // the caller counts one
    return PCT_OK;
}

int continuous_policy_random(pct_env_batch *h, int32_t *leaf_idx, uint64_t seed, int64_t t, cudaStream_t st) {
    pctc_policy_random_kernel<<<(h->n_envs + 127) / 128, 128, 0, st>>>((const CEnv *)h->c_state, h->n_envs, h->cfg.env_id_base, seed, t, leaf_idx);
    return cudaGetLastError() == cudaSuccess ? PCT_OK : PCT_ERR_CUDA;
}

int continuous_get_state(pct_env_batch *h, int env, pct_state_dump *out) {
    CEnv *tmp = (CEnv *)malloc(sizeof(CEnv));
    if (cudaMemcpy(tmp, (CEnv *)h->c_state + env, sizeof(CEnv), cudaMemcpyDeviceToHost) != cudaSuccess) { free(tmp); return PCT_ERR_CUDA; }
    memset(out, 0, sizeof(*out));
    out->n_boxes = tmp->h.n_box; out->n_ems = tmp->h.n_ems; out->n_leaf = tmp->h.n_leaf; out->flags = tmp->h.flags;
    out->draw_pos = tmp->h.draw_pos; out->next_den = tmp->h.next_den;
    for (int i = 0; i < 3; i++) out->next_box[i] = tmp->h.next_box[i];
    for (int i = 0; i < tmp->h.n_box && i < 80; i++) {
        const double *b = tmp->box[i];
        out->boxes[i][0] = b[0]; out->boxes[i][1] = b[1]; out->boxes[i][2] = b[2];
        out->boxes[i][3] = b[0] + b[3]; out->boxes[i][4] = b[1] + b[4]; out->boxes[i][5] = b[2] + b[5];
        out->boxes[i][6] = tmp->den[i];
    }
    for (int i = 0; i < tmp->h.n_ems && i < 256; i++)
        for (int t = 0; t < 6; t++) out->ems[i][t] = tmp->ems[i][t];
    free(tmp);
    return PCT_OK;
}

}  // namespace pct

#include "pct_heuristics_continuous.cuh"
