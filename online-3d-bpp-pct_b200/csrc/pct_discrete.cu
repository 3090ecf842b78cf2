// Discrete PCT environment: batched reset / step kernels for sm_100a.
//
// One warp owns one environment for the whole step:
//   TMA bulk load of the env's packed record (header + placed boxes + EMS list) HBM -> shared memory
//   -> decode action -> real placement (warp max-reduce over placed boxes for the resting height,
//      lane 0 runs the load-propagating stability update) -> EMS update (warp ballot / scan compaction)
//   -> candidate leaves in CPython-set order (hash table in shared memory)
//   -> feasibility, ONE LANE PER CANDIDATE (bounds, resting height over all placed boxes, stacking stability)
//   -> ordered compaction of the first `leaf_node_holder` feasible leaves (ballot + popc)
//   -> coalesced observation write, TMA bulk store of the record back to HBM.
//
// Reference behaviour restated here (D: = pct_envs/PctDiscrete0/ in the reference repo):
//   PackingDiscrete.step / reset / cur_observation / get_possible_position / LeafNode2Action  D:bin3D.py:61-188
//   Space.drop_box / drop_box_virtual / check_box / update_height_graph                       D:space.py:316-454
//   Space.GENEMS / Difference / EliminateInscribedEMS / EMSPoint                               D:space.py:457-570
//   ShmemVecEnv worker auto-reset                                                              wrapper/shmem_vec_env.py:139-143
// The height map of the reference is not materialised: max(plain[lx:lx+x, ly:ly+y]) equals the maximum top
// over placed boxes whose footprint overlaps the query footprint (update_height_graph sets covered cells to
// the new top, which is >= every older value there).
//
// Code-size discipline: the first version of this kernel was instruction-fetch bound (ncu r1a:
// stalled_no_instruction 11.3 of 19 stalled warps per issue, 202 KB of SASS).  Phases are __noinline__
// functions, loops over chunks are dynamic, candidate keys are canonical integers compared with one
// instruction instead of being re-derived from the EMS list on every probe.
#include "pct_common.cuh"
#include "pct_stability.cuh"
#include "pct_kernels.h"
#include "pct_geom.cuh"
#include "pct_walkq.cuh"
#include "pct_records.cuh"

namespace pct {

// ------------------------------------------------------------------------------------------------------
// NodeD / GeomD (geometry policy of the stability routine) and rest_height: pct_geom.cuh

// ---- shared-memory layout of one warp ------------------------------------------------------------------
// Candidate keys are canonical integers: xs | ys << B | zs << 2B | rot << 3B  (rot = first rotation index with
// the same oriented dims).  B = 4 bits when every container side is <= 16 (16-bit table slots), else 8 bits
// (32-bit slots).
// The CPython-set emulation walks table sizes 8 -> 32 -> 128 -> 512 -> 2048, alternating between two buffers:
// A holds the 8 / 128 / 2048 stages, B the 32 / 512 stages.  BIGSM = true keeps the 2048 stage in shared memory
// (setting 2: 6 orientations, hundreds of candidates per step); BIGSM = false (settings 1/3: <= 306 candidates in
// practice) keeps A at 128 slots and spills the rare 2048 stage to the env's cold record in HBM, which lets 28
// warps (= 4096 envs / 148 SMs) be resident per SM.
template <typename SlotT, bool BIGSM>
struct Lay {
    static constexpr int A_SLOTS = BIGSM ? TAB_A : 128;
    static constexpr int HOT = 0;
    static constexpr int TAB_A_OFF = HOT_PREFIX;
    static constexpr int TAB_B_OFF = TAB_A_OFF + A_SLOTS * sizeof(SlotT);
    static constexpr int LEAF = TAB_B_OFF + TAB_B * sizeof(SlotT);  // NL_MAX x 6 x i16
    static constexpr int MISC = LEAF + NL_MAX * 12;                 // mbarrier (8) + lock (4) + pad (4) + RotTab (32) + SetStage (384)
    static constexpr int PER_WARP = MISC + 48 + 384;
    static constexpr int BITS = sizeof(SlotT) == 2 ? 4 : 8;
    static_assert(TAB_A_OFF % 16 == 0 && PER_WARP % 16 == 0, "alignment");
    static_assert(E_MAX * 12 <= MISC - TAB_A_OFF, "EMS temp aliases tables + leaf buffer");
};

struct RotTab {   // per env/item: oriented dims of the R rotations (D:space.py:540-562), validity, canonical index
    uint8_t d[6][3];
    uint8_t valid, canon[6];
};

__device__ __forceinline__ void make_rot_tab(const int nb[3], int R, RotTab &rt) {
    const int perm[6][3] = {{0, 1, 2}, {1, 0, 2}, {0, 2, 1}, {1, 2, 0}, {2, 0, 1}, {2, 1, 0}};
    rt.valid = 0;
#pragma unroll
    for (int r = 0; r < 6; r++) {
        const int sx = nb[perm[r][0]], sy = nb[perm[r][1]], sz = nb[perm[r][2]];
        rt.d[r][0] = (uint8_t)sx; rt.d[r][1] = (uint8_t)sy; rt.d[r][2] = (uint8_t)sz;
        bool v = r < R;
        if (r == 1 || r == 4 || r == 5) v = v && sx != sy;
        if (r == 2 || r == 3) v = v && !(sx == sy && sy == sz);
        if (v) rt.valid |= 1 << r;
        int c = r;
        for (int q = r - 1; q >= 0; q--)
            if (rt.d[q][0] == sx && rt.d[q][1] == sy && rt.d[q][2] == sz) c = q;
        rt.canon[r] = (uint8_t)c;
    }
}

template <int BITS>
__device__ __forceinline__ uint32_t key_pack(int xs, int ys, int zs, int rot) {
    return (uint32_t)xs | ((uint32_t)ys << BITS) | ((uint32_t)zs << (2 * BITS)) | ((uint32_t)rot << (3 * BITS));
}
template <int BITS>
__device__ __forceinline__ void key_unpack(uint32_t k, int &xs, int &ys, int &zs, int &rot) {
    constexpr uint32_t M = (1u << BITS) - 1;
    xs = k & M; ys = (k >> BITS) & M; zs = (k >> (2 * BITS)) & M; rot = (k >> (3 * BITS)) & 7;
}
template <int BITS>
__device__ __noinline__ uint64_t key_hash(uint32_t k, const RotTab *rt) {
    int xs, ys, zs, rot;
    key_unpack<BITS>(k, xs, ys, zs, rot);
    const uint64_t l[6] = {(uint64_t)xs, (uint64_t)ys, (uint64_t)zs, (uint64_t)(xs + rt->d[rot][0]), (uint64_t)(ys + rt->d[rot][1]),
                           (uint64_t)(zs + rt->d[rot][2])};
    return tuple_hash6(l);
}

// ---- EMS update (GENEMS + Difference + EliminateInscribedEMS, D:space.py:457-531) -------------------------
__device__ __noinline__ int genems_warp(int16_t (*ems)[6], const int n0, int16_t (*tmp)[6], uint2 *pk, const int16_t *it, double low_bound, int lane,
                                        int &flags) {
    const double lb = low_bound == 0 ? 0.1 : low_bound;
    const int nch = (n0 + 31) >> 5;
    // pass 1: survivors (EMS not intersecting the new box) keep their order
    int off = 0;
#pragma unroll 1
    for (int c = 0; c < nch; c++) {
        const int i = c * 32 + lane;
        bool keep = false;
        if (i < n0) {
            const int16_t *m = ems[i];
            keep = !(max((int)m[0], (int)it[0]) < min((int)m[3], (int)it[3]) && max((int)m[1], (int)it[1]) < min((int)m[4], (int)it[4]) &&
                     max((int)m[2], (int)it[2]) < min((int)m[5], (int)it[5]));
        }
        const uint32_t bm = __ballot_sync(FULL, keep);
        if (keep) {
            const int p = off + __popc(bm & ((1u << lane) - 1));
#pragma unroll
            for (int t = 0; t < 6; t++) tmp[p][t] = ems[i][t];
        }
        off += __popc(bm);
    }
    // pass 2: children of the intersected EMS, parent order then fixed child order (left, right, front, back, top)
    bool overflow = false;
#pragma unroll 1
    for (int c = 0; c < nch; c++) {
        const int i = c * 32 + lane;
        uint32_t cm = 0;
        int a1 = 0, b1 = 0, c1 = 0, a2 = 0, b2 = 0, c2 = 0, x1 = 0, y1 = 0, x2 = 0, y2 = 0, z2 = 0;
        if (i < n0) {
            const int16_t *m = ems[i];
            a1 = m[0]; b1 = m[1]; c1 = m[2]; a2 = m[3]; b2 = m[4]; c2 = m[5];
            x1 = max(a1, (int)it[0]); y1 = max(b1, (int)it[1]);
            const int z1 = max(c1, (int)it[2]);
            x2 = min(a2, (int)it[3]); y2 = min(b2, (int)it[4]); z2 = min(c2, (int)it[5]);
            if (x1 < x2 && y1 < y2 && z1 < z2) {  // clamp + degenerate test of D:space.py:464-475
                const bool ux = (double)(a2 - a1) >= lb, uy = (double)(b2 - b1) >= lb, uz = (double)(c2 - c1) >= lb;
                if ((double)(x1 - a1) >= lb && uy && uz) cm |= 1;
                if ((double)(a2 - x2) >= lb && uy && uz) cm |= 2;
                if (ux && (double)(y1 - b1) >= lb && uz) cm |= 4;
                if (ux && (double)(b2 - y2) >= lb && uz) cm |= 8;
                if (ux && uy && (double)(c2 - z2) >= lb) cm |= 16;
            }
        }
        const int cnt = __popc(cm);
        const int incl = warp_incl_scan(cnt, lane);
        int p = off + incl - cnt;
#pragma unroll 1
        for (int ch = 0; ch < 5 && cm; ch++) {
            if (!(cm & (1u << ch))) continue;
            int q0 = a1, q1 = b1, q2 = c1, q3 = a2, q4 = b2, q5 = c2;
            if (ch == 0) q3 = x1;
            else if (ch == 1) q0 = x2;
            else if (ch == 2) q4 = y1;
            else if (ch == 3) q1 = y2;
            else q2 = z2;
            if (p < EMS_TMP_MAX) {
                tmp[p][0] = (int16_t)q0; tmp[p][1] = (int16_t)q1; tmp[p][2] = (int16_t)q2;
                tmp[p][3] = (int16_t)q3; tmp[p][4] = (int16_t)q4; tmp[p][5] = (int16_t)q5;
            } else overflow = true;
            p++;
        }
        off += __shfl_sync(FULL, incl, 31);
    }
    if (__any_sync(FULL, overflow)) flags |= PCT_FLAG_EMS_OVERFLOW;
    const int n = off < EMS_TMP_MAX ? off : EMS_TMP_MAX;  // intermediate list (survivors + children), before the inscribed-EMS purge
    __syncwarp();
    // EliminateInscribedEMS: drop i if some j != i contains it (non-strict; identical twins delete each other).
    // The O(n^2) containment test was 28 % of the apply kernel's warp instructions (ncu r2, profiles/r2_k1_head_source.txt): six 16-bit loads and
    // six compares per pair.  Coordinates are <= 255 (pct_create), so an EMS packs into two words of three 9-bit fields — lows as they are, highs
    // as 255 - v, which turns all six tests into "field of a >= field of b" — and with a guard bit per field one subtraction tests three fields:
    // ((a | G) - b) keeps the guard of a field iff a_f >= b_f (fields are >= 1 after the OR, so no borrow crosses a field).
    constexpr uint32_t G = (1u << 8) | (1u << 17) | (1u << 26);
    for (int i = lane; i < n; i += 32) {
        const int16_t *m = tmp[i];
        pk[i] = make_uint2((uint32_t)m[0] | ((uint32_t)m[1] << 9) | ((uint32_t)m[2] << 18),
                           (uint32_t)(255 - m[3]) | ((uint32_t)(255 - m[4]) << 9) | ((uint32_t)(255 - m[5]) << 18));
    }
    __syncwarp();
    int w = 0;
    const int nch2 = (n + 31) >> 5;
#pragma unroll 1
    for (int c = 0; c < nch2; c++) {
        const int i = c * 32 + lane;
        bool keep = false;
        if (i < n) {
            const uint2 a = pk[i];
            const uint32_t aL = a.x | G, aH = a.y | G;
            int hit = 0;
#pragma unroll 4
            for (int j = 0; j < n; j++) {
                const uint2 b = pk[j];
                hit |= (int)(((aL - b.x) & (aH - b.y) & G) == G && j != i);
            }
            keep = !hit;
        }
        const uint32_t bm = __ballot_sync(FULL, keep);
        if (keep) {
            const int p = w + __popc(bm & ((1u << lane) - 1));
            if (p < E_MAX) {
#pragma unroll
                for (int t = 0; t < 6; t++) ems[p][t] = tmp[i][t];
            }
        }
        w += __popc(bm);
    }
    if (w > E_MAX) { flags |= PCT_FLAG_EMS_OVERFLOW; w = E_MAX; }
    __syncwarp();
    return w;
}

// ---- candidate leaves in CPython set order (EMSPoint, D:space.py:534-570) ---------------------------------
// set_insert_clean (setobject.c) for a key known to be absent: plain scalar probe loop, run by ONE lane
template <typename SlotT>
__device__ __forceinline__ void table_insert_clean(SlotT *tab, uint32_t mask, uint64_t hash, SlotT key) {
    uint64_t perturb = hash;
    uint32_t i = (uint32_t)hash & mask;
#pragma unroll 1
    for (;;) {
        if (tab[i] == (SlotT)~(SlotT)0) { tab[i] = key; return; }
        if (i + 9 <= mask) {
#pragma unroll 1
            for (int j = 1; j <= 9; j++)
                if (tab[i + j] == (SlotT)~(SlotT)0) { tab[i + j] = key; return; }
        }
        perturb >>= 5;
        i = (uint32_t)((uint64_t)i * 5 + 1 + perturb) & mask;
    }
}

struct SetStage {  // per-warp staging of (hash, key) pairs for the serial insertion
    uint64_t h[32];
    uint32_t k[32];
};

// returns the candidate count; the ordered keys end up at the start of `out`.
// Inserting a key that is already in the set is a no-op, so only FIRST occurrences have to go through the
// order-defining serial insertion: every lane first looks its key up in the current table (read-only, the
// lookup of a present key follows exactly the probe sequence that placed it), duplicates inside the 32-wide
// chunk are collapsed onto their lowest lane with __match_any_sync, the surviving new keys are compacted into a
// shared-memory staging buffer in lane (= reference insertion) order and inserted by lane 0 with a scalar
// set_insert_clean (the kernel is instruction-issue bound: a one-lane scalar loop costs ~3x fewer warp
// instructions than a ballot-based warp-wide probe).  Resizes re-hash the old table in parallel, 32 slots at a time.
template <typename SlotT>
__device__ __noinline__ int build_candidates(const int16_t (*ems)[6], int n_ems, const RotTab *rt, int R, SlotT *tabA, SlotT *tabB, SlotT *tabBig,
                                             SetStage *stg, SlotT *&out, int lane, int &flags, const uint32_t *raw_keys = nullptr, int n_raw = 0) {
    constexpr int BITS = sizeof(SlotT) == 2 ? 4 : 8;
    constexpr SlotT EMPTY = (SlotT)~(SlotT)0;
    SlotT *tab = tabA;
    uint32_t mask = 7;
    int fill = 0;
    if (lane < 8) tab[lane] = EMPTY;
    __syncwarp();
    const int raw = raw_keys ? n_raw : n_ems * R * 4;  // raw_keys: insertion sequence produced by an EV / EP / CP / FC generator
    bool stop = false;
#pragma unroll 1
    for (int base = 0; base < raw && !stop; base += 32) {
        const int r = base + lane;
        bool valid = false;
        uint64_t hash = 0;
        uint32_t key = 0xFFFFFFFFu;
        if (r < raw && raw_keys) {
            valid = true;
            key = raw_keys[r];
            hash = key_hash<BITS>(key, rt);
        } else if (r < raw) {
            const int q = r & 3, er = r >> 2;
            const int rot = er % R, ei = er / R;
            if (rt->valid & (1 << rot)) {
                const int sx = rt->d[rot][0], sy = rt->d[rot][1], sz = rt->d[rot][2];
                const int16_t *m = ems[ei];
                if (m[3] - m[0] >= sx && m[4] - m[1] >= sy && m[5] - m[2] >= sz) {
                    valid = true;
                    const int xs = (q & 1) ? m[3] - sx : m[0];
                    const int ys = (q & 2) ? m[4] - sy : m[1];
                    key = key_pack<BITS>(xs, ys, m[2], rt->canon[rot]);
                    hash = key_hash<BITS>(key, rt);
                }
            }
        }
        // first occurrence inside the chunk
        const uint32_t same = __match_any_sync(FULL, key);
        if (valid && (same & ((1u << lane) - 1))) valid = false;
        // already in the set?  (set_add_entry probe sequence, read-only)
        if (valid) {
            uint64_t perturb = hash;
            uint32_t i = (uint32_t)hash & mask;
            bool open = true;
            while (open) {
                const int probes = (i + 9 <= mask) ? 9 : 0;
                for (int j = 0; j <= probes; j++) {
                    const SlotT e = tab[i + j];
                    if (e == EMPTY) { open = false; break; }
                    if (e == (SlotT)key) { open = false; valid = false; break; }
                }
                perturb >>= 5;
                i = (uint32_t)((uint64_t)i * 5 + 1 + perturb) & mask;
            }
        }
        const uint32_t vm = __ballot_sync(FULL, valid);
        int n_new = __popc(vm);
        if (valid) {
            const int pos = __popc(vm & ((1u << lane) - 1));
            stg->h[pos] = hash;
            stg->k[pos] = key;
        }
        __syncwarp();
        int done = 0;
#pragma unroll 1
        while (done < n_new) {
            // lane 0: insert staged keys until the set has to grow
            int upto = n_new;
            if (lane == 0) {
#pragma unroll 1
                for (int t = done; t < n_new; t++) {
                    table_insert_clean<SlotT>(tab, mask, stg->h[t], (SlotT)stg->k[t]);
                    if ((uint32_t)(++fill) * 5 >= mask * 3) { upto = t + 1; break; }
                }
            }
            upto = __shfl_sync(FULL, upto, 0);
            fill = __shfl_sync(FULL, fill, 0);
            done = upto;
            __syncwarp();
            if ((uint32_t)fill * 5 >= mask * 3) {
                // set_table_resize(used * 4): smallest power of two > 4 * used, re-insert in slot order
                uint32_t newsize = 8;
                while (newsize <= (uint32_t)fill * 4) newsize <<= 1;
                if (newsize > TAB_A) { flags |= PCT_FLAG_CAND_OVERFLOW; stop = true; break; }
                SlotT *nt = newsize == TAB_A ? tabBig : ((tab == tabA) ? tabB : tabA);
                for (uint32_t t = lane; t < newsize; t += 32) nt[t] = EMPTY;
                // the staged keys not inserted yet must survive: move them to registers
                const uint64_t keep_h = (done + lane < n_new) ? stg->h[done + lane] : 0;
                const uint32_t keep_k = (done + lane < n_new) ? stg->k[done + lane] : 0;
                __syncwarp();
#pragma unroll 1
                for (uint32_t b2 = 0; b2 <= mask; b2 += 32) {
                    const uint32_t s = b2 + lane;
                    const SlotT e = s <= mask ? tab[s] : EMPTY;
                    const uint32_t em = __ballot_sync(FULL, e != EMPTY);
                    if (e != EMPTY) {
                        const int pos = __popc(em & ((1u << lane) - 1));
                        stg->h[pos] = key_hash<BITS>(e, rt);
                        stg->k[pos] = e;
                    }
                    __syncwarp();
                    if (lane == 0) {
                        const int m2 = __popc(em);
#pragma unroll 1
                        for (int t = 0; t < m2; t++) table_insert_clean<SlotT>(nt, newsize - 1, stg->h[t], (SlotT)stg->k[t]);
                    }
                    __syncwarp();
                }
                tab = nt;
                mask = newsize - 1;
                // restore the pending keys at the front of the staging buffer
                if (done + lane < n_new) { stg->h[lane] = keep_h; stg->k[lane] = keep_k; }
                // (indices shift: pending key t now sits at t - done)
                __syncwarp();
                n_new -= done;  // the pending keys now sit at staged[0 .. n_new)
                done = 0;
            }
        }
    }
    __syncwarp();
    // iteration order = slot order: compact the keys in place
    int cnt = 0;
#pragma unroll 1
    for (uint32_t b2 = 0; b2 <= mask; b2 += 32) {
        const uint32_t s = b2 + lane;
        const SlotT e = s <= mask ? tab[s] : EMPTY;
        const uint32_t em = __ballot_sync(FULL, e != EMPTY);
        __syncwarp();
        if (e != EMPTY) tab[cnt + __popc(em & ((1u << lane) - 1))] = e;
        cnt += __popc(em);
        __syncwarp();
    }
    out = tab;
    return cnt;
}

// ---- the other leaf-node expansion schemes (D:bin3D.py:101-112): generators of the set-insertion sequence --------------
constexpr int RAW_MAX = 2048;

// FullCoord (D:space.py:573-610): every cell x valid rotation with lz = height of the cell, rot-major / lx / ly order
template <int BITS>
__device__ __noinline__ int gen_full_coord(const int16_t (*box)[6], int n_box, const RotTab *rt, int R, int W, int L, int H, uint32_t *raw,
                                           int lane, int &flags) {
    int n = 0;
    const int cells = W * L;
#pragma unroll 1
    for (int rot = 0; rot < R; rot++) {
        if (!(rt->valid & (1 << rot))) continue;
        const int sx = rt->d[rot][0], sy = rt->d[rot][1], sz = rt->d[rot][2];
#pragma unroll 1
        for (int b = 0; b < cells; b += 32) {
            const int c = b + lane, lx = c / L, ly = c - lx * L;
            bool ok = false;
            int lz = 0;
            if (c < cells) {
                lz = rest_height(box, 0, n_box, 1, lx, ly, lx + 1, ly + 1);
                ok = lx + sx <= W && ly + sy <= L && lz + sz <= H;
            }
            const uint32_t m = __ballot_sync(FULL, ok);
            if (ok) {
                const int p = n + __popc(m & ((1u << lane) - 1));
                if (p < RAW_MAX) raw[p] = key_pack<BITS>(lx, ly, lz, rt->canon[rot]);
            }
            n += __popc(m);
        }
    }
    if (n > RAW_MAX) { flags |= PCT_FLAG_CAND_OVERFLOW; n = RAW_MAX; }
    __syncwarp();
    return n;
}

// EventPoint (D:space.py:613-693) as the reference actually behaves: GENEMS (which maintains EMS and ZMAP) only runs for
// LNES == 'EMS' (D:bin3D.py:172-175), so ZMAP stays {0: x_up [0], y_left [0], x_bottom [W], y_right [L]} and the EMS list
// stays [whole bin]: four bin-corner placements per rotation at z = 0 (oversized rotations produce nothing valid).
template <int BITS>
__device__ __noinline__ int gen_event_point(const RotTab *rt, int R, int W, int L, uint32_t *raw, int lane) {
    int n = 0;
    if (lane == 0) {
        for (int rot = 0; rot < R; rot++) {
            if (!(rt->valid & (1 << rot))) continue;
            const int sx = rt->d[rot][0], sy = rt->d[rot][1], c = rt->canon[rot];
            if (sx > W || sy > L) continue;
            raw[n++] = key_pack<BITS>(0, 0, 0, c);
            raw[n++] = key_pack<BITS>(0, L - sy, 0, c);
            raw[n++] = key_pack<BITS>(W - sx, 0, 0, c);
            raw[n++] = key_pack<BITS>(W - sx, L - sy, 0, c);
        }
    }
    n = __shfl_sync(FULL, n, 0);
    __syncwarp();
    return n;
}

// ExtremePoint2D (ep = true, D:space.py:696-750 + PctTools.extreme2D :107-135) and CornerPoint (ep = false,
// D:space.py:752-806 + PctTools.corners2D :137-159): per distinct top level k, the 2-D points of the boxes whose top is
// above k; points new w.r.t. the previous level x rotations.  Small serial algorithms over <= 80 boxes: lane 0 runs them.
// Returns -2 for the empty-bin special case (two hard-coded placements, a list, no set).
template <int BITS>
__device__ __noinline__ int gen_level_points(const int16_t (*box)[6], int n_box, const RotTab *rt, int R, int W, int L, int H, bool ep,
                                             uint32_t *raw, int lane, int &flags) {
    if (n_box == 0) return -2;
    int n = 0;
    if (lane == 0) {
        int16_t tset[NB_MAX + 1];
        int nt = 0;
        tset[nt++] = 0;
        for (int i = 0; i < n_box; i++) {
            const int16_t t = box[i][5];
            bool f = false;
            for (int k = 0; k < nt; k++) f |= tset[k] == t;
            if (!f) tset[nt++] = t;
        }
        for (int i = 1; i < nt; i++) { int16_t v = tset[i]; int j = i - 1; while (j >= 0 && tset[j] > v) { tset[j + 1] = tset[j]; j--; } tset[j + 1] = v; }
        uint8_t ord[NB_MAX], em[NB_MAX];
        int16_t cur[2 * NB_MAX + 2][2], last[2 * NB_MAX + 2][2];
        int nlast = 0;
        bool over = false;
        for (int ti = 0; ti < nt; ti++) {
            const int k = tset[ti];
            int nr = 0, nc = 0;
            for (int i = 0; i < n_box; i++)
                if (box[i][5] > k) ord[nr++] = (uint8_t)i;  // IK in box order
            if (nr == 0) { cur[0][0] = 0; cur[0][1] = 0; nc = 1; }
            else if (!ep) {
                // corners2D: stable sort by (y_end, x_end) descending, staircase of the items that extend x
                for (int i = 1; i < nr; i++) {
                    const uint8_t o = ord[i];
                    int j = i - 1;
                    while (j >= 0 && (box[ord[j]][4] < box[o][4] || (box[ord[j]][4] == box[o][4] && box[ord[j]][3] < box[o][3]))) { ord[j + 1] = ord[j]; j--; }
                    ord[j + 1] = o;
                }
                int xrec = 0, m = 0;
                for (int i = 0; i < nr; i++)
                    if (box[ord[i]][3] > xrec) { em[m++] = ord[i]; xrec = box[ord[i]][3]; }
                cur[nc][0] = 0; cur[nc][1] = box[ord[0]][4]; nc++;
                for (int i = 1; i < m; i++) { cur[nc][0] = box[em[i - 1]][3]; cur[nc][1] = box[em[i]][4]; nc++; }
                cur[nc][0] = box[em[m - 1]][3]; cur[nc][1] = 0; nc++;
            } else {
                // extreme2D: stable sort by (ly, x_end) ascending; the two `demo` walls use the reference's hard-coded 10
                for (int i = 1; i < nr; i++) {
                    const uint8_t o = ord[i];
                    int j = i - 1;
                    while (j >= 0 && (box[ord[j]][1] > box[o][1] || (box[ord[j]][1] == box[o][1] && box[ord[j]][3] > box[o][3]))) { ord[j + 1] = ord[j]; j--; }
                    ord[j + 1] = o;
                }
                for (int i = 0; i < nr; i++) {
                    const int16_t *ni = box[ord[i]];
                    int maxb0 = -10, maxb2 = -10, e0x = 0, e0y = 0, e2x = 0, e2y = 0;
                    bool has0 = false, has2 = false;
                    bool first2 = false;  // newEps is a dict: .values() lists key 2 before key 0 when newEps[2] was assigned first (D:PctTools.py:121-127)
                    for (int b = 0; b < 2 + i; b++) {
                        int bx2, bx3;
                        if (b == 0) { bx2 = 0; bx3 = 10; } else if (b == 1) { bx2 = 10; bx3 = 0; } else { bx2 = box[ord[b - 2]][3]; bx3 = box[ord[b - 2]][4]; }
                        if (ni[0] >= bx2 && ni[4] < bx3 && bx2 > maxb0) { e0x = bx2; e0y = ni[4]; maxb0 = bx2; has0 = true; }
                        if (ni[1] >= bx3 && ni[3] < bx2 && bx3 > maxb2) { e2x = ni[3]; e2y = bx3; maxb2 = bx3; if (!has2 && !has0) first2 = true; has2 = true; }
                    }
                    int w = 0;  // deleteEps2D
                    for (int q = 0; q < nc; q++)
                        if (!(cur[q][0] >= ni[0] && cur[q][0] < ni[3] && cur[q][1] >= ni[1] && cur[q][1] < ni[4])) { cur[w][0] = cur[q][0]; cur[w][1] = cur[q][1]; w++; }
                    nc = w;
                    if (has0 && has2 && !(e0x == e2x && e0y == e2y)) {
                        // list(set(newEps.values())): CPython order of two int 2-tuples in an 8-slot table; the values are inserted in the
                        // dict's key order, the first takes its home slot, the second probes from its own (perturb path); iteration = slot order
                        uint64_t l0[2] = {(uint64_t)e0x, (uint64_t)e0y}, l2[2] = {(uint64_t)e2x, (uint64_t)e2y};
                        const uint64_t h0 = tuple_hash_n(l0, 2), h2 = tuple_hash_n(l2, 2);
                        uint64_t s0 = h0 & 7, s2 = h2 & 7;
                        if (first2) { uint64_t pert = h0; while (s0 == s2) { pert >>= 5; s0 = (s0 * 5 + 1 + pert) & 7; } }
                        else { uint64_t pert = h2; while (s2 == s0) { pert >>= 5; s2 = (s2 * 5 + 1 + pert) & 7; } }
                        if (s0 < s2) { cur[nc][0] = e0x; cur[nc][1] = e0y; nc++; cur[nc][0] = e2x; cur[nc][1] = e2y; nc++; }
                        else { cur[nc][0] = e2x; cur[nc][1] = e2y; nc++; cur[nc][0] = e0x; cur[nc][1] = e0y; nc++; }
                    } else if (has0) { cur[nc][0] = e0x; cur[nc][1] = e0y; nc++; }
                    else if (has2) { cur[nc][0] = e2x; cur[nc][1] = e2y; nc++; }
                }
            }
            for (int q = 0; q < nc; q++) {
                bool f = false;
                for (int u = 0; u < nlast; u++) f |= last[u][0] == cur[q][0] && last[u][1] == cur[q][1];
                if (f) continue;
                for (int rot = 0; rot < R; rot++) {  // CI point x rotation -> insertion sequence of posVec
                    if (!(rt->valid & (1 << rot))) continue;
                    if (cur[q][0] + rt->d[rot][0] <= W && cur[q][1] + rt->d[rot][1] <= L && k + rt->d[rot][2] <= H) {
                        if (n < RAW_MAX && cur[q][0] >= 0 && cur[q][1] >= 0) raw[n++] = key_pack<BITS>(cur[q][0], cur[q][1], k, rt->canon[rot]);
                        else over = true;
                    }
                }
            }
            for (int q = 0; q < nc; q++) { last[q][0] = cur[q][0]; last[q][1] = cur[q][1]; }
            nlast = nc;
        }
        if (over) flags |= PCT_FLAG_CAND_OVERFLOW;
    }
    n = __shfl_sync(FULL, n, 0);
    __syncwarp();
    return n;
}

// ---- item source ------------------------------------------------------------------------------------------
__device__ __noinline__ void draw_item(const DParams &p, int e, DHdr &h) {
    const uint64_t gid = (uint64_t)h.item_env;  // the env's own global id unless a saved record was loaded into it
    const uint64_t d = (uint64_t)h.draw_pos;
    const double *it;
    if (p.item_mode == 0) {
        it = p.item_set + (rnd_u64(p.seed, gid, d) % (uint64_t)p.n_items) * 3;
        h.next_den = p.setting == 3 ? rnd_density(p.seed, gid, d) : 1.0;
    } else {
        it = p.stream + ((size_t)(h.item_env - p.env_id_base) * p.stream_len + (size_t)(d % (uint64_t)p.stream_len)) * 4;
        h.next_den = p.setting == 3 ? it[3] : 1.0;
    }
    h.next_box[0] = (int)it[0];
    h.next_box[1] = (int)it[1];
    h.next_box[2] = (int)it[2];
    h.draw_pos++;
}

// Space.reset (D:space.py:290-314) + box_creator.reset / generate_box_size (D:bin3D.py:62-65)
__device__ __noinline__ void reset_space(DEnvHot *hot, const DParams &p, int e, int lane) {
    if (lane == 0) {
        DHdr &h = hot->h;
        h.n_box = 0; h.n_ems = 1; h.n_leaf = 0; h.flags = 0; h.n_edge = 0; h.n_poly = 0; h.vol_sum = 0; h.ep_len = 0; h.ep_reward = 0;
        hot->ems[0][0] = 0; hot->ems[0][1] = 0; hot->ems[0][2] = 0;
        hot->ems[0][3] = (int16_t)p.W; hot->ems[0][4] = (int16_t)p.L; hot->ems[0][5] = (int16_t)p.H;
        if (p.traj_len > 0 && h.draw_pos % p.traj_len) h.draw_pos += p.traj_len - h.draw_pos % p.traj_len;  // LoadBoxCreator.reset
        draw_item(p, e, h);
    }
    __syncwarp();
}

// PART: 0 = the whole observation (round 1's block kernel), 1 = internal-node rows + item row (written by the candidates kernel since round 2: they
// are final after the apply kernel, and on the zero-copy host path their PCIe traffic then overlaps the walk kernels), 2 = leaf rows (emit kernel).
template <typename OT, int PART = 0>
__device__ __noinline__ void write_obs(const DParams &p, int e, const DEnvHot *hot, const DEnvCold *cold, const int16_t (*leaf)[6], int n_leaf,
                                       int tid, int nthreads) {
    OT *obs = (OT *)p.obs + (size_t)e * (size_t)((p.nb + p.nl + 1) * 9);
    const int n_box = hot->h.n_box;
    int s0 = hot->h.next_box[0], s1 = hot->h.next_box[1], s2 = hot->h.next_box[2];
    if (s1 < s0) { int t = s0; s0 = s1; s1 = t; }
    if (s2 < s1) { int t = s1; s1 = s2; s2 = t; }
    if (s1 < s0) { int t = s0; s0 = s1; s1 = t; }
    const OT den = (OT)hot->h.next_den;
    const bool s3 = p.setting == 3;
    const int r_lo = PART == 2 ? p.nb : 0, r_hi = PART == 1 ? p.nb : (PART == 2 ? p.nb + p.nl : p.nb + p.nl + 1);
    const int f_lo = r_lo * 9, f_hi = r_hi * 9;
#pragma unroll 4
    for (int f = f_lo + tid; f < f_hi + (PART == 1 ? 9 : 0); f += nthreads) {
        int row = f / 9;
        const int col = f - row * 9;
        if (PART == 1 && row >= p.nb) row = p.nb + p.nl;  // the 9 extra elements of PART 1 are the item row
        OT v = 0;
        if (row < p.nb) {
            if (row < n_box) {
                if (col < 6) v = (OT)hot->box[row][col];
                else if (col == 6) v = s3 ? (OT)cold->density[row] : (OT)1;
                else if (col == 8) v = 1;
            } else if (row == 0 && col == 8) v = 1;  // D:space.py:294-295
        } else if (row < p.nb + p.nl) {
            const int k = row - p.nb;
            if (k < n_leaf) {
                if (col < 5) v = (OT)leaf[k][col];
                else if (col == 5) v = (OT)p.H;  // D:bin3D.py:128 — bin height, not ze
                else if (col == 8) v = 1;
            }
        } else {
            if (col == 0) v = den;
            else if (col == 3) v = (OT)s0;
            else if (col == 4) v = (OT)s1;
            else if (col == 5) v = (OT)s2;
            else if (col == 8) v = 1;
        }
        obs[row * 9 + col] = v;
    }
}

// Delta variant (default, PCT_B200_OBS_DELTA=0 disables): the caller hands back the SAME observation buffer every step, and prev[0] / prev[1]
// hold how many internal / leaf rows of it may be non-zero.  75 % of the (NB + NL + 1) x 9 observation is zero padding, so only the
// rows below max(now, prev) and the next-item row are written (and prev is updated); every other row is zero already.  The written
// values are the ones write_obs computes.  The host resets prev to {NB, NL} whenever the buffer changes.
template <typename OT, bool WARP_SCOPE = false, int PART = 0>
__device__ __noinline__ void write_obs_delta(const DParams &p, int e, const DEnvHot *hot, const DEnvCold *cold, const int16_t (*leaf)[6], int n_leaf,
                                             int tid, int nthreads) {
    OT *obs = (OT *)p.obs + (size_t)e * (size_t)((p.nb + p.nl + 1) * 9);
    int32_t *prev = p.aux[e].obs_prev;
    const int n_box = hot->h.n_box;
    const int pb = min(prev[0], p.nb), pl = min(prev[1], p.nl);
    if constexpr (WARP_SCOPE) __syncwarp(); else __syncthreads();  // every thread of the env has read prev before thread 0 replaces it below
    const int wb = PART == 2 ? 0 : max(max(n_box, pb), 1);  // row 0 always carries its valid flag (D:space.py:294-295)
    const int wl = PART == 1 ? 0 : max(n_leaf, pl);
    int s0 = hot->h.next_box[0], s1 = hot->h.next_box[1], s2 = hot->h.next_box[2];
    if (s1 < s0) { int t = s0; s0 = s1; s1 = t; }
    if (s2 < s1) { int t = s1; s1 = s2; s2 = t; }
    if (s1 < s0) { int t = s0; s0 = s1; s1 = t; }
    const OT den = (OT)hot->h.next_den;
    const bool s3 = p.setting == 3;
    const int total = (wb + wl + (PART == 2 ? 0 : 1)) * 9;
#pragma unroll 1
    for (int f = tid; f < total; f += nthreads) {
        const int r = f / 9, col = f - r * 9;
        OT v = 0;
        int row;
        if (r < wb) {
            row = r;
            if (row < n_box) {
                if (col < 6) v = (OT)hot->box[row][col];
                else if (col == 6) v = s3 ? (OT)cold->density[row] : (OT)1;
                else if (col == 8) v = 1;
            } else if (row == 0 && col == 8) v = 1;
        } else if (r < wb + wl) {
            const int k = r - wb;
            row = p.nb + k;
            if (k < n_leaf) {
                if (col < 5) v = (OT)leaf[k][col];
                else if (col == 5) v = (OT)p.H;
                else if (col == 8) v = 1;
            }
        } else {
            row = p.nb + p.nl;
            if (col == 0) v = den;
            else if (col == 3) v = (OT)s0;
            else if (col == 4) v = (OT)s1;
            else if (col == 5) v = (OT)s2;
            else if (col == 8) v = 1;
        }
        obs[row * 9 + col] = v;
    }
    if (tid == 0) {
        if (PART != 2) prev[0] = max(n_box, 1);
        if (PART != 1) prev[1] = n_leaf;
    }
}

// ======================================================================================================
// The step is a pipeline of three kernels (plus the optional synthetic-policy kernel).  A monolithic
// one-warp-per-env kernel was measured first (profiles/r1_monolithic_*.txt): it was instruction-fetch bound
// (each warp streamed ~80 KB of SASS once per step, warps of an SM sat in different phases) and its duration
// was the latency of the slowest env.  Splitting by phase keeps every kernel's code small and hot in the
// instruction cache and lets the heavy phase run one THREAD per candidate leaf.
//   K1 apply      warp / env    action decode, real placement (+ load-propagating stability), EMS update,
//                               reward / done / info, auto-reset, next item
//   K2 candidates warp / env    EMSPoint in CPython-set order -> ordered candidate list in HBM
//   K3 feas_emit  block / env   thread per candidate: bounds, resting height, virtual stability;
//                               ordered compaction into the leaf slots; observation write
// ======================================================================================================
#ifdef PCT_PHASE_TIMERS
__device__ __forceinline__ long long gtime() { long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#define KT_BEGIN() const long long kt0_ = gtime(); const long long kc0_ = clock64()
#define KT_END(e, k) do { if (p.mode == 1 && p.dbg) { p.dbg[(size_t)(e) * 16 + (k) * 4 + 0] = kt0_; p.dbg[(size_t)(e) * 16 + (k) * 4 + 1] = gtime(); \
        p.dbg[(size_t)(e) * 16 + (k) * 4 + 2] = clock64() - kc0_; } } while (0)
#else
#define KT_BEGIN()
#define KT_END(e, k)
#endif
#ifndef K1_MINB
#define K1_MINB 6   // sweep (r1): 168 regs / 6 blocks per SM beats 72 regs / 14 blocks — spills cost more than occupancy gives
#endif
#ifndef K3_MINB
#define K3_MINB 8   // sweep (r1): 128 regs / 8 blocks per SM
#endif
// ---- block scheduling order (longest-processing-time-first) --------------------------------------------------------------------------
// A launch lasts as long as its slowest block and blocks are dispatched in index order, so the envs with the most expected work (boxes placed
// drive the real stability descent and the EMS update) get the lowest slots.  No sorting pass: pct_apply_kernel files every env under its
// work key for the NEXT step (one atomicAdd into a 64-bucket histogram + one store into that bucket's list), and the apply / candidates
// kernels of the next step turn their slot into an env with a 64-entry warp scan.  Two parities: a step reads what the previous step
// wrote; the emit kernel (last of the sequence) empties the buckets just consumed and flips the parity ON THE DEVICE, so captured graphs replay
// correctly.  Layout of DParams::order (int32): [0] parity, [2 + 64 * par + j] count of bucket j = 63 - key, [ORD_LIST + (64 * par + j) * n_envs + i] envs.
constexpr int ORD_BUCKETS = 64, ORD_CNT = 2, ORD_LIST = ORD_CNT + 2 * ORD_BUCKETS;
__device__ __forceinline__ int order_lookup(const int32_t *ord, int n_envs, int slot, int lane) {
    const int par = *(volatile const int32_t *)ord & 1;
    const int32_t *cnt = ord + ORD_CNT + ORD_BUCKETS * par;
    const int a = cnt[2 * lane], b = cnt[2 * lane + 1];
    int incl = a + b;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(FULL, incl, d);
        if (lane >= d) incl += t;
    }
    const uint32_t m = __ballot_sync(FULL, slot < incl);
    if (m == 0) return slot;  // not a whole-batch history (cannot happen after pct_create's initialisation): identity
    const int f = __ffs(m) - 1;
    const int incl_f = __shfl_sync(FULL, incl, f), a_f = __shfl_sync(FULL, a, f), b_f = __shfl_sync(FULL, b, f);
    int off = slot - (incl_f - a_f - b_f), j = 2 * f;
    if (off >= a_f) { off -= a_f; j++; }
    return ord[ORD_LIST + (size_t)(ORD_BUCKETS * par + j) * n_envs + off];
}
__device__ __forceinline__ void order_file(int32_t *ord, int n_envs, int e, int n_box, int n_ems) {
    const int par = *(volatile const int32_t *)ord & 1;
    const int j = 63 - min(63, n_box + (n_ems >> 1));
    const int pos = atomicAdd(ord + ORD_CNT + ORD_BUCKETS * (par ^ 1) + j, 1);
    if (pos < n_envs) ord[ORD_LIST + (size_t)(ORD_BUCKETS * (par ^ 1) + j) * n_envs + pos] = e;
}

constexpr int K1_SM_PER_WARP = sizeof(DEnvHot) + EMS_TMP_MAX * 12 + 16 + EDGE_STAGE * 32 + POLY_STAGE * 16 + EMS_TMP_MAX * 8;  // record + EMS temp + mbarrier/lock + staged loads + packed EMS temp
static_assert(K1_SM_PER_WARP % 16 == 0, "alignment");

template <bool STAB, bool ALIAS = false>
__global__ void __launch_bounds__(32 * WARPS_PER_BLOCK, K1_MINB) pct_apply_kernel(const DParams p) {  // ALIAS: see EdgePoolA (the default; PCT_B200_ALIAS=0 selects the snapshot kernel)
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int slot = blockIdx.x * WARPS_PER_BLOCK + warp;
    if (slot >= p.n_envs) return;
    const int e = (p.order && p.mode == 1) ? order_lookup(p.order, p.n_envs, slot, lane) : slot;  // heaviest envs first (longest-processing-time-first)
    unsigned char *sm = smem_raw + (size_t)warp * K1_SM_PER_WARP;
    DEnvHot *hot = (DEnvHot *)sm;
    // per-warp layout: record | EMS temp (3 KB) | packed EMS temp (2 KB) | mbarrier + lock | staged loads | staged polygons.  The two EMS areas are
    // only used by GENEMS, after the descent: the descent's working arrays (StabScratch, 4 KB) are aliased onto them
    int16_t (*ems_tmp)[6] = (int16_t (*)[6])(sm + sizeof(DEnvHot));
    uint2 *ems_pk = (uint2 *)(sm + sizeof(DEnvHot) + EMS_TMP_MAX * 12);
    static_assert(sizeof(StabScratch) <= EMS_TMP_MAX * 12 + EMS_TMP_MAX * 8 && sizeof(DEnvHot) % 8 == 0, "the descent's scratch fits the EMS temp areas");
    StabScratch *scr = (StabScratch *)ems_tmp;
    uint64_t *mbar = (uint64_t *)(sm + sizeof(DEnvHot) + EMS_TMP_MAX * 12 + EMS_TMP_MAX * 8);
    int *lock = (int *)(mbar + 1);
    Stack4 *st_sm = (Stack4 *)(sm + sizeof(DEnvHot) + EMS_TMP_MAX * 12 + EMS_TMP_MAX * 8 + 16);
    double *poly_sm = (double *)(st_sm + EDGE_STAGE);
    DEnvHot *ghot = p.hot + e;
    DEnvCold *cold = p.cold + e;
    DHdr &h = hot->h;
    KT_BEGIN();
    if (p.ready) pdl_launch_dependents();
    if (lane == 0) *lock = 0;
    float reward = 0.f;
    int done = 0;
    pct_step_info info{};

    if (p.mode == 0) {
        // ---------------- reset (D:bin3D.py:61-67, D:space.py:290-314) ----------------
        const int64_t dp = p.keep_draw ? ghot->h.draw_pos : 0;  // box_creator.reset() does not rewind the item source
        const int64_t ie = p.keep_draw ? ghot->h.item_env : p.env_id_base + e;  // ... nor change the sequence it follows
        for (int t = lane; t < (int)(sizeof(DEnvHot) / 4); t += 32) ((uint32_t *)hot)[t] = 0;
        __syncwarp();
        if (lane == 0) { hot->h.draw_pos = dp; hot->h.item_env = ie; }
        __syncwarp();
        reset_space(hot, p, e, lane);
    } else {
        // ---------------- stage the env record: HBM -> smem via TMA ----------------
        if (lane == 0) {
            mbar_init(mbar, 1);
            fence_proxy_async();
        }
        __syncwarp();
        if (lane == 0) {
            mbar_expect_tx(mbar, (uint32_t)sizeof(DEnvHot));
            tma_load_1d(hot, ghot, (uint32_t)sizeof(DEnvHot), mbar);
        }
        mbar_wait(mbar, 0);
        __syncwarp();
        if (STAB && h.n_edge > 0) {  // stage the load edges and support polygons too (second phase of the same mbarrier)
            const uint32_t bytes = (uint32_t)min(h.n_edge, EDGE_STAGE) * (uint32_t)sizeof(Stack4);
            const uint32_t pbytes = (uint32_t)min(h.n_poly, POLY_STAGE) * 16u;
            if (lane == 0) {
                mbar_expect_tx(mbar, bytes + pbytes);
                tma_load_1d(st_sm, cold->e_st, bytes, mbar);
                if (pbytes) tma_load_1d(poly_sm, cold->poly, pbytes, mbar);
            }
            mbar_wait(mbar, 1);
            __syncwarp();
        }

        const int nb0 = h.next_box[0], nb1 = h.next_box[1], nb2 = h.next_box[2];
        const int n_box0 = h.n_box, n_leaf0 = h.n_leaf, flags0 = h.flags;
        const double next_den0 = h.next_den;
        __syncwarp();
        // ---- LeafNode2Action (D:bin3D.py:139-149) ----
        int lx = 0, ly = 0, x = nb0, y = nb1, z = nb2;
        bool bad = false;
        {
            double a0 = 0, a1 = 0, a3 = 0, a4 = 0;
            bool zero = true;
            if (p.leaf_idx) {
                const int k = p.leaf_idx[e];
                if (k >= 0 && k < n_leaf0) {
                    zero = false;
                    const int16_t *l = cold->leaf[k];
                    a0 = l[0]; a1 = l[1]; a3 = l[3]; a4 = l[4];
                }
            } else {
                double a[6], s = 0;
#pragma unroll
                for (int t = 0; t < 6; t++) {
                    a[t] = p.action_f64 ? ((const double *)p.actions)[(size_t)e * 9 + t] : (double)((const float *)p.actions)[(size_t)e * 9 + t];
                    s += a[t];
                }
                zero = (s == 0);
                a0 = a[0]; a1 = a[1]; a3 = a[3]; a4 = a[4];
            }
            if (!zero) {
                x = (int)(a3 - a0);
                y = (int)(a4 - a1);
                // z = what is left of next_box after list.remove(x), list.remove(y)
                int r0 = nb0, r1 = nb1, r2 = nb2, n = 3;
                if (r0 == x) { r0 = r1; r1 = r2; n = 2; }
                else if (r1 == x) { r1 = r2; n = 2; }
                else if (r2 == x) n = 2;
                else bad = true;
                if (n == 2) {
                    if (r0 == y) r0 = r1;
                    else if (r1 != y) bad = true;
                }
                z = r0;
                lx = (int)a0;
                ly = (int)a1;
            }
        }
        // ---- Space.drop_box (D:space.py:347-389) ----
        const int maxax = max(p.W, p.L);
        bool ok = !bad && lx >= 0 && ly >= 0 && lx < maxax && ly < maxax && x > 0 && y > 0;
        int max_h = 0;
        if (STAB && lane == 0) {  // CSR slot / incoming-list head of the box about to be placed
            hot->e_off[n_box0] = (uint16_t)h.n_edge;
            hot->poly_off[n_box0] = (uint16_t)h.n_poly;
            hot->first_in[n_box0 < NB_MAX ? n_box0 : 0] = EDGE_NIL;
        }
        __syncwarp();
        if (ok) {
            // resting height: warp max-reduce over the placed boxes whose footprint overlaps
            max_h = __reduce_max_sync(FULL, rest_height(hot->box, lane, n_box0, 32, lx, ly, lx + x, ly + y));
            if (lx + x > p.W || ly + y > p.L) ok = false;
            else if (max_h + z > p.H) ok = false;
            else if (STAB && max_h != 0) {
                int res = 0;
                if (lane == 0) {
                    int fl = 0;
                    GeomD g{hot->box, n_box0, p.setting == 3 ? cold->density : nullptr};
                    NodeD root{lx, ly, max_h, x, y, z, (double)(x * y * z) * next_den0};
                    if constexpr (ALIAS) {  // the reference's object semantics of the load entries (DESIGN.md section 3 (b))
                        EdgePoolA pool;
                        static_cast<EdgePool &>(pool) = EdgePool{hot->e_lower, hot->e_next, hot->e_off, hot->first_in, hot->last_in, cold->e_st, st_sm, h.n_edge,
                                                                 hot->poly_off, &cold->poly[0][0], poly_sm, h.n_poly};
                        DEnvAux *ax = p.aux + e;
                        pool.box_st = ax->box_st; pool.e_upper = ax->e_upper; pool.e_alias = ax->e_alias;
                        res = stability_check<true, GeomD, true>(g, root, pool, &cold->big, lock, n_box0, fl, nullptr, scr);
                        if (!res) alias_sync_loads(pool);
                        h.n_edge = pool.n;
                        h.n_poly = pool.n_poly;
                    } else {
                    EdgePool pool{hot->e_lower, hot->e_next, hot->e_off, hot->first_in, hot->last_in, cold->e_st, st_sm, h.n_edge,
                                  hot->poly_off, &cold->poly[0][0], poly_sm, h.n_poly};
                    res = stability_check<true, GeomD>(g, root, pool, &cold->big, lock, n_box0, fl, nullptr, scr);
                    h.n_edge = pool.n;
                    h.n_poly = pool.n_poly;
                    }
                    h.flags |= fl;
                }
                __syncwarp();
                ok = __shfl_sync(FULL, res, 0) != 0;
            }
            if (ok && n_box0 >= p.nb) {
                ok = false;
                if (lane == 0) h.flags |= PCT_FLAG_BOX_OVERFLOW;
            }
        }
        if (bad && lane == 0) h.flags |= PCT_FLAG_BAD_ACTION;
        __syncwarp();
        const double binvol = (double)(p.W * p.L * p.H);
        if (ok) {
            int16_t *b = hot->box[n_box0];
            if (lane == 0) {
                b[0] = (int16_t)lx; b[1] = (int16_t)ly; b[2] = (int16_t)max_h;
                b[3] = (int16_t)(lx + x); b[4] = (int16_t)(ly + y); b[5] = (int16_t)(max_h + z);
                if (p.setting == 3) cold->density[n_box0] = next_den0;
                h.n_box = n_box0 + 1;
                h.vol_sum += x * y * z;
                if (STAB) { hot->e_off[n_box0 + 1] = (uint16_t)h.n_edge; hot->poly_off[n_box0 + 1] = (uint16_t)h.n_poly; }
            }
            const int n_ems0 = h.n_ems;
            __syncwarp();
            int fl = 0;
            // GENEMS only runs for LNES == 'EMS' (D:bin3D.py:172-175)
            const int n_ems = p.lnes == 0 ? genems_warp(hot->ems, n_ems0, ems_tmp, ems_pk, b, p.low_bound, lane, fl) : n_ems0;
            const double rw = (double)(nb0 * nb1 * nb2) / binvol * 10;  // D:bin3D.py:180-183
            reward = (float)rw;
            info.counter = n_box0 + 1;
            info.flags = flags0 | fl;
            if (lane == 0) {
                h.n_ems = n_ems;
                h.flags |= fl;
                h.ep_len++;
                h.ep_reward += rw;
                draw_item(p, e, h);
            }
            __syncwarp();
        } else {
            // terminal step (D:bin3D.py:160-165) followed by the worker's auto-reset (shmem_vec_env.py:141-142)
            done = 1;
            info.counter = n_box0;
            info.flags = h.flags;
            info.ratio = (float)((double)h.vol_sum / binvol);
            info.ep_reward = (float)h.ep_reward;
            info.ep_len = h.ep_len + 1;
            __syncwarp();
            if (!p.no_auto_reset) reset_space(hot, p, e, lane);
        }
    }
    fence_proxy_async();
    __syncwarp();
    if (lane == 0) {
        if (p.reward) p.reward[e] = reward;
        if (p.done) p.done[e] = (uint8_t)done;
        if (p.info) p.info[e] = info;
        if (p.order) order_file(p.order, p.n_envs, e, h.n_box, h.n_ems);  // this env's slot in the next step's launches
        // record back to HBM: smem -> global via TMA bulk store
        tma_store_1d(ghot, hot, (uint32_t)sizeof(DEnvHot));
        if (STAB && p.mode == 1 && h.n_edge > 0) tma_store_1d(cold->e_st, st_sm, (uint32_t)min(h.n_edge, EDGE_STAGE) * (uint32_t)sizeof(Stack4));
        if (STAB && p.mode == 1 && h.n_poly > 0) tma_store_1d(cold->poly, poly_sm, (uint32_t)min(h.n_poly, POLY_STAGE) * 16u);
        if (p.ready) {  // overlapped mode: the record must be globally visible before the hand-over flag
            tma_store_commit_wait_all();
            fence_proxy_async_all();
            env_publish(p.ready + e, p.epoch);
        } else
            tma_store_commit_wait();
        KT_END(p.env_id_base + e - p.env_id_base0, 0);
    }
}

// ---- K2: candidate leaves -----------------------------------------------------------------------------------
template <typename SlotT, bool BIGSM>
__global__ void __launch_bounds__(32 * WARPS_PER_BLOCK) pct_candidates_kernel(const DParams p) {
    typedef Lay<SlotT, BIGSM> LY;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int slot = blockIdx.x * WARPS_PER_BLOCK + warp;
    if (slot >= p.n_envs) return;
    const int e = (p.order && p.mode == 1) ? order_lookup(p.order, p.n_envs, slot, lane) : slot;
    unsigned char *sm = smem_raw + (size_t)warp * LY::PER_WARP;
    DEnvHot *hot = (DEnvHot *)(sm + LY::HOT);
    SlotT *tabA = (SlotT *)(sm + LY::TAB_A_OFF), *tabB = (SlotT *)(sm + LY::TAB_B_OFF);
    uint64_t *mbar = (uint64_t *)(sm + LY::MISC);
    RotTab *rt = (RotTab *)(sm + LY::MISC + 16);
    SetStage *stg = (SetStage *)(sm + LY::MISC + 48);
    static_assert(sizeof(RotTab) <= 32 && sizeof(SetStage) == 384, "RotTab / SetStage slots");
    DEnvHot *ghot = p.hot + e;
    DEnvCold *cold = p.cold + e;
    KT_BEGIN();
    int sync_fl = 0;
    if (p.ready) {  // overlapped mode: wait for the apply kernel's hand-over of THIS env
        pdl_launch_dependents();
        if (lane == 0 && !env_wait(p.ready + e, p.epoch)) sync_fl = PCT_FLAG_SYNC_TIMEOUT;
        __syncwarp();
    }
    if (lane == 0) {
        mbar_init(mbar, 1);
        fence_proxy_async_all();
    }
    __syncwarp();
    if (lane == 0) {  // header + boxes + EMS list only
        mbar_expect_tx(mbar, (uint32_t)HOT_PREFIX);
        tma_load_1d(hot, ghot, (uint32_t)HOT_PREFIX, mbar);
    }
    mbar_wait(mbar, 0);
    __syncwarp();
    const DHdr &h = hot->h;
    const int nb3[3] = {h.next_box[0], h.next_box[1], h.next_box[2]};
    const int R = p.setting == 2 ? 6 : 2;
    if (lane == 0) make_rot_tab(nb3, R, *rt);
    __syncwarp();
    SlotT *cand = nullptr;
    int fl = 0, n_cand;
    SlotT *out = (SlotT *)cold->cand;
    constexpr int KB = sizeof(SlotT) == 2 ? 4 : 8;
    if (p.lnes == 0) {
        n_cand = build_candidates<SlotT>(hot->ems, h.n_ems, rt, R, tabA, tabB, BIGSM ? tabA : (SlotT *)cold->tab_big, stg, cand, lane, fl);
    } else {
        uint32_t *raw = cold->raw;
        int n_raw;
        if (p.lnes == 4) n_raw = gen_full_coord<KB>(hot->box, h.n_box, rt, R, p.W, p.L, p.H, raw, lane, fl);
        else if (p.lnes == 1) n_raw = gen_event_point<KB>(rt, R, p.W, p.L, raw, lane);
        else n_raw = gen_level_points<KB>(hot->box, h.n_box, rt, R, p.W, p.L, p.H, p.lnes == 2, raw, lane, fl);
        if (n_raw == -2) {  // empty bin under EP / CP: the reference returns a 2-element LIST (D:space.py:700-701)
            if (lane < 2) out[lane] = (SlotT)key_pack<KB>(0, 0, 0, rt->canon[lane]);
            n_cand = 2;
            cand = out;
        } else
            n_cand = build_candidates<SlotT>(hot->ems, h.n_ems, rt, R, tabA, tabB, BIGSM ? tabA : (SlotT *)cold->tab_big, stg, cand, lane, fl, raw, n_raw);
    }
    if (cand != out)
        for (int t = lane; t < n_cand; t += 32) out[t] = cand[t];
    fl |= sync_fl;
    __syncwarp();
    if (p.shuffle) {  // scratch: cold->raw + cold->tab_big (contiguous, 16 KB, free once the list is in `out`): keys at 0, permuted list at 10 KB
        static_assert(offsetof(DEnvCold, tab_big) == offsetof(DEnvCold, raw) + sizeof(uint32_t) * RAW_MAX, "raw and tab_big are contiguous");
        static_assert(CAND_MAX * 8 <= 10240 && 10240 + CAND_MAX * 4 <= (RAW_MAX + TAB_A) * 4, "shuffle scratch fits");
        shuffle_candidates<SlotT>(out, n_cand, (uint64_t *)cold->raw, (SlotT *)((char *)cold->raw + 10240), p.seed, (uint64_t)h.item_env,
                                  (uint64_t)h.draw_pos, lane);
        cand = out;
    }
    if (p.walkq) {
        // ---- classify (round 2; see "K3 (round 2)" below): drop_box_virtual (D:space.py:393-433) + check_box (:436-454), integer part ----
        constexpr bool STAB = !BIGSM;
        const int n_box = h.n_box, nl = p.nl;
        const uint32_t lt = (1u << lane) - 1;
        int pos = 0, nf = 0, n_walk = 0;
#pragma unroll 1
        while (pos < n_cand && nf < nl) {
            const int c = pos + lane;
            bool feas = false, pend = false;
            int mh = 0, k = 0, xs = 0, ys = 0, zs = 0, rot = 0, sx = 0, sy = 0, sz = 0;
            uint32_t pack = 0;
            if (c < n_cand) {
                key_unpack<KB>((uint32_t)cand[c], xs, ys, zs, rot);
                sx = rt->d[rot][0]; sy = rt->d[rot][1]; sz = rt->d[rot][2];
                bool far_out = false;
                if (STAB) mh = rest_height_supports(hot->box, n_box, xs, ys, xs + sx, ys + sy, k, pack, far_out);
                else mh = rest_height(hot->box, 0, n_box, 1, xs, ys, xs + sx, ys + sy);
                if (xs + sx > p.W || ys + sy > p.L) feas = false;
                else if (mh + sz > p.H) feas = false;
                else if (!STAB || mh == 0) feas = true;
                else pend = !far_out;  // far_out: the centre is outside the supports' bounding box -> the root test fails (rest_height_supports)
            }
            const uint32_t fm = __ballot_sync(FULL, feas), pm = __ballot_sync(FULL, pend);
            if (lane == 0) cold->fbits[pos >> 5] = fm;
            nf += __popc(fm);
            n_walk += __popc(pm);
            if (pm) {
                int qb = 0;
                if (lane == 0) qb = atomicAdd(p.walk_ctr, __popc(pm));
                qb = __shfl_sync(FULL, qb, 0);
                if (pend) {
                    WalkItem it;
                    it.env = (uint32_t)e; it.pack = pack; it.c = (uint16_t)c;
                    it.xs = (uint8_t)xs; it.ys = (uint8_t)ys; it.mh = (uint8_t)mh; it.sx = (uint8_t)sx; it.sy = (uint8_t)sy; it.sz = (uint8_t)sz;
                    it.k = (uint8_t)min(k, 255); it.pad_ = 0;
                    p.walkq[qb + __popc(pm & lt)] = it;
                }
            }
            pos += 32;
        }
        if (lane == 0) { cold->n_fw = pos >> 5; cold->n_pending = n_walk; }
        // cur_observation, part 1 (D:bin3D.py:70-93): internal-node rows + item row are final since the apply kernel
        if (p.obs) {
            const bool delta = (p.opt & PCT_OPT_DELTA) != 0;
            if (p.obs_f64) { if (delta) write_obs_delta<double, true, 1>(p, e, hot, cold, nullptr, 0, lane, 32); else write_obs<double, 1>(p, e, hot, cold, nullptr, 0, lane, 32); }
            else { if (delta) write_obs_delta<float, true, 1>(p, e, hot, cold, nullptr, 0, lane, 32); else write_obs<float, 1>(p, e, hot, cold, nullptr, 0, lane, 32); }
        }
    }
    if (lane == 0) {
        ghot->h.n_cand = n_cand;
        if (fl) ghot->h.flags = h.flags | fl;
        if (p.ready) env_publish(p.ready + p.n_envs + e, p.epoch);
        KT_END(p.env_id_base + e - p.env_id_base0, 1);
    }
}

// ---- K3: feasibility (thread per candidate) + leaf compaction + observation ------------------------------------
#ifndef FEAS_WARPS_N
#define FEAS_WARPS_N 2
#endif
constexpr int FEAS_WARPS = FEAS_WARPS_N;
constexpr int FEAS_THREADS = 32 * FEAS_WARPS;
constexpr int K3_SMEM = sizeof(DEnvHot) + NL_MAX * 12 + 64 + EDGE_STAGE * 32 + POLY_STAGE * 16;

template <typename OT, bool STAB, typename SlotT, bool DELTA = false>
__global__ void __launch_bounds__(FEAS_THREADS, K3_MINB) pct_feas_emit_kernel(const DParams p) {
    constexpr int BITS = sizeof(SlotT) == 2 ? 4 : 8;
    __shared__ __align__(16) unsigned char sm[K3_SMEM];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int e = blockIdx.x;  // (round 1's heaviest-first permutation of this kernel went with the sorting pass; the legacy mode runs in env order)
    DEnvHot *hot = (DEnvHot *)sm;
    int16_t (*leaf)[6] = (int16_t (*)[6])(sm + sizeof(DEnvHot));
    uint64_t *mbar = (uint64_t *)(sm + sizeof(DEnvHot) + NL_MAX * 12);
    int *lock = (int *)(mbar + 1);
    uint32_t *wb = (uint32_t *)(mbar + 2);             // per-warp feasibility ballots of the current pass
    RotTab *rt = (RotTab *)(sm + sizeof(DEnvHot) + NL_MAX * 12 + 32);
    Stack4 *st_sm = (Stack4 *)(sm + sizeof(DEnvHot) + NL_MAX * 12 + 64);
    double *poly_sm = (double *)(st_sm + EDGE_STAGE);
    DEnvHot *ghot = p.hot + e;
    DEnvCold *cold = p.cold + e;
    KT_BEGIN();
    if (tid == 0) {
        *lock = 0;
        mbar_init(mbar, 1);
        fence_proxy_async();
    }
    __syncthreads();
    if (tid == 0) {
        if (p.ready) {  // overlapped mode: wait for the candidates kernel's hand-over of THIS env
            if (!env_wait(p.ready + p.n_envs + e, p.epoch)) atomicOr(&ghot->h.flags, PCT_FLAG_SYNC_TIMEOUT);
            fence_proxy_async_all();
        }
        mbar_expect_tx(mbar, (uint32_t)sizeof(DEnvHot));
        tma_load_1d(hot, ghot, (uint32_t)sizeof(DEnvHot), mbar);
    }
    mbar_wait(mbar, 0);
    __syncthreads();  // every thread must have observed phase 0 before the barrier is re-armed
    const DHdr &h = hot->h;
    if (STAB && h.n_edge > 0) {  // stage the load edges (second phase of the same mbarrier)
        const uint32_t bytes = (uint32_t)min(h.n_edge, EDGE_STAGE) * (uint32_t)sizeof(Stack4);
        const uint32_t pbytes = (uint32_t)min(h.n_poly, POLY_STAGE) * 16u;
        if (tid == 0) {
            mbar_expect_tx(mbar, bytes + pbytes);
            tma_load_1d(st_sm, cold->e_st, bytes, mbar);
            if (pbytes) tma_load_1d(poly_sm, cold->poly, pbytes, mbar);
        }
        mbar_wait(mbar, 1);
    }
    const int nb3[3] = {h.next_box[0], h.next_box[1], h.next_box[2]};
    if (tid == 0) make_rot_tab(nb3, p.setting == 2 ? 6 : 2, *rt);
    __syncthreads();
    const int n_cand = h.n_cand, n_box = h.n_box;
    const double den = h.next_den;
    const SlotT *cand = (const SlotT *)cold->cand;
    GeomD g{hot->box, n_box, p.setting == 3 ? cold->density : nullptr};
    EdgePool pool{hot->e_lower, hot->e_next, hot->e_off, hot->first_in, hot->last_in, cold->e_st, st_sm, h.n_edge,
                  hot->poly_off, &cold->poly[0][0], poly_sm, h.n_poly};
    int n_leaf = 0, fl = 0;
    // ---------------- get_possible_position (D:bin3D.py:100-136): first `nl` feasible candidates in order ----------------
#pragma unroll 1
    for (int base = 0; base < n_cand && n_leaf < p.nl; base += FEAS_THREADS) {
        const int c = base + tid;
        bool feas = false;
        int xs = 0, ys = 0, zs = 0, rot = 0, sx = 0, sy = 0, sz = 0;
        if (c < n_cand) {
            key_unpack<BITS>(cand[c], xs, ys, zs, rot);
            sx = rt->d[rot][0]; sy = rt->d[rot][1]; sz = rt->d[rot][2];
            // drop_box_virtual (D:space.py:393-433) + check_box (:436-454)
            const int mh = rest_height(hot->box, 0, n_box, 1, xs, ys, xs + sx, ys + sy);
            if (xs + sx > p.W || ys + sy > p.L) feas = false;
            else if (mh + sz > p.H) feas = false;
            else if (!STAB || mh == 0) feas = true;
            else {
                NodeD root{xs, ys, mh, sx, sy, sz, (double)(sx * sy * sz) * den};
#ifdef PCT_PHASE_TIMERS
                const long long c0 = clock64();
                int fl2 = 0;
                long long prof[6];
                feas = stability_check<false, GeomD>(g, root, pool, &cold->big, lock, 0, fl2, prof) != 0;
                const long long dc = clock64() - c0;
                fl |= fl2 & 0xFFFF;
                if (p.mode == 1 && p.dbg) {
                    unsigned long long packed = ((unsigned long long)dc << 24) | ((unsigned long long)((fl2 >> 16) & 0xFF) << 8) | (unsigned long long)((fl2 >> 24) & 0xFF);
                    long long *slot = &p.dbg[(size_t)(p.env_id_base + e - p.env_id_base0) * 16];
                    if (atomicMax((unsigned long long *)&slot[12], packed) < packed)
                        { slot[3] = prof[0]; slot[7] = prof[1]; slot[11] = prof[2]; slot[13] = prof[3]; slot[14] = prof[4]; }
                }
#else
                feas = stability_check<false, GeomD>(g, root, pool, &cold->big, lock, 0, fl) != 0;
#endif
            }
        }
        const uint32_t fm = __ballot_sync(FULL, feas);
        if (lane == 0) wb[warp] = fm;
        __syncthreads();
        int before = 0, total = 0;
#pragma unroll
        for (int w = 0; w < FEAS_WARPS; w++) {
            const int cnt = __popc(wb[w]);
            if (w < warp) before += cnt;
            total += cnt;
        }
        if (feas) {
            const int k = n_leaf + before + __popc(fm & ((1u << lane) - 1));
            if (k < p.nl) {
                leaf[k][0] = (int16_t)xs; leaf[k][1] = (int16_t)ys; leaf[k][2] = (int16_t)zs;
                leaf[k][3] = (int16_t)(xs + sx); leaf[k][4] = (int16_t)(ys + sy); leaf[k][5] = (int16_t)(zs + sz);
            }
        }
        n_leaf += total;
        __syncthreads();
    }
    if (n_leaf > p.nl) n_leaf = p.nl;
    fl = __reduce_or_sync(FULL, fl);
    if (fl && lane == 0) atomicOr(&ghot->h.flags, fl);
    __syncthreads();
    // persist the emitted leaves for the leaf-index action path; header / info
    for (int t = tid; t < n_leaf * 6; t += FEAS_THREADS) ((int16_t *)cold->leaf)[t] = ((int16_t *)leaf)[t];
    if (tid == 0) {
        ghot->h.n_leaf = n_leaf;
        if (p.info) {
            p.info[e].n_leaf = n_leaf;
            p.info[e].n_cand = n_cand;
            p.info[e].n_ems = h.n_ems;
            p.info[e].flags |= h.flags;
        }
    }
    // ---------------- cur_observation (D:bin3D.py:70-93) ----------------
    if constexpr (DELTA) write_obs_delta<OT>(p, e, hot, cold, leaf, n_leaf, tid, FEAS_THREADS);
    else write_obs<OT>(p, e, hot, cold, leaf, n_leaf, tid, FEAS_THREADS);
    if (tid == 0) KT_END(p.env_id_base + e - p.env_id_base0, 2);
}

// ---- K3 (round 2): pooled stability walks + emit ---------------------------------------------------------------------
// ncu of the kernel above at round 1's HEAD (profiles/r2_k3_head_*.txt) and of a warp-per-env variant (profiles/r2_k3_warp_per_env.txt):
// the launch lasts 2x the SMs' mean active time — it ends when the env with the most and deepest stability walks ends (a serial chain
// inside one block) —, 60 % of the warp instructions sit in the walk at 2-5 active lanes, every candidate scans the boxes twice, and capping
// registers for occupancy only trades stalls for spills.  Round 2 cuts the work by KIND instead of by env:
//   classify  (end of K2, warp per env, integer only) bounds + ONE pass over the boxes for resting height, supports and the exact
//             quick reject (rest_height_supports) -> infeasible / feasible / needs a stability walk; feasibility bits per 32-candidate
//             chunk; the walks of ALL envs go into one global pool;
//   walk      two kernels over the pool, 32 walks per warp from whichever envs (a heavy env's walks spread over many warps and SMs):
//             pct_walk_light_kernel runs every walk's LIGHT PREFIX (stab_light: visits of nodes with <= 1 support; 81 % of the walks are
//             nothing else) and hands the rest — walks standing in front of a node with >= 2 supports, with (node, stack) — to
//             pct_walk_kernel, whose lanes therefore all START with a heavy visit (dense) and finish through stab_virtual;
//   emit      pct_emit_kernel (warp per env): the first `nl` set feasibility bits in candidate order -> leaf slots, observation.
// get_possible_position stops at `nl` feasible candidates (D:bin3D.py:117-136); here classification stops once `nl` candidates are KNOWN
// feasible and the emit kernel takes the first `nl` set bits: the same ordered prefix (walks past the cut are wasted work, not wrong).
#ifndef WALK_MINB
#define WALK_MINB 8
#endif
#ifndef LIGHT_MINB
#define LIGHT_MINB 6
#endif
constexpr int WALK_WARPS = 2, LIGHT_WARPS = 4;

// a walk of this env has delivered its verdict (fbits / flags written before): release-decrement the env's counter of running walks
__device__ __forceinline__ void walk_done(int32_t *n_pending) {
    __threadfence();
    atomicSub(n_pending, 1);
}

// per-lane view of one pooled walk: the env's record stays in global memory (L1 / L2) — the lanes of a warp belong to different envs
struct WalkView {
    GeomD g;
    EdgePool pool;
    NodeD root;
    DEnvCold *cold;
    const DEnvHot *hot;
};
__device__ __forceinline__ WalkView walk_view(const DParams &p, const WalkItem &it, bool has) {
    const DEnvHot *hot = p.hot + it.env;
    DEnvCold *cold = p.cold + it.env;
    const DHdr &h = hot->h;
    const int sx = it.sx, sy = it.sy, sz = it.sz;
    return WalkView{GeomD{hot->box, has ? h.n_box : 0, p.setting == 3 ? cold->density : nullptr},
                    EdgePool{const_cast<uint8_t *>(hot->e_lower), const_cast<uint8_t *>(hot->e_next), const_cast<uint16_t *>(hot->e_off),
                             const_cast<uint8_t *>(hot->first_in), const_cast<uint8_t *>(hot->last_in), cold->e_st, cold->e_st, has ? h.n_edge : 0,
                             const_cast<uint16_t *>(hot->poly_off), &cold->poly[0][0], &cold->poly[0][0], has ? h.n_poly : 0},
                    NodeD{(int)it.xs, (int)it.ys, (int)it.mh, sx, sy, sz, (double)(sx * sy * sz) * (has ? h.next_den : 1.0)}, cold, hot};
}

// walk, stage 1: the light prefix of EVERY pooled walk, one lane per walk (stab_light: single-support visits only — small code, no local arrays).
// 81 % of the walks end here; the rest goes to the continuation pool with (node, stack).
__global__ void __launch_bounds__(32 * LIGHT_WARPS, LIGHT_MINB) pct_walk_light_kernel(const DParams p) {
    const int lane = threadIdx.x & 31;
    const int total = *(volatile const int32_t *)p.walk_ctr;
    const int nwarps = gridDim.x * LIGHT_WARPS;
    const int cap = p.n_envs * WALK_CONT_PER_ENV;
#pragma unroll 1
    for (int base = (blockIdx.x * LIGHT_WARPS + (threadIdx.x >> 5)) * 32; base < total; base += nwarps * 32) {
        const int i = base + lane;
        const bool has = i < total;
        WalkItem it{};
        if (has) it = p.walkq[i];
        const WalkView v = walk_view(p, it, has);
        int node = NODE_NEW, res = 0;
        Stack4 st{};
        if (has) res = stab_light<GeomD>(v.g, v.root, (int)it.k, it.pack, v.pool, node, st);
        if (res == 1) atomicOr(&v.cold->fbits[it.c >> 5], 1u << (it.c & 31));
        if (has && res != 2) walk_done(&v.cold->n_pending);
        // continuations: walks high up in the bin descend through the deepest support DAGs (host statistics: resting height >= 0.6 H -> up to 8 heavy
        // visits, below -> at most 2), so they are pooled apart (from the END of the pool) and get fewer lanes per warp in pct_walk_kernel
        if (p.walk_fork) {  // fork-join continuation kernel: one queue of pieces, "enter `node` with the stack st" (pct_walkq.cuh)
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
                    } else {  // never silent: the candidate stays infeasible and the env is flagged
                        atomicOr(const_cast<int32_t *>(&v.hot->h.flags), PCT_FLAG_CAND_OVERFLOW);
                        walk_done(&v.cold->n_pending);
                        pq_piece_done(pq);
                    }
                }
            }
            continue;
        }
        const bool tall = (int)it.mh * 5 >= p.H * 3;
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
                const int idx = tall ? qt + __popc(pt & lt) : qs + __popc(ps & lt);  // each class owns half of the pool (the counters may overshoot; the consumer clamps)
                if (idx < cap / 2) p.contq[tall ? cap - 1 - idx : idx] = WalkCont{(uint32_t)i, (uint32_t)node, st};
                else { atomicOr(const_cast<int32_t *>(&v.hot->h.flags), PCT_FLAG_CAND_OVERFLOW); walk_done(&v.cold->n_pending); }  // never silent: the candidate stays infeasible and the env is flagged
            }
        }
    }
}

// walk, stage 2: the continuations — every lane starts with the heavy visit its walk stopped at, then runs the general light / heavy state
// machine to the end of the walk.  Only `p.walk_lanes` lanes of a warp carry a walk (default 16; 4 for the walks resting at >= 0.6 H): there are few
// continuations (3 per env) and each is a long serial chain; a full warp of them (ncu r2, profiles/r2_walk_two_stage_32lanes.txt: 400 warps on 592
// schedulers, 20 k instructions per warp, 116 us) leaves too few warps, 4-8 per warp multiply the warp instructions (measured sweep: DESIGN.md 5d).
__global__ void __launch_bounds__(32 * WALK_WARPS, WALK_MINB) pct_walk_kernel(const DParams p) {
    const int lane = threadIdx.x & 31;
    const int cap = p.n_envs * WALK_CONT_PER_ENV;
    const int n_short = min(*(volatile const int32_t *)p.cont_ctr, cap / 2), n_tall = min(*(volatile const int32_t *)(p.cont_ctr + 1), cap / 2);
    __syncthreads();
    pdl_launch_dependents();  // the emit kernel's blocks may become resident now (it also empties the pool counters: read above); each waits for ITS env's last walk
    const int nwarps = gridDim.x * WALK_WARPS, Ls = p.walk_lanes, Lt = p.walk_lanes_tall;
    const int w_tall = (n_tall + Lt - 1) / Lt, w_all = w_tall + (n_short + Ls - 1) / Ls;
#pragma unroll 1
    for (int w = blockIdx.x * WALK_WARPS + (threadIdx.x >> 5); w < w_all; w += nwarps) {  // the tall walks (longest chains) are dealt first
        const bool tw = w < w_tall;
        const int L = tw ? Lt : Ls;
        const unsigned mask = L >= 32 ? FULL : ((1u << L) - 1u);
        if (lane >= L) continue;
        const int i = tw ? w * Lt + lane : (w - w_tall) * Ls + lane;
        const bool has = i < (tw ? n_tall : n_short);
        WalkCont ct{};
        WalkItem it{};
        if (has) { ct = p.contq[tw ? cap - 1 - i : i]; it = p.walkq[ct.item]; }
        const WalkView v = walk_view(p, it, has);
        int fl = 0;
        const bool ok = stab_virtual<GeomD>(v.g, v.root, (int)it.k, it.pack, v.pool, &v.cold->big, &v.cold->lock, fl, has, mask,
                                            has ? (int)ct.node : NODE_NEW, &ct.st) != 0;
        if (has && ok) atomicOr(&v.cold->fbits[it.c >> 5], 1u << (it.c & 31));
        if (has && fl) atomicOr(const_cast<int32_t *>(&v.hot->h.flags), fl);
        if (has) walk_done(&v.cold->n_pending);
    }
}

// walk, stage 2, fork-join form (opt-in, PCT_B200_WALK=fork): the queue holds PIECES of walks (stab_piece: one chain of visits; a node with k >= 2 supports keeps
// its first subtree and publishes the other k - 1 as new pieces; protocol: pct_walkq.cuh).  A walk's verdict is the AND over its pieces:
// walk_pend[item] counts them, the piece that brings it to zero sets the feasibility bit (unless one failed) and releases the env's n_pending.
// The critical chain of a step's longest walk becomes its longest root-to-floor PATH instead of the sum over its visits (host statistics,
// scratch/stats_paths.py: 51 -> 34 visit units at the 99.99 % quantile) — and the stage does not get faster (B200, 4096 envs: walk + emit group 0.180 ms
// against 0.171 ms, whatever the number of helper warps, blocks per SM or pieces per warp): the continuation stage is bound by the issue rate of a few
// hundred divergent, latency-bound warps (warp instructions = thread instructions / 4.8 lanes, ~10 cycles each), not by its longest walk.  Kept as an
// opt-in because it is the measured answer to "would independent subtrees on separate lanes help?" and is parity-tested (tests/test_gpu_walk_fork.py).
struct PieceFork {
    PieceQueue pq;
    int32_t *pend;
    uint32_t item;
    int n_init;
    bool overflow;
    __device__ __forceinline__ void operator()(int child, int skip, double vx, double vy, double vm) {
        if (!pq_fork(pq, n_init, pend, WalkPiece{item, (uint8_t)child, (uint8_t)skip, 1, 0, vx, vy, vm})) overflow = true;
    }
};
// one piece: the chain of visits, then the walk's AND-reduction (walk_pend) and the queue's bookkeeping
__device__ __forceinline__ void run_piece(const DParams &p, const PieceQueue &pq, int n_init, int slot) {
    const WalkPiece pc = pq.q[slot];
    if (slot >= n_init) pq.ready[slot] = 0;
    const WalkItem it = p.walkq[pc.item];
    const WalkView v = walk_view(p, it, true);
    int32_t *pend = p.walk_pend + pc.item;
    int fl = 0, ok = 0;
    if (!(*(volatile const int32_t *)pend & WALK_FAILED)) {  // a failed sibling has already decided the walk
        PieceFork fork{pq, pend, pc.item, n_init, false};
        ok = stab_piece<GeomD>(v.g, v.root, (int)it.k, it.pack, v.pool, &v.cold->big, &v.cold->lock, fl, (int)pc.node, (int)pc.kind, (int)pc.skip,
                               pc.a, pc.b, pc.c, fork);
        if (fork.overflow) { fl |= PCT_FLAG_CAND_OVERFLOW; ok = 0; }  // never silent: the candidate stays infeasible and the env is flagged
    }
    if (fl) atomicOr(const_cast<int32_t *>(&v.hot->h.flags), fl);
    if (!ok) atomicOr(pend, WALK_FAILED);
    __threadfence();
    const int r = atomicSub(pend, 1);
    if ((r & (WALK_FAILED - 1)) == 1) {  // the walk's last piece
        if (!(r & WALK_FAILED)) atomicOr(&v.cold->fbits[it.c >> 5], 1u << (it.c & 31));
        walk_done(&v.cold->n_pending);
    }
    pq_piece_done(pq);
}
__global__ void __launch_bounds__(32 * WALK_WARPS, WALK_MINB) pct_walk_fork_kernel(const DParams p) {
    const int lane = threadIdx.x & 31;
    const int wid = blockIdx.x * WALK_WARPS + (threadIdx.x >> 5), n_warps = gridDim.x * WALK_WARPS;
    const PieceQueue pq{(WalkPiece *)p.contq, p.piece_ready, p.cont_ctr, p.piece_cap};
    const int n_init = min(*(volatile const int32_t *)(pq.ctr + PQ_NINIT), pq.cap);  // written by the light-prefix kernel only (completed)
    const int L = p.walk_lanes;
    pdl_launch_dependents();  // the emit kernel's blocks may become resident; each waits for ITS env's last walk
    if (n_init > 0) {
        // the light-prefix kernel's pieces: dealt statically
#pragma unroll 1
        for (int b = wid * L; b < n_init; b += n_warps * L) {
            if (lane < L && b + lane < n_init) run_piece(p, pq, n_init, b + lane);
            __syncwarp();
        }
        // forked pieces: tickets
        const bool keep = wid < p.walk_keep;
#pragma unroll 1
        for (;;) {
            int t0 = -1;
            if (lane == 0 && (keep || *(volatile const int32_t *)(pq.ctr + PQ_ALLOC) - *(volatile const int32_t *)(pq.ctr + PQ_HEAD) > 0))
                t0 = atomicAdd(pq.ctr + PQ_HEAD, L);
            t0 = __shfl_sync(FULL, t0, 0);
            if (t0 < 0) break;  // not a helper and nothing unclaimed in the queue: leave (SM slots for the emit kernel)
            bool fin = false;
            if (lane < L) {
                const int slot = n_init + t0 + lane;
                if (pq_wait(pq, slot)) run_piece(p, pq, n_init, slot);
                else fin = true;
            }
            __syncwarp();
            if (__any_sync(FULL, fin)) break;  // a lane saw the end of all work
        }
    }
    if (lane == 0) pq_warp_exit(pq, n_warps, p.walk_ctr);
}

constexpr int EMIT_WARPS = 4;
constexpr int EMIT_STAGE = sizeof(DHdr) + NB_MAX * 12;  // header + placed boxes: all the observation needs from the hot record
constexpr int EMIT_SM_PER_WARP = EMIT_STAGE + NL_MAX * 12 + 48;
static_assert(EMIT_STAGE % 16 == 0 && EMIT_SM_PER_WARP % 16 == 0, "TMA bulk copies move multiples of 16 bytes");

template <typename OT, typename SlotT, bool DELTA>
__global__ void __launch_bounds__(32 * EMIT_WARPS) pct_emit_kernel(const DParams p) {
    constexpr int BITS = sizeof(SlotT) == 2 ? 4 : 8;
    __shared__ __align__(16) unsigned char smem[EMIT_WARPS * EMIT_SM_PER_WARP];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int e = blockIdx.x * EMIT_WARPS + warp;
    // last kernel of the launch sequence that touches the walk pools (both walk kernels have completed: plain stream order): empty them for the next step
    if (blockIdx.x == 0 && threadIdx.x == 0 && p.walk_ctr && !p.walk_fork) { *p.walk_ctr = 0; p.cont_ctr[0] = 0; p.cont_ctr[1] = 0; }  // (the fork-join kernel's counters are live while this kernel starts: its last warp empties them)
    if (blockIdx.x == 0 && p.order) {
        // ... and the last one of the step: the apply and candidates kernels have consumed this parity's buckets (both completed before the walk kernels
        // started) and the apply kernel has filled the other parity's; empty the consumed ones and flip
        const int par = *(volatile const int32_t *)p.order & 1;
        if (threadIdx.x < ORD_BUCKETS) p.order[ORD_CNT + ORD_BUCKETS * par + threadIdx.x] = 0;
        __syncthreads();
        if (threadIdx.x == 0) { __threadfence(); *(volatile int32_t *)p.order = par ^ 1; }
    }
    if (e >= p.n_envs) return;
    unsigned char *sm = smem + warp * EMIT_SM_PER_WARP;
    DEnvHot *hot = (DEnvHot *)sm;  // only the header and the boxes are staged
    int16_t (*leaf)[6] = (int16_t (*)[6])(sm + EMIT_STAGE);
    uint64_t *mbar = (uint64_t *)(sm + EMIT_STAGE + NL_MAX * 12);
    RotTab *rt = (RotTab *)(sm + EMIT_STAGE + NL_MAX * 12 + 16);
    DEnvHot *ghot = p.hot + e;
    DEnvCold *cold = p.cold + e;
    const uint32_t lt = (1u << lane) - 1;
    if (lane == 0) {
        mbar_init(mbar, 1);
        fence_proxy_async();
        // launched as a programmatic dependent of the continuation kernel: this block may run while walks are still in flight.  The classification
        // (a fully completed kernel) set n_pending; the walk kernels release-decrement it after their last write of this env.
        int spins = 0;
        while (*(volatile const int32_t *)&cold->n_pending > 0) {
            __nanosleep(spins < 16 ? 100 : 1000);
            if (++spins > (1 << 22)) { atomicOr(&ghot->h.flags, PCT_FLAG_SYNC_TIMEOUT); break; }
        }
        __threadfence();
        fence_proxy_async_all();
    }
    __syncwarp();
    if (lane == 0) {
        mbar_expect_tx(mbar, (uint32_t)EMIT_STAGE);
        tma_load_1d(hot, ghot, (uint32_t)EMIT_STAGE, mbar);
    }
    mbar_wait(mbar, 0);
    __syncwarp();
    const DHdr &h = hot->h;
    const int nb3[3] = {h.next_box[0], h.next_box[1], h.next_box[2]};
    if (lane == 0) make_rot_tab(nb3, p.setting == 2 ? 6 : 2, *rt);
    __syncwarp();
    const int nl = p.nl, nw = cold->n_fw;
    const SlotT *cand = (const SlotT *)cold->cand;
    // ---------------- leaves = the first `nl` feasible candidates in order ----------------
    int base = 0;
#pragma unroll 1
    for (int w = 0; w < nw && base < nl; w++) {
        const uint32_t bits = cold->fbits[w];
        if ((bits >> lane) & 1u) {
            const int kk = base + __popc(bits & lt);
            if (kk < nl) {
                int xs, ys, zs, rot;
                key_unpack<BITS>(cand[w * 32 + lane], xs, ys, zs, rot);
                leaf[kk][0] = (int16_t)xs; leaf[kk][1] = (int16_t)ys; leaf[kk][2] = (int16_t)zs;
                leaf[kk][3] = (int16_t)(xs + rt->d[rot][0]); leaf[kk][4] = (int16_t)(ys + rt->d[rot][1]); leaf[kk][5] = (int16_t)(zs + rt->d[rot][2]);
            }
        }
        base += __popc(bits);
    }
    const int n_leaf = min(base, nl);
    __syncwarp();
    // persist the emitted leaves for the leaf-index action path; header / info
    for (int t = lane; t < n_leaf * 6; t += 32) ((int16_t *)cold->leaf)[t] = ((int16_t *)leaf)[t];
    if (lane == 0) {
        ghot->h.n_leaf = n_leaf;
        if (p.info) {
            p.info[e].n_leaf = n_leaf;
            p.info[e].n_cand = h.n_cand;
            p.info[e].n_ems = h.n_ems;
            p.info[e].flags |= h.flags;
        }
    }
    // ---------------- cur_observation (D:bin3D.py:70-93) ----------------
    if constexpr (DELTA) write_obs_delta<OT, true, 2>(p, e, hot, cold, leaf, n_leaf, lane, 32);  // leaf rows: the rest was written by the candidates kernel
    else write_obs<OT, 2>(p, e, hot, cold, leaf, n_leaf, lane, 32);
}

// uniform-random valid-leaf policy (SURVEY.md §8(d)): reads only the record headers
__global__ void pct_policy_random_kernel(const DEnvHot *hot, int n_envs, int64_t env_id_base, uint64_t seed, int64_t t, const int64_t *t_dev,
                                         int32_t *leaf_idx) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_envs) return;
    if (t_dev) t = *t_dev;
    const int n = hot[e].h.n_leaf;
    leaf_idx[e] = n > 0 ? (int32_t)(rnd_u64(seed, (uint64_t)(env_id_base + e), (uint64_t)t) % (uint64_t)n) : 0;
}

__global__ void pct_fill_prev_kernel(DEnvAux *aux, int n, int nb, int nl) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { aux[i].obs_prev[0] = nb; aux[i].obs_prev[1] = nl; }
}
void launch_fill_prev(DEnvAux *aux, int n_envs, int nb, int nl, cudaStream_t st) {
    pct_fill_prev_kernel<<<(n_envs + 255) / 256, 256, 0, st>>>(aux, n_envs, nb, nl);
}

// ---- saved env records (pct_save_envs / pct_load_envs) ------------------------------------------------------------------------------------
// What stays live between two calls, read off the kernels above (everything else is per-step scratch, rebuilt by the next step before it is read):
//   DEnvHot              whole (3.5 KB): header (counts, item source position + item_env, episode sums, flags, next item), boxes, EMS list,
//                        load-edge topology (e_off / e_lower / e_next / first_in / last_in / poly_off)
//   DEnvCold::leaf       [0, n_leaf)   leaves of the last observation (leaf-index actions, observation on load)
//   DEnvCold::density    [0, n_box)    per placed box (setting 3)
//   DEnvCold::e_st       [0, n_edge)   loads of the edge pool (stability settings)
//   DEnvCold::poly       [0, n_poly)   support-polygon vertices
//   DEnvAux::box_st      [0, n_box]    ALIAS handles only (PCT_B200_ALIAS=0 handles never write it); entry n_box is the stack of the last placement
//                                      attempt, rewritten by the next one before it is read — saved anyway, it costs 32 bytes
//   DEnvAux::e_upper     [0, n_edge), DEnvAux::e_alias (32 bytes)   ALIAS handles only
//   LSAH footprint       4 int32 (pct_heuristic_actions)
// Not saved: cand / raw / tab_big (written by K2 before K3 / emit read them), fbits / n_fw (written by K2's classification, read by the walk
// and emit kernels of the same step), big (per-descent scratch), lock / n_pending (zeroed on load; both are zero between calls), obs_prev
// (set to "every row" on load).  No kernel reads an array beyond its count: after an auto-reset every array still holds the previous episode.
struct alignas(16) DRec {
    RecHdr s;
    DEnvHot hot;
    int16_t leaf[NL_MAX][6];
    double density[NB_MAX];
    Stack4 e_st[EDGE_MAX + 1];
    double poly[POLY_MAX][2];
    Stack4 box_st[NB_MAX + 1];
    uint8_t e_upper[EDGE_MAX + 1];
    uint32_t e_alias[(EDGE_MAX + 32) / 32];
    int32_t hstate[4];
};
static_assert(offsetof(DEnvCold, leaf) % 16 == 0 && offsetof(DEnvCold, density) % 16 == 0 && offsetof(DEnvCold, e_st) % 16 == 0 &&
              offsetof(DEnvCold, poly) % 16 == 0 && sizeof(DEnvCold) % 16 == 0, "cold arrays are copied in 16-byte units");
static_assert(offsetof(DEnvAux, e_upper) % 8 == 0 && sizeof(DEnvAux) % 8 == 0 && sizeof(DEnvAux::e_alias) == 32, "aux arrays are copied in 8-byte units");
static_assert(offsetof(DRec, leaf) % 16 == 0 && offsetof(DRec, density) % 16 == 0 && offsetof(DRec, e_st) % 16 == 0 && offsetof(DRec, poly) % 16 == 0 &&
              offsetof(DRec, box_st) % 16 == 0 && offsetof(DRec, e_upper) % 16 == 0 && offsetof(DRec, hstate) % 16 == 0, "record layout");
int64_t discrete_record_bytes() { return (int64_t)sizeof(DRec); }

// One warp per record.  Counts come from the source's header (clamped to the capacities).
template <bool LOAD, typename OT>
__global__ void __launch_bounds__(128, 4) pct_env_record_kernel(const DParams p, const RecArgs s) {
    const int lane = threadIdx.x & 31, i = blockIdx.x * 4 + (threadIdx.x >> 5);
    if (i >= s.n) return;
    const int e = s.ids ? s.ids[i] : i;
    DRec *r = (DRec *)(s.rec + (size_t)i * (size_t)s.rec_bytes);
    if (e < 0 || e >= p.n_envs) {
        if (LOAD) { if (lane == 0 && s.status) s.status[i] = REC_BAD_ENV; }
        else if (lane == 0) { RecHdr z{}; z.magic = REC_MAGIC; z.version = REC_VERSION; r->s = z; }  // valid = 0
        return;
    }
    DEnvHot *hot = p.hot + e;
    DEnvCold *cold = p.cold + e;
    DEnvAux *aux = p.aux ? p.aux + e : nullptr;
    const DHdr &src = LOAD ? r->hot.h : hot->h;
    if (LOAD) {
        int st = 0;
        if (lane == 0) st = rec_check(r->s, PCT_DISCRETE, src.item_env, s, p.env_id_base, p.n_envs);
        st = __shfl_sync(FULL, st, 0);
        if (lane == 0 && s.status) s.status[i] = st;
        if (st) return;  // a rejected record leaves its env untouched
    } else if (lane == 0) {
        RecHdr z{};
        z.magic = REC_MAGIC; z.version = REC_VERSION; z.domain = PCT_DISCRETE; z.valid = 1; z.fingerprint = s.fingerprint;
        const int64_t row = src.item_env - p.env_id_base;
        z.row_hash = (s.row_hash && row >= 0 && row < p.n_envs) ? s.row_hash[row] : 0;
        r->s = z;
    }
    const int n_box = min(max(src.n_box, 0), NB_MAX), n_leaf = min(max(src.n_leaf, 0), NL_MAX);
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
    cp(&r->hot, hot, (int)sizeof(DEnvHot));
    cp(r->leaf, cold->leaf, n_leaf * 12);
    cp(r->density, cold->density, n_box * 8);
    cp(r->e_st, cold->e_st, n_edge * (int)sizeof(Stack4));
    cp(r->poly, cold->poly, n_poly * 16);
    if (s.alias) {
        cp8(r->box_st, aux->box_st, min(n_box + 1, NB_MAX + 1) * (int)sizeof(Stack4));
        cp8(r->e_upper, aux->e_upper, n_edge);
        if (lane < (EDGE_MAX + 32) / 32) { if (LOAD) aux->e_alias[lane] = r->e_alias[lane]; else r->e_alias[lane] = aux->e_alias[lane]; }
    }
    if (lane == 0) {
        uint4 *hs = (uint4 *)((int32_t *)s.hstate + (size_t)e * 4);
        if (LOAD) *hs = *(const uint4 *)r->hstate; else *(uint4 *)r->hstate = *hs;
    }
    if (LOAD) {
        if (lane == 0) { cold->lock = 0; cold->n_pending = 0; }
        if (aux && lane == 0) { aux->obs_prev[0] = p.nb; aux->obs_prev[1] = p.nl; }  // the next step rewrites every row of whichever buffer it gets
        if (p.obs) {
            __syncwarp();  // the warp's copies above are visible to all its lanes
            write_obs<OT, 0>(p, e, hot, cold, cold->leaf, n_leaf, lane, 32);
        }
    }
}

// Plain stream-ordered launches (no programmatic serialisation): a save / load sits between the previous step's emit kernel and the next
// step's apply kernel.  The LPT bucket lists (order_file / order_lookup) stay a permutation of the envs after a load, so they need no update;
// d_ready / epoch belong to the step's kernels and are not touched.
cudaError_t launch_records_discrete(const DParams &p, const RecArgs &s, int load, cudaStream_t st) {
    if (s.n <= 0) return cudaSuccess;
    const int blocks = (s.n + 3) / 4;
    if (!load) pct_env_record_kernel<false, float><<<blocks, 128, 0, st>>>(p, s);
    else if (p.obs_f64) pct_env_record_kernel<true, double><<<blocks, 128, 0, st>>>(p, s);
    else pct_env_record_kernel<true, float><<<blocks, 128, 0, st>>>(p, s);
    return cudaGetLastError();
}

// ---- launchers ---------------------------------------------------------------------------------------------
template <typename K>
static cudaError_t set_smem(K kernel, size_t smem) {
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
}

template <typename OT, bool STAB, typename SlotT>
static cudaError_t launch_t(const DParams &p_in, cudaStream_t st, cudaEvent_t *prof) {
    constexpr bool BIGSM = !STAB;
    static bool attr_set = false;
    static int n_sm = 0;
    const size_t smem1 = (size_t)K1_SM_PER_WARP * WARPS_PER_BLOCK;
    const size_t smem2 = (size_t)Lay<SlotT, BIGSM>::PER_WARP * WARPS_PER_BLOCK;
    DParams p = p_in;
    const bool k3_old = (p.opt & PCT_OPT_K3_BLOCK) != 0 || !p.walkq;  // PCT_B200_K3=block: round 1's block-per-env / thread-per-candidate kernel (A/B measurements)
    if (k3_old) p.walkq = nullptr;  // K2 then skips the classification
    if (!attr_set) {
        cudaError_t err = set_smem(pct_apply_kernel<STAB>, smem1);
        if (err == cudaSuccess && STAB) err = set_smem(pct_apply_kernel<STAB, STAB>, smem1);  // the ALIAS variant (stability settings only)
        if (err == cudaSuccess) err = set_smem(pct_candidates_kernel<SlotT, BIGSM>, smem2);
        int dev = 0;
        if (err == cudaSuccess) err = cudaGetDevice(&dev);
        if (err == cudaSuccess) err = cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
        if (err != cudaSuccess) return err;
        attr_set = true;
    }
    const int blocks = (p.n_envs + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK;
    if (prof) cudaEventRecord(prof[0], st);
    if (STAB && (p.opt & PCT_OPT_ALIAS)) pct_apply_kernel<STAB, STAB><<<blocks, 32 * WARPS_PER_BLOCK, smem1, st>>>(p);
    else pct_apply_kernel<STAB><<<blocks, 32 * WARPS_PER_BLOCK, smem1, st>>>(p);
    if (prof) cudaEventRecord(prof[1], st);
    cudaError_t err = cudaSuccess;
    if (p.ready) {
        // overlapped mode (programmatic dependent launch): the candidates blocks become resident while the apply kernel's tail is
        // still running and pick their env up through the per-env hand-over flags
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        cudaLaunchConfig_t cfg{};
        cfg.stream = st; cfg.attrs = at; cfg.numAttrs = 1;
        cfg.gridDim = dim3(blocks); cfg.blockDim = dim3(32 * WARPS_PER_BLOCK); cfg.dynamicSmemBytes = smem2;
        err = cudaLaunchKernelEx(&cfg, pct_candidates_kernel<SlotT, BIGSM>, p);
        if (err != cudaSuccess) return err;
        if (k3_old) {
            cfg.gridDim = dim3(p.n_envs); cfg.blockDim = dim3(FEAS_THREADS); cfg.dynamicSmemBytes = 0;
            err = (p.opt & PCT_OPT_DELTA) ? cudaLaunchKernelEx(&cfg, pct_feas_emit_kernel<OT, STAB, SlotT, true>, p)
                             : cudaLaunchKernelEx(&cfg, pct_feas_emit_kernel<OT, STAB, SlotT>, p);
            if (err != cudaSuccess) return err;
        }
    } else {
        pct_candidates_kernel<SlotT, BIGSM><<<blocks, 32 * WARPS_PER_BLOCK, smem2, st>>>(p);
        if (prof) cudaEventRecord(prof[2], st);
        if (k3_old) {
            if (p.opt & PCT_OPT_DELTA) pct_feas_emit_kernel<OT, STAB, SlotT, true><<<p.n_envs, FEAS_THREADS, 0, st>>>(p);
            else pct_feas_emit_kernel<OT, STAB, SlotT><<<p.n_envs, FEAS_THREADS, 0, st>>>(p);
        }
    }
    if (!k3_old) {
        // the pooled walks need EVERY env's classification (plain stream order = full dependency), the emit kernel every walk
        if (p.ready && prof) cudaEventRecord(prof[2], st);
        if (STAB) {
            pct_walk_light_kernel<<<n_sm * LIGHT_MINB, 32 * LIGHT_WARPS, 0, st>>>(p);
            if (p.walk_fork) pct_walk_fork_kernel<<<n_sm * max(1, min(p.walk_blocks, WALK_MINB)), 32 * WALK_WARPS, 0, st>>>(p);  // one resident wave
            else pct_walk_kernel<<<n_sm * WALK_MINB, 32 * WALK_WARPS, 0, st>>>(p);  // one resident wave (every block starts at once: the emit kernel may follow)
        }
        const int eb = (p.n_envs + EMIT_WARPS - 1) / EMIT_WARPS;
        {   // programmatic dependent of the continuation kernel (setting 2: of the candidates kernel, whose blocks never trigger early -> plain order)
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            at[0].val.programmaticStreamSerializationAllowed = 1;
            cudaLaunchConfig_t cfg{};
            cfg.stream = st; cfg.attrs = at; cfg.numAttrs = (STAB && p.ready && !(p.opt & PCT_OPT_NO_EMIT_PDL)) ? 1 : 0;
            cfg.gridDim = dim3(eb); cfg.blockDim = dim3(32 * EMIT_WARPS); cfg.dynamicSmemBytes = 0;
            err = (p.opt & PCT_OPT_DELTA) ? cudaLaunchKernelEx(&cfg, pct_emit_kernel<OT, SlotT, true>, p) : cudaLaunchKernelEx(&cfg, pct_emit_kernel<OT, SlotT, false>, p);
            if (err != cudaSuccess) return err;
        }
    }
    if (prof) cudaEventRecord(prof[3], st);
    return cudaGetLastError();
}
template <typename OT, bool STAB>
static cudaError_t launch_s(const DParams &p, cudaStream_t st, cudaEvent_t *prof) {
    if (p.W <= 16 && p.L <= 16 && p.H <= 16) return launch_t<OT, STAB, uint16_t>(p, st, prof);
    return launch_t<OT, STAB, uint32_t>(p, st, prof);
}

// number of kernels one reset / step enqueues (for pct_kernel_launches): apply, candidates (+ classify), [walk], emit, order / pool reset
int discrete_kernels_per_step(const DParams &p) {
    if ((p.opt & PCT_OPT_K3_BLOCK) || !p.walkq) return 3;
    return 3 + (p.setting != 2 ? 2 : 0);
}

cudaError_t launch_discrete(const DParams &p, cudaStream_t st, cudaEvent_t *prof) {
    const bool stab = p.setting != 2;
    if (p.obs_f64) return stab ? launch_s<double, true>(p, st, prof) : launch_s<double, false>(p, st, prof);
    return stab ? launch_s<float, true>(p, st, prof) : launch_s<float, false>(p, st, prof);
}

cudaError_t launch_policy_random_discrete(const DEnvHot *hot, int n_envs, int64_t env_id_base, uint64_t seed, int64_t t, int32_t *leaf_idx,
                                          cudaStream_t st, const int64_t *t_dev) {
    pct_policy_random_kernel<<<(n_envs + 127) / 128, 128, 0, st>>>(hot, n_envs, env_id_base, seed, t, t_dev, leaf_idx);
    return cudaGetLastError();
}

}  // namespace pct

#include "pct_heuristics.cuh"
