// Device helpers of the saved env records (pct_save_envs / pct_load_envs), shared by both domains.
#pragma once
#include "pct_common.cuh"
#include "pct_kernels.h"

namespace pct {

// the live prefix [0, bytes) of an array, rounded up to 16-byte units (every array's capacity is a multiple of 16 bytes); one warp, coalesced
__device__ __forceinline__ void warp_copy16(void *dst, const void *src, int bytes, int lane) {
    uint4 *d = (uint4 *)dst;
    const uint4 *s = (const uint4 *)src;
    const int n = (bytes + 15) >> 4;
#pragma unroll 4
    for (int i = lane; i < n; i += 32) d[i] = s[i];
}
// same in 8-byte units, for DEnvAux (its 2888-byte stride leaves every other env 8-byte aligned only)
__device__ __forceinline__ void warp_copy8(void *dst, const void *src, int bytes, int lane) {
    uint2 *d = (uint2 *)dst;
    const uint2 *s = (const uint2 *)src;
    const int n = (bytes + 7) >> 3;
#pragma unroll 4
    for (int i = lane; i < n; i += 32) d[i] = s[i];
}
// header check of a record against the loading handle: 0, REC_BAD_RECORD or REC_ROW_OUTSIDE
__device__ __forceinline__ int rec_check(const RecHdr &r, uint32_t domain, int64_t item_env, const RecArgs &s, int64_t env_id_base, int n_envs) {
    if (r.magic != REC_MAGIC || r.version != REC_VERSION || r.domain != domain || !r.valid || r.fingerprint != s.fingerprint) return REC_BAD_RECORD;
    if (s.row_hash) {
        const int64_t row = item_env - env_id_base;
        if (row < 0 || row >= n_envs) return REC_ROW_OUTSIDE;
        if (s.row_hash[row] != r.row_hash) return REC_BAD_RECORD;
    }
    return 0;
}

}  // namespace pct
