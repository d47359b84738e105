// Shared host/device helpers for the nanosnp_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include "../../include/nanosnp_b200.h"

namespace nsnp {

int set_error(int code, const char* fmt, ...);   // records a thread-local message, returns code
int cuda_status(const char* what);               // maps cudaGetLastError() to NSNP_E_CUDA / NSNP_OK

// RAII bracket around one kernel launch when profiling is on (api.cu)
struct ProfScope {
    int slot; cudaStream_t stream; void* pending;
    ProfScope(int slot_, cudaStream_t s);
    ~ProfScope();
};

constexpr int kNumSMs = 148;                     // B200: 2 dies x 74 SMs

// device-side status words (status_dev[4])
enum { ST_ERR = 0, ST_DETAIL = 1, ST_AUX0 = 2, ST_AUX1 = 3 };
enum { DEV_OK = 0, DEV_E_DEPTH = 1, DEV_E_INDEL_SLAB = 2, DEV_E_SEQ_SPAN = 3, DEV_E_CAND_CAP = 4, DEV_E_UNSORTED = 5, DEV_E_CIGAR = 6 };

__device__ __forceinline__ void dev_fail(int32_t* status, int code, int detail) {
    if (atomicCAS(&status[ST_ERR], 0, code) == 0) status[ST_DETAIL] = detail;
}

// streaming (read-once / write-once) global accesses: keep them out of L1
__device__ __forceinline__ int4 ld_stream(const int4* p) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ int2 ld_stream(const int2* p) {
    int2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.s32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream(int4* p, const int4& v) {
    asm volatile("st.global.L1::no_allocate.v4.s32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void st_stream(int2* p, const int2& v) {
    asm volatile("st.global.L1::no_allocate.v2.s32 [%0], {%1,%2};" ::"l"(p), "r"(v.x), "r"(v.y) : "memory");
}

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

// reference base classification (cpp_aux.cpp nst_nt4_table: ACGTacgt -> 0..3, everything else 4)
__host__ __device__ __forceinline__ int nt4(uint8_t c) {
    switch (c) {
        case 'A': case 'a': return 0;
        case 'C': case 'c': return 1;
        case 'G': case 'g': return 2;
        case 'T': case 't': return 3;
        default: return 4;
    }
}

// Target intervals of nsnp_pileup_counts_targets / nsnp_select_candidates_targets: n half-open [start, end) int32 pairs in
// contig coordinates (host memory), non-empty, ascending and disjoint (adjacent allowed), inside [lo, hi).
inline int check_targets(const char* fn, const int32_t* iv, int64_t n, int64_t lo, int64_t hi) {
    if (n < 0 || (n > 0 && !iv)) return set_error(NSNP_E_INVALID, "%s: bad interval list", fn);
    int64_t prev = lo;
    for (int64_t k = 0; k < n; ++k) {
        const int64_t s = iv[2 * k], e = iv[2 * k + 1];
        if (s < prev || e <= s || e > hi)
            return set_error(NSNP_E_INVALID, "%s: interval %lld [%lld,%lld) is empty, unsorted, overlapping or outside [%lld,%lld)", fn,
                             (long long)k, (long long)s, (long long)e, (long long)lo, (long long)hi);
        prev = e;
    }
    return NSNP_OK;
}

}  // namespace nsnp
