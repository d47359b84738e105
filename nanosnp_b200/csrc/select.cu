// s1 steps B and C: candidate selection (ordered stream compaction) and window gather.
//
// select: replaces the gate + 33-row contiguity rule of create_pileup_tensor (main.cpp:174-217):
//   position c is a site  <=>  GATE(c)  and  COVERED(p) for every p in [c-16, c+16].
//   Three small kernels over the 1-byte flag array: per-segment counts (ballot/popc), single-block scan,
//   ordered write.  Reads 1 B/position when the pileup epilogue already produced the GATE bit.
// gather: a window is the contiguous 33*18 int32 span counts[c-16 .. c+16][:], so the kernel is N_s
//   independent 2376-byte copies, one warp each, 8-byte vector accesses (rows are only 8-byte aligned).
#include "common.cuh"

namespace nsnp {
namespace {

constexpr int kSelThreads = 256;
constexpr int kPerThread = 8;
constexpr int kSeg = kSelThreads * kPerThread;          // 2048 positions per CTA

struct SelArgs {
    const uint8_t* flags;      // [region_len]
    int64_t region_start, region_len;
    int64_t emit_start, emit_end;      // contig coordinates
    const int32_t* targets;            // nullptr, or n_targets sorted disjoint [start, end) pairs (contig coordinates)
    int n_targets;
    const uint8_t* ref;                // sites mode: the contig, for the centre-base rule
};

// target bits of the 8 positions [c0, c0 + 8): binary search for the first interval ending after c0, then at most 8 more
// (intervals are non-empty and disjoint)
__device__ __forceinline__ uint32_t target_mask8(const SelArgs& a, int64_t c0) {
    int lo = 0, hi = a.n_targets;
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (__ldg(a.targets + 2 * mid + 1) > c0) hi = mid; else lo = mid + 1; }
    uint32_t t = 0;
    for (int k = lo; k < a.n_targets; ++k) {
        const int64_t s = __ldg(a.targets + 2 * k), e = __ldg(a.targets + 2 * k + 1);
        if (s >= c0 + 8) break;
        const int b0 = (int)(max(s, c0) - c0), b1 = (int)(min(e, c0 + 8) - c0);
        t |= ((1u << (b1 - b0)) - 1u) << b0;
    }
    return t;
}

// 8-bit candidate mask of positions [seg0 + 8*tid, +8): bit j set <=> site
template <bool kSites>
__device__ __forceinline__ uint32_t cand_mask8(const SelArgs& a, int64_t seg0, uint32_t* covw /* smem, (kSeg+64)/32 + 2 words */) {
    const int tid = threadIdx.x;
    uint8_t* cov8 = reinterpret_cast<uint8_t*>(covw);
    // covered bits of [seg0-16, seg0+kSeg+16) as bytes of 8 positions; byte j <-> positions seg0 - 16 + 8j
    auto pack8 = [&](int64_t i0, uint32_t& gate) -> uint32_t {
        uint32_t c = 0; gate = 0;
        if (i0 >= 0 && i0 + 8 <= a.region_len && ((uintptr_t)(a.flags + i0) & 7) == 0) {
            const uint2 v = *reinterpret_cast<const uint2*>(a.flags + i0);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t f0 = (v.x >> (8 * j)) & 0xFF, f1 = (v.y >> (8 * j)) & 0xFF;
                c |= (f0 & 1u) << j; gate |= ((f0 >> 1) & 1u) << j;
                c |= (f1 & 1u) << (j + 4); gate |= ((f1 >> 1) & 1u) << (j + 4);
            }
        } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int64_t i = i0 + j;
                const uint32_t f = (i >= 0 && i < a.region_len) ? a.flags[i] : 0u;
                c |= (f & 1u) << j; gate |= ((f >> 1) & 1u) << j;
            }
        }
        return c;
    };
    uint32_t gate = 0, gdummy;
    const int64_t i0 = seg0 + (int64_t)tid * 8;
    const uint32_t own = pack8(i0, gate);
    cov8[tid + 2] = (uint8_t)own;
    if constexpr (kSites) {
        // the pileup epilogue folds the ACGT centre-base rule (make_predict_data/main.cpp:92, SURVEY 8a P10) into the GATE
        // bit; the listed covered positions replace that bit here, so the rule is applied again
        gate = own ? own & target_mask8(a, a.region_start + i0) : 0u;
        for (uint32_t g = gate; g; g &= g - 1) {
            const int j = __ffs(g) - 1;
            if (nt4(__ldg(a.ref + a.region_start + i0 + j)) >= 4) gate &= ~(1u << j);
        }
    }
    if (tid < 2) cov8[tid] = (uint8_t)pack8(seg0 - 16 + 8 * tid, gdummy);
    else if (tid < 4) cov8[kSelThreads + tid] = (uint8_t)pack8(seg0 + kSeg + 8 * (tid - 2), gdummy);
    else if (tid < 12) cov8[kSelThreads + tid] = 0;              // padding read by the unaligned extraction
    __syncthreads();
    uint32_t m = 0;
    while (gate) {
        const int j = __ffs(gate) - 1; gate &= gate - 1;
        const int64_t c = a.region_start + i0 + j;
        if (c < a.emit_start || c >= a.emit_end) continue;
        const int b = tid * 8 + j;                         // window [c-16, c+16] <-> bits [b, b+32] of cov
        const uint32_t lo = __funnelshift_r(covw[b >> 5], covw[(b >> 5) + 1], b & 31);
        const uint32_t hi = (covw[(b >> 5) + 1] >> (b & 31)) & 1u;
        if (lo == 0xFFFFFFFFu && hi) m |= 1u << j;
    }
    if (!kSites && a.targets && m) m &= target_mask8(a, a.region_start + i0);
    return m;
}

template <bool kSites>
__global__ void __launch_bounds__(kSelThreads) select_count_kernel(SelArgs a, int32_t* seg_counts) {
    __shared__ uint32_t covw[(kSeg + 64) / 32 + 4];
    __shared__ int wsum[kSelThreads / 32];
    const int64_t seg0 = (int64_t)blockIdx.x * kSeg;
    const int cnt = __popc(cand_mask8<kSites>(a, seg0, covw));
    const int ws = __reduce_add_sync(0xffffffffu, cnt);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = ws;
    __syncthreads();
    if (threadIdx.x == 0) { int s = 0; for (int w = 0; w < kSelThreads / 32; ++w) s += wsum[w]; seg_counts[blockIdx.x] = s; }
}

// exclusive scan of seg_counts in place (single block), total -> n_dev
__global__ void __launch_bounds__(1024) select_scan_kernel(int32_t* seg_counts, int n_seg, int32_t* n_dev, int64_t capacity, int32_t* status) {
    __shared__ int wtot[32];
    __shared__ int carry_s;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) carry_s = 0;
    __syncthreads();
    for (int base = 0; base < n_seg; base += 1024) {
        const int i = base + tid;
        const int v = i < n_seg ? seg_counts[i] : 0;
        int inc = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += t; }
        if (lane == 31) wtot[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            int w = wtot[lane];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(0xffffffffu, w, d); if (lane >= d) w += t; }
            wtot[lane] = w;
        }
        __syncthreads();
        const int carry = carry_s;
        const int excl = carry + (warp ? wtot[warp - 1] : 0) + inc - v;
        if (i < n_seg) seg_counts[i] = excl;
        __syncthreads();
        if (tid == 1023) carry_s = carry + wtot[31];
        __syncthreads();
    }
    if (tid == 0) {
        const int total = carry_s;
        *n_dev = total;
        if ((int64_t)total > capacity) dev_fail(status, DEV_E_CAND_CAP, total);
    }
}

template <bool kSites>
__global__ void __launch_bounds__(kSelThreads) select_write_kernel(SelArgs a, const int32_t* seg_offsets, int32_t* pos_out, int64_t capacity) {
    __shared__ uint32_t covw[(kSeg + 64) / 32 + 4];
    __shared__ int wsum[kSelThreads / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t seg0 = (int64_t)blockIdx.x * kSeg;
    uint32_t m = cand_mask8<kSites>(a, seg0, covw);
    const int cnt = __popc(m);
    int inc = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += t; }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    int off = seg_offsets[blockIdx.x] + inc - cnt;
    for (int w = 0; w < warp; ++w) off += wsum[w];
    const int64_t c0 = a.region_start + seg0 + (int64_t)tid * 8;
    while (m) {
        const int j = __ffs(m) - 1; m &= m - 1;
        if (off < capacity) pos_out[off] = (int32_t)(c0 + j);
        ++off;
    }
}

// recompute the GATE bit from the final count rows (stand-alone use of nsnp_select_candidates)
__global__ void __launch_bounds__(256) regate_kernel(const int32_t* __restrict__ counts, uint8_t* flags, const uint8_t* __restrict__ ref,
                                                     int64_t region_start, int64_t region_len, nsnp_params_t prm) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < region_len; i += (int64_t)gridDim.x * blockDim.x) {
        const int2* row2 = reinterpret_cast<const int2*>(counts + i * 18);
        int v[18];
#pragma unroll
        for (int j = 0; j < 9; ++j) { const int2 t = row2[j]; v[2 * j] = t.x; v[2 * j + 1] = t.y; }
        const int rc4 = nt4(ref[region_start + i]);
        const int chr = rc4 < 4 ? rc4 : 0;
        // undo the reference-channel overwrite (tensor_maker.cpp:230-246): v[chr] = -(A+C+G+T)
        int mf = 0, mr = 0, oth = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) { if (b == chr) { mf = -v[b]; mr = -v[9 + b]; } else oth += v[b] + v[9 + b]; }
        int tally[6];
        tally[0] = chr == 0 ? mf + mr - oth : v[0] + v[9];
        tally[1] = chr == 1 ? mf + mr - oth : v[1] + v[10];
        tally[2] = v[6] + v[15];
        tally[3] = chr == 2 ? mf + mr - oth : v[2] + v[11];
        tally[4] = v[4] + v[13];
        tally[5] = chr == 3 ? mf + mr - oth : v[3] + v[12];
        const int depth = mf + mr + v[8] + v[17];
        const int den = depth ? depth : 1;
        int top = -1, topc = 0;
#pragma unroll
        for (int k = 0; k < 6; ++k) if (tally[k] > topc) { topc = tally[k]; top = k; }
        const int chr_key = chr == 0 ? 0 : chr == 1 ? 1 : chr == 2 ? 3 : 5;
        bool pass = top >= 0 && top != chr_key;
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            if (k == chr_key || tally[k] == 0) continue;
            pass = pass || (1.0 * tally[k] / den >= ((k == 2 || k == 4) ? prm.indel_min_af : prm.snp_min_af));
        }
        const uint8_t f = flags[i];
        const bool gate = (f & NSNP_F_COVERED) && rc4 < 4 && pass && depth >= prm.min_coverage;
        flags[i] = (uint8_t)((f & ~NSNP_F_GATE) | (gate ? NSNP_F_GATE : 0));
    }
}

__global__ void __launch_bounds__(256) gather_kernel(const int32_t* __restrict__ counts, const uint8_t* __restrict__ ref,
                                                     int64_t region_start, int64_t region_len, const int32_t* __restrict__ pos,
                                                     const int32_t* __restrict__ n_dev, int64_t n_max,
                                                     int32_t* __restrict__ xi, float* __restrict__ xf, uint8_t* __restrict__ refbase)
{
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    int64_t n = n_max;
    if (n_dev) { const int64_t nd = *n_dev; if (nd < n) n = nd; }
    constexpr int kPairs = NSNP_WINDOW * NSNP_CHANNELS / 2;        // 297 int2 per window
    for (int64_t s = warp0; s < n; s += nwarps) {
        const int64_t c = pos[s];
        const int64_t i0 = c - region_start - NSNP_FLANK;           // first window row, region coordinates
        if (i0 < 0 || i0 + NSNP_WINDOW > region_len) continue;      // cannot happen for sites produced by select
        const int2* src = reinterpret_cast<const int2*>(counts + i0 * NSNP_CHANNELS);
        int2 v[10];
#pragma unroll
        for (int j = 0; j < 10; ++j) { const int k = lane + 32 * j; if (k < kPairs) v[j] = __ldg(src + k); }
        if (xi) {
            int2* dst = reinterpret_cast<int2*>(xi + s * (NSNP_WINDOW * NSNP_CHANNELS));
#pragma unroll
            for (int j = 0; j < 10; ++j) { const int k = lane + 32 * j; if (k < kPairs) st_stream(dst + k, v[j]); }
        }
        if (xf) {
            float2* dst = reinterpret_cast<float2*>(xf + s * (NSNP_WINDOW * NSNP_CHANNELS));
#pragma unroll
            for (int j = 0; j < 10; ++j) { const int k = lane + 32 * j; if (k < kPairs) dst[k] = make_float2((float)v[j].x, (float)v[j].y); }
        }
        if (refbase && lane == 0) { uint8_t r = ref[c]; if (r >= 'a' && r <= 'z') r = (uint8_t)(r - 32); refbase[s] = r; }
    }
}

}  // namespace
}  // namespace nsnp

using namespace nsnp;

extern "C" {

size_t nsnp_select_workspace_bytes(int64_t region_len) {
    const int64_t n_seg = (region_len + kSeg - 1) / kSeg;
    return (size_t)(n_seg + 1) * 4 + 256;
}

}  // extern "C"

// targets == nullptr && n_targets < 0: every position of the emit range (nsnp_select_candidates)
// sites: listed positions replace the gate (nsnp_select_candidates_sites; params and recompute_gate are unused)
static int select_candidates(const int32_t* counts_dev, uint8_t* flags_dev, const uint8_t* ref_dev, int64_t contig_len,
                             int64_t region_start, int64_t region_len, int64_t emit_start, int64_t emit_end,
                             const int32_t* targets, int64_t n_targets, const nsnp_params_t* params, int recompute_gate,
                             int32_t* pos_dev, int64_t capacity, int32_t* n_dev, void* workspace_dev, size_t workspace_bytes,
                             int32_t* status_dev, void* stream_, bool sites = false)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!flags_dev || !pos_dev || !n_dev || !workspace_dev || !status_dev || (!params && !sites) || (sites && !ref_dev))
        return set_error(NSNP_E_INVALID, "nsnp_select_candidates: null argument");
    if (recompute_gate && (!counts_dev || !ref_dev)) return set_error(NSNP_E_INVALID, "nsnp_select_candidates: recompute_gate needs counts and ref");
    if (region_start < 0 || region_len < 0 || region_start + region_len > contig_len || capacity < 0)
        return set_error(NSNP_E_INVALID, "nsnp_select_candidates: bad region");
    if (n_targets >= 0) {
        if (int e = check_targets(sites ? "nsnp_select_candidates_sites" : "nsnp_select_candidates_targets", targets, n_targets,
                                  region_start, region_start + region_len)) return e;
    }
    const size_t ws_need = n_targets >= 0 ? nsnp_select_targets_workspace_bytes(region_len, n_targets) : nsnp_select_workspace_bytes(region_len);
    if (workspace_bytes < ws_need) return set_error(NSNP_E_WORKSPACE, "select workspace too small");
    if (nsnp_device_count() == 0) return set_error(NSNP_E_NO_DEVICE, "no CUDA device (there is no CPU fallback)");
    if (region_len == 0 || emit_end <= emit_start || n_targets == 0) { cudaMemsetAsync(n_dev, 0, 4, stream); return cuda_status("memset n"); }
    if (recompute_gate) {
        int blocks = (int)((region_len + 255) / 256); if (blocks > kNumSMs * 16) blocks = kNumSMs * 16;
        regate_kernel<<<blocks, 256, 0, stream>>>(counts_dev, flags_dev, ref_dev, region_start, region_len, *params);
        if (int e = cuda_status("regate_kernel")) return e;
    }
    ProfScope prof(NSNP_PROF_SELECT, stream);
    SelArgs a{flags_dev, region_start, region_len, emit_start, emit_end, nullptr, 0, ref_dev};
    const int n_seg = (int)((region_len + kSeg - 1) / kSeg);
    int32_t* seg = (int32_t*)workspace_dev;
    if (n_targets > 0) {                        // the interval copy sits behind the segment counts
        int32_t* iv = (int32_t*)((char*)workspace_dev + nsnp_select_workspace_bytes(region_len));
        cudaMemcpyAsync(iv, targets, (size_t)n_targets * 8, cudaMemcpyHostToDevice, stream);
        a.targets = iv; a.n_targets = (int)n_targets;
    }
    if (sites) select_count_kernel<true><<<n_seg, kSelThreads, 0, stream>>>(a, seg);
    else select_count_kernel<false><<<n_seg, kSelThreads, 0, stream>>>(a, seg);
    select_scan_kernel<<<1, 1024, 0, stream>>>(seg, n_seg, n_dev, capacity, status_dev);
    if (sites) select_write_kernel<true><<<n_seg, kSelThreads, 0, stream>>>(a, seg, pos_dev, capacity);
    else select_write_kernel<false><<<n_seg, kSelThreads, 0, stream>>>(a, seg, pos_dev, capacity);
    return cuda_status("select kernels");
}

extern "C" {

int nsnp_select_candidates(const int32_t* counts_dev, uint8_t* flags_dev, const uint8_t* ref_dev, int64_t contig_len,
                           int64_t region_start, int64_t region_len, int64_t emit_start, int64_t emit_end,
                           const nsnp_params_t* params, int recompute_gate, int32_t* pos_dev, int64_t capacity,
                           int32_t* n_dev, void* workspace_dev, size_t workspace_bytes, int32_t* status_dev, void* stream)
{
    return select_candidates(counts_dev, flags_dev, ref_dev, contig_len, region_start, region_len, emit_start, emit_end, nullptr, -1,
                             params, recompute_gate, pos_dev, capacity, n_dev, workspace_dev, workspace_bytes, status_dev, stream);
}

size_t nsnp_select_targets_workspace_bytes(int64_t region_len, int64_t n_targets) {
    return nsnp_select_workspace_bytes(region_len) + (size_t)(n_targets < 0 ? 0 : n_targets) * 8 + 256;
}

int nsnp_select_candidates_targets(const int32_t* counts_dev, uint8_t* flags_dev, const uint8_t* ref_dev, int64_t contig_len,
                                   int64_t region_start, int64_t region_len, int64_t emit_start, int64_t emit_end,
                                   const int32_t* targets, int64_t n_targets, const nsnp_params_t* params, int recompute_gate,
                                   int32_t* pos_dev, int64_t capacity, int32_t* n_dev, void* workspace_dev, size_t workspace_bytes,
                                   int32_t* status_dev, void* stream)
{
    if (n_targets < 0) return set_error(NSNP_E_INVALID, "nsnp_select_candidates_targets: negative interval count");
    return select_candidates(counts_dev, flags_dev, ref_dev, contig_len, region_start, region_len, emit_start, emit_end, targets,
                             n_targets, params, recompute_gate, pos_dev, capacity, n_dev, workspace_dev, workspace_bytes, status_dev, stream);
}

size_t nsnp_select_sites_workspace_bytes(int64_t region_len, int64_t n_sites) {
    return nsnp_select_targets_workspace_bytes(region_len, n_sites);
}

int nsnp_select_candidates_sites(const uint8_t* flags_dev, const uint8_t* ref_dev, int64_t contig_len, int64_t region_start,
                                 int64_t region_len, int64_t emit_start, int64_t emit_end, const int32_t* sites, int64_t n_sites,
                                 int32_t* pos_dev, int64_t capacity, int32_t* n_dev, void* workspace_dev, size_t workspace_bytes,
                                 int32_t* status_dev, void* stream)
{
    if (n_sites < 0) return set_error(NSNP_E_INVALID, "nsnp_select_candidates_sites: negative interval count");
    return select_candidates(nullptr, const_cast<uint8_t*>(flags_dev), ref_dev, contig_len, region_start, region_len, emit_start,
                             emit_end, sites, n_sites, nullptr, 0, pos_dev, capacity, n_dev, workspace_dev, workspace_bytes,
                             status_dev, stream, true);
}

int nsnp_gather_windows(const int32_t* counts_dev, const uint8_t* ref_dev, int64_t region_start, int64_t region_len,
                        const int32_t* pos_dev, const int32_t* n_dev, int64_t n_max, int32_t* x_i32_dev, float* x_f32_dev,
                        uint8_t* refbase_dev, void* stream_)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!counts_dev || !pos_dev || (!x_i32_dev && !x_f32_dev && !refbase_dev)) return set_error(NSNP_E_INVALID, "nsnp_gather_windows: null argument");
    if (refbase_dev && !ref_dev) return set_error(NSNP_E_INVALID, "nsnp_gather_windows: refbase needs ref");
    if (((uintptr_t)counts_dev & 7) || ((uintptr_t)x_i32_dev & 7) || ((uintptr_t)x_f32_dev & 7))
        return set_error(NSNP_E_INVALID, "nsnp_gather_windows: 8-byte alignment required");
    if (nsnp_device_count() == 0) return set_error(NSNP_E_NO_DEVICE, "no CUDA device (there is no CPU fallback)");
    if (n_max <= 0) return NSNP_OK;
    int64_t blocks = (n_max + 7) / 8; if (blocks > kNumSMs * 16) blocks = kNumSMs * 16;
    ProfScope prof(NSNP_PROF_GATHER, stream);
    gather_kernel<<<(int)blocks, 256, 0, stream>>>(counts_dev, ref_dev, region_start, region_len, pos_dev, n_dev, n_max, x_i32_dev, x_f32_dev, refbase_dev);
    return cuda_status("gather_kernel");
}

}  // extern "C"
