// s2 on the 5th-generation tensor cores: the LSTM gate contractions of PileupModel (model.py:18-25,34-35)
// as tcgen05.mma with TMEM accumulators, hand-written for sm_100a.
//
// One CTA = 128 candidate sites x one direction of one layer; per time step
//     gates[128 x 256] = [in_t | h_{t-1}] [128 x K]  .  W^T [K x 256]            (K = 96 layer 0, 192 layer 1)
// runs as K/16 x 3 tcgen05.mma (M=128 or 256, N=256, K=16, kind::f16, fp32 accumulate in 256 TMEM columns).
//
// Precision: fp32-grade results from fp16 tensor-core inputs by hi/lo operand splitting,
//     a.w  ~=  a_hi.w_hi + a_hi.w_lo + a_lo.w_hi        (dropped term a_lo.w_lo ~ 2^-22 relative)
// implemented as three K-passes into the same accumulator.  Counts (layer-0 inputs, integers that reach
// hundreds) use a pre-scaled low part -- (x_hi 2^-10).(w_lo 2^10) -- so the low weight halves stay in the
// normal fp16 range.  Layer 0's bias rides in the GEMM as a constant-1 input column (its input k-blocks have spare
// columns); layer 1 is tensor-bound, so its bias is added in the epilogue instead of costing a k-block.  The activation
// scales (-log2 e, -2 log2 e) are folded into the packed weights: every exponential is a bare ex2 of an accumulator.
//
// Operands sit in shared memory in the UMMA canonical K-major / no-swizzle layout: 8x(16-byte) core
// matrices, [k/8][row][k%8]; a thread owns one site row, so it writes whole 16-byte core-matrix rows
// (conflict free) and the next step's A operand is produced directly by the epilogue.
//
// Epilogue (8 warps = 2 per TMEM lane quadrant): tcgen05.ld 32 columns = (i,f,g,o) of 8 hidden units,
// cell update with one reciprocal per (c', h) pair (5 ex2 + 2 rcp on the MUFU pipe), h -> fp16 hi/lo ->
// st.shared (next step's operand) and -> global for layer 1.
//
// CG = 2 pairs two CTAs (cta_group::2): M = 256, each CTA holds half of W (N/2 rows) -- that is what makes the
// layer-1 weights (2 x 96 KB) fit; the leader CTA issues the MMAs, tcgen05.commit multicasts completion.
//
// Kernels: lstm0_pair2_kernel (layer 0, production), lstm1_pair2x3_kernel (layer 1, production), lstm1_pair2_kernel
// (layer 1, single-pass NSNP_PREC_F16X1), lstm_tc_kernel<1,2,4> (layer-1 alternative NSNP_L1_VARIANT=0 and the debug entry),
// lstm_tc_kernel<0,...> (layer-0 alternative NSNP_L0_VARIANT=0 and the raw-accumulator debug entry), tail_tc_kernel.
#include <cuda_fp16.h>
#include <stdlib.h>
#include "model_common.cuh"
#include "tc_ptx.cuh"

namespace nsnp {
namespace {

constexpr int kRows = 128;             // sites per CTA = TMEM lanes
constexpr float kLog2e = 1.4426950408889634f;

// hi copy of integer counts scaled by 2^-10 (exact: counts are integers, results stay normal or zero)
__device__ __forceinline__ uint4 scale_hi(const uint4& hi) {
    const __half2 k = __float2half2_rn(1.0f / kTcLoScale);
    auto m = [&](uint32_t x) { __half2 t = *reinterpret_cast<__half2*>(&x); return h2_bits(__hmul2(t, k)); };
    return make_uint4(m(hi.x), m(hi.y), m(hi.z), m(hi.w));
}

template <int LAYER> struct TcCfg;
template <> struct TcCfg<0> { static constexpr int K = kTcK0, IN = kTcIn0, STEPS = 33; };
template <> struct TcCfg<1> { static constexpr int K = kTcK1, IN = kTcIn1, STEPS = 17; };

template <int LAYER, int CG> struct TcSmem {
    static constexpr int K = TcCfg<LAYER>::K;
    static constexpr int RB = 256 / CG;                        // weight rows held by this CTA
    static constexpr size_t b_bytes = (size_t)K * RB * 2;      // one of hi / lo
    static constexpr size_t a_bytes = (size_t)K * kRows * 2;
    static constexpr size_t sc_bytes = LAYER == 0 ? (size_t)kTcIn0 * kRows * 2 : 0;
    static constexpr size_t off_bhi = 0, off_blo = b_bytes, off_ahi = 2 * b_bytes, off_alo = off_ahi + a_bytes,
                            off_asc = off_alo + a_bytes, off_bar = off_asc + sc_bytes, off_bias = off_bar + 64,
                            total = off_bias + (LAYER == 1 ? 256 * sizeof(float) : 0);
};

// NWQ warps share each TMEM lane quadrant (each thread = one site row x 64/NWQ hidden units).
// DEBUG: dump the raw accumulators of the first step and return.
template <int LAYER, int CG, int NWQ, bool DEBUG>
__global__ void __launch_bounds__(128 * NWQ + (LAYER == 1 ? 32 : 0), (LAYER == 0 && CG == 2 && NWQ == 2) ? 2 : 1)
lstm_tc_kernel(const unsigned char* __restrict__ blob, const int32_t* __restrict__ xi, const float* __restrict__ xf,
               const __half* __restrict__ h0_in, __half* __restrict__ h0_out, float* __restrict__ h16, float* __restrict__ dbg,
               int64_t n, int dir_override)
{
    using C = TcCfg<LAYER>;
    using S = TcSmem<LAYER, CG>;
    constexpr int K = C::K, IN = C::IN, RB = S::RB;
    constexpr int KB = K / 16;                                   // MMA k-blocks per pass
    constexpr int kThreads = 128 * NWQ + (LAYER == 1 ? 32 : 0);     // layer 1: + one producer warp (bulk copies of the next input)
    constexpr int kEpiWarps = 4 * NWQ;
    constexpr int UB = 8 / NWQ;                                  // blocks of 8 hidden units per thread
    constexpr uint32_t LBO_A = kRows * 16, LBO_B = RB * 16, SBO = 128;
    extern __shared__ __align__(1024) unsigned char smem[];
    unsigned char* sBhi = smem + S::off_bhi; unsigned char* sBlo = smem + S::off_blo;
    unsigned char* sAhi = smem + S::off_ahi; unsigned char* sAlo = smem + S::off_alo; unsigned char* sAsc = smem + S::off_asc;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + S::off_bar);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + S::off_bar + 32);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool producer = LAYER == 1 && warp == kEpiWarps;       // warp-uniform
    const int quad = warp & 3, sub = producer ? 0 : (warp >> 2);
    const int row = quad * 32 + lane;                            // site row = TMEM lane
    const int dir = DEBUG ? dir_override : (int)blockIdx.y;
    const uint32_t cta_rank = CG == 2 ? cluster_ctarank() : 0u;
    const int64_t site0 = (int64_t)blockIdx.x * kRows;
    int64_t site = site0 + row;
    const bool live = site < n;
    if (!live) site = n - 1;                                     // clamp loads, skip stores

    // ---- one-time setup ----
    if (tid == 0) { mbar_init(bar, 1); mbar_init(bar + 1, 1); mbar_init(bar + 2, 1); fence_mbar_init(); }
    if (warp == 0) tmem_alloc<CG>(tmem_slot, LAYER == 1 ? 512 : 256);
    {   // this CTA's weight rows: global [K/8][256][8] halfs -> shared [K/8][RB][8]
        const uint4* ghi = reinterpret_cast<const uint4*>(blob + tc_off(LAYER, dir, 0));
        const uint4* glo = reinterpret_cast<const uint4*>(blob + tc_off(LAYER, dir, 1));
        uint4* dhi = reinterpret_cast<uint4*>(sBhi); uint4* dlo = reinterpret_cast<uint4*>(sBlo);
        for (int i = tid; i < (K / 8) * RB; i += kThreads) {
            const int ch = i / RB, r = i - ch * RB;
            const int g = ch * 256 + (int)cta_rank * RB + r;
            dhi[i] = __ldg(ghi + g); dlo[i] = __ldg(glo + g);
        }
        uint4* a = reinterpret_cast<uint4*>(sAhi);
        const int n16 = (int)((2 * S::a_bytes + S::sc_bytes) / 16);
        for (int i = tid; i < n16; i += kThreads) a[i] = make_uint4(0, 0, 0, 0);
    }
    __syncthreads();
    // constant chunk holding the bias column (1.0) -- layer 0: chunk 2 is rewritten every step with x16, x17
    // layer 1: the (scaled) bias of this direction, added to the accumulators in the epilogue
    const float* sBias = reinterpret_cast<const float*>(smem + S::off_bias);
    if (LAYER == 1) {
        const float* gb = reinterpret_cast<const float*>(blob + kOffTcBias1) + dir * 256;
        for (int i = tid; i < 256; i += kThreads) reinterpret_cast<float*>(smem + S::off_bias)[i] = __ldg(gb + i);
        __syncthreads();
    }

    float c[UB][8];
#pragma unroll
    for (int j = 0; j < UB; ++j)
#pragma unroll
        for (int u = 0; u < 8; ++u) c[j][u] = 0.f;

    // ---- input staging.  Layer 0: counts row -> registers (prefetch) -> fp16 hi / lo / scaled-hi chunks.
    //      Layer 1: layer-0 output is already fp16 hi|lo in global memory -> cp.async straight into the operand. ----
    // layer 0 work split: sub 0 converts x[0..15] (chunks 0,1); the last sub converts x16, x17 + the bias column (chunk 2)
    int2 xraw[8];                                                    // raw bits: converted only when stored (no stall at the load)
    auto load_x = [&](int t) {
        if (LAYER != 0) return;
        const int2* g = reinterpret_cast<const int2*>(xi ? (const void*)(xi + (site * kT + t) * kF) : (const void*)(xf + (site * kT + t) * kF));
        if (sub == 0) {
#pragma unroll
            for (int j = 0; j < 8; ++j) xraw[j] = ldg_nc_volatile(g + j);
        } else if (sub == NWQ - 1) {
            xraw[0] = ldg_nc_volatile(g + 8);
        }
    };
    auto xval = [&](int j) -> float {
        const int2 p = xraw[j >> 1];
        const int b = (j & 1) ? p.y : p.x;
        return xi ? (float)b : __int_as_float(b);
    };
    auto store_x = [&]() {
        if (LAYER != 0) return;
        if (sub == 0) {
#pragma unroll
            for (int ch = 0; ch < 2; ++ch) {
                float v[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) v[j] = xval(ch * 8 + j);
                const HiLo8 s = split8(v);
                reinterpret_cast<uint4*>(sAhi + ch * LBO_A)[row] = s.hi;
                reinterpret_cast<uint4*>(sAlo + ch * LBO_A)[row] = s.lo;
                reinterpret_cast<uint4*>(sAsc + ch * LBO_A)[row] = scale_hi(s.hi);
            }
        } else if (sub == NWQ - 1) {
            const float v[8] = {xval(0), xval(1), 1.0f, 0.f, 0.f, 0.f, 0.f, 0.f};  // x16, x17, bias column
            const HiLo8 s = split8(v);
            reinterpret_cast<uint4*>(sAhi + 2 * LBO_A)[row] = s.hi;
            reinterpret_cast<uint4*>(sAlo + 2 * LBO_A)[row] = s.lo;
            reinterpret_cast<uint4*>(sAsc + 2 * LBO_A)[row] = scale_hi(s.hi);
        }
    };
    // layer 1: the layer-0 output of one (tile, t) is stored exactly in operand layout, hi part then lo part, 32 KB each:
    //     h0[tile][t][hi|lo][chunk 16][row 128][8 halfs]
    uint64_t* barS = bar + 2;                                        // "input part of A for the next step has landed"
    constexpr uint32_t kPartBytes = 16u * kRows * 16u;               // 32 KB
    const bool l2_prefetch = (dir_override >> 8) & 1;
    const int npass = ((dir_override >> 16) & 3) ? ((dir_override >> 16) & 3) : 3;   // NSNP_PREC_F16X1: the hi.hi pass only
    // the padding CTA of an odd tile count (clusters come in pairs) re-reads the last real tile: it must not touch memory
    // past the layer-0 output (found by compute-sanitizer memcheck)
    const size_t src_tile = min((size_t)blockIdx.x, (size_t)((n + kRows - 1) / kRows - 1));
    auto stage_h0_bulk = [&](int t) {                                // one thread
        const __half* src = h0_in + (src_tile * kT + t) * (2 * kPartBytes / 2);
        mbar_expect_tx(barS, 2 * kPartBytes);
        bulk_g2s(sAhi, src, kPartBytes, barS);
        bulk_g2s(sAlo, src + kPartBytes / 2, kPartBytes, barS);
        // the rows of the step after this one: pull them into L2 now, so that their bulk copy (issued when the operand
        // buffer is free again, one step from now) pays L2 latency instead of DRAM latency
        const int tp = dir == 0 ? t + 1 : t - 1;
        if (l2_prefetch && tp >= 0 && tp < kT) bulk_prefetch_l2(h0_in + (src_tile * kT + tp) * (2 * kPartBytes / 2), 2 * kPartBytes);
    };
    constexpr int XB = IN / 16;                                  // k-blocks of the input part; the rest is the h part
    constexpr uint32_t kTmemCols = LAYER == 1 ? 512 : 256;       // layer 1 double-buffers the accumulator
    uint64_t* barH = bar;                                        // "gates of this step are complete"
    uint64_t* barX = bar + 1;                                    // layer 1: "input part of the NEXT step is accumulated"
    {
        const int t0 = dir == 0 ? 0 : kT - 1;
        load_x(t0); store_x();
        fence_async_smem();
    }

    tc_fence_before();
    if (CG == 2) cluster_sync_all(); else __syncthreads();         // barriers initialised, operands zeroed, TMEM allocated
    tc_fence_after();
    uint32_t phaseH = 0, phaseX = 0, phaseS = 0;
    if (LAYER == 1) {
        if (producer && lane == 0) stage_h0_bulk(dir == 0 ? 0 : kT - 1);
        mbar_wait(barS, phaseS); phaseS ^= 1;
        tc_fence_before();
        if (CG == 2) cluster_sync_all(); else __syncthreads();     // both CTAs of the pair have their first input
        tc_fence_after();
    }
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t a_hi = smem_u32(sAhi), a_lo = smem_u32(sAlo), a_sc = smem_u32(sAsc), b_hi = smem_u32(sBhi), b_lo = smem_u32(sBlo);
    constexpr uint32_t idesc = make_idesc(128 * CG, 256);
    const bool issuer = cta_rank == 0 && tid == 0;
    // k-blocks [kb0, kb1) x three hi/lo passes into the accumulator at tmem_d
    auto issue = [&](int kb0, int kb1, uint32_t tmem_d, uint32_t acc) {
#pragma unroll 1
        for (int pass = 0; pass < npass; ++pass) {
#pragma unroll 1
            for (int kb = kb0; kb < kb1; ++kb) {
                // pass 0: a_hi.w_hi   pass 1: a_hi.w_lo (layer-0 counts: scaled copy)   pass 2: a_lo.w_hi
                uint32_t aa = pass == 2 ? a_lo : a_hi;
                if (LAYER == 0 && pass == 1 && kb < kTcIn0 / 16) aa = a_sc;
                const uint32_t bb = pass == 1 ? b_lo : b_hi;
                umma_f16<CG>(tmem_d, make_desc(aa + kb * 2 * LBO_A, LBO_A, SBO), make_desc(bb + kb * 2 * LBO_B, LBO_B, SBO), idesc, acc);
                acc = 1;
            }
        }
    };
    if (LAYER == 1) {
        // software pipeline: the input part of step t+1 (24 of 36 MMAs, independent of h_t) runs on the tensor core
        // while the epilogue of step t runs on the SM; only the 12 h-part MMAs stay on the per-step critical path
        if (issuer) { tc_fence_after(); issue(0, XB, tmem_base, 0); umma_commit<CG>(barX); }
        if (producer) {
            mbar_wait(barX, phaseX); phaseX ^= 1;
            if (lane == 0 && C::STEPS > 1 && !DEBUG) stage_h0_bulk(dir == 0 ? 1 : kT - 2);
        }
    }

    for (int step = 0; step < C::STEPS; ++step) {
        const int t = dir == 0 ? step : (kT - 1 - step);
        const int tn = dir == 0 ? step + 1 : (kT - 2 - step);
        const bool more = !DEBUG && step + 1 < C::STEPS;
        const uint32_t acc_cols = LAYER == 1 ? (uint32_t)(step & 1) * 256u : 0u;
        // ---- operands written by the generic proxy -> visible to the tensor core; TMEM reads of the last step retired ----
        if (LAYER == 1 && more) { mbar_wait(barS, phaseS); phaseS ^= 1; }      // the input rows of step t+1 have landed (their MMAs are issued below)
        fence_async_smem();
        tc_fence_before();
        if (CG == 2) cluster_sync_exec(); else __syncthreads();
        if (issuer) {
            tc_fence_after();
            if (LAYER == 1) {
                issue(XB, KB, tmem_base + acc_cols, 1);                       // += W_hh . h_{t-1}
                umma_commit<CG>(barH);
                if (more) { issue(0, XB, tmem_base + (acc_cols ^ 256u), 0); umma_commit<CG>(barX); }
            } else {
                issue(0, KB, tmem_base, 0);
                umma_commit<CG>(barH);
            }
        }
        if (producer) {
            // producer warp: once the input-part MMAs of step t+1 have completed, their operand region takes the rows of
            // step t+2 (two 32 KB bulk copies); it never touches TMEM and skips the epilogue
            if (more) {
                mbar_wait(barX, phaseX); phaseX ^= 1;
                if (lane == 0 && step + 2 < C::STEPS) stage_h0_bulk(dir == 0 ? step + 2 : kT - 3 - step);
            }
            if (DEBUG) break;
            continue;
        }
        if (more) load_x(tn);                                       // global latency hides under the MMAs
        mbar_wait(barH, phaseH);
        phaseH ^= 1;
        tc_fence_after();

        if (DEBUG) {
#pragma unroll 1
            for (int jb = sub * UB; jb < sub * UB + UB; ++jb) {
                float v[32];
                tmem_ld32(tmem_base + acc_cols + ((uint32_t)(quad * 32) << 16) + jb * 32, v);
                if (live) for (int i = 0; i < 32; ++i) dbg[(site0 + row) * 256 + jb * 32 + i] = v[i] + (LAYER == 1 ? sBias[jb * 32 + i] : 0.f);
            }
            break;
        }

        // ---- epilogue: UB blocks of 8 hidden units per thread, as 2*UB half blocks of 4 units whose TMEM loads are
        //      software pipelined (the 16 columns of a half block are i,f,g,o of its 4 units) ----
        uint32_t vb[2][16];
        const uint32_t tacc = tmem_base + acc_cols + ((uint32_t)(quad * 32) << 16) + (uint32_t)(sub * UB) * 32u;
        tmem_ld16_nowait(tacc, vb[0]);
        tmem_wait_ld();
        float hv[8];
#pragma unroll
        for (int hb = 0; hb < 2 * UB; ++hb) {
            const int jl = hb >> 1, uh = hb & 1, jb = sub * UB + jl;
            if (hb + 1 < 2 * UB) tmem_ld16_nowait(tacc + (hb + 1) * 16, vb[(hb + 1) & 1]);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const uint32_t* v = vb[hb & 1];
                // The packed weights carry the activation scales (pack_tc_weights): the accumulators are
                //     xi = -log2e i,  xf = -log2e f,  xg = -2 log2e g,  xo = -log2e o
                // so every exponential is a bare ex2, and the cell state is kept as cs = -2 log2e c, which makes the
                // argument of tanh(c')'s exponential the state itself.
                // Only the upper clamps are needed: a huge argument would give ex2 = +inf and inf * 0 below, a very negative
                // one gives ex2 = 0, which is exact.  With the clamps every (1 + e) factor is <= 2^36 + 1, so the triple
                // product stays below 2^108 and its reciprocal stays a normal float.  |c'| <= 33 after 33 steps, so
                // ex2(cs') <= 2^96 needs no clamp; an overflowing (1 + eo) makes rcp return 0 = the exact limit.
                const float* bq = sBias + jb * 32 + uh * 16 + u;              // layer 1 only: bias of gate columns i, f, g, o
                const float bi_ = LAYER == 1 ? bq[0] : 0.f, bf_ = LAYER == 1 ? bq[4] : 0.f, bg_ = LAYER == 1 ? bq[8] : 0.f, bo_ = LAYER == 1 ? bq[12] : 0.f;
                const float xi_ = fminf(__uint_as_float(v[u]) + bi_, 36.f), xf_ = fminf(__uint_as_float(v[4 + u]) + bf_, 36.f);
                const float xg_ = fminf(__uint_as_float(v[8 + u]) + bg_, 36.f), xo_ = __uint_as_float(v[12 + u]) + bo_;
                const float ei = ex2_approx(xi_), ef = ex2_approx(xf_), eg = ex2_approx(xg_), eo = ex2_approx(xo_);
                const float pi = 1.f + ei, pf = 1.f + ef, pg = 1.f + eg;
                // cs' = sigmoid(f) cs + K sigmoid(i) tanh(g), K = -2 log2e, over one common denominator
                const float pig = pi * pg;
                const float num = fmaf(c[jl][uh * 4 + u], pig, fmaf(eg, 2.f * kLog2e, -2.f * kLog2e) * pf);
                const float cn = num * rcp_approx(pf * pig);
                c[jl][uh * 4 + u] = cn;
                const float ec = ex2_approx(cn);
                hv[uh * 4 + u] = (1.f - ec) * rcp_approx((1.f + eo) * (1.f + ec));        // sigmoid(o) tanh(c')
            }
            if (hb + 1 < 2 * UB) tmem_wait_ld();
            if (uh == 1) {
                const HiLo8 s = split8(hv);
                reinterpret_cast<uint4*>(sAhi + (IN / 8 + jb) * LBO_A)[row] = s.hi;
                reinterpret_cast<uint4*>(sAlo + (IN / 8 + jb) * LBO_A)[row] = s.lo;
                if (live) {
                    if (LAYER == 0) {
                        // layer-1 operand layout h0[tile][t][hi|lo][chunk][row][8]: a warp writes 512 contiguous bytes
                        __half* o = h0_out + ((((size_t)blockIdx.x * kT + t) * 2) * 16 + (dir * 8 + jb)) * (kRows * 8) + row * 8;
                        *reinterpret_cast<uint4*>(o) = s.hi;
                        *reinterpret_cast<uint4*>(o + 16 * kRows * 8) = s.lo;
                    } else if (step == C::STEPS - 1) {
                        float4* o = reinterpret_cast<float4*>(h16 + site * 128 + dir * kH + jb * 8);
                        o[0] = make_float4(hv[0], hv[1], hv[2], hv[3]); o[1] = make_float4(hv[4], hv[5], hv[6], hv[7]);
                    }
                }
            }
        }
        if (more) store_x();
    }

    // ---- teardown: nobody may still be reading TMEM / the peer's shared memory ----
    tc_fence_before();
    if (CG == 2) cluster_sync_all(); else __syncthreads();
    if (warp == 0) tmem_dealloc<CG>(tmem_base, kTmemCols);
}


__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ------------------------------------------------------------------------------------------------------------------
// Layer 0, "two groups per CTA" variant.  A clock64 trace of lstm_tc_kernel<0,2,2> (two independent CTAs per SM) shows a
// step period of 8100 cycles while the two co-resident CTAs alternate (one waits for its MMAs while the other runs its
// cell updates) and 10400 once later waves have drifted into phase: then both wait for the tensor pipe together and both
// fight for the MUFU pipe together.  Here the alternation is built in: one CTA per SM holds TWO 128-site groups
// (16 warps, 2 x 256 TMEM columns, one copy of this CTA's half of W), still paired with a second CTA through
// cta_group::2.  There is no cluster barrier: every warp reports "my part of the epilogue is done" on an mbarrier of the
// leader CTA (remote arrive from the peer), the leader's thread 0 of the group issues the 18 MMAs and tcgen05.commit
// multicasts completion to both CTAs.  A second pair of mbarriers passes a token between the two groups so that their
// MMA bursts strictly alternate.
constexpr int kP2GroupThreads = 256, kP2Threads = 2 * kP2GroupThreads;
struct P2Smem {
    static constexpr size_t b_bytes = (size_t)kTcK0 * 128 * 2;                  // this CTA's half of W, one of hi / lo
    static constexpr size_t a_bytes = (size_t)kTcK0 * kRows * 2;
    static constexpr size_t sc_bytes = (size_t)kTcIn0 * kRows * 2;
    static constexpr size_t a_stride = 2 * a_bytes + sc_bytes;
    static constexpr size_t off_bhi = 0, off_blo = b_bytes, off_a = 2 * b_bytes, off_bar = off_a + 2 * a_stride, total = off_bar + 128;
};

__global__ void __launch_bounds__(kP2Threads, 1)
lstm0_pair2_kernel(const unsigned char* __restrict__ blob, const int32_t* __restrict__ xi, const float* __restrict__ xf,
                   __half* __restrict__ h0_out, int64_t n, const int32_t* __restrict__ pos, int64_t pos_bias, int npass)
{
    // pos != nullptr: xi is the region's count tensor [L][18] and site j's window is its contiguous row span starting at
    // pos[j] - pos_bias (pos_bias = region_start + 16): the [n][33][18] feature tensor is never materialised
    using S = P2Smem;
    constexpr int K = kTcK0, IN = kTcIn0, KB = K / 16, RB = 128, UB = 4;
    constexpr uint32_t LBO_A = kRows * 16, LBO_B = RB * 16, SBO = 128;
    extern __shared__ __align__(1024) unsigned char smem[];
    const int grp = (int)threadIdx.x / kP2GroupThreads;
    const int tid = (int)threadIdx.x - grp * kP2GroupThreads, lane = tid & 31, warp = tid >> 5;
    unsigned char* sBhi = smem + S::off_bhi; unsigned char* sBlo = smem + S::off_blo;
    unsigned char* sAhi = smem + S::off_a + grp * S::a_stride; unsigned char* sAlo = sAhi + S::a_bytes; unsigned char* sAsc = sAlo + S::a_bytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::off_bar);
    uint64_t* barH = bars + grp;               // [0,1]  gates of this group complete (commit, multicast to both CTAs)
    uint64_t* barReady = bars + 2 + grp;       // [2,3]  leader CTA: all 16 warps of this group (both CTAs) finished their epilogue
    uint64_t* barTurn = bars + 4;              // [4,5]  leader CTA: token, barTurn[g] = "group g may issue"
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + S::off_bar + 64);

    const int quad = warp & 3, sub = warp >> 2;
    const int row = quad * 32 + lane;
    // Persistent: cluster k works in direction k & 1 on the tile quads k >> 1, k >> 1 + stride, ... (a quad = the four
    // 128-site tiles of one cluster: two groups in each of the two CTAs).  Weights, TMEM and barriers are set up once.
    const uint32_t cta_rank = cluster_ctarank();
    const int cluster_id = (int)(blockIdx.x >> 1);
    const int dir = cluster_id & 1;
    const int quad_stride = (int)(gridDim.x >> 2);
    const int n_quads = (int)((n + 4 * kRows - 1) / (4 * kRows));
    const int q0 = cluster_id >> 1;
    const int my_quads = q0 < n_quads ? (n_quads - q0 + quad_stride - 1) / quad_stride : 0;
    const int total_g = my_quads * kT;                          // this group's stream of (quad, step) pairs
    auto tile_of = [&](int qi) -> int64_t { return (int64_t)(q0 + qi * quad_stride) * 4 + (int64_t)cta_rank * 2 + grp; };

    if (threadIdx.x == 0) {
        mbar_init(bars + 0, 1); mbar_init(bars + 1, 1); mbar_init(bars + 2, 16); mbar_init(bars + 3, 16);
        mbar_init(bars + 4, 1); mbar_init(bars + 5, 1);
        fence_mbar_init();
    }
    if (threadIdx.x < 32) tmem_alloc<2>(tmem_slot, 512);
    {
        const uint4* ghi = reinterpret_cast<const uint4*>(blob + tc_off(0, dir, 0));
        const uint4* glo = reinterpret_cast<const uint4*>(blob + tc_off(0, dir, 1));
        uint4* dhi = reinterpret_cast<uint4*>(sBhi); uint4* dlo = reinterpret_cast<uint4*>(sBlo);
        for (int i = (int)threadIdx.x; i < (K / 8) * RB; i += kP2Threads) {
            const int ch = i / RB, r = i - ch * RB;
            const int g = ch * 256 + (int)cta_rank * RB + r;
            dhi[i] = __ldg(ghi + g); dlo[i] = __ldg(glo + g);
        }
        uint4* a = reinterpret_cast<uint4*>(sAhi);
        for (int i = tid; i < (int)(S::a_stride / 16); i += kP2GroupThreads) a[i] = make_uint4(0, 0, 0, 0);
    }
    __syncthreads();

    float c[UB][8];
#pragma unroll
    for (int j = 0; j < UB; ++j)
#pragma unroll
        for (int u = 0; u < 8; ++u) c[j][u] = 0.f;

    int2 xraw[8];
    int64_t win0 = 0;                                           // first row of this thread's window in the count tensor
    auto load_x = [&](int gstep) {                              // count row of stream element gstep
        const int qi = gstep / kT, st = gstep - qi * kT;
        const int t = dir == 0 ? st : (kT - 1 - st);
        int64_t site = tile_of(qi) * kRows + row;
        if (site >= n) site = n - 1;
        if (pos && st == 0) win0 = (int64_t)__ldg(pos + site) - pos_bias;
        const int2* g = pos ? reinterpret_cast<const int2*>(xi + (win0 + t) * kF)
                            : reinterpret_cast<const int2*>(xi ? (const void*)(xi + (site * kT + t) * kF) : (const void*)(xf + (site * kT + t) * kF));
        if (sub == 0) {
#pragma unroll
            for (int j = 0; j < 8; ++j) xraw[j] = ldg_nc_volatile(g + j);
        } else {
            xraw[0] = ldg_nc_volatile(g + 8);
        }
    };
    auto xval = [&](int j) -> float {
        const int2 p = xraw[j >> 1];
        const int b = (j & 1) ? p.y : p.x;
        return xi ? (float)b : __int_as_float(b);
    };
    auto store_x = [&]() {
        if (sub == 0) {
#pragma unroll
            for (int ch = 0; ch < 2; ++ch) {
                float v[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) v[j] = xval(ch * 8 + j);
                const HiLo8 sp = split8(v);
                reinterpret_cast<uint4*>(sAhi + ch * LBO_A)[row] = sp.hi;
                reinterpret_cast<uint4*>(sAlo + ch * LBO_A)[row] = sp.lo;
                reinterpret_cast<uint4*>(sAsc + ch * LBO_A)[row] = scale_hi(sp.hi);
            }
        } else {
            const float v[8] = {xval(0), xval(1), 1.0f, 0.f, 0.f, 0.f, 0.f, 0.f};  // x16, x17, bias column
            const HiLo8 sp = split8(v);
            reinterpret_cast<uint4*>(sAhi + 2 * LBO_A)[row] = sp.hi;
            reinterpret_cast<uint4*>(sAlo + 2 * LBO_A)[row] = sp.lo;
            reinterpret_cast<uint4*>(sAsc + 2 * LBO_A)[row] = scale_hi(sp.hi);
        }
    };
    // "this warp's operand rows are written and its TMEM reads have retired": one arrival per warp on the leader's barrier
    auto report_ready = [&]() {
        fence_async_smem();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_remote_relaxed(barReady, 0);      // the leader maps to itself
    };
    if (total_g > 0) { load_x(0); store_x(); }
    tc_fence_before();
    cluster_sync_all();                                            // barriers initialised, operands zeroed, TMEM allocated (both CTAs)
    tc_fence_after();
    if (total_g > 0) report_ready();

    const uint32_t tmem_base = *tmem_slot + (uint32_t)grp * 256u;
    const uint32_t a_hi = smem_u32(sAhi), a_lo = smem_u32(sAlo), a_sc = smem_u32(sAsc), b_hi = smem_u32(sBhi), b_lo = smem_u32(sBlo);
    constexpr uint32_t idesc = make_idesc(256, 256);
    const bool issuer = cta_rank == 0 && tid == 0;
    uint32_t phaseH = 0, phaseR = 0, phaseT = 0;
    if (cta_rank == 0 && threadIdx.x == 0) mbar_arrive(barTurn + 0);          // group 0 issues first

    int step = 0, qi = 0;
    for (int g = 0; g < total_g; ++g) {
        const int t = dir == 0 ? step : (kT - 1 - step);
        const bool more = g + 1 < total_g;
        const int64_t tile_idx = tile_of(qi);
        const bool live = tile_idx * kRows + row < n;
        if (step == 0) {                                            // a new tile: the recurrence starts from c = 0, h = 0
#pragma unroll
            for (int j = 0; j < UB; ++j)
#pragma unroll
                for (int u = 0; u < 8; ++u) c[j][u] = 0.f;
        }
        if (issuer) {
            mbar_wait_cluster(barReady, phaseR);                   // every warp of this group, in both CTAs, has reported
            mbar_wait(barTurn + grp, phaseT);                      // and it is this group's turn on the tensor pipe
            tc_fence_after();
#pragma unroll 1
            for (int pass = 0; pass < npass; ++pass) {
#pragma unroll 1
                for (int kb = 0; kb < (step == 0 ? IN / 16 : KB); ++kb) {      // h = 0 at the first step of a tile: input k-blocks only
                    uint32_t aa = pass == 2 ? a_lo : a_hi;
                    if (pass == 1 && kb < IN / 16) aa = a_sc;
                    const uint32_t bb = pass == 1 ? b_lo : b_hi;
                    umma_f16<2>(tmem_base, make_desc(aa + kb * 2 * LBO_A, LBO_A, SBO), make_desc(bb + kb * 2 * LBO_B, LBO_B, SBO), idesc,
                                (pass | kb) ? 1u : 0u);
                }
            }
            umma_commit<2>(barH);
            mbar_arrive(barTurn + (grp ^ 1));                      // hand the token to the other group
        }
        phaseR ^= 1; phaseT ^= 1;
        if (more) load_x(g + 1);
        mbar_wait(barH, phaseH);
        phaseH ^= 1;
        tc_fence_after();

        uint32_t vb[2][16];
        const uint32_t tacc = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(sub * UB) * 32u;
        tmem_ld16_nowait(tacc, vb[0]);
        tmem_wait_ld();
        float hv[8];
#pragma unroll
        for (int hb = 0; hb < 2 * UB; ++hb) {
            const int jl = hb >> 1, uh = hb & 1, jb = sub * UB + jl;
            if (hb + 1 < 2 * UB) tmem_ld16_nowait(tacc + (hb + 1) * 16, vb[(hb + 1) & 1]);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const uint32_t* v = vb[hb & 1];
                // same cell update as lstm_tc_kernel (scales folded into the weights, scaled cell state)
                const float xi_ = fminf(__uint_as_float(v[u]), 36.f), xf_ = fminf(__uint_as_float(v[4 + u]), 36.f);
                const float xg_ = fminf(__uint_as_float(v[8 + u]), 36.f), xo_ = __uint_as_float(v[12 + u]);
                const float ei = ex2_approx(xi_), ef = ex2_approx(xf_), eg = ex2_approx(xg_), eo = ex2_approx(xo_);
                const float pi = 1.f + ei, pf = 1.f + ef, pg = 1.f + eg;
                const float pig = pi * pg;
                const float num = fmaf(c[jl][uh * 4 + u], pig, fmaf(eg, 2.f * kLog2e, -2.f * kLog2e) * pf);
                const float cn = num * rcp_approx(pf * pig);
                c[jl][uh * 4 + u] = cn;
                const float ec = ex2_approx(cn);
                hv[uh * 4 + u] = (1.f - ec) * rcp_approx((1.f + eo) * (1.f + ec));
            }
            if (hb + 1 < 2 * UB) tmem_wait_ld();
            if (uh == 1) {
                const HiLo8 sp = split8(hv);
                reinterpret_cast<uint4*>(sAhi + (IN / 8 + jb) * LBO_A)[row] = sp.hi;
                if (npass == 3) reinterpret_cast<uint4*>(sAlo + (IN / 8 + jb) * LBO_A)[row] = sp.lo;
                if (live) {
                    __half* o = h0_out + ((((size_t)tile_idx * kT + t) * 2) * 16 + (dir * 8 + jb)) * (kRows * 8) + row * 8;
                    *reinterpret_cast<uint4*>(o) = sp.hi;
                    if (npass == 3) *reinterpret_cast<uint4*>(o + 16 * kRows * 8) = sp.lo;     // single pass: layer 1 reads the hi halves only
                }
            }
        }
        if (more) { store_x(); report_ready(); }
        if (++step == kT) { step = 0; ++qi; }
    }

    tc_fence_before();
    cluster_sync_all();
    if (threadIdx.x < 32) tmem_dealloc<2>(*tmem_slot, 512);
}

// ------------------------------------------------------------------------------------------------------------------
// Layer 1, single-pass (NSNP_PREC_F16X1) variant with the same two-groups-per-CTA alternation.  With one fp16 pass only the
// hi halves of W and of the operands are needed: this CTA's half of W (48 KB) + two 128-site operand buffers (48 KB each) fit
// one SM, and layer 1 stops being a serial "12 MMAs, then the cell update" chain per SM (lstm_tc_kernel<1> with one pass:
// 2,300 + 4,150 cycles per step, MUFU pipe 55 % busy): one group's MMAs run under the other group's cell update.
// The input rows of a step (layer-0 output, already in operand layout: 32 KB per tile and position) arrive by one bulk copy
// per group and CTA, issued as soon as the MMAs that read the previous rows have completed; the warp that issued it waits for
// the copy before it reports the group ready.  Same MMA order and cell arithmetic as lstm_tc_kernel<1> with npass = 1:
// bit-identical output.
struct P2Smem1 {
    static constexpr size_t b_bytes = (size_t)kTcK1 * 128 * 2;                  // this CTA's half of W (hi)
    static constexpr size_t a_bytes = (size_t)kTcK1 * kRows * 2;               // one group's operand (hi): 128 input + 64 hidden columns
    static constexpr size_t off_b = 0, off_a = b_bytes, off_bias = off_a + 2 * a_bytes, off_bar = off_bias + 256 * sizeof(float), total = off_bar + 128;
};

__global__ void __launch_bounds__(kP2Threads, 1)
lstm1_pair2_kernel(const unsigned char* __restrict__ blob, const __half* __restrict__ h0_in, float* __restrict__ h16, int64_t n)
{
    using S = P2Smem1;
    constexpr int K = kTcK1, IN = kTcIn1, KB = K / 16, XB = IN / 16, RB = 128, UB = 4, kS = TcCfg<1>::STEPS;
    constexpr uint32_t LBO_A = kRows * 16, LBO_B = RB * 16, SBO = 128;
    constexpr uint32_t kPartBytes = 16u * kRows * 16u;              // 32 KB: the hi half of one (tile, position) of the layer-0 output
    extern __shared__ __align__(1024) unsigned char smem[];
    const int grp = (int)threadIdx.x / kP2GroupThreads;
    const int tid = (int)threadIdx.x - grp * kP2GroupThreads, lane = tid & 31, warp = tid >> 5;
    unsigned char* sB = smem + S::off_b;
    unsigned char* sA = smem + S::off_a + grp * S::a_bytes;
    float* sBias = reinterpret_cast<float*>(smem + S::off_bias);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::off_bar);
    uint64_t* barH = bars + grp;               // [0,1]  gates of this group complete (commit, multicast to both CTAs)
    uint64_t* barReady = bars + 2 + grp;       // [2,3]  leader CTA: all 16 warps of this group (both CTAs) are ready for the next step
    uint64_t* barTurn = bars + 4;              // [4,5]  leader CTA: token, barTurn[g] = "group g may issue"
    uint64_t* barIn = bars + 6 + grp;          // [6,7]  this CTA: the input rows of this group's next step have landed
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + S::off_bar + 64);

    const int quad = warp & 3, sub = warp >> 2;
    const int row = quad * 32 + lane;
    const uint32_t cta_rank = cluster_ctarank();
    const int cluster_id = (int)(blockIdx.x >> 1);
    const int dir = cluster_id & 1;
    const int quad_stride = (int)(gridDim.x >> 2);
    const int n_quads = (int)((n + 4 * kRows - 1) / (4 * kRows));
    const int64_t last_tile = (n + kRows - 1) / kRows - 1;
    const int q0 = cluster_id >> 1;
    const int my_quads = q0 < n_quads ? (n_quads - q0 + quad_stride - 1) / quad_stride : 0;
    const int total_g = my_quads * kS;                          // this group's stream of (quad, step) pairs
    auto tile_of = [&](int qi) -> int64_t { return (int64_t)(q0 + qi * quad_stride) * 4 + (int64_t)cta_rank * 2 + grp; };

    if (threadIdx.x == 0) {
        mbar_init(bars + 0, 1); mbar_init(bars + 1, 1); mbar_init(bars + 2, 16); mbar_init(bars + 3, 16);
        mbar_init(bars + 4, 1); mbar_init(bars + 5, 1); mbar_init(bars + 6, 1); mbar_init(bars + 7, 1);
        fence_mbar_init();
    }
    if (threadIdx.x < 32) tmem_alloc<2>(tmem_slot, 512);
    {
        const uint4* ghi = reinterpret_cast<const uint4*>(blob + tc_off(1, dir, 0));
        uint4* dhi = reinterpret_cast<uint4*>(sB);
        for (int i = (int)threadIdx.x; i < (K / 8) * RB; i += kP2Threads) {
            const int ch = i / RB, r = i - ch * RB;
            dhi[i] = __ldg(ghi + ch * 256 + (int)cta_rank * RB + r);
        }
        const float* gb = reinterpret_cast<const float*>(blob + kOffTcBias1) + dir * 256;
        for (int i = (int)threadIdx.x; i < 256; i += kP2Threads) sBias[i] = __ldg(gb + i);
    }
    __syncthreads();

    float c[UB][8];
#pragma unroll
    for (int j = 0; j < UB; ++j)
#pragma unroll
        for (int u = 0; u < 8; ++u) c[j][u] = 0.f;

    // input rows of stream element gstep: h0[tile][t][hi][16 chunks][128 rows][8]; a padding tile re-reads the last real one
    auto stage_in = [&](int gstep) {                            // one thread per group and CTA
        const int qi = gstep / kS, st = gstep - qi * kS;
        const int t = dir == 0 ? st : (kT - 1 - st);
        const int64_t tile = min(tile_of(qi), last_tile);
        mbar_expect_tx(barIn, kPartBytes);
        bulk_g2s(sA, h0_in + ((size_t)tile * kT + t) * (size_t)kPartBytes, kPartBytes, barIn);     // kPartBytes halfs = hi + lo per (tile, t)
    };
    auto report_ready = [&]() {
        fence_async_smem();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_remote_relaxed(barReady, 0);      // the leader maps to itself
    };
    uint32_t phaseIn = 0;
    if (total_g > 0 && tid == 0) stage_in(0);
    tc_fence_before();
    cluster_sync_all();                                            // barriers initialised, TMEM allocated (both CTAs)
    tc_fence_after();
    if (total_g > 0) {
        if (warp == 0) { mbar_wait(barIn, phaseIn); phaseIn ^= 1; }
        report_ready();
    }

    const uint32_t tmem_base = *tmem_slot + (uint32_t)grp * 256u;
    const uint32_t a_hi = smem_u32(sA), b_hi = smem_u32(sB);
    constexpr uint32_t idesc = make_idesc(256, 256);
    const bool issuer = cta_rank == 0 && tid == 0;
    uint32_t phaseH = 0, phaseR = 0, phaseT = 0;
    if (cta_rank == 0 && threadIdx.x == 0) mbar_arrive(barTurn + 0);          // group 0 issues first

    int step = 0, qi = 0;
    for (int g = 0; g < total_g; ++g) {
        const bool more = g + 1 < total_g;
        const int64_t site = tile_of(qi) * kRows + row;
        const bool live = site < n;
        if (step == 0) {                                            // a new tile: the recurrence starts from c = 0, h = 0
#pragma unroll
            for (int j = 0; j < UB; ++j)
#pragma unroll
                for (int u = 0; u < 8; ++u) c[j][u] = 0.f;
        }
        if (issuer) {
            mbar_wait_cluster(barReady, phaseR);                   // every warp of this group, in both CTAs, has reported
            mbar_wait(barTurn + grp, phaseT);                      // and it is this group's turn on the tensor pipe
            tc_fence_after();
#pragma unroll 1
            for (int kb = 0; kb < (step == 0 ? XB : KB); ++kb)      // h = 0 at the first step of a tile: input k-blocks only
                umma_f16<2>(tmem_base, make_desc(a_hi + kb * 2 * LBO_A, LBO_A, SBO), make_desc(b_hi + kb * 2 * LBO_B, LBO_B, SBO), idesc, kb ? 1u : 0u);
            umma_commit<2>(barH);
            mbar_arrive(barTurn + (grp ^ 1));                      // hand the token to the other group
        }
        phaseR ^= 1; phaseT ^= 1;
        mbar_wait(barH, phaseH);
        phaseH ^= 1;
        tc_fence_after();
        if (more && tid == 0) stage_in(g + 1);                      // the MMAs that read the input rows are complete: fetch the next ones

        uint32_t vb[2][16];
        const uint32_t tacc = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(sub * UB) * 32u;
        tmem_ld16_nowait(tacc, vb[0]);
        tmem_wait_ld();
        float hv[8];
#pragma unroll
        for (int hb = 0; hb < 2 * UB; ++hb) {
            const int jl = hb >> 1, uh = hb & 1, jb = sub * UB + jl;
            if (hb + 1 < 2 * UB) tmem_ld16_nowait(tacc + (hb + 1) * 16, vb[(hb + 1) & 1]);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const uint32_t* v = vb[hb & 1];
                // same cell update as lstm_tc_kernel<1> (scales folded into the weights, scaled cell state, bias in the epilogue)
                const float* bq = sBias + jb * 32 + uh * 16 + u;
                const float xi_ = fminf(__uint_as_float(v[u]) + bq[0], 36.f), xf_ = fminf(__uint_as_float(v[4 + u]) + bq[4], 36.f);
                const float xg_ = fminf(__uint_as_float(v[8 + u]) + bq[8], 36.f), xo_ = __uint_as_float(v[12 + u]) + bq[12];
                const float ei = ex2_approx(xi_), ef = ex2_approx(xf_), eg = ex2_approx(xg_), eo = ex2_approx(xo_);
                const float pi = 1.f + ei, pf = 1.f + ef, pg = 1.f + eg;
                const float pig = pi * pg;
                const float num = fmaf(c[jl][uh * 4 + u], pig, fmaf(eg, 2.f * kLog2e, -2.f * kLog2e) * pf);
                const float cn = num * rcp_approx(pf * pig);
                c[jl][uh * 4 + u] = cn;
                const float ec = ex2_approx(cn);
                hv[uh * 4 + u] = (1.f - ec) * rcp_approx((1.f + eo) * (1.f + ec));
            }
            if (hb + 1 < 2 * UB) tmem_wait_ld();
            if (uh == 1) {
                const HiLo8 sp = split8(hv);
                reinterpret_cast<uint4*>(sA + (IN / 8 + jb) * LBO_A)[row] = sp.hi;
                if (live && step == kS - 1) {
                    float4* o = reinterpret_cast<float4*>(h16 + site * 128 + dir * kH + jb * 8);
                    o[0] = make_float4(hv[0], hv[1], hv[2], hv[3]); o[1] = make_float4(hv[4], hv[5], hv[6], hv[7]);
                }
            }
        }
        if (more) {
            if (warp == 0) { mbar_wait(barIn, phaseIn); phaseIn ^= 1; }
            report_ready();
        }
        if (++step == kS) { step = 0; ++qi; }
    }

    tc_fence_before();
    cluster_sync_all();
    if (threadIdx.x < 32) tmem_dealloc<2>(*tmem_slot, 512);
}

// ------------------------------------------------------------------------------------------------------------------
// Layer 1, three-pass (default NSNP_PREC_F16X3) variant with the same two-groups-per-CTA alternation.  Two groups' full
// operands (2 x 96 KB) next to W hi + lo (96 KB) would not fit, but the input part of the operand (the layer-0 output,
// 128 of the 192 columns) is only read during its own group's MMA burst and the bursts strictly alternate: the two groups
// share ONE input buffer and keep only their h part (64 columns, hi + lo) to themselves.  The input buffer is refilled
// per burst by a producer warp in two halves, each with a full and an empty mbarrier:
//     hi half (passes 0 and 1 read it): empty once pass 1 of the input part has completed -- the copy of the other group's
//             rows overlaps pass 2 and the 12 h-part MMAs;
//     lo half (pass 2 reads it): empty once pass 2 of the input part has completed.
// The full barriers exist per group (a group waits for its own rows only, one phase per step of that group); warp 0 of the
// group waits for them before it reports the group ready, so barReady covers "both CTAs' input rows have landed".  Same MMA
// order (input part: 3 passes over kb 0-7, then h part: 3 passes over kb 8-11) and cell arithmetic as lstm_tc_kernel<1>:
// bit-identical output.
constexpr int kP2x3Threads = kP2Threads + 32;                   // + the producer warp
struct P2Smem1x3 {
    static constexpr size_t b_bytes = (size_t)kTcK1 * 128 * 2;                  // this CTA's half of W, one of hi / lo
    static constexpr size_t in_bytes = (size_t)kTcIn1 * kRows * 2;             // input part, one of hi / lo (shared by both groups)
    static constexpr size_t h_bytes = (size_t)kH * kRows * 2;                  // one group's h part, one of hi / lo
    static constexpr size_t off_bhi = 0, off_blo = b_bytes, off_in = 2 * b_bytes, off_h = off_in + 2 * in_bytes,
                            off_bias = off_h + 4 * h_bytes, off_bar = off_bias + 256 * sizeof(float), total = off_bar + 128;
};
static_assert(P2Smem1x3::total <= 232448, "lstm1_pair2x3_kernel: shared memory above the per-block opt-in limit");

__global__ void __launch_bounds__(kP2x3Threads, 1)
lstm1_pair2x3_kernel(const unsigned char* __restrict__ blob, const __half* __restrict__ h0_in, float* __restrict__ h16, int64_t n)
{
    using S = P2Smem1x3;
    constexpr int K = kTcK1, IN = kTcIn1, KB = K / 16, XB = IN / 16, RB = 128, UB = 4, kS = TcCfg<1>::STEPS;
    constexpr uint32_t LBO_A = kRows * 16, LBO_B = RB * 16, SBO = 128;
    constexpr uint32_t kPartBytes = 16u * kRows * 16u;              // 32 KB: the hi (or lo) half of one (tile, position) of the layer-0 output
    extern __shared__ __align__(1024) unsigned char smem[];
    const bool producer = threadIdx.x >= kP2Threads;               // warp-uniform
    const int grp = producer ? 0 : (int)threadIdx.x / kP2GroupThreads;
    const int tid = (int)threadIdx.x - grp * kP2GroupThreads, lane = tid & 31, warp = tid >> 5;
    unsigned char* sBhi = smem + S::off_bhi; unsigned char* sBlo = smem + S::off_blo;
    unsigned char* sInHi = smem + S::off_in; unsigned char* sInLo = sInHi + S::in_bytes;
    unsigned char* sHhi = smem + S::off_h + grp * 2 * S::h_bytes; unsigned char* sHlo = sHhi + S::h_bytes;
    float* sBias = reinterpret_cast<float*>(smem + S::off_bias);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::off_bar);
    uint64_t* barH = bars + grp;               // [0,1]   gates of this group complete (commit, multicast to both CTAs)
    uint64_t* barReady = bars + 2 + grp;       // [2,3]   leader CTA: all 16 warps of this group (both CTAs) are ready, input rows landed
    uint64_t* barTurn = bars + 4;              // [4,5]   leader CTA: token, barTurn[g] = "group g may issue"
    uint64_t* barHiFull = bars + 6;            // [6,7]   this CTA: the hi input rows of group g's next step have landed
    uint64_t* barLoFull = bars + 8;            // [8,9]   this CTA: the lo input rows of group g's next step have landed
    uint64_t* barHiEmpty = bars + 10;          // [10]    passes 0 and 1 of the last burst's input part are complete (multicast)
    uint64_t* barLoEmpty = bars + 11;          // [11]    pass 2 of the last burst's input part is complete (multicast)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + S::off_bar + 96);

    const int quad = warp & 3, sub = warp >> 2;
    const int row = quad * 32 + lane;
    const uint32_t cta_rank = cluster_ctarank();
    const int cluster_id = (int)(blockIdx.x >> 1);
    const int dir = cluster_id & 1;
    const int quad_stride = (int)(gridDim.x >> 2);
    const int n_quads = (int)((n + 4 * kRows - 1) / (4 * kRows));
    const int64_t last_tile = (n + kRows - 1) / kRows - 1;
    const int q0 = cluster_id >> 1;
    const int my_quads = q0 < n_quads ? (n_quads - q0 + quad_stride - 1) / quad_stride : 0;
    const int total_g = my_quads * kS;                          // each group's stream of (quad, step) pairs; bursts alternate g0, g1, g0, ...
    auto tile_of = [&](int qi, int g) -> int64_t { return (int64_t)(q0 + qi * quad_stride) * 4 + (int64_t)cta_rank * 2 + g; };

    if (threadIdx.x == 0) {
        mbar_init(bars + 0, 1); mbar_init(bars + 1, 1); mbar_init(bars + 2, 16); mbar_init(bars + 3, 16);
        for (int i = 4; i < 12; ++i) mbar_init(bars + i, 1);
        fence_mbar_init();
    }
    if (threadIdx.x < 32) tmem_alloc<2>(tmem_slot, 512);
    {
        const uint4* ghi = reinterpret_cast<const uint4*>(blob + tc_off(1, dir, 0));
        const uint4* glo = reinterpret_cast<const uint4*>(blob + tc_off(1, dir, 1));
        uint4* dhi = reinterpret_cast<uint4*>(sBhi); uint4* dlo = reinterpret_cast<uint4*>(sBlo);
        for (int i = (int)threadIdx.x; i < (K / 8) * RB; i += kP2x3Threads) {
            const int ch = i / RB, r = i - ch * RB;
            const int g = ch * 256 + (int)cta_rank * RB + r;
            dhi[i] = __ldg(ghi + g); dlo[i] = __ldg(glo + g);
        }
        const float* gb = reinterpret_cast<const float*>(blob + kOffTcBias1) + dir * 256;
        for (int i = (int)threadIdx.x; i < 256; i += kP2x3Threads) sBias[i] = __ldg(gb + i);
    }
    __syncthreads();

    // input rows of burst b (group b & 1, its stream element b >> 1): h0[tile][t][hi|lo][16 chunks][128 rows][8];
    // a padding tile re-reads the last real one
    auto rows_of = [&](int b) -> const __half* {
        const int gs = b >> 1, qi = gs / kS, st = gs - qi * kS;
        const int t = dir == 0 ? st : (kT - 1 - st);
        const int64_t tile = min(tile_of(qi, b & 1), last_tile);
        return h0_in + ((size_t)tile * kT + t) * (size_t)kPartBytes;       // kPartBytes halfs = hi + lo per (tile, t)
    };
    const int total_b = 2 * total_g;
    if (producer && lane == 0 && total_b > 0) {                 // the first burst's rows: the buffer is free
        const __half* src = rows_of(0);
        mbar_expect_tx(barHiFull, kPartBytes); bulk_g2s(sInHi, src, kPartBytes, barHiFull);
        mbar_expect_tx(barLoFull, kPartBytes); bulk_g2s(sInLo, src + kPartBytes / 2, kPartBytes, barLoFull);
        if (total_b > 1) bulk_prefetch_l2(rows_of(1), 2 * kPartBytes);
    }
    auto report_ready = [&]() {
        fence_async_smem();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_remote_relaxed(barReady, 0);      // the leader maps to itself
    };
    uint32_t phaseIn = 0;                                           // parity of this group's full barriers
    auto wait_input = [&]() {                                       // warp 0 of a group: both halves of its next rows have landed
        mbar_wait(barHiFull + grp, phaseIn);
        mbar_wait(barLoFull + grp, phaseIn);
        phaseIn ^= 1;
    };
    tc_fence_before();
    cluster_sync_all();                                            // barriers initialised, TMEM allocated (both CTAs)
    tc_fence_after();

    if (producer) {
        // producer warp: burst b's rows go into the buffer as soon as burst b - 1 has finished reading each half; it never
        // touches TMEM and skips the epilogue
        if (lane == 0) {
            for (int b = 1; b < total_b; ++b) {
                const __half* src = rows_of(b);
                uint64_t* full_hi = barHiFull + (b & 1); uint64_t* full_lo = barLoFull + (b & 1);
                mbar_wait(barHiEmpty, (uint32_t)((b - 1) & 1));
                mbar_expect_tx(full_hi, kPartBytes); bulk_g2s(sInHi, src, kPartBytes, full_hi);
                // the next burst's rows: pull them into L2 now, so that their copy (one burst from now) pays L2 latency instead of DRAM latency
                if (b + 1 < total_b) bulk_prefetch_l2(rows_of(b + 1), 2 * kPartBytes);
                mbar_wait(barLoEmpty, (uint32_t)((b - 1) & 1));
                mbar_expect_tx(full_lo, kPartBytes); bulk_g2s(sInLo, src + kPartBytes / 2, kPartBytes, full_lo);
            }
        }
        __syncwarp();
    } else {
        float c[UB][8];
#pragma unroll
        for (int j = 0; j < UB; ++j)
#pragma unroll
            for (int u = 0; u < 8; ++u) c[j][u] = 0.f;

        if (total_g > 0) {
            if (warp == 0) wait_input();
            report_ready();
        }

        const uint32_t tmem_base = *tmem_slot + (uint32_t)grp * 256u;
        const uint32_t in_hi = smem_u32(sInHi), in_lo = smem_u32(sInLo), h_hi = smem_u32(sHhi), h_lo = smem_u32(sHlo);
        const uint32_t b_hi = smem_u32(sBhi), b_lo = smem_u32(sBlo);
        constexpr uint32_t idesc = make_idesc(256, 256);
        const bool issuer = cta_rank == 0 && tid == 0;
        uint32_t phaseH = 0, phaseR = 0, phaseT = 0;
        if (cta_rank == 0 && threadIdx.x == 0) mbar_arrive(barTurn + 0);          // group 0 issues first

        int step = 0, qi = 0;
        for (int g = 0; g < total_g; ++g) {
            const bool more = g + 1 < total_g;
            const int64_t site = tile_of(qi, grp) * kRows + row;
            const bool live = site < n;
            float* const out = h16 + site * 128 + dir * kH + sub * UB * 8;      // this thread's hidden units of the t = 16 state
            if (step == 0) {                                        // a new tile: the recurrence starts from c = 0, h = 0
#pragma unroll
                for (int j = 0; j < UB; ++j)
#pragma unroll
                    for (int u = 0; u < 8; ++u) c[j][u] = 0.f;
            }
            if (issuer) {
                const bool refill = more || grp == 0;              // another burst follows this one
                mbar_wait_cluster(barReady, phaseR);               // every warp of this group, in both CTAs, has reported
                mbar_wait(barTurn + grp, phaseT);                  // and it is this group's turn on the tensor pipe
                tc_fence_after();
                // pass 0: a_hi.w_hi   pass 1: a_hi.w_lo   pass 2: a_lo.w_hi; input part first, then the h part
#pragma unroll 1
                for (int pass = 0; pass < 3; ++pass) {
#pragma unroll 1
                    for (int kb = 0; kb < XB; ++kb)
                        umma_f16<2>(tmem_base, make_desc((pass == 2 ? in_lo : in_hi) + kb * 2 * LBO_A, LBO_A, SBO),
                                    make_desc((pass == 1 ? b_lo : b_hi) + kb * 2 * LBO_B, LBO_B, SBO), idesc, (pass | kb) ? 1u : 0u);
                    if (pass == 1 && refill) umma_commit<2>(barHiEmpty);     // the hi input rows are read: the producer may refill them
                }
                if (refill) umma_commit<2>(barLoEmpty);
                if (step > 0) {                                    // h = 0 at the first step of a tile: input k-blocks only
#pragma unroll 1
                    for (int pass = 0; pass < 3; ++pass) {
#pragma unroll 1
                        for (int kb = XB; kb < KB; ++kb)
                            umma_f16<2>(tmem_base, make_desc((pass == 2 ? h_lo : h_hi) + (kb - XB) * 2 * LBO_A, LBO_A, SBO),
                                        make_desc((pass == 1 ? b_lo : b_hi) + kb * 2 * LBO_B, LBO_B, SBO), idesc, 1u);
                    }
                }
                umma_commit<2>(barH);
                mbar_arrive(barTurn + (grp ^ 1));                  // hand the token to the other group
            }
            phaseR ^= 1; phaseT ^= 1;
            mbar_wait(barH, phaseH);
            phaseH ^= 1;
            tc_fence_after();

            uint32_t vb[2][16];
            const uint32_t tacc = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(sub * UB) * 32u;
            tmem_ld16_nowait(tacc, vb[0]);
            tmem_wait_ld();
            float hv[8];
#pragma unroll
            for (int hb = 0; hb < 2 * UB; ++hb) {
                const int jl = hb >> 1, uh = hb & 1, jb = sub * UB + jl;
                if (hb + 1 < 2 * UB) tmem_ld16_nowait(tacc + (hb + 1) * 16, vb[(hb + 1) & 1]);
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const uint32_t* v = vb[hb & 1];
                    // same cell update as lstm_tc_kernel<1> (scales folded into the weights, scaled cell state, bias in the epilogue)
                    const float* bq = sBias + jb * 32 + uh * 16 + u;
                    const float xi_ = fminf(__uint_as_float(v[u]) + bq[0], 36.f), xf_ = fminf(__uint_as_float(v[4 + u]) + bq[4], 36.f);
                    const float xg_ = fminf(__uint_as_float(v[8 + u]) + bq[8], 36.f), xo_ = __uint_as_float(v[12 + u]) + bq[12];
                    const float ei = ex2_approx(xi_), ef = ex2_approx(xf_), eg = ex2_approx(xg_), eo = ex2_approx(xo_);
                    const float pi = 1.f + ei, pf = 1.f + ef, pg = 1.f + eg;
                    const float pig = pi * pg;
                    const float num = fmaf(c[jl][uh * 4 + u], pig, fmaf(eg, 2.f * kLog2e, -2.f * kLog2e) * pf);
                    const float cn = num * rcp_approx(pf * pig);
                    c[jl][uh * 4 + u] = cn;
                    const float ec = ex2_approx(cn);
                    hv[uh * 4 + u] = (1.f - ec) * rcp_approx((1.f + eo) * (1.f + ec));
                }
                if (hb + 1 < 2 * UB) tmem_wait_ld();
                if (uh == 1) {
                    const HiLo8 sp = split8(hv);
                    reinterpret_cast<uint4*>(sHhi + jb * LBO_A)[row] = sp.hi;
                    reinterpret_cast<uint4*>(sHlo + jb * LBO_A)[row] = sp.lo;
                    if (live && step == kS - 1) {
                        float4* o = reinterpret_cast<float4*>(out + jl * 8);
                        o[0] = make_float4(hv[0], hv[1], hv[2], hv[3]); o[1] = make_float4(hv[4], hv[5], hv[6], hv[7]);
                    }
                }
            }
            if (more) {
                if (warp == 0) wait_input();
                report_ready();
            }
            if (++step == kS) { step = 0; ++qi; }
        }
    }

    tc_fence_before();
    cluster_sync_all();
    if (threadIdx.x < 32) tmem_dealloc<2>(*tmem_slot, 512);
}

template <class Kern, class... Args>
int launch_pair2(Kern kern, const char* name, size_t smem_bytes, int threads, int64_t m, cudaStream_t stream, Args... args) {
    // persistent: at most one CTA per SM; clusters alternate between the two directions, so an even number of clusters
    const unsigned quads = (unsigned)((m + 4 * kRows - 1) / (4 * kRows));
    unsigned clusters = 2 * quads; if (clusters > (unsigned)kNumSMs / 2) clusters = ((unsigned)kNumSMs / 2) & ~1u;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * clusters, 1, 1);
    cfg.blockDim = dim3((unsigned)threads, 1, 1);
    cfg.dynamicSmemBytes = smem_bytes;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kern, args...);
    if (e != cudaSuccess) return set_error(NSNP_E_CUDA, "%s: %s", name, cudaGetErrorString(e));
    return NSNP_OK;
}

int launch_l0_pair2(const void* blob, const int32_t* xi, const float* xf, void* h0_out, int64_t m, const int32_t* pos, int64_t pos_bias, int npass, cudaStream_t stream) {
    static bool attr_done = false;
    if (!attr_done) {
        if (cudaFuncSetAttribute(lstm0_pair2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P2Smem::total) != cudaSuccess)
            return cuda_status("cudaFuncSetAttribute(lstm0_pair2_kernel)");
        attr_done = true;
    }
    return launch_pair2(lstm0_pair2_kernel, "lstm0_pair2_kernel", P2Smem::total, kP2Threads, m, stream, (const unsigned char*)blob, xi, xf, (__half*)h0_out, m, pos, pos_bias, npass);
}

int launch_l1_pair2(const void* blob, const void* h0_in, float* h16, int64_t m, cudaStream_t stream) {
    static bool attr_done = false;
    if (!attr_done) {
        if (cudaFuncSetAttribute(lstm1_pair2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P2Smem1::total) != cudaSuccess)
            return cuda_status("cudaFuncSetAttribute(lstm1_pair2_kernel)");
        attr_done = true;
    }
    return launch_pair2(lstm1_pair2_kernel, "lstm1_pair2_kernel", P2Smem1::total, kP2Threads, m, stream, (const unsigned char*)blob, (const __half*)h0_in, h16, m);
}

int launch_l1_pair2x3(const void* blob, const void* h0_in, float* h16, int64_t m, cudaStream_t stream) {
    static bool attr_done = false;
    if (!attr_done) {
        if (cudaFuncSetAttribute(lstm1_pair2x3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P2Smem1x3::total) != cudaSuccess)
            return cuda_status("cudaFuncSetAttribute(lstm1_pair2x3_kernel)");
        attr_done = true;
    }
    return launch_pair2(lstm1_pair2x3_kernel, "lstm1_pair2x3_kernel", P2Smem1x3::total, kP2x3Threads, m, stream, (const unsigned char*)blob, (const __half*)h0_in, h16, m);
}

// ------------------------------------------------------------------------------------------------------------------
// Tail: probabilities from the t = 16 state (model.py:36-39,66-73 with output_proj folded into dense).
//   d[128 sites x 256] = h16[128 x 128] . W'^T     24 tcgen05.mma (8 k-blocks x 3 hi/lo passes), fp32 in TMEM
//   t = tanh(d + b'), logits = t . Wh + bh (24 = 21 genotype + 3 zygosity), two softmaxes.
// One persistent CTA per SM, W' (2 x 64 KB) resident.  Warp roles:
//   warps 0-7  epilogue: one site row x 128 dense outputs per thread; TMEM -> bias + tanh (1 ex2 + 1 rcp) -> 24 running
//              dot products against Wh (shared-memory broadcasts); the two halves of a row meet in a small exchange
//              buffer; softmax -> global.
//   warps 8-11 loaders: the next tile's h16 rows -> fp16 hi/lo operand in shared memory
//   warp  12   MMA issuer.
// TMEM is double buffered (2 x 256 columns): the MMAs of tile g+1 run under the epilogue of tile g.
constexpr int kTtEpiWarps = 8, kTtLoadWarps = 4;
constexpr int kTtThreads = (kTtEpiWarps + kTtLoadWarps + 1) * 32;
struct TailSmem {
    static constexpr size_t w_bytes = kTcBytesTail;                 // one of hi / lo
    static constexpr size_t a_bytes = (size_t)128 * kRows * 2;
    static constexpr size_t off_whi = 0, off_wlo = w_bytes, off_ahi = 2 * w_bytes, off_alo = off_ahi + a_bytes,
                            off_head = off_alo + a_bytes,            // float [256][24]
                            off_bias = off_head + 256 * 24 * 4,      // float [256] dense bias, float [24] head bias
                            off_xch = off_bias + (256 + 32) * 4,     // float [128][12] partial-logit exchange
                            off_bar = off_xch + 128 * 12 * 4, total = off_bar + 64;
};

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

__global__ void __launch_bounds__(kTtThreads, 1)
tail_tc_kernel(const unsigned char* __restrict__ blob, const float* __restrict__ h16, int64_t n_max, const int32_t* __restrict__ n_dev,
               float* __restrict__ gt, float* __restrict__ zy)
{
    using S = TailSmem;
    constexpr uint32_t LBO_A = kRows * 16, LBO_B = 256 * 16, SBO = 128;
    extern __shared__ __align__(1024) unsigned char smem[];
    unsigned char* sWhi = smem + S::off_whi; unsigned char* sWlo = smem + S::off_wlo;
    unsigned char* sAhi = smem + S::off_ahi; unsigned char* sAlo = smem + S::off_alo;
    float* sHead = reinterpret_cast<float*>(smem + S::off_head);
    float* sBias = reinterpret_cast<float*>(smem + S::off_bias);
    float* sXch = reinterpret_cast<float*>(smem + S::off_xch);
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + S::off_bar);     // [0,1] barH, [2] barIn, [3,4] barFree
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + S::off_bar + 48);
    uint64_t* barH = bar; uint64_t* barIn = bar + 2; uint64_t* barFree = bar + 3;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int64_t n = n_max;
    if (n_dev) { const int64_t nd = *n_dev; if (nd < n) n = nd; }
    const int n_tiles = (int)((n + kRows - 1) / kRows);
    const int my_tiles = (int)blockIdx.x < n_tiles ? (n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;

    if (tid == 0) {
        mbar_init(barH, 1); mbar_init(barH + 1, 1); mbar_init(barIn, kTtLoadWarps);
        mbar_init(barFree, kTtEpiWarps); mbar_init(barFree + 1, kTtEpiWarps);
        fence_mbar_init();
    }
    if (warp == 0) tmem_alloc<1>(tmem_slot, 512);
    {
        const uint4* ghi = reinterpret_cast<const uint4*>(blob + kOffTcTail);
        const uint4* glo = reinterpret_cast<const uint4*>(blob + kOffTcTail + kTcBytesTail);
        uint4* dhi = reinterpret_cast<uint4*>(sWhi); uint4* dlo = reinterpret_cast<uint4*>(sWlo);
        for (int i = tid; i < (int)(S::w_bytes / 16); i += kTtThreads) { dhi[i] = __ldg(ghi + i); dlo[i] = __ldg(glo + i); }
        const float* fb = reinterpret_cast<const float*>(blob);
        for (int i = tid; i < 256 * 24; i += kTtThreads) sHead[i] = __ldg(fb + kOffHeadW + i);
        for (int i = tid; i < 256; i += kTtThreads) sBias[i] = __ldg(fb + kOffDenseB + i);
        if (tid < 24) sBias[256 + tid] = __ldg(fb + kOffHeadB + tid);
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == kTtEpiWarps + kTtLoadWarps) {
        // ---- MMA issuer ----
        if (lane == 0) {
            const uint32_t a_hi = smem_u32(sAhi), a_lo = smem_u32(sAlo), b_hi = smem_u32(sWhi), b_lo = smem_u32(sWlo);
            constexpr uint32_t idesc = make_idesc(128, 256);
            for (int g = 0; g < my_tiles; ++g) {
                const int b = g & 1;
                mbar_wait(barIn, (uint32_t)(g & 1));                                     // operand of tile g staged
                if (g >= 2) mbar_wait(barFree + b, (uint32_t)(((g >> 1) - 1) & 1));      // accumulator b drained by tile g-2
                tc_fence_after();
                const uint32_t acc = tmem_base + (uint32_t)b * 256u;
#pragma unroll 1
                for (int kb = 0; kb < 8; ++kb) {
                    const uint64_t bh = make_desc(b_hi + kb * 2 * LBO_B, LBO_B, SBO), bl = make_desc(b_lo + kb * 2 * LBO_B, LBO_B, SBO);
                    const uint64_t ah = make_desc(a_hi + kb * 2 * LBO_A, LBO_A, SBO), al = make_desc(a_lo + kb * 2 * LBO_A, LBO_A, SBO);
                    umma_f16<1>(acc, ah, bh, idesc, kb == 0 ? 0u : 1u);
                    umma_f16<1>(acc, ah, bl, idesc, 1u);
                    umma_f16<1>(acc, al, bh, idesc, 1u);
                }
                umma_commit<1>(barH + b);
            }
        }
    } else if (warp >= kTtEpiWarps) {
        // ---- loaders: thread = one site row; 16 chunks of 8 values = two float4 loads each.  The accumulators are double
        //      buffered and the epilogue of a tile outlasts MMA + staging, so the loads need not be hoisted above the wait ----
        const int row = (warp - kTtEpiWarps) * 32 + lane;
        for (int g = 0; g < my_tiles; ++g) {
            const int tile = (int)blockIdx.x + g * (int)gridDim.x;
            int64_t site = (int64_t)tile * kRows + row; if (site >= n) site = n - 1;
            const float4* src = reinterpret_cast<const float4*>(h16 + site * 128);
            float4 pre[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) pre[i] = __ldg(src + i);
            if (g >= 1) mbar_wait(barH + ((g - 1) & 1), (uint32_t)(((g - 1) >> 1) & 1));    // the MMAs of the previous tile have read the operand
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {
                if (hf == 1) {
#pragma unroll
                    for (int i = 0; i < 16; ++i) pre[i] = __ldg(src + 16 + i);
                }
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const float v[8] = {pre[2 * c].x, pre[2 * c].y, pre[2 * c].z, pre[2 * c].w, pre[2 * c + 1].x, pre[2 * c + 1].y, pre[2 * c + 1].z, pre[2 * c + 1].w};
                    const HiLo8 sp = split8(v);
                    reinterpret_cast<uint4*>(sAhi + (hf * 8 + c) * LBO_A)[row] = sp.hi;
                    reinterpret_cast<uint4*>(sAlo + (hf * 8 + c) * LBO_A)[row] = sp.lo;
                }
            }
            fence_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(barIn);
        }
    } else {
        // ---- epilogue: warp & 3 = TMEM lane quadrant, warp >> 2 = half of the 256 dense outputs; thread = site row ----
        const int quad = warp & 3, half = warp >> 2;
        const int row = quad * 32 + lane;
        for (int g = 0; g < my_tiles; ++g) {
            const int b = g & 1;
            const int tile = (int)blockIdx.x + g * (int)gridDim.x;
            const int64_t site = (int64_t)tile * kRows + row;
            mbar_wait(barH + b, (uint32_t)((g >> 1) & 1));
            tc_fence_after();
            float lg[24];
#pragma unroll
            for (int j = 0; j < 24; ++j) lg[j] = half == 0 ? sBias[256 + j] : 0.f;
            uint32_t vb[2][16];
            const uint32_t tacc = tmem_base + (uint32_t)b * 256u + ((uint32_t)(quad * 32) << 16) + (uint32_t)half * 128u;
            tmem_ld16_nowait(tacc, vb[0]);
            tmem_wait_ld();
#pragma unroll 2
            for (int cb = 0; cb < 8; ++cb) {
                if (cb + 1 < 8) tmem_ld16_nowait(tacc + (cb + 1) * 16, vb[(cb + 1) & 1]);
                // tanh(d) = (1 - e) / (1 + e), e = exp(-2 d); d >= -20 keeps e finite (tanh(-20) = -1 to the last bit)
                float t[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const float d = fmaxf(__uint_as_float(vb[cb & 1][j]) + sBias[half * 128 + cb * 16 + j], -20.f);
                    const float e = ex2_approx(-2.f * kLog2e * d);
                    t[j] = (1.f - e) * rcp_approx(1.f + e);
                }
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const float4* wr = reinterpret_cast<const float4*>(sHead + (half * 128 + cb * 16 + j) * 24);
#pragma unroll
                    for (int q = 0; q < 6; ++q) {
                        const float4 w = wr[q];
                        lg[4 * q] = fmaf(t[j], w.x, lg[4 * q]); lg[4 * q + 1] = fmaf(t[j], w.y, lg[4 * q + 1]);
                        lg[4 * q + 2] = fmaf(t[j], w.z, lg[4 * q + 2]); lg[4 * q + 3] = fmaf(t[j], w.w, lg[4 * q + 3]);
                    }
                }
                if (cb + 1 < 8) tmem_wait_ld();
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(barFree + b);
            // the two halves of a quadrant add their partial logits through a 6 KB exchange buffer, 12 values per round
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                float4* x = reinterpret_cast<float4*>(sXch + row * 12);
                if (half == 1) {
#pragma unroll
                    for (int q = 0; q < 3; ++q) x[q] = make_float4(lg[12 * r + 4 * q], lg[12 * r + 4 * q + 1], lg[12 * r + 4 * q + 2], lg[12 * r + 4 * q + 3]);
                }
                named_bar_sync(1 + quad, 64);
                if (half == 0) {
#pragma unroll
                    for (int q = 0; q < 3; ++q) { const float4 v = x[q]; lg[12 * r + 4 * q] += v.x; lg[12 * r + 4 * q + 1] += v.y; lg[12 * r + 4 * q + 2] += v.z; lg[12 * r + 4 * q + 3] += v.w; }
                }
                named_bar_sync(1 + quad, 64);
            }
            if (half == 0 && site < n) {
                float m = lg[0];
#pragma unroll
                for (int j = 1; j < 21; ++j) m = fmaxf(m, lg[j]);
                float sum = 0.f;
#pragma unroll
                for (int j = 0; j < 21; ++j) { lg[j] = expf(lg[j] - m); sum += lg[j]; }
#pragma unroll
                for (int j = 0; j < 21; ++j) gt[site * 21 + j] = lg[j] / sum;
                const float m2 = fmaxf(lg[21], fmaxf(lg[22], lg[23]));
                const float e0 = expf(lg[21] - m2), e1 = expf(lg[22] - m2), e2 = expf(lg[23] - m2);
                const float s2 = e0 + e1 + e2;
                zy[site * 3 + 0] = e0 / s2; zy[site * 3 + 1] = e1 / s2; zy[site * 3 + 2] = e2 / s2;
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<1>(tmem_base, 512);
}

template <int LAYER, int CG, int NWQ, bool DEBUG>
int launch_one(const void* blob, const int32_t* xi, const float* xf, const void* h0_in, void* h0_out, float* h16, float* dbg,
               int64_t m, int dir_override, cudaStream_t stream)
{
    using S = TcSmem<LAYER, CG>;
    auto kern = lstm_tc_kernel<LAYER, CG, NWQ, DEBUG>;
    static bool attr_done = false;
    if (!attr_done) {
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::total) != cudaSuccess) return cuda_status("cudaFuncSetAttribute(lstm_tc_kernel)");
        attr_done = true;
    }
    unsigned gx = (unsigned)((m + kRows - 1) / kRows);
    if (CG == 2 && (gx & 1)) ++gx;                               // whole clusters; the padding CTA works on clamped rows
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(gx, DEBUG ? 1 : 2, 1);
    cfg.blockDim = dim3(128 * NWQ + (LAYER == 1 ? 32 : 0), 1, 1);
    cfg.dynamicSmemBytes = S::total;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CG; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kern, (const unsigned char*)blob, xi, xf, (const __half*)h0_in, (__half*)h0_out, h16, dbg, m, dir_override);
    if (e != cudaSuccess) return set_error(NSNP_E_CUDA, "lstm_tc_kernel<%d,%d,%d>: %s", LAYER, CG, NWQ, cudaGetErrorString(e));
    return NSNP_OK;
}

}  // namespace

int launch_tail_tc(const void* blob, const float* h16, int64_t n_max, const int32_t* n_dev, float* gt, float* zy, cudaStream_t stream) {
    using S = TailSmem;
    static bool attr_done = false;
    if (!attr_done) {
        if (cudaFuncSetAttribute(tail_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::total) != cudaSuccess)
            return cuda_status("cudaFuncSetAttribute(tail_tc_kernel)");
        attr_done = true;
    }
    const int64_t n_tiles = (n_max + kRows - 1) / kRows;
    const int grid = (int)(n_tiles < kNumSMs ? n_tiles : kNumSMs);
    tail_tc_kernel<<<grid, kTtThreads, S::total, stream>>>((const unsigned char*)blob, h16, n_max, n_dev, gt, zy);
    return cuda_status("tail_tc_kernel");
}

int launch_lstm_tc(const void* blob, const int32_t* xi, const float* xf, void* h0, float* h16, int64_t m, const int32_t* pos, int64_t pos_bias, int npass, cudaStream_t stream) {
    // layer 0: CTA pairs share W (53 KB each) so two CTAs fit per SM and one CTA's MMAs overlap the other's epilogue
    {
        ProfScope prof(NSNP_PROF_LSTM0, stream);
        // default: two alternating groups per CTA (lstm0_pair2_kernel); NSNP_L0_VARIANT=0 selects two independent CTAs per SM
        static const int variant = [] { const char* v = getenv("NSNP_L0_VARIANT"); return v ? atoi(v) : 1; }();
        if (pos && variant != 1) return set_error(NSNP_E_UNSUPPORTED, "window reads from the count tensor need the default layer-0 kernel");
        if (int e = variant == 1 ? launch_l0_pair2(blob, xi, xf, h0, m, pos, pos_bias, npass, stream)
                                 : launch_one<0, 2, 2, false>(blob, xi, xf, nullptr, h0, nullptr, nullptr, m, npass << 16, stream)) return e;
    }
    // layer 1: W only fits split across a CTA pair (2 x 96 KB hi + lo); one CTA per SM
    ProfScope prof(NSNP_PROF_LSTM1, stream);
    static const int pf = [] { const char* v = getenv("NSNP_L1_PREFETCH"); return v ? atoi(v) : 1; }();
    // default: two alternating groups per CTA (lstm1_pair2x3_kernel, single pass: lstm1_pair2_kernel);
    // NSNP_L1_VARIANT=0 keeps the one-group kernel lstm_tc_kernel<1,2,4> (A/B, tests)
    static const int l1_variant = [] { const char* v = getenv("NSNP_L1_VARIANT"); return v ? atoi(v) : 1; }();
    if (npass == 1 && l1_variant == 1) return launch_l1_pair2(blob, h0, h16, m, stream);
    if (npass == 3 && l1_variant == 1) return launch_l1_pair2x3(blob, h0, h16, m, stream);
    return launch_one<1, 2, 4, false>(blob, nullptr, nullptr, h0, nullptr, h16, nullptr, m, (pf << 8) | (npass << 16), stream);
}

int debug_tc_gates(const void* blob, const int32_t* xi, int layer, int dir, int cg, const void* h0, float* gates_out, int64_t m, cudaStream_t stream) {
    if (layer == 0 && cg == 1) return launch_one<0, 1, 2, true>(blob, xi, nullptr, nullptr, nullptr, nullptr, gates_out, m, dir, stream);
    if (layer == 0 && cg == 2) return launch_one<0, 2, 2, true>(blob, xi, nullptr, nullptr, nullptr, nullptr, gates_out, m, dir, stream);
    if (layer == 1 && cg == 2) return launch_one<1, 2, 4, true>(blob, nullptr, nullptr, h0, nullptr, nullptr, gates_out, m, dir, stream);
    return set_error(NSNP_E_UNSUPPORTED, "debug_tc_gates: layer %d with cta_group %d is not built", layer, cg);
}

// host: fp16 hi/lo split weights in the [k/8][n][k%8] operand layout
int pack_tc_weights(const nsnp_model_weights_t* w, unsigned char* blob) {
    for (int layer = 0; layer < 2; ++layer) {
        const int K = layer == 0 ? kTcK0 : kTcK1, IN = layer == 0 ? kTcIn0 : kTcIn1, nin = layer == 0 ? kF : 128;
        for (int d = 0; d < 2; ++d) {
            __half* hi = reinterpret_cast<__half*>(blob + tc_off(layer, d, 0));
            __half* lo = reinterpret_cast<__half*>(blob + tc_off(layer, d, 1));
            const float *wih = w->w_ih[layer][d], *whh = w->w_hh[layer][d], *bi = w->b_ih[layer][d], *bh = w->b_hh[layer][d];
            for (int n = 0; n < 256; ++n) {
                const int jb = n >> 5, uh = (n >> 4) & 1, gate = (n >> 2) & 3, u4 = n & 3;
                const int rowi = gate * kH + jb * 8 + uh * 4 + u4;       // PyTorch gate-major row
                for (int k = 0; k < K; ++k) {
                    float v = 0.f;
                    if (k < nin) v = wih[rowi * nin + k];
                    else if (layer == 0 && k == nin) v = bi[rowi] + bh[rowi];          // layer 0: bias rides as a constant-1 input column
                    else if (k >= IN) v = whh[rowi * kH + (k - IN)];
                    v *= gate == 2 ? -2.0f * kLog2e : -kLog2e;         // activation scale folded into the weights (see the epilogue)
                    const float scale = (layer == 0 && k < IN) ? kTcLoScale : 1.0f;
                    const __half h = __float2half_rn(v);
                    const __half l = __float2half_rn((v - __half2float(h)) * scale);
                    const size_t idx = ((size_t)(k >> 3) * 256 + n) * 8 + (k & 7);
                    hi[idx] = h; lo[idx] = l;
                }
                if (layer == 1) reinterpret_cast<float*>(blob + kOffTcBias1)[d * 256 + n] = (bi[rowi] + bh[rowi]) * (gate == 2 ? -2.0f * kLog2e : -kLog2e);
            }
        }
    }
    // tail: folded dense weights (float [128 k][256 n], written by nsnp_model_pack_weights before this call)
    {
        const float* Wd = reinterpret_cast<const float*>(blob) + kOffDenseW;
        __half* hi = reinterpret_cast<__half*>(blob + kOffTcTail);
        __half* lo = reinterpret_cast<__half*>(blob + kOffTcTail + kTcBytesTail);
        for (int n = 0; n < 256; ++n)
            for (int k = 0; k < 128; ++k) {
                const float v = Wd[(size_t)k * 256 + n];
                const __half h = __float2half_rn(v);
                const size_t idx = ((size_t)(k >> 3) * 256 + n) * 8 + (k & 7);
                hi[idx] = h; lo[idx] = __float2half_rn(v - __half2float(h));
            }
    }
    return NSNP_OK;
}

}  // namespace nsnp

extern "C" int nsnp_debug_lstm_tc_gates(const void* blob_dev, const int32_t* x_i32_dev, int layer, int dir, int cg, const void* h0_dev,
                                        float* gates_out_dev, int64_t m, void* stream)
{
    if (!blob_dev || !gates_out_dev || m <= 0 || dir < 0 || dir > 1) return nsnp::set_error(NSNP_E_INVALID, "nsnp_debug_lstm_tc_gates: bad argument");
    if (nsnp_device_count() == 0) return nsnp::set_error(NSNP_E_NO_DEVICE, "no CUDA device (there is no CPU fallback)");
    return nsnp::debug_tc_gates(blob_dev, x_i32_dev, layer, dir, cg, h0_dev, gates_out_dev, m, (cudaStream_t)stream);
}
