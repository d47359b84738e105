// HaplotypeModel s5 forward pass on the 5th-generation tensor cores (opt-in, precision f16x3): the same network as
// nsnp_hap_model_forward (haplotype.cu, the fp32 parity reference), hand-written for sm_100a.
//
// One fused kernel per time step, shared by all six recurrences (2 encoders x 3 layers, 2 directions each):
//     gates[128 sites x 256] = [in_t | h_{t-1}] [128 x K]  .  W'^T [K x 256]  + b'
// One CTA = one 128-site tile x one slice of 256 gate columns (64 hidden units; the packed rows interleave the four gates of a
// unit, column = unit * 4 + gate, so one TMEM lane holds i, f, g, o of its units and the cell update runs in the epilogue).
// The independent recurrences of a (layer, step) -- both encoders, both directions -- share a launch through grid.z, so a
// chunk of sites takes 33 + 33 + 17 = 83 step launches.
//
// Operands.  K runs in k-blocks of 32 bytes per row: A [hi|lo][2 core-matrix columns][128 rows][16 B] = 8 KB and
// B [hi|lo][2][256 rows][16 B] = 16 KB, both in the UMMA canonical K-major no-swizzle layout.  A warp of the CTA streams the
// k-blocks (W' from L2, the A rows from the layer buffers) into a kStages-deep shared-memory ring with cp.async.bulk; another
// warp issues three MMAs per k-block into one fp32 TMEM accumulator (256 columns):
//     a.w  ~=  a_hi.w_hi + a_hi.w_lo + a_lo.w_hi
//   * layer-0 input (the 105 feature channels, padded to 112): kind::tf32 with hi = tf32(x), lo = x - hi.  Features are not
//     bounded (counts reach the row depth, quality sums ~1e7 > fp16's 65504), tf32 keeps fp32's exponent range.
//   * h and the outputs of layers 0-1 (in [-1, 1]): kind::f16, hi = fp16(v), lo = fp16(v - hi), as model_tc.cu.
// Layer outputs are written once by the epilogue, as fp16 hi/lo, directly in the operand layout that the next step (its h part:
// this direction's half at position t -+ 1) and the next layer (its input part) read: Y[tile][position][32 k-blocks][8 KB].
// The cell state stays in an fp32 [m][256] buffer per recurrence.  The last layer runs only the steps its centre output needs and
// writes only the centre h, in fp32; output_proj, dense and the heads (0.3 % of the work) run on haplotype.cu's fp32 kernels.
//
// Cell update as model_tc.cu: the activation scales (-log2 e, -2 log2 e) are folded into the packed weights and bias, every
// exponential is a bare ex2.approx and the cell state is kept scaled.  Every site's arithmetic is the same wherever it sits in
// a batch (one TMEM lane, fixed k order), so results do not depend on the batch.
#include <math.h>
#include "hap_common.cuh"
#include "tc_ptx.cuh"

namespace nsnp {
namespace {

constexpr int kH = 256, kG = 4 * kH, kDim = 105, kLayers = 3, kLp = 33, kLh = 11;
constexpr int kRows = 128;                       // sites per tile = TMEM lanes
constexpr int kSlices = kG / 256;                // gate-column slices of 256 (64 hidden units) per tile
constexpr int kKb0 = 14;                         // layer-0 input k-blocks: 105 channels padded to 112, tf32 (K = 8 per MMA)
constexpr int kKbIn = 32;                        // layer 1-2 input k-blocks: 512 = [fwd 256 | rev 256], fp16 (K = 16 per MMA)
constexpr int kKbH = 16;                         // recurrent k-blocks: 256, fp16
constexpr uint32_t kABytes = 8192, kBBytes = 16384, kHalfA = kABytes / 2, kHalfB = kBBytes / 2;
constexpr size_t kTileT = (size_t)kKbIn * kABytes;   // one (tile, position) of a layer output: 256 KB
constexpr size_t kTileT0 = (size_t)kKb0 * kABytes;   // one (tile, position) of the layer-0 input: 112 KB
constexpr int kStages = 4;                       // 4 x 24 KB: two CTAs per SM, one's epilogue under the other's MMAs
constexpr int kThreads = 192;                    // warps 0-3 epilogue (one TMEM lane quadrant each), 4 bulk copies, 5 MMA issuer
constexpr size_t kSmemBytes = (size_t)kStages * (kABytes + kBBytes) + 128;
constexpr float kLog2e = 1.4426950408889634f;
constexpr int64_t kChunk = 4096;                 // sites per pass: bounds the workspace (~27 MB per 128-site tile)

inline int nkb_of(int layer) { return (layer == 0 ? kKb0 : kKbIn) + kKbH; }
__host__ __device__ inline float gate_scale(int gate) { return gate == 2 ? -2.0f * kLog2e : -kLog2e; }

// ---- packed blob (bytes) ----
//   fp32 tail: proj_w[2] [256][512], proj_b[2] [256], dense_w [256][512], dense_b [256], gt_w [10][256], gt_b, zy_w [3][256], zy_b
//   per (encoder e, layer l, direction d): bias' float [1024] (column order, activation-scaled), then
//       W' k-blocks [slice 4][kb][hi|lo][2][256 rows][16 B]   (kb < kKb0 of layer 0: tf32 words, otherwise fp16)
struct TcBlob {
    size_t proj_w[2], proj_b[2], dense_w, dense_b, gt_w, gt_b, zy_w, zy_b;    // float offsets
    size_t bias[2][kLayers][2], w[2][kLayers][2], total;                     // byte offsets
};
inline TcBlob tc_blob_layout() {
    TcBlob B; size_t o = 0;
    for (int e = 0; e < 2; ++e) { B.proj_w[e] = o; o += (size_t)kH * 2 * kH; B.proj_b[e] = o; o += kH; }
    B.dense_w = o; o += (size_t)kH * 2 * kH; B.dense_b = o; o += kH;
    B.gt_w = o; o += 10 * kH; B.gt_b = o; o += 10; B.zy_w = o; o += 3 * kH; B.zy_b = o; o += 3;
    size_t b = (o * 4 + 1023) / 1024 * 1024;
    for (int e = 0; e < 2; ++e)
        for (int l = 0; l < kLayers; ++l)
            for (int d = 0; d < 2; ++d) {
                B.bias[e][l][d] = b; b += (size_t)kG * 4;
                B.w[e][l][d] = b; b += (size_t)kSlices * nkb_of(l) * kBBytes;
            }
    B.total = b;
    return B;
}

// tf32 round to nearest, ties away from zero (cvt.rna.tf32.f32): the hi part is then exact in the MMA's tf32 operand
inline float tf32_rna_host(float v) {
    uint32_t b; memcpy(&b, &v, 4);
    if ((b & 0x7f800000u) != 0x7f800000u) b = (b + 0x1000u) & 0xffffe000u;
    memcpy(&v, &b, 4); return v;
}
__device__ __forceinline__ float tf32_rna(float x) { uint32_t r; asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x)); return __uint_as_float(r); }

// ---- layer-0 operand: x [m][105][L] -> X0[tile][t][kb 14][hi|lo][2][128 rows][4 floats]; padding rows and channels are 0 ----
__global__ void __launch_bounds__(256) hap_x0_kernel(const float* __restrict__ x, int L, int64_t m, int64_t tiles, unsigned char* __restrict__ x0)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= tiles * L * (2 * kKb0) * kRows) return;
    const int row = (int)(i % kRows), col = (int)((i / kRows) % (2 * kKb0)), t = (int)((i / (kRows * 2 * kKb0)) % L);
    const int64_t tile = i / ((int64_t)kRows * 2 * kKb0 * L);
    const int64_t site = tile * kRows + row;
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int ch = col * 4 + j;
        v[j] = (site < m && ch < kDim) ? x[(site * kDim + ch) * L + t] : 0.f;
    }
    float4 hi, lo;
    hi.x = tf32_rna(v[0]); hi.y = tf32_rna(v[1]); hi.z = tf32_rna(v[2]); hi.w = tf32_rna(v[3]);
    lo.x = v[0] - hi.x; lo.y = v[1] - hi.y; lo.z = v[2] - hi.z; lo.w = v[3] - hi.w;
    unsigned char* o = x0 + (tile * L + t) * kTileT0 + (size_t)(col >> 1) * kABytes + (col & 1) * 2048 + row * 16;
    *reinterpret_cast<float4*>(o) = hi;
    *reinterpret_cast<float4*>(o + kHalfA) = lo;
}

// ---- one time step ----
struct Rec {                       // one recurrence (encoder, direction) of the launch's layer
    const unsigned char* w;        // W' k-blocks of this (encoder, layer, direction)
    const float* bias;             // bias' [1024], column order
    const unsigned char* in;       // input rows: X0 (layer 0) or the previous layer's Y, in_stride bytes per (tile, position)
    unsigned char* y;              // this layer's Y [tile][L][256 KB]: h_{t-1} is read from it, h_t written to it
    float* c;                      // cell state [m][256], scaled by -2 log2 e
    float* hout;                   // last layer, centre step: fp32 h -> hout[site][dir * 256 + unit] (rows of 512), no Y write
    float* dbg;                    // test aid: unscaled gate pre-activations [m][1024] in PyTorch order, nothing else written
    int L, t, dir, first;
};
struct StepArgs { Rec r[4]; int64_t m; int nkb_in, tf32_in; size_t in_stride; };

__global__ void __launch_bounds__(kThreads, 2) hap_step_kernel(const __grid_constant__ StepArgs a)
{
    extern __shared__ __align__(1024) unsigned char smem[];
    const Rec& R = a.r[blockIdx.z];
    const int tile = (int)blockIdx.x, slice = (int)blockIdx.y;
    const int warp = (int)threadIdx.x >> 5, lane = (int)threadIdx.x & 31;
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + kStages * (kABytes + kBBytes));   // [kStages] k-block landed
    uint64_t* empty = full + kStages;                                                     // [kStages] its MMAs have completed
    uint64_t* done = empty + kStages;                                                     // all MMAs of the step have completed
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);
    const int nkb = a.nkb_in + (R.first ? 0 : kKbH);                                      // h = 0 at the first step

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 1); }
        mbar_init(done, 1);
        fence_mbar_init();
    }
    if (warp == 0) tmem_alloc<1>(tmem_slot, 256);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == 4) {
        if (lane == 0) {                                                                   // producer: k-block kb -> stage kb % kStages
            const int tp = R.dir == 0 ? R.t - 1 : R.t + 1;
            const unsigned char* ain = R.in + ((size_t)tile * R.L + R.t) * a.in_stride;
            const unsigned char* ah = R.y + ((int64_t)tile * R.L + tp) * (int64_t)kTileT + (int64_t)R.dir * kKbH * kABytes;
            const unsigned char* wb = R.w + (size_t)slice * (a.nkb_in + kKbH) * kBBytes;
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % kStages;
                if (kb >= kStages) mbar_wait(empty + s, (uint32_t)((kb / kStages - 1) & 1));
                unsigned char* st = smem + s * (kABytes + kBBytes);
                mbar_expect_tx(full + s, kABytes + kBBytes);
                bulk_g2s(st, kb < a.nkb_in ? ain + (size_t)kb * kABytes : ah + (size_t)(kb - a.nkb_in) * kABytes, kABytes, full + s);
                bulk_g2s(st + kABytes, wb + (size_t)kb * kBBytes, kBBytes, full + s);
            }
        }
    } else if (warp == 5) {
        if (lane == 0) {                                                                   // MMA issuer
            constexpr uint32_t idesc16 = make_idesc(kRows, 256);
            constexpr uint32_t idesc32 = idesc16 | (2u << 7) | (2u << 10);                 // A, B format tf32
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % kStages;
                mbar_wait(full + s, (uint32_t)((kb / kStages) & 1));
                tc_fence_after();
                const uint32_t base = smem_u32(smem + s * (kABytes + kBBytes));
                const uint64_t ahi = make_desc(base, 2048, 128), alo = make_desc(base + kHalfA, 2048, 128);
                const uint64_t bhi = make_desc(base + kABytes, 4096, 128), blo = make_desc(base + kABytes + kHalfB, 4096, 128);
                if (a.tf32_in && kb < a.nkb_in) {
                    umma_tf32(tmem, ahi, bhi, idesc32, kb > 0);
                    umma_tf32(tmem, ahi, blo, idesc32, 1u);
                    umma_tf32(tmem, alo, bhi, idesc32, 1u);
                } else {
                    umma_f16<1>(tmem, ahi, bhi, idesc16, kb > 0);
                    umma_f16<1>(tmem, ahi, blo, idesc16, 1u);
                    umma_f16<1>(tmem, alo, bhi, idesc16, 1u);
                }
                umma_commit<1>(empty + s);
            }
            umma_commit<1>(done);
        }
    } else {
        // ---- epilogue: thread = one site row (TMEM lane), 8 blocks of 8 hidden units = 32 columns (i, f, g, o per unit) ----
        const int row = warp * 32 + lane;
        const int64_t site = (int64_t)tile * kRows + row;
        const bool live = site < a.m;
        const float* bias = R.bias + slice * 256;
        mbar_wait(done, 0);
        tc_fence_after();
        const uint32_t tacc = tmem + ((uint32_t)(warp * 32) << 16);
#pragma unroll 1
        for (int ub = 0; ub < 8; ++ub) {
            float v[32];
            tmem_ld32(tacc + ub * 32, v);
            if (R.dbg) {
                if (live)
                    for (int j = 0; j < 32; ++j) {
                        const int col = ub * 32 + j, unit = slice * 64 + col / 4, gate = col % 4;
                        R.dbg[site * kG + gate * kH + unit] = (v[j] + __ldg(bias + col)) / gate_scale(gate);
                    }
                continue;
            }
            const int unit0 = slice * 64 + ub * 8;
            float cs[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            if (!R.first && live) {
                const float4 c0 = *reinterpret_cast<const float4*>(R.c + site * kH + unit0), c1 = *reinterpret_cast<const float4*>(R.c + site * kH + unit0 + 4);
                cs[0] = c0.x; cs[1] = c0.y; cs[2] = c0.z; cs[3] = c0.w; cs[4] = c1.x; cs[5] = c1.y; cs[6] = c1.z; cs[7] = c1.w;
            }
            float hv[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                // accumulators: xi = -log2e i, xf = -log2e f, xg = -2 log2e g, xo = -log2e o; cs = -2 log2e c (model_tc.cu)
                const float* bq = bias + ub * 32 + u * 4;
                const float xi_ = fminf(v[4 * u] + __ldg(bq), 36.f), xf_ = fminf(v[4 * u + 1] + __ldg(bq + 1), 36.f);
                const float xg_ = fminf(v[4 * u + 2] + __ldg(bq + 2), 36.f), xo_ = v[4 * u + 3] + __ldg(bq + 3);
                const float ei = ex2_approx(xi_), ef = ex2_approx(xf_), eg = ex2_approx(xg_), eo = ex2_approx(xo_);
                const float pi = 1.f + ei, pf = 1.f + ef, pg = 1.f + eg;
                const float pig = pi * pg;
                const float num = fmaf(cs[u], pig, fmaf(eg, 2.f * kLog2e, -2.f * kLog2e) * pf);
                const float cn = num * rcp_approx(pf * pig);
                cs[u] = cn;
                const float ec = ex2_approx(cn);
                hv[u] = (1.f - ec) * rcp_approx((1.f + eo) * (1.f + ec));                   // sigmoid(o) tanh(c')
            }
            if (live) {                                                                     // padding rows: nothing stored
                float4* cw = reinterpret_cast<float4*>(R.c + site * kH + unit0);
                cw[0] = make_float4(cs[0], cs[1], cs[2], cs[3]); cw[1] = make_float4(cs[4], cs[5], cs[6], cs[7]);
                if (R.hout) {
                    float4* o = reinterpret_cast<float4*>(R.hout + site * (2 * kH) + R.dir * kH + unit0);
                    o[0] = make_float4(hv[0], hv[1], hv[2], hv[3]); o[1] = make_float4(hv[4], hv[5], hv[6], hv[7]);
                } else {
                    const HiLo8 sp = split8(hv);
                    const int ch = R.dir * 32 + unit0 / 8;                                   // 16-byte column of the 512-wide layer output
                    unsigned char* o = R.y + ((size_t)tile * R.L + R.t) * kTileT + (size_t)(ch >> 1) * kABytes + (ch & 1) * 2048 + row * 16;
                    *reinterpret_cast<uint4*>(o) = sp.hi;
                    *reinterpret_cast<uint4*>(o + kHalfA) = sp.lo;
                }
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<1>(tmem, 256);
}

int launch_step(const StepArgs& a, int nrec, int64_t tiles, cudaStream_t st)
{
    static bool attr_done = false;
    if (!attr_done) {
        if (cudaFuncSetAttribute(hap_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes) != cudaSuccess)
            return cuda_status("cudaFuncSetAttribute(hap_step_kernel)");
        attr_done = true;
    }
    hap_step_kernel<<<dim3((unsigned)tiles, kSlices, (unsigned)nrec), kThreads, kSmemBytes, st>>>(a);
    return cuda_status("hap_step_kernel");
}

int launch_x0(const float* x, int L, int64_t m, int64_t tiles, unsigned char* x0, cudaStream_t st)
{
    const int64_t total = tiles * L * (2 * kKb0) * kRows;
    hap_x0_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(x, L, m, tiles, x0);
    return cuda_status("hap_x0_kernel");
}

struct TcWs { unsigned char *x0[2], *ya[2], *yb[2]; float *c[4], *cat[2], *enc, *hid; };
inline size_t carve_tc_ws(void* base, int64_t n, TcWs* w) {
    const int64_t m = n < kChunk ? n : kChunk, tiles = (m + kRows - 1) / kRows;
    size_t off = 0;
    auto take = [&](size_t bytes) { unsigned char* p = base ? (unsigned char*)base + off : nullptr; off += (bytes + 1023) / 1024 * 1024; return p; };
    for (int e = 0; e < 2; ++e) {
        const int L = e == 0 ? kLp : kLh;
        w->x0[e] = take((size_t)tiles * L * kTileT0);
        w->ya[e] = take((size_t)tiles * L * kTileT);
        w->yb[e] = take((size_t)tiles * L * kTileT);
        w->cat[e] = (float*)take((size_t)m * 2 * kH * 4);     // centre h of the last layer, fwd | rev
    }
    for (int r = 0; r < 4; ++r) w->c[r] = (float*)take((size_t)m * kH * 4);
    w->enc = (float*)take((size_t)m * 2 * kH * 4);            // output_proj of both encoders, pileup | haplotype
    w->hid = (float*)take((size_t)m * kH * 4);
    return off;
}

}  // namespace
}  // namespace nsnp

using namespace nsnp;

extern "C" {

size_t nsnp_hap_model_tc_blob_bytes(void) { return tc_blob_layout().total; }

int nsnp_hap_model_tc_pack_weights(const nsnp_hap_weights_t* w, void* host_blob, size_t blob_bytes)
{
    if (!w || !host_blob) return set_error(NSNP_E_INVALID, "nsnp_hap_model_tc_pack_weights: null argument");
    const TcBlob B = tc_blob_layout();
    if (blob_bytes < B.total) return set_error(NSNP_E_WORKSPACE, "haplotype tensor-core blob: need %zu bytes", B.total);
    unsigned char* blob = (unsigned char*)host_blob;
    float* f = (float*)host_blob;
    for (int e = 0; e < 2; ++e)
        for (int l = 0; l < kLayers; ++l)
            for (int d = 0; d < 2; ++d) {
                const int in = l == 0 ? kDim : 2 * kH, nkb_in = l == 0 ? kKb0 : kKbIn, nkb = nkb_of(l);
                const float *wi = w->w_ih[e][l][d], *wh = w->w_hh[e][l][d], *bi = w->b_ih[e][l][d], *bh = w->b_hh[e][l][d];
                if (!wi || !wh || !bi || !bh) return set_error(NSNP_E_INVALID, "nsnp_hap_model_tc_pack_weights: missing LSTM tensor");
                float* bias = (float*)(blob + B.bias[e][l][d]);
                for (int s = 0; s < kSlices; ++s)
                    for (int r = 0; r < 256; ++r) {
                        const int unit = s * 64 + r / 4, gate = r % 4, prow = gate * kH + unit;       // PyTorch row of column r
                        const float sc = gate_scale(gate);
                        bias[s * 256 + r] = (bi[prow] + bh[prow]) * sc;
                        for (int kb = 0; kb < nkb; ++kb) {
                            unsigned char* blk = blob + B.w[e][l][d] + ((size_t)s * nkb + kb) * kBBytes;
                            for (int sub = 0; sub < 2; ++sub) {
                                if (l == 0 && kb < nkb_in) {                                          // tf32 words
                                    float* hi = (float*)(blk + ((size_t)sub * 256 + r) * 16);
                                    float* lo = (float*)(blk + kHalfB + ((size_t)sub * 256 + r) * 16);
                                    for (int j = 0; j < 4; ++j) {
                                        const int k = kb * 8 + sub * 4 + j;
                                        const float v = k < in ? wi[(size_t)prow * in + k] * sc : 0.f;
                                        hi[j] = tf32_rna_host(v); lo[j] = v - hi[j];
                                    }
                                } else {                                                               // fp16 halves
                                    __half* hi = (__half*)(blk + ((size_t)sub * 256 + r) * 16);
                                    __half* lo = (__half*)(blk + kHalfB + ((size_t)sub * 256 + r) * 16);
                                    for (int j = 0; j < 8; ++j) {
                                        float v;
                                        if (kb < nkb_in) v = wi[(size_t)prow * in + kb * 16 + sub * 8 + j] * sc;
                                        else v = wh[(size_t)prow * kH + (kb - nkb_in) * 16 + sub * 8 + j] * sc;
                                        hi[j] = __float2half_rn(v); lo[j] = __float2half_rn(v - __half2float(hi[j]));
                                    }
                                }
                            }
                        }
                    }
            }
    for (int e = 0; e < 2; ++e) {
        if (!w->proj_w[e] || !w->proj_b[e]) return set_error(NSNP_E_INVALID, "nsnp_hap_model_tc_pack_weights: missing output_proj");
        memcpy(f + B.proj_w[e], w->proj_w[e], (size_t)kH * 2 * kH * 4); memcpy(f + B.proj_b[e], w->proj_b[e], kH * 4);
    }
    if (!w->dense_w || !w->dense_b || !w->gt_w || !w->gt_b || !w->zy_w || !w->zy_b) return set_error(NSNP_E_INVALID, "nsnp_hap_model_tc_pack_weights: missing head tensor");
    memcpy(f + B.dense_w, w->dense_w, (size_t)kH * 2 * kH * 4); memcpy(f + B.dense_b, w->dense_b, kH * 4);
    memcpy(f + B.gt_w, w->gt_w, 10 * kH * 4); memcpy(f + B.gt_b, w->gt_b, 10 * 4);
    memcpy(f + B.zy_w, w->zy_w, 3 * kH * 4); memcpy(f + B.zy_b, w->zy_b, 3 * 4);
    return NSNP_OK;
}

size_t nsnp_hap_model_tc_workspace_bytes(int64_t n) { TcWs w; return carve_tc_ws(nullptr, n < 1 ? 1 : n, &w); }

int nsnp_hap_model_tc_forward(const void* blob_dev, const float* xp_dev, const float* xh_dev, int64_t n, float* gt_prob_dev, float* zy_prob_dev,
                              void* workspace_dev, size_t workspace_bytes, void* stream_)
{
    cudaStream_t st = (cudaStream_t)stream_;
    if (n < 0 || (n > 0 && (!blob_dev || !xp_dev || !xh_dev || !gt_prob_dev || !zy_prob_dev || !workspace_dev)))
        return set_error(NSNP_E_INVALID, "nsnp_hap_model_tc_forward: bad argument");
    if (n == 0) return NSNP_OK;
    if (nsnp_device_count() == 0) return set_error(NSNP_E_NO_DEVICE, "no CUDA device (there is no CPU fallback)");
    TcWs w;
    if (carve_tc_ws(workspace_dev, n, &w) > workspace_bytes) return set_error(NSNP_E_WORKSPACE, "haplotype tensor-core workspace too small");
    const TcBlob B = tc_blob_layout();
    const unsigned char* blob = (const unsigned char*)blob_dev;
    const float* f = (const float*)blob_dev;
    for (int64_t s0 = 0; s0 < n; s0 += kChunk) {
        const int64_t m = n - s0 < kChunk ? n - s0 : kChunk, tiles = (m + kRows - 1) / kRows;
        for (int e = 0; e < 2; ++e) {
            const int L = e == 0 ? kLp : kLh;
            if (int rc = launch_x0((e == 0 ? xp_dev : xh_dev) + s0 * kDim * L, L, m, tiles, w.x0[e], st)) return rc;
        }
        for (int l = 0; l < kLayers; ++l) {
            const bool last = l == kLayers - 1;
            StepArgs a = {};
            a.m = m; a.nkb_in = l == 0 ? kKb0 : kKbIn; a.tf32_in = l == 0; a.in_stride = l == 0 ? kTileT0 : kTileT;
            const int steps_p = last ? kLp / 2 + 1 : kLp;
            for (int s = 0; s < steps_p; ++s) {
                int nrec = 0;
                for (int e = 0; e < 2; ++e) {
                    const int L = e == 0 ? kLp : kLh, ctr = L / 2;
                    if (s >= (last ? ctr + 1 : L)) continue;
                    for (int d = 0; d < 2; ++d) {
                        Rec& r = a.r[nrec++];
                        r.w = blob + B.w[e][l][d]; r.bias = (const float*)(blob + B.bias[e][l][d]);
                        r.in = l == 0 ? w.x0[e] : (l == 1 ? w.ya[e] : w.yb[e]);
                        r.y = l == 1 ? w.yb[e] : w.ya[e];                 // layer 2 reuses layer 0's buffer
                        r.c = w.c[e * 2 + d];
                        r.L = L; r.dir = d; r.first = s == 0;
                        r.t = d == 0 ? s : L - 1 - s;
                        r.hout = last && r.t == ctr ? w.cat[e] : nullptr;
                        r.dbg = nullptr;
                    }
                }
                if (int rc = launch_step(a, nrec, tiles, st)) return rc;
            }
        }
        for (int e = 0; e < 2; ++e)                                        // output_proj at the centre row (model_dev.py:84, :105-106)
            if (int rc = hap_sgemm_nt(w.cat[e], 2 * kH, f + B.proj_w[e], f + B.proj_b[e], w.enc + e * kH, 2 * kH, m, kH, 2 * kH, 0, st)) return rc;
        if (int rc = hap_sgemm_nt(w.enc, 2 * kH, f + B.dense_w, f + B.dense_b, w.hid, kH, m, kH, 2 * kH, 1, st)) return rc;
        if (int rc = hap_heads(w.hid, f + B.gt_w, f + B.gt_b, f + B.zy_w, f + B.zy_b, gt_prob_dev + s0 * 10, zy_prob_dev + s0 * 3, m, st)) return rc;
    }
    return cuda_status("nsnp_hap_model_tc_forward");
}

int nsnp_debug_hap_tc_gates(const void* blob_dev, const float* x_dev, int encoder, int dir, float* gates_out_dev, int64_t m, void* stream_)
{
    if (!blob_dev || !x_dev || !gates_out_dev || m <= 0 || encoder < 0 || encoder > 1 || dir < 0 || dir > 1)
        return set_error(NSNP_E_INVALID, "nsnp_debug_hap_tc_gates: bad argument");
    if (nsnp_device_count() == 0) return set_error(NSNP_E_NO_DEVICE, "no CUDA device (there is no CPU fallback)");
    cudaStream_t st = (cudaStream_t)stream_;
    const TcBlob B = tc_blob_layout();
    const int L = encoder == 0 ? kLp : kLh;
    const int64_t tiles = (m + kRows - 1) / kRows;
    void* x0 = nullptr;
    if (cudaMallocAsync(&x0, (size_t)tiles * L * kTileT0, st) != cudaSuccess) return cuda_status("nsnp_debug_hap_tc_gates: cudaMallocAsync");
    int rc = launch_x0(x_dev, L, m, tiles, (unsigned char*)x0, st);
    if (rc == NSNP_OK) {
        StepArgs a = {};
        a.m = m; a.nkb_in = kKb0; a.tf32_in = 1; a.in_stride = kTileT0;
        Rec& r = a.r[0];
        r.w = (const unsigned char*)blob_dev + B.w[encoder][0][dir]; r.bias = (const float*)((const unsigned char*)blob_dev + B.bias[encoder][0][dir]);
        r.in = (const unsigned char*)x0; r.L = L; r.dir = dir; r.first = 1; r.t = dir == 0 ? 0 : L - 1; r.dbg = gates_out_dev;
        rc = launch_step(a, 1, tiles, st);
    }
    cudaFreeAsync(x0, st);
    return rc;
}

}  // extern "C"
