// s2: PileupModel forward (PileupModel/model.py:14-73,114-119; config/ont_pileup.yaml:6-20).
//
//   x[N,33,18] -> BiLSTM(18->64) -> BiLSTM(128->64) -> Linear(128->128) -> Linear(128->256)+tanh @t=16
//             -> Linear(256->21), Linear(256->3) -> softmax
//
// Exact-output pruning (SURVEY appendix D.3): layer 1 runs only the 17 steps per direction that reach
// t=16, output_proj/dense run only at t=16, the two indel heads are never computed.
//
// This file holds the fp32 path (NSNP_PREC_FP32): plain FFMA with fp32 accumulation and accurate
// expf/tanhf -- it is the parity path and the fallback for low-margin sites of the tensor-core path.
//   lstm_dir_kernel<L0>  one CTA = 64 sites x one direction, weights resident in shared memory (85 KB),
//                        lanes own hidden-unit pairs, warps own site groups, cell state in registers.
//   lstm_dir_kernel<L1>  one CTA = 32 sites x one direction, 197 KB of weights resident.
//   tail_kernel          proj + dense/tanh + heads + softmax on the t=16 state.
#include "model_common.cuh"

namespace nsnp {
namespace {

// column of gate row (gate g, unit u) in the shared-memory weight tile: two lane-contiguous halves so that
// every LDS.128 of a warp is conflict free.  half = g>>1, lane = u>>1.
__host__ __device__ constexpr int gate_col(int g, int u) { return (g >> 1) * 128 + (u >> 1) * 4 + (g & 1) * 2 + (u & 1); }

__device__ __forceinline__ float sigmoid_acc(float x) { return 1.0f / (1.0f + expf(-x)); }

template <int LAYER> struct Cfg;
template <> struct Cfg<0> { static constexpr int KP = kKP0, IN = kIn0, S = 64, STEPS = 33; };
template <> struct Cfg<1> { static constexpr int KP = kKP1, IN = kIn1, S = 32, STEPS = 17; };

template <int LAYER>
__global__ void __launch_bounds__(256, 1) lstm_dir_kernel(const float* __restrict__ blob, const int32_t* __restrict__ xi,
                                                          const float* __restrict__ xf, const float* __restrict__ h0_in,
                                                          float* __restrict__ out, int64_t n_max, const int32_t* __restrict__ n_dev)
{
    using C = Cfg<LAYER>;
    constexpr int KP = C::KP, IN = C::IN, S = C::S, SPT = S / 8;
    extern __shared__ __align__(16) float smem[];
    float* W = smem;                       // [KP][256]
    float* bias = W + KP * kG;             // [256]
    float* act = bias + kG;                // [S][KP]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int dir = blockIdx.y;
    int64_t n = n_max;
    if (n_dev) { const int64_t nd = *n_dev; if (nd < n) n = nd; }
    const int64_t site0 = (int64_t)blockIdx.x * S;
    if (site0 >= n) return;

    {   // weights of this (layer, direction) -> shared memory
        const float* gw = blob + (LAYER == 0 ? kOffW0 : kOffW1) + (size_t)dir * KP * kG;
        const float4* g4 = reinterpret_cast<const float4*>(gw);
        float4* s4 = reinterpret_cast<float4*>(W);
        for (int i = tid; i < KP * kG / 4; i += 256) s4[i] = __ldg(g4 + i);
        bias[tid] = __ldg(blob + (LAYER == 0 ? kOffB0 : kOffB1) + dir * kG + tid);
        for (int i = tid; i < S * KP; i += 256) act[i] = 0.0f;
    }
    float c[2][SPT];
#pragma unroll
    for (int s = 0; s < SPT; ++s) { c[0][s] = 0.f; c[1][s] = 0.f; }
    __syncthreads();

    for (int step = 0; step < C::STEPS; ++step) {
        const int t = dir == 0 ? step : (kT - 1 - step);
        // ---- stage the input rows of time t ----
        if (LAYER == 0) {
            for (int i = tid; i < S * kF; i += 256) {
                const int s = i / kF, j = i - s * kF;
                int64_t site = site0 + s; if (site >= n) site = n - 1;
                const int64_t g = (site * kT + t) * kF + j;
                act[s * KP + j] = xi ? (float)__ldg(xi + g) : __ldg(xf + g);
            }
        } else {
            for (int i = tid; i < S * (kIn1 / 4); i += 256) {
                const int s = i / (kIn1 / 4), j = i - s * (kIn1 / 4);
                int64_t site = site0 + s; if (site >= n) site = n - 1;
                const float4 v = __ldg(reinterpret_cast<const float4*>(h0_in + (site * kT + t) * kIn1) + j);
                *reinterpret_cast<float4*>(act + s * KP + 4 * j) = v;
            }
        }
        __syncthreads();
        // ---- gates = W . [in ; h] + b ----
        float acc[4][2][SPT];
        {
            const float4 b0 = *reinterpret_cast<const float4*>(bias + lane * 4);
            const float4 b1 = *reinterpret_cast<const float4*>(bias + 128 + lane * 4);
#pragma unroll
            for (int s = 0; s < SPT; ++s) {
                acc[0][0][s] = b0.x; acc[0][1][s] = b0.y; acc[1][0][s] = b0.z; acc[1][1][s] = b0.w;
                acc[2][0][s] = b1.x; acc[2][1][s] = b1.y; acc[3][0][s] = b1.z; acc[3][1][s] = b1.w;
            }
        }
        const float* arow = act + (warp * SPT) * KP;
#pragma unroll 2
        for (int k4 = 0; k4 < KP / 4; ++k4) {
            float4 a[SPT];
#pragma unroll
            for (int s = 0; s < SPT; ++s) a[s] = *reinterpret_cast<const float4*>(arow + s * KP + 4 * k4);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                const float4 w0 = *reinterpret_cast<const float4*>(W + (4 * k4 + kk) * kG + lane * 4);
                const float4 w1 = *reinterpret_cast<const float4*>(W + (4 * k4 + kk) * kG + 128 + lane * 4);
#pragma unroll
                for (int s = 0; s < SPT; ++s) {
                    const float av = kk == 0 ? a[s].x : kk == 1 ? a[s].y : kk == 2 ? a[s].z : a[s].w;
                    acc[0][0][s] = fmaf(w0.x, av, acc[0][0][s]); acc[0][1][s] = fmaf(w0.y, av, acc[0][1][s]);
                    acc[1][0][s] = fmaf(w0.z, av, acc[1][0][s]); acc[1][1][s] = fmaf(w0.w, av, acc[1][1][s]);
                    acc[2][0][s] = fmaf(w1.x, av, acc[2][0][s]); acc[2][1][s] = fmaf(w1.y, av, acc[2][1][s]);
                    acc[3][0][s] = fmaf(w1.z, av, acc[3][0][s]); acc[3][1][s] = fmaf(w1.w, av, acc[3][1][s]);
                }
            }
        }
        __syncthreads();                   // everyone is done reading h_{t-1}
        // ---- cell update (PyTorch gate order i, f, g, o) ----
#pragma unroll
        for (int s = 0; s < SPT; ++s) {
            float hv[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const float ig = sigmoid_acc(acc[0][u][s]), fg = sigmoid_acc(acc[1][u][s]);
                const float gg = tanhf(acc[2][u][s]), og = sigmoid_acc(acc[3][u][s]);
                c[u][s] = fg * c[u][s] + ig * gg;
                hv[u] = og * tanhf(c[u][s]);
            }
            const int sl = warp * SPT + s;
            *reinterpret_cast<float2*>(act + sl * KP + IN + 2 * lane) = make_float2(hv[0], hv[1]);
            const int64_t site = site0 + sl;
            if (site < n) {
                if (LAYER == 0) *reinterpret_cast<float2*>(out + (site * kT + t) * 128 + dir * kH + 2 * lane) = make_float2(hv[0], hv[1]);
                else if (step == C::STEPS - 1) *reinterpret_cast<float2*>(out + site * 128 + dir * kH + 2 * lane) = make_float2(hv[0], hv[1]);
            }
        }
        // the next iteration's staging writes only act[.. < IN]; the barrier after it orders the h writes
    }
}

// ---- tail: output_proj -> dense + tanh -> heads -> softmax on the t = 16 state (model.py:37, 67-72, 117-118) ----
// output_proj has no non-linearity, so it is folded into dense on the host (W' = W_dense W_proj, b' = W_dense b_proj +
// b_dense, formed in double precision): one 128 -> 256 layer instead of 128 -> 128 -> 256.
// One CTA = 32 sites (48 KB smem, 4 CTAs/SM).  Each layer is a register-tiled fp32 GEMM: a thread owns 4 adjacent
// output columns x SPT sites, weights stream k-major from global memory (coalesced float4 rows, L1/L2 resident),
// activations are float4 broadcasts from shared memory.
constexpr int kTailS = 32;

template <int IN, int OUT, bool TANH>
__device__ __forceinline__ void dense_tile(const float* __restrict__ in, const float* __restrict__ Wt, const float* __restrict__ b,
                                           float* __restrict__ outp)
{
    constexpr int CG = OUT / 4;                  // column groups
    constexpr int SGN = 256 / CG;                // site groups
    constexpr int SPT = kTailS / SGN;            // sites per thread
    const int cg = threadIdx.x % CG, sg = threadIdx.x / CG;
    float acc[SPT][4];
    const float4 bb = __ldg(reinterpret_cast<const float4*>(b) + cg);
#pragma unroll
    for (int s = 0; s < SPT; ++s) { acc[s][0] = bb.x; acc[s][1] = bb.y; acc[s][2] = bb.z; acc[s][3] = bb.w; }
    const float* arow = in + (sg * SPT) * IN;
#pragma unroll 4
    for (int k = 0; k < IN; k += 4) {
        float4 w[4];
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) w[kk] = __ldg(reinterpret_cast<const float4*>(Wt + (size_t)(k + kk) * OUT) + cg);
#pragma unroll
        for (int s = 0; s < SPT; ++s) {
            const float4 a = *reinterpret_cast<const float4*>(arow + s * IN + k);
            const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                acc[s][0] = fmaf(w[kk].x, av[kk], acc[s][0]); acc[s][1] = fmaf(w[kk].y, av[kk], acc[s][1]);
                acc[s][2] = fmaf(w[kk].z, av[kk], acc[s][2]); acc[s][3] = fmaf(w[kk].w, av[kk], acc[s][3]);
            }
        }
    }
#pragma unroll
    for (int s = 0; s < SPT; ++s) {
        float4 o = make_float4(acc[s][0], acc[s][1], acc[s][2], acc[s][3]);
        if (TANH) o = make_float4(tanhf(o.x), tanhf(o.y), tanhf(o.z), tanhf(o.w));
        *reinterpret_cast<float4*>(outp + (sg * SPT + s) * OUT + 4 * cg) = o;
    }
}

__global__ void __launch_bounds__(256, 4) tail_kernel(const float* __restrict__ blob, const float* __restrict__ h16, int64_t n_max,
                                                      const int32_t* __restrict__ n_dev, float* __restrict__ gt, float* __restrict__ zy)
{
    extern __shared__ __align__(16) float tsm[];
    float* in = tsm;                         // [32][128]   (later: logits [32][24])
    float* dn = in + kTailS * 128;           // [32][256]
    int64_t n = n_max;
    if (n_dev) { const int64_t nd = *n_dev; if (nd < n) n = nd; }
    const int64_t site0 = (int64_t)blockIdx.x * kTailS;
    if (site0 >= n) return;
    for (int i = threadIdx.x; i < kTailS * 32; i += 256) {
        const int s = i >> 5, j = i & 31;        // 32 float4 per site
        int64_t site = site0 + s; if (site >= n) site = n - 1;
        reinterpret_cast<float4*>(in)[i] = __ldg(reinterpret_cast<const float4*>(h16 + site * 128) + j);
    }
    __syncthreads();
    dense_tile<128, 256, true>(in, blob + kOffDenseW, blob + kOffDenseB, dn);       // (dense o output_proj) + tanh
    __syncthreads();
    // heads: 24 logits per site (21 genotype + 3 zygosity), thread = (site, 3 logits)
    float* lg = in;
    {
        const int s = threadIdx.x >> 3, c0 = (threadIdx.x & 7) * 3;
        float acc[3];
#pragma unroll
        for (int j = 0; j < 3; ++j) acc[j] = __ldg(blob + kOffHeadB + c0 + j);
        const float* drow = dn + s * 256;
#pragma unroll 4
        for (int k = 0; k < 256; k += 4) {
            const float4 a = *reinterpret_cast<const float4*>(drow + k);
            const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                const float* wr = blob + kOffHeadW + (size_t)(k + kk) * 24 + c0;
                acc[0] = fmaf(__ldg(wr), av[kk], acc[0]); acc[1] = fmaf(__ldg(wr + 1), av[kk], acc[1]); acc[2] = fmaf(__ldg(wr + 2), av[kk], acc[2]);
            }
        }
#pragma unroll
        for (int j = 0; j < 3; ++j) lg[s * 24 + c0 + j] = acc[j];
    }
    __syncthreads();
    if (threadIdx.x < kTailS) {
        const int s = threadIdx.x;
        const int64_t site = site0 + s;
        if (site < n) {
            const float* l = lg + s * 24;
            float m = l[0];
            for (int j = 1; j < 21; ++j) m = fmaxf(m, l[j]);
            float e[21], sum = 0.f;
            for (int j = 0; j < 21; ++j) { e[j] = expf(l[j] - m); sum += e[j]; }
            for (int j = 0; j < 21; ++j) gt[site * 21 + j] = e[j] / sum;
            float m2 = fmaxf(l[21], fmaxf(l[22], l[23]));
            const float e0 = expf(l[21] - m2), e1 = expf(l[22] - m2), e2 = expf(l[23] - m2);
            const float s2 = e0 + e1 + e2;
            zy[site * 3 + 0] = e0 / s2; zy[site * 3 + 1] = e1 / s2; zy[site * 3 + 2] = e2 / s2;
        }
    }
}
constexpr size_t kTailSmem = (size_t)kTailS * (128 + 256) * sizeof(float);

// sites per LSTM launch: four whole waves of 128-site tiles on 148 SMs for both LSTM kernels; bounds the layer-0 output
// buffer (16.9 KB per site)
constexpr int64_t kChunkSites = (int64_t)148 * 128 * 4;


// ---- NSNP_PREC_F16X1: single-pass tensor-core LSTM + re-evaluation of the low-margin sites in NSNP_PREC_F16X3 -------------
// One fp16 MMA per product leaves operand rounding errors of 2^-11: |dp| up to 3e-3 (profiles/r02_precision_experiment.md),
// enough to flip an argmax only where the two best classes of a head are closer than that.  Every site whose top-2 margin is
// below kX1Margin in EITHER head is therefore run again through the three-pass path (its result replaces the single-pass
// one), so genotype / zygosity calls are those of NSNP_PREC_F16X3; the other sites keep probabilities within the stated 5e-3.
// That error bound holds for ordinary counts.  The single pass drops the low bits of a count above 2048 (fp16 holds every
// integer up to 2048), and the errors grow with the counts: deep windows (chrM, collapsed repeats) reach |dp| ~ 1e-2 without a
// flip.  Sites whose window holds such a count are re-evaluated as well.
constexpr float kX1Margin = 0.02f;           // > 6x the largest single-pass error observed
constexpr float kX1ExactCount = 2048.f;
constexpr int kX1Cap = 4096;                 // re-evaluated sites per call (expected: ~0.07 % of the sites); beyond it
                                             // nsnp_model_f16x1_reevaluated reports the overflow
struct X1Work { int32_t* cnt; int32_t* idx; int32_t* pos_low; float* gt_low; float* zy_low; int32_t* x_low; };
constexpr size_t kX1FixedBytes = 256 + (size_t)kX1Cap * (4 + 4 + 24 * 4);
constexpr size_t kX1WindowBytes = (size_t)kX1Cap * kT * kF * 4;

// one warp per site: the lanes scan the site's window (int32 or float32 rows, or its row span of the count tensor when pos is given)
__global__ void x1_margin_kernel(const float* __restrict__ gt, const float* __restrict__ zy, int64_t n, const int32_t* __restrict__ n_dev,
                                 float tau, const int32_t* __restrict__ x, const float* __restrict__ xf, const int32_t* __restrict__ pos,
                                 int64_t pos_bias, int32_t* __restrict__ cnt, int32_t* __restrict__ idx)
{
    const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (i >= n || (n_dev && i >= *n_dev)) return;           // warp-uniform
    const int64_t w0 = pos ? ((int64_t)pos[i] - pos_bias) * kF : i * kT * kF;
    bool deep = false;
    for (int j = lane; j < kT * kF; j += 32) deep |= !(fabsf(x ? (float)x[w0 + j] : xf[w0 + j]) <= kX1ExactCount);
    deep = __any_sync(0xffffffffu, deep);
    if (lane != 0) return;
    float a = -1.f, b = -1.f;
    for (int k = 0; k < 21; ++k) { const float v = gt[i * 21 + k]; if (v > a) { b = a; a = v; } else if (v > b) b = v; }
    float c = -1.f, d = -1.f;
    for (int k = 0; k < 3; ++k) { const float v = zy[i * 3 + k]; if (v > c) { d = c; c = v; } else if (v > d) d = v; }
    if (deep || !(a - b >= tau) || !(c - d >= tau)) {         // also catches NaN
        const int k = atomicAdd(cnt, 1);
        if (k < kX1Cap) idx[k] = (int32_t)i;
    }
}
// inputs of the re-evaluation batch (always kX1Cap sites: slots beyond the count repeat site 0, their results are dropped)
__global__ void x1_gather_kernel(const int32_t* __restrict__ cnt, const int32_t* __restrict__ idx, const int32_t* __restrict__ pos,
                                 const int32_t* __restrict__ x, const float* __restrict__ xf, int32_t* __restrict__ pos_low, int32_t* __restrict__ x_low)
{
    const int k = blockIdx.x;
    const int m = min(*cnt, kX1Cap);
    const int64_t src = k < m ? idx[k] : 0;
    if (pos) { if (threadIdx.x == 0) pos_low[k] = pos[src]; return; }
    const int32_t* from = x ? x : reinterpret_cast<const int32_t*>(xf);          // 4-byte words either way
    for (int j = threadIdx.x; j < kT * kF; j += blockDim.x) x_low[(int64_t)k * kT * kF + j] = from[src * kT * kF + j];
}
__global__ void x1_scatter_kernel(int32_t* __restrict__ cnt, const int32_t* __restrict__ idx, const float* __restrict__ gt_low,
                                  const float* __restrict__ zy_low, float* __restrict__ gt, float* __restrict__ zy)
{
    const int k = blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicMax(cnt + 1, *cnt);            // sticky maximum: an overflow stays visible
    if (k >= min(*cnt, kX1Cap)) return;
    const int64_t dst = idx[k];
    if (lane < 21) gt[dst * 21 + lane] = gt_low[(int64_t)k * 21 + lane];
    else if (lane < 24) zy[dst * 3 + lane - 21] = zy_low[(int64_t)k * 3 + lane - 21];
}

}  // namespace
}  // namespace nsnp

using namespace nsnp;

extern "C" {

size_t nsnp_model_blob_bytes(void) { return kBlobBytes; }

int nsnp_model_pack_weights(const nsnp_model_weights_t* w, void* host_blob, size_t blob_bytes) {
    if (!w || !host_blob) return set_error(NSNP_E_INVALID, "nsnp_model_pack_weights: null argument");
    if (blob_bytes < nsnp_model_blob_bytes()) return set_error(NSNP_E_WORKSPACE, "model blob too small");
    float* b = (float*)host_blob;
    memset(b, 0, nsnp_model_blob_bytes());
    for (int d = 0; d < 2; ++d) {
        // layer 0: rows k = [x 0..17 | pad | h 20..83]
        const float *wih = w->w_ih[0][d], *whh = w->w_hh[0][d], *bi = w->b_ih[0][d], *bh = w->b_hh[0][d];
        if (!wih || !whh || !bi || !bh) return set_error(NSNP_E_INVALID, "missing layer-0 weights");
        float* W0 = b + kOffW0 + (size_t)d * kKP0 * kG;
        for (int g = 0; g < 4; ++g) for (int u = 0; u < kH; ++u) {
            const int row = g * kH + u, col = gate_col(g, u);
            for (int k = 0; k < kF; ++k) W0[k * kG + col] = wih[row * kF + k];
            for (int k = 0; k < kH; ++k) W0[(kIn0 + k) * kG + col] = whh[row * kH + k];
            b[kOffB0 + d * kG + col] = bi[row] + bh[row];
        }
        const float *wih1 = w->w_ih[1][d], *whh1 = w->w_hh[1][d], *bi1 = w->b_ih[1][d], *bh1 = w->b_hh[1][d];
        if (!wih1 || !whh1 || !bi1 || !bh1) return set_error(NSNP_E_INVALID, "missing layer-1 weights");
        float* W1 = b + kOffW1 + (size_t)d * kKP1 * kG;
        for (int g = 0; g < 4; ++g) for (int u = 0; u < kH; ++u) {
            const int row = g * kH + u, col = gate_col(g, u);
            for (int k = 0; k < kIn1; ++k) W1[k * kG + col] = wih1[row * kIn1 + k];
            for (int k = 0; k < kH; ++k) W1[(kIn1 + k) * kG + col] = whh1[row * kH + k];
            b[kOffB1 + d * kG + col] = bi1[row] + bh1[row];
        }
    }
    if (!w->proj_w || !w->proj_b || !w->dense_w || !w->dense_b || !w->gt_w || !w->gt_b || !w->zy_w || !w->zy_b)
        return set_error(NSNP_E_INVALID, "missing head weights");
    for (int o = 0; o < 128; ++o) { for (int k = 0; k < 128; ++k) b[kOffProjW + k * 128 + o] = w->proj_w[o * 128 + k]; b[kOffProjB + o] = w->proj_b[o]; }
    // dense o output_proj folded in double precision: W'[o][k] = sum_j Wd[o][j] Wp[j][k], b'[o] = sum_j Wd[o][j] bp[j] + bd[o]
    for (int o = 0; o < 256; ++o) {
        for (int k = 0; k < 128; ++k) {
            double acc = 0.0;
            for (int j = 0; j < 128; ++j) acc += (double)w->dense_w[o * 128 + j] * (double)w->proj_w[j * 128 + k];
            b[kOffDenseW + k * 256 + o] = (float)acc;
        }
        double bacc = (double)w->dense_b[o];
        for (int j = 0; j < 128; ++j) bacc += (double)w->dense_w[o * 128 + j] * (double)w->proj_b[j];
        b[kOffDenseB + o] = (float)bacc;
    }
    for (int o = 0; o < 21; ++o) { for (int k = 0; k < 256; ++k) b[kOffHeadW + k * 24 + o] = w->gt_w[o * 256 + k]; b[kOffHeadB + o] = w->gt_b[o]; }
    for (int o = 0; o < 3; ++o) { for (int k = 0; k < 256; ++k) b[kOffHeadW + k * 24 + 21 + o] = w->zy_w[o * 256 + k]; b[kOffHeadB + 21 + o] = w->zy_b[o]; }
    return pack_tc_weights(w, (unsigned char*)host_blob);
}

size_t nsnp_model_workspace_bytes(int64_t n_sites) {
    int64_t ch = n_sites < kChunkSites ? n_sites : kChunkSites; if (ch < 1) ch = 1;
    ch = (ch + 127) / 128 * 128;                      // the tensor-core path stores layer-0 output in whole 128-site tiles
    // layer-0 output of one chunk + the t = 16 state of ALL sites (the tail runs once per call, not once per chunk)
    const int64_t np = ((n_sites < 1 ? 1 : n_sites) + 127) / 128 * 128;
    // + the re-evaluation batch of NSNP_PREC_F16X1 (index list, outputs, gathered windows for the window-tensor entry point)
    // 256-byte header first (NSNP_PREC_F16X1 counters: [0] low-margin sites of the last call, [1] their maximum since the reset)
    return 256 + (size_t)ch * kT * 128 * sizeof(float) + (size_t)np * 128 * sizeof(float) + 256 + kX1FixedBytes + kX1WindowBytes;
}

static X1Work x1_carve(void* workspace_dev, int64_t n) {
    const int64_t ch0 = n < kChunkSites ? n : kChunkSites;
    const int64_t ch = ((ch0 < 1 ? 1 : ch0) + 127) / 128 * 128, np = ((n < 1 ? 1 : n) + 127) / 128 * 128;
    char* p = (char*)workspace_dev + 256 + ((size_t)ch * kT * 128 + (size_t)np * 128) * sizeof(float) + 256;
    X1Work w;
    w.cnt = (int32_t*)workspace_dev;
    w.idx = (int32_t*)p; p += (size_t)kX1Cap * 4;
    w.pos_low = (int32_t*)p; p += (size_t)kX1Cap * 4;
    w.gt_low = (float*)p; p += (size_t)kX1Cap * 21 * 4;
    w.zy_low = (float*)p; p += (size_t)kX1Cap * 3 * 4;
    w.x_low = (int32_t*)p;
    return w;
}

int nsnp_model_f16x1_reset(void* workspace_dev, void* stream_) {
    if (!workspace_dev) return set_error(NSNP_E_INVALID, "nsnp_model_f16x1_reset: null argument");
    if (cudaMemsetAsync(workspace_dev, 0, 256, (cudaStream_t)stream_) != cudaSuccess) return cuda_status("nsnp_model_f16x1_reset");
    return NSNP_OK;
}

int nsnp_model_f16x1_reevaluated(const void* workspace_dev, int64_t* count_out, void* stream_) {
    if (!workspace_dev || !count_out) return set_error(NSNP_E_INVALID, "nsnp_model_f16x1_reevaluated: null argument");
    int32_t c[2] = {0, 0};
    if (cudaMemcpyAsync(c, workspace_dev, 8, cudaMemcpyDeviceToHost, (cudaStream_t)stream_) != cudaSuccess || cudaStreamSynchronize((cudaStream_t)stream_) != cudaSuccess)
        return cuda_status("nsnp_model_f16x1_reevaluated");
    *count_out = c[0];
    if (c[1] > kX1Cap) return set_error(NSNP_E_OVERFLOW, "NSNP_PREC_F16X1: a call found %d low-margin sites, only %d were re-evaluated; use NSNP_PREC_F16X3 for this input", c[1], kX1Cap);
    return NSNP_OK;
}

static int model_forward(const void* blob_dev, const int32_t* x_i32_dev, const float* x_f32_dev, int64_t n,
                         const int32_t* n_dev, float* gt_prob_dev, float* zy_prob_dev, void* workspace_dev,
                         size_t workspace_bytes, int precision, const int32_t* pos_dev, int64_t pos_bias, void* stream_);

int nsnp_pileup_model_forward(const void* blob_dev, const int32_t* x_i32_dev, const float* x_f32_dev, int64_t n,
                              const int32_t* n_dev, float* gt_prob_dev, float* zy_prob_dev, void* workspace_dev,
                              size_t workspace_bytes, int precision, void* stream_)
{
    return model_forward(blob_dev, x_i32_dev, x_f32_dev, n, n_dev, gt_prob_dev, zy_prob_dev, workspace_dev, workspace_bytes, precision, nullptr, 0, stream_);
}

int nsnp_pileup_model_forward_sites(const void* blob_dev, const int32_t* counts_dev, int64_t region_start, int64_t region_len,
                                    const int32_t* pos_dev, int64_t n, const int32_t* n_dev, float* gt_prob_dev, float* zy_prob_dev,
                                    void* workspace_dev, size_t workspace_bytes, int precision, void* stream_)
{
    if (n == 0) return NSNP_OK;
    if (!counts_dev || !pos_dev || region_len < NSNP_WINDOW) return set_error(NSNP_E_INVALID, "nsnp_pileup_model_forward_sites: bad argument");
    if (precision != NSNP_PREC_F16X3 && precision != NSNP_PREC_F16X1) return set_error(NSNP_E_UNSUPPORTED, "window reads from the count tensor are built for the tensor-core path; gather the windows for the fp32 path");
    return model_forward(blob_dev, counts_dev, nullptr, n, n_dev, gt_prob_dev, zy_prob_dev, workspace_dev, workspace_bytes, precision, pos_dev,
                         region_start + NSNP_FLANK, stream_);
}

static int model_forward(const void* blob_dev, const int32_t* x_i32_dev, const float* x_f32_dev, int64_t n,
                         const int32_t* n_dev, float* gt_prob_dev, float* zy_prob_dev, void* workspace_dev,
                         size_t workspace_bytes, int precision, const int32_t* pos_dev, int64_t pos_bias, void* stream_)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    if (n == 0) return NSNP_OK;          // empty batch: nothing to launch (pointers of empty tensors may be null)
    if (!blob_dev || (!x_i32_dev == !x_f32_dev) || !gt_prob_dev || !zy_prob_dev || !workspace_dev)
        return set_error(NSNP_E_INVALID, "nsnp_pileup_model_forward: null argument (exactly one of x_i32/x_f32)");
    if (precision != NSNP_PREC_FP32 && precision != NSNP_PREC_F16X3 && precision != NSNP_PREC_F16X1) return set_error(NSNP_E_UNSUPPORTED, "unknown precision %d", precision);
    if (n < 0) return set_error(NSNP_E_INVALID, "negative n");
    if (workspace_bytes < nsnp_model_workspace_bytes(n)) return set_error(NSNP_E_WORKSPACE, "model workspace too small");
    if (nsnp_device_count() == 0) return set_error(NSNP_E_NO_DEVICE, "no CUDA device (there is no CPU fallback)");
    if (n == 0) return NSNP_OK;
    const float* blob = (const float*)blob_dev;
    const size_t smem0 = (size_t)(kKP0 * kG + kG + Cfg<0>::S * kKP0) * sizeof(float);
    const size_t smem1 = (size_t)(kKP1 * kG + kG + Cfg<1>::S * kKP1) * sizeof(float);
    static bool attr_done = false;
    if (!attr_done) {
        if (cudaFuncSetAttribute(lstm_dir_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem0) != cudaSuccess ||
            cudaFuncSetAttribute(lstm_dir_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1) != cudaSuccess ||
            cudaFuncSetAttribute(tail_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTailSmem) != cudaSuccess)
            return cuda_status("cudaFuncSetAttribute(lstm_dir_kernel)");
        attr_done = true;
    }
    float* h0 = (float*)((char*)workspace_dev + 256);          // after the header
    const int64_t ch = n < kChunkSites ? n : kChunkSites;
    const bool tc = precision == NSNP_PREC_F16X3 || precision == NSNP_PREC_F16X1;
    // single pass only pays for batches well above the re-evaluation batch; smaller ones run the three-pass path directly
    const bool x1 = precision == NSNP_PREC_F16X1 && n > 4 * (int64_t)kX1Cap;
    float* h16 = h0 + ((ch + 127) / 128 * 128) * kT * 128;
    // n_dev (device-side site count) only makes sense for a single chunk; larger batches are chunked by the host count
    for (int64_t off = 0; off < n; off += ch) {
        const int64_t m = (n - off) < ch ? (n - off) : ch;
        const int32_t* nd = (off == 0 && n <= ch) ? n_dev : nullptr;
        const int32_t* xi = x_i32_dev ? (pos_dev ? x_i32_dev : x_i32_dev + off * kT * kF) : nullptr;       // pos_dev: the count tensor itself
        const float* xf = x_f32_dev ? x_f32_dev + off * kT * kF : nullptr;
        dim3 g0((unsigned)((m + Cfg<0>::S - 1) / Cfg<0>::S), 2), g1((unsigned)((m + Cfg<1>::S - 1) / Cfg<1>::S), 2);
        if (tc) {
            if (int e = launch_lstm_tc(blob_dev, xi, xf, h0, h16 + off * 128, m, pos_dev ? pos_dev + off : nullptr, pos_bias, x1 ? 1 : 3, stream)) return e;
            continue;                                // one tensor-core tail launch over all chunks below
        }
        { ProfScope prof(NSNP_PROF_LSTM0, stream); lstm_dir_kernel<0><<<g0, 256, smem0, stream>>>(blob, xi, xf, nullptr, h0, m, nd); }
        { ProfScope prof(NSNP_PROF_LSTM1, stream); lstm_dir_kernel<1><<<g1, 256, smem1, stream>>>(blob, nullptr, nullptr, h0, h16, m, nd); }
        ProfScope prof(NSNP_PROF_TAIL, stream);
        tail_kernel<<<(unsigned)((m + kTailS - 1) / kTailS), 256, kTailSmem, stream>>>(blob, h16, m, nd, gt_prob_dev + off * 21, zy_prob_dev + off * 3);
        if (int e = cuda_status("pileup model kernels")) return e;
    }
    if (tc) {
        ProfScope prof(NSNP_PROF_TAIL, stream);
        if (int e = launch_tail_tc(blob_dev, h16, n, n <= ch ? n_dev : nullptr, gt_prob_dev, zy_prob_dev, stream)) return e;
    }
    if (precision == NSNP_PREC_F16X1 && cudaMemsetAsync(x1_carve(workspace_dev, n).cnt, 0, 4, stream) != cudaSuccess) return cuda_status("cudaMemsetAsync");
    if (x1) {
        // low-margin sites -> one three-pass batch of kX1Cap sites (layer-0 buffer and h16 of the main pass are free again)
        const X1Work w = x1_carve(workspace_dev, n);
        x1_margin_kernel<<<(unsigned)((n + 7) / 8), 256, 0, stream>>>(gt_prob_dev, zy_prob_dev, n, n <= ch ? n_dev : nullptr, kX1Margin,
                                                                     x_i32_dev, x_f32_dev, pos_dev, pos_bias, w.cnt, w.idx);
        x1_gather_kernel<<<kX1Cap, 128, 0, stream>>>(w.cnt, w.idx, pos_dev, pos_dev ? nullptr : x_i32_dev, x_f32_dev, w.pos_low, w.x_low);
        if (int e = cuda_status("x1 margin / gather kernels")) return e;
        const int32_t* xi_low = pos_dev ? x_i32_dev : (x_i32_dev ? w.x_low : nullptr);
        const float* xf_low = (!pos_dev && x_f32_dev) ? reinterpret_cast<const float*>(w.x_low) : nullptr;
        if (int e = launch_lstm_tc(blob_dev, xi_low, xf_low, h0, h16, kX1Cap, pos_dev ? w.pos_low : nullptr, pos_bias, 3, stream)) return e;
        if (int e = launch_tail_tc(blob_dev, h16, kX1Cap, nullptr, w.gt_low, w.zy_low, stream)) return e;
        x1_scatter_kernel<<<kX1Cap / 8, 256, 0, stream>>>(w.cnt, w.idx, w.gt_low, w.zy_low, gt_prob_dev, zy_prob_dev);
        if (int e = cuda_status("x1 re-evaluation")) return e;
    }
    return NSNP_OK;
}

}  // extern "C"
