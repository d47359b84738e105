// BASELINE configs[4]: HaplotypeModel s5 on the GPU (SURVEY 8a rows H4, H5).
//
//   hap_feature_kernel   HaplotypeModel/dataset_dev.py:11-87,337-349: read x position matrices (base code, baseQ, MAPQ, HP) ->
//                        26 statistics x {all, HP1, HP2, unphased} + reference code = 105 channels, evaluated in IEEE double
//                        exactly as NumPy does and rounded once to float32 (predict_dev.py:35 `.type(FloatTensor)`): bit-exact.
//   nsnp_hap_model_forward  HaplotypeModel/model_dev.py:59-143: two 3-layer BiLSTM-256 encoders (33 and 11 positions) + Linear,
//                        centre rows, dense/tanh, genotype (10) / zygosity (3) heads, softmax.  fp32 FFMA: the input
//                        projection of a layer is one tiled GEMM over all positions; every recurrent step is one fused
//                        kernel (h W_hh^T tile + projected input -> LSTM cell update in the epilogue: the packed weight rows
//                        interleave the four gates of a unit, so one thread holds i, f, g, o of its unit).  The last layer only
//                        runs the steps its centre output needs.  This path sees the few low-QUAL sites of a sample
//                        (~0.32 GFLOP/site) and is the parity reference of the opt-in tensor-core path
//                        (nsnp_hap_model_tc_forward, haplotype_tc.cu), which runs its tail through sgemm_nt_kernel / heads_kernel.
#include <math.h>
#include "hap_common.cuh"

namespace nsnp {
namespace {

constexpr int kH = 256, kG = 4 * kH, kDim = 105, kLayers = 3;
constexpr int kLp = 33, kLh = 11;

// ------------------------------------------------------------------------------------------------ features
__global__ void __launch_bounds__(128) hap_feature_kernel(const int32_t* __restrict__ seq, const int32_t* __restrict__ bq,
                                                          const int32_t* __restrict__ mq, const int32_t* __restrict__ hp,
                                                          const int32_t* __restrict__ refcode, int depth, int L, float* __restrict__ out)
{
    extern __shared__ uint8_t rowtag[];                         // per read row: bit t set when any position carries HP tag t
    const int64_t site = blockIdx.x;
    const int32_t* s = seq + site * depth * L; const int32_t* b = bq + site * depth * L;
    const int32_t* m = mq + site * depth * L; const int32_t* h = hp + site * depth * L;
    for (int d = threadIdx.x; d < depth; d += blockDim.x) {
        uint32_t t = 0;
        for (int l = 0; l < L; ++l) { const int v = h[d * L + l]; if (v >= 1 && v <= 3) t |= 1u << v; }
        rowtag[d] = (uint8_t)t;
    }
    __syncthreads();
    float* o = out + site * kDim * L;
    for (int idx = threadIdx.x; idx < 4 * L; idx += blockDim.x) {
        const int g = idx / L, l = idx % L;
        long long cnt[5] = {0, 0, 0, 0, 0}, bs[4] = {0, 0, 0, 0}, ms[4] = {0, 0, 0, 0};
        for (int d = 0; d < depth; ++d) {
            if (g && !((rowtag[d] >> g) & 1u)) continue;
            const int v = s[d * L + l];
            const int c = v == -1 ? 4 : (v >= 1 && v <= 4) ? v - 1 : -1;
            if (c < 0) continue;
            ++cnt[c];
            if (c < 4) { bs[c] += b[d * L + l]; ms[c] += m[d * L + l]; }
        }
        const double total = (double)(cnt[0] + cnt[1] + cnt[2] + cnt[3] + cnt[4]) + 1e-6;      // dataset_dev.py:17
        float* og = o + (size_t)g * 26 * L + l;
        for (int c = 0; c < 5; ++c) { og[c * L] = (float)((double)cnt[c] / total); og[(5 + c) * L] = (float)cnt[c]; }
        for (int c = 0; c < 4; ++c) {
            og[(10 + c) * L] = (float)bs[c]; og[(14 + c) * L] = (float)((double)bs[c] / ((double)cnt[c] + 1e-9));   // dataset_dev.py:30-33
            og[(18 + c) * L] = (float)ms[c]; og[(22 + c) * L] = (float)((double)ms[c] / ((double)cnt[c] + 1e-9));
        }
    }
    for (int l = threadIdx.x; l < L; l += blockDim.x) o[(size_t)104 * L + l] = (float)refcode[site * L + l];
}

// ------------------------------------------------------------------------------------------------ model: packed weights
// per encoder e, layer l, direction d:  W_ih' [1024][in]  W_hh' [1024][256]  b' [1024]   rows interleaved: row' = unit * 4 + gate
// then per encoder: proj_w [256][512], proj_b [256]; then dense_w [256][512], dense_b, gt_w [10][256], gt_b, zy_w [3][256], zy_b
struct Blob {
    size_t w_ih[2][kLayers][2], w_hh[2][kLayers][2], b[2][kLayers][2], proj_w[2], proj_b[2], dense_w, dense_b, gt_w, gt_b, zy_w, zy_b, total;
};
inline Blob blob_layout() {
    Blob L; size_t o = 0;
    for (int e = 0; e < 2; ++e)
        for (int l = 0; l < kLayers; ++l)
            for (int d = 0; d < 2; ++d) {
                const int in = l == 0 ? kDim : 2 * kH;
                L.w_ih[e][l][d] = o; o += (size_t)kG * in;
                L.w_hh[e][l][d] = o; o += (size_t)kG * kH;
                L.b[e][l][d] = o; o += kG;
            }
    for (int e = 0; e < 2; ++e) { L.proj_w[e] = o; o += (size_t)kH * 2 * kH; L.proj_b[e] = o; o += kH; }
    L.dense_w = o; o += (size_t)kH * 2 * kH; L.dense_b = o; o += kH;
    L.gt_w = o; o += 10 * kH; L.gt_b = o; o += 10; L.zy_w = o; o += 3 * kH; L.zy_b = o; o += 3;
    L.total = o;
    return L;
}

// C[M][N] = A[M][K] . B[N][K]^T + bias[N]      (A rows lda apart, C rows ldc apart); 64x64 tile, 16-wide k slices, 4x4 per thread
__global__ void __launch_bounds__(256) sgemm_nt_kernel(const float* __restrict__ A, int64_t lda, const float* __restrict__ B, const float* __restrict__ bias,
                                                       float* __restrict__ C, int64_t ldc, int64_t M, int N, int K, int act_tanh)
{
    __shared__ float As[16][64 + 4], Bs[16][64 + 4];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int64_t m0 = (int64_t)blockIdx.y * 64; const int n0 = blockIdx.x * 64;
    float acc[4][4] = {};
    for (int k0 = 0; k0 < K; k0 += 16) {
        for (int i = threadIdx.x; i < 64 * 16; i += 256) {
            const int r = i >> 4, c = i & 15;
            As[c][r] = (m0 + r < M && k0 + c < K) ? A[(m0 + r) * lda + k0 + c] : 0.f;
            Bs[c][r] = (n0 + r < N && k0 + c < K) ? B[(int64_t)(n0 + r) * K + k0 + c] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            float a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) { a[i] = As[k][ty * 4 + i]; b[i] = Bs[k][tx * 4 + i]; }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int64_t m = m0 + ty * 4 + i; const int n = n0 + tx * 4 + j;
            if (m < M && n < N) { float v = acc[i][j] + (bias ? bias[n] : 0.f); if (act_tanh) v = tanhf(v); C[m * ldc + n] = v; }
        }
}

// One LSTM step for all sites: gates = xp[site][t][.] + h_prev . W_hh'^T, cell update in the epilogue.
// xp rows are (site * L + t) * 1024; y: layer output [site][L][512] (this direction's half), may be null; h/c: [n][256].
__global__ void __launch_bounds__(256) lstm_step_kernel(const float* __restrict__ xp, int L, int t, const float* __restrict__ whh,
                                                        const float* __restrict__ h_prev, float* __restrict__ h_next, float* __restrict__ c,
                                                        float* __restrict__ y, int y_off, int64_t n, int first)
{
    __shared__ float As[16][64 + 4], Bs[16][64 + 4];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int64_t m0 = (int64_t)blockIdx.y * 64; const int n0 = blockIdx.x * 64;          // 64 gate columns = 16 units
    float acc[4][4] = {};
    if (!first) {
        for (int k0 = 0; k0 < kH; k0 += 16) {
            for (int i = threadIdx.x; i < 64 * 16; i += 256) {
                const int r = i >> 4, cc = i & 15;
                As[cc][r] = (m0 + r < n) ? h_prev[(m0 + r) * kH + k0 + cc] : 0.f;
                Bs[cc][r] = whh[(int64_t)(n0 + r) * kH + k0 + cc];
            }
            __syncthreads();
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                float a[4], b[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) { a[i] = As[k][ty * 4 + i]; b[i] = Bs[k][tx * 4 + i]; }
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
            }
            __syncthreads();
        }
    }
    const int unit = (n0 >> 2) + tx;                                                       // this thread's 4 columns = i f g o of one unit
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int64_t m = m0 + ty * 4 + i;
        if (m >= n) continue;
        const float4 x4 = *reinterpret_cast<const float4*>(xp + ((m * L + t) * (int64_t)kG) + n0 + tx * 4);
        const float gi = acc[i][0] + x4.x, gf = acc[i][1] + x4.y, gg = acc[i][2] + x4.z, go = acc[i][3] + x4.w;
        const float ig = 1.f / (1.f + expf(-gi)), fg = 1.f / (1.f + expf(-gf)), og = 1.f / (1.f + expf(-go));
        const float cp = first ? 0.f : c[m * kH + unit];
        const float cn = fg * cp + ig * tanhf(gg);
        const float hn = og * tanhf(cn);
        c[m * kH + unit] = cn;
        h_next[m * kH + unit] = hn;
        if (y) y[(m * L + t) * (int64_t)(2 * kH) + y_off + unit] = hn;
    }
}

// [n][105][L] -> [n][L][105]   (model_dev.py:136-137 permute(0, 2, 1))
__global__ void permute_kernel(const float* __restrict__ x, float* __restrict__ y, int64_t n, int L)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * kDim * L) return;
    const int64_t s = i / (kDim * L); const int r = (int)(i % (kDim * L)); const int l = r / kDim, ch = r % kDim;
    y[i] = x[(s * kDim + ch) * L + l];
}

// centre rows of both encoders' last layers: cat[n][1024] = [fwd_p | rev_p | fwd_h | rev_h] handled by the caller's pointers
__global__ void heads_kernel(const float* __restrict__ hid, const float* __restrict__ gw, const float* __restrict__ gb,
                             const float* __restrict__ zw, const float* __restrict__ zb, float* __restrict__ gt, float* __restrict__ zy, int64_t n)
{
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    const float* h = hid + s * kH;
    float lg[10], lz[3];
    for (int k = 0; k < 10; ++k) { float a = gb[k]; for (int j = 0; j < kH; ++j) a = fmaf(h[j], gw[k * kH + j], a); lg[k] = a; }
    for (int k = 0; k < 3; ++k) { float a = zb[k]; for (int j = 0; j < kH; ++j) a = fmaf(h[j], zw[k * kH + j], a); lz[k] = a; }
    float mx = lg[0]; for (int k = 1; k < 10; ++k) mx = fmaxf(mx, lg[k]);
    float sum = 0.f; for (int k = 0; k < 10; ++k) { lg[k] = expf(lg[k] - mx); sum += lg[k]; }
    for (int k = 0; k < 10; ++k) gt[s * 10 + k] = lg[k] / sum;
    mx = fmaxf(lz[0], fmaxf(lz[1], lz[2]));
    sum = 0.f; for (int k = 0; k < 3; ++k) { lz[k] = expf(lz[k] - mx); sum += lz[k]; }
    for (int k = 0; k < 3; ++k) zy[s * 3 + k] = lz[k] / sum;
}

constexpr int64_t kChunk = 2048;            // sites per pass: bounds the workspace (projected inputs: chunk * 33 * 1024 floats)

struct Ws { float *xperm, *ya, *yb, *xp, *h0, *h1, *c, *cat, *enc, *hid; };
inline size_t carve_ws(void* base, int64_t n, Ws* w) {
    const int64_t m = n < kChunk ? n : kChunk;
    size_t off = 0;
    auto take = [&](size_t floats) { float* p = base ? (float*)((char*)base + off) : nullptr; off += (floats * 4 + 255) / 256 * 256; return p; };
    w->xperm = take((size_t)m * kLp * kDim);
    w->ya = take((size_t)m * kLp * 2 * kH);
    w->yb = take((size_t)m * kLp * 2 * kH);
    w->xp = take((size_t)m * kLp * kG);
    w->h0 = take((size_t)m * kH); w->h1 = take((size_t)m * kH); w->c = take((size_t)m * kH);
    w->cat = take((size_t)m * 2 * kH);          // centre rows of the last layer, fwd | rev
    w->enc = take((size_t)m * 2 * kH);          // output_proj of both encoders, pileup | haplotype
    w->hid = take((size_t)m * kH);
    return off;
}

}  // namespace

// the fp32 tail kernels, for the tensor-core path (haplotype_tc.cu)
int hap_sgemm_nt(const float* A, int64_t lda, const float* B, const float* bias, float* C, int64_t ldc, int64_t M, int N, int K, int act_tanh,
                 cudaStream_t st)
{
    sgemm_nt_kernel<<<dim3((unsigned)((N + 63) / 64), (unsigned)((M + 63) / 64)), 256, 0, st>>>(A, lda, B, bias, C, ldc, M, N, K, act_tanh);
    return cuda_status("sgemm_nt_kernel");
}

int hap_heads(const float* hid, const float* gw, const float* gb, const float* zw, const float* zb, float* gt, float* zy, int64_t n, cudaStream_t st)
{
    heads_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(hid, gw, gb, zw, zb, gt, zy, n);
    return cuda_status("heads_kernel");
}

}  // namespace nsnp

using namespace nsnp;

extern "C" {

int nsnp_hap_features(const int32_t* seq_dev, const int32_t* bq_dev, const int32_t* mq_dev, const int32_t* hp_dev, const int32_t* refcode_dev,
                      int64_t n, int32_t depth, int32_t L, float* out_dev, void* stream_)
{
    if (n < 0 || depth < 0 || L <= 0 || (n > 0 && (!seq_dev || !bq_dev || !mq_dev || !hp_dev || !refcode_dev || !out_dev)))
        return set_error(NSNP_E_INVALID, "nsnp_hap_features: bad argument");
    if (depth > 40000) return set_error(NSNP_E_UNSUPPORTED, "nsnp_hap_features: more than 40000 read rows per site");
    if (n == 0) return NSNP_OK;
    if (nsnp_device_count() == 0) return set_error(NSNP_E_NO_DEVICE, "no CUDA device (there is no CPU fallback)");
    hap_feature_kernel<<<(unsigned)n, 128, (size_t)depth + 16, (cudaStream_t)stream_>>>(seq_dev, bq_dev, mq_dev, hp_dev, refcode_dev, depth, L, out_dev);
    return cuda_status("hap_feature_kernel");
}

size_t nsnp_hap_model_blob_bytes(void) { return blob_layout().total * 4; }

int nsnp_hap_model_pack_weights(const nsnp_hap_weights_t* w, void* host_blob, size_t blob_bytes)
{
    if (!w || !host_blob) return set_error(NSNP_E_INVALID, "nsnp_hap_model_pack_weights: null argument");
    const Blob L = blob_layout();
    if (blob_bytes < L.total * 4) return set_error(NSNP_E_WORKSPACE, "haplotype model blob: need %zu bytes", L.total * 4);
    float* o = (float*)host_blob;
    for (int e = 0; e < 2; ++e)
        for (int l = 0; l < kLayers; ++l)
            for (int d = 0; d < 2; ++d) {
                const int in = l == 0 ? kDim : 2 * kH;
                const float *wi = w->w_ih[e][l][d], *wh = w->w_hh[e][l][d], *bi = w->b_ih[e][l][d], *bh = w->b_hh[e][l][d];
                if (!wi || !wh || !bi || !bh) return set_error(NSNP_E_INVALID, "nsnp_hap_model_pack_weights: missing LSTM tensor");
                for (int g = 0; g < 4; ++g)                          // PyTorch gate order i f g o, rows g * 256 + unit
                    for (int u = 0; u < kH; ++u) {
                        const size_t src = (size_t)g * kH + u, dst = (size_t)u * 4 + g;
                        memcpy(o + L.w_ih[e][l][d] + dst * in, wi + src * in, (size_t)in * 4);
                        memcpy(o + L.w_hh[e][l][d] + dst * kH, wh + src * kH, (size_t)kH * 4);
                        o[L.b[e][l][d] + dst] = bi[src] + bh[src];
                    }
            }
    for (int e = 0; e < 2; ++e) {
        if (!w->proj_w[e] || !w->proj_b[e]) return set_error(NSNP_E_INVALID, "nsnp_hap_model_pack_weights: missing output_proj");
        memcpy(o + L.proj_w[e], w->proj_w[e], (size_t)kH * 2 * kH * 4); memcpy(o + L.proj_b[e], w->proj_b[e], kH * 4);
    }
    if (!w->dense_w || !w->dense_b || !w->gt_w || !w->gt_b || !w->zy_w || !w->zy_b) return set_error(NSNP_E_INVALID, "nsnp_hap_model_pack_weights: missing head tensor");
    memcpy(o + L.dense_w, w->dense_w, (size_t)kH * 2 * kH * 4); memcpy(o + L.dense_b, w->dense_b, kH * 4);
    memcpy(o + L.gt_w, w->gt_w, 10 * kH * 4); memcpy(o + L.gt_b, w->gt_b, 10 * 4);
    memcpy(o + L.zy_w, w->zy_w, 3 * kH * 4); memcpy(o + L.zy_b, w->zy_b, 3 * 4);
    return NSNP_OK;
}

size_t nsnp_hap_model_workspace_bytes(int64_t n) { Ws w; return carve_ws(nullptr, n < 1 ? 1 : n, &w); }

int nsnp_hap_model_forward(const void* blob_dev, const float* xp_dev, const float* xh_dev, int64_t n, float* gt_prob_dev, float* zy_prob_dev,
                           void* workspace_dev, size_t workspace_bytes, void* stream_)
{
    cudaStream_t st = (cudaStream_t)stream_;
    if (n < 0 || (n > 0 && (!blob_dev || !xp_dev || !xh_dev || !gt_prob_dev || !zy_prob_dev || !workspace_dev)))
        return set_error(NSNP_E_INVALID, "nsnp_hap_model_forward: bad argument");
    if (n == 0) return NSNP_OK;
    if (nsnp_device_count() == 0) return set_error(NSNP_E_NO_DEVICE, "no CUDA device (there is no CPU fallback)");
    Ws w;
    if (carve_ws(workspace_dev, n, &w) > workspace_bytes) return set_error(NSNP_E_WORKSPACE, "haplotype model workspace too small");
    const Blob B = blob_layout();
    const float* blob = (const float*)blob_dev;
    for (int64_t s0 = 0; s0 < n; s0 += kChunk) {
        const int64_t m = n - s0 < kChunk ? n - s0 : kChunk;
        for (int e = 0; e < 2; ++e) {
            const int L = e == 0 ? kLp : kLh, ctr = L / 2;
            const float* x = (e == 0 ? xp_dev : xh_dev) + s0 * kDim * L;
            permute_kernel<<<(unsigned)((m * kDim * L + 255) / 256), 256, 0, st>>>(x, w.xperm, m, L);
            const float* in = w.xperm; int in_dim = kDim;
            float* outs[2] = {w.ya, w.yb};
            for (int l = 0; l < kLayers; ++l) {
                float* y = outs[l & 1];
                const bool last = l == kLayers - 1;
                for (int d = 0; d < 2; ++d) {
                    // input projection of every position: [m * L, in] x [1024, in]^T + (b_ih + b_hh)
                    sgemm_nt_kernel<<<dim3(kG / 64, (unsigned)((m * L + 63) / 64)), 256, 0, st>>>(in, in_dim, blob + B.w_ih[e][l][d], blob + B.b[e][l][d],
                                                                                               w.xp, kG, m * L, kG, in_dim, 0);
                    float* hp = w.h0; float* hn = w.h1;
                    const int t_begin = d == 0 ? 0 : L - 1, t_end = last ? ctr : (d == 0 ? L - 1 : 0), dt = d == 0 ? 1 : -1;
                    for (int t = t_begin;; t += dt) {
                        lstm_step_kernel<<<dim3(kG / 64, (unsigned)((m + 63) / 64)), 256, 0, st>>>(w.xp, L, t, blob + B.w_hh[e][l][d], hp, hn, w.c,
                                                                                                 last ? nullptr : y, d * kH, m, t == t_begin);
                        float* tmp = hp; hp = hn; hn = tmp;
                        if (t == t_end) break;
                    }
                    if (last)                                   // centre state of this direction -> cat[:, d * 256 ...]
                        cudaMemcpy2DAsync(w.cat + d * kH, 2 * kH * 4, hp, kH * 4, kH * 4, (size_t)m, cudaMemcpyDeviceToDevice, st);
                }
                in = y; in_dim = 2 * kH;
            }
            // output_proj at the centre row (model_dev.py:84, :105-106)
            sgemm_nt_kernel<<<dim3(kH / 64, (unsigned)((m + 63) / 64)), 256, 0, st>>>(w.cat, 2 * kH, blob + B.proj_w[e], blob + B.proj_b[e],
                                                                                   w.enc + e * kH, 2 * kH, m, kH, 2 * kH, 0);
        }
        sgemm_nt_kernel<<<dim3(kH / 64, (unsigned)((m + 63) / 64)), 256, 0, st>>>(w.enc, 2 * kH, blob + B.dense_w, blob + B.dense_b, w.hid, kH, m, kH, 2 * kH, 1);
        heads_kernel<<<(unsigned)((m + 127) / 128), 128, 0, st>>>(w.hid, blob + B.gt_w, blob + B.gt_b, blob + B.zy_w, blob + B.zy_b,
                                                                 gt_prob_dev + s0 * 10, zy_prob_dev + s0 * 3, m);
    }
    return cuda_status("nsnp_hap_model_forward");
}

}  // extern "C"
