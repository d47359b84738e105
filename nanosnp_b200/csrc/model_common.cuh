// Shared constants of the PileupModel kernels: dimensions and the packed weight blob layout.
#pragma once
#include "common.cuh"

namespace nsnp {

constexpr int kH = 64;               // hidden size
constexpr int kG = 256;              // 4 gates x 64
constexpr int kT = NSNP_WINDOW;      // 33
constexpr int kF = NSNP_CHANNELS;    // 18
constexpr int kMid = NSNP_FLANK;     // 16
constexpr int kKP0 = 84;             // [x 18 | pad 2 | h 64]
constexpr int kIn0 = 20;
constexpr int kKP1 = 192;            // [l0 fwd 64 | l0 rev 64 | h 64]
constexpr int kIn1 = 128;

// blob layout (floats)
constexpr size_t kOffW0 = 0;                                        // [2][kKP0][256]
constexpr size_t kOffB0 = kOffW0 + 2 * (size_t)kKP0 * kG;           // [2][256]
constexpr size_t kOffW1 = kOffB0 + 2 * kG;                          // [2][kKP1][256]
constexpr size_t kOffB1 = kOffW1 + 2 * (size_t)kKP1 * kG;           // [2][256]
constexpr size_t kOffProjW = kOffB1 + 2 * kG;                       // [128 k][128]
constexpr size_t kOffProjB = kOffProjW + 128 * 128;
constexpr size_t kOffDenseW = kOffProjB + 128;                      // [128 k][256]
constexpr size_t kOffDenseB = kOffDenseW + 128 * 256;
constexpr size_t kOffHeadW = kOffDenseB + 256;                      // [256 k][24]
constexpr size_t kOffHeadB = kOffHeadW + 256 * 24;
constexpr size_t kBlobFloats = kOffHeadB + 24 + 8;


// ---- tensor-core section of the blob (fp16 hi/lo split weights in the UMMA K-major no-swizzle layout) ----
//   B[k/8][n][k%8] halfs, n = unit_block*32 + unit_half*16 + gate*4 + unit_in_half  (TMEM column order: every
//   16 columns hold i,f,g,o of 4 hidden units, so the epilogue can pipeline 16-column TMEM loads)
//   layer 0: K = 96  = [x 0..17 | bias column 18 | pad ..31 | h 32..95]; lo part of k < 32 is pre-scaled by 2^10, hi part
//            of k < 32 by 2^8 (the inputs are staged as x 2^-8, see kTcInScale)
//   layer 1: K = 192 = [l0 out 0..127 | h 128..191]; its bias is added in the epilogue (a bias column would cost a whole
//            k-block = 2 of 38 MMAs per step on a tensor-bound kernel): float [2 dirs][256] in column order n, at kOffTcBias1
constexpr int kTcK0 = 96, kTcIn0 = 32, kTcK1 = 192, kTcIn1 = 128;
constexpr float kTcLoScale = 1024.0f;
// Layer-0 inputs (counts) are staged as x 2^-8 with a saturating fp16 conversion, so that counts up to 65504 x 2^8 =
// 16 769 024 keep their fp16 hi/lo split (fp16 itself ends at 65504: a raw count of 65 520 would round to inf and turn the
// gates into inf - inf = NaN); larger ones saturate at twice that.  The hi weight halves of those columns carry 2^8 back: every
// product, hence every accumulator, is the unscaled one for integer counts below 65 520.  It limits those weights to
// |w| < 65504 / 2^8 / (2 log2 e).
constexpr float kTcInScale = 256.0f;
constexpr size_t kTcBytes0 = (size_t)kTcK0 * 256 * 2;       // one (hi or lo) array of one direction
constexpr size_t kTcBytes1 = (size_t)kTcK1 * 256 * 2;
constexpr size_t kOffTcBytes = ((kBlobFloats * 4 + 255) / 256) * 256;
// order: L0 d0 hi, L0 d0 lo, L0 d1 hi, L0 d1 lo, L1 d0 hi, L1 d0 lo, L1 d1 hi, L1 d1 lo
constexpr size_t tc_off(int layer, int dir, int lo) {
    return kOffTcBytes + (layer == 0 ? (size_t)(dir * 2 + lo) * kTcBytes0 : 4 * kTcBytes0 + (size_t)(dir * 2 + lo) * kTcBytes1);
}
// tail: W' = dense o output_proj, [k/8 = 16][n = 256 dense outputs][k%8] halfs, hi then lo (64 KB each)
constexpr size_t kTcBytesTail = (size_t)128 * 256 * 2;
constexpr size_t kOffTcTail = kOffTcBytes + 4 * kTcBytes0 + 4 * kTcBytes1;
constexpr size_t kOffTcBias1 = kOffTcTail + 2 * kTcBytesTail;
constexpr size_t kBlobBytes = kOffTcBias1 + 2 * 256 * sizeof(float);

// fp16 hi/lo tensor-core LSTM (model_tc.cu).  h0: fp16 [site][33][2][128]; h16: fp32 [site][128].
int launch_lstm_tc(const void* blob, const int32_t* xi, const float* xf, void* h0, float* h16, int64_t m, const int32_t* pos, int64_t pos_bias, int npass, cudaStream_t stream);
int pack_tc_weights(const nsnp_model_weights_t* w, unsigned char* blob);
// (dense o output_proj) + tanh on the tensor cores, heads + softmax on the FMA pipe (model_tc.cu)
int launch_tail_tc(const void* blob, const float* h16, int64_t n_max, const int32_t* n_dev, float* gt, float* zy, cudaStream_t stream);
int debug_tc_gates(const void* blob, const int32_t* xi, int layer, int dir, int cg, const void* h0, float* gates_out, int64_t m, cudaStream_t stream);

}  // namespace nsnp
