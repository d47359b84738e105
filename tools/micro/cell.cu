// LSTM cell-update epilogue in isolation: how close to the MUFU rate (16 ops/clk/SM) does the instruction stream of
// lstm0_pair2_kernel get without the tensor core, TMEM and barriers, and which ingredient costs what?
//   MODE 0: math only (gates from registers)      MODE 1: + fp16 hi/lo split and st.shared of h
//   MODE 2: + fence.proxy.async + __syncthreads per step      MODE 3: + global stores of h (layer-0 output)
#include <cstdio>
#include <cstdint>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
__device__ __forceinline__ float ex2a(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcpa(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ uint32_t h2b(__half2 h) { return *reinterpret_cast<uint32_t*>(&h); }

template <int MODE, int UNITS>   // UNITS hidden units per thread and step (32 for NWQ=2, 16 for NWQ=4)
__global__ void __launch_bounds__(512) cell(float* out, __half* gout, int steps) {
    extern __shared__ __align__(16) unsigned char sm[];
    float c[UNITS];
#pragma unroll
    for (int u = 0; u < UNITS; ++u) c[u] = 0.001f * (threadIdx.x + u);
    float acc = 0.f;
    const int row = threadIdx.x & 127;
    for (int s = 0; s < steps; ++s) {
#pragma unroll
        for (int hb = 0; hb < UNITS / 4; ++hb) {
            float hv[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float base = c[hb * 4 + u] * 0.37f + acc * 1e-3f;            // stand-ins for the four accumulators
                const float xi = fminf(base + 0.1f * u, 36.f), xf = fminf(base - 0.2f, 36.f), xg = fminf(0.5f - base, 36.f), xo = base * 0.5f;
                const float ei = ex2a(xi), ef = ex2a(xf), eg = ex2a(xg), eo = ex2a(xo);
                const float pi = 1.f + ei, pf = 1.f + ef, pg = 1.f + eg;
                const float pig = pi * pg;
                const float num = fmaf(c[hb * 4 + u], pig, fmaf(eg, 2.885f, -2.885f) * pf);
                const float cn = num * rcpa(pf * pig);
                c[hb * 4 + u] = cn;
                const float ec = ex2a(cn);
                hv[u] = (1.f - ec) * rcpa((1.f + eo) * (1.f + ec));
            }
            acc += hv[0] + hv[1] + hv[2] + hv[3];
            if (MODE >= 1) {
                const __half2 h01 = __floats2half2_rn(hv[0], hv[1]), h23 = __floats2half2_rn(hv[2], hv[3]);
                const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
                const uint2 hi = make_uint2(h2b(h01), h2b(h23));
                const uint2 lo = make_uint2(h2b(__floats2half2_rn(hv[0] - f01.x, hv[1] - f01.y)), h2b(__floats2half2_rn(hv[2] - f23.x, hv[3] - f23.y)));
                *reinterpret_cast<uint2*>(sm + (hb >> 1) * 2048 + row * 16 + (hb & 1) * 8) = hi;
                *reinterpret_cast<uint2*>(sm + 16384 + (hb >> 1) * 2048 + row * 16 + (hb & 1) * 8) = lo;
                if (MODE >= 3) {
                    __half* o = gout + ((size_t)(blockIdx.x * steps + s) * 32 + (hb >> 1)) * 1024 + row * 8 + (hb & 1) * 4;
                    *reinterpret_cast<uint2*>(o) = hi; *reinterpret_cast<uint2*>(o + 16 * 1024) = lo;
                }
            }
        }
        if (MODE >= 2) { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); __syncthreads(); }
    }
    if (acc == 123.456f) out[0] = acc;
}

template <int MODE, int UNITS> void run(int threads, int ctas_per_sm, float* d, __half* g, int sms, int clk) {
    const int steps = 2000;
    cudaFuncSetAttribute(cell<MODE, UNITS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
    cell<MODE, UNITS><<<sms * ctas_per_sm, threads, 100 * 1024>>>(d, g, 10); cudaDeviceSynchronize();
    cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
    cudaEventRecord(a); cell<MODE, UNITS><<<sms * ctas_per_sm, threads, 100 * 1024>>>(d, g, steps); cudaEventRecord(b); cudaEventSynchronize(b);
    float ms; cudaEventElapsedTime(&ms, a, b);
    const double mufu = (double)sms * ctas_per_sm * threads * UNITS * 7.0 * steps;
    printf("mode %d units/thread %2d threads %3d x %d CTA/SM: %.2f ms  %.2f MUFU/clk/SM (nominal %d MHz)  err=%s\n", MODE, UNITS, threads, ctas_per_sm, ms,
           mufu / (ms * 1e-3) / sms / (clk * 1e3), clk / 1000, cudaGetErrorString(cudaGetLastError()));
}
int main() {
    cudaDeviceProp p; cudaGetDeviceProperties(&p, 0);
    int clk; cudaDeviceGetAttribute(&clk, cudaDevAttrClockRate, 0);
    float* d; cudaMalloc(&d, 4);
    __half* g; cudaMalloc(&g, (size_t)p.multiProcessorCount * 2 * 2000 * 32 * 1024 * 2 + (1 << 20));
    run<0, 32>(256, 2, d, g, p.multiProcessorCount, clk);
    run<1, 32>(256, 2, d, g, p.multiProcessorCount, clk);
    run<2, 32>(256, 2, d, g, p.multiProcessorCount, clk);
    run<3, 32>(256, 2, d, g, p.multiProcessorCount, clk);
    run<0, 16>(512, 1, d, g, p.multiProcessorCount, clk);
    run<2, 16>(512, 1, d, g, p.multiProcessorCount, clk);
    run<0, 16>(512, 2, d, g, p.multiProcessorCount, clk);
    run<0, 32>(256, 1, d, g, p.multiProcessorCount, clk);
    return 0;
}
