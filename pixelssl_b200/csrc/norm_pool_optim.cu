// NHWC BatchNorm (train / eval, forward / backward), 3x3/2 max-pool, fused SGD+EMA.
// All HBM-bound: every kernel moves 128-bit vectors along the channel dimension, one pass per
// tensor, with per-channel reductions finished in fp64 atomics (tiny: 2*C doubles per layer).
#include "common.cuh"
#include <stdlib.h>
#include <math_constants.h>
#include <cuda_fp16.h>

// ------------------------------------------------------------------------------------------
// thread layout shared by the per-channel reductions: a block covers CW = 4*TX channels
// (TX lanes x float4) and strides over rows with TY = 256/TX row lanes.
// ------------------------------------------------------------------------------------------
struct RedLayout { int TX, TY, colBlocks, rowBlocks; int64_t rowsPerBlock; };

static RedLayout red_layout(int64_t rows, int C) {
    RedLayout L;
    int c4 = C / 4;
    L.TX = c4 >= 32 ? 32 : (c4 >= 16 ? 16 : (c4 >= 8 ? 8 : (c4 >= 4 ? 4 : (c4 >= 2 ? 2 : 1))));
    L.TY = 256 / L.TX;
    L.colBlocks = (int)pxl_cdiv(c4, L.TX);
    // 8 CTAs per SM in total, but every CTA ends with 2 fp64 atomics per channel: cap the row blocks (= atomics per
    // address) at one per 256 KB of tensor, at least one per SM - on a 17 MB layer ~550 contended atomics per
    // address cost more than streaming the layer (tools/bench_bn.py: 45 us vs 20 us)
    int64_t target = (int64_t)PXL_NUM_SMS * 8 / L.colBlocks;
    int64_t cap = rows * C / 65536;
    if (cap < PXL_NUM_SMS) cap = PXL_NUM_SMS;
    if (target > cap) target = cap;
    if (target < 1) target = 1;
    int64_t rpb = pxl_cdiv(rows, target);
    if (rpb < L.TY * 4) rpb = L.TY * 4;
    L.rowsPerBlock = rpb;
    L.rowBlocks = (int)pxl_cdiv(rows, rpb);
    return L;
}

__device__ __forceinline__ float4 f4add(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
__device__ __forceinline__ float4 f4mul(float4 a, float4 b) { return make_float4(a.x * b.x, a.y * b.y, a.z * b.z, a.w * b.w); }

// reduce two float4 accumulators over the TY row-lanes of the block, then fp64 atomics
__device__ __forceinline__ void block_reduce_cols(float4 s0, float4 s1, int TX, int TY, int c4, int c4max,
                                                  double* out0, double* out1) {
    __shared__ float4 sm0[256];
    __shared__ float4 sm1[256];
    const int tx = threadIdx.x % TX, ty = threadIdx.x / TX;
    sm0[threadIdx.x] = s0;
    sm1[threadIdx.x] = s1;
    __syncthreads();
    for (int h = TY >> 1; h > 0; h >>= 1) {
        if (ty < h) {
            sm0[threadIdx.x] = f4add(sm0[threadIdx.x], sm0[threadIdx.x + h * TX]);
            sm1[threadIdx.x] = f4add(sm1[threadIdx.x], sm1[threadIdx.x + h * TX]);
        }
        __syncthreads();
    }
    if (ty == 0 && c4 < c4max) {
        float4 a = sm0[tx], b = sm1[tx];
        atomicAdd(out0 + 4 * c4 + 0, (double)a.x); atomicAdd(out0 + 4 * c4 + 1, (double)a.y);
        atomicAdd(out0 + 4 * c4 + 2, (double)a.z); atomicAdd(out0 + 4 * c4 + 3, (double)a.w);
        atomicAdd(out1 + 4 * c4 + 0, (double)b.x); atomicAdd(out1 + 4 * c4 + 1, (double)b.y);
        atomicAdd(out1 + 4 * c4 + 2, (double)b.z); atomicAdd(out1 + 4 * c4 + 3, (double)b.w);
    }
}


// ------------------------------------------------------------------------------------------
// fp16-pair outputs (csrc/h16_prep.cu): v*s = hi + lo, 4 channels -> one 8-byte store per plane.
// Returns true when a value had to be clipped to the fp16 range.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ bool h16_store4(float4 v, float s, uint2* __restrict__ hi, uint2* __restrict__ lo, int64_t i) {
    const float t[4] = {v.x * s, v.y * s, v.z * s, v.w * s};
    unsigned short h[4], l[4];
    bool clipped = false;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float c = fminf(fmaxf(t[k], -65504.f), 65504.f);
        clipped |= (c != t[k]) && (t[k] == t[k]);
        const __half hh = __float2half_rn(c);
        h[k] = __half_as_ushort(hh);
        l[k] = __half_as_ushort(__float2half_rn(c - __half2float(hh)));
    }
    hi[i] = make_uint2((uint32_t)h[0] | ((uint32_t)h[1] << 16), (uint32_t)h[2] | ((uint32_t)h[3] << 16));
    if (lo) lo[i] = make_uint2((uint32_t)l[0] | ((uint32_t)l[1] << 16), (uint32_t)l[2] | ((uint32_t)l[3] << 16));
    return clipped;
}

// ------------------------------------------------------------------------------------------
// forward statistics: sums[0:C] += sum x ; sums[C:2C] += sum x^2
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
bn_stats_kernel(const float* __restrict__ x, int64_t rows, int C, int TX, int TY, int64_t rowsPerBlock,
                double* __restrict__ sums) {
    const int tx = threadIdx.x % TX, ty = threadIdx.x / TX;
    const int c4 = blockIdx.y * TX + tx, c4max = C >> 2;
    const int64_t r0 = (int64_t)blockIdx.x * rowsPerBlock;
    const int64_t r1 = min(rows, r0 + rowsPerBlock);
    float4 s = make_float4(0, 0, 0, 0), q = make_float4(0, 0, 0, 0);
    if (c4 < c4max) {
        const float4* xp = reinterpret_cast<const float4*>(x) + c4;
#pragma unroll 8
        for (int64_t r = r0 + ty; r < r1; r += TY) {
            float4 v = __ldg(xp + r * c4max);
            s = f4add(s, v);
            q = f4add(q, f4mul(v, v));
        }
    }
    block_reduce_cols(s, q, TX, TY, c4, c4max, sums, sums + C);
}

extern "C" int pxl_bn_stats(const float* x, int64_t rows, int C, double* sums, void* stream) {
    if (!x || !sums || rows <= 0 || C <= 0 || (C & 3)) return PXL_ERR_BAD_ARG;
    RedLayout L = red_layout(rows, C);
    dim3 grid(L.rowBlocks, L.colBlocks);
    bn_stats_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, rows, C, L.TX, L.TY, L.rowsPerBlock, sums);
    PXL_CHECK_LAUNCH();
    return 0;
}

__global__ void bn_finalize_kernel(const double* __restrict__ sums, double count, int C,
                                   const float* __restrict__ gamma, const float* __restrict__ beta,
                                   float* running_mean, float* running_var, float momentum, float eps,
                                   int clamp_mode, float* mean, float* invstd, float* scale, float* shift) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const double m = sums[c] / count;
    double var = sums[C + c] / count - m * m;     // biased
    if (var < 0.0) var = 0.0;
    const float mf = (float)m;
    float is;
    if (clamp_mode) is = 1.0f / sqrtf(fmaxf((float)var, eps));   // batchnorm.py:125 multi-replica path
    else is = 1.0f / sqrtf((float)var + eps);                    // F.batch_norm path (batchnorm.py:50-53)
    if (running_mean) {
        const double unbiased = count > 1.0 ? var * count / (count - 1.0) : var;
        running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * mf;
        running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
    }
    mean[c] = mf;
    invstd[c] = is;
    const float sc = gamma[c] * is;
    scale[c] = sc;
    shift[c] = beta[c] - mf * sc;
}

extern "C" int pxl_bn_finalize(const double* sums, double count, int C, const float* gamma, const float* beta,
                               float* running_mean, float* running_var, float momentum, float eps,
                               int clamp_mode, float* mean, float* invstd, float* scale, float* shift,
                               void* stream) {
    if (!sums || !gamma || !beta || !mean || !invstd || !scale || !shift || C <= 0 || count <= 0) return PXL_ERR_BAD_ARG;
    bn_finalize_kernel<<<(C + 127) / 128, 128, 0, (cudaStream_t)stream>>>(sums, count, C, gamma, beta, running_mean, running_var,
                                                                         momentum, eps, clamp_mode, mean, invstd, scale, shift);
    PXL_CHECK_LAUNCH();
    return 0;
}

__global__ void bn_eval_coeffs_kernel(int C, const float* gamma, const float* beta, const float* rm,
                                      const float* rv, float eps, float* scale, float* shift) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const float sc = gamma[c] / sqrtf(rv[c] + eps);
    scale[c] = sc;
    shift[c] = beta[c] - rm[c] * sc;
}

extern "C" int pxl_bn_eval_coeffs(int C, const float* gamma, const float* beta, const float* running_mean,
                                  const float* running_var, float eps, float* scale, float* shift, void* stream) {
    if (!gamma || !beta || !running_mean || !running_var || !scale || !shift || C <= 0) return PXL_ERR_BAD_ARG;
    bn_eval_coeffs_kernel<<<(C + 127) / 128, 128, 0, (cudaStream_t)stream>>>(C, gamma, beta, running_mean, running_var, eps, scale, shift);
    PXL_CHECK_LAUNCH();
    return 0;
}

// ------------------------------------------------------------------------------------------
// apply: y = x*scale + shift (+ residual) (ReLU)        8 B/elem (12 with residual)
// ------------------------------------------------------------------------------------------
// ReLU mask of a float4 (bit k: lane k of the result is > 0): 1 byte per 4 values, written by the forward apply of a
// block output and read by its backward instead of the fp32 result (0.25 B/element instead of 4, twice per step)
__device__ __forceinline__ uint8_t relu_mask4(const float4& v) {
    return (uint8_t)((v.x > 0.f ? 1u : 0u) | (v.y > 0.f ? 2u : 0u) | (v.z > 0.f ? 4u : 0u) | (v.w > 0.f ? 8u : 0u));
}
__device__ __forceinline__ void apply_mask4(float4& d, unsigned m) {
    d.x = (m & 1u) ? d.x : 0.f; d.y = (m & 2u) ? d.y : 0.f; d.z = (m & 4u) ? d.z : 0.f; d.w = (m & 8u) ? d.w : 0.f;
}

template <bool RES, bool RELU>
__global__ void __launch_bounds__(256)
bn_apply_kernel(const float4* __restrict__ x, const float4* __restrict__ scale, const float4* __restrict__ shift,
                const float4* __restrict__ res, float4* __restrict__ y, int64_t n4, int c4max,
                uint2* __restrict__ hi, uint2* __restrict__ lo, float hscale, int* __restrict__ sat,
                uint8_t* __restrict__ mask) {
    PXL_PDL_SYNC();
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    bool clipped = false;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        const int c = (int)(i % c4max);
        float4 v = __ldcs(x + i);
        const float4 sc = __ldg(scale + c), sh = __ldg(shift + c);
        v.x = fmaf(v.x, sc.x, sh.x); v.y = fmaf(v.y, sc.y, sh.y);
        v.z = fmaf(v.z, sc.z, sh.z); v.w = fmaf(v.w, sc.w, sh.w);
        if (RES) { float4 r = __ldcs(res + i); v = f4add(v, r); }
        if (RELU) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
        if (y) y[i] = v;
        if (hi) clipped |= h16_store4(v, hscale, hi, lo, i);
        if (mask) mask[i] = relu_mask4(v);
    }
    if (clipped && sat) atomicAdd(sat, 1);
}

extern "C" int* pxl_h16_sat_counter(void);

extern "C" int pxl_bn_apply_h16(const float* x, const float* scale, const float* shift, const float* residual,
                                int relu, float* y, int64_t rows, int C, void* hi, void* lo, float hscale, void* relu_mask,
                                void* stream);

extern "C" int pxl_bn_apply(const float* x, const float* scale, const float* shift, const float* residual,
                            int relu, float* y, int64_t rows, int C, void* stream) {
    if (!y) return PXL_ERR_BAD_ARG;
    return pxl_bn_apply_h16(x, scale, shift, residual, relu, y, rows, C, nullptr, nullptr, 1.f, nullptr, stream);
}

// y nullable when the fp16 pair (hi, lo nullable) is the only output wanted; relu_mask (nullable, rows*C/4 bytes)
// receives the sign bits of the result for the backward (pxl_bn_bwd_*_h16)
extern "C" int pxl_bn_apply_h16(const float* x, const float* scale, const float* shift, const float* residual,
                                int relu, float* y, int64_t rows, int C, void* hi, void* lo, float hscale, void* relu_mask,
                                void* stream) {
    if (!x || !scale || !shift || (!y && !hi) || rows <= 0 || C <= 0 || (C & 3)) return PXL_ERR_BAD_ARG;
    const int64_t n4 = rows * (C / 4);
    int blocks = (int)(pxl_cdiv(n4, 256 * 2) < PXL_NUM_SMS * 8 ? pxl_cdiv(n4, 256 * 2) : PXL_NUM_SMS * 8);
    cudaStream_t st = (cudaStream_t)stream;
    const float4 *x4 = (const float4*)x, *s4 = (const float4*)scale, *h4 = (const float4*)shift, *r4 = (const float4*)residual;
    float4* y4 = (float4*)y;
    int* sat = hi ? pxl_h16_sat_counter() : nullptr;
    if (sat) sat += 2;
#define PXL_AP_ARGS x4, s4, h4, r4, y4, n4, C / 4, (uint2*)hi, (uint2*)lo, hscale, sat, (uint8_t*)relu_mask
    if (residual && relu) pxl_launch_pdl(bn_apply_kernel<true, true>, dim3(blocks), dim3(256), 0, st, PXL_AP_ARGS);
    else if (residual) pxl_launch_pdl(bn_apply_kernel<true, false>, dim3(blocks), dim3(256), 0, st, PXL_AP_ARGS);
    else if (relu) pxl_launch_pdl(bn_apply_kernel<false, true>, dim3(blocks), dim3(256), 0, st, PXL_AP_ARGS);
    else pxl_launch_pdl(bn_apply_kernel<false, false>, dim3(blocks), dim3(256), 0, st, PXL_AP_ARGS);
#undef PXL_AP_ARGS
    PXL_CHECK_LAUNCH();
    return 0;
}

// ------------------------------------------------------------------------------------------
// training forward in one launch: finalize (the arithmetic of bn_finalize_kernel, per thread for its 4 channels,
// from the fp64 sums) + apply.  The CTAs of row block 0 also store mean / inv_std / scale / shift for the backward
// and update the running statistics.  Same 2-D decomposition as bn_bwd_dx_kernel.
// ------------------------------------------------------------------------------------------
// BN_PRE: rows whose loads are issued before the per-channel prologue (0 or 2; registers: 4 CTAs of 256 threads per SM)
template <bool RES, bool RELU, int BN_PRE>
__global__ void __launch_bounds__(256, 4)
bn_finalize_apply_kernel(const float4* __restrict__ x, const double* __restrict__ sums, double count, double inv_count,
                         const float* __restrict__ gamma, const float* __restrict__ beta,
                         float* running_mean, float* running_var, float momentum, float eps, int clamp_mode,
                         float* mean, float* invstd, float* scale, float* shift,
                         const float4* __restrict__ res, float4* __restrict__ y,
                         int64_t rows, int C, int TX, int TY, int64_t rowsPerBlock,
                         uint2* __restrict__ hi, uint2* __restrict__ lo, float hscale, int* __restrict__ sat,
                         uint8_t* __restrict__ mask) {
    PXL_PDL_SYNC();
    const int tx = threadIdx.x % TX, ty = threadIdx.x / TX;
    const int c4 = blockIdx.y * TX + tx, c4max = C >> 2;
    if (c4 >= c4max) return;
    bool clipped = false;
    const int64_t r0 = (int64_t)blockIdx.x * rowsPerBlock;
    const int64_t r1 = min(rows, r0 + rowsPerBlock);
    // the first trip's loads go out BEFORE the per-channel prologue (fp64 finalize, 16 parameter loads): a 17 MB
    // layer-3 tensor is one wave of CTAs, and the prologue's latency chain in front of the first load was a
    // sizeable part of such a launch
    float4 px[BN_PRE > 0 ? BN_PRE : 1], pq[BN_PRE > 0 ? BN_PRE : 1];
#pragma unroll
    for (int u = 0; u < BN_PRE; ++u) {
        const int64_t r = r0 + ty + (int64_t)u * TY;
        px[u] = make_float4(0.f, 0.f, 0.f, 0.f); pq[u] = px[u];
        if (r < r1) {
            px[u] = __ldcs(x + r * c4max + c4);
            if (RES) pq[u] = __ldcs(res + r * c4max + c4);
        }
    }
    float sc[4], sh[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int c = 4 * c4 + k;
        // reciprocal multiply instead of bn_finalize_kernel's fp64 divisions: every thread of every CTA runs this
        // prologue before its first load, and two fp64 divisions per channel cost ~10 us per launch
        const double m = __ldg(sums + c) * inv_count;
        double var = fma(__ldg(sums + C + c), inv_count, -m * m);     // biased
        if (var < 0.0) var = 0.0;
        const float mf = (float)m;
        float is;
        if (clamp_mode) is = 1.0f / sqrtf(fmaxf((float)var, eps));
        else is = 1.0f / sqrtf((float)var + eps);
        sc[k] = __ldg(gamma + c) * is;
        sh[k] = __ldg(beta + c) - mf * sc[k];
        if (blockIdx.x == 0 && ty == 0) {
            if (running_mean) {
                const double unbiased = count > 1.0 ? var * count / (count - 1.0) : var;
                running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * mf;
                running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
            }
            mean[c] = mf; invstd[c] = is; scale[c] = sc[k]; shift[c] = sh[k];
        }
    }
    auto emit = [&](int64_t i, float4 v, const float4& q) {
        v.x = fmaf(v.x, sc[0], sh[0]); v.y = fmaf(v.y, sc[1], sh[1]);
        v.z = fmaf(v.z, sc[2], sh[2]); v.w = fmaf(v.w, sc[3], sh[3]);
        if (RES) v = f4add(v, q);
        if (RELU) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
        if (y) y[i] = v;
        if (hi) clipped |= h16_store4(v, hscale, hi, lo, i);
        if (mask) mask[i] = relu_mask4(v);
    };
#pragma unroll
    for (int u = 0; u < BN_PRE; ++u) {
        const int64_t r = r0 + ty + (int64_t)u * TY;
        if (r < r1) emit(r * c4max + c4, px[u], pq[u]);
    }
#pragma unroll 4
    for (int64_t r = r0 + ty + BN_PRE * (int64_t)TY; r < r1; r += TY) {
        const int64_t i = r * c4max + c4;
        const float4 v = __ldcs(x + i);
        float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
        if (RES) q = __ldcs(res + i);
        emit(i, v, q);
    }
    if (clipped && sat) atomicAdd(sat, 1);
}

// PXL_BN_PREFETCH (default 2; 0 = loads after the prologue): A/B switch of the first-trip prefetch
static int bn_prefetch_rows() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("PXL_BN_PREFETCH"); v = e ? atoi(e) : 2; }
    return v;
}

static RedLayout stream_layout(int64_t rows, int C) {
    RedLayout L;
    const int c4 = C / 4;
    // as many lanes along the channel axis as fit (<= 256): a CTA then streams whole contiguous NHWC rows
    // (a 32-lane split left every CTA reading 512-byte pieces with a row stride: ~12 % slower on HBM)
    L.TX = 1;
    while (L.TX * 2 <= c4 && L.TX < 256) L.TX *= 2;
    L.TY = 256 / L.TX;
    L.colBlocks = (int)pxl_cdiv(c4, L.TX);
    int64_t target = (int64_t)PXL_NUM_SMS * 8 / L.colBlocks;
    if (target < 1) target = 1;
    int64_t rpb = pxl_cdiv(rows, target);
    if (rpb < L.TY * 4) rpb = L.TY * 4;
    L.rowsPerBlock = rpb;
    L.rowBlocks = (int)pxl_cdiv(rows, rpb);
    return L;
}

extern "C" int pxl_bn_finalize_apply_h16(const float* x, const double* sums, double count, const float* gamma,
                                         const float* beta, float* running_mean, float* running_var, float momentum,
                                         float eps, int clamp_mode, float* mean, float* invstd, float* scale, float* shift,
                                         const float* residual, int relu, float* y, int64_t rows, int C,
                                         void* hi, void* lo, float hscale, void* relu_mask, void* stream);

extern "C" int pxl_bn_finalize_apply(const float* x, const double* sums, double count, const float* gamma,
                                     const float* beta, float* running_mean, float* running_var, float momentum,
                                     float eps, int clamp_mode, float* mean, float* invstd, float* scale, float* shift,
                                     const float* residual, int relu, float* y, int64_t rows, int C, void* stream) {
    if (!y) return PXL_ERR_BAD_ARG;
    return pxl_bn_finalize_apply_h16(x, sums, count, gamma, beta, running_mean, running_var, momentum, eps, clamp_mode, mean,
                                     invstd, scale, shift, residual, relu, y, rows, C, nullptr, nullptr, 1.f, nullptr, stream);
}

// the same launch also (or only: y nullable) writes the result as the fp16 pair the next convolution reads
extern "C" int pxl_bn_finalize_apply_h16(const float* x, const double* sums, double count, const float* gamma,
                                         const float* beta, float* running_mean, float* running_var, float momentum,
                                         float eps, int clamp_mode, float* mean, float* invstd, float* scale, float* shift,
                                         const float* residual, int relu, float* y, int64_t rows, int C,
                                         void* hi, void* lo, float hscale, void* relu_mask, void* stream) {
    if (!x || !sums || !gamma || !beta || !mean || !invstd || !scale || !shift || (!y && !hi) || rows <= 0 || C <= 0 || (C & 3) || count <= 0)
        return PXL_ERR_BAD_ARG;
    int* sat = hi ? pxl_h16_sat_counter() : nullptr;
    if (sat) sat += 2;
    const RedLayout L = stream_layout(rows, C);
    dim3 grid(L.rowBlocks, L.colBlocks);
    cudaStream_t st = (cudaStream_t)stream;
#define PXL_FA_ARGS (const float4*)x, sums, count, 1.0 / count, gamma, beta, running_mean, running_var, momentum, eps, clamp_mode, mean, invstd, \
                    scale, shift, (const float4*)residual, (float4*)y, rows, C, L.TX, L.TY, L.rowsPerBlock, \
                    (uint2*)hi, (uint2*)lo, hscale, sat, (uint8_t*)relu_mask
    if (residual && relu) { if (bn_prefetch_rows()) pxl_launch_pdl(bn_finalize_apply_kernel<true, true, 2>, dim3(grid), dim3(256), 0, st, PXL_FA_ARGS); else pxl_launch_pdl(bn_finalize_apply_kernel<true, true, 0>, dim3(grid), dim3(256), 0, st, PXL_FA_ARGS); }
    else if (residual) { if (bn_prefetch_rows()) pxl_launch_pdl(bn_finalize_apply_kernel<true, false, 2>, dim3(grid), dim3(256), 0, st, PXL_FA_ARGS); else pxl_launch_pdl(bn_finalize_apply_kernel<true, false, 0>, dim3(grid), dim3(256), 0, st, PXL_FA_ARGS); }
    else if (relu) { if (bn_prefetch_rows()) pxl_launch_pdl(bn_finalize_apply_kernel<false, true, 2>, dim3(grid), dim3(256), 0, st, PXL_FA_ARGS); else pxl_launch_pdl(bn_finalize_apply_kernel<false, true, 0>, dim3(grid), dim3(256), 0, st, PXL_FA_ARGS); }
    else { if (bn_prefetch_rows()) pxl_launch_pdl(bn_finalize_apply_kernel<false, false, 2>, dim3(grid), dim3(256), 0, st, PXL_FA_ARGS); else pxl_launch_pdl(bn_finalize_apply_kernel<false, false, 0>, dim3(grid), dim3(256), 0, st, PXL_FA_ARGS); }
#undef PXL_FA_ARGS
    PXL_CHECK_LAUNCH();
    return 0;
}

// ------------------------------------------------------------------------------------------
// backward.  dz = dy * (y > 0) when the ReLU was fused.
//   reduce: dsums[0:C] += sum dz ; dsums[C:2C] += sum dz * xhat
//   dx = gamma*invstd * (dz - dsums0/count - xhat*dsums1/count)
// ------------------------------------------------------------------------------------------
// RELU: 0 none, 1 mask from y, 2 mask recomputed from x (fmaf(x, scale, shift) > 0, no residual)
template <int RELU>
__global__ void __launch_bounds__(256)
bn_bwd_reduce_kernel(const float* __restrict__ x, const float* __restrict__ y, const float* __restrict__ dy,
                     const float* __restrict__ mean, const float* __restrict__ invstd, int64_t rows, int C,
                     int TX, int TY, int64_t rowsPerBlock, double* __restrict__ dsums,
                     const float* __restrict__ scale, const float* __restrict__ shift, float* __restrict__ amax_slot,
                     const uint8_t* __restrict__ mask) {
    PXL_PDL_SYNC();
    const int tx = threadIdx.x % TX, ty = threadIdx.x / TX;
    const int c4 = blockIdx.y * TX + tx, c4max = C >> 2;
    const int64_t r0 = (int64_t)blockIdx.x * rowsPerBlock;
    const int64_t r1 = min(rows, r0 + rowsPerBlock);
    float4 s = make_float4(0, 0, 0, 0), q = make_float4(0, 0, 0, 0);
    float amax = 0.f;
    if (c4 < c4max) {
        const float4 m = __ldg(reinterpret_cast<const float4*>(mean) + c4);
        const float4 is = __ldg(reinterpret_cast<const float4*>(invstd) + c4);
        const float4* xp = reinterpret_cast<const float4*>(x) + c4;
        const float4* yp = reinterpret_cast<const float4*>(y) + c4;
        const float4* dp = reinterpret_cast<const float4*>(dy) + c4;
        float4 sc = make_float4(0, 0, 0, 0), sh = sc;
        if (RELU == 2) { sc = __ldg(reinterpret_cast<const float4*>(scale) + c4); sh = __ldg(reinterpret_cast<const float4*>(shift) + c4); }
        // 4 rows per trip: 12 independent 16-byte loads in flight per thread (these launches are short, the
        // loop is latency-bound otherwise)
#pragma unroll 4
        for (int64_t r = r0 + ty; r < r1; r += TY) {
            float4 d = __ldg(dp + r * c4max);
            float4 v = __ldg(xp + r * c4max);
            if (RELU == 1) {
                float4 o = __ldg(yp + r * c4max);
                d.x = o.x > 0.f ? d.x : 0.f; d.y = o.y > 0.f ? d.y : 0.f;
                d.z = o.z > 0.f ? d.z : 0.f; d.w = o.w > 0.f ? d.w : 0.f;
            } else if (RELU == 2) {
                d.x = fmaf(v.x, sc.x, sh.x) > 0.f ? d.x : 0.f; d.y = fmaf(v.y, sc.y, sh.y) > 0.f ? d.y : 0.f;
                d.z = fmaf(v.z, sc.z, sh.z) > 0.f ? d.z : 0.f; d.w = fmaf(v.w, sc.w, sh.w) > 0.f ? d.w : 0.f;
            } else if (RELU == 3) {
                apply_mask4(d, __ldg(mask + r * c4max + c4));
            }
            float4 xh = make_float4((v.x - m.x) * is.x, (v.y - m.y) * is.y, (v.z - m.z) * is.z, (v.w - m.w) * is.w);
            s = f4add(s, d);
            q = f4add(q, f4mul(d, xh));
            amax = fmaxf(amax, fmaxf(fmaxf(fabsf(d.x), fabsf(d.y)), fmaxf(fabsf(d.z), fabsf(d.w))));
        }
    }
    if (amax_slot) {
        // absmax of dz for the fp16-pair scale of dx (bn_bwd_dx_kernel): one atomicMax per warp that saw a larger value
        amax = warp_max(amax);
        if ((threadIdx.x & 31) == 0 && amax > 0.f && __float_as_uint(amax) > ((volatile unsigned*)amax_slot)[2])
            atomicMax((unsigned*)amax_slot + 2, __float_as_uint(amax));
    }
    block_reduce_cols(s, q, TX, TY, c4, c4max, dsums, dsums + C);
}

extern "C" int pxl_bn_bwd_reduce_h16(const float* x, const float* y, const float* dy, const float* mean,
                                     const float* invstd, int relu, int64_t rows, int C, double* dsums,
                                     const float* scale, const float* shift, float* amax_slot, const void* relu_mask,
                                     void* stream);

extern "C" int pxl_bn_bwd_reduce(const float* x, const float* y, const float* dy, const float* mean,
                                 const float* invstd, int relu, int64_t rows, int C, double* dsums,
                                 const float* scale, const float* shift, void* stream) {
    return pxl_bn_bwd_reduce_h16(x, y, dy, mean, invstd, relu, rows, C, dsums, scale, shift, nullptr, nullptr, stream);
}

// amax_slot (nullable DEVICE float[4], zeroed): slot[2] = max(slot[2], absmax(dz)) as a bit pattern
// ReLU mask source, in this order: relu_mask (bytes written by pxl_bn_*apply_h16), y (the forward result), else
// recomputed from x*scale+shift (no residual)
extern "C" int pxl_bn_bwd_reduce_h16(const float* x, const float* y, const float* dy, const float* mean,
                                     const float* invstd, int relu, int64_t rows, int C, double* dsums,
                                     const float* scale, const float* shift, float* amax_slot, const void* relu_mask,
                                     void* stream) {
    if (!x || !dy || !mean || !invstd || !dsums || rows <= 0 || C <= 0 || (C & 3) || (relu && !y && !relu_mask && !(scale && shift))) return PXL_ERR_BAD_ARG;
    RedLayout L = red_layout(rows, C);
    dim3 grid(L.rowBlocks, L.colBlocks);
    cudaStream_t st = (cudaStream_t)stream;
    const uint8_t* mk = (const uint8_t*)relu_mask;
    if (relu && mk) pxl_launch_pdl(bn_bwd_reduce_kernel<3>, dim3(grid), dim3(256), 0, st, x, y, dy, mean, invstd, rows, C, L.TX, L.TY, L.rowsPerBlock, dsums, scale, shift, amax_slot, mk);
    else if (relu && y) pxl_launch_pdl(bn_bwd_reduce_kernel<1>, dim3(grid), dim3(256), 0, st, x, y, dy, mean, invstd, rows, C, L.TX, L.TY, L.rowsPerBlock, dsums, scale, shift, amax_slot, mk);
    else if (relu) pxl_launch_pdl(bn_bwd_reduce_kernel<2>, dim3(grid), dim3(256), 0, st, x, y, dy, mean, invstd, rows, C, L.TX, L.TY, L.rowsPerBlock, dsums, scale, shift, amax_slot, mk);
    else pxl_launch_pdl(bn_bwd_reduce_kernel<0>, dim3(grid), dim3(256), 0, st, x, y, dy, mean, invstd, rows, C, L.TX, L.TY, L.rowsPerBlock, dsums, scale, shift, amax_slot, mk);
    PXL_CHECK_LAUNCH();
    return 0;
}

// dx = A*dz + B*x + K per channel with A = gamma*invstd, B = -A*invstd*mean(dz*xhat), K = -A*mean(dz) - B*mean:
// a thread owns 4 fixed channels (coefficients in registers, computed once from the fp64 sums) and walks down
// the rows, 4 rows per trip.
template <int RELU, bool DRES, int BN_PRE>
__global__ void __launch_bounds__(256, 4)
bn_bwd_dx_kernel(const float4* __restrict__ x, const float4* __restrict__ y, const float4* __restrict__ dy,
                 const float* __restrict__ mean, const float* __restrict__ invstd, const float* __restrict__ gamma,
                 const double* __restrict__ dsums, double inv_count, float4* __restrict__ dx, float4* __restrict__ dres,
                 int64_t rows, int C, int TX, int TY, int64_t rowsPerBlock,
                 const float* __restrict__ scale, const float* __restrict__ shift,
                 float* dgamma_acc, float* dbeta_acc,
                 uint2* __restrict__ dhi, uint2* __restrict__ dlo, float* __restrict__ slot, int target_log2,
                 int* __restrict__ sat, const uint8_t* __restrict__ mask) {
    PXL_PDL_SYNC();
    const int tx = threadIdx.x % TX, ty = threadIdx.x / TX;
    const int c4 = blockIdx.y * TX + tx, c4max = C >> 2;
    const int64_t r0 = (int64_t)blockIdx.x * rowsPerBlock;
    const int64_t r1 = min(rows, r0 + rowsPerBlock);
    // first trip's loads before the prologue (scale reduction with a barrier, fp64 coefficient math), see
    // bn_finalize_apply_kernel
    float4 pd[BN_PRE > 0 ? BN_PRE : 1], pv[BN_PRE > 0 ? BN_PRE : 1], po[BN_PRE > 0 ? BN_PRE : 1];
    unsigned pm[BN_PRE > 0 ? BN_PRE : 1];
#pragma unroll
    for (int u = 0; u < BN_PRE; ++u) {
        const int64_t r = r0 + ty + (int64_t)u * TY;
        pd[u] = make_float4(0.f, 0.f, 0.f, 0.f); pv[u] = pd[u]; po[u] = pd[u]; pm[u] = 0u;
        if (c4 < c4max && r < r1) {
            const int64_t i = r * c4max + c4;
            pd[u] = __ldcs(dy + i);
            pv[u] = __ldcs(x + i);
            if (RELU == 1) po[u] = __ldcs(y + i);
            if (RELU == 3) pm[u] = __ldg(mask + i);
        }
    }
    float hs = 1.f;
    if (dhi) {
        // fp16-pair scale of dx: |dx| <= max_c |gamma*invstd| * (absmax(dz) + |mean dz| + |xhat| |mean dz*xhat|); the
        // first factor times absmax(dz) is mapped to <= 2^target_log2, the mean terms live in the headroom above it
        // (values that still leave the fp16 range saturate and are counted).  Every CTA derives the same number.
        __shared__ float smax[8];
        float a = 0.f;
        for (int c = threadIdx.x; c < C; c += blockDim.x) a = fmaxf(a, fabsf(__ldg(gamma + c) * __ldg(invstd + c)));
        a = warp_max(a);
        if ((threadIdx.x & 31) == 0) smax[threadIdx.x >> 5] = a;
        __syncthreads();
        a = smax[0];
#pragma unroll
        for (int w = 1; w < 8; ++w) a = fmaxf(a, smax[w]);
        hs = pxl_pow2_scale(a * __uint_as_float(((const unsigned*)slot)[2]), target_log2);
        if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) { slot[0] = hs; slot[1] = 1.f / hs; }
    }
    if (c4 >= c4max) return;
    bool clipped = false;
    if (dgamma_acc && blockIdx.x == 0 && ty == 0) {
        // parameter gradients (what bn_bwd_params_kernel does), accumulated straight into gamma.grad / beta.grad
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int c = 4 * c4 + k;
            dbeta_acc[c] += (float)__ldg(dsums + c);
            dgamma_acc[c] += (float)__ldg(dsums + C + c);
        }
    }
    float A[4], B[4], K[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int c = 4 * c4 + k;
        const float m = __ldg(mean + c), is = __ldg(invstd + c), g = __ldg(gamma + c);
        const float mdz = (float)(__ldg(dsums + c) * inv_count);
        const float mdzx = (float)(__ldg(dsums + C + c) * inv_count);
        A[k] = g * is;
        B[k] = -A[k] * is * mdzx;
        K[k] = -A[k] * mdz - B[k] * m;
    }
    float4 sc = make_float4(0, 0, 0, 0), sh = sc;
    if (RELU == 2) { sc = __ldg(reinterpret_cast<const float4*>(scale) + c4); sh = __ldg(reinterpret_cast<const float4*>(shift) + c4); }
    auto emit = [&](int64_t i, float4 d, const float4& v, const float4& o, unsigned m) {
        if (RELU == 1) {
            d.x = o.x > 0.f ? d.x : 0.f; d.y = o.y > 0.f ? d.y : 0.f;
            d.z = o.z > 0.f ? d.z : 0.f; d.w = o.w > 0.f ? d.w : 0.f;
        } else if (RELU == 2) {
            d.x = fmaf(v.x, sc.x, sh.x) > 0.f ? d.x : 0.f; d.y = fmaf(v.y, sc.y, sh.y) > 0.f ? d.y : 0.f;
            d.z = fmaf(v.z, sc.z, sh.z) > 0.f ? d.z : 0.f; d.w = fmaf(v.w, sc.w, sh.w) > 0.f ? d.w : 0.f;
        } else if (RELU == 3) {
            apply_mask4(d, m);
        }
        if (DRES) dres[i] = d;
        float4 o4;
        o4.x = fmaf(A[0], d.x, fmaf(B[0], v.x, K[0]));
        o4.y = fmaf(A[1], d.y, fmaf(B[1], v.y, K[1]));
        o4.z = fmaf(A[2], d.z, fmaf(B[2], v.z, K[2]));
        o4.w = fmaf(A[3], d.w, fmaf(B[3], v.w, K[3]));
        if (dx) dx[i] = o4;
        if (dhi) clipped |= h16_store4(o4, hs, dhi, dlo, i);
    };
#pragma unroll
    for (int u = 0; u < BN_PRE; ++u) {
        const int64_t r = r0 + ty + (int64_t)u * TY;
        if (r < r1) emit(r * c4max + c4, pd[u], pv[u], po[u], pm[u]);
    }
#pragma unroll 4
    for (int64_t r = r0 + ty + BN_PRE * (int64_t)TY; r < r1; r += TY) {
        const int64_t i = r * c4max + c4;
        const float4 d = __ldcs(dy + i);
        const float4 v = __ldcs(x + i);
        float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
        unsigned m = 0u;
        if (RELU == 1) o = __ldcs(y + i);
        if (RELU == 3) m = __ldg(mask + i);
        emit(i, d, v, o, m);
    }
    if (clipped && sat) atomicAdd(sat, 1);
}

extern "C" int pxl_bn_bwd_dx_h16(const float* x, const float* y, const float* dy, const float* mean,
                                 const float* invstd, const float* gamma, const double* dsums, double count,
                                 int relu, float* dx, float* dres, int64_t rows, int C,
                                 const float* scale, const float* shift, float* dgamma_acc, float* dbeta_acc,
                                 void* dhi, void* dlo, float* slot, int target_log2, const void* relu_mask, void* stream);

extern "C" int pxl_bn_bwd_dx(const float* x, const float* y, const float* dy, const float* mean,
                             const float* invstd, const float* gamma, const double* dsums, double count,
                             int relu, float* dx, float* dres, int64_t rows, int C,
                             const float* scale, const float* shift, float* dgamma_acc, float* dbeta_acc, void* stream) {
    if (!dx) return PXL_ERR_BAD_ARG;
    return pxl_bn_bwd_dx_h16(x, y, dy, mean, invstd, gamma, dsums, count, relu, dx, dres, rows, C, scale, shift,
                             dgamma_acc, dbeta_acc, nullptr, nullptr, nullptr, 0, nullptr, stream);
}

// dx also (or only: dx nullable) as the fp16 pair (dhi, dlo nullable) the dgrad / wgrad convolutions read; slot = the
// DEVICE float[4] pxl_bn_bwd_reduce_h16 left absmax(dz) in: this launch stores the pair's scale s / 1/s in slot[0..1]
extern "C" int pxl_bn_bwd_dx_h16(const float* x, const float* y, const float* dy, const float* mean,
                                 const float* invstd, const float* gamma, const double* dsums, double count,
                                 int relu, float* dx, float* dres, int64_t rows, int C,
                                 const float* scale, const float* shift, float* dgamma_acc, float* dbeta_acc,
                                 void* dhi, void* dlo, float* slot, int target_log2, const void* relu_mask, void* stream) {
    if ((!dx && !dhi) || (dhi && !slot)) return PXL_ERR_BAD_ARG;
    int* sat = dhi ? pxl_h16_sat_counter() : nullptr;
    if (sat) sat += 3;
    if (!x || !dy || !mean || !invstd || !gamma || !dsums || rows <= 0 || C <= 0 || (C & 3) || (relu && !y && !relu_mask && !(scale && shift))) return PXL_ERR_BAD_ARG;
    const RedLayout L = stream_layout(rows, C);     // the reductions' decomposition without their atomics
    dim3 grid(L.rowBlocks, L.colBlocks);
    cudaStream_t st = (cudaStream_t)stream;
    const float4 *x4 = (const float4*)x, *y4 = (const float4*)y, *d4 = (const float4*)dy;
    float4 *o4 = (float4*)dx, *r4 = (float4*)dres;
    const double ic = 1.0 / count;
#define PXL_DX_ARGS x4, y4, d4, mean, invstd, gamma, dsums, ic, o4, r4, rows, C, L.TX, L.TY, L.rowsPerBlock, scale, shift, \
                    (dgamma_acc && dbeta_acc) ? dgamma_acc : nullptr, dbeta_acc, (uint2*)dhi, (uint2*)dlo, slot, target_log2, sat, (const uint8_t*)relu_mask
    const int mode = relu ? (relu_mask ? 3 : (y ? 1 : 2)) : 0;
    if (mode == 3 && dres) { if (bn_prefetch_rows()) pxl_launch_pdl(bn_bwd_dx_kernel<3, true, 2>, dim3(grid), dim3(256), 0, st, PXL_DX_ARGS); else pxl_launch_pdl(bn_bwd_dx_kernel<3, true, 0>, dim3(grid), dim3(256), 0, st, PXL_DX_ARGS); }
    else if (mode == 3) { if (bn_prefetch_rows()) pxl_launch_pdl(bn_bwd_dx_kernel<3, false, 2>, dim3(grid), dim3(256), 0, st, PXL_DX_ARGS); else pxl_launch_pdl(bn_bwd_dx_kernel<3, false, 0>, dim3(grid), dim3(256), 0, st, PXL_DX_ARGS); }
    else if (mode == 1 && dres) { if (bn_prefetch_rows()) pxl_launch_pdl(bn_bwd_dx_kernel<1, true, 2>, dim3(grid), dim3(256), 0, st, PXL_DX_ARGS); else pxl_launch_pdl(bn_bwd_dx_kernel<1, true, 0>, dim3(grid), dim3(256), 0, st, PXL_DX_ARGS); }
    else if (mode == 1) { if (bn_prefetch_rows()) pxl_launch_pdl(bn_bwd_dx_kernel<1, false, 2>, dim3(grid), dim3(256), 0, st, PXL_DX_ARGS); else pxl_launch_pdl(bn_bwd_dx_kernel<1, false, 0>, dim3(grid), dim3(256), 0, st, PXL_DX_ARGS); }
    else if (mode == 2 && dres) { if (bn_prefetch_rows()) pxl_launch_pdl(bn_bwd_dx_kernel<2, true, 2>, dim3(grid), dim3(256), 0, st, PXL_DX_ARGS); else pxl_launch_pdl(bn_bwd_dx_kernel<2, true, 0>, dim3(grid), dim3(256), 0, st, PXL_DX_ARGS); }
    else if (mode == 2) { if (bn_prefetch_rows()) pxl_launch_pdl(bn_bwd_dx_kernel<2, false, 2>, dim3(grid), dim3(256), 0, st, PXL_DX_ARGS); else pxl_launch_pdl(bn_bwd_dx_kernel<2, false, 0>, dim3(grid), dim3(256), 0, st, PXL_DX_ARGS); }
    else if (dres) { if (bn_prefetch_rows()) pxl_launch_pdl(bn_bwd_dx_kernel<0, true, 2>, dim3(grid), dim3(256), 0, st, PXL_DX_ARGS); else pxl_launch_pdl(bn_bwd_dx_kernel<0, true, 0>, dim3(grid), dim3(256), 0, st, PXL_DX_ARGS); }
    else { if (bn_prefetch_rows()) pxl_launch_pdl(bn_bwd_dx_kernel<0, false, 2>, dim3(grid), dim3(256), 0, st, PXL_DX_ARGS); else pxl_launch_pdl(bn_bwd_dx_kernel<0, false, 0>, dim3(grid), dim3(256), 0, st, PXL_DX_ARGS); }
#undef PXL_DX_ARGS
    PXL_CHECK_LAUNCH();
    return 0;
}

__global__ void bn_bwd_params_kernel(const double* __restrict__ dsums, int C, float* dgamma, float* dbeta, int accumulate) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const float db = (float)dsums[c], dg = (float)dsums[C + c];
    if (accumulate) { dgamma[c] += dg; dbeta[c] += db; }
    else { dgamma[c] = dg; dbeta[c] = db; }
}

extern "C" int pxl_bn_bwd_params(const double* dsums, int C, float* dgamma, float* dbeta, int accumulate, void* stream) {
    if (!dsums || !dgamma || !dbeta || C <= 0) return PXL_ERR_BAD_ARG;
    bn_bwd_params_kernel<<<(C + 127) / 128, 128, 0, (cudaStream_t)stream>>>(dsums, C, dgamma, dbeta, accumulate);
    PXL_CHECK_LAUNCH();
    return 0;
}

// ------------------------------------------------------------------------------------------
// MaxPool2d(kernel 3, stride 2, padding 1), NHWC (resnet.py:72).  Backward routes each output
// gradient to the FIRST maximum in row-major window order (strict '>' scan, like ATen).
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
maxpool_fwd_kernel(const float4* __restrict__ x, float4* __restrict__ y, int N, int H, int W, int c4max, int OH, int OW) {
    const int64_t total = (int64_t)N * OH * OW * c4max;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int c = (int)(i % c4max);
        int64_t p = i / c4max;
        const int ox = (int)(p % OW); p /= OW;
        const int oy = (int)(p % OH);
        const int n = (int)(p / OH);
        float4 m = make_float4(-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F);
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const int iy = oy * 2 - 1 + r;
            if (iy < 0 || iy >= H) continue;
#pragma unroll
            for (int s = 0; s < 3; ++s) {
                const int ix = ox * 2 - 1 + s;
                if (ix < 0 || ix >= W) continue;
                const float4 v = __ldg(x + ((int64_t)(n * H + iy) * W + ix) * c4max + c);
                m.x = fmaxf(m.x, v.x); m.y = fmaxf(m.y, v.y); m.z = fmaxf(m.z, v.z); m.w = fmaxf(m.w, v.w);
            }
        }
        y[i] = m;
    }
}

extern "C" int pxl_maxpool3x3s2_fwd(const float* x, float* y, int N, int H, int W, int C, int OH, int OW, void* stream) {
    if (!x || !y || N <= 0 || (C & 3) || OH != (H + 2 - 3) / 2 + 1 || OW != (W + 2 - 3) / 2 + 1) return PXL_ERR_BAD_ARG;
    const int64_t total = (int64_t)N * OH * OW * (C / 4);
    int blocks = (int)(pxl_cdiv(total, 256) < PXL_NUM_SMS * 16 ? pxl_cdiv(total, 256) : PXL_NUM_SMS * 16);
    maxpool_fwd_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>((const float4*)x, (float4*)y, N, H, W, C / 4, OH, OW);
    PXL_CHECK_LAUNCH();
    return 0;
}

// One launch per parity class (oy % 2, ox % 2) of the output windows: 3x3 windows at stride 2 whose rows (columns)
// have the same parity do not overlap, so within a launch every dx element receives at most one gradient and the four
// launches add them in a fixed order (atomics in arrival order would make the sums differ from run to run).
__global__ void __launch_bounds__(256)
maxpool_bwd_kernel(const float* __restrict__ x, const float* __restrict__ dy, float* __restrict__ dx,
                   int N, int H, int W, int C, int OH, int OW, int py, int px) {
    const int PH = (OH - py + 1) / 2, PW = (OW - px + 1) / 2;
    const int64_t total = (int64_t)N * PH * PW * C;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < total; j += stride) {
        const int c = (int)(j % C);
        int64_t p = j / C;
        const int ox = 2 * (int)(p % PW) + px; p /= PW;
        const int oy = 2 * (int)(p % PH) + py;
        const int n = (int)(p / PH);
        const int64_t i = ((int64_t)(n * OH + oy) * OW + ox) * C + c;
        float m = -CUDART_INF_F;
        int64_t arg = -1;
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const int iy = oy * 2 - 1 + r;
            if (iy < 0 || iy >= H) continue;
#pragma unroll
            for (int s = 0; s < 3; ++s) {
                const int ix = ox * 2 - 1 + s;
                if (ix < 0 || ix >= W) continue;
                const int64_t idx = ((int64_t)(n * H + iy) * W + ix) * C + c;
                const float v = __ldg(x + idx);
                if (arg < 0 || v > m || isnan(v)) { m = v; arg = idx; }
            }
        }
        if (arg >= 0) dx[arg] += __ldg(dy + i);
    }
}

extern "C" int pxl_maxpool3x3s2_bwd(const float* x, const float* y, const float* dy, float* dx,
                                    int N, int H, int W, int C, int OH, int OW, void* stream) {
    (void)y;
    if (!x || !dy || !dx || N <= 0) return PXL_ERR_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(dx, 0, sizeof(float) * (size_t)N * H * W * C, st);
    if (e != cudaSuccess) return (int)e;
    for (int cls = 0; cls < 4; ++cls) {
        const int py = cls >> 1, px = cls & 1;
        const int64_t total = (int64_t)N * ((OH - py + 1) / 2) * ((OW - px + 1) / 2) * C;
        if (total <= 0) continue;
        int blocks = (int)(pxl_cdiv(total, 256) < PXL_NUM_SMS * 16 ? pxl_cdiv(total, 256) : PXL_NUM_SMS * 16);
        maxpool_bwd_kernel<<<blocks, 256, 0, st>>>(x, dy, dx, N, H, W, C, OH, OW, py, px);
        PXL_CHECK_LAUNCH();
    }
    return 0;
}

// ------------------------------------------------------------------------------------------
// fused SGD(momentum, weight decay) + teacher EMA over a flat parameter arena
//   (nn/optimizer.py:57-75 ; ssl_mt.py:359-363).  28 B/param: r p, r g, r buf, r t ; w p, w buf, w t
// ------------------------------------------------------------------------------------------
template <bool EMA, bool FIRST>
__global__ void __launch_bounds__(256)
sgd_ema_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ buf, float* __restrict__ t,
               int64_t n, float lr, float mom, float wd, float d) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const float omd = 1.f - d;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const float pv = p[i];
        // torch: d_p = g.add(p, alpha=wd); buf = d_p (first) | buf.mul_(mom).add_(d_p); p.add_(buf, alpha=-lr)
        float dp = fmaf(wd, pv, g[i]);
        float b;
        if (FIRST) b = dp;
        else b = __fadd_rn(__fmul_rn(buf[i], mom), dp);
        buf[i] = b;
        const float np = fmaf(-lr, b, pv);
        p[i] = np;
        if (EMA) t[i] = fmaf(omd, np, __fmul_rn(t[i], d));   // t.mul_(d).add_(s, alpha=1-d)
    }
}

extern "C" int pxl_sgd_ema(float* p, const float* g, float* buf, float* teacher, int64_t n, float lr,
                           float momentum, float weight_decay, float ema_d, int first_step, void* stream) {
    if (!p || !g || !buf || n <= 0) return PXL_ERR_BAD_ARG;
    int blocks = (int)(pxl_cdiv(n, 256 * 4) < PXL_NUM_SMS * 8 ? pxl_cdiv(n, 256 * 4) : PXL_NUM_SMS * 8);
    cudaStream_t st = (cudaStream_t)stream;
    if (teacher && first_step) sgd_ema_kernel<true, true><<<blocks, 256, 0, st>>>(p, g, buf, teacher, n, lr, momentum, weight_decay, ema_d);
    else if (teacher) sgd_ema_kernel<true, false><<<blocks, 256, 0, st>>>(p, g, buf, teacher, n, lr, momentum, weight_decay, ema_d);
    else if (first_step) sgd_ema_kernel<false, true><<<blocks, 256, 0, st>>>(p, g, buf, teacher, n, lr, momentum, weight_decay, ema_d);
    else sgd_ema_kernel<false, false><<<blocks, 256, 0, st>>>(p, g, buf, teacher, n, lr, momentum, weight_decay, ema_d);
    PXL_CHECK_LAUNCH();
    return 0;
}

__global__ void __launch_bounds__(256)
ema_kernel(float* __restrict__ t, const float* __restrict__ s, int64_t n, float d) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const float omd = 1.f - d;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        t[i] = fmaf(omd, s[i], __fmul_rn(t[i], d));
}

extern "C" int pxl_ema(float* teacher, const float* student, int64_t n, float ema_d, void* stream) {
    if (!teacher || !student || n <= 0) return PXL_ERR_BAD_ARG;
    int blocks = (int)(pxl_cdiv(n, 256 * 4) < PXL_NUM_SMS * 8 ? pxl_cdiv(n, 256 * 4) : PXL_NUM_SMS * 8);
    ema_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(teacher, student, n, ema_d);
    PXL_CHECK_LAUNCH();
    return 0;
}
