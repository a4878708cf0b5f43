// Pixel-wise loss kernels on planar [n, C, H*W] maps: MSE consistency (the metric kernel),
// cross-entropy with ignore_index, channel softmax, fused softmax+MSE, CutMix mix/confidence.
#include "common.cuh"
#include <stdlib.h>
#include <math_constants.h>

// ------------------------------------------------------------------------------------------
// launch accounting
// ------------------------------------------------------------------------------------------
static int64_t g_launches = 0;
extern "C" void pxl_count_launch_(int n) { g_launches += n; }
// programmatic dependent launch switch (common.cuh): environment PXL_PDL, read once; default on
extern "C" int pxl_pdl_enabled_(void) {
    static int v = -1;
    if (v < 0) { const char* e = getenv("PXL_PDL"); v = e ? (atoi(e) != 0) : 1; }
    return v;
}
// 2: relu_mask argument of the pxl_bn_*_h16 entry points; 3: caller-provided workspace of the wgrad launches
extern "C" int pxl_abi_version(void) { return 3; }
extern "C" int64_t pxl_launch_count(void) { return g_launches; }
extern "C" void pxl_reset_launch_count(void) { g_launches = 0; }

// ------------------------------------------------------------------------------------------
// MSE consistency  (ssl_mt.py:115,179-187)
//   algorithmic traffic: read s, read t (8 B/elem) [+ write grad (4 B/elem)]
//   design: persistent grid = 148 SMs x 4 CTAs x 256 threads, 128-bit streaming loads, 4-deep
//   unroll (8 independent LDG.128 in flight per thread), warp-shuffle + smem block reduction,
//   fp64 per-block partials, last-block-done deterministic final sum.
// ------------------------------------------------------------------------------------------
#define MSE_THREADS 256
#define MSE_MAX_BLOCKS (PXL_NUM_SMS * 4)
#define MSE_UNROLL 4

struct MseWorkspace {
    double partial[MSE_MAX_BLOCKS];
    unsigned int ticket;
    unsigned int pad[3];
    double scalar_acc;      // accumulator of the softmax+MSE kernel, kept zero between launches
};

extern "C" int64_t pxl_mse_workspace_bytes(void) { return (int64_t)sizeof(MseWorkspace); }

__device__ __forceinline__ float sq_acc4(float4 a, float4 b, float gs, float4& g) {
    float dx = a.x - b.x, dy = a.y - b.y, dz = a.z - b.z, dw = a.w - b.w;
    g = make_float4(gs * dx, gs * dy, gs * dz, gs * dw);
    return dx * dx + dy * dy + dz * dz + dw * dw;
}

__device__ __forceinline__ void block_finish(float acc, MseWorkspace* ws, double final_scale,
                                             float* loss_out) {
    __shared__ float warp_part[MSE_THREADS / 32];
    __shared__ bool is_last;
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) warp_part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double b = 0.0;
#pragma unroll
        for (int i = 0; i < MSE_THREADS / 32; ++i) b += (double)warp_part[i];
        ws->partial[blockIdx.x] = b;
        __threadfence();
        unsigned int t = atomicAdd(&ws->ticket, 1u);
        is_last = (t == gridDim.x - 1);
    }
    __syncthreads();
    if (is_last) {
        __threadfence();
        double s = 0.0;
        for (int i = threadIdx.x; i < (int)gridDim.x; i += MSE_THREADS) s += ((volatile double*)ws->partial)[i];
        s = warp_sum_d(s);
        __shared__ double wp[MSE_THREADS / 32];
        if ((threadIdx.x & 31) == 0) wp[threadIdx.x >> 5] = s;
        __syncthreads();
        if (threadIdx.x == 0) {
            double tot = 0.0;
#pragma unroll
            for (int i = 0; i < MSE_THREADS / 32; ++i) tot += wp[i];
            loss_out[0] = (float)(tot * final_scale);
            ws->ticket = 0;  // restore for the next launch
        }
    }
}

template <bool WRITE_GRAD>
__global__ void __launch_bounds__(MSE_THREADS, 4)
mse_vec_kernel(const float* __restrict__ s, const float* __restrict__ t, int64_t n, int64_t head,
               float gscale, double final_scale, float* __restrict__ grad, float* loss_out,
               MseWorkspace* ws) {
    // elements [0, head) and the tail after the last full float4 are handled scalar by block 0
    const int64_t nvec = (n - head) >> 2;
    const float* sv = s + head;
    const float* tv = t + head;
    float* gv = WRITE_GRAD ? grad + head : nullptr;
    float acc = 0.f;
    const int64_t stride = (int64_t)gridDim.x * MSE_THREADS;
    int64_t i = (int64_t)blockIdx.x * MSE_THREADS + threadIdx.x;
    for (; i + (MSE_UNROLL - 1) * stride < nvec; i += MSE_UNROLL * stride) {
        float4 a[MSE_UNROLL], b[MSE_UNROLL];
#pragma unroll
        for (int u = 0; u < MSE_UNROLL; ++u) {
            a[u] = ld_stream4(sv + 4 * (i + u * stride));
            b[u] = ld_stream4(tv + 4 * (i + u * stride));
        }
#pragma unroll
        for (int u = 0; u < MSE_UNROLL; ++u) {
            float4 g;
            acc += sq_acc4(a[u], b[u], gscale, g);
            if (WRITE_GRAD) st_stream4(gv + 4 * (i + u * stride), g);
        }
    }
    for (; i < nvec; i += stride) {
        float4 a = ld_stream4(sv + 4 * i), b = ld_stream4(tv + 4 * i), g;
        acc += sq_acc4(a, b, gscale, g);
        if (WRITE_GRAD) st_stream4(gv + 4 * i, g);
    }
    if (blockIdx.x == 0) {
        const int64_t tail0 = head + (nvec << 2);
        for (int64_t j = threadIdx.x; j < head + (n - tail0); j += MSE_THREADS) {
            int64_t idx = j < head ? j : tail0 + (j - head);
            float d = s[idx] - t[idx];
            acc += d * d;
            if (WRITE_GRAD) grad[idx] = gscale * d;
        }
    }
    block_finish(acc, ws, final_scale, loss_out);
}

template <bool WRITE_GRAD>
__global__ void __launch_bounds__(MSE_THREADS, 4)
mse_scalar_kernel(const float* __restrict__ s, const float* __restrict__ t, int64_t n, float gscale,
                  double final_scale, float* __restrict__ grad, float* loss_out, MseWorkspace* ws) {
    float acc = 0.f;
    const int64_t stride = (int64_t)gridDim.x * MSE_THREADS;
    for (int64_t i = (int64_t)blockIdx.x * MSE_THREADS + threadIdx.x; i < n; i += stride) {
        float d = s[i] - t[i];
        acc += d * d;
        if (WRITE_GRAD) grad[i] = gscale * d;
    }
    block_finish(acc, ws, final_scale, loss_out);
}

extern "C" int pxl_mse_consistency(const float* s, const float* t, int64_t n, float loss_scale,
                                   float* loss_out, float* grad_s, void* workspace, void* stream) {
    if (!s || !t || !loss_out || !workspace || n <= 0) return PXL_ERR_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    MseWorkspace* ws = (MseWorkspace*)workspace;
    const double final_scale = (double)loss_scale / (double)n;
    const float gscale = (float)(2.0 * (double)loss_scale / (double)n);
    // vector path needs s, t (and grad) congruent mod 16 bytes
    uintptr_t as = (uintptr_t)s & 15, at = (uintptr_t)t & 15, ag = grad_s ? ((uintptr_t)grad_s & 15) : as;
    bool vec = (as == at) && (as == ag) && ((as & 3) == 0) && n >= 1024;
    int64_t work = vec ? (n >> 2) : n;
    int blocks = (int)(pxl_cdiv(work, MSE_THREADS * MSE_UNROLL) < MSE_MAX_BLOCKS
                           ? pxl_cdiv(work, MSE_THREADS * MSE_UNROLL) : MSE_MAX_BLOCKS);
    if (blocks < 1) blocks = 1;
    if (vec) {
        int64_t head = as ? (16 - (int64_t)as) / 4 : 0;
        if (grad_s) mse_vec_kernel<true><<<blocks, MSE_THREADS, 0, st>>>(s, t, n, head, gscale, final_scale, grad_s, loss_out, ws);
        else mse_vec_kernel<false><<<blocks, MSE_THREADS, 0, st>>>(s, t, n, head, gscale, final_scale, nullptr, loss_out, ws);
    } else {
        if (grad_s) mse_scalar_kernel<true><<<blocks, MSE_THREADS, 0, st>>>(s, t, n, gscale, final_scale, grad_s, loss_out, ws);
        else mse_scalar_kernel<false><<<blocks, MSE_THREADS, 0, st>>>(s, t, n, gscale, final_scale, nullptr, loss_out, ws);
    }
    PXL_CHECK_LAUNCH();
    return 0;
}

__global__ void __launch_bounds__(256)
mse_bwd_kernel(const float* __restrict__ s, const float* __restrict__ t, int64_t n, float c,
               const float* __restrict__ upstream, float* __restrict__ grad) {
    const float g = c * upstream[0];
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        grad[i] = g * (s[i] - t[i]);
}

extern "C" int pxl_mse_consistency_bwd(const float* s, const float* t, int64_t n, float loss_scale,
                                       const float* upstream, float* grad_s, void* stream) {
    if (!s || !t || !upstream || !grad_s || n <= 0) return PXL_ERR_BAD_ARG;
    int blocks = (int)(pxl_cdiv(n, 256 * 4) < PXL_NUM_SMS * 8 ? pxl_cdiv(n, 256 * 4) : PXL_NUM_SMS * 8);
    mse_bwd_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(s, t, n, (float)(2.0 * loss_scale / (double)n), upstream, grad_s);
    PXL_CHECK_LAUNCH();
    return 0;
}

// ------------------------------------------------------------------------------------------
// Cross entropy with ignore_index (task/sseg/criterion.py:24-38).  One thread per pixel, the C
// channel planes are read coalesced (consecutive threads = consecutive pixels of one plane).
//   algorithmic traffic: 4*C + 4 B/pixel forward, + 4*C B/pixel when the gradient is written.
// ------------------------------------------------------------------------------------------
#define CE_MAXC 32
template <bool WRITE_GRAD>
__global__ void __launch_bounds__(256)
ce2d_kernel(const float* __restrict__ logits, const float* __restrict__ labels, int C, int64_t HW,
            int ignore_index, float* __restrict__ per_sample, float* __restrict__ grad,
            const float* __restrict__ upstream, float upstream_const) {
    const int b = blockIdx.y;
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const float* lg = logits + (int64_t)b * C * HW;
    float loss = 0.f;
    if (p < HW) {
        float v[CE_MAXC];
        float m = -CUDART_INF_F;
#pragma unroll
        for (int c = 0; c < CE_MAXC; ++c)
            if (c < C) { v[c] = lg[(int64_t)c * HW + p]; m = fmaxf(m, v[c]); }
        float se = 0.f;
#pragma unroll
        for (int c = 0; c < CE_MAXC; ++c)
            if (c < C) { v[c] = expf(v[c] - m); se += v[c]; }
        const float lab_f = labels[(int64_t)b * HW + p];
        const long long lab = (long long)lab_f;     // .long(): truncation toward zero
        const bool valid = (lab != (long long)ignore_index) && lab >= 0 && lab < C;
        float x_lab = 0.f;
        if (valid) {
            // re-read the target logit (L1/L2 hit) instead of dynamic register indexing
            x_lab = lg[(int64_t)lab * HW + p];
            loss = (logf(se) + m) - x_lab;
        }
        if (WRITE_GRAD) {
            const float g = (upstream ? upstream[b] : upstream_const) / (float)HW;
            const float inv = valid ? g / se : 0.f;
            float* gp = grad + (int64_t)b * C * HW + p;
#pragma unroll
            for (int c = 0; c < CE_MAXC; ++c)
                if (c < C) {
                    float gv = v[c] * inv;
                    if (valid && c == (int)lab) gv -= g;
                    gp[(int64_t)c * HW] = gv;
                }
        }
    }
    // block reduce -> one atomic per block
    __shared__ float wp[8];
    loss = warp_sum(loss);
    if ((threadIdx.x & 31) == 0) wp[threadIdx.x >> 5] = loss;
    __syncthreads();
    if (threadIdx.x == 0) {
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) s += wp[i];
        atomicAdd(per_sample + b, s / (float)HW);
    }
}

extern "C" int pxl_ce2d(const float* logits, const float* labels, int n, int C, int64_t HW,
                        int ignore_index, float* per_sample, float* grad_logits,
                        const float* upstream, float upstream_const, void* stream) {
    if (!logits || !labels || !per_sample || n <= 0 || C <= 0 || HW <= 0) return PXL_ERR_BAD_ARG;
    if (C > CE_MAXC) return PXL_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(per_sample, 0, sizeof(float) * n, st);
    if (e != cudaSuccess) return (int)e;
    dim3 grid((unsigned)pxl_cdiv(HW, 256), (unsigned)n);
    if (grad_logits) ce2d_kernel<true><<<grid, 256, 0, st>>>(logits, labels, C, HW, ignore_index, per_sample, grad_logits, upstream, upstream_const);
    else ce2d_kernel<false><<<grid, 256, 0, st>>>(logits, labels, C, HW, ignore_index, per_sample, nullptr, nullptr, 0.f);
    PXL_CHECK_LAUNCH();
    return 0;
}

// ------------------------------------------------------------------------------------------
// channel softmax fwd / bwd on planar maps (task/sseg/model.py:62)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
softmax_planar_kernel(const float* __restrict__ logits, float* __restrict__ prob, int C, int64_t HW) {
    const int b = blockIdx.y;
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= HW) return;
    const float* lg = logits + (int64_t)b * C * HW + p;
    float* pr = prob + (int64_t)b * C * HW + p;
    float v[CE_MAXC];
    float m = -CUDART_INF_F;
#pragma unroll
    for (int c = 0; c < CE_MAXC; ++c)
        if (c < C) { v[c] = lg[(int64_t)c * HW]; m = fmaxf(m, v[c]); }
    float se = 0.f;
#pragma unroll
    for (int c = 0; c < CE_MAXC; ++c)
        if (c < C) { v[c] = expf(v[c] - m); se += v[c]; }
    const float inv = 1.f / se;
#pragma unroll
    for (int c = 0; c < CE_MAXC; ++c)
        if (c < C) pr[(int64_t)c * HW] = v[c] * inv;
}

extern "C" int pxl_softmax_planar(const float* logits, float* prob, int n, int C, int64_t HW, void* stream) {
    if (!logits || !prob || n <= 0 || C <= 0 || HW <= 0) return PXL_ERR_BAD_ARG;
    if (C > CE_MAXC) return PXL_ERR_UNSUPPORTED;
    dim3 grid((unsigned)pxl_cdiv(HW, 256), (unsigned)n);
    softmax_planar_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(logits, prob, C, HW);
    PXL_CHECK_LAUNCH();
    return 0;
}

__global__ void __launch_bounds__(256)
softmax_planar_bwd_kernel(const float* __restrict__ prob, const float* __restrict__ gprob,
                          float* __restrict__ glogits, int C, int64_t HW) {
    const int b = blockIdx.y;
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= HW) return;
    const int64_t base = (int64_t)b * C * HW + p;
    float pv[CE_MAXC], gv[CE_MAXC];
    float dot = 0.f;
#pragma unroll
    for (int c = 0; c < CE_MAXC; ++c)
        if (c < C) { pv[c] = prob[base + (int64_t)c * HW]; gv[c] = gprob[base + (int64_t)c * HW]; dot += pv[c] * gv[c]; }
#pragma unroll
    for (int c = 0; c < CE_MAXC; ++c)
        if (c < C) glogits[base + (int64_t)c * HW] = pv[c] * (gv[c] - dot);
}

extern "C" int pxl_softmax_planar_bwd(const float* prob, const float* grad_prob, float* grad_logits,
                                      int n, int C, int64_t HW, void* stream) {
    if (!prob || !grad_prob || !grad_logits || n <= 0 || C <= 0 || HW <= 0) return PXL_ERR_BAD_ARG;
    if (C > CE_MAXC) return PXL_ERR_UNSUPPORTED;
    dim3 grid((unsigned)pxl_cdiv(HW, 256), (unsigned)n);
    softmax_planar_bwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(prob, grad_prob, grad_logits, C, HW);
    PXL_CHECK_LAUNCH();
    return 0;
}

// ------------------------------------------------------------------------------------------
// fused softmax(student logits) + MSE against target probabilities (+ gradient through the
// softmax): the CutMix / GCT / CCT consistency tail (ssl_cutmix.py:206-215)
// ------------------------------------------------------------------------------------------
template <bool WRITE_PROB, bool WRITE_GRAD>
__global__ void __launch_bounds__(256)
softmax_mse_kernel(const float* __restrict__ logits, const float* __restrict__ tprob, int C, int64_t HW,
                   float gscale, float* __restrict__ prob_out, float* __restrict__ grad,
                   double* __restrict__ partial) {
    const int b = blockIdx.y;
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    float acc = 0.f;
    if (p < HW) {
        const int64_t base = (int64_t)b * C * HW + p;
        float v[CE_MAXC], d[CE_MAXC];
        float m = -CUDART_INF_F;
#pragma unroll
        for (int c = 0; c < CE_MAXC; ++c)
            if (c < C) { v[c] = logits[base + (int64_t)c * HW]; m = fmaxf(m, v[c]); }
        float se = 0.f;
#pragma unroll
        for (int c = 0; c < CE_MAXC; ++c)
            if (c < C) { v[c] = expf(v[c] - m); se += v[c]; }
        const float inv = 1.f / se;
        float dot = 0.f;
#pragma unroll
        for (int c = 0; c < CE_MAXC; ++c)
            if (c < C) {
                v[c] *= inv;
                if (WRITE_PROB) prob_out[base + (int64_t)c * HW] = v[c];
                d[c] = v[c] - tprob[base + (int64_t)c * HW];
                acc += d[c] * d[c];
                dot += d[c] * v[c];
            }
        if (WRITE_GRAD) {
#pragma unroll
            for (int c = 0; c < CE_MAXC; ++c)
                if (c < C) grad[base + (int64_t)c * HW] = gscale * v[c] * (d[c] - dot);
        }
    }
    __shared__ float wp[8];
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) wp[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
#pragma unroll
        for (int i = 0; i < 8; ++i) s += (double)wp[i];
        atomicAdd(partial, s);
    }
}

__global__ void finalize_scalar_kernel(double* acc, double scale, float* out) {
    out[0] = (float)(acc[0] * scale);
    acc[0] = 0.0;
}

extern "C" int pxl_softmax_mse(const float* s_logits, const float* t_prob, int n, int C, int64_t HW,
                               float loss_scale, float* loss_out, float* prob_out, float* grad_logits,
                               void* workspace, void* stream) {
    if (!s_logits || !t_prob || !loss_out || !workspace || n <= 0 || C <= 0 || HW <= 0) return PXL_ERR_BAD_ARG;
    if (C > CE_MAXC) return PXL_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    MseWorkspace* ws = (MseWorkspace*)workspace;
    const double N = (double)n * C * (double)HW;
    const float gscale = (float)(2.0 * loss_scale / N);
    dim3 grid((unsigned)pxl_cdiv(HW, 256), (unsigned)n);
    double* acc = &ws->scalar_acc;
    if (prob_out && grad_logits) softmax_mse_kernel<true, true><<<grid, 256, 0, st>>>(s_logits, t_prob, C, HW, gscale, prob_out, grad_logits, acc);
    else if (prob_out) softmax_mse_kernel<true, false><<<grid, 256, 0, st>>>(s_logits, t_prob, C, HW, gscale, prob_out, nullptr, acc);
    else if (grad_logits) softmax_mse_kernel<false, true><<<grid, 256, 0, st>>>(s_logits, t_prob, C, HW, gscale, nullptr, grad_logits, acc);
    else softmax_mse_kernel<false, false><<<grid, 256, 0, st>>>(s_logits, t_prob, C, HW, gscale, nullptr, nullptr, acc);
    PXL_CHECK_LAUNCH();
    finalize_scalar_kernel<<<1, 1, 0, st>>>(acc, (double)loss_scale / N, loss_out);
    PXL_CHECK_LAUNCH();
    return 0;
}

// ------------------------------------------------------------------------------------------
// CutMix mix: out = mask*a + (1-mask)*b  -- bit-exact with the reference's separately rounded
// fp32 ops (ssl_cutmix.py:195,428): __fmul_rn/__fadd_rn forbid FMA contraction.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
cutmix_mix_kernel(const float* __restrict__ mask, const float* __restrict__ a, const float* __restrict__ b,
                  float* __restrict__ out, int C, int64_t HW) {
    const int n = blockIdx.z, c = blockIdx.y;
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= HW) return;
    const float m = mask[(int64_t)n * HW + p];
    const int64_t i = ((int64_t)n * C + c) * HW + p;
    const float one_minus = __fsub_rn(1.0f, m);
    out[i] = __fadd_rn(__fmul_rn(m, a[i]), __fmul_rn(one_minus, b[i]));
}

extern "C" int pxl_cutmix_mix(const float* mask, const float* a, const float* b, float* out,
                              int n, int C, int64_t HW, void* stream) {
    if (!mask || !a || !b || !out || n <= 0 || C <= 0 || HW <= 0) return PXL_ERR_BAD_ARG;
    if (C > 65535 || n > 65535) return PXL_ERR_UNSUPPORTED;
    dim3 grid((unsigned)pxl_cdiv(HW, 256), (unsigned)C, (unsigned)n);
    cutmix_mix_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(mask, a, b, out, C, HW);
    PXL_CHECK_LAUNCH();
    return 0;
}

__global__ void __launch_bounds__(256)
cutmix_conf_kernel(const float* __restrict__ prob, int C, int64_t HW, float thr,
                   unsigned long long* __restrict__ count) {
    const int b = blockIdx.y;
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int hit = 0;
    if (p < HW) {
        const float* pr = prob + (int64_t)b * C * HW + p;
        float m = -CUDART_INF_F;
        for (int c = 0; c < C; ++c) m = fmaxf(m, pr[(int64_t)c * HW]);
        hit = m > thr;
    }
    unsigned int ballot = __ballot_sync(0xffffffffu, hit);
    __shared__ int wp[8];
    if ((threadIdx.x & 31) == 0) wp[threadIdx.x >> 5] = __popc(ballot);
    __syncthreads();
    if (threadIdx.x == 0) {
        int s = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) s += wp[i];
        if (s) atomicAdd(count, (unsigned long long)s);
    }
}

extern "C" int pxl_cutmix_confidence(const float* prob, int n, int C, int64_t HW, float thr,
                                     unsigned long long* count_out, void* stream) {
    if (!prob || !count_out || n <= 0 || C <= 0 || HW <= 0) return PXL_ERR_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(count_out, 0, sizeof(unsigned long long), st);
    if (e != cudaSuccess) return (int)e;
    dim3 grid((unsigned)pxl_cdiv(HW, 256), (unsigned)n);
    cutmix_conf_kernel<<<grid, 256, 0, st>>>(prob, C, HW, thr, count_out);
    PXL_CHECK_LAUNCH();
    return 0;
}
