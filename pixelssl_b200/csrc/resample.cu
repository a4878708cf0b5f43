// Bilinear resize forward / backward (F.interpolate(mode='bilinear'), both align_corners flavours)
//   deeplab_v2.py:32, _pspnet.py:99-100,127, ssl_gct.py:580, ssl_adv.py:488, ssl_cct.py:482
// Output (and grad_out) are planar [n, C, H, W]; the small input is planar or NHWC (ldc stride).
// Forward is write-bound: 4*C B per output pixel.  The source-index arithmetic mirrors ATen's
// area_pixel_compute_source_index so results agree to fp32 round-off.
#include "common.cuh"

__device__ __forceinline__ float src_index(float scale, int dst, bool align_corners) {
    if (align_corners) return scale * (float)dst;
    float s = scale * ((float)dst + 0.5f) - 0.5f;
    return s < 0.f ? 0.f : s;
}

static inline float resize_scale(int in, int out, int align_corners) {
    if (align_corners) return out > 1 ? (float)(in - 1) / (float)(out - 1) : 0.f;
    return (float)in / (float)out;
}

#define BL_MAXC 32
template <bool NHWC>
__global__ void __launch_bounds__(256)
bilinear_fwd_kernel(const float* __restrict__ in, float* __restrict__ out, int C, int h, int w, int H, int W,
                    float sh, float sw, bool ac, int ldc) {
    const int b = blockIdx.z;
    const int y = blockIdx.y;
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= W) return;
    const float fy = src_index(sh, y, ac), fx = src_index(sw, x, ac);
    const int y0 = (int)fy, x0 = (int)fx;
    const int y1 = y0 + (y0 < h - 1 ? 1 : 0), x1 = x0 + (x0 < w - 1 ? 1 : 0);
    const float ly1 = fy - (float)y0, lx1 = fx - (float)x0;
    const float ly0 = 1.f - ly1, lx0 = 1.f - lx1;
    const int64_t HW = (int64_t)H * W;
    float* op = out + (int64_t)b * C * HW + (int64_t)y * W + x;
    if (NHWC) {
        const float* p00 = in + ((int64_t)(b * h + y0) * w + x0) * ldc;
        const float* p01 = in + ((int64_t)(b * h + y0) * w + x1) * ldc;
        const float* p10 = in + ((int64_t)(b * h + y1) * w + x0) * ldc;
        const float* p11 = in + ((int64_t)(b * h + y1) * w + x1) * ldc;
        for (int c = 0; c < C; ++c)
            op[(int64_t)c * HW] = ly0 * (lx0 * __ldg(p00 + c) + lx1 * __ldg(p01 + c)) +
                                  ly1 * (lx0 * __ldg(p10 + c) + lx1 * __ldg(p11 + c));
    } else {
        const int64_t hw = (int64_t)h * w;
        const float* base = in + (int64_t)b * C * hw;
        for (int c = 0; c < C; ++c) {
            const float* pc = base + (int64_t)c * hw;
            op[(int64_t)c * HW] = ly0 * (lx0 * __ldg(pc + y0 * w + x0) + lx1 * __ldg(pc + y0 * w + x1)) +
                                  ly1 * (lx0 * __ldg(pc + y1 * w + x0) + lx1 * __ldg(pc + y1 * w + x1));
        }
    }
}

extern "C" int pxl_bilinear_fwd(const float* in, float* out, int n, int C, int h, int w, int H, int W,
                                int align_corners, int in_nhwc, int ldc, void* stream) {
    if (!in || !out || n <= 0 || C <= 0 || h <= 0 || w <= 0 || H <= 0 || W <= 0) return PXL_ERR_BAD_ARG;
    if (H > 65535 || n > 65535) return PXL_ERR_UNSUPPORTED;
    const float sh = resize_scale(h, H, align_corners), sw = resize_scale(w, W, align_corners);
    dim3 grid((unsigned)pxl_cdiv(W, 256), (unsigned)H, (unsigned)n);
    cudaStream_t st = (cudaStream_t)stream;
    if (in_nhwc) bilinear_fwd_kernel<true><<<grid, 256, 0, st>>>(in, out, C, h, w, H, W, sh, sw, align_corners != 0, ldc);
    else bilinear_fwd_kernel<false><<<grid, 256, 0, st>>>(in, out, C, h, w, H, W, sh, sw, align_corners != 0, C);
    PXL_CHECK_LAUNCH();
    return 0;
}

// ------------------------------------------------------------------------------------------
// backward: grad_in[b,c,i,j] = sum over the output pixels whose 2x2 support includes (i,j).
// One CTA per (low-res row i, channel c, sample b).  Its warps stream the contributing
// high-res rows (coalesced along x), weight by the y-coefficient and scatter along x into a
// shared-memory row accumulator with shared atomics; each high-res row is read by the (at
// most) two low-res rows it touches.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void y_support(int i, int h, int H, float sh, bool ac, int& ylo, int& yhi) {
    // conservative bounds on {y : y0(y) == i or y1(y) == i}; refined per row in the loop
    if (sh <= 0.f) { ylo = 0; yhi = H - 1; return; }
    float lo, hi;
    if (ac) { lo = ((float)i - 1.f) / sh; hi = ((float)i + 1.f) / sh; }
    else { lo = ((float)i - 0.5f) / sh - 0.5f; hi = ((float)i + 1.5f) / sh - 0.5f; }
    ylo = (int)floorf(lo) - 1; yhi = (int)ceilf(hi) + 1;
    if (i == 0) ylo = 0;           // align_corners=False clamps negative sources to row 0
    if (ylo < 0) ylo = 0;
    if (yhi > H - 1) yhi = H - 1;
}

// v3: no contended atomics, no per-element weight arithmetic.
//   * per CTA (low-res row i, channel c, image b): the horizontal weights wx(x, j) depend only on the
//     column pair, so they are tabulated once in shared memory (wtab[j][t], t over the <= SUP high-res
//     columns under low-res column j);
//   * the ~2/sh contributing high-res rows are staged G at a time by the whole CTA (coalesced loads,
//     G*W/128 independent loads per thread), stored at x + x/R so that lanes walking supports that
//     start R apart hit distinct banks;
//   * work item = (staged row g, column j): a SUP-long dot product from shared memory, added into the
//     accumulator row of slot g (the same thread owns item (g, j) in every group, so no atomics); the G slot
//     rows are summed in slot order at the end - the same result every run.
template <bool NHWC>
__global__ void __launch_bounds__(128)
bilinear_bwd_kernel(const float* __restrict__ gout, float* __restrict__ gin, int C, int h, int w, int H, int W,
                    float sh, float sw, bool ac, int ldc, int R, int rowbuf, int SUP, int G) {
    extern __shared__ float smem[];
    const int wpad = (w + 31) & ~31;
    float* acc = smem;                                   // [G][wpad]
    int4* meta = reinterpret_cast<int4*>(smem + G * wpad);   // [wpad] {xlo, count, padded start, xlo % R}
    float* wtab = smem + G * wpad + 4 * wpad;            // [w][SUP]
    float* rb = wtab + (((size_t)w * SUP + 3) & ~(size_t)3);   // [G][rowbuf]
    const int i = blockIdx.x, b = blockIdx.z;

    // column tables: the same for every channel, built once per CTA; the CTA then walks over its channels
    // (blockIdx.y, blockIdx.y + gridDim.y, ...) - one CTA per channel spent half its time on these tables
    for (int j = threadIdx.x; j < w; j += blockDim.x) {
        int xlo, xhi;
        if (sw <= 0.f) { xlo = 0; xhi = W - 1; }
        else {
            float lo, hi;
            if (ac) { lo = ((float)j - 1.f) / sw; hi = ((float)j + 1.f) / sw; }
            else { lo = ((float)j - 0.5f) / sw - 0.5f; hi = ((float)j + 1.5f) / sw - 0.5f; }
            xlo = (int)floorf(lo) - 1; xhi = (int)ceilf(hi) + 1;
            if (j == 0 || xlo < 0) xlo = 0;
            if (xhi > W - 1) xhi = W - 1;
        }
        // trim to the columns that really touch j and tabulate their weights
        int first = -1, last = -2;
        for (int x = xlo; x <= xhi; ++x) {
            const float fx = src_index(sw, x, ac);
            const int x0 = (int)fx;
            const int x1 = x0 + (x0 < w - 1 ? 1 : 0);
            if (x0 == j || x1 == j) { if (first < 0) first = x; last = x; }
        }
        int cnt = last - first + 1;
        if (first < 0) { first = 0; cnt = 0; }
        if (cnt > SUP) cnt = SUP;                         // cannot happen (SUP is a host-side bound)
        for (int t = 0; t < cnt; ++t) {
            const int x = first + t;
            const float fx = src_index(sw, x, ac);
            const int x0 = (int)fx;
            const int x1 = x0 + (x0 < w - 1 ? 1 : 0);
            const float lx1 = fx - (float)x0;
            float wx = 0.f;
            if (x0 == j) wx += 1.f - lx1;
            if (x1 == j) wx += lx1;
            wtab[j * SUP + t] = wx;
        }
        meta[j] = make_int4(first, cnt, first + first / R, first % R);
    }
    int ylo, yhi;
    y_support(i, h, H, sh, ac, ylo, yhi);
    for (int c = blockIdx.y; c < C; c += gridDim.y) {
    __syncthreads();                                      // tables ready / previous channel written out
    for (int j = threadIdx.x; j < G * wpad; j += blockDim.x) acc[j] = 0.f;
    const float* gp = gout + ((int64_t)b * C + c) * (int64_t)H * W;
    for (int y0g = ylo; y0g <= yhi; y0g += G) {
        const int rows = min(G, yhi - y0g + 1);
        __syncthreads();                                  // previous group consumed / tables ready
        {   // x / R advanced incrementally (x grows by blockDim.x per trip): no integer division in the loop
            const int dq = (int)blockDim.x / R, dr = (int)blockDim.x - dq * R;
            int q = (int)threadIdx.x / R, r = (int)threadIdx.x - q * R;
            for (int x = threadIdx.x; x < W; x += blockDim.x) {
                const float* src = gp + (int64_t)y0g * W + x;
                float* dst = rb + x + q;
#pragma unroll 4
                for (int g = 0; g < rows; ++g) dst[g * rowbuf] = __ldg(src + (int64_t)g * W);
                q += dq; r += dr;
                if (r >= R) { r -= R; ++q; }
            }
        }
        __syncthreads();
        for (int item = threadIdx.x; item < rows * w; item += blockDim.x) {
            const int g = item / w, j = item - g * w;
            const int y = y0g + g;
            const float fy = src_index(sh, y, ac);
            const int yy0 = (int)fy;
            const int yy1 = yy0 + (yy0 < h - 1 ? 1 : 0);
            const float ly1 = fy - (float)yy0;
            float wy = 0.f;
            if (yy0 == i) wy += 1.f - ly1;
            if (yy1 == i) wy += ly1;
            if (wy == 0.f) continue;
            const int4 m = meta[j];
            const float* wt = wtab + j * SUP;
            const float* rp = rb + g * rowbuf;
            int pidx = m.z, rem = m.w;
            float sacc = 0.f;
            for (int t = 0; t < m.y; ++t) {
                sacc = fmaf(rp[pidx], wt[t], sacc);
                ++pidx;
                if (++rem == R) { rem = 0; ++pidx; }
            }
            acc[g * wpad + j] += sacc * wy;
        }
    }
    __syncthreads();
    for (int j = threadIdx.x; j < w; j += blockDim.x) {
        float s = acc[j];
        for (int g = 1; g < G; ++g) s += acc[g * wpad + j];
        if (NHWC) gin[((int64_t)(b * h + i) * w + j) * ldc + c] = s;
        else gin[(((int64_t)b * C + c) * h + i) * w + j] = s;
    }
    }
}

extern "C" int pxl_bilinear_bwd(const float* grad_out, float* grad_in, int n, int C, int h, int w, int H, int W,
                                int align_corners, int in_nhwc, int ldc, void* stream) {
    if (!grad_out || !grad_in || n <= 0 || C <= 0 || h <= 0 || w <= 0 || H <= 0 || W <= 0) return PXL_ERR_BAD_ARG;
    if (C > 65535 || n > 65535) return PXL_ERR_UNSUPPORTED;
    const float sh = resize_scale(h, H, align_corners), sw = resize_scale(w, W, align_corners);
    // channel groups: enough CTAs for ~8 per SM, each walking over C / groups channels with one set of column tables
    int64_t cgroups = pxl_cdiv((int64_t)PXL_NUM_SMS * 8, (int64_t)h * n);
    if (cgroups > C) cgroups = C;
    if (cgroups < 1) cgroups = 1;
    dim3 grid((unsigned)h, (unsigned)cgroups, (unsigned)n);
    cudaStream_t st = (cudaStream_t)stream;
    int R = sw > 0.f ? (int)(1.f / sw + 0.5f) : W;
    if (R < 1) R = 1;
    // high-res columns under one low-res column: < 2/sw + 2; odd so that wtab rows start in distinct banks
    int SUP = sw > 0.f ? (int)ceilf(2.f / sw) + 3 : W;
    if (SUP > W) SUP = W;
    SUP |= 1;
    const int rowbuf = ((W + W / R + 1) + 31) & ~31;
    const int wpad = (w + 31) & ~31;
    const size_t fixed = (size_t)wpad * 4 + (((size_t)w * SUP + 3) & ~(size_t)3);
    const size_t budget = 48 * 1024 / sizeof(float);
    if (fixed + (size_t)(rowbuf + wpad) > budget) return PXL_ERR_UNSUPPORTED;
    int G = (int)((budget - fixed) / (rowbuf + wpad));      // per staged row: its buffer and its accumulator row
    if (G > 8) G = 8;
    const size_t smem = (fixed + (size_t)G * (rowbuf + wpad)) * sizeof(float);
    if (in_nhwc) bilinear_bwd_kernel<true><<<grid, 128, smem, st>>>(grad_out, grad_in, C, h, w, H, W, sh, sw, align_corners != 0, ldc, R, rowbuf, SUP, G);
    else bilinear_bwd_kernel<false><<<grid, 128, smem, st>>>(grad_out, grad_in, C, h, w, H, W, sh, sw, align_corners != 0, C, R, rowbuf, SUP, G);
    PXL_CHECK_LAUNCH();
    return 0;
}
