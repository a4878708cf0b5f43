// FP32 (FFMA, exact fp32 accumulate) implicit-GEMM convolution on NHWC activations with a tap
// table: forward, dgrad (same kernel, transposed weights + negated taps), wgrad (split-K with
// fp32 atomics), weight transpose, bias gradient and the 7x7/2 stem.  This is the precise path
// (precision == 0) and the fallback for shapes the tcgen05 kernels do not cover.
//
// GEMM view:  out[M = N*OH*OW, Cout] = A[M, K = ntaps*Cin] * W^T[K, Cout], A gathered on the fly
// (im2col-free): row m, k = (tap, ci) reads in[n, (oy*mul+dy_t)/div, (ox*mul+dx_t)/div, ci].
#include "common.cuh"

struct ConvP {
    int N, H, W, Cin, OH, OW, Cout, ldo, mul, div, ntaps;
    int64_t M;
    short dy[PXL_MAX_TAPS], dx[PXL_MAX_TAPS];
};

static int fill_params(const pxl_conv_geom* g, const int* taps, ConvP& p) {
    if (!g || !taps) return PXL_ERR_BAD_ARG;
    if (g->ntaps <= 0 || g->ntaps > PXL_MAX_TAPS || g->mul <= 0 || g->div <= 0) return PXL_ERR_BAD_ARG;
    if (g->N <= 0 || g->H <= 0 || g->W <= 0 || g->Cin <= 0 || g->OH <= 0 || g->OW <= 0 || g->Cout <= 0 || g->ldo < g->Cout)
        return PXL_ERR_BAD_ARG;
    p.N = g->N; p.H = g->H; p.W = g->W; p.Cin = g->Cin; p.OH = g->OH; p.OW = g->OW; p.Cout = g->Cout;
    p.ldo = g->ldo; p.mul = g->mul; p.div = g->div; p.ntaps = g->ntaps;
    p.M = (int64_t)g->N * g->OH * g->OW;
    for (int t = 0; t < g->ntaps; ++t) {
        if (taps[2 * t] < -32768 || taps[2 * t] > 32767 || taps[2 * t + 1] < -32768 || taps[2 * t + 1] > 32767) return PXL_ERR_BAD_ARG;
        p.dy[t] = (short)taps[2 * t]; p.dx[t] = (short)taps[2 * t + 1];
    }
    return 0;
}

// ------------------------------------------------------------------------------------------
// forward / dgrad.  CTA tile 128 (pixels) x 64 (out channels) x 16 (k), 256 threads, 8x4 per
// thread, register-prefetch double buffering through shared memory.
// ------------------------------------------------------------------------------------------
#define CF_BM 128
#define CF_BN 64
#define CF_BK 16
#define CF_APAD 4
#define CF_BPAD 4

template <bool VEC>
__global__ void __launch_bounds__(256, 2)
conv_fwd_fp32_kernel(const ConvP p, const float* __restrict__ in, const float* __restrict__ w,
                     const float* __restrict__ bias, float* __restrict__ out) {
    __shared__ float As[2][CF_BK][CF_BM + CF_APAD];
    __shared__ float Bs[2][CF_BK][CF_BN + CF_BPAD];
    __shared__ int rowBase[CF_BM];   // n*H*W, or -1 when the row is past M
    __shared__ int rowY[CF_BM], rowX[CF_BM];

    const int tid = threadIdx.x;
    const int64_t m0 = (int64_t)blockIdx.x * CF_BM;
    const int n0 = blockIdx.y * CF_BN;
    if (tid < CF_BM) {
        const int64_t m = m0 + tid;
        if (m < p.M) {
            const int ox = (int)(m % p.OW);
            const int64_t q = m / p.OW;
            const int oy = (int)(q % p.OH);
            const int n = (int)(q / p.OH);
            rowBase[tid] = n * p.H * p.W;
            rowY[tid] = oy * p.mul;
            rowX[tid] = ox * p.mul;
        } else {
            rowBase[tid] = -1; rowY[tid] = 0; rowX[tid] = 0;
        }
    }
    __syncthreads();

    const int K = p.ntaps * p.Cin;
    const int numK = (K + CF_BK - 1) / CF_BK;
    float4 ra[2], rb;

    auto load_chunk = [&](int kc) {
        if (VEC) {
            const int cpt = p.Cin / CF_BK;
            const int tap = kc / cpt, c0 = (kc - tap * cpt) * CF_BK;
            const int dy = p.dy[tap], dx = p.dx[tap];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int idx = tid + j * 256;
                const int row = idx >> 2, kq = idx & 3;
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                const int base = rowBase[row];
                if (base >= 0) {
                    int iy = rowY[row] + dy, ix = rowX[row] + dx;
                    bool ok = iy >= 0 && ix >= 0;
                    if (p.div > 1) {
                        ok = ok && (iy % p.div == 0) && (ix % p.div == 0);
                        iy /= p.div; ix /= p.div;
                    }
                    if (ok && iy < p.H && ix < p.W)
                        v = __ldg(reinterpret_cast<const float4*>(in + ((int64_t)base + (int64_t)iy * p.W + ix) * p.Cin + c0 + kq * 4));
                }
                ra[j] = v;
            }
            {
                const int row = tid >> 2, kq = tid & 3;
                const int co = n0 + row;
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (co < p.Cout)
                    v = __ldg(reinterpret_cast<const float4*>(w + ((int64_t)co * p.ntaps + tap) * p.Cin + c0 + kq * 4));
                rb = v;
            }
        } else {
            // generic path: any Cin; k = tap*Cin + ci decoded per element
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int idx = tid + j * 256;
                const int row = idx >> 2, kq = idx & 3;
                float vv[4] = {0.f, 0.f, 0.f, 0.f};
                const int base = rowBase[row];
                if (base >= 0) {
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int k = kc * CF_BK + kq * 4 + e;
                        if (k < K) {
                            const int tap = k / p.Cin, ci = k - tap * p.Cin;
                            int iy = rowY[row] + p.dy[tap], ix = rowX[row] + p.dx[tap];
                            bool ok = iy >= 0 && ix >= 0;
                            if (p.div > 1) { ok = ok && (iy % p.div == 0) && (ix % p.div == 0); iy /= p.div; ix /= p.div; }
                            if (ok && iy < p.H && ix < p.W) vv[e] = __ldg(in + ((int64_t)base + (int64_t)iy * p.W + ix) * p.Cin + ci);
                        }
                    }
                }
                ra[j] = make_float4(vv[0], vv[1], vv[2], vv[3]);
            }
            {
                const int row = tid >> 2, kq = tid & 3;
                const int co = n0 + row;
                float vv[4] = {0.f, 0.f, 0.f, 0.f};
                if (co < p.Cout) {
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int k = kc * CF_BK + kq * 4 + e;
                        if (k < K) vv[e] = __ldg(w + (int64_t)co * K + k);
                    }
                }
                rb = make_float4(vv[0], vv[1], vv[2], vv[3]);
            }
        }
    };
    auto store_chunk = [&](int buf) {
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int idx = tid + j * 256;
            const int row = idx >> 2, kq = idx & 3;
            As[buf][kq * 4 + 0][row] = ra[j].x; As[buf][kq * 4 + 1][row] = ra[j].y;
            As[buf][kq * 4 + 2][row] = ra[j].z; As[buf][kq * 4 + 3][row] = ra[j].w;
        }
        const int row = tid >> 2, kq = tid & 3;
        Bs[buf][kq * 4 + 0][row] = rb.x; Bs[buf][kq * 4 + 1][row] = rb.y;
        Bs[buf][kq * 4 + 2][row] = rb.z; Bs[buf][kq * 4 + 3][row] = rb.w;
    };

    float acc[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    const int tx = tid & 15, ty = tid >> 4;
    load_chunk(0);
    store_chunk(0);
    __syncthreads();
    for (int kc = 0; kc < numK; ++kc) {
        const int cur = kc & 1;
        if (kc + 1 < numK) load_chunk(kc + 1);
#pragma unroll
        for (int k = 0; k < CF_BK; ++k) {
            const float4 a0 = *reinterpret_cast<const float4*>(&As[cur][k][ty * 8]);
            const float4 a1 = *reinterpret_cast<const float4*>(&As[cur][k][ty * 8 + 4]);
            const float4 b = *reinterpret_cast<const float4*>(&Bs[cur][k][tx * 4]);
            const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float bb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
        }
        if (kc + 1 < numK) store_chunk(cur ^ 1);
        __syncthreads();
    }

    const int co0 = n0 + tx * 4;
    float bv[4] = {0.f, 0.f, 0.f, 0.f};
    if (bias) {
#pragma unroll
        for (int j = 0; j < 4; ++j) if (co0 + j < p.Cout) bv[j] = __ldg(bias + co0 + j);
    }
    const bool vec_out = ((p.ldo & 3) == 0) && (co0 + 3 < p.Cout);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int64_t m = m0 + ty * 8 + i;
        if (m >= p.M) continue;
        float* op = out + m * p.ldo + co0;
        if (vec_out) {
            *reinterpret_cast<float4*>(op) = make_float4(acc[i][0] + bv[0], acc[i][1] + bv[1], acc[i][2] + bv[2], acc[i][3] + bv[3]);
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) if (co0 + j < p.Cout) op[j] = acc[i][j] + bv[j];
        }
    }
}

extern "C" int pxl_conv_fp32_impl(const pxl_conv_geom* geom, const int* taps, const float* in, const float* w,
                                  const float* bias, float* out, void* stream) {
    ConvP p;
    int rc = fill_params(geom, taps, p);
    if (rc) return rc;
    if (!in || !w || !out) return PXL_ERR_BAD_ARG;
    if ((int64_t)p.N * p.H * p.W >= (1ll << 31)) return PXL_ERR_UNSUPPORTED;
    dim3 grid((unsigned)pxl_cdiv(p.M, CF_BM), (unsigned)pxl_cdiv(p.Cout, CF_BN));
    cudaStream_t st = (cudaStream_t)stream;
    if (p.Cin % CF_BK == 0) conv_fwd_fp32_kernel<true><<<grid, 256, 0, st>>>(p, in, w, bias, out);
    else conv_fwd_fp32_kernel<false><<<grid, 256, 0, st>>>(p, in, w, bias, out);
    PXL_CHECK_LAUNCH();
    return 0;
}

// ------------------------------------------------------------------------------------------
// wgrad: dW[co][t][ci] += sum_m dy[m][co] * in[pix(m,t)][ci].  CTA tile 64 (co) x 64 (ci) for one
// tap and one slice of the pixel range (split-K), 16 pixels per stage, 4x4 per thread, fp32
// atomics into dW (the caller's .grad buffer, zeroed at the start of the step).
// ------------------------------------------------------------------------------------------
#define WG_BM 64
#define WG_BN 64
#define WG_BK 16

template <bool VEC>
__global__ void __launch_bounds__(256, 2)
conv_wgrad_fp32_kernel(const ConvP p, const float* __restrict__ in, const float* __restrict__ dy,
                       float* __restrict__ dw, int tiles_ci, int64_t chunk) {
    __shared__ float As[2][WG_BK][WG_BM];
    __shared__ float Bs[2][WG_BK][WG_BN];
    const int tid = threadIdx.x;
    const int tile_co = blockIdx.x / tiles_ci, tile_ci = blockIdx.x % tiles_ci;
    const int co0 = tile_co * WG_BM, ci0 = tile_ci * WG_BN;
    const int tap = blockIdx.y;
    const int tdy = p.dy[tap], tdx = p.dx[tap];
    const int64_t mBeg = (int64_t)blockIdx.z * chunk;
    const int64_t mEnd = min(p.M, mBeg + chunk);
    const int numK = (int)((mEnd - mBeg + WG_BK - 1) / WG_BK);
    if (numK <= 0) return;

    float4 ra, rb;
    const int lp = tid >> 4, lq = tid & 15;   // pixel within stage, float4 column
    auto load_chunk = [&](int kc) {
        const int64_t m = mBeg + (int64_t)kc * WG_BK + lp;
        float4 va = make_float4(0.f, 0.f, 0.f, 0.f), vb = va;
        if (m < mEnd) {
            const int ox = (int)(m % p.OW);
            const int64_t q = m / p.OW;
            const int oy = (int)(q % p.OH);
            const int n = (int)(q / p.OH);
            int iy = oy * p.mul + tdy, ix = ox * p.mul + tdx;
            bool ok = iy >= 0 && ix >= 0;
            if (p.div > 1) { ok = ok && (iy % p.div == 0) && (ix % p.div == 0); iy /= p.div; ix /= p.div; }
            ok = ok && iy < p.H && ix < p.W;
            if (ok) {   // a pixel whose input tap is padding contributes nothing
                const float* dp = dy + m * p.ldo + co0 + lq * 4;
                const float* xp = in + ((int64_t)(n * p.H + iy) * p.W + ix) * p.Cin + ci0 + lq * 4;
                if (VEC) {
                    if (co0 + lq * 4 + 3 < p.ldo) va = __ldg(reinterpret_cast<const float4*>(dp));
                    if (ci0 + lq * 4 + 3 < p.Cin) vb = __ldg(reinterpret_cast<const float4*>(xp));
                } else {
                    float a[4] = {0, 0, 0, 0}, b[4] = {0, 0, 0, 0};
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        if (co0 + lq * 4 + e < p.Cout) a[e] = __ldg(dp + e);
                        if (ci0 + lq * 4 + e < p.Cin) b[e] = __ldg(xp + e);
                    }
                    va = make_float4(a[0], a[1], a[2], a[3]); vb = make_float4(b[0], b[1], b[2], b[3]);
                }
            }
        }
        ra = va; rb = vb;
    };
    auto store_chunk = [&](int buf) {
        *reinterpret_cast<float4*>(&As[buf][lp][lq * 4]) = ra;
        *reinterpret_cast<float4*>(&Bs[buf][lp][lq * 4]) = rb;
    };

    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    const int tx = tid & 15, ty = tid >> 4;   // tx -> ci quad, ty -> co quad

    load_chunk(0);
    store_chunk(0);
    __syncthreads();
    for (int kc = 0; kc < numK; ++kc) {
        const int cur = kc & 1;
        if (kc + 1 < numK) load_chunk(kc + 1);
#pragma unroll
        for (int k = 0; k < WG_BK; ++k) {
            const float4 a = *reinterpret_cast<const float4*>(&As[cur][k][ty * 4]);
            const float4 b = *reinterpret_cast<const float4*>(&Bs[cur][k][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        if (kc + 1 < numK) store_chunk(cur ^ 1);
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int co = co0 + ty * 4 + i;
        if (co >= p.Cout) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int ci = ci0 + tx * 4 + j;
            if (ci < p.Cin) atomicAdd(dw + ((int64_t)co * p.ntaps + tap) * p.Cin + ci, acc[i][j]);
        }
    }
}

extern "C" int pxl_conv_wgrad_fp32_impl(const pxl_conv_geom* geom, const int* taps, const float* in,
                                        const float* dy, float* dw, void* stream) {
    ConvP p;
    int rc = fill_params(geom, taps, p);
    if (rc) return rc;
    if (!in || !dy || !dw) return PXL_ERR_BAD_ARG;
    const int tiles_co = (int)pxl_cdiv(p.Cout, WG_BM), tiles_ci = (int)pxl_cdiv(p.Cin, WG_BN);
    const int64_t tiles = (int64_t)tiles_co * tiles_ci * p.ntaps;
    int64_t split = pxl_cdiv((int64_t)PXL_NUM_SMS * 4, tiles);
    const int64_t maxSplit = pxl_cdiv(p.M, 4 * WG_BK);
    if (split > maxSplit) split = maxSplit;
    if (split < 1) split = 1;
    if (split > 65535) split = 65535;
    int64_t chunk = pxl_cdiv(pxl_cdiv(p.M, split), WG_BK) * WG_BK;
    split = pxl_cdiv(p.M, chunk);
    dim3 grid((unsigned)(tiles_co * tiles_ci), (unsigned)p.ntaps, (unsigned)split);
    cudaStream_t st = (cudaStream_t)stream;
    const bool vec = (p.Cin % 4 == 0) && (p.ldo % 4 == 0);
    if (vec) conv_wgrad_fp32_kernel<true><<<grid, 256, 0, st>>>(p, in, dy, dw, tiles_ci, chunk);
    else conv_wgrad_fp32_kernel<false><<<grid, 256, 0, st>>>(p, in, dy, dw, tiles_ci, chunk);
    PXL_CHECK_LAUNCH();
    return 0;
}

// ------------------------------------------------------------------------------------------
// weight transpose [Cout][T][Cin] -> [Cin][T][Cout] (operand of dgrad), 32x32 smem tiles
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
transpose_w_kernel(const float* __restrict__ w, float* __restrict__ wt, int Cout, int T, int Cin) {
    __shared__ float tile[32][33];
    const int t = blockIdx.z;
    const int ci0 = blockIdx.x * 32, co0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int r = ty; r < 32; r += 8) {
        const int co = co0 + r, ci = ci0 + tx;
        tile[r][tx] = (co < Cout && ci < Cin) ? __ldg(w + ((int64_t)co * T + t) * Cin + ci) : 0.f;
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        const int ci = ci0 + r, co = co0 + tx;
        if (ci < Cin && co < Cout) wt[((int64_t)ci * T + t) * Cout + co] = tile[tx][r];
    }
}

extern "C" int pxl_conv_transpose_weights(const float* w, float* wt, int Cout, int T, int Cin, void* stream) {
    if (!w || !wt || Cout <= 0 || T <= 0 || Cin <= 0 || T > 65535) return PXL_ERR_BAD_ARG;
    dim3 grid((unsigned)pxl_cdiv(Cin, 32), (unsigned)pxl_cdiv(Cout, 32), (unsigned)T);
    transpose_w_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(w, wt, Cout, T, Cin);
    PXL_CHECK_LAUNCH();
    return 0;
}

// All conv weights of a parameter arena in ONE launch: table[n][6] = {src offset, dst offset, Cout, T, Cin, first tile}
// (element offsets into src_base / dst_base; tiles = 32x32 (co, ci) blocks per tap, numbered tensor by tensor).
// Replaces ~100 per-layer launches per step whose cost was launch latency, not bytes.
__global__ void __launch_bounds__(256)
transpose_w_batched_kernel(const float* __restrict__ src_base, float* __restrict__ dst_base,
                           const long long* __restrict__ table, int n) {
    __shared__ float tile[32][33];
    __shared__ long long ent[6];
    if (threadIdx.x == 0) {
        int lo = 0, hi = n - 1;                    // last tensor whose first tile <= blockIdx.x
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (table[mid * 6 + 5] <= (long long)blockIdx.x) lo = mid; else hi = mid - 1;
        }
        for (int k = 0; k < 6; ++k) ent[k] = table[lo * 6 + k];
    }
    __syncthreads();
    const float* w = src_base + ent[0];
    float* wt = dst_base + ent[1];
    const int Cout = (int)ent[2], T = (int)ent[3], Cin = (int)ent[4];
    const int local = (int)((long long)blockIdx.x - ent[5]);
    const int tiles_ci = (Cin + 31) / 32, tiles_co = (Cout + 31) / 32;
    const int t = local / (tiles_ci * tiles_co);
    const int rem = local - t * tiles_ci * tiles_co;
    const int ci0 = (rem % tiles_ci) * 32, co0 = (rem / tiles_ci) * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int r = ty; r < 32; r += 8) {
        const int co = co0 + r, ci = ci0 + tx;
        tile[r][tx] = (co < Cout && ci < Cin) ? __ldg(w + ((int64_t)co * T + t) * Cin + ci) : 0.f;
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        const int ci = ci0 + r, co = co0 + tx;
        if (ci < Cin && co < Cout) wt[((int64_t)ci * T + t) * Cout + co] = tile[tx][r];
    }
}

extern "C" int pxl_conv_transpose_weights_batched(const float* src_base, float* dst_base, const int64_t* table, int n,
                                                  int64_t total_tiles, void* stream) {
    if (!src_base || !dst_base || !table || n <= 0 || total_tiles <= 0 || total_tiles >= (1ll << 31)) return PXL_ERR_BAD_ARG;
    transpose_w_batched_kernel<<<(unsigned)total_tiles, 256, 0, (cudaStream_t)stream>>>(
        src_base, dst_base, reinterpret_cast<const long long*>(table), n);
    PXL_CHECK_LAUNCH();
    return 0;
}

// ------------------------------------------------------------------------------------------
// bias gradient: dbias[co] (+)= sum_rows dy[row*ldo + co]
// Two passes in a fixed order, so the result is the same in every run: each CTA of the first sums its row block into
// one partial per channel, the second adds the partials in row-block order.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
bias_grad_partial_kernel(const float* __restrict__ dy, int64_t rows, int Cout, int ldo, int64_t rowsPerBlock,
                         float* __restrict__ partial) {
    // thread (c = tid % 32, r = tid / 32); Cout <= 32 per grid.y slice
    const int c = blockIdx.y * 32 + (threadIdx.x & 31), rl = threadIdx.x >> 5;
    const int64_t r0 = (int64_t)blockIdx.x * rowsPerBlock, r1 = min(rows, r0 + rowsPerBlock);
    float s = 0.f;
    if (c < Cout)
        for (int64_t r = r0 + rl; r < r1; r += 8) s += __ldg(dy + r * ldo + c);
    __shared__ float sm[8][32];
    sm[rl][threadIdx.x & 31] = s;
    __syncthreads();
    if (rl == 0 && c < Cout) {
        float t = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) t += sm[i][threadIdx.x & 31];
        partial[(int64_t)blockIdx.x * Cout + c] = t;
    }
}

__global__ void bias_grad_sum_kernel(const float* __restrict__ partial, int nblocks, int Cout, float* __restrict__ dbias) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= Cout) return;
    float t = 0.f;
    for (int b = 0; b < nblocks; ++b) t += partial[(int64_t)b * Cout + c];
    dbias[c] += t;
}

extern "C" int pxl_bias_grad(const float* dy, int64_t rows, int Cout, int ldo, float* dbias, int accumulate, void* stream) {
    if (!dy || !dbias || rows <= 0 || Cout <= 0 || ldo < Cout) return PXL_ERR_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (!accumulate) {
        cudaError_t e = cudaMemsetAsync(dbias, 0, sizeof(float) * Cout, st);
        if (e != cudaSuccess) return (int)e;
    }
    int64_t rb = pxl_cdiv(rows, PXL_NUM_SMS * 4);
    if (rb < 64) rb = 64;
    const int nblocks = (int)pxl_cdiv(rows, rb);
    float* partial = nullptr;         // stream-ordered scratch: launches on other streams get their own
    cudaError_t e = cudaMallocAsync((void**)&partial, sizeof(float) * (size_t)nblocks * Cout, st);
    if (e != cudaSuccess) return (int)e;
    dim3 grid((unsigned)nblocks, (unsigned)pxl_cdiv(Cout, 32));
    bias_grad_partial_kernel<<<grid, 256, 0, st>>>(dy, rows, Cout, ldo, rb, partial);
    PXL_CHECK_LAUNCH();
    bias_grad_sum_kernel<<<(unsigned)pxl_cdiv(Cout, 128), 128, 0, st>>>(partial, nblocks, Cout, dbias);
    PXL_CHECK_LAUNCH();
    e = cudaFreeAsync(partial, st);
    return e == cudaSuccess ? 0 : (int)e;
}

// ------------------------------------------------------------------------------------------
// stem: conv 7x7 / stride 2 / pad 3, planar [N,3,H,W] image -> NHWC [N,OH,OW,64] (resnet.py:69)
// CTA: one output row segment of 64 pixels x 64 channels; the 7 x 133 x 3 input patch and the
// 147 x 64 weights live in shared memory.  thread = 4 pixels x 4 channels.
// ------------------------------------------------------------------------------------------
#define ST_PX 64
#define ST_IW (2 * ST_PX + 5)      // 133 input columns
#define ST_K 147

__global__ void __launch_bounds__(256)
stem_fwd_kernel(const float* __restrict__ img, const float* __restrict__ w, float* __restrict__ out,
                int N, int H, int W, int OH, int OW) {
    extern __shared__ float smem[];
    float* ws = smem;                         // [147][64]   k = (r*7+s)*3 + c
    float* is = smem + ST_K * 64;             // [3][7][ST_IW + 1]
    const int n = blockIdx.z, oy = blockIdx.y, ox0 = blockIdx.x * ST_PX;
    const int tid = threadIdx.x;
    for (int i = tid; i < ST_K * 64; i += 256) {
        const int co = i & 63, k = i >> 6;
        ws[i] = __ldg(w + (int64_t)co * ST_K + k);
    }
    const int ix0 = ox0 * 2 - 3, iy0 = oy * 2 - 3;
    for (int i = tid; i < 3 * 7 * ST_IW; i += 256) {
        const int xx = i % ST_IW, r = (i / ST_IW) % 7, c = i / (ST_IW * 7);
        const int iy = iy0 + r, ix = ix0 + xx;
        float v = 0.f;
        if (iy >= 0 && iy < H && ix >= 0 && ix < W) v = __ldg(img + ((int64_t)(n * 3 + c) * H + iy) * W + ix);
        is[(c * 7 + r) * (ST_IW + 1) + xx] = v;
    }
    __syncthreads();
    const int tx = tid & 15, ty = tid >> 4;   // tx: channel quad, ty: pixel quad
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (int r = 0; r < 7; ++r)
        for (int s = 0; s < 7; ++s)
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const int k = (r * 7 + s) * 3 + c;
                const float4 wv = *reinterpret_cast<const float4*>(ws + k * 64 + tx * 4);
                const float* ip = is + (c * 7 + r) * (ST_IW + 1) + s + ty * 8;
                const float a[4] = {ip[0], ip[2], ip[4], ip[6]};
                const float b[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
            }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int ox = ox0 + ty * 4 + i;
        if (ox < OW)
            *reinterpret_cast<float4*>(out + (((int64_t)n * OH + oy) * OW + ox) * 64 + tx * 4) =
                make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
    }
}

extern "C" int pxl_stem_conv7x7s2(const float* img, const float* w, float* out, int N, int H, int W,
                                  int OH, int OW, void* stream) {
    if (!img || !w || !out || N <= 0 || OH != (H + 6 - 7) / 2 + 1 || OW != (W + 6 - 7) / 2 + 1) return PXL_ERR_BAD_ARG;
    if (OH > 65535 || N > 65535) return PXL_ERR_UNSUPPORTED;
    const size_t smem = (ST_K * 64 + 3 * 7 * (ST_IW + 1)) * sizeof(float);
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(stem_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        attr_set = true;
    }
    dim3 grid((unsigned)pxl_cdiv(OW, ST_PX), (unsigned)OH, (unsigned)N);
    stem_fwd_kernel<<<grid, 256, smem, (cudaStream_t)stream>>>(img, w, out, N, H, W, OH, OW);
    PXL_CHECK_LAUNCH();
    return 0;
}

// stem wgrad: dW[co][k] += sum_pixels dy[pix][co] * patch[pix][k].  Persistent CTAs loop over
// (n, oy) output rows; thread (co = tid%64, ks = tid/64) owns k = ks, ks+4, ... (37 values).
#define SW_SLOTS 37
__global__ void __launch_bounds__(256)
stem_wgrad_kernel(const float* __restrict__ img, const float* __restrict__ dy, float* __restrict__ dw,
                  int N, int H, int W, int OH, int OW) {
    extern __shared__ float smem[];
    float* dys = smem;                               // [ST_PX][64]
    float* is = smem + ST_PX * 64;                   // [3][7][ST_IW + 1]
    const int tid = threadIdx.x;
    const int co = tid & 63, ks = tid >> 6;
    float acc[SW_SLOTS];
#pragma unroll
    for (int j = 0; j < SW_SLOTS; ++j) acc[j] = 0.f;
    const int segs = (OW + ST_PX - 1) / ST_PX;
    const int64_t units = (int64_t)N * OH * segs;
    for (int64_t u = blockIdx.x; u < units; u += gridDim.x) {
        const int seg = (int)(u % segs);
        const int oy = (int)((u / segs) % OH);
        const int n = (int)(u / ((int64_t)segs * OH));
        const int ox0 = seg * ST_PX;
        __syncthreads();
        for (int i = tid; i < ST_PX * 64; i += 256) {
            const int px = i >> 6, c = i & 63;
            const int ox = ox0 + px;
            dys[i] = ox < OW ? __ldg(dy + (((int64_t)n * OH + oy) * OW + ox) * 64 + c) : 0.f;
        }
        const int ix0 = ox0 * 2 - 3, iy0 = oy * 2 - 3;
        for (int i = tid; i < 3 * 7 * ST_IW; i += 256) {
            const int xx = i % ST_IW, r = (i / ST_IW) % 7, c = i / (ST_IW * 7);
            const int iy = iy0 + r, ix = ix0 + xx;
            float v = 0.f;
            if (iy >= 0 && iy < H && ix >= 0 && ix < W) v = __ldg(img + ((int64_t)(n * 3 + c) * H + iy) * W + ix);
            is[(c * 7 + r) * (ST_IW + 1) + xx] = v;
        }
        __syncthreads();
        for (int px = 0; px < ST_PX; ++px) {
            const float d = dys[px * 64 + co];
#pragma unroll
            for (int j = 0; j < SW_SLOTS; ++j) {
                const int k = ks + 4 * j;
                if (k < ST_K) {
                    const int c = k % 3, rs = k / 3, r = rs / 7, s = rs % 7;
                    acc[j] = fmaf(d, is[(c * 7 + r) * (ST_IW + 1) + 2 * px + s], acc[j]);
                }
            }
        }
    }
#pragma unroll
    for (int j = 0; j < SW_SLOTS; ++j) {
        const int k = ks + 4 * j;
        if (k < ST_K) atomicAdd(dw + (int64_t)co * ST_K + k, acc[j]);
    }
}

extern "C" int pxl_stem_conv7x7s2_wgrad(const float* img, const float* dy, float* dw, int N, int H, int W,
                                        int OH, int OW, void* stream) {
    if (!img || !dy || !dw || N <= 0) return PXL_ERR_BAD_ARG;
    const size_t smem = (ST_PX * 64 + 3 * 7 * (ST_IW + 1)) * sizeof(float);
    stem_wgrad_kernel<<<PXL_NUM_SMS * 2, 256, smem, (cudaStream_t)stream>>>(img, dy, dw, N, H, W, OH, OW);
    PXL_CHECK_LAUNCH();
    return 0;
}

// ------------------------------------------------------------------------------------------
// stem im2col for the tensor-core path: cols[pixel][k], k = (r*7 + s)*3 + c for k < 147 (the physical
// order of the channels_last [64,3,7,7] weight), zero for 147 <= k < 160.  The 7x7/2 stem then runs as a
// flat 1x1 convolution with 160 input lanes on tcgen05 (forward and wgrad share the matrix).
// ------------------------------------------------------------------------------------------
#define ST_KP 160
__global__ void __launch_bounds__(256)
stem_im2col_kernel(const float* __restrict__ img, float* __restrict__ cols, int N, int H, int W, int OH, int OW) {
    const int64_t total4 = (int64_t)N * OH * OW * (ST_KP / 4);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += (int64_t)gridDim.x * blockDim.x) {
        const int k4 = (int)(i % (ST_KP / 4));
        const int64_t pix = i / (ST_KP / 4);
        const int ox = (int)(pix % OW), oy = (int)((pix / OW) % OH), n = (int)(pix / ((int64_t)OW * OH));
        float v[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int k = k4 * 4 + e;
            float x = 0.f;
            if (k < ST_K) {
                const int c = k % 3, rs = k / 3, r = rs / 7, sx = rs - r * 7;
                const int iy = oy * 2 - 3 + r, ix = ox * 2 - 3 + sx;
                if (iy >= 0 && iy < H && ix >= 0 && ix < W) x = __ldg(img + ((int64_t)(n * 3 + c) * H + iy) * W + ix);
            }
            v[e] = x;
        }
        reinterpret_cast<float4*>(cols)[i] = make_float4(v[0], v[1], v[2], v[3]);
    }
}

extern "C" int pxl_stem_im2col(const float* img, float* cols, int N, int H, int W, int OH, int OW, void* stream) {
    if (!img || !cols || N <= 0 || H <= 0 || W <= 0 || OH <= 0 || OW <= 0) return PXL_ERR_BAD_ARG;
    const int64_t total4 = (int64_t)N * OH * OW * (ST_KP / 4);
    int64_t blocks = pxl_cdiv(total4, 256 * 4);
    if (blocks > PXL_NUM_SMS * 16) blocks = PXL_NUM_SMS * 16;
    stem_im2col_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(img, cols, N, H, W, OH, OW);
    PXL_CHECK_LAUNCH();
    return 0;
}

// fp16-pair variant for the kind::f16 tensor-core path (csrc/h16_prep.cu): the unfolded stem matrix is written directly
// as hi / lo planes [pixels][192] (147 taps*channels + 45 zero lanes: K must be a multiple of the 64-element operand
// row), value * scale = hi + lo.  768 B per output pixel instead of 640 B of fp32, and no separate split pass.
#include <cuda_fp16.h>
#define ST_KH 192
#define IM_TOX 32                       // output tile of a CTA: 32 x 4 pixels of one image
#define IM_TOY 4
#define IM_PW (2 * IM_TOX + 5)          // input patch it touches: 69 x 13 pixels x 3 channels (10.8 KB of shared memory)
#define IM_PH (2 * IM_TOY + 5)
__constant__ int c_im_koff[ST_KH];      // k -> offset of tap k inside the patch for the tile's first pixel (-1: zero lane)

// The patch is staged once in shared memory (coalesced rows, zero outside the image = the convolution's padding); every
// thread then emits 4-lane groups of the [pixels][192] matrix with one table lookup + one shared-memory load per value
// instead of a div/mod chain and a scattered global load (the round-2 first version: 0.71 ms per launch).
__global__ void __launch_bounds__(256)
stem_im2col_h16_kernel(const float* __restrict__ img, uint2* __restrict__ hi, uint2* __restrict__ lo, float scale,
                       int N, int H, int W, int OH, int OW, int tilesX, int tilesY, int* __restrict__ sat) {
    __shared__ float patch[3 * IM_PH * IM_PW];
    __shared__ short koff_s[ST_KH];          // the lanes of a warp index the table with 32 different k: from constant memory
                                             // that serialises 32-fold (it bounded the kernel: 1.57 ms -> see profiles/)
    for (int i = threadIdx.x; i < ST_KH; i += blockDim.x) koff_s[i] = (short)c_im_koff[i];
    const int t = blockIdx.x;
    const int tx = t % tilesX, ty = (t / tilesX) % tilesY, n = t / (tilesX * tilesY);
    const int ox0 = tx * IM_TOX, oy0 = ty * IM_TOY;
    const int ix0 = ox0 * 2 - 3, iy0 = oy0 * 2 - 3;
    for (int i = threadIdx.x; i < 3 * IM_PH * IM_PW; i += blockDim.x) {
        const int px = i % IM_PW, py = (i / IM_PW) % IM_PH, c = i / (IM_PW * IM_PH);
        const int iy = iy0 + py, ix = ix0 + px;
        patch[i] = (iy >= 0 && iy < H && ix >= 0 && ix < W) ? __ldg(img + ((int64_t)(n * 3 + c) * H + iy) * W + ix) * scale : 0.f;
    }
    __syncthreads();
    bool clipped = false;
    for (int i = threadIdx.x; i < IM_TOX * IM_TOY * (ST_KH / 4); i += blockDim.x) {
        const int k4 = i % (ST_KH / 4), p = i / (ST_KH / 4);
        const int lx = p % IM_TOX, ly = p / IM_TOX;
        const int ox = ox0 + lx, oy = oy0 + ly;
        if (ox >= OW || oy >= OH) continue;
        const int base = (2 * ly) * IM_PW + 2 * lx;
        unsigned short h[4], l[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int off = koff_s[k4 * 4 + e];
            const float v = off >= 0 ? patch[off + base] : 0.f;
            const float cl = fminf(fmaxf(v, -65504.f), 65504.f);
            clipped |= (cl != v) && (v == v);
            const __half hh = __float2half_rn(cl);
            h[e] = __half_as_ushort(hh);
            l[e] = __half_as_ushort(__float2half_rn(cl - __half2float(hh)));
        }
        const int64_t o = (((int64_t)n * OH + oy) * OW + ox) * (ST_KH / 4) + k4;
        hi[o] = make_uint2((uint32_t)h[0] | ((uint32_t)h[1] << 16), (uint32_t)h[2] | ((uint32_t)h[3] << 16));
        if (lo) lo[o] = make_uint2((uint32_t)l[0] | ((uint32_t)l[1] << 16), (uint32_t)l[2] | ((uint32_t)l[3] << 16));
    }
    if (clipped && sat) atomicAdd(sat, 1);
}

extern "C" int* pxl_h16_sat_counter(void);

extern "C" int pxl_stem_im2col_h16(const float* img, void* hi, void* lo, float scale, int N, int H, int W, int OH, int OW,
                                   void* stream) {
    if (!img || !hi || !(scale > 0.f) || N <= 0 || H <= 0 || W <= 0 || OH <= 0 || OW <= 0) return PXL_ERR_BAD_ARG;
    static bool table = false;
    if (!table) {
        int koff[ST_KH];
        for (int k = 0; k < ST_KH; ++k) {
            if (k >= ST_K) { koff[k] = -1; continue; }
            const int c = k % 3, rs = k / 3, r = rs / 7, sx = rs - r * 7;
            koff[k] = (c * IM_PH + r) * IM_PW + sx;
        }
        if (cudaMemcpyToSymbol(c_im_koff, koff, sizeof(koff)) != cudaSuccess) return PXL_ERR_BAD_ARG;
        table = true;
    }
    const int tilesX = (OW + IM_TOX - 1) / IM_TOX, tilesY = (OH + IM_TOY - 1) / IM_TOY;
    const int64_t blocks = (int64_t)N * tilesX * tilesY;
    if (blocks > 0x7fffffff) return PXL_ERR_UNSUPPORTED;
    stem_im2col_h16_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(img, (uint2*)hi, (uint2*)lo, scale, N, H, W, OH, OW,
                                                                              tilesX, tilesY, pxl_h16_sat_counter());
    PXL_CHECK_LAUNCH();
    return 0;
}
