// tcgen05 (5th-gen tensor core) implicit-GEMM convolution for sm_100a: forward / dgrad (wgrad at the end of the file).
//
//   D[128 output pixels, BN out channels] (fp32, in TMEM) += A[128, K] * B[BN, K]^T  per (tap, 128-byte channel chunk)
//   K per chunk: 64 fp16 values (kind::f16, the benchmarked modes) or 32 tf32 values (kind::tf32)
//
// * A (activations, NHWC) is staged by TMA as a 4-D box {chunk, BW, BH, 1}: one 128-byte row per
//   output pixel of a BH x BW spatial tile, shifted by the tap offset; out-of-image coordinates
//   are zero-filled by the TMA unit, which IS the convolution's zero padding (im2col-free).
//   1x1 convolutions use the same path with the pixel axis flattened (BW = 128, BH = 1).
// * B (weights [Cout][tap][Cin], K-major) is a 2-D box {chunk, BN}.
// * Both land in shared memory in the canonical K-major SWIZZLE_128B layout and feed tcgen05.mma (four MMAs of
//   32 bytes of K per operand pair and stage); accumulators live in TMEM (double-buffered in the persistent
//   kernels) and are read back with tcgen05.ld by the epilogue warps.
// * precision 3 ("f16x3", default of bench.py): both operands arrive as fp16 PAIRS x*s = hi + lo written by the
//   producing kernels (csrc/h16_prep.cu), D += A_hi*B_hi + A_lo*B_hi + A_hi*B_lo recovers fp32-grade products with
//   fp32 accumulation; the epilogue multiplies by the operands' inverse power-of-two scales.  precision 4 ("f16"):
//   hi*hi only.  precision 1 / 2: kind::tf32 single pass / 3xTF32 (activations split in shared memory by the
//   transform warps, "a_inkernel").
// * warp roles: warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer - both run their loops with all 32 lanes
//   converged and predicate the TMA / tcgen05 instructions with elect.sync (see elect_one) -, warps 2..9 = epilogue
//   in two groups of four on alternate 32-column slabs (TMEM lane quarter = warp_idx % 4); in the 3xTF32 mode
//   warps 6..9 are the operand transform instead.  mbarrier full/empty ring.
// * epilogue: TMEM -> registers -> scale / bias -> 128B-swizzled staging slab -> TMA store (or TMA reduce-add when the
//   launch accumulates into its output); BatchNorm statistics by a column walk over the staged slab, accumulated per
//   CTA across tiles, combined across the four warps of a group, one fp64 atomic pair per channel and CTA.
// * three kernels share this scheme: conv_tc_persist_kernel (one CTA per SM walks over tiles), conv_tc_pair_kernel
//   (cta_group::2: a CTA pair computes 256 pixels x BN per step, each CTA stages half of the weight tile; selected per
//   shape, see conv_tc_launch_core) and conv_tc_kernel (one tile per CTA, single-pass TF32 multi-tap layers only).
// * launched with programmatic stream serialization: everything before PXL_PDL_SYNC() overlaps the previous kernel.
//
// Every mbarrier wait has a watchdog: on expiry the kernel raises a device-side flag and bails
// out, so a protocol bug can never hang the GPU.
#include "common.cuh"
#include <cuda.h>
#include <cstdlib>

// ------------------------------------------------------------------------------------------
// driver entry point for tensor-map encoding (no link-time dependency on libcuda)
// ------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

// NHWC fp32 tensor viewed as (C, W, H, N), box {32, bw, bh, 1}, 128-byte swizzle, zero OOB fill
// estride = traversal stride of the W/H dims (2 for stride-2 convolutions: the box spans 2x the pixels
// and the TMA unit picks every 2nd one)
// f16: the tensor holds __half (one half of an fp16 pair, see h16_prep.cu); a 128-byte row is then 64 channels
static int make_act_map(CUtensorMap* m, const void* base, int C, int W, int H, int N, int bw, int bh, int estride = 1, int f16 = 0) {
    EncodeTiledFn enc = get_encode();
    if (!enc) return PXL_ERR_UNSUPPORTED;
    const cuuint64_t eb = f16 ? 2 : 4;
    cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
    cuuint64_t strides[3] = {(cuuint64_t)C * eb, (cuuint64_t)W * C * eb, (cuuint64_t)H * W * C * eb};
    cuuint32_t box[4] = {(cuuint32_t)(f16 ? 64 : 32), (cuuint32_t)(bw * estride), (cuuint32_t)(bh * estride), 1};
    cuuint32_t es[4] = {1, (cuuint32_t)estride, (cuuint32_t)estride, 1};
    if (box[1] > 256 || box[2] > 256) return PXL_ERR_UNSUPPORTED;
    CUresult r = enc(m, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void*)base, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : PXL_ERR_BAD_ARG;
}

// NHWC fp32 output viewed as (Cout, W, H, N) with pixel stride ldo: box {32, bw, bh, 1}, 128-byte swizzle.
// Used by the epilogue's TMA store: channels >= Cout and pixels outside the image are clipped by the TMA unit.
static int make_out_map(CUtensorMap* m, const float* base, int Cout, int ldo, int W, int H, int N, int bw, int bh) {
    EncodeTiledFn enc = get_encode();
    if (!enc) return PXL_ERR_UNSUPPORTED;
    cuuint64_t dims[4] = {(cuuint64_t)Cout, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
    cuuint64_t strides[3] = {(cuuint64_t)ldo * 4, (cuuint64_t)W * ldo * 4, (cuuint64_t)H * W * ldo * 4};
    cuuint32_t box[4] = {32, (cuuint32_t)bw, (cuuint32_t)bh, 1};
    cuuint32_t es[4] = {1, 1, 1, 1};
    if (box[1] > 256 || box[2] > 256) return PXL_ERR_UNSUPPORTED;
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void*)base, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : PXL_ERR_BAD_ARG;
}

// weights [rows][K] fp32, box {32, bn}
static int make_w_map(CUtensorMap* m, const void* base, int64_t K, int rows, int bn, int f16 = 0) {
    EncodeTiledFn enc = get_encode();
    if (!enc) return PXL_ERR_UNSUPPORTED;
    cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)K * (f16 ? 2 : 4)};
    cuuint32_t box[2] = {(cuuint32_t)(f16 ? 64 : 32), (cuuint32_t)bn};
    cuuint32_t es[2] = {1, 1};
    CUresult r = enc(m, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : PXL_ERR_BAD_ARG;
}

// ------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ bool mbar_try_wait_cluster(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ bool mbar_wait_cluster(uint64_t* bar, uint32_t parity, int* flag, int code) {
    for (uint32_t spin = 0; spin < (1u << 22); ++spin) {
        if (mbar_try_wait_cluster(bar, parity)) return true;
        if ((spin & 1023u) == 1023u && *(volatile int*)flag != 0) return false;
    }
    atomicCAS(flag, 0, code);
    return false;
}
// bounded wait: returns false (and raises *flag) if the barrier never completes
__device__ __forceinline__ bool mbar_wait(uint64_t* bar, uint32_t parity, int* flag, int code) {
    for (uint32_t spin = 0; spin < (1u << 22); ++spin) {
        if (mbar_try_wait(bar, parity)) return true;
        if ((spin & 1023u) == 1023u && *(volatile int*)flag != 0) return false;   // another CTA already failed
    }
    atomicCAS(flag, 0, code);
    return false;
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_store_4d(const void* src, const CUtensorMap* map, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
        ::"l"(map), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
// out[box] += shared[box] (fp32): lets a dgrad launch add its result into a tensor that already holds another
// gradient (the residual branch of a bottleneck), instead of a separate elementwise add over both tensors
__device__ __forceinline__ void tma_reduce_add_4d(const void* src, const CUtensorMap* map, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.reduce.async.bulk.tensor.4d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
        ::"l"(map), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_store_commit_and_wait_read() {
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// one K step (32 bytes of K per operand row: 8 tf32 or 16 fp16 values) of the selected kind
__device__ __forceinline__ void umma_any(int f16, uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    if (f16) umma_f16(tmem_d, adesc, bdesc, idesc, accumulate);
    else umma_tf32(tmem_d, adesc, bdesc, idesc, accumulate);
}
// One lane of a converged warp (deterministic for a given member mask).  The producer and MMA warps run their loops
// with all 32 lanes in uniform control flow and predicate only the TMA / tcgen05 instructions with this: addresses
// and descriptors then live in uniform registers.  A loop entered by `if (lane == 0)` instead costs ~40 SASS
// instructions per tcgen05.mma (VOTEU / ELECT / R2UR per operand plus integer divisions for the ring indices) and
// the issuing thread, not the tensor pipe, bounds the kernel (ncu source view, profiles/r02_ncu_l1.conv2_*).
__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile(
        "{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\t"
        "elect.sync rx|px, 0xffffffff;\n\t"
        "@px mov.s32 %0, 1;\n\t}"
        : "+r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// the MMAs of one 128-byte K slice of a stage (4 steps of 32 bytes; hi*hi + lo*hi + hi*lo when the operands are split)
template <int F16>
__device__ __forceinline__ void umma_slice(uint32_t acc, uint64_t da, uint64_t db, uint64_t dal, uint64_t dbl,
                                           uint32_t idesc, uint32_t acc0, bool split3) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (F16) umma_f16(acc, da + 2 * k, db + 2 * k, idesc, k ? 1u : acc0);
        else umma_tf32(acc, da + 2 * k, db + 2 * k, idesc, k ? 1u : acc0);
    }
    if (split3) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (F16) umma_f16(acc, dal + 2 * k, db + 2 * k, idesc, 1u);
            else umma_tf32(acc, dal + 2 * k, db + 2 * k, idesc, 1u);
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (F16) umma_f16(acc, da + 2 * k, dbl + 2 * k, idesc, 1u);
            else umma_tf32(acc, da + 2 * k, dbl + 2 * k, idesc, 1u);
        }
    }
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
        "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor):
//   start address >> 4 | LBO (unused for swizzled K-major, =1) << 16 | SBO = 1024 B (8 rows x 128 B) >> 4 << 32
//   | version 1 << 46 | layout SWIZZLE_128B (2) << 61
__device__ __forceinline__ uint64_t kmajor_sw128_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// kind::tf32 instruction descriptor (cute::UMMA::InstrDescriptor): D fp32, A/B tf32, both K-major, M=128, N
__device__ __forceinline__ uint32_t tf32_idesc(int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}
// kind::f16 with fp16 operands (a_format = b_format = 0), D fp32, K-major, M = 128, N
__device__ __forceinline__ uint32_t f16_idesc(int N) {
    return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}

// ------------------------------------------------------------------------------------------
struct TcParams {
    int Cin, Cout, ldo, ntaps, kchunks;
    int N, OH, OW;
    int BW, BH, tilesW, tilesH;
    int BN, stages, nsplit;
    int nacc;       // TMEM accumulators used round-robin over k-iterations (summed with RN adds in the epilogue)
    int a_inkernel; // 3xTF32 only: A arrives as raw fp32 and is split hi/lo in shared memory by the epilogue warps
    int in_mul;     // input pixel = output pixel * in_mul + tap (stride-2 forward uses the TMA traversal stride)
    int out_mul, out_offy, out_offx, outH, outW;   // output pixel (oy,ox) is stored at (oy*out_mul+offy, ox*out_mul+offx)
    int ntilesN, total_tiles;   // persistent kernel: N tiles per pixel tile, tiles in total
    int tma_store;  // epilogue stages 32-channel slabs in the (drained) operand ring and writes them with TMA
    int f16;        // operands are fp16 (kind::f16); nsplit == 3 then means the fp16 pair hi/lo of both operands
    int kc;         // K elements per 128-byte operand row: 32 (tf32) or 64 (fp16)
    float out_scale;   // the accumulator is multiplied by this (and by *oscale_ptr) before bias / statistics / store
    int out_acc;       // TMA-store epilogue adds into `out` (cp.reduce.async.bulk .add) instead of overwriting it
    int stats_smem;    // BN statistics: column walk over the staged slab instead of the register butterfly
    short dy[PXL_MAX_TAPS], dx[PXL_MAX_TAPS], widx[PXL_MAX_TAPS];
};

#define TC_A_BYTES (128 * 128)          // 128 rows x 128 B

__global__ void __launch_bounds__(192, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapAlo,
               const __grid_constant__ CUtensorMap mapB, const __grid_constant__ CUtensorMap mapBlo,
               const __grid_constant__ CUtensorMap mapOut,
               const TcParams p, const float* __restrict__ bias, float* __restrict__ out, double* __restrict__ stats,
               int* __restrict__ err_flag, const float* __restrict__ oscale_ptr) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ uint64_t full_bar[8], empty_bar[8], ready_bar[8], acc_bar;
    __shared__ uint32_t tmem_base_slot;

    // 1024-byte aligned operand ring
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const int b_bytes = p.BN * 128;
    const int per_op = TC_A_BYTES + b_bytes;                 // A + B of one precision part
    const int stage_bytes = per_op * (p.nsplit == 3 ? 2 : 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tile = blockIdx.x;
    const int tw = tile % p.tilesW, th = (tile / p.tilesW) % p.tilesH, n = tile / (p.tilesW * p.tilesH);
    const int w0 = tw * p.BW, h0 = th * p.BH;
    const int n0 = blockIdx.y * p.BN;
    const int iters = p.ntaps * p.kchunks;
    // The tensor core's fp32 accumulator truncates instead of rounding to nearest (measured: error
    // grows ~5e-9 * K), so long reductions are spread over `nacc` independent TMEM accumulators.
    const uint32_t acc_cols = p.BN < 32 ? 32 : p.BN;           // BN in {32,64,128,256}
    const uint32_t tmem_cols = acc_cols * p.nacc;              // power of two, <= 512

    if (threadIdx.x == 0) {
        for (int s = 0; s < p.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); mbar_init(&ready_bar[s], 128); }
        mbar_init(&acc_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(&tmem_base_slot, tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_d = tmem_base_slot;
    PXL_PDL_SYNC();          // everything above overlapped the previous kernel's tail; global memory from here on

    if (warp == 0) {
        // ================= TMA producer (whole warp converged, TMA under elect.sync) =================
        // bytes the TMA unit will deliver per stage: full boxes, OOB parts are zero-filled but counted
        uint32_t tx = (uint32_t)((p.BW * p.BH * 128 + b_bytes) * (p.nsplit == 3 ? 2 : 1));
        if (p.a_inkernel) tx -= (uint32_t)(p.BW * p.BH * 128);      // no A_lo box: it is produced in shared memory
        uint32_t s = 0, ph = 0;
        int tap = 0, c0 = 0;
        for (int it = 0; it < iters; ++it) {
            if (!__all_sync(0xffffffffu, mbar_wait(&empty_bar[s], ph ^ 1u, err_flag, 1))) break;
            uint8_t* sa = smem + (size_t)s * stage_bytes;
            const int ax = w0 * p.in_mul + p.dx[tap], ay = h0 * p.in_mul + p.dy[tap];
            const int bk = p.widx[tap] * p.Cin + c0;
            if (elect_one()) {
                mbar_expect_tx(&full_bar[s], tx);
                tma_load_4d(sa, &mapA, &full_bar[s], c0, ax, ay, n);
                tma_load_2d(sa + TC_A_BYTES, &mapB, &full_bar[s], bk, n0);
                if (p.nsplit == 3) {
                    if (!p.a_inkernel) tma_load_4d(sa + per_op, &mapAlo, &full_bar[s], c0, ax, ay, n);
                    tma_load_2d(sa + per_op + TC_A_BYTES, &mapBlo, &full_bar[s], bk, n0);
                }
            }
            __syncwarp();
            c0 += p.kc; if (c0 >= p.Cin) { c0 = 0; ++tap; }
            if (++s == (uint32_t)p.stages) { s = 0; ph ^= 1u; }
        }
    } else if (warp == 1) {
        // ================= MMA issuer (whole warp converged, tcgen05 under elect.sync) =================
        const uint32_t idesc = p.f16 ? f16_idesc(p.BN) : tf32_idesc(p.BN);
        const uint32_t smem_base = smem_u32(smem);
        uint32_t s = 0, ph = 0, a = 0;
        for (int it = 0; it < iters; ++it) {
            if (!__all_sync(0xffffffffu, mbar_wait(p.a_inkernel ? &ready_bar[s] : &full_bar[s], ph, err_flag, 2))) break;
            tc_fence_after();
            const uint32_t sa = smem_base + s * (uint32_t)stage_bytes;
            const uint64_t da = kmajor_sw128_desc(sa), db = kmajor_sw128_desc(sa + TC_A_BYTES);
            const uint64_t dal = kmajor_sw128_desc(sa + per_op), dbl = kmajor_sw128_desc(sa + per_op + TC_A_BYTES);
            const uint32_t acc = tmem_d + a * acc_cols;
            const uint32_t acc0 = it >= p.nacc ? 1u : 0u;
            if (elect_one()) {
                if (p.f16) umma_slice<1>(acc, da, db, dal, dbl, idesc, acc0, p.nsplit == 3);
                else umma_slice<0>(acc, da, db, dal, dbl, idesc, acc0, p.nsplit == 3);
                umma_commit(&empty_bar[s]);      // frees the smem slot once these MMAs have read it
                if (it == iters - 1) umma_commit(&acc_bar);       // accumulator complete -> epilogue
            }
            __syncwarp();
            if (++s == (uint32_t)p.stages) { s = 0; ph ^= 1u; }
            if (++a == (uint32_t)p.nacc) a = 0;
        }
    } else {
        // ================= epilogue: TMEM -> registers -> global (NHWC rows) =================
        const int q = warp & 3;                  // TMEM lane quarter this warp may access
        const int r = q * 32 + lane;             // tile row = output pixel within the spatial tile
        if (p.a_inkernel) {
            // ---- operand transform: raw fp32 A tile -> (hi in place, lo) ; elementwise, so the TMA
            // swizzle is preserved.  Thread t owns the 16-byte chunks t, t+128, ... (conflict-free).
            const int t = threadIdx.x - 64;
            bool okt = true;
            for (int it = 0; it < iters && okt; ++it) {
                const int s = it % p.stages;
                const uint32_t ph = (uint32_t)(it / p.stages) & 1u;
                okt = mbar_wait(&full_bar[s], ph, err_flag, 4);
                if (!okt) break;
                float4* a_hi = reinterpret_cast<float4*>(smem + (size_t)s * stage_bytes);
                float4* a_lo = reinterpret_cast<float4*>(smem + (size_t)s * stage_bytes + per_op);
#pragma unroll
                for (int c = 0; c < TC_A_BYTES / 16 / 128; ++c) {
                    const float4 v = a_hi[t + c * 128];
                    float4 h, l;
                    const float* vp = &v.x; float* hp = &h.x; float* lp = &l.x;
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        uint32_t u;
                        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(vp[e]));
                        u &= 0xFFFFE000u;
                        hp[e] = __uint_as_float(u);
                        lp[e] = vp[e] - hp[e];
                    }
                    a_hi[t + c * 128] = h;
                    a_lo[t + c * 128] = l;
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to UMMA
                asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&ready_bar[s])) : "memory");
            }
        }
        const bool ok = __all_sync(0xffffffffu, mbar_wait(&acc_bar, 0, err_flag, 3));
        tc_fence_after();
        if (ok) {
            const int hy = r / p.BW, wx = r - hy * p.BW;
            const int oy = h0 + hy, ox = w0 + wx;
            const bool valid = hy < p.BH && oy < p.OH && ox < p.OW;
            float* orow = out + ((int64_t)(n * p.outH + oy * p.out_mul + p.out_offy) * p.outW + ox * p.out_mul + p.out_offx) * p.ldo;
            const int used = iters < p.nacc ? iters : p.nacc;
            const float osc = p.out_scale * (oscale_ptr ? __ldg(oscale_ptr) : 1.f);
            for (int j = 0; j < p.BN; j += 32) {
                float v[32];
                tmem_ld32(tmem_d + ((uint32_t)(q * 32) << 16) + (uint32_t)j, v);   // warp-collective
                for (int a = 1; a < used; ++a) {
                    float u[32];
                    tmem_ld32(tmem_d + ((uint32_t)(q * 32) << 16) + (uint32_t)a * acc_cols + (uint32_t)j, u);
#pragma unroll
                    for (int c = 0; c < 32; ++c) v[c] += u[c];
                }
                if (osc != 1.f) {
#pragma unroll
                    for (int c = 0; c < 32; ++c) v[c] *= osc;
                }
                const int cb = n0 + j;
                if (stats) {
                    // per-channel sum / sum of squares of this tile for the BatchNorm that follows
                    // (sync_batchnorm/batchnorm.py:60-62): warp transpose-reduce over the 32 rows, then one
                    // fp64 atomic per channel and warp.  Rows outside the image contribute nothing.
                    float sv[32], sq[32];
#pragma unroll
                    for (int c = 0; c < 32; ++c) {
                        const float o = valid ? v[c] + ((bias && cb + c < p.Cout) ? __ldg(bias + cb + c) : 0.f) : 0.f;
                        sv[c] = o; sq[c] = o * o;
                    }
#pragma unroll
                    for (int off = 16; off >= 1; off >>= 1) {
                        const bool up = (lane & off) != 0;
#pragma unroll
                        for (int i = 0; i < off; ++i) {
                            const float s_send = up ? sv[i] : sv[i + off], q_send = up ? sq[i] : sq[i + off];
                            const float s_recv = __shfl_xor_sync(0xffffffffu, s_send, off);
                            const float q_recv = __shfl_xor_sync(0xffffffffu, q_send, off);
                            sv[i] = (up ? sv[i + off] : sv[i]) + s_recv;
                            sq[i] = (up ? sq[i + off] : sq[i]) + q_recv;
                        }
                    }
                    if (cb + lane < p.Cout) {
                        atomicAdd(stats + cb + lane, (double)sv[0]);
                        atomicAdd(stats + p.Cout + cb + lane, (double)sq[0]);
                    }
                }
                if (p.tma_store) {
                    // stage this warp's 32 rows of the slab in the drained operand ring (canonical 128B-swizzled
                    // rows: conflict-free float4 writes), TMA-store the whole 128-row slab once all four warps
                    // are done.  The ring holds `fit` slabs; a round = up to `fit` consecutive slabs.
                    const int fit = (p.stages * stage_bytes) / TC_A_BYTES;
                    const int slab = (j >> 5) % fit;
                    float4* dst = reinterpret_cast<float4*>(smem + (size_t)slab * TC_A_BYTES + (size_t)r * 128);
                    if (cb < p.Cout) {
#pragma unroll
                        for (int c = 0; c < 8; ++c) {
                            float4 o = make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
                            if (bias) {
                                const int cc = cb + 4 * c;
                                if (cc < p.Cout) o.x += __ldg(bias + cc);
                                if (cc + 1 < p.Cout) o.y += __ldg(bias + cc + 1);
                                if (cc + 2 < p.Cout) o.z += __ldg(bias + cc + 2);
                                if (cc + 3 < p.Cout) o.w += __ldg(bias + cc + 3);
                            }
                            dst[c ^ (r & 7)] = o;
                        }
                    }
                    const bool round_end = (slab == fit - 1) || (j + 32 >= p.BN);
                    if (round_end) {
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        asm volatile("bar.sync 1, 128;" ::: "memory");
                        if (threadIdx.x == 64) {
                            const int first = j - slab * 32;          // first column of this round
                            for (int jj = 0; jj <= slab; ++jj) {
                                const int cs = n0 + first + jj * 32;
                                if (cs < p.Cout)
                                    tma_store_4d(smem + (size_t)jj * TC_A_BYTES, &mapOut, cs, w0, h0, n);
                            }
                            tma_store_commit_and_wait_read();
                        }
                        if (j + 32 < p.BN) asm volatile("bar.sync 1, 128;" ::: "memory");   // ring reusable
                    }
                    continue;
                }
                if (!valid) continue;
                if (cb + 31 < p.Cout && (p.ldo & 3) == 0) {
#pragma unroll
                    for (int c = 0; c < 32; c += 4) {
                        float4 o = make_float4(v[c], v[c + 1], v[c + 2], v[c + 3]);
                        if (bias) { o.x += __ldg(bias + cb + c); o.y += __ldg(bias + cb + c + 1); o.z += __ldg(bias + cb + c + 2); o.w += __ldg(bias + cb + c + 3); }
                        *reinterpret_cast<float4*>(orow + cb + c) = o;
                    }
                } else {
#pragma unroll
                    for (int c = 0; c < 32; ++c)
                        if (cb + c < p.Cout) orow[cb + c] = v[c] + (bias ? __ldg(bias + cb + c) : 0.f);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_d, tmem_cols);
}


// ------------------------------------------------------------------------------------------
// Persistent variant: one CTA per SM walks over output tiles (static stride).  The operand ring keeps
// streaming across tile boundaries, the accumulator is double-buffered in TMEM (set = tile & 1) and the
// epilogue of tile t (TMEM -> registers -> swizzled staging slab -> TMA store) overlaps the main loop of
// tile t+1.  Warp roles: 0 TMA producer, 1 MMA issuer (+TMEM allocator), 2..5 epilogue, 6..9 operand
// transform (3xTF32 with raw activations only: hi/lo split of the A tile in shared memory).
// ------------------------------------------------------------------------------------------
#define TC_STG_SLABS 2

__device__ __forceinline__ void tc_tile_coords(const TcParams& p, int tile, int& n0, int& w0, int& h0, int& n) {
    const int nt = tile % p.ntilesN, pix = tile / p.ntilesN;
    const int tw = pix % p.tilesW, th = (pix / p.tilesW) % p.tilesH;
    n = pix / (p.tilesW * p.tilesH);
    w0 = tw * p.BW; h0 = th * p.BH; n0 = nt * p.BN;
}

__global__ void __launch_bounds__(320, 1)
conv_tc_persist_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapAlo,
                       const __grid_constant__ CUtensorMap mapB, const __grid_constant__ CUtensorMap mapBlo,
                       const __grid_constant__ CUtensorMap mapOut,
                       const TcParams p, const float* __restrict__ bias, float* __restrict__ out,
                       double* __restrict__ stats, int* __restrict__ err_flag, const float* __restrict__ oscale_ptr) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ uint64_t full_bar[8], empty_bar[8], ready_bar[8], acc_full[2], acc_empty[2];
    __shared__ uint32_t tmem_base_slot;

    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const int b_bytes = p.BN * 128;
    const int per_op = TC_A_BYTES + b_bytes;
    const int stage_bytes = per_op * (p.nsplit == 3 ? 2 : 1);
    uint8_t* staging = smem + (size_t)p.stages * stage_bytes;        // TC_STG_SLABS x 16 KB, 1024-aligned

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int iters = p.ntaps * p.kchunks;
    const uint32_t acc_cols = p.BN < 32 ? 32 : p.BN;
    const uint32_t set_cols = acc_cols * p.nacc;
    const uint32_t tmem_cols = 512;

    if (threadIdx.x == 0) {
        for (int s = 0; s < p.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); mbar_init(&ready_bar[s], 128); }
        for (int a = 0; a < 2; ++a) { mbar_init(&acc_full[a], 1); mbar_init(&acc_empty[a], 128 * (p.a_inkernel ? 1 : 2)); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(&tmem_base_slot, tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_d = tmem_base_slot;
    PXL_PDL_SYNC();          // everything above overlapped the previous kernel's tail; global memory from here on

    if (warp == 0) {
        // ================= TMA producer (whole warp converged, TMA under elect.sync) =================
        uint32_t tx = (uint32_t)((p.BW * p.BH * 128 + b_bytes) * (p.nsplit == 3 ? 2 : 1));
        if (p.a_inkernel) tx -= (uint32_t)(p.BW * p.BH * 128);
        uint32_t s = 0, ph = 0;
        bool ok = true;
        for (int tile = blockIdx.x; tile < p.total_tiles && ok; tile += gridDim.x) {
            int n0, w0, h0, n;
            tc_tile_coords(p, tile, n0, w0, h0, n);
            int tap = 0, c0 = 0;
            for (int it = 0; it < iters; ++it) {
                ok = __all_sync(0xffffffffu, mbar_wait(&empty_bar[s], ph ^ 1u, err_flag, 1));
                if (!ok) break;
                uint8_t* sa = smem + (size_t)s * stage_bytes;
                const int ax = w0 * p.in_mul + p.dx[tap], ay = h0 * p.in_mul + p.dy[tap];
                const int bk = p.widx[tap] * p.Cin + c0;
                if (elect_one()) {
                    mbar_expect_tx(&full_bar[s], tx);
                    tma_load_4d(sa, &mapA, &full_bar[s], c0, ax, ay, n);
                    tma_load_2d(sa + TC_A_BYTES, &mapB, &full_bar[s], bk, n0);
                    if (p.nsplit == 3) {
                        if (!p.a_inkernel) tma_load_4d(sa + per_op, &mapAlo, &full_bar[s], c0, ax, ay, n);
                        tma_load_2d(sa + per_op + TC_A_BYTES, &mapBlo, &full_bar[s], bk, n0);
                    }
                }
                __syncwarp();
                c0 += p.kc; if (c0 >= p.Cin) { c0 = 0; ++tap; }
                if (++s == (uint32_t)p.stages) { s = 0; ph ^= 1u; }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer (whole warp converged, tcgen05 under elect.sync) =================
        const uint32_t idesc = p.f16 ? f16_idesc(p.BN) : tf32_idesc(p.BN);
        const uint32_t smem_base = smem_u32(smem);
        uint32_t s = 0, ph = 0, tcount = 0;
        bool ok = true;
        for (int tile = blockIdx.x; tile < p.total_tiles && ok; tile += gridDim.x, ++tcount) {
            const uint32_t set = tcount & 1u, aph = (tcount >> 1) & 1u;
            ok = __all_sync(0xffffffffu, mbar_wait(&acc_empty[set], aph ^ 1u, err_flag, 5));       // epilogue drained this set
            if (!ok) break;
            tc_fence_after();
            const uint32_t set_base = tmem_d + set * set_cols;
            uint32_t a = 0;
            for (int it = 0; it < iters; ++it) {
                ok = __all_sync(0xffffffffu, mbar_wait(p.a_inkernel ? &ready_bar[s] : &full_bar[s], ph, err_flag, 2));
                if (!ok) break;
                tc_fence_after();
                const uint32_t sa = smem_base + s * (uint32_t)stage_bytes;
                const uint64_t da = kmajor_sw128_desc(sa), db = kmajor_sw128_desc(sa + TC_A_BYTES);
                const uint64_t dal = kmajor_sw128_desc(sa + per_op), dbl = kmajor_sw128_desc(sa + per_op + TC_A_BYTES);
                const uint32_t acc = set_base + a * acc_cols;
                const uint32_t acc0 = it >= p.nacc ? 1u : 0u;
                if (elect_one()) {
                    if (p.f16) umma_slice<1>(acc, da, db, dal, dbl, idesc, acc0, p.nsplit == 3);
                    else umma_slice<0>(acc, da, db, dal, dbl, idesc, acc0, p.nsplit == 3);
                    umma_commit(&empty_bar[s]);
                    if (it == iters - 1) umma_commit(&acc_full[set]);
                }
                __syncwarp();
                if (++s == (uint32_t)p.stages) { s = 0; ph ^= 1u; }
                if (++a == (uint32_t)p.nacc) a = 0;
            }
        }
    } else if (warp < 6 || !p.a_inkernel) {
        // ================= epilogue =================
        // Without an operand transform (every mode but 3xTF32 on raw activations) warps 6..9 form a second epilogue
        // group: the two groups take alternate 32-column slabs of the tile (TMEM lane quarter = warp % 4 either
        // way), each with its own staging slab and named barrier.
        const int grp = warp >= 6 ? 1 : 0;
        const int ngrp = p.a_inkernel ? 1 : 2;
        const int q = warp & 3;
        const int r = q * 32 + lane;
        const int et = threadIdx.x - 64 - 128 * grp;     // 0..127 within the group
        const int barid = 1 + grp;
        uint32_t tcount = 0, sc = 0;
        const float osc = p.out_scale * (oscale_ptr ? __ldg(oscale_ptr) : 1.f);
        // BatchNorm statistics are accumulated per lane across the tiles this CTA processes for one channel block
        // and flushed with ONE pair of fp64 atomics per channel when the channel block changes / at the end: the
        // stem and layer1 convolutions run ~50 tiles per CTA onto 64..256 channels, and per-tile atomics serialise on
        // those few addresses (33 K atomics per address for the stem).  fp32 partials over <= a few thousand rows.
        float st_s0 = 0.f, st_s1 = 0.f, st_s2 = 0.f, st_s3 = 0.f, st_q0 = 0.f, st_q1 = 0.f, st_q2 = 0.f, st_q3 = 0.f;
        int st_n0 = -1;
        auto flush_stats = [&]() {
            if (stats && st_n0 >= 0) {
                // the four warps of a group hold the four row quarters of the same channels: combine them through the
                // group's (idle) staging slab so that ONE thread per channel issues the fp64 atomics - a single-wave
                // layer-3 launch otherwise sends 548 atomics to each of 512 addresses at the same moment (+8 us)
                float* scratch = reinterpret_cast<float*>(staging + (size_t)(ngrp == 1 ? 0 : grp) * TC_A_BYTES);
                if (et == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                asm volatile("bar.sync %0, 128;" ::"r"(barid) : "memory");
                scratch[0 * 128 + r] = st_s0; scratch[1 * 128 + r] = st_q0;
                scratch[2 * 128 + r] = st_s1; scratch[3 * 128 + r] = st_q1;
                scratch[4 * 128 + r] = st_s2; scratch[5 * 128 + r] = st_q2;
                scratch[6 * 128 + r] = st_s3; scratch[7 * 128 + r] = st_q3;
                asm volatile("bar.sync %0, 128;" ::"r"(barid) : "memory");
                const int slab = grp + q * ngrp;              // warp q of the group reduces accumulator slot si = q
                const int cbf = st_n0 + 32 * slab + lane;
                if (32 * slab < p.BN && cbf < p.Cout) {
                    const float* ps = scratch + (2 * q) * 128 + lane;
                    const float sv = (ps[0] + ps[32]) + (ps[64] + ps[96]);
                    const float qv = (ps[128] + ps[160]) + (ps[192] + ps[224]);
                    if (sv != 0.f || qv != 0.f) {
                        atomicAdd(stats + cbf, (double)sv);
                        atomicAdd(stats + p.Cout + cbf, (double)qv);
                    }
                }
            }
            st_s0 = st_s1 = st_s2 = st_s3 = st_q0 = st_q1 = st_q2 = st_q3 = 0.f;
        };
        bool ok = true;
        for (int tile = blockIdx.x; tile < p.total_tiles && ok; tile += gridDim.x, ++tcount) {
            const uint32_t set = tcount & 1u, aph = (tcount >> 1) & 1u;
            ok = __all_sync(0xffffffffu, mbar_wait(&acc_full[set], aph, err_flag, 3));
            if (!ok) break;
            tc_fence_after();
            int n0, w0, h0, n;
            tc_tile_coords(p, tile, n0, w0, h0, n);
            if (n0 != st_n0) { flush_stats(); st_n0 = n0; }
            const int hy = r / p.BW, wx = r - hy * p.BW;
            const int oy = h0 + hy, ox = w0 + wx;
            const bool valid = hy < p.BH && oy < p.OH && ox < p.OW;
            float* orow = out + ((int64_t)(n * p.outH + oy * p.out_mul + p.out_offy) * p.outW + ox * p.out_mul + p.out_offx) * p.ldo;
            const int used = iters < p.nacc ? iters : p.nacc;
            const uint32_t tbase = tmem_d + set * set_cols + ((uint32_t)(q * 32) << 16);
            for (int j = 32 * grp; j < p.BN; j += 32 * ngrp) {
                const int cb = n0 + j;
                if (cb >= p.Cout) break;                  // uniform: nothing left to store for this tile
                float v[32];
                tmem_ld32(tbase + (uint32_t)j, v);
                for (int a = 1; a < used; ++a) {
                    float u[32];
                    tmem_ld32(tbase + (uint32_t)a * acc_cols + (uint32_t)j, u);
#pragma unroll
                    for (int c = 0; c < 32; ++c) v[c] += u[c];
                }
                if (osc != 1.f) {
#pragma unroll
                    for (int c = 0; c < 32; ++c) v[c] *= osc;
                }
                if (bias) {
#pragma unroll
                    for (int c = 0; c < 32; ++c) if (cb + c < p.Cout) v[c] += __ldg(bias + cb + c);
                }
                const bool walk = stats && p.stats_smem && p.tma_store;
                float col_s = 0.f, col_q = 0.f;              // this lane's column over this warp's 32 rows
                if (stats && !walk) {
                    float sv[32], sq[32];
#pragma unroll
                    for (int c = 0; c < 32; ++c) { const float o = valid ? v[c] : 0.f; sv[c] = o; sq[c] = o * o; }
#pragma unroll
                    for (int off = 16; off >= 1; off >>= 1) {
                        const bool up = (lane & off) != 0;
#pragma unroll
                        for (int i = 0; i < off; ++i) {
                            const float s_send = up ? sv[i] : sv[i + off], q_send = up ? sq[i] : sq[i + off];
                            const float s_recv = __shfl_xor_sync(0xffffffffu, s_send, off);
                            const float q_recv = __shfl_xor_sync(0xffffffffu, q_send, off);
                            sv[i] = (up ? sv[i + off] : sv[i]) + s_recv;
                            sq[i] = (up ? sq[i + off] : sq[i]) + q_recv;
                        }
                    }
                    col_s = sv[0]; col_q = sq[0];
                }
                if (walk && !valid) {                        // rows outside the image are clipped by the TMA store; zero them for the sums
#pragma unroll
                    for (int c = 0; c < 32; ++c) v[c] = 0.f;
                }
                if (p.tma_store) {
                    // one group: two staging slabs used alternately (slab b was last stored two slabs ago);
                    // two groups: one slab each, its previous TMA read must be over before it is rewritten
                    const uint32_t b = ngrp == 1 ? (sc & 1u) : (uint32_t)grp;
                    if (et == 0) {
                        if (ngrp == 1) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
                        else asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                    }
                    asm volatile("bar.sync %0, 128;" ::"r"(barid) : "memory");
                    float4* dst = reinterpret_cast<float4*>(staging + (size_t)b * TC_A_BYTES + (size_t)r * 128);
#pragma unroll
                    for (int c = 0; c < 8; ++c)
                        dst[c ^ (r & 7)] = make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    asm volatile("bar.sync %0, 128;" ::"r"(barid) : "memory");
                    if (et == 0) {
                        if (p.out_acc) tma_reduce_add_4d(staging + (size_t)b * TC_A_BYTES, &mapOut, cb, w0, h0, n);
                        else tma_store_4d(staging + (size_t)b * TC_A_BYTES, &mapOut, cb, w0, h0, n);
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    }
                    if (walk) {
                        // column `lane` of rows 32q .. 32q+31 of the staged slab: one 128-byte row per step, the 32 lanes
                        // read its 32 words (16-byte chunks XOR-swizzled by row & 7), conflict-free
                        const float* srow = reinterpret_cast<const float*>(staging + (size_t)b * TC_A_BYTES + (size_t)(q * 32) * 128);
                        const int cq = lane >> 2, cw = lane & 3;
#pragma unroll 8
                        for (int rr = 0; rr < 32; ++rr) {
                            const float o = srow[rr * 32 + (((cq ^ (rr & 7)) << 2) | cw)];
                            col_s += o; col_q = fmaf(o, o, col_q);
                        }
                    }
                    ++sc;
                } else if (valid) {
                    if (cb + 31 < p.Cout && (p.ldo & 3) == 0) {
#pragma unroll
                        for (int c = 0; c < 32; c += 4)
                            *reinterpret_cast<float4*>(orow + cb + c) = make_float4(v[c], v[c + 1], v[c + 2], v[c + 3]);
                    } else {
#pragma unroll
                        for (int c = 0; c < 32; ++c)
                            if (cb + c < p.Cout) orow[cb + c] = v[c];
                    }
                }
                if (stats) {
                    const int si = (j / 32 - grp) / ngrp;
                    if (si < 4) {
                        switch (si) {
                            case 0: st_s0 += col_s; st_q0 += col_q; break;
                            case 1: st_s1 += col_s; st_q1 += col_q; break;
                            case 2: st_s2 += col_s; st_q2 += col_q; break;
                            default: st_s3 += col_s; st_q3 += col_q; break;
                        }
                    } else if (cb + lane < p.Cout) {          // BN = 256 with one epilogue group: slabs 4..7 go out per tile
                        atomicAdd(stats + cb + lane, (double)col_s);
                        atomicAdd(stats + p.Cout + cb + lane, (double)col_q);
                    }
                }
            }
            // this accumulator set may be overwritten by the MMA warp now
            tc_fence_before();
            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&acc_empty[set])) : "memory");
        }
        flush_stats();
        if (et == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    } else {
        // ================= operand transform (3xTF32, raw activations) =================
        if (p.a_inkernel) {
            const int t = threadIdx.x - 192;
            uint32_t gs = 0;
            bool okt = true;
            for (int tile = blockIdx.x; tile < p.total_tiles && okt; tile += gridDim.x) {
                for (int it = 0; it < iters; ++it, ++gs) {
                    const int s = gs % p.stages;
                    const uint32_t ph = (gs / p.stages) & 1u;
                    okt = mbar_wait(&full_bar[s], ph, err_flag, 4);
                    if (!okt) break;
                    float4* a_hi = reinterpret_cast<float4*>(smem + (size_t)s * stage_bytes);
                    float4* a_lo = reinterpret_cast<float4*>(smem + (size_t)s * stage_bytes + per_op);
#pragma unroll
                    for (int c = 0; c < TC_A_BYTES / 16 / 128; ++c) {
                        const float4 v = a_hi[t + c * 128];
                        float4 h, l;
                        const float* vp = &v.x; float* hp = &h.x; float* lp = &l.x;
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            uint32_t u;
                            asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(vp[e]));
                            u &= 0xFFFFE000u;
                            hp[e] = __uint_as_float(u);
                            lp[e] = vp[e] - hp[e];
                        }
                        a_hi[t + c * 128] = h;
                        a_lo[t + c * 128] = l;
                    }
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&ready_bar[s])) : "memory");
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_d, tmem_cols);
}


// ------------------------------------------------------------------------------------------
// CTA-pair variant (tcgen05 cta_group::2, cluster of two CTAs on one TPC): the pair computes a
// 256-pixel x BN tile per step.  Each CTA stages ITS 128 pixels of A and HALF of the B tile (BN/2 weight
// rows); one tcgen05.mma.cta_group::2 issued by the leader CTA reads A and B from both CTAs' shared memory
// and writes rows 0..127 into the leader's TMEM and rows 128..255 into the peer's.  Operand traffic per
// FLOP drops by a third compared with two independent 128 x BN tiles, and the shared-memory stage shrinks
// so the ring gets deeper.  Same persistent structure as conv_tc_persist_kernel.
//
// Barriers (identical shared-memory offsets in both CTAs):
//   full[s]   single-pass TF32: leader's only, count 1 + tx bytes of BOTH CTAs (2-SM TMA form signals the
//             leader's barrier).  3xTF32 in-kernel split: per CTA, local loads.
//   ready[s]  3xTF32: leader's only, count 256 = transform threads of both CTAs (peer arrives remotely)
//   empty[s]  per CTA, count 1, arrival = multicast tcgen05.commit of the leader's MMA thread
//   acc_full[2]  per CTA, count 1, multicast commit;   acc_empty[2]  leader's only, count 256 per epilogue group
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
    uint32_t r; asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank)); return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tma2_load_4d(void* dst, const CUtensorMap* map, uint32_t bar_cluster_addr, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma2_load_2d(void* dst, const CUtensorMap* map, uint32_t bar_cluster_addr, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma2_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma2_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma2_any(int f16, uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    if (f16) umma2_f16(tmem_d, adesc, bdesc, idesc, accumulate);
    else umma2_tf32(tmem_d, adesc, bdesc, idesc, accumulate);
}
template <int F16>
__device__ __forceinline__ void umma2_slice(uint32_t acc, uint64_t da, uint64_t db, uint64_t dal, uint64_t dbl,
                                            uint32_t idesc, uint32_t acc0, bool split3) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (F16) umma2_f16(acc, da + 2 * k, db + 2 * k, idesc, k ? 1u : acc0);
        else umma2_tf32(acc, da + 2 * k, db + 2 * k, idesc, k ? 1u : acc0);
    }
    if (split3) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (F16) umma2_f16(acc, dal + 2 * k, db + 2 * k, idesc, 1u);
            else umma2_tf32(acc, dal + 2 * k, db + 2 * k, idesc, 1u);
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (F16) umma2_f16(acc, da + 2 * k, dbl + 2 * k, idesc, 1u);
            else umma2_tf32(acc, da + 2 * k, dbl + 2 * k, idesc, 1u);
        }
    }
}
__device__ __forceinline__ void umma2_commit_mc(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}

__device__ __forceinline__ void tc_pair_coords(const TcParams& p, int work, uint32_t rank, int& n0, int& w0, int& h0, int& n) {
    const int nt = work % p.ntilesN, pix = 2 * (work / p.ntilesN) + (int)rank;
    const int tw = pix % p.tilesW, th = (pix / p.tilesW) % p.tilesH;
    n = pix / (p.tilesW * p.tilesH);                     // == p.N for the padding tile of an odd tile count
    w0 = tw * p.BW; h0 = th * p.BH; n0 = nt * p.BN;
}

__global__ void __launch_bounds__(320, 1)
conv_tc_pair_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapAlo,
                    const __grid_constant__ CUtensorMap mapB, const __grid_constant__ CUtensorMap mapBlo,
                    const __grid_constant__ CUtensorMap mapOut,
                    const TcParams p, const float* __restrict__ bias, float* __restrict__ out,
                    double* __restrict__ stats, int* __restrict__ err_flag, const float* __restrict__ oscale_ptr) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ uint64_t full_bar[8], empty_bar[8], ready_bar[8], acc_full[2], acc_empty[2];
    __shared__ uint32_t tmem_base_slot;

    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const int bh_rows = p.BN / 2;                         // weight rows staged by this CTA
    const int b_bytes = bh_rows * 128;
    const int per_op = TC_A_BYTES + b_bytes;
    const int stage_bytes = per_op * (p.nsplit == 3 ? 2 : 1);
    uint8_t* staging = smem + (size_t)p.stages * stage_bytes;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;
    const int iters = p.ntaps * p.kchunks;
    const uint32_t acc_cols = p.BN;
    const uint32_t set_cols = acc_cols * p.nacc;
    const uint32_t tmem_cols = 512;
    const int cid = blockIdx.x >> 1, nclusters = gridDim.x >> 1;

    if (threadIdx.x == 0) {
        for (int s = 0; s < p.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); mbar_init(&ready_bar[s], 256); }
        for (int a = 0; a < 2; ++a) { mbar_init(&acc_full[a], 1); mbar_init(&acc_empty[a], 256 * (p.a_inkernel ? 1 : 2)); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc2(&tmem_base_slot, tmem_cols);
    tc_fence_before();
    cluster_sync_all();                                   // peer barriers initialised, TMEM allocated in both CTAs
    tc_fence_after();
    const uint32_t tmem_d = tmem_base_slot;
    PXL_PDL_SYNC();          // everything above overlapped the previous kernel's tail; global memory from here on

    if (warp == 0) {
        // ================= TMA producer (both CTAs; whole warp converged, TMA under elect.sync) =================
        const uint32_t my_bytes = (uint32_t)((p.BW * p.BH * 128 + b_bytes) * (p.nsplit == 3 ? 2 : 1)) -
                                  (p.a_inkernel ? (uint32_t)(p.BW * p.BH * 128) : 0u);
        uint32_t s = 0, ph = 0;
        bool ok = true;
        for (int work = cid; work < p.total_tiles && ok; work += nclusters) {
            int n0, w0, h0, n;
            tc_pair_coords(p, work, rank, n0, w0, h0, n);
            const int brow = n0 + (int)rank * bh_rows;
            int tap = 0, c0 = 0;
            for (int it = 0; it < iters; ++it) {
                ok = __all_sync(0xffffffffu, mbar_wait(&empty_bar[s], ph ^ 1u, err_flag, 1));
                if (!ok) break;
                uint8_t* sa = smem + (size_t)s * stage_bytes;
                const int ax = w0 * p.in_mul + p.dx[tap], ay = h0 * p.in_mul + p.dy[tap];
                const int bk = p.widx[tap] * p.Cin + c0;
                const uint32_t fb = mapa_u32(smem_u32(&full_bar[s]), 0);
                if (elect_one()) {
                    if (p.a_inkernel) {
                        // local barrier: this CTA's transform warps wait for this CTA's bytes
                        mbar_expect_tx(&full_bar[s], my_bytes);
                        tma_load_4d(sa, &mapA, &full_bar[s], c0, ax, ay, n);
                        tma_load_2d(sa + TC_A_BYTES, &mapB, &full_bar[s], bk, brow);
                        tma_load_2d(sa + per_op + TC_A_BYTES, &mapBlo, &full_bar[s], bk, brow);
                    } else {
                        // the leader's barrier collects the bytes of both CTAs
                        if (leader) mbar_expect_tx(&full_bar[s], 2u * my_bytes);
                        tma2_load_4d(sa, &mapA, fb, c0, ax, ay, n);
                        tma2_load_2d(sa + TC_A_BYTES, &mapB, fb, bk, brow);
                        if (p.nsplit == 3) {
                            tma2_load_4d(sa + per_op, &mapAlo, fb, c0, ax, ay, n);
                            tma2_load_2d(sa + per_op + TC_A_BYTES, &mapBlo, fb, bk, brow);
                        }
                    }
                }
                __syncwarp();
                c0 += p.kc; if (c0 >= p.Cin) { c0 = 0; ++tap; }
                if (++s == (uint32_t)p.stages) { s = 0; ph ^= 1u; }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer (leader CTA; whole warp converged, tcgen05 under elect.sync) =================
        if (leader) {
            // M = 256 (bits 24..28 = M >> 4), N = BN
            const uint32_t idesc = (1u << 4) | (p.f16 ? 0u : ((2u << 7) | (2u << 10))) | ((uint32_t)(p.BN >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
            const uint32_t smem_base = smem_u32(smem);
            uint32_t s = 0, ph = 0, tcount = 0;
            bool ok = true;
            for (int work = cid; work < p.total_tiles && ok; work += nclusters, ++tcount) {
                const uint32_t set = tcount & 1u, aph = (tcount >> 1) & 1u;
                ok = __all_sync(0xffffffffu, mbar_wait_cluster(&acc_empty[set], aph ^ 1u, err_flag, 5));
                if (!ok) break;
                tc_fence_after();
                const uint32_t set_base = tmem_d + set * set_cols;
                uint32_t a = 0;
                for (int it = 0; it < iters; ++it) {
                    ok = __all_sync(0xffffffffu, mbar_wait_cluster(p.a_inkernel ? &ready_bar[s] : &full_bar[s], ph, err_flag, 2));
                    if (!ok) break;
                    tc_fence_after();
                    const uint32_t sa = smem_base + s * (uint32_t)stage_bytes;
                    const uint64_t da = kmajor_sw128_desc(sa), db = kmajor_sw128_desc(sa + TC_A_BYTES);
                    const uint64_t dal = kmajor_sw128_desc(sa + per_op), dbl = kmajor_sw128_desc(sa + per_op + TC_A_BYTES);
                    const uint32_t acc = set_base + a * acc_cols;
                    const uint32_t acc0 = it >= p.nacc ? 1u : 0u;
                    if (elect_one()) {
                        if (p.f16) umma2_slice<1>(acc, da, db, dal, dbl, idesc, acc0, p.nsplit == 3);
                        else umma2_slice<0>(acc, da, db, dal, dbl, idesc, acc0, p.nsplit == 3);
                        umma2_commit_mc(&empty_bar[s]);          // frees the slot in both CTAs
                        if (it == iters - 1) umma2_commit_mc(&acc_full[set]);
                    }
                    __syncwarp();
                    if (++s == (uint32_t)p.stages) { s = 0; ph ^= 1u; }
                    if (++a == (uint32_t)p.nacc) a = 0;
                }
            }
        }
    } else if (warp < 6 || !p.a_inkernel) {
        // ================= epilogue (both CTAs, own 128 rows; two 4-warp groups on alternate slabs like the
        // persistent kernel when there is no operand transform) =================
        const int grp = warp >= 6 ? 1 : 0;
        const int ngrp = p.a_inkernel ? 1 : 2;
        const int q = warp & 3;
        const int r = q * 32 + lane;
        const int et = threadIdx.x - 64 - 128 * grp;
        const int barid = 1 + grp;
        uint32_t tcount = 0, sc = 0;
        const float osc = p.out_scale * (oscale_ptr ? __ldg(oscale_ptr) : 1.f);
        float st_s0 = 0.f, st_s1 = 0.f, st_s2 = 0.f, st_s3 = 0.f, st_q0 = 0.f, st_q1 = 0.f, st_q2 = 0.f, st_q3 = 0.f;
        int st_n0 = -1;
        auto flush_stats = [&]() {
            if (stats && st_n0 >= 0) {
                // the four warps of a group hold the four row quarters of the same channels: combine them through the
                // group's (idle) staging slab so that ONE thread per channel issues the fp64 atomics - a single-wave
                // layer-3 launch otherwise sends 548 atomics to each of 512 addresses at the same moment (+8 us)
                float* scratch = reinterpret_cast<float*>(staging + (size_t)(ngrp == 1 ? 0 : grp) * TC_A_BYTES);
                if (et == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                asm volatile("bar.sync %0, 128;" ::"r"(barid) : "memory");
                scratch[0 * 128 + r] = st_s0; scratch[1 * 128 + r] = st_q0;
                scratch[2 * 128 + r] = st_s1; scratch[3 * 128 + r] = st_q1;
                scratch[4 * 128 + r] = st_s2; scratch[5 * 128 + r] = st_q2;
                scratch[6 * 128 + r] = st_s3; scratch[7 * 128 + r] = st_q3;
                asm volatile("bar.sync %0, 128;" ::"r"(barid) : "memory");
                const int slab = grp + q * ngrp;              // warp q of the group reduces accumulator slot si = q
                const int cbf = st_n0 + 32 * slab + lane;
                if (32 * slab < p.BN && cbf < p.Cout) {
                    const float* ps = scratch + (2 * q) * 128 + lane;
                    const float sv = (ps[0] + ps[32]) + (ps[64] + ps[96]);
                    const float qv = (ps[128] + ps[160]) + (ps[192] + ps[224]);
                    if (sv != 0.f || qv != 0.f) {
                        atomicAdd(stats + cbf, (double)sv);
                        atomicAdd(stats + p.Cout + cbf, (double)qv);
                    }
                }
            }
            st_s0 = st_s1 = st_s2 = st_s3 = st_q0 = st_q1 = st_q2 = st_q3 = 0.f;
        };
        bool ok = true;
        for (int work = cid; work < p.total_tiles && ok; work += nclusters, ++tcount) {
            const uint32_t set = tcount & 1u, aph = (tcount >> 1) & 1u;
            ok = __all_sync(0xffffffffu, mbar_wait(&acc_full[set], aph, err_flag, 3));
            if (!ok) break;
            tc_fence_after();
            int n0, w0, h0, n;
            tc_pair_coords(p, work, rank, n0, w0, h0, n);
            if (n0 != st_n0) { flush_stats(); st_n0 = n0; }
            const int hy = r / p.BW, wx = r - hy * p.BW;
            const int oy = h0 + hy, ox = w0 + wx;
            const bool valid = n < p.N && hy < p.BH && oy < p.OH && ox < p.OW;
            float* orow = out + ((int64_t)(n * p.outH + oy * p.out_mul + p.out_offy) * p.outW + ox * p.out_mul + p.out_offx) * p.ldo;
            const int used = iters < p.nacc ? iters : p.nacc;
            const uint32_t tbase = tmem_d + set * set_cols + ((uint32_t)(q * 32) << 16);
            for (int j = 32 * grp; j < p.BN; j += 32 * ngrp) {
                const int cb = n0 + j;
                if (cb >= p.Cout || n >= p.N) break;
                float v[32];
                tmem_ld32(tbase + (uint32_t)j, v);
                for (int a = 1; a < used; ++a) {
                    float u[32];
                    tmem_ld32(tbase + (uint32_t)a * acc_cols + (uint32_t)j, u);
#pragma unroll
                    for (int c = 0; c < 32; ++c) v[c] += u[c];
                }
                if (osc != 1.f) {
#pragma unroll
                    for (int c = 0; c < 32; ++c) v[c] *= osc;
                }
                if (bias) {
#pragma unroll
                    for (int c = 0; c < 32; ++c) if (cb + c < p.Cout) v[c] += __ldg(bias + cb + c);
                }
                const bool walk = stats && p.stats_smem && p.tma_store;
                float col_s = 0.f, col_q = 0.f;
                if (stats && !walk) {
                    float sv[32], sq[32];
#pragma unroll
                    for (int c = 0; c < 32; ++c) { const float o = valid ? v[c] : 0.f; sv[c] = o; sq[c] = o * o; }
#pragma unroll
                    for (int off = 16; off >= 1; off >>= 1) {
                        const bool up = (lane & off) != 0;
#pragma unroll
                        for (int i = 0; i < off; ++i) {
                            const float s_send = up ? sv[i] : sv[i + off], q_send = up ? sq[i] : sq[i + off];
                            const float s_recv = __shfl_xor_sync(0xffffffffu, s_send, off);
                            const float q_recv = __shfl_xor_sync(0xffffffffu, q_send, off);
                            sv[i] = (up ? sv[i + off] : sv[i]) + s_recv;
                            sq[i] = (up ? sq[i + off] : sq[i]) + q_recv;
                        }
                    }
                    col_s = sv[0]; col_q = sq[0];
                }
                if (walk && !valid) {
#pragma unroll
                    for (int c = 0; c < 32; ++c) v[c] = 0.f;
                }
                if (p.tma_store) {
                    const uint32_t b = ngrp == 1 ? (sc & 1u) : (uint32_t)grp;
                    if (et == 0) {
                        if (ngrp == 1) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
                        else asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                    }
                    asm volatile("bar.sync %0, 128;" ::"r"(barid) : "memory");
                    float4* dst = reinterpret_cast<float4*>(staging + (size_t)b * TC_A_BYTES + (size_t)r * 128);
#pragma unroll
                    for (int c = 0; c < 8; ++c)
                        dst[c ^ (r & 7)] = make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    asm volatile("bar.sync %0, 128;" ::"r"(barid) : "memory");
                    if (et == 0) {
                        if (p.out_acc) tma_reduce_add_4d(staging + (size_t)b * TC_A_BYTES, &mapOut, cb, w0, h0, n);
                        else tma_store_4d(staging + (size_t)b * TC_A_BYTES, &mapOut, cb, w0, h0, n);
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    }
                    if (walk) {
                        const float* srow = reinterpret_cast<const float*>(staging + (size_t)b * TC_A_BYTES + (size_t)(q * 32) * 128);
                        const int cq = lane >> 2, cw = lane & 3;
#pragma unroll 8
                        for (int rr = 0; rr < 32; ++rr) {
                            const float o = srow[rr * 32 + (((cq ^ (rr & 7)) << 2) | cw)];
                            col_s += o; col_q = fmaf(o, o, col_q);
                        }
                    }
                    ++sc;
                } else if (valid) {
                    if (cb + 31 < p.Cout && (p.ldo & 3) == 0) {
#pragma unroll
                        for (int c = 0; c < 32; c += 4)
                            *reinterpret_cast<float4*>(orow + cb + c) = make_float4(v[c], v[c + 1], v[c + 2], v[c + 3]);
                    } else {
#pragma unroll
                        for (int c = 0; c < 32; ++c)
                            if (cb + c < p.Cout) orow[cb + c] = v[c];
                    }
                }
                if (stats) {
                    const int si = (j / 32 - grp) / ngrp;
                    if (si < 4) {
                        switch (si) {
                            case 0: st_s0 += col_s; st_q0 += col_q; break;
                            case 1: st_s1 += col_s; st_q1 += col_q; break;
                            case 2: st_s2 += col_s; st_q2 += col_q; break;
                            default: st_s3 += col_s; st_q3 += col_q; break;
                        }
                    } else if (cb + lane < p.Cout) {
                        atomicAdd(stats + cb + lane, (double)col_s);
                        atomicAdd(stats + p.Cout + cb + lane, (double)col_q);
                    }
                }
            }
            // release this accumulator set to the leader's MMA thread (arrivals of both CTAs' epilogue threads)
            tc_fence_before();
            mbar_arrive_cluster(mapa_u32(smem_u32(&acc_empty[set]), 0));
        }
        flush_stats();
        if (et == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    } else {
        // ================= operand transform (3xTF32 with raw activations; both CTAs) =================
        if (p.a_inkernel) {
            const int t = threadIdx.x - 192;
            uint32_t gs = 0;
            bool okt = true;
            for (int work = cid; work < p.total_tiles && okt; work += nclusters) {
                for (int it = 0; it < iters; ++it, ++gs) {
                    const int s = gs % p.stages;
                    const uint32_t ph = (gs / p.stages) & 1u;
                    okt = mbar_wait(&full_bar[s], ph, err_flag, 4);
                    if (!okt) break;
                    float4* a_hi = reinterpret_cast<float4*>(smem + (size_t)s * stage_bytes);
                    float4* a_lo = reinterpret_cast<float4*>(smem + (size_t)s * stage_bytes + per_op);
#pragma unroll
                    for (int c = 0; c < TC_A_BYTES / 16 / 128; ++c) {
                        const float4 v = a_hi[t + c * 128];
                        float4 h, l;
                        const float* vp = &v.x; float* hp = &h.x; float* lp = &l.x;
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            uint32_t u;
                            asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(vp[e]));
                            u &= 0xFFFFE000u;
                            hp[e] = __uint_as_float(u);
                            lp[e] = vp[e] - hp[e];
                        }
                        a_hi[t + c * 128] = h;
                        a_lo[t + c * 128] = l;
                    }
                    asm volatile("fence.proxy.async;" ::: "memory");      // generic writes -> async proxy (both SMs' tensor cores)
                    mbar_arrive_cluster(mapa_u32(smem_u32(&ready_bar[s]), 0));
                }
            }
        }
    }
    tc_fence_before();
    cluster_sync_all();                                   // nobody leaves while the peer may still touch its smem/TMEM
    if (warp == 1) tmem_dealloc2(tmem_d, tmem_cols);
}

// ------------------------------------------------------------------------------------------
// tf32 split: hi = x with the low 13 mantissa bits cleared after round-to-nearest, lo = x - hi
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
split_tf32_kernel(const float4* __restrict__ x, float4* __restrict__ hi, float4* __restrict__ lo, int64_t n4) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        const float4 v = __ldcs(x + i);
        float4 h, l;
        const float* vp = &v.x; float* hp = &h.x; float* lp = &l.x;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            uint32_t u;
            asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(vp[k]));
            u &= 0xFFFFE000u;
            hp[k] = __uint_as_float(u);
            lp[k] = vp[k] - hp[k];
        }
        hi[i] = h;
        lo[i] = l;
    }
}

extern "C" int pxl_split_tf32(const float* x, float* hi, float* lo, int64_t n, void* stream) {
    if (!x || !hi || !lo || n <= 0 || (n & 3)) return PXL_ERR_BAD_ARG;
    const int64_t n4 = n / 4;
    int blocks = (int)(pxl_cdiv(n4, 256 * 2) < PXL_NUM_SMS * 8 ? pxl_cdiv(n4, 256 * 2) : PXL_NUM_SMS * 8);
    split_tf32_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>((const float4*)x, (float4*)hi, (float4*)lo, n4);
    PXL_CHECK_LAUNCH();
    return 0;
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static int* g_err_flag = nullptr;

static void pick_tile(int OH, int OW, bool flat, int& BW, int& BH) {
    if (flat) { BW = 128; BH = 1; return; }
    // choose BW x BH <= 128 maximising useful pixels per 128-row MMA tile
    double best = -1.0;
    BW = 16; BH = 8;
    for (int bw = 4; bw <= 128 && bw <= 256; ++bw) {
        int bh = 128 / bw;
        if (bh < 1) break;
        if (bh > 256) bh = 256;
        const int64_t tiles = (int64_t)((OW + bw - 1) / bw) * ((OH + bh - 1) / bh);
        const double eff = (double)OH * OW / ((double)tiles * 128.0);
        if (eff > best + 1e-9) { best = eff; BW = bw; BH = bh; }
    }
}

static int conv_tc_launch_core(const pxl_conv_geom* g, const int* taps, const pxl_conv_tc_ext* ext,
                               const void* in_hi, const void* in_lo, const void* w_hi, const void* w_lo,
                               const float* bias, float* out, void* stream);

// lo parts: for precision 2 the caller passes hi/lo through `in`/`w` (hi) and the extra pointers
extern "C" int pxl_conv_tc_launch(const pxl_conv_geom* g, const int* taps, const float* in_hi, const float* in_lo,
                                  const float* w_hi, const float* w_lo, const float* bias, float* out, void* stream) {
    if (g && g->precision > 2) return PXL_ERR_BAD_ARG;      // fp16 operands go through pxl_conv_h16_launch
    return conv_tc_launch_core(g, taps, nullptr, in_hi, in_lo, w_hi, w_lo, bias, out, stream);
}

extern "C" int pxl_conv_tc_launch_ex(const pxl_conv_geom* g, const int* taps, const pxl_conv_tc_ext* ext,
                                     const float* in_hi, const float* in_lo, const float* w_hi, const float* w_lo,
                                     const float* bias, float* out, void* stream) {
    if (g && g->precision > 2) return PXL_ERR_BAD_ARG;
    return conv_tc_launch_core(g, taps, ext, in_hi, in_lo, w_hi, w_lo, bias, out, stream);
}

// fp16-pair operands (h16_prep.cu): precision 3 = hi*hi + lo*hi + hi*lo (fp32-grade), 4 = hi*hi only (11-bit
// significands = TF32-grade)
extern "C" int pxl_conv_h16_launch(const pxl_conv_geom* g, const int* taps, const pxl_conv_tc_ext* ext,
                                   const void* in_hi, const void* in_lo, const void* w_hi, const void* w_lo,
                                   const float* bias, float* out, void* stream) {
    if (!g || (g->precision != 3 && g->precision != 4)) return PXL_ERR_BAD_ARG;
    return conv_tc_launch_core(g, taps, ext, in_hi, in_lo, w_hi, w_lo, bias, out, stream);
}

static int conv_tc_launch_core(const pxl_conv_geom* g, const int* taps, const pxl_conv_tc_ext* ext,
                               const void* in_hi, const void* in_lo, const void* w_hi, const void* w_lo,
                               const float* bias, float* out, void* stream) {
    if (!g || !taps || !in_hi || !w_hi || !out) return PXL_ERR_BAD_ARG;
    if ((g->mul != 1 && g->mul != 2) || g->div != 1) return PXL_ERR_UNSUPPORTED;
    const int f16 = g->precision >= 3 ? 1 : 0;
    const int kc = f16 ? 64 : 32;
    if (g->Cin % kc != 0 || g->ntaps > PXL_MAX_TAPS) return PXL_ERR_UNSUPPORTED;
    const int wtaps = ext && ext->w_ntaps > 0 ? ext->w_ntaps : g->ntaps;    // taps in the weight tensor
    const int nsplit = (g->precision == 2 || g->precision == 3) ? 3 : 1;
    if (nsplit == 3 && !w_lo) return PXL_ERR_BAD_ARG;
    if (f16 && nsplit == 3 && !in_lo) return PXL_ERR_BAD_ARG;    // fp16 pairs are always split by their producer
    const int a_inkernel = (!f16 && nsplit == 3 && !in_lo) ? 1 : 0;       // in_hi then holds the raw fp32 activations
    const int omul = (ext && ext->out_mul > 0) ? ext->out_mul : 1;
    const bool has_out_xform = ext && (omul != 1 || ext->out_offy != 0 || ext->out_offx != 0);
    bool flat = (g->ntaps == 1 && taps[0] == 0 && taps[1] == 0 && g->OH == g->H && g->OW == g->W && g->mul == 1 &&
                 !has_out_xform);
    TcParams p;
    p.Cin = g->Cin; p.Cout = g->Cout; p.ldo = g->ldo; p.ntaps = g->ntaps; p.kchunks = g->Cin / kc;
    p.nsplit = nsplit; p.a_inkernel = a_inkernel; p.f16 = f16; p.kc = kc;
    p.out_scale = (ext && ext->out_scale != 0.f) ? ext->out_scale : 1.f;
    const float* oscale_ptr = ext ? ext->out_scale_dev : nullptr;
    for (int t = 0; t < g->ntaps; ++t) {
        p.dy[t] = (short)taps[2 * t]; p.dx[t] = (short)taps[2 * t + 1];
        p.widx[t] = (short)((ext && ext->widx_host) ? ext->widx_host[t] : t);
        if (p.widx[t] < 0 || p.widx[t] >= wtaps) return PXL_ERR_BAD_ARG;
    }
    p.in_mul = g->mul;
    p.out_mul = omul; p.out_offy = has_out_xform ? ext->out_offy : 0; p.out_offx = has_out_xform ? ext->out_offx : 0;
    int mapW, mapH, mapN;
    if (flat) {
        const int64_t M = (int64_t)g->N * g->H * g->W;
        if (M >= (1ll << 31)) return PXL_ERR_UNSUPPORTED;
        p.N = 1; p.OH = 1; p.OW = (int)M;
        mapW = (int)M; mapH = 1; mapN = 1;
        p.outH = 1; p.outW = (int)M;
    } else {
        p.N = g->N; p.OH = g->OH; p.OW = g->OW;
        mapW = g->W; mapH = g->H; mapN = g->N;
        p.outH = has_out_xform ? ext->out_H : g->OH; p.outW = has_out_xform ? ext->out_W : g->OW;
    }
    pick_tile(p.OH, p.OW, flat, p.BW, p.BH);
    if (g->mul == 2 && (p.BW > 128 || p.BH > 128)) return PXL_ERR_UNSUPPORTED;
    // tuning knobs (environment, read once): shared-memory budget per CTA in KB (<= ~100 lets two CTAs share
    // an SM so one CTA's epilogue overlaps the other's main loop), N-tile cap, accumulator count
    static int cfg_budget_kb = -1, cfg_bn_max1 = 256, cfg_bn_max3 = 128, cfg_nacc3 = 4;
    static int cfg_bn_max_h3 = 256, cfg_bn_max_h1 = 256, cfg_nacc_h3 = 4, cfg_nacc_h1 = 1;   // measured: tools/sweep_h16.sh
    if (cfg_budget_kb < 0) {
        const char* e = getenv("PXL_TC_SMEM_KB"); cfg_budget_kb = e ? atoi(e) : 200;
        if ((e = getenv("PXL_TC_BN_MAX_TF32"))) cfg_bn_max1 = atoi(e);
        if ((e = getenv("PXL_TC_BN_MAX_TF32X3"))) cfg_bn_max3 = atoi(e);
        if ((e = getenv("PXL_TC_NACC_TF32X3"))) cfg_nacc3 = atoi(e);
        if ((e = getenv("PXL_TC_BN_MAX_F16X3"))) cfg_bn_max_h3 = atoi(e);
        if ((e = getenv("PXL_TC_BN_MAX_F16"))) cfg_bn_max_h1 = atoi(e);
        if ((e = getenv("PXL_TC_NACC_F16X3"))) cfg_nacc_h3 = atoi(e);
        if ((e = getenv("PXL_TC_NACC_F16"))) cfg_nacc_h1 = atoi(e);
    }
    p.BN = g->Cout > 128 ? 256 : (g->Cout > 64 ? 128 : (g->Cout > 32 ? 64 : 32));
    const int bn_cap = f16 ? (nsplit == 3 ? cfg_bn_max_h3 : cfg_bn_max_h1) : (nsplit == 3 ? cfg_bn_max3 : cfg_bn_max1);
    if (p.BN > bn_cap) p.BN = bn_cap;
    static int cfg_persist = -1;
    if (cfg_persist < 0) { const char* e = getenv("PXL_TC_PERSIST"); cfg_persist = e ? atoi(e) : 1; }
    // measured per layer shape (tools/bench_conv.py): the persistent kernel wins everywhere for 3xTF32 and for
    // single-pass TF32 except multi-tap convolutions with more than one wave of tiles, where two co-resident
    // non-persistent CTAs per SM pull more L2 bandwidth (those layers are operand-traffic bound)
    int use_persist = cfg_persist;
    if (cfg_persist == 1 && nsplit == 1 && g->ntaps > 1) {
        int bw, bh;
        pick_tile(p.OH, p.OW, flat, bw, bh);
        const int64_t tiles = (int64_t)p.N * ((p.OW + bw - 1) / bw) * ((p.OH + bh - 1) / bh) * ((g->Cout + p.BN - 1) / p.BN);
        if (tiles > PXL_NUM_SMS) use_persist = 0;
    }
    // CTA pairs (cta_group::2): 256 pixels x BN per step, each CTA stages half of the weight tile
    // PXL_TC_PAIR: 0 never, 1 whenever possible, 2 (default) = the fp16 modes on layers with >= 256 output channels and
    // a reduction of >= 256 (ResNet layer3 / layer4): there the halved weight traffic per SM pays (measured per
    // shape, tools/bench_conv.py: -6..-10 %); narrower layers are epilogue / L2 bound and lose with M = 256 tiles
    static int cfg_pair = -1;
    if (cfg_pair < 0) { const char* e = getenv("PXL_TC_PAIR"); cfg_pair = e ? atoi(e) : 2; }
    int use_pair = 0;
    // auto rule, re-measured after the issue-loop rewrite (tools/bench_conv.py, PXL_TC_PAIR=0/1): pairs win when the
    // reduction is long enough to amortise the cluster start-up (K >= 256) - except the 1x1 layers with K = 256 and a
    // 4x wider output (layer3 conv3 / conv1-dgrad: epilogue-bound, 33.3 vs 36.9 us) - and also on 3x3 layers with only
    // 128 output channels (layer2 conv2: 48 vs 57 us).  3 = the rule of the first half of round 2 (Cout >= 256).
    const int64_t kred = (int64_t)g->Cin * g->ntaps;
    const bool wide_1x1 = g->ntaps == 1 && kred < 512 && g->Cout >= 4 * g->Cin;
    const bool pair_auto = f16 && kred >= 256 && !wide_1x1 && (g->Cout >= 256 || g->ntaps > 1);
    const bool pair_wanted = cfg_pair == 1 || (cfg_pair == 2 && pair_auto) ||
                             (cfg_pair == 3 && f16 && g->Cout >= 256 && kred >= 256);
    if (pair_wanted && cfg_persist && p.BN >= 128) {
        int bw, bh;
        pick_tile(p.OH, p.OW, flat, bw, bh);
        const int64_t pix_tiles = (int64_t)p.N * ((p.OW + bw - 1) / bw) * ((p.OH + bh - 1) / bh);
        if (pix_tiles >= 2) use_pair = 1;
    }
    if (use_pair) use_persist = 1;
    p.nacc = f16 ? (nsplit == 3 ? cfg_nacc_h3 : cfg_nacc_h1) : (nsplit == 3 ? cfg_nacc3 : 1);
    if (p.nacc < 1) p.nacc = 1;
    // TMEM: 512 columns per SM; the persistent kernel keeps two accumulator sets (epilogue / main loop overlap)
    while (p.nacc > 1 && (p.BN < 32 ? 32 : p.BN) * p.nacc * (use_persist ? 2 : 1) > 512) p.nacc >>= 1;
    const int per_op = TC_A_BYTES + (use_pair ? p.BN / 2 : p.BN) * 128;
    const int stage_bytes = per_op * (nsplit == 3 ? 2 : 1);
    // measured (tools/sweep_tc.sh, MT step): single-pass TF32 is 6.5 % faster with two co-resident CTAs per SM
    // (<= 100 KB each: one CTA's epilogue overlaps the other's main loop); 3xTF32 needs the deeper ring
    pick_tile(p.OH, p.OW, flat, p.BW, p.BH);
    p.tilesW = (p.OW + p.BW - 1) / p.BW; p.tilesH = (p.OH + p.BH - 1) / p.BH;
    const int64_t n_ctas = (int64_t)p.N * p.tilesH * p.tilesW * ((g->Cout + p.BN - 1) / p.BN);
    // a grid that fits one wave at one CTA per SM gets the deep ring instead of a co-resident CTA
    const int budget = (getenv("PXL_TC_SMEM_KB") ? cfg_budget_kb : ((nsplit == 3 || n_ctas <= PXL_NUM_SMS) ? 200 : 100)) * 1024;
    p.ntilesN = (g->Cout + p.BN - 1) / p.BN;
    p.total_tiles = (int)n_ctas;
    const size_t persist_fixed = 1024 + (size_t)TC_STG_SLABS * TC_A_BYTES;     // alignment slack + staging slabs
    if (use_persist) p.stages = (int)((227 * 1024 - 2048 - persist_fixed) / stage_bytes);
    else p.stages = budget / stage_bytes;
    if (p.stages > 8) p.stages = 8;
    if (p.stages < 2) return PXL_ERR_UNSUPPORTED;
    const size_t smem = use_persist ? (size_t)p.stages * stage_bytes + persist_fixed : (size_t)p.stages * stage_bytes + 1024;

    CUtensorMap mA, mAlo, mB, mBlo;
    int rc = make_act_map(&mA, in_hi, g->Cin, mapW, mapH, mapN, p.BW, p.BH, g->mul, f16);
    if (rc) return rc;
    const int b_box_rows = use_pair ? p.BN / 2 : p.BN;
    rc = make_w_map(&mB, w_hi, (int64_t)wtaps * g->Cin, g->Cout, b_box_rows, f16);
    if (rc) return rc;
    if (nsplit == 3) {
        if (a_inkernel) mAlo = mA;
        else {
            rc = make_act_map(&mAlo, in_lo, g->Cin, mapW, mapH, mapN, p.BW, p.BH, g->mul, f16);
            if (rc) return rc;
        }
        rc = make_w_map(&mBlo, w_lo, (int64_t)wtaps * g->Cin, g->Cout, b_box_rows, f16);
        if (rc) return rc;
    } else {
        mAlo = mA; mBlo = mB;
    }
    // TMA-store epilogue: needs 16-byte pixel strides and the plain output mapping
    static int cfg_tma_store = -1;
    if (cfg_tma_store < 0) { const char* e = getenv("PXL_TC_TMA_STORE"); cfg_tma_store = e ? atoi(e) : 1; }
    p.tma_store = (cfg_tma_store && !has_out_xform && (g->ldo % 4) == 0 && ((uintptr_t)out % 16) == 0) ? 1 : 0;
    CUtensorMap mO = mA;
    if (p.tma_store) {
        rc = make_out_map(&mO, out, g->Cout, g->ldo, p.outW, p.outH, p.N, p.BW, p.BH);
        if (rc) p.tma_store = 0;
    }
    static int cfg_stats_smem = -1;
    if (cfg_stats_smem < 0) { const char* e = getenv("PXL_TC_STATS_SMEM"); cfg_stats_smem = e ? atoi(e) : 1; }
    p.stats_smem = cfg_stats_smem;
    p.out_acc = (ext && ext->out_accumulate) ? 1 : 0;
    if (p.out_acc && !(p.tma_store && use_persist)) return PXL_ERR_UNSUPPORTED;      // accumulation exists in the TMA-store epilogues only
    cudaStream_t st = (cudaStream_t)stream;
    if (!g_err_flag) {
        cudaError_t e = cudaMalloc(&g_err_flag, sizeof(int));
        if (e != cudaSuccess) return (int)e;
        e = cudaMemset(g_err_flag, 0, sizeof(int));
        if (e != cudaSuccess) return (int)e;
    }
    static bool attr = false;
    if (!attr) {
        cudaError_t e = cudaFuncSetAttribute(conv_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 2048);
        if (e != cudaSuccess) return (int)e;
        attr = true;
    }
    if (use_pair) {
        static bool attr3 = false;
        if (!attr3) {
            cudaError_t e = cudaFuncSetAttribute(conv_tc_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 2048);
            if (e != cudaSuccess) return (int)e;
            attr3 = true;
        }
        const int64_t pix_tiles = (int64_t)p.N * p.tilesH * p.tilesW;
        p.total_tiles = (int)(((pix_tiles + 1) / 2) * p.ntilesN);          // work items of a pair
        int nclusters = p.total_tiles < PXL_NUM_SMS / 2 ? p.total_tiles : PXL_NUM_SMS / 2;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(2 * nclusters), 1, 1);
        cfg.blockDim = dim3(320, 1, 1);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute at[2];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[1].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at; cfg.numAttrs = pxl_pdl_enabled_() ? 2 : 1;
        double* st_ptr = ext ? (double*)ext->bn_stats : nullptr;
        cudaError_t e = cudaLaunchKernelEx(&cfg, conv_tc_pair_kernel, mA, mAlo, mB, mBlo, mO, p, bias, out, st_ptr, g_err_flag, oscale_ptr);
        if (e != cudaSuccess) return (int)e;
        pxl_count_launch_(1);
        return 0;
    }
    if (use_persist) {
        static bool attr2 = false;
        if (!attr2) {
            cudaError_t e = cudaFuncSetAttribute(conv_tc_persist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 2048);
            if (e != cudaSuccess) return (int)e;
            attr2 = true;
        }
        const unsigned nblk = (unsigned)(p.total_tiles < PXL_NUM_SMS ? p.total_tiles : PXL_NUM_SMS);
        cudaError_t le = pxl_launch_pdl(conv_tc_persist_kernel, dim3(nblk), dim3(320), smem, st, mA, mAlo, mB, mBlo, mO, p, bias, out,
                                        ext ? (double*)ext->bn_stats : (double*)nullptr, g_err_flag, oscale_ptr);
        if (le != cudaSuccess) return (int)le;
        PXL_CHECK_LAUNCH();
        return 0;
    }
    dim3 grid((unsigned)((int64_t)p.N * p.tilesH * p.tilesW), (unsigned)((g->Cout + p.BN - 1) / p.BN));
    cudaError_t le = pxl_launch_pdl(conv_tc_kernel, grid, dim3(192), smem, st, mA, mAlo, mB, mBlo, mO, p, bias, out,
                                    ext ? (double*)ext->bn_stats : (double*)nullptr, g_err_flag, oscale_ptr);
    if (le != cudaSuccess) return (int)le;
    PXL_CHECK_LAUNCH();
    return 0;
}

// watchdog status: 0 = fine, otherwise the role (1 producer, 2 mma, 3 epilogue) that timed out
extern "C" int pxl_conv_tc_status(void) {
    if (!g_err_flag) return 0;
    int v = 0;
    if (cudaMemcpy(&v, g_err_flag, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    return v;
}

extern "C" int pxl_conv_tc_impl(const pxl_conv_geom* g, const int* taps, const float* in, const float* w,
                                const float* bias, float* out, void* stream) {
    if (!g) return PXL_ERR_BAD_ARG;
    if (g->precision == 2) return PXL_ERR_UNSUPPORTED;     // 3xTF32 needs the split operands: pxl_conv_tc_launch
    return pxl_conv_tc_launch(g, taps, in, nullptr, w, nullptr, bias, out, stream);
}

// ==========================================================================================
// wgrad on tcgen05:  dW[co][tap][ci] += sum_pixels dY[pix][co] * X[pix + tap][ci]
//
//   D[128 co, BN ci] (TMEM) += A^T[K = pixels, 128 co] * B[K = pixels, BN ci]
//
// Both operands are "MN-major" (the reduction index = pixel row is the slow one), which is exactly
// what NHWC gives: a TMA box {32 channels, BW, BH, 1} is (BW*BH pixel rows) x 128 B and lands as one
// SWIZZLE_128B_ATOM_32B slab; 4 slabs of dY (128 co) and BN/32 slabs of X (tap-shifted, OOB zero-filled)
// form a stage.  Each tcgen05.mma.kind::tf32 consumes 8 pixel rows (one 1024-B swizzle atom per
// slab).  Rows between BW*BH and the 8-aligned allocation are zeroed once and never written.
// The pixel range is split over gridDim.z CTAs.  Each writes its tile into its own slot of a workspace
// [split][Cout][taps][Cin]; wg_slot_sum_kernel then adds the slots into dW in split order, so dW does not depend on
// the order in which the CTAs finish (fp32 adds from different CTAs in arrival order would make every run differ).
// ==========================================================================================
struct WgParams {
    int Cin, Cout, ldo, ntaps;
    int N, OH, OW, mul;
    int BW, BH, tilesW, tilesH, rows, rows_alloc;
    int BN, stages, nsplit, nacc;
    int inkernel;      // 3xTF32: dY / X arrive raw and are split hi/lo in shared memory by the epilogue warps
    int f16;           // fp16 operands (kind::f16): 64-channel slabs, 16 pixel rows per MMA, plain SWIZZLE_128B
    int slab_ch;       // channels per 128-byte slab row: 32 (tf32) or 64 (fp16)
    float out_scale;   // the tile is multiplied by this (and by *oscale_ptr) before it is added into dW
    int tma_red;       // epilogue: stage 32-column slabs in the drained ring and TMA-store them into the slot
                       // (PXL_WG_TMA_REDUCE=0: plain stores; the name dates from the reduce-add epilogue)
    int tiles_ci, ktiles_per_cta, ktiles_total;
    short dy[PXL_MAX_TAPS], dx[PXL_MAX_TAPS];
};

// MN-major tf32 operands only exist in the SWIZZLE_128B_BASE32B layout (cutlass sm100_common.inl:92;
// cute Layout_MN_SW128_32B_Atom = Swizzle<2,5,2> over 4 rows x 128 B): 128-byte rows, 32-byte swizzle
// granularity, atoms of 4 K-rows.  LBO = byte distance between 32-element MN slabs, SBO = byte
// distance between 4-row K atoms (512 B for densely packed rows).  TMA writes this layout with
// CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B.
__device__ __forceinline__ uint64_t mnmajor_sw128_desc(uint32_t smem_addr, uint32_t lbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)(512 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)1 << 61;       // LayoutType::SWIZZLE_128B_BASE32B
    return d;
}

// MN-major 16-bit operands use the plain SWIZZLE_128B layout (cute Layout_MN_SW128_Atom: 64 elements x 8 K-rows,
// Swizzle<3,4,3>): LBO = byte distance between 64-element MN slabs, SBO = 1024 B between 8-row K groups.
__device__ __forceinline__ uint64_t mnmajor_sw128_f16_desc(uint32_t smem_addr, uint32_t lbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;       // LayoutType::SWIZZLE_128B
    return d;
}

__global__ void __launch_bounds__(320, 1)
conv_wgrad_tc_kernel(const __grid_constant__ CUtensorMap mapDy, const __grid_constant__ CUtensorMap mapDyLo,
                     const __grid_constant__ CUtensorMap mapX, const __grid_constant__ CUtensorMap mapXLo,
                     const __grid_constant__ CUtensorMap mapDw,
                     const WgParams p, float* __restrict__ ws, int* __restrict__ err_flag,
                     const float* __restrict__ oscale_ptr) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ uint64_t full_bar[8], empty_bar[8], ready_bar[8], acc_bar;
    __shared__ uint32_t tmem_base_slot;
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);

    const int slab_bytes = p.rows_alloc * 128;
    const int slabsA = 128 / p.slab_ch;                  // dY slabs (128 output channels)
    const int slabsB = p.BN / p.slab_ch;
    const int per_op = (slabsA + slabsB) * slab_bytes;
    const int stage_bytes = per_op * (p.nsplit == 3 ? 2 : 1);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tile_co = blockIdx.x / p.tiles_ci, tile_ci = blockIdx.x % p.tiles_ci;
    const int co0 = tile_co * 128, ci0 = tile_ci * p.BN;
    const int tap = blockIdx.y;
    const int kt0 = blockIdx.z * p.ktiles_per_cta;
    int kt1 = kt0 + p.ktiles_per_cta;
    if (kt1 > p.ktiles_total) kt1 = p.ktiles_total;
    const int iters = kt1 - kt0;
    const uint32_t acc_cols = p.BN < 32 ? 32 : p.BN;
    const uint32_t tmem_cols = acc_cols * p.nacc;
    // slabs that actually exist (the others stay zero)
    int nsA = (p.ldo - co0 + p.slab_ch - 1) / p.slab_ch; if (nsA > slabsA) nsA = slabsA;
    int nsB = (p.Cin - ci0 + p.slab_ch - 1) / p.slab_ch; if (nsB > slabsB) nsB = slabsB;

    // zero the operand ring once: rows the TMA never writes must contribute nothing
    {
        uint4 z = make_uint4(0, 0, 0, 0);
        const int total16 = p.stages * stage_bytes / 16;
        for (int i = threadIdx.x; i < total16; i += blockDim.x) reinterpret_cast<uint4*>(smem)[i] = z;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (threadIdx.x == 0) {
        for (int s = 0; s < p.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); mbar_init(&ready_bar[s], blockDim.x - 64); }
        mbar_init(&acc_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(&tmem_base_slot, tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_d = tmem_base_slot;
    PXL_PDL_SYNC();          // everything above overlapped the previous kernel's tail; global memory from here on

    if (iters > 0) {
        if (warp == 0) {
            // TMA producer: whole warp converged, TMA under elect.sync
            const uint32_t box_bytes = (uint32_t)(p.rows * 128);
            const int nparts = (p.nsplit == 3 && !p.inkernel) ? 2 : 1;
            const uint32_t tx = box_bytes * (uint32_t)(nsA + nsB) * (uint32_t)nparts;
            const int tdy = p.dy[tap], tdx = p.dx[tap];
            int tw = kt0 % p.tilesW, th = (kt0 / p.tilesW) % p.tilesH, n = kt0 / (p.tilesW * p.tilesH);
            uint32_t s = 0, ph = 0;
            for (int it = 0; it < iters; ++it) {
                if (!__all_sync(0xffffffffu, mbar_wait(&empty_bar[s], ph ^ 1u, err_flag, 11))) break;
                const int w0 = tw * p.BW, h0 = th * p.BH;
                uint8_t* sa = smem + (size_t)s * stage_bytes;
                if (elect_one()) {
                    mbar_expect_tx(&full_bar[s], tx);
                    for (int part = 0; part < nparts; ++part) {
                        uint8_t* base = sa + (size_t)part * per_op;
                        const CUtensorMap* mdy = part ? &mapDyLo : &mapDy;
                        const CUtensorMap* mx = part ? &mapXLo : &mapX;
                        for (int j = 0; j < nsA; ++j)
                            tma_load_4d(base + (size_t)j * slab_bytes, mdy, &full_bar[s], co0 + p.slab_ch * j, w0, h0, n);
                        for (int j = 0; j < nsB; ++j)
                            tma_load_4d(base + (size_t)(slabsA + j) * slab_bytes, mx, &full_bar[s], ci0 + p.slab_ch * j,
                                        w0 * p.mul + tdx, h0 * p.mul + tdy, n);
                    }
                }
                __syncwarp();
                if (++tw == p.tilesW) { tw = 0; if (++th == p.tilesH) { th = 0; ++n; } }
                if (++s == (uint32_t)p.stages) { s = 0; ph ^= 1u; }
            }
        } else if (warp == 1) {
            // MMA issuer: whole warp converged, tcgen05 under elect.sync
            // D fp32, A/B tf32 or fp16, both MN-major (bits 15,16), M = 128, N = BN
            const uint32_t idesc = (p.f16 ? f16_idesc(p.BN) : tf32_idesc(p.BN)) | (1u << 15) | (1u << 16);
            const int krows = p.f16 ? 16 : 8;                 // pixel rows one MMA consumes
            const int kmma = p.rows_alloc / krows;
            const uint64_t kstep = (uint64_t)(krows * 128 / 16);   // descriptor start-address advance per MMA
            const uint32_t smem_base = smem_u32(smem);
            const uint32_t offB = (uint32_t)(slabsA * slab_bytes);
            uint32_t s = 0, ph = 0, a = 0;
            for (int it = 0; it < iters; ++it) {
                if (!__all_sync(0xffffffffu, mbar_wait(p.inkernel ? &ready_bar[s] : &full_bar[s], ph, err_flag, 12))) break;
                tc_fence_after();
                const uint32_t sa = smem_base + s * (uint32_t)stage_bytes;
                const uint32_t sb = sa + offB;
                const uint32_t acc = tmem_d + a * acc_cols;
                const uint32_t acc0 = it >= p.nacc ? 1u : 0u;
                uint64_t da, db, dal, dbl;
                if (p.f16) {
                    da = mnmajor_sw128_f16_desc(sa, (uint32_t)slab_bytes); db = mnmajor_sw128_f16_desc(sb, (uint32_t)slab_bytes);
                    dal = mnmajor_sw128_f16_desc(sa + per_op, (uint32_t)slab_bytes); dbl = mnmajor_sw128_f16_desc(sb + per_op, (uint32_t)slab_bytes);
                } else {
                    da = mnmajor_sw128_desc(sa, (uint32_t)slab_bytes); db = mnmajor_sw128_desc(sb, (uint32_t)slab_bytes);
                    dal = mnmajor_sw128_desc(sa + per_op, (uint32_t)slab_bytes); dbl = mnmajor_sw128_desc(sb + per_op, (uint32_t)slab_bytes);
                }
                if (elect_one()) {
                    if (p.f16) {
                        for (int k = 0; k < kmma; ++k) umma_f16(acc, da + kstep * k, db + kstep * k, idesc, k ? 1u : acc0);
                        if (p.nsplit == 3) {
                            for (int k = 0; k < kmma; ++k) umma_f16(acc, dal + kstep * k, db + kstep * k, idesc, 1u);
                            for (int k = 0; k < kmma; ++k) umma_f16(acc, da + kstep * k, dbl + kstep * k, idesc, 1u);
                        }
                    } else {
                        for (int k = 0; k < kmma; ++k) umma_tf32(acc, da + kstep * k, db + kstep * k, idesc, k ? 1u : acc0);
                        if (p.nsplit == 3) {
                            for (int k = 0; k < kmma; ++k) umma_tf32(acc, dal + kstep * k, db + kstep * k, idesc, 1u);
                            for (int k = 0; k < kmma; ++k) umma_tf32(acc, da + kstep * k, dbl + kstep * k, idesc, 1u);
                        }
                    }
                    umma_commit(&empty_bar[s]);
                    if (it == iters - 1) umma_commit(&acc_bar);
                }
                __syncwarp();
                if (++s == (uint32_t)p.stages) { s = 0; ph ^= 1u; }
                if (++a == (uint32_t)p.nacc) a = 0;
            }
        } else {
            const int q = warp & 3;
            const int co = co0 + q * 32 + lane;
            if (p.inkernel) {
                // raw fp32 slabs -> hi (in place) / lo (second half of the stage); elementwise, layout-agnostic.
                // All warps from 2 up take part (8 of them in the 3xTF32 launch: the split of BOTH operands is
                // as much work per stage as its 12 MMAs, four warps could not keep up)
                const int t = threadIdx.x - 64;
                const int tstride = blockDim.x - 64;
                const int chunks = per_op / 16;
                bool okt = true;
                for (int it = 0; it < iters && okt; ++it) {
                    const int s = it % p.stages;
                    const uint32_t ph = (uint32_t)(it / p.stages) & 1u;
                    okt = mbar_wait(&full_bar[s], ph, err_flag, 14);
                    if (!okt) break;
                    float4* hi = reinterpret_cast<float4*>(smem + (size_t)s * stage_bytes);
                    float4* lo = reinterpret_cast<float4*>(smem + (size_t)s * stage_bytes + per_op);
                    for (int c = t; c < chunks; c += tstride) {
                        const float4 v = hi[c];
                        float4 h, l;
                        const float* vp = &v.x; float* hp = &h.x; float* lp = &l.x;
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            uint32_t u;
                            asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(vp[e]));
                            u &= 0xFFFFE000u;
                            hp[e] = __uint_as_float(u);
                            lp[e] = vp[e] - hp[e];
                        }
                        hi[c] = h;
                        lo[c] = l;
                    }
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&ready_bar[s])) : "memory");
                }
            }
            const bool ok = warp < 6 && __all_sync(0xffffffffu, mbar_wait(&acc_bar, 0, err_flag, 13));
            tc_fence_after();
            if (ok) {
                const int used = iters < p.nacc ? iters : p.nacc;
                const float osc = p.out_scale * (oscale_ptr ? __ldg(oscale_ptr) : 1.f);
                float* drow = ws + (((int64_t)blockIdx.z * p.Cout + co) * p.ntaps + tap) * p.Cin;
                const int r = q * 32 + lane;
                const int et = threadIdx.x - 64;
                uint32_t sc = 0;
                for (int j = 0; j < p.BN; j += 32) {
                    if (p.tma_red && ci0 + j >= p.Cin) break;          // uniform
                    float v[32];
                    tmem_ld32(tmem_d + ((uint32_t)(q * 32) << 16) + (uint32_t)j, v);
                    for (int a = 1; a < used; ++a) {
                        float u[32];
                        tmem_ld32(tmem_d + ((uint32_t)(q * 32) << 16) + (uint32_t)a * acc_cols + (uint32_t)j, u);
#pragma unroll
                        for (int c = 0; c < 32; ++c) v[c] += u[c];
                    }
                    if (p.tma_red) {
                        // the operand ring is drained (acc_bar): two 16 KB slabs of it stage the tile, 128 rows (co) x
                        // 32 floats (ci) in the 128B-swizzled layout, and the TMA unit stores them into the slot
                        const uint32_t b = sc & 1u;
                        if (et == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
                        asm volatile("bar.sync 1, 128;" ::: "memory");
                        float4* dst = reinterpret_cast<float4*>(smem + (size_t)b * 16384 + (size_t)r * 128);
#pragma unroll
                        for (int c = 0; c < 8; ++c)
                            dst[c ^ (r & 7)] = make_float4(v[4 * c] * osc, v[4 * c + 1] * osc, v[4 * c + 2] * osc, v[4 * c + 3] * osc);
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        asm volatile("bar.sync 1, 128;" ::: "memory");
                        if (et == 0) {
                            tma_store_4d(smem + (size_t)b * 16384, &mapDw, ci0 + j, tap, co0, blockIdx.z);
                            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                        }
                        ++sc;
                        continue;
                    }
                    if (co >= p.Cout) continue;
#pragma unroll
                    for (int c = 0; c < 32; ++c) {
                        const int ci = ci0 + j + c;
                        if (ci < p.Cin) drow[ci] = v[c] * osc;
                    }
                }
                if (p.tma_red && et == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_d, tmem_cols);
}

// activation map for wgrad: optional traversal stride (stride-2 convolutions read every 2nd pixel)
static int make_act_map_strided(CUtensorMap* m, const void* base, int C, int W, int H, int N, int bw, int bh, int estride, int f16 = 0) {
    EncodeTiledFn enc = get_encode();
    if (!enc) return PXL_ERR_UNSUPPORTED;
    const cuuint64_t eb = f16 ? 2 : 4;
    cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
    cuuint64_t strides[3] = {(cuuint64_t)C * eb, (cuuint64_t)W * C * eb, (cuuint64_t)H * W * C * eb};
    cuuint32_t box[4] = {(cuuint32_t)(f16 ? 64 : 32), (cuuint32_t)(bw * estride), (cuuint32_t)(bh * estride), 1};
    cuuint32_t es[4] = {1, (cuuint32_t)estride, (cuuint32_t)estride, 1};
    if (box[1] > 256 || box[2] > 256) return PXL_ERR_UNSUPPORTED;
    CUresult r = enc(m, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void*)base, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, f16 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : PXL_ERR_BAD_ARG;
}

static void pick_ktile(int OH, int OW, bool flat, int maxrows, int& BW, int& BH, int unit = 8) {
    if (flat) { BW = maxrows; BH = 1; return; }
    double best = -1.0;
    BW = 8; BH = maxrows / 8;
    for (int bw = 1; bw <= maxrows && bw <= 256; ++bw) {
        int bh = maxrows / bw;
        if (bh < 1) break;
        if (bh > 256) bh = 256;
        const int alloc = (bw * bh + unit - 1) / unit * unit;
        const int64_t tiles = (int64_t)((OW + bw - 1) / bw) * ((OH + bh - 1) / bh);
        // useful rows per allocated row, discounted for narrow boxes: a TMA box is fetched as bh separate runs of
        // bw pixels, and short runs stream poorly (PXL_WG_WIDE_BIAS, measured with tools/bench_conv.py)
        static double bias = -1.0;
        if (bias < 0.0) { const char* e = getenv("PXL_WG_WIDE_BIAS"); bias = e ? atof(e) : 0.0; }
        const double eff = (double)OH * OW / ((double)tiles * alloc) * (1.0 - bias / (bias + bw));
        if (eff > best + 1e-9) { best = eff; BW = bw; BH = bh; }
    }
}

// ws_need != NULL: only report the workspace size (split * Cout * taps * Cin floats) the launch would need
static int conv_wgrad_tc_core(const pxl_conv_geom* g, const int* taps, const void* in_hi, const void* in_lo,
                              const void* dy_hi, const void* dy_lo, float* dw, float out_scale, const float* oscale_ptr,
                              float* ws, int64_t ws_floats, int64_t* ws_need, void* stream);

// dw[i] += slot[0][i] + slot[1][i] + ... in split order (n floats per slot)
__global__ void __launch_bounds__(256)
wg_slot_sum_kernel(const float* __restrict__ ws, float* __restrict__ dw, int64_t n, int split) {
    PXL_PDL_SYNC();
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        float s = __ldg(ws + i);
        for (int z = 1; z < split; ++z) s += __ldg(ws + (int64_t)z * n + i);
        dw[i] += s;
    }
}

extern "C" int64_t pxl_conv_wgrad_workspace_floats(const pxl_conv_geom* g, const int* taps) {
    int64_t need = 0;
    const int rc = conv_wgrad_tc_core(g, taps, nullptr, nullptr, nullptr, nullptr, nullptr, 1.f, nullptr, nullptr, 0, &need, nullptr);
    return rc ? (int64_t)rc : need;
}

extern "C" int pxl_conv_wgrad_tc_launch(const pxl_conv_geom* g, const int* taps, const float* in_hi, const float* in_lo,
                                        const float* dy_hi, const float* dy_lo, float* dw, float* ws, int64_t ws_floats,
                                        void* stream) {
    if (g && g->precision > 2) return PXL_ERR_BAD_ARG;      // fp16 operands go through pxl_conv_wgrad_h16_launch
    return conv_wgrad_tc_core(g, taps, in_hi, in_lo, dy_hi, dy_lo, dw, 1.f, nullptr, ws, ws_floats, nullptr, stream);
}

// fp16-pair operands; dw += out_scale * (*out_scale_dev) * sum(dy * x)
extern "C" int pxl_conv_wgrad_h16_launch(const pxl_conv_geom* g, const int* taps, const void* in_hi, const void* in_lo,
                                         const void* dy_hi, const void* dy_lo, float* dw, float out_scale,
                                         const float* out_scale_dev, float* ws, int64_t ws_floats, void* stream) {
    if (!g || (g->precision != 3 && g->precision != 4)) return PXL_ERR_BAD_ARG;
    return conv_wgrad_tc_core(g, taps, in_hi, in_lo, dy_hi, dy_lo, dw, out_scale != 0.f ? out_scale : 1.f, out_scale_dev,
                              ws, ws_floats, nullptr, stream);
}

static int conv_wgrad_tc_core(const pxl_conv_geom* g, const int* taps, const void* in_hi, const void* in_lo,
                              const void* dy_hi, const void* dy_lo, float* dw, float out_scale, const float* oscale_ptr,
                              float* ws, int64_t ws_floats, int64_t* ws_need, void* stream) {
    if (!g || !taps) return PXL_ERR_BAD_ARG;
    if (!ws_need && (!in_hi || !dy_hi || !dw || !ws)) return PXL_ERR_BAD_ARG;
    if (g->div != 1 || (g->mul != 1 && g->mul != 2)) return PXL_ERR_UNSUPPORTED;   // stride 2 via TMA traversal stride
    const int f16 = g->precision >= 3 ? 1 : 0;
    const int slab_ch = f16 ? 64 : 32;
    if (g->Cin % slab_ch != 0 || g->ldo % slab_ch != 0 || g->ntaps > PXL_MAX_TAPS) return PXL_ERR_UNSUPPORTED;
    const int nsplit = (g->precision == 2 || g->precision == 3) ? 3 : 1;
    if (!ws_need && nsplit == 3 && ((in_lo == nullptr) != (dy_lo == nullptr))) return PXL_ERR_BAD_ARG;
    if (!ws_need && f16 && nsplit == 3 && !in_lo) return PXL_ERR_BAD_ARG;
    const int inkernel = (!f16 && nsplit == 3 && !in_lo) ? 1 : 0;         // in_hi / dy_hi then hold the raw fp32 tensors
    const bool flat = (g->ntaps == 1 && taps[0] == 0 && taps[1] == 0 && g->OH == g->H && g->OW == g->W && g->mul == 1);
    WgParams p;
    p.Cin = g->Cin; p.Cout = g->Cout; p.ldo = g->ldo; p.ntaps = g->ntaps; p.mul = g->mul; p.nsplit = nsplit; p.inkernel = inkernel;
    p.f16 = f16; p.slab_ch = slab_ch; p.out_scale = out_scale;
    for (int t = 0; t < g->ntaps; ++t) { p.dy[t] = (short)taps[2 * t]; p.dx[t] = (short)taps[2 * t + 1]; }
    int mapW, mapH, mapN, inW, inH;
    if (flat) {
        const int64_t M = (int64_t)g->N * g->H * g->W;
        if (M >= (1ll << 31)) return PXL_ERR_UNSUPPORTED;
        p.N = 1; p.OH = 1; p.OW = (int)M; mapW = (int)M; mapH = 1; mapN = 1; inW = (int)M; inH = 1;
    } else {
        p.N = g->N; p.OH = g->OH; p.OW = g->OW; mapW = g->OW; mapH = g->OH; mapN = g->N; inW = g->W; inH = g->H;
    }
    static int cfg_wg_bn_max = -1, cfg_wg_bn_max_h3 = 256, cfg_wg_bn_max_h1 = 256, cfg_wg_rows_h3 = 64, cfg_wg_rows_h1 = 128;
    if (cfg_wg_bn_max < 0) {
        const char* e = getenv("PXL_WG_BN_MAX"); cfg_wg_bn_max = e ? atoi(e) : 128;
        if ((e = getenv("PXL_WG_BN_MAX_F16X3"))) cfg_wg_bn_max_h3 = atoi(e);
        if ((e = getenv("PXL_WG_BN_MAX_F16"))) cfg_wg_bn_max_h1 = atoi(e);
        if ((e = getenv("PXL_WG_ROWS_F16X3"))) cfg_wg_rows_h3 = atoi(e);
        if ((e = getenv("PXL_WG_ROWS_F16"))) cfg_wg_rows_h1 = atoi(e);
    }
    const bool wide = !f16 && nsplit == 1 && cfg_wg_bn_max >= 256 && g->Cin >= 256;     // 128 x 256 tile, 32-row stages
    int maxrows = nsplit == 3 ? 32 : (wide ? 32 : 64);
    if (f16) maxrows = nsplit == 3 ? cfg_wg_rows_h3 : cfg_wg_rows_h1;
    const int kunit = f16 ? 16 : 8;                      // pixel rows per MMA
    pick_ktile(p.OH, p.OW, flat, maxrows, p.BW, p.BH, kunit);
    p.rows = p.BW * p.BH;
    p.rows_alloc = (p.rows + kunit - 1) / kunit * kunit;
    p.tilesW = (p.OW + p.BW - 1) / p.BW; p.tilesH = (p.OH + p.BH - 1) / p.BH;
    p.BN = wide ? 256 : (g->Cin > 64 ? 128 : (g->Cin > 32 ? 64 : 32));
    if (f16) {
        const int cap = nsplit == 3 ? cfg_wg_bn_max_h3 : cfg_wg_bn_max_h1;
        p.BN = g->Cin > 128 ? 256 : (g->Cin > 64 ? 128 : 64);
        if (p.BN > cap) p.BN = cap < 64 ? 64 : cap;
    }
    p.nacc = 512 / (p.BN < 32 ? 32 : p.BN); if (p.nacc > 4) p.nacc = 4;
    p.tiles_ci = (g->Cin + p.BN - 1) / p.BN;
    const int tiles_co = (g->Cout + 127) / 128;
    const int stage_bytes = (128 / slab_ch + p.BN / slab_ch) * p.rows_alloc * 128 * (nsplit == 3 ? 2 : 1);
    p.stages = (200 * 1024) / stage_bytes;
    if (p.stages > 8) p.stages = 8;
    if (p.stages < 2) return PXL_ERR_UNSUPPORTED;
    p.ktiles_total = p.N * p.tilesH * p.tilesW;
    // split the pixel range: enough CTAs to fill the GPU, and at most ~4096 pixel rows per CTA so the
    // truncating TMEM accumulation stays at fp32 level (the per-split slots are summed with round to nearest)
    const int64_t base_ctas = (int64_t)tiles_co * p.tiles_ci * g->ntaps;
    int64_t by_rows = pxl_cdiv((int64_t)p.ktiles_total * p.rows_alloc, 4096);
    if (by_rows < 1) by_rows = 1;
    // one CTA per SM (the ring takes ~200 KB): pick the pixel split that minimises
    //   rounds x (main-loop iterations per CTA + a fixed prologue/epilogue cost)
    // so that the grid fills whole waves instead of leaving a mostly idle last one
    int64_t split = by_rows, best_cost = -1;
    int64_t hi = pxl_cdiv((int64_t)PXL_NUM_SMS * 4, base_ctas) + 1;
    if (hi < by_rows) hi = by_rows;
    if (hi > p.ktiles_total) hi = p.ktiles_total;
    for (int64_t sp = by_rows; sp <= hi; ++sp) {
        const int64_t per = pxl_cdiv(p.ktiles_total, sp);
        const int64_t ctas = base_ctas * pxl_cdiv(p.ktiles_total, per);
        const int64_t cost = pxl_cdiv(ctas, PXL_NUM_SMS) * (per + 6);
        if (best_cost < 0 || cost < best_cost) { best_cost = cost; split = sp; }
    }
    if (split > p.ktiles_total) split = p.ktiles_total;
    if (split < 1) split = 1;
    if (split > 65535) split = 65535;
    p.ktiles_per_cta = (int)pxl_cdiv(p.ktiles_total, split);
    split = pxl_cdiv(p.ktiles_total, p.ktiles_per_cta);
    // every CTA writes its whole tile into the slot of its pixel range (each slot element is written by exactly one
    // CTA, so the slots need no clearing); the caller owns the workspace, one per stream
    const int64_t n = (int64_t)g->Cout * g->ntaps * g->Cin;
    if (ws_need) { *ws_need = split * n; return 0; }
    if (ws_floats < split * n) return PXL_ERR_BAD_ARG;

    CUtensorMap mDy, mDyLo, mX, mXLo;
    int rc = make_act_map_strided(&mDy, dy_hi, g->ldo, mapW, mapH, mapN, p.BW, p.BH, 1, f16);
    if (rc) return rc;
    rc = make_act_map_strided(&mX, in_hi, g->Cin, inW, inH, mapN, p.BW, p.BH, g->mul, f16);
    if (rc) return rc;
    if (nsplit == 3 && !inkernel) {
        rc = make_act_map_strided(&mDyLo, dy_lo, g->ldo, mapW, mapH, mapN, p.BW, p.BH, 1, f16);
        if (rc) return rc;
        rc = make_act_map_strided(&mXLo, in_lo, g->Cin, inW, inH, mapN, p.BW, p.BH, g->mul, f16);
        if (rc) return rc;
    } else { mDyLo = mDy; mXLo = mX; }
    if (!g_err_flag) {
        cudaError_t e = cudaMalloc(&g_err_flag, sizeof(int));
        if (e != cudaSuccess) return (int)e;
        e = cudaMemset(g_err_flag, 0, sizeof(int));
        if (e != cudaSuccess) return (int)e;
    }
    static bool attr = false;
    if (!attr) {
        cudaError_t e = cudaFuncSetAttribute(conv_wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 2048);
        if (e != cudaSuccess) return (int)e;
        attr = true;
    }
    const size_t smem = (size_t)p.stages * stage_bytes + 1024;
    // the slots [split][Cout][taps][Cin] as a 4-D tensor (Cin, taps, Cout, split): box {32, 1, 128, 1}, 128-byte swizzle
    static int cfg_wg_red = -1;
    if (cfg_wg_red < 0) { const char* e = getenv("PXL_WG_TMA_REDUCE"); cfg_wg_red = e ? atoi(e) : 1; }
    CUtensorMap mDw = mDy;
    p.tma_red = 0;
    if (cfg_wg_red && (g->Cin % 4) == 0 && ((uintptr_t)ws % 16) == 0 && (size_t)p.stages * stage_bytes >= 32768) {
        EncodeTiledFn enc = get_encode();
        cuuint64_t dims[4] = {(cuuint64_t)g->Cin, (cuuint64_t)g->ntaps, (cuuint64_t)g->Cout, (cuuint64_t)split};
        cuuint64_t strides[3] = {(cuuint64_t)g->Cin * 4, (cuuint64_t)g->ntaps * g->Cin * 4, (cuuint64_t)n * 4};
        cuuint32_t box[4] = {32, 1, 128, 1};
        cuuint32_t es[4] = {1, 1, 1, 1};
        if (enc && enc(&mDw, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void*)ws, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                       CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS)
            p.tma_red = 1;
    }
    dim3 grid((unsigned)(tiles_co * p.tiles_ci), (unsigned)g->ntaps, (unsigned)split);
    cudaError_t le = pxl_launch_pdl(conv_wgrad_tc_kernel, grid, dim3(inkernel ? 320 : 192), smem, (cudaStream_t)stream, mDy, mDyLo, mX, mXLo,
                                    mDw, p, ws, g_err_flag, oscale_ptr);
    if (le != cudaSuccess) return (int)le;
    PXL_CHECK_LAUNCH();
    int blocks = (int)(pxl_cdiv(n, 256) < PXL_NUM_SMS * 8 ? pxl_cdiv(n, 256) : PXL_NUM_SMS * 8);
    le = pxl_launch_pdl(wg_slot_sum_kernel, dim3(blocks), dim3(256), 0, (cudaStream_t)stream,
                        (const float*)ws, dw, n, (int)split);
    if (le != cudaSuccess) return (int)le;
    PXL_CHECK_LAUNCH();
    return 0;
}

extern "C" int pxl_conv_wgrad_tc_impl(const pxl_conv_geom* g, const int* taps, const float* in, const float* dy,
                                      float* dw, void* stream) {
    if (!g) return PXL_ERR_BAD_ARG;
    if (g->precision == 2) return PXL_ERR_UNSUPPORTED;     // needs split operands: pxl_conv_wgrad_tc_launch
    // this entry point takes no workspace: a stream-ordered one for this launch only
    const int64_t need = pxl_conv_wgrad_workspace_floats(g, taps);
    if (need < 0) return (int)need;
    float* ws = nullptr;
    cudaError_t e = cudaMallocAsync((void**)&ws, (size_t)need * sizeof(float), (cudaStream_t)stream);
    if (e != cudaSuccess) return (int)e;
    const int rc = pxl_conv_wgrad_tc_launch(g, taps, in, nullptr, dy, nullptr, dw, ws, need, stream);
    e = cudaFreeAsync(ws, (cudaStream_t)stream);
    return rc ? rc : (int)e;
}
