// wgrad_kernels.cu -- weight gradient of the policy's 3x3 convolutions on the 5th-generation tensor
// cores (tcgen05 + TMEM), operands staged by TMA.
//
// The PPO update spends more time in the weight gradient of conv4 (128 -> 128 channels on the 15x10
// board, inversus_rl/policies.py:40-43) than in any other kernel: the library's implicit-GEMM wgrad
// reaches 0.24 PFLOP/s there (profiles/r2_explore_policy.txt) because the output is tiny
// (128 x 1152) and the reduction runs over batch x positions. This kernel is built for exactly that
// shape:
//
//   dW[co][ky][kx][ci] = sum over (n, y, x) of dY[n, y, x, co] * X[n, y + ky - 1, x + kx - 1, ci]
//
//   * A CTA owns one kernel column kx and a contiguous range of samples. Its three accumulators
//     (ky = 0, 1, 2), each 128 (co) x CIN fp32, live in TMEM for the whole kernel.
//   * Per sample, TMA brings dY as a [10 x 16] position box and X as a [12 x 16] box shifted by
//     (kx - 1, -1): the boxes hang over the 15 x 10 board and TMA zero-fills what is outside, which
//     is exactly the convolution's zero padding. Row r of the dY box and row r + 16*ky of the X box
//     then face each other for tap (ky, kx), so the three taps are three MMAs over the SAME shared
//     memory tile at three 2 KB-aligned offsets -- no im2col, no shifted copies.
//   * Both operands are "MN-major" for the MMA (channels are contiguous in memory, positions are
//     the reduction dimension): 128-byte-swizzled rows of 64 channels, 8 rows per 1 KB atom.
//   * warp 0 = TMA producer, warp 1 = MMA issuer (one elected lane), warps 2-5 = epilogue, which
//     runs once: TMEM -> registers -> per-CTA fp32 partials; a small kernel sums the partials.
//   * conv2 (32 -> 64 channels) uses the same kernel with M = 64, N = 32: all nine taps fit one CTA's
//     TMEM (9 x 32 columns), so dY is loaded once per sample and X as three kx-shifted boxes of
//     64-byte rows (64-byte swizzle).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "../../include/inversus_b200.h"
#include "launch_common.h"

namespace {

constexpr int kBoxW = 16;                 // 15 board columns + 1 (zero-filled or neighbour halo)
constexpr int kRowsA = 10 * kBoxW;        // 160 positions of dY per sample (K of the GEMM)
constexpr int kRowsB = 12 * kBoxW;        // 192 positions of X per sample: rows y = -1 .. 10
constexpr int kThreads = 192;
constexpr uint32_t kTmemCols = 512;

// Shape of one instantiation. NKX = kernel columns handled by one CTA (3 ky each).
template <int COUT, int CIN, int NKX>
struct Shape {
    static_assert((COUT == 128 || COUT == 64) && (CIN == 128 || CIN == 64 || CIN == 32) && NKX >= 1 && NKX <= 3, "unsupported shape");
    static constexpr int kAHalves = COUT / 64;               // 64-channel column blocks of the dY tile
    static constexpr int kHalfA = kRowsA * 128;              // bytes of one block (128-byte rows)
    static constexpr int kBRowBytes = CIN >= 64 ? 128 : 64;  // X rows: 64 or 32 channels per swizzled row
    static constexpr int kBHalves = CIN >= 64 ? CIN / 64 : 1;
    static constexpr int kHalfB = kRowsB * kBRowBytes;
    static constexpr int kBBox = kBHalves * kHalfB;          // one kx-shifted X tile
    static constexpr int kStageBytes = kAHalves * kHalfA + NKX * kBBox;
    static constexpr int kStages = kStageBytes > 80 * 1024 ? 2 : 3;
    static constexpr uint32_t kBLayout = CIN >= 64 ? 2u : 4u; // UMMA layout type: SWIZZLE_128B / SWIZZLE_64B
    static constexpr uint32_t kBSbo = CIN >= 64 ? 1024u : 512u; // bytes between 8-row groups
    static_assert(NKX * 3 * CIN <= (int)kTmemCols, "accumulators exceed TMEM");
};

__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    uint32_t done = 0;
    for (uint32_t spins = 0; !done; ++spins) {
        asm volatile("{\n\t.reg .pred p;\n\t"
                     "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                     "selp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done)
                     : "r"(bar), "r"(parity)
                     : "memory");
        if (spins > (1u << 26)) __trap(); // a protocol error surfaces as a CUDA error, never as a hung GPU
    }
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap *map, int c0, int c1, int c2, int c3,
                                            uint32_t bar)
{
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
                 ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(bar)
                 : "memory");
}
// shared-memory matrix descriptor, MN-major, 128-byte swizzle (cute::UMMA::SmemDescriptor):
// start address, leading-dimension byte offset (between 64-element column blocks), stride byte
// offset (between 8-row groups along K), version 1, layout type 2 = SWIZZLE_128B
__device__ __forceinline__ uint64_t umma_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout = 2u)
{
    return (uint64_t)((addr & 0x3FFFFu) >> 4) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46) | ((uint64_t)layout << 61);
}
// instruction descriptor (cute::UMMA::InstrDescriptor): D = f32, A = B = bf16, both MN-major
__host__ __device__ constexpr uint32_t umma_idesc(int M, int N)
{
    return (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(N >> 3) << 17) |
           ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
                 : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// partials: [parts][ky][kx][co][CIN] fp32
// One CTA: kernel columns [kx0, kx0 + NKX), samples [part * per_part, ...). STAGES ring stages of
// Shape<COUT, CIN, NKX>::kStageBytes each must fit the dynamic shared memory of the launch.
template <int COUT, int CIN, int NKX, int STAGES>
__device__ __forceinline__ void wgrad_cta(const CUtensorMap &map_dy, const CUtensorMap &map_x, int64_t B, int kx0, int part,
                                          int per_part, float *__restrict__ partials)
{
    typedef Shape<COUT, CIN, NKX> S;
    constexpr int SB = S::kStageBytes;
    extern __shared__ __align__(1024) unsigned char smem[];
    __shared__ __align__(8) uint64_t s_full[STAGES], s_empty[STAGES], s_done;
    __shared__ uint32_t s_tmem;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t first = (int64_t)part * per_part;
    const int64_t last = first + per_part < B ? first + per_part : B;
    const int nsamp = last > first ? (int)(last - first) : 0;
    const uint32_t base = (smem_addr(smem) + 1023u) & ~1023u; // TMA swizzle atoms are 1 KB aligned

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(smem_addr(&s_full[s]), 1);
            mbar_init(smem_addr(&s_empty[s]), 1);
        }
        mbar_init(smem_addr(&s_done), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) { // TMEM: the NKX x 3 accumulators (CIN columns each) in one 512-column allocation
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_addr(&s_tmem)), "n"(kTmemCols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = s_tmem;

    if (warp == 0) {
        // ================================================================= TMA producer
        if (lane == 0) {
            for (int i = 0; i < nsamp; ++i) {
                const int st = i % STAGES;
                if (i >= STAGES) mbar_wait(smem_addr(&s_empty[st]), (uint32_t)((i / STAGES) - 1) & 1u);
                const uint32_t bar = smem_addr(&s_full[st]);
                const uint32_t a0 = base + (uint32_t)st * SB, b0 = a0 + S::kAHalves * S::kHalfA;
                mbar_expect_tx(bar, (uint32_t)SB);
                const int n = (int)(first + i);
#pragma unroll
                for (int h = 0; h < S::kAHalves; ++h) tma_load_4d(a0 + h * S::kHalfA, &map_dy, 64 * h, 0, 0, n, bar);
#pragma unroll
                for (int k = 0; k < NKX; ++k)
#pragma unroll
                    for (int h = 0; h < S::kBHalves; ++h)
                        tma_load_4d(b0 + k * S::kBBox + h * S::kHalfB, &map_x, 64 * h, kx0 + k - 1, -1, n, bar);
            }
        }
    } else if (warp == 1) {
        // ================================================================= MMA issuer
        if (lane == 0) {
            // With several kernel columns per CTA (conv2) their X boxes sit side by side in the MMA's N
            // dimension: one MMA of N = NKX * CIN per kernel row, the column blocks LBO = one box apart.
            // Accumulator of kernel row ky: columns [ky * NKX * CIN, +NKX * CIN), kx-major inside.
            constexpr uint32_t idesc = umma_idesc(COUT, NKX * CIN);
            constexpr uint32_t lbo_b = NKX > 1 ? (uint32_t)S::kBBox : (uint32_t)S::kHalfB;
            static_assert(NKX == 1 || S::kBHalves == 1, "merged kernel columns need one column block per box");
            for (int i = 0; i < nsamp; ++i) {
                const int st = i % STAGES;
                mbar_wait(smem_addr(&s_full[st]), (uint32_t)(i / STAGES) & 1u);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t a0 = base + (uint32_t)st * SB, b0 = a0 + S::kAHalves * S::kHalfA;
                // 30 MMAs per sample, 16 positions (one board row) each. Order measured per shape
                // (profiles/r2_wgrad.txt): row-by-row per accumulator for the large shapes (interleaving
                // cost conv3 20 %), accumulators interleaved for conv2's small MMAs.
#pragma unroll
                for (int t = 0; t < 3 * (kRowsA / 16); ++t) {
                    constexpr bool kInterleave = CIN < 64;
                    const int ky = kInterleave ? t % 3 : t / (kRowsA / 16), kk = kInterleave ? t / 3 : t % (kRowsA / 16);
                    const uint64_t da = umma_desc(a0 + kk * 16 * 128, S::kHalfA, 1024);
                    const uint64_t db = umma_desc(b0 + (ky * 16 + kk * 16) * S::kBRowBytes, lbo_b, S::kBSbo, S::kBLayout);
                    umma_f16(tmem + ky * NKX * CIN, da, db, idesc, (i > 0 || kk > 0) ? 1u : 0u);
                }
                umma_commit(smem_addr(&s_empty[st])); // the stage is free once these MMAs have read it
            }
            umma_commit(smem_addr(&s_done));
        }
    } else {
        // ================================================================= epilogue (once)
        // TMEM lane quadrant q belongs to warp q (mod 4). M = 128: accumulator row = lane index;
        // M = 64: rows 16q .. 16q+15 sit in the first 16 lanes of quadrant q.
        const int q = warp & 3;
        const int co = COUT == 128 ? q * 32 + lane : q * 16 + lane;
        const bool row_ok = COUT == 128 || lane < 16;
        if (nsamp > 0) {
            mbar_wait(smem_addr(&s_done), 0);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        }
#pragma unroll 1
        for (int t = 0; t < NKX * 3; ++t) {
            const int k = t / 3, ky = t % 3;
            float *out = partials + ((((size_t)part * 3 + ky) * 3 + (kx0 + k)) * COUT + co) * CIN;
#pragma unroll 1
            for (int c = 0; c < CIN / 32; ++c) {
                uint32_t v[32];
                if (nsamp > 0) {
                    const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)((ky * NKX + k) * CIN + c * 32);
                    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                                   "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                                   "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                                 : "r"(taddr));
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = 0u;
                }
                if (row_ok) {
                    uint4 *o4 = reinterpret_cast<uint4 *>(out + c * 32);
#pragma unroll
                    for (int j = 0; j < 8; ++j) o4[j] = make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(kTmemCols));
}

// Uniform grid: 3 / NKX CTAs per sample range, one per group of kernel columns.
template <int COUT, int CIN, int NKX>
__global__ void __launch_bounds__(kThreads, 1)
conv3x3_wgrad_kernel(const __grid_constant__ CUtensorMap map_dy, const __grid_constant__ CUtensorMap map_x, int64_t B,
                     int per_part, float *__restrict__ partials)
{
    constexpr int KXG = 3 / NKX;
    wgrad_cta<COUT, CIN, NKX, Shape<COUT, CIN, NKX>::kStages>(map_dy, map_x, B, (blockIdx.x % KXG) * NKX, blockIdx.x / KXG,
                                                             per_part, partials);
}

__global__ void wgrad_reduce_kernel(const float *__restrict__ partials, int parts, int cin, int cout, float *__restrict__ dw)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int total = 9 * cout * cin;
    if (i >= total) return;
    const int ci = i % cin, co = (i / cin) % cout, tap = i / (cin * cout);
    float a = 0.f;
#pragma unroll 8
    for (int p = 0; p < parts; ++p) a += partials[(size_t)p * total + i];
    dw[((size_t)co * 9 + tap) * cin + ci] = a;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn()
{
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// [B][10][15][C] bf16 channels-last activations as a 4-D tensor; box = 64 channels x 16 x rows x 1 sample
bool make_map(CUtensorMap *map, const void *ptr, int64_t B, int C, int box_rows)
{
    EncodeTiledFn enc = encode_fn();
    if (!enc) return false;
    const int inner = C >= 64 ? 64 : C; // channels per swizzled row: 128-byte rows, or 64-byte rows for C = 32
    const cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)INV_BOARD_W, (cuuint64_t)INV_BOARD_H, (cuuint64_t)B};
    const cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)C * 2 * INV_BOARD_W, (cuuint64_t)C * 2 * INV_BOARD_W * INV_BOARD_H};
    const cuuint32_t box[4] = {(cuuint32_t)inner, (cuuint32_t)kBoxW, (cuuint32_t)box_rows, 1};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    return enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void *>(ptr), dims, strides, box, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, inner == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
               CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int COUT, int CIN, int NKX>
int launch_wgrad(const void *dy, const void *x, int64_t B, float *dw, float *partials, cudaStream_t st)
{
    const char *who = "inv_conv3x3_wgrad";
    typedef Shape<COUT, CIN, NKX> S;
    CUtensorMap map_dy, map_x;
    if (!make_map(&map_dy, dy, B, COUT, 10) || !make_map(&map_x, x, B, CIN, 12))
        return inv_host::set_error(INV_ERR_CUDA, who, "cuTensorMapEncodeTiled failed");
    constexpr size_t smem = (size_t)S::kStages * S::kStageBytes + 1024;
    auto kern = conv3x3_wgrad_kernel<COUT, CIN, NKX>;
    if (inv_host::allow_dynamic_smem((const void *)kern, smem) != cudaSuccess) return inv_host::launch_status(who);
    constexpr int KXG = 3 / NKX;
    int parts = inv_host::sm_count() / KXG;
    if (parts > B) parts = (int)B;
    if (parts < 1) parts = 1;
    const int per_part = (int)((B + parts - 1) / parts);
    kern<<<KXG * parts, kThreads, smem, st>>>(map_dy, map_x, B, per_part, partials);
    if (int rc = inv_host::launch_status(who)) return rc;
    const int total = 9 * COUT * CIN;
    wgrad_reduce_kernel<<<(total + 255) / 256, 256, 0, st>>>(partials, parts, CIN, COUT, dw);
    return inv_host::launch_status(who);
}

} // namespace

extern "C" {

int64_t inv_conv3x3_wgrad_scratch_floats(int32_t cin, int32_t cout)
{
    const int kxg = cin == 128 ? 3 : 1; // conv4: three CTAs per sample range; conv2 / conv3: up to one part per SM
    return (int64_t)(inv_host::sm_count() / kxg) * 9 * cout * cin;
}

int inv_conv3x3_wgrad(const void *dy, const void *x, int64_t B, int32_t cin, int32_t cout, float *dw, float *partials,
                      void *stream)
{
    const char *who = "inv_conv3x3_wgrad";
    if (int rc = inv_host::require_sm100(who)) return rc;
    if (!dy || !x || !dw || !partials || B <= 0) return inv_host::set_error(INV_ERR_INVALID_ARG, who, "null pointer or B <= 0");
    if (((uintptr_t)dy | (uintptr_t)x) & 15u)
        return inv_host::set_error(INV_ERR_INVALID_ARG, who, "dy and x must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    if (cout == 128 && cin == 128) return launch_wgrad<128, 128, 1>(dy, x, B, dw, partials, st);
    if (cout == 128 && cin == 64) return launch_wgrad<128, 64, 1>(dy, x, B, dw, partials, st);
    if (cout == 64 && cin == 32) return launch_wgrad<64, 32, 3>(dy, x, B, dw, partials, st);
    return inv_host::set_error(INV_ERR_INVALID_ARG, who, "(cout, cin) must be (128, 128), (128, 64) or (64, 32)");
}

} // extern "C"
