// policy_kernels.cu -- fused LayerNorm(+residual)+ReLU for the policy's channels-last bf16 path.
//
// The policy CNN (inversus_rl/policies.py:27-45, :94-100) applies LayerNorm over the whole
// [C,H,W] feature map after every convolution, then ReLU (and a residual add before the fourth).
// The contractions stay in cuDNN/cuBLAS; this file fuses the memory-bound glue between them:
//
//   forward   y = relu( LN(x [+ res]) * gamma + beta )          one read of x (and res), one write of y
//   backward  dx = LN'(relu'(dy)) ; dgamma, dbeta               one read of dy, x (and res), one write of dx
//
// Layout: a sample is D = H*W*C contiguous bf16 values in HWC order (the memory of a
// channels-last tensor); gamma/beta are [D] bf16 in the same order. Statistics and all arithmetic
// are fp32. Both kernels are persistent. The forward walks over samples with one CTA per sample.
// The backward (round 2) splits the FEATURE dimension over a thread-block cluster: each of the
// 2/4/8 CTAs of a cluster owns D/CS columns, one 8-column vector per thread, so gamma/beta and the
// dgamma/dbeta/dbias accumulators of those columns live in registers for the whole kernel (the
// round-1 kernel kept 2*D floats per CTA in shared memory, which pinned it at one CTA per SM and
// 0.24-0.41 of the HBM peak). The two per-sample row sums of the LayerNorm backward are combined
// across the cluster through distributed shared memory, two samples per cluster barrier. Partials
// are written per cluster and reduced by a second small kernel -- deterministic, no atomics.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include <type_traits>

#include "../../include/inversus_b200.h"
#include "launch_common.h"

namespace {

constexpr int kLnThreads = 512;

__device__ __forceinline__ void unpack8(const uint4 &v, float (&f)[8])
{
    const __nv_bfloat162 *h = reinterpret_cast<const __nv_bfloat162 *>(&v);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 t = __bfloat1622float2(h[i]);
        f[2 * i] = t.x;
        f[2 * i + 1] = t.y;
    }
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8])
{
    uint4 v;
    __nv_bfloat162 *h = reinterpret_cast<__nv_bfloat162 *>(&v);
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
    return v;
}

// ---- packed fp32x2 arithmetic (FFMA2 / FADD2 / FMUL2 on sm_100): two lanes per issue slot. The
// LayerNorm backward is bound by instruction issue, not by HBM, so this is where its time goes.
typedef unsigned long long f2;
__device__ __forceinline__ f2 f2_make(float lo, float hi)
{
    f2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void f2_split(f2 v, float &lo, float &hi)
{
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f2 f2_fma(f2 a, f2 b, f2 c)
{
    f2 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ f2 f2_add(f2 a, f2 b)
{
    f2 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f2 f2_mul(f2 a, f2 b)
{
    f2 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
// two bf16 in one 32-bit word -> two fp32
__device__ __forceinline__ f2 bf2_to_f2(uint32_t w) { return f2_make(__uint_as_float(w << 16), __uint_as_float(w & 0xFFFF0000u)); }
__device__ __forceinline__ uint32_t f2_to_bf2(f2 v)
{
    float lo, hi;
    f2_split(v, lo, hi);
    const __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<const uint32_t *>(&h);
}
__device__ __forceinline__ uint32_t word_of(const uint4 &v, int p) { return p == 0 ? v.x : p == 1 ? v.y : p == 2 ? v.z : v.w; }

// sum of (a, b) over the CTA; result broadcast to every thread
__device__ __forceinline__ float2 block_sum2(float a, float b, float2 *scratch)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __syncthreads(); // scratch may still be read from the previous call
    if (lane == 0) scratch[warp] = make_float2(a, b);
    __syncthreads();
    float2 t = lane < (kLnThreads / 32) ? scratch[lane] : make_float2(0.f, 0.f);
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) {
        t.x += __shfl_xor_sync(0xffffffffu, t.x, o);
        t.y += __shfl_xor_sync(0xffffffffu, t.y, o);
    }
    return make_float2(__shfl_sync(0xffffffffu, t.x, 0), __shfl_sync(0xffffffffu, t.y, 0));
}

// Two CTAs per SM (<= 64 registers at 512 threads): while one CTA sits in its block reduction the
// other streams. gamma/beta are re-read per sample from L1/L2 (caching them in registers would not
// fit the 64-register budget together with the packed inputs).
template <int MAXV, bool HAS_RES>
__global__ void __launch_bounds__(kLnThreads, 2)
ln_relu_fwd_kernel(const uint4 *__restrict__ x, const uint4 *__restrict__ res, const uint4 *__restrict__ cbias,
                   int cvecs, const uint4 *__restrict__ gamma, const uint4 *__restrict__ beta, int64_t B, int nvec,
                   float eps, uint4 *__restrict__ y, float *__restrict__ mean_out, float *__restrict__ rstd_out)
{
    __shared__ float2 scratch[kLnThreads / 32];
    const int tid = threadIdx.x;
    // per-channel convolution bias, folded in here so cuDNN runs bias-free: the element (i*8 + j) of
    // an HWC sample belongs to channel ((i mod C/8)*8 + j), and since kLnThreads is a multiple of
    // C/8 every vector of a thread sees the same 8 channels -> four register pairs per thread
    const uint4 cbv = cbias ? cbias[tid % cvecs] : make_uint4(0u, 0u, 0u, 0u);
    f2 cb2[4];
#pragma unroll
    for (int p = 0; p < 4; ++p) cb2[p] = bf2_to_f2(word_of(cbv, p));
    constexpr bool kCacheGB = MAXV <= 1;
    uint4 g[kCacheGB ? MAXV : 1], bt[kCacheGB ? MAXV : 1];
    if (kCacheGB) {
#pragma unroll
        for (int k = 0; k < MAXV; ++k) {
            const int i = k * kLnThreads + tid;
            if (i < nvec) { g[k] = gamma[i]; bt[k] = beta[i]; }
        }
    }
    const float inv_d = 1.0f / (float)(nvec * 8);
    // All arithmetic is packed fp32x2 (FFMA2 / FADD2 / FMUL2): at ~10 instructions per element instead
    // of ~17 the kernel stops being bound by instruction issue.
    for (int64_t s = blockIdx.x; s < B; s += gridDim.x) {
        const uint4 *xs = x + s * nvec;
        uint4 xv[MAXV], rv[HAS_RES ? MAXV : 1]; // inputs stay packed (bf16) between the two passes
#pragma unroll
        for (int k = 0; k < MAXV; ++k) {
            const int i = k * kLnThreads + tid;
            if (i < nvec) {
                xv[k] = xs[i];
                if (HAS_RES) rv[k] = res[s * nvec + i];
            }
        }
        f2 sum2 = f2_make(0.f, 0.f), sq2 = f2_make(0.f, 0.f);
#pragma unroll
        for (int k = 0; k < MAXV; ++k) {
            const int i = k * kLnThreads + tid;
            if (i < nvec) {
#pragma unroll
                for (int p = 0; p < 4; ++p) {
                    f2 z = f2_add(bf2_to_f2(word_of(xv[k], p)), cb2[p]);
                    if (HAS_RES) z = f2_add(z, bf2_to_f2(word_of(rv[k], p)));
                    sum2 = f2_add(sum2, z);
                    sq2 = f2_fma(z, z, sq2);
                }
            }
        }
        float s0, s1, q0, q1;
        f2_split(sum2, s0, s1);
        f2_split(sq2, q0, q1);
        const float2 t = block_sum2(s0 + s1, q0 + q1, scratch);
        const float mean = t.x * inv_d;
        const float var = fmaxf(t.y * inv_d - mean * mean, 0.f);
        const float rstd = rsqrtf(var + eps);
        if (tid == 0) { mean_out[s] = mean; rstd_out[s] = rstd; }
        const f2 rs2 = f2_make(rstd, rstd), nm2 = f2_make(-mean, -mean);
#pragma unroll
        for (int k = 0; k < MAXV; ++k) {
            const int i = k * kLnThreads + tid;
            if (i < nvec) {
                const uint4 gk = kCacheGB ? g[k] : gamma[i], bk = kCacheGB ? bt[k] : beta[i];
                uint32_t ow[4];
#pragma unroll
                for (int p = 0; p < 4; ++p) {
                    f2 z = f2_add(bf2_to_f2(word_of(xv[k], p)), cb2[p]);
                    if (HAS_RES) z = f2_add(z, bf2_to_f2(word_of(rv[k], p)));
                    // (z - mean) * rstd * gamma + beta  =  z * (rstd*gamma) + (beta - mean*rstd*gamma)
                    const f2 sg = f2_mul(bf2_to_f2(word_of(gk, p)), rs2);
                    const f2 o = f2_fma(z, sg, f2_fma(sg, nm2, bf2_to_f2(word_of(bk, p))));
                    float o0, o1;
                    f2_split(o, o0, o1);
                    const __nv_bfloat162 h = __floats2bfloat162_rn(fmaxf(o0, 0.f), fmaxf(o1, 0.f));
                    ow[p] = *reinterpret_cast<const uint32_t *>(&h);
                }
                y[s * nvec + i] = make_uint4(ow[0], ow[1], ow[2], ow[3]);
            }
        }
    }
}

// dynamic smem: float acc[2][nvec*8]  (dgamma, dbeta of this CTA)
template <int MAXV, bool HAS_RES>
__global__ void __launch_bounds__(kLnThreads)
ln_relu_bwd_kernel(const uint4 *__restrict__ dy, const uint4 *__restrict__ x, const uint4 *__restrict__ res,
                   const uint4 *__restrict__ cbias, int cvecs, const uint4 *__restrict__ gamma,
                   const uint4 *__restrict__ beta, const float *__restrict__ mean_in,
                   const float *__restrict__ rstd_in, int64_t B, int nvec, uint4 *__restrict__ dx,
                   float *__restrict__ partials)
{
    extern __shared__ float acc[];
    __shared__ float2 scratch[kLnThreads / 32];
    const int tid = threadIdx.x;
    const int D = nvec * 8;
    float cb[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (cbias) unpack8(cbias[tid % cvecs], cb);
    float db[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}; // d(conv bias) of this thread's 8 channels
    for (int i = tid; i < 2 * D; i += kLnThreads) acc[i] = 0.f;
    __syncthreads();
    // gamma/beta live in registers across samples when the slice is small; for the two 19200-wide
    // layers (MAXV >= 4) that would spill, so they are re-read per sample (they stay L1/L2-resident)
    constexpr bool kCacheGB = MAXV <= 3;
    uint4 g[kCacheGB ? MAXV : 1], bt[kCacheGB ? MAXV : 1];
    if (kCacheGB) {
#pragma unroll
        for (int k = 0; k < MAXV; ++k) {
            const int i = k * kLnThreads + tid;
            if (i < nvec) { g[k] = gamma[i]; bt[k] = beta[i]; }
        }
    }
    const float inv_d = 1.0f / (float)D;
    // from here on each thread only touches its own accumulator slots: no barrier needed around acc
    for (int64_t s = blockIdx.x; s < B; s += gridDim.x) {
        const float mean = mean_in[s], rstd = rstd_in[s];
        // issue every global load of this sample before touching the data (memory-level
        // parallelism); the packed inputs stay in registers for both passes
        uint4 xv[MAXV], dv[MAXV], rv[HAS_RES ? MAXV : 1];
#pragma unroll
        for (int k = 0; k < MAXV; ++k) {
            const int i = k * kLnThreads + tid;
            if (i < nvec) {
                xv[k] = x[s * nvec + i];
                dv[k] = dy[s * nvec + i];
                if (HAS_RES) rv[k] = res[s * nvec + i];
            }
        }
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int k = 0; k < MAXV; ++k) {
            const int i = k * kLnThreads + tid;
            if (i < nvec) {
                float z[8], d[8], gf[8], bf[8];
                unpack8(xv[k], z);
#pragma unroll
                for (int j = 0; j < 8; ++j) z[j] += cb[j];
                if (HAS_RES) {
                    float r[8];
                    unpack8(rv[k], r);
#pragma unroll
                    for (int j = 0; j < 8; ++j) z[j] += r[j];
                }
                unpack8(dv[k], d);
                unpack8(kCacheGB ? g[k] : gamma[i], gf);
                unpack8(kCacheGB ? bt[k] : beta[i], bf);
                // accumulators are element-major (acc[j*nvec + i]) so that the 32 lanes of a warp
                // hit 32 different banks; i*8 + j would be an 8-way conflict on every access
                float *ag = acc + i, *ab = acc + D + i;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float h = (z[j] - mean) * rstd;
                    const float gy = (h * gf[j] + bf[j] > 0.f) ? d[j] : 0.f; // relu'
                    ag[j * nvec] += gy * h;
                    ab[j * nvec] += gy;
                    const float w = gy * gf[j];
                    s1 += w;
                    s2 += w * h;
                }
            }
        }
        const float2 t = block_sum2(s1, s2, scratch);
        const float m1 = t.x * inv_d, m2 = t.y * inv_d;
#pragma unroll
        for (int k = 0; k < MAXV; ++k) {
            const int i = k * kLnThreads + tid;
            if (i < nvec) {
                float z[8], d[8], gf[8], bf[8], o[8];
                unpack8(xv[k], z);
#pragma unroll
                for (int j = 0; j < 8; ++j) z[j] += cb[j];
                if (HAS_RES) {
                    float r[8];
                    unpack8(rv[k], r);
#pragma unroll
                    for (int j = 0; j < 8; ++j) z[j] += r[j];
                }
                unpack8(dv[k], d);
                unpack8(kCacheGB ? g[k] : gamma[i], gf);
                unpack8(kCacheGB ? bt[k] : beta[i], bf);
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float h = (z[j] - mean) * rstd;
                    const float w = (h * gf[j] + bf[j] > 0.f) ? d[j] * gf[j] : 0.f;
                    o[j] = rstd * (w - m1 - h * m2);
                    db[j] += o[j];
                }
                dx[s * nvec + i] = pack8(o);
            }
        }
    }
    const int C = cvecs * 8;
    float *out = partials + (size_t)blockIdx.x * (2 * D + C);
    for (int k = 0; k < MAXV; ++k) {
        const int i = k * kLnThreads + tid;
        if (i < nvec) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                out[i * 8 + j] = acc[j * nvec + i];
                out[D + i * 8 + j] = acc[D + j * nvec + i];
            }
        }
    }
    // d(conv bias): every thread holds sums for channels (tid % cvecs)*8 .. +7; fold the
    // kLnThreads / cvecs threads of each channel group through shared memory (acc is free now)
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[tid * 8 + j] = db[j];
    __syncthreads();
    if (tid < C) {
        const int grp = tid >> 3, j = tid & 7;
        float sum = 0.f;
        for (int t = grp; t < kLnThreads; t += cvecs) sum += acc[t * 8 + j];
        out[2 * D + tid] = sum;
    }
}

__global__ void reduce_partials_kernel(const float *__restrict__ partials, int nparts, int width,
                                       float *__restrict__ dgamma, float *__restrict__ dbeta,
                                       float *__restrict__ dcbias, int D)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= width) return;
    float s = 0.f;
    for (int p = 0; p < nparts; ++p) s += partials[(size_t)p * width + i];
    if (i < D) dgamma[i] = s;
    else if (i < 2 * D) dbeta[i - D] = s;
    else if (dcbias) dcbias[i - 2 * D] = s;
}

// ---- distributed-shared-memory helpers (raw PTX: the cooperative-groups cluster.sync() compiles
// to MEMBAR.ALL.GPU + an L1 invalidate, far too heavy to sit in a streaming loop) ----
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t map_to_rank(uint32_t local_smem_addr, uint32_t rank)
{
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// a 4-byte store into a peer CTA's shared memory that completes `bytes` on the peer's mbarrier
__device__ __forceinline__ void st_async_f32(uint32_t remote_addr, float v, uint32_t remote_bar)
{
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.f32 [%0], %1, [%2];" ::"r"(remote_addr),
                 "f"(v), "r"(remote_bar)
                 : "memory");
}
// Spin until the barrier's phase with the given parity has completed; traps instead of hanging.
// Default (CTA-scope) acquire on purpose: what is waited for -- TMA bulk copies and the peers'
// st.async words -- lands in THIS CTA's shared memory through the async proxy and is published by the
// barrier's own transaction count. A cluster-scope acquire makes ptxas emit CCTL.IVALL (an L1
// invalidate) after every wait: 26 % of the stall samples of this kernel in the first ncu capture.
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
        if (spins > (1u << 26)) __trap(); // a protocol error must surface as a CUDA error, never as a hung GPU
    }
}
__device__ __forceinline__ void cluster_sync_all()
{
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// 1-D bulk copy global -> this CTA's shared memory, completion counted in bytes on an mbarrier (TMA)
__device__ __forceinline__ void bulk_load(uint32_t dst_smem, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}

// ------------------------------------------------------------------------------------------------
// Clustered backward (round 2). Grid = nclusters * CS CTAs of kBwdThreads threads; cluster c walks
// over sample groups c, c + nclusters, ... of S samples each. Thread `slot = rank * kBwdThreads +
// tid` owns columns [8*slot, 8*slot + 8) of every sample: gamma/beta/conv-bias and the three
// gradient accumulators of those columns are registers for the whole kernel.
//
// Per group of S samples:
//   pass 1   reads the group's x / dy / residual slices from shared memory, where TMA bulk copies put
//            them one to two groups ahead (2-stage ring), forms h and w = relu'(.) * dy * gamma --
//            kept in registers -- accumulates dgamma / dbeta and the CTA's share of the row sums;
//   exchange the 2*S sums go to every CTA of the cluster with st.async into distributed shared
//            memory, counted by the receiver's mbarrier (no cluster barrier, no fence in the loop);
//            the other CTA resident on the SM works while this one waits;
//   pass 2   dx = rstd * (w - m1 - h * m2) from the registers, d(bias) accumulation, 16-byte stores.
// All arithmetic is packed fp32x2. One __syncthreads per group.
// partials layout (floats): [nclusters][2][D] (dgamma, dbeta) followed by [grid][C] (d conv bias).
constexpr int kBwdThreads = 320;
constexpr int kMaxCluster = 8;
constexpr int kBwdStages = 2;
constexpr int kSumSlots = 2; // a peer is at most one group ahead of the slowest reader (see below)

template <int S, bool HAS_RES>
constexpr size_t bwd_cluster_smem() { return (size_t)kBwdStages * S * (HAS_RES ? 3 : 2) * kBwdThreads * 16; }

template <int S, bool HAS_RES>
__global__ void __launch_bounds__(kBwdThreads, 2)
ln_relu_bwd_cluster_kernel(const uint4 *__restrict__ dy, const uint4 *__restrict__ x, const uint4 *__restrict__ res,
                           const uint4 *__restrict__ cbias, int cvecs, const uint4 *__restrict__ gamma,
                           const uint4 *__restrict__ beta, const float *__restrict__ mean_in,
                           const float *__restrict__ rstd_in, int64_t B, int nvec, uint4 *__restrict__ dx,
                           float *__restrict__ partials)
{
    constexpr int NT = HAS_RES ? 3 : 2;
    uint32_t cs, rank;
    asm volatile("mov.u32 %0, %%cluster_nctaid.x;" : "=r"(cs));
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
    const int nclusters = gridDim.x / cs, cid = blockIdx.x / cs;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int slot = rank * kBwdThreads + tid;
    const bool active = slot < nvec;
    const int D = nvec * 8;
    const float inv_d = 1.0f / (float)D;
    const int myvec = min(kBwdThreads, nvec - (int)rank * kBwdThreads); // > 0 by construction of cs
    const uint32_t slice_bytes = (uint32_t)myvec * 16u;

    extern __shared__ __align__(128) unsigned char dsm[];
    uint4 *ring = reinterpret_cast<uint4 *>(dsm); // [stage][sample][tensor][kBwdThreads]
    __shared__ __align__(8) uint64_t s_full[kBwdStages]; // TMA completion per ring stage
    __shared__ __align__(8) uint64_t s_sum[kSumSlots];   // peers' row-sum bytes per group slot
    __shared__ float s_peer[kSumSlots][kMaxCluster][2 * S];
    __shared__ float s_warp[2][kBwdThreads / 32][2 * S]; // by group parity (see the exchange below)
    __shared__ float s_cb[kBwdThreads * 8];
    __shared__ float s_stat[kBwdStages][2 * S]; // rstd[S], mean[S] of the group in each ring stage

    // gamma, beta and the conv bias of this thread's 8 columns stay packed (4 registers each);
    // kBwdThreads % cvecs == 0, so slot % cvecs == tid % cvecs
    const uint4 gv = active ? gamma[slot] : make_uint4(0u, 0u, 0u, 0u);
    const uint4 bv = active ? beta[slot] : make_uint4(0u, 0u, 0u, 0u);
    const uint4 cbv = cbias ? cbias[tid % cvecs] : make_uint4(0u, 0u, 0u, 0u);
    f2 dg[4], db[4], dcb[4]; // column pairs (2p, 2p+1) of this thread's 8 columns
#pragma unroll
    for (int p = 0; p < 4; ++p) dg[p] = db[p] = dcb[p] = f2_make(0.f, 0.f);

    const int64_t groups = (B + S - 1) / S;
    const int G = cid < groups ? (int)((groups - cid + nclusters - 1) / nclusters) : 0; // same in every CTA of the cluster

    auto stage_ptr = [&](int stage, int k, int t) { return ring + ((size_t)(stage * S + k) * NT + t) * kBwdThreads; };
    auto issue = [&](int i) { // thread 0: TMA loads of this CTA's column slice of group i
        const int64_t grp = cid + (int64_t)i * nclusters;
        const int stage = i % kBwdStages;
        const int nvalid = (int)min((int64_t)S, B - grp * S);
        const uint32_t bar = smem_u32(&s_full[stage]);
        mbar_expect_tx(bar, (uint32_t)nvalid * NT * slice_bytes);
        for (int k = 0; k < nvalid; ++k) {
            const int64_t off = (grp * S + k) * nvec + (int64_t)rank * kBwdThreads;
            bulk_load(smem_u32(stage_ptr(stage, k, 0)), x + off, slice_bytes, bar);
            bulk_load(smem_u32(stage_ptr(stage, k, 1)), dy + off, slice_bytes, bar);
            if (HAS_RES) bulk_load(smem_u32(stage_ptr(stage, k, 2)), res + off, slice_bytes, bar);
        }
    };

    if (tid == 0) {
        for (int q = 0; q < kBwdStages; ++q) mbar_init(smem_u32(&s_full[q]), 1);
        for (int q = 0; q < kSumSlots; ++q) mbar_init(smem_u32(&s_sum[q]), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // The groups' mean / rstd travel through shared memory one ring turn ahead, like the tensors: a
    // global load inside pass 1 sat on the critical path of every group (top stall in the ncu capture).
    auto stat_load = [&](int i, int j) -> float { // j < S: rstd of sample j, j >= S: mean of sample j - S
        const int64_t smp = (cid + (int64_t)i * nclusters) * S + (j % S);
        return smp < B ? (j < S ? rstd_in : mean_in)[smp] : 0.f;
    };
    if (tid < 2 * S)
        for (int q = 0; q < kBwdStages && q < G; ++q) s_stat[q][tid] = stat_load(q, tid);
    cluster_sync_all(); // every CTA's barriers exist before any peer signals them (and s_stat is visible)
    if (tid == 0) {
        if (G > 0) issue(0);
        if (G > 1) issue(1);
    }
    const uint32_t sum_bytes = (uint32_t)(2 * S * cs * sizeof(float));

    for (int i = 0; i < G; ++i) {
        const int64_t grp = cid + (int64_t)i * nclusters;
        const int stage = i % kBwdStages, q = i % kSumSlots;
        mbar_wait(smem_u32(&s_full[stage]), (uint32_t)(i / kBwdStages) & 1u);
        // ---------------------------------------------------------------- pass 1
        // S = 2: h and w stay fp32 pairs (32 registers). S = 4 (no residual): they are parked as bf16
        // pairs (32 registers again) -- dx is a bf16 output, and twice the samples per exchange
        // halves the number of cluster exchanges, which is what bounds this kernel.
        constexpr bool kPack = S > 2;
        typedef typename std::conditional<kPack, uint32_t, f2>::type hw_t;
        hw_t h[S][4], w[S][4];
        float p1[S], p2[S], rs[S];
#pragma unroll
        for (int k = 0; k < S; ++k) {
            p1[k] = p2[k] = rs[k] = 0.f;
            const int64_t smp = grp * S + k;
            if (active && smp < B) {
                rs[k] = s_stat[stage][k];
                const float nmr = -s_stat[stage][S + k] * rs[k];
                const f2 rs2 = f2_make(rs[k], rs[k]), nmr2 = f2_make(nmr, nmr);
                const uint4 xv = stage_ptr(stage, k, 0)[tid], dv = stage_ptr(stage, k, 1)[tid];
                uint4 rv = make_uint4(0u, 0u, 0u, 0u);
                if (HAS_RES) rv = stage_ptr(stage, k, 2)[tid];
                f2 s1 = f2_make(0.f, 0.f), s2 = f2_make(0.f, 0.f);
#pragma unroll
                for (int p = 0; p < 4; ++p) {
                    f2 z = f2_add(bf2_to_f2(word_of(xv, p)), bf2_to_f2(word_of(cbv, p)));
                    if (HAS_RES) z = f2_add(z, bf2_to_f2(word_of(rv, p)));
                    const f2 g2 = bf2_to_f2(word_of(gv, p));
                    const f2 hh = f2_fma(z, rs2, nmr2);
                    float pre0, pre1;
                    f2_split(f2_fma(hh, g2, bf2_to_f2(word_of(bv, p))), pre0, pre1);
                    const uint32_t dw = word_of(dv, p);
                    const f2 gy = f2_make(pre0 > 0.f ? __uint_as_float(dw << 16) : 0.f,      // relu'
                                          pre1 > 0.f ? __uint_as_float(dw & 0xFFFF0000u) : 0.f);
                    dg[p] = f2_fma(gy, hh, dg[p]);
                    db[p] = f2_add(db[p], gy);
                    const f2 ww = f2_mul(gy, g2);
                    if constexpr (kPack) {
                        h[k][p] = f2_to_bf2(hh);
                        w[k][p] = f2_to_bf2(ww);
                    } else {
                        h[k][p] = hh;
                        w[k][p] = ww;
                    }
                    s1 = f2_add(s1, ww);
                    s2 = f2_fma(ww, hh, s2);
                }
                float a0, a1, b0, b1;
                f2_split(s1, a0, a1);
                f2_split(s2, b0, b1);
                p1[k] = a0 + a1;
                p2[k] = b0 + b1;
            } else {
#pragma unroll
                for (int p = 0; p < 4; ++p) h[k][p] = w[k][p] = hw_t(0);
            }
        }
        // Warp reduction of the 2*S sums, transposed: every butterfly step halves the number of values a
        // lane carries (the half it gives away goes to the partner lane), so 2*S values cost
        // 2*S - 1 + (5 - log2(2*S)) shuffles instead of 5 * 2*S. Lane l ends with the total of value l / kRep.
        {
            constexpr int V = 2 * S, kRep = 32 / V;
            float v[V];
#pragma unroll
            for (int k = 0; k < S; ++k) {
                v[2 * k] = p1[k];
                v[2 * k + 1] = p2[k];
            }
            int o = 16;
#pragma unroll
            for (int n = V / 2; n >= 1; n >>= 1, o >>= 1) {
                const bool up = (lane & o) != 0;
#pragma unroll
                for (int j = 0; j < n; ++j) {
                    const float give = up ? v[j] : v[j + n], keep = up ? v[j + n] : v[j];
                    v[j] = keep + __shfl_xor_sync(0xffffffffu, give, o);
                }
            }
#pragma unroll
            for (; o > 0; o >>= 1) v[0] += __shfl_xor_sync(0xffffffffu, v[0], o);
            if ((lane & (kRep - 1)) == 0) s_warp[i & 1][warp][lane / kRep] = v[0];
        }
        __syncthreads(); // s_warp is complete, and every thread is done reading ring stage `stage`
        if (tid == 0 && i + kBwdStages < G) issue(i + kBwdStages);
        const bool stat_thread = tid >= 32 && tid < 32 + 2 * S && i + kBwdStages < G;
        float stat_next = 0.f; // in flight during the exchange and pass 2, stored at the end of the iteration
        if (stat_thread) stat_next = stat_load(i + kBwdStages, tid - 32);
        // ---------------------------------------------------------------- exchange
        // This CTA's 2*S sums go to every CTA of the cluster (itself included); the receiver's mbarrier
        // counts the bytes. Two slots are enough: a peer sends group i+1 only after it has passed its
        // wait for group i, and it sends group i+2 only after THIS CTA's sums of i+1 -- sent after all
        // its warps finished reading slot i -- have reached it.
        // s_warp has two buffers by group parity. The readers below (2*S*cs threads: warps 0 AND 1 for
        // S = 4, cs = 8) are ordered only before this CTA's own __syncthreads of group i + 1, not before
        // the other warps' writes of group i + 1: the wait below completes on the send of whichever
        // warp holds this CTA's own entries, so a warp may run into pass 1 of group i + 1 while the other
        // reading warp still reads. Group i + 1 writes the other buffer; group i + 2 writes this one
        // again only after the __syncthreads of group i + 1, which every reader of group i has reached.
        const uint32_t bar = smem_u32(&s_sum[q]);
        if (tid == 0) mbar_expect_tx(bar, sum_bytes);
        for (int e = tid; e < 2 * S * (int)cs; e += kBwdThreads) {
            const int v = e % (2 * S), dst = e / (2 * S);
            float a = 0.f;
#pragma unroll
            for (int ww = 0; ww < kBwdThreads / 32; ++ww) a += s_warp[i & 1][ww][v];
            st_async_f32(map_to_rank(smem_u32(&s_peer[q][rank][v]), (uint32_t)dst), a, map_to_rank(bar, (uint32_t)dst));
        }
        mbar_wait(bar, (uint32_t)(i / kSumSlots) & 1u);
        float t = 0.f;
        if (lane < 2 * S)
            for (int r = 0; r < (int)cs; ++r) t += s_peer[q][r][lane];
        // ---------------------------------------------------------------- pass 2 (from registers)
#pragma unroll
        for (int k = 0; k < S; ++k) {
            const float t1 = __shfl_sync(0xffffffffu, t, 2 * k), t2 = __shfl_sync(0xffffffffu, t, 2 * k + 1);
            const int64_t smp = grp * S + k;
            if (active && smp < B) {
                const float a = -(t1 * inv_d * rs[k]), b = -(t2 * inv_d * rs[k]); // -m1 * rstd, -m2 * rstd
                const f2 rs2 = f2_make(rs[k], rs[k]), a2 = f2_make(a, a), b2 = f2_make(b, b);
                uint32_t ow[4];
#pragma unroll
                for (int p = 0; p < 4; ++p) {
                    f2 hh, ww;
                    if constexpr (kPack) {
                        hh = bf2_to_f2(h[k][p]);
                        ww = bf2_to_f2(w[k][p]);
                    } else {
                        hh = h[k][p];
                        ww = w[k][p];
                    }
                    const f2 o = f2_fma(hh, b2, f2_fma(ww, rs2, a2)); // w*rstd - m1*rstd - h*m2*rstd
                    dcb[p] = f2_add(dcb[p], o);
                    ow[p] = f2_to_bf2(o);
                }
                dx[smp * nvec + slot] = make_uint4(ow[0], ow[1], ow[2], ow[3]);
            }
        }
        // every thread read s_stat[stage] before this iteration's __syncthreads; its next readers come
        // after the next iteration's
        if (stat_thread) s_stat[stage][tid - 32] = stat_next;
    }

    if (active) {
        float *out = partials + (size_t)cid * 2 * D + (size_t)slot * 8;
#pragma unroll
        for (int p = 0; p < 4; ++p) {
            f2_split(dg[p], out[2 * p], out[2 * p + 1]);
            f2_split(db[p], out[D + 2 * p], out[D + 2 * p + 1]);
        }
    }
    // d(conv bias): fold the threads that share a channel group (tid % cvecs) through shared memory
#pragma unroll
    for (int p = 0; p < 4; ++p) f2_split(dcb[p], s_cb[tid * 8 + 2 * p], s_cb[tid * 8 + 2 * p + 1]);
    __syncthreads();
    const int C = cvecs * 8;
    if (tid < C) {
        const int grp = tid >> 3, j = tid & 7;
        float sum = 0.f;
        for (int q = grp; q < kBwdThreads; q += cvecs) sum += s_cb[q * 8 + j];
        partials[(size_t)nclusters * 2 * D + (size_t)blockIdx.x * C + tid] = sum;
    }
    cluster_sync_all(); // no CTA leaves while a peer may still write into its shared memory
}

// sums the clustered backward's partials: thread i < 2D -> dgamma/dbeta (over clusters),
// 2D <= i < 2D + C -> d conv bias (over CTAs)
__global__ void reduce_cluster_partials_kernel(const float *__restrict__ partials, int nclusters, int nctas, int D,
                                               int C, float *__restrict__ dgamma, float *__restrict__ dbeta,
                                               float *__restrict__ dcbias)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 2 * D) {
        float s = 0.f;
#pragma unroll 8
        for (int p = 0; p < nclusters; ++p) s += partials[(size_t)p * 2 * D + i];
        if (i < D) dgamma[i] = s;
        else dbeta[i - D] = s;
    } else if (i < 2 * D + C && dcbias) {
        const float *cbp = partials + (size_t)nclusters * 2 * D;
        float s = 0.f;
#pragma unroll 8
        for (int p = 0; p < nctas; ++p) s += cbp[(size_t)p * C + (i - 2 * D)];
        dcbias[i - 2 * D] = s;
    }
}

// Per-row transpose with dtype conversion: dst[r][b*A + a] = src[r][a*B + b] for a < A, b < B.
// Used to bring the 19200 trunk columns of the fused head weight from the checkpoint's CHW order
// (fp32 master) to the HWC order of the channels-last activations (bf16 working copy), and to
// carry the gradient back. 32x32 shared-memory tiles, coalesced on both sides.
template <typename TS, typename TD>
__global__ void transpose_cast_kernel(const TS *__restrict__ src, int64_t ld_src, TD *__restrict__ dst,
                                      int64_t ld_dst, int A, int B)
{
    __shared__ float tile[32][33];
    const int64_t r = blockIdx.z;
    const int a0 = blockIdx.y * 32, b0 = blockIdx.x * 32;
    const TS *s = src + r * ld_src;
    TD *d = dst + r * ld_dst;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int a = a0 + i, b = b0 + threadIdx.x;
        if (a < A && b < B) tile[i][threadIdx.x] = (float)s[(int64_t)a * B + b];
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int b = b0 + i, a = a0 + threadIdx.x;
        if (a < A && b < B) d[(int64_t)b * A + a] = (TD)tile[threadIdx.x][i];
    }
}

constexpr const char *kBadC = "unsupported C: needs C % 8 == 0, D % C == 0 and C / 8 dividing the block size";
constexpr const char *kBadD = "D must be at most 20480";

} // namespace

// INV_LN_BWD=percta: the pointers, B and D have been checked by inv_ln_relu_bwd
static int ln_relu_bwd_percta(const void *dy, const void *x, const void *res, const void *cbias, const void *gamma,
                    const void *beta, const float *mean, const float *rstd, int64_t B, int32_t D, int32_t C,
                    void *dx, float *dgamma, float *dbeta, float *dcbias, float *partials, void *stream)
{
    const char *who = "inv_ln_relu_bwd";
    if (C <= 0 || C % 8 || D % C || kLnThreads % (C / 8) || C > kLnThreads)
        return inv_host::set_error(INV_ERR_INVALID_ARG, who, kBadC);
    const int cvecs = C / 8;
    const int nvec = D / 8;
    const int maxv = (nvec + kLnThreads - 1) / kLnThreads;
    if (maxv > 5) return inv_host::set_error(INV_ERR_INVALID_ARG, who, kBadD);
    const int nsm = inv_host::sm_count();
    const unsigned grid = (unsigned)(B < nsm ? B : nsm); // one CTA per SM: 2*D floats of shared memory each
    size_t smem = (size_t)2 * D * sizeof(float);
    if (smem < (size_t)kLnThreads * 8 * sizeof(float)) smem = (size_t)kLnThreads * 8 * sizeof(float);
    cudaStream_t st = (cudaStream_t)stream;
    using Kern = decltype(&ln_relu_bwd_kernel<1, false>);
    static const Kern kerns[5][2] = {{ln_relu_bwd_kernel<1, false>, ln_relu_bwd_kernel<1, true>},
                                     {ln_relu_bwd_kernel<2, false>, ln_relu_bwd_kernel<2, true>},
                                     {ln_relu_bwd_kernel<3, false>, ln_relu_bwd_kernel<3, true>},
                                     {ln_relu_bwd_kernel<4, false>, ln_relu_bwd_kernel<4, true>},
                                     {ln_relu_bwd_kernel<5, false>, ln_relu_bwd_kernel<5, true>}};
    const Kern kern = kerns[maxv - 1][res != nullptr];
    if (inv_host::allow_dynamic_smem((const void *)kern, smem) != cudaSuccess) return inv_host::launch_status(who);
    kern<<<grid, kLnThreads, smem, st>>>((const uint4 *)dy, (const uint4 *)x, (const uint4 *)res, (const uint4 *)cbias,
                                        cvecs, (const uint4 *)gamma, (const uint4 *)beta, mean, rstd, B, nvec, (uint4 *)dx,
                                        partials);
    if (int rc = inv_host::launch_status(who)) return rc;
    const int width = 2 * D + C;
    reduce_partials_kernel<<<(width + 255) / 256, 256, 0, st>>>(partials, (int)grid, width, dgamma, dbeta, dcbias, D);
    return inv_host::launch_status(who);
}


extern "C" {

int inv_transpose_cast(const void *src, int32_t src_is_f32, int64_t ld_src, void *dst, int32_t dst_is_f32,
                       int64_t ld_dst, int64_t rows, int32_t A, int32_t B, void *stream)
{
    const char *who = "inv_transpose_cast";
    if (int rc = inv_host::require_sm100(who)) return rc;
    if (!src || !dst || rows < 0 || A <= 0 || B <= 0 || rows > 65535)
        return inv_host::set_error(INV_ERR_INVALID_ARG, who, "null pointer, or rows outside [0, 65535], or A or B not positive");
    if (src_is_f32 == dst_is_f32) return inv_host::set_error(INV_ERR_INVALID_ARG, who, "exactly one side must be fp32");
    if (rows == 0) return INV_OK;
    const dim3 grid((B + 31) / 32, (A + 31) / 32, (unsigned)rows), block(32, 8);
    cudaStream_t st = (cudaStream_t)stream;
    if (src_is_f32)
        transpose_cast_kernel<float, __nv_bfloat16><<<grid, block, 0, st>>>(
            (const float *)src, ld_src, (__nv_bfloat16 *)dst, ld_dst, A, B);
    else
        transpose_cast_kernel<__nv_bfloat16, float><<<grid, block, 0, st>>>(
            (const __nv_bfloat16 *)src, ld_src, (float *)dst, ld_dst, A, B);
    return inv_host::launch_status(who);
}

int inv_ln_relu_partials(int32_t D) { (void)D; return 2 * inv_host::sm_count(); }

int inv_ln_relu_fwd(const void *x, const void *res, const void *cbias, const void *gamma, const void *beta,
                    int64_t B, int32_t D, int32_t C, float eps, void *y, float *mean, float *rstd, void *stream)
{
    const char *who = "inv_ln_relu_fwd";
    if (int rc = inv_host::require_sm100(who)) return rc;
    if (!x || !gamma || !beta || !y || !mean || !rstd || B < 0 || D <= 0 || D % 8)
        return inv_host::set_error(INV_ERR_INVALID_ARG, who, "null pointer, B < 0, or D not a positive multiple of 8");
    if (C <= 0 || C % 8 || D % C || kLnThreads % (C / 8)) return inv_host::set_error(INV_ERR_INVALID_ARG, who, kBadC);
    const int cvecs = C / 8;
    if (B == 0) return INV_OK;
    const int nvec = D / 8;
    const int maxv = (nvec + kLnThreads - 1) / kLnThreads;
    if (maxv > 5) return inv_host::set_error(INV_ERR_INVALID_ARG, who, kBadD);
    const int64_t cap = (int64_t)inv_host::sm_count() * 4;
    const unsigned grid = (unsigned)(B < cap ? B : cap);
    cudaStream_t st = (cudaStream_t)stream;
#define LAUNCH(MV)                                                                                              \
    if (res)                                                                                                    \
        ln_relu_fwd_kernel<MV, true><<<grid, kLnThreads, 0, st>>>((const uint4 *)x, (const uint4 *)res,         \
            (const uint4 *)cbias, cvecs, (const uint4 *)gamma, (const uint4 *)beta, B, nvec, eps, (uint4 *)y,    \
            mean, rstd);                                                                                        \
    else                                                                                                        \
        ln_relu_fwd_kernel<MV, false><<<grid, kLnThreads, 0, st>>>((const uint4 *)x, nullptr,                   \
            (const uint4 *)cbias, cvecs, (const uint4 *)gamma, (const uint4 *)beta, B, nvec, eps, (uint4 *)y,    \
            mean, rstd);
    switch (maxv) {
    case 1: LAUNCH(1) break;
    case 2: LAUNCH(2) break;
    case 3: LAUNCH(3) break;
    case 4: LAUNCH(4) break;
    default: LAUNCH(5) break;
    }
#undef LAUNCH
    return inv_host::launch_status(who);
}

int inv_ln_relu_bwd(const void *dy, const void *x, const void *res, const void *cbias, const void *gamma,
                    const void *beta, const float *mean, const float *rstd, int64_t B, int32_t D, int32_t C,
                    void *dx, float *dgamma, float *dbeta, float *dcbias, float *partials, void *stream)
{
    const char *who = "inv_ln_relu_bwd";
    if (int rc = inv_host::require_sm100(who)) return rc;
    if (!dy || !x || !gamma || !beta || !mean || !rstd || !dx || !dgamma || !dbeta || !partials || B <= 0 ||
        D <= 0 || D % 8)
        return inv_host::set_error(INV_ERR_INVALID_ARG, who, "null pointer, B <= 0, or D not a positive multiple of 8");
    {   // default: the cluster-split kernel; INV_LN_BWD=percta selects the round-1 kernel (one CTA per
        // SM, shared-memory accumulators) for A/B measurements
        static int use_cluster = -1;
        if (use_cluster < 0) {
            const char *e = getenv("INV_LN_BWD");
            use_cluster = (e && e[0] == 'p' && e[1] == 'e') ? 0 : 1; // "percta"
        }
        if (!use_cluster)
            return ln_relu_bwd_percta(dy, x, res, cbias, gamma, beta, mean, rstd, B, D, C, dx, dgamma, dbeta, dcbias,
                                      partials, stream);
    }
    if (C <= 0 || C % 8 || D % C || kBwdThreads % (C / 8) || C > kBwdThreads)
        return inv_host::set_error(INV_ERR_INVALID_ARG, who, kBadC);
    const int cvecs = C / 8;
    const int nvec = D / 8;
    const int cs = (nvec + kBwdThreads - 1) / kBwdThreads; // CTAs per cluster: 2 / 4 / 8 for D = 4800 / 9600 / 19200
    if (cs > kMaxCluster) return inv_host::set_error(INV_ERR_INVALID_ARG, who, kBadD);
    cudaStream_t st = (cudaStream_t)stream;
    // samples per cluster exchange: 4 without a residual input (INV_LN_BWD_S=2 selects 2, for A/B runs), 2 with
    static int s_nores = -1;
    if (s_nores < 0) {
        const char *e = getenv("INV_LN_BWD_S");
        s_nores = (e && e[0] == '2') ? 2 : 4;
    }
    const int S = res ? 2 : s_nores;
    auto kern = res ? ln_relu_bwd_cluster_kernel<2, true>
                    : (S == 4 ? ln_relu_bwd_cluster_kernel<4, false> : ln_relu_bwd_cluster_kernel<2, false>);

    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)cs;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    const size_t smem = res ? bwd_cluster_smem<2, true>() : (S == 4 ? bwd_cluster_smem<4, false>() : bwd_cluster_smem<2, false>());
    if (inv_host::allow_dynamic_smem((const void *)kern, smem) != cudaSuccess) return inv_host::launch_status(who);
    cfg.blockDim = dim3(kBwdThreads, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    // as many clusters as the GPU keeps resident at once (the work split is static per cluster)
    static int resident[64][kMaxCluster + 1][3] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    int ncl = 0;
    const int variant = res ? 1 : (S == 4 ? 2 : 0);
    if (dev >= 0 && dev < 64) ncl = resident[dev][cs][variant];
    if (ncl == 0) {
        cfg.gridDim = dim3((unsigned)(cs * 64), 1, 1);
        if (cudaOccupancyMaxActiveClusters(&ncl, kern, &cfg) != cudaSuccess || ncl <= 0) {
            cudaGetLastError();
            ncl = inv_host::sm_count() / cs; // conservative: one CTA per SM
        }
        const int cap = 2 * inv_host::sm_count() / cs; // the partials buffer holds 2 * SMs parts
        if (ncl > cap) ncl = cap;
        if (dev >= 0 && dev < 64) resident[dev][cs][variant] = ncl;
    }
    const int64_t groups = (B + S - 1) / S;
    if (ncl > groups) ncl = (int)groups;
    if (ncl < 1) ncl = 1;
    cfg.gridDim = dim3((unsigned)(ncl * cs), 1, 1);
    const uint4 *dy4 = (const uint4 *)dy, *x4 = (const uint4 *)x, *res4 = (const uint4 *)res, *cb4 = (const uint4 *)cbias;
    const uint4 *g4 = (const uint4 *)gamma, *b4 = (const uint4 *)beta;
    uint4 *dx4 = (uint4 *)dx;
    if (cudaLaunchKernelEx(&cfg, kern, dy4, x4, res4, cb4, cvecs, g4, b4, mean, rstd, B, nvec, dx4, partials) != cudaSuccess)
        return inv_host::launch_status(who);
    const int width = 2 * D + C;
    reduce_cluster_partials_kernel<<<(width + 255) / 256, 256, 0, st>>>(partials, ncl, ncl * cs, D, C, dgamma, dbeta, dcbias);
    return inv_host::launch_status(who);
}

} // extern "C"
