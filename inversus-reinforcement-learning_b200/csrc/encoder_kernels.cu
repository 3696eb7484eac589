// encoder_kernels.cu -- layer 1 of the policy computed straight from packed env states.
//
// The policy's first block is conv1 (3x3, 12 -> 32) + bias + LayerNorm([32,10,15]) + ReLU
// (inversus_rl/policies.py:27-31, :94) applied to the 12-plane observation of
// build_observation (inversus_rl/env_wrappers.py:173-245). Those planes hold only 0 and 1, and all
// of them are a function of the 80-byte packed state. So instead of materialising the observation
// (3.6-7.2 KB per sample), converting it to channels-last and running a K=108 convolution that
// cuDNN serves with Ampere-generation kernels, this file evaluates the same function directly:
//
//   * the two tile planes (ch0 = BLACK, ch1 = WHITE, exactly one of them set per tile) contribute,
//     for every output position and kernel row, one of 24 pre-summed weight vectors selected by the
//     3-tile colour pattern under that kernel row (table T, built from the fp32 master weights);
//   * the ten sparse planes (two players, eight bullet planes) contribute weight vectors scattered
//     around the few set positions (table S).
//
// One warp owns one sample, lane = output channel. The pre-LayerNorm feature map lives in shared
// memory as bf16 (what the cuDNN path stores too), statistics are fp32, the output is the
// channels-last bf16 activation [B, 10, 15, 32] the rest of the trunk consumes. The backward kernel
// recomputes the feature map from the packed state, applies the LayerNorm+ReLU backward and turns
// the result directly into the gradients of conv1's weight and bias and of the LayerNorm affine --
// there is no input gradient to produce. No atomics: every accumulator has one owner, so results
// are deterministic.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/inversus_b200.h"
#include "launch_common.h"

namespace {

constexpr int kBW = INV_BOARD_W, kBH = INV_BOARD_H, kPos = kBW * kBH; // 15 x 10 = 150 positions
constexpr int kCo = 32;                                                // conv1 output channels = lanes
constexpr int kCi = INV_OBS_CHANNELS;                                  // 12 input planes
constexpr int kD = kPos * kCo;                                         // 4800 features per sample
constexpr int kWords = kD / 2;                                         // bf16 pairs per sample
constexpr int kPat = 24;                                               // (edge 0..2) x (3-tile pattern 0..7)
constexpr int kSparse = kCi - 2;                                       // planes ch2..ch11
constexpr int kFwdWarps = 16, kBwdWarps = 8;
constexpr unsigned kFull = 0xffffffffu;

struct Tables {
    float T[3][kPat][kCo];      // dense part: kernel row r, pattern -> sum over the row's valid taps
    float S[kSparse][9][kCo];   // sparse part: plane (ch - 2), tap -> weight
};

// (float)(k / 6.0) as numpy computes it (env_wrappers.py:238-240); same table as the step kernel
__constant__ float kAmmoNormEnc[8] = {0x0.0p+0f, 0x1.555556p-3f, 0x1.555556p-2f, 0x1.0p-1f,
                                      0x1.555556p-1f, 0x1.aaaaaap-1f, 0x1.0p+0f, 0x1.2aaaaap+0f};

// w1 is the checkpoint layout [co][ci][ky][kx] (fp32 master weights).
__device__ void build_tables(Tables &tb, const float *__restrict__ w1)
{
    for (int i = threadIdx.x; i < 3 * kPat * kCo; i += blockDim.x) {
        const int co = i % kCo, pat = (i / kCo) % kPat, r = i / (kCo * kPat);
        const int edge = pat >> 3, win = pat & 7; // edge 1: x == 0 (left tap outside), 2: x == 14 (right tap outside)
        float acc = 0.f;
        for (int dx = 0; dx < 3; ++dx) {
            if ((edge == 1 && dx == 0) || (edge == 2 && dx == 2)) continue;
            const int colour = (win >> dx) & 1; // 1 = WHITE -> plane 1, 0 = BLACK -> plane 0
            acc += w1[((co * kCi + colour) * 3 + r) * 3 + dx];
        }
        tb.T[r][pat][co] = acc;
    }
    for (int i = threadIdx.x; i < kSparse * 9 * kCo; i += blockDim.x) {
        const int co = i % kCo, tap = (i / kCo) % 9, c = i / (kCo * 9);
        tb.S[c][tap][co] = w1[(co * kCi + c + 2) * 9 + tap];
    }
}

// What a warp needs of one env, identical in every lane except `bul` (lane i < 16: bullet slot i).
// Packed layout: DESIGN.md section 3 / csrc/inversus_kernels.cuh (five 16-byte planes).
struct EnvBits {
    uint32_t rb[kBH]; // 15 tile bits per board row, 1 = WHITE
    uint32_t p1w, p2w, bul;
    int nb;
};

__device__ __forceinline__ void load_env_bits(const uint32_t *__restrict__ planes, int64_t stride, int64_t e, int lane,
                                              EnvBits &o)
{
    uint32_t v = 0;
    if (lane < 20) v = planes[((int64_t)(lane >> 2) * stride + e) * 4 + (lane & 3)];
    uint32_t t[6];
#pragma unroll
    for (int k = 0; k < 5; ++k) t[k] = __shfl_sync(kFull, v, k);
    t[5] = 0u;
    o.p1w = __shfl_sync(kFull, v, 5);
    o.p2w = __shfl_sync(kFull, v, 6);
    o.nb = (int)(o.p1w >> 20) & 31;
    const uint32_t wd = __shfl_sync(kFull, v, 12 + ((lane & 15) >> 1));
    o.bul = (wd >> ((lane & 1) * 16)) & 0xFFFFu;
#pragma unroll
    for (int y = 0; y < kBH; ++y) {
        const int off = y * kBW, w = off >> 5, sh = off & 31;
        const uint64_t two = ((uint64_t)t[w + 1] << 32) | t[w];
        o.rb[y] = (uint32_t)(two >> sh) & 0x7FFFu;
    }
}

__device__ __forceinline__ float4 extra_of(const EnvBits &eb, int view)
{
    const uint32_t vw = view ? eb.p2w : eb.p1w, ew = view ? eb.p1w : eb.p2w;
    const bool va = (vw >> 16) & 1u, ea = (ew >> 16) & 1u;
    return make_float4(va ? kAmmoNormEnc[(vw >> 8) & 7u] : 0.f, ea ? kAmmoNormEnc[(ew >> 8) & 7u] : 0.f,
                       va ? 1.f : 0.f, ea ? 1.f : 0.f);
}

// Calls fn(plane, x, y) once per set bit of the ten sparse observation planes (plane = channel - 2):
// ch2 viewer, ch3 enemy (if alive), ch4-7 viewer's bullets by direction, ch8-11 enemy's bullets.
// Bullets that coincide in tile, direction and owner set the same bit and are visited once.
template <typename Fn>
__device__ __forceinline__ void for_each_object(const EnvBits &eb, int view, int lane, Fn fn)
{
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const uint32_t w = i ? eb.p2w : eb.p1w;
        if ((w >> 16) & 1u) fn(i == view ? 0 : 1, (int)(w & 15u), (int)((w >> 4) & 15u));
    }
    const bool valid = lane < 16 && lane < eb.nb;
    const uint32_t key = valid ? (eb.bul & 0x7FFu) : (0x8000u + (uint32_t)lane);
    const uint32_t same = __match_any_sync(kFull, key);
    const bool keep = valid && (same & ((1u << lane) - 1u)) == 0u;
    uint32_t todo = __ballot_sync(kFull, keep);
    while (todo) {
        const int j = __ffs(todo) - 1;
        todo &= todo - 1u;
        const uint32_t b = __shfl_sync(kFull, eb.bul, j);
        const int owner = (b >> 10) & 1u, dir = (b >> 8) & 3u;
        fn((owner == view ? 2 : 6) + dir, (int)(b & 15u), (int)((b >> 4) & 15u));
    }
}

// conv1 + bias of one sample into zb[pos * 32 + lane] (bf16). Dense part, then the sparse planes.
__device__ __forceinline__ void conv1_to_smem(const Tables &tb, const EnvBits &eb, int view, float bias, int lane,
                                              __nv_bfloat16 *zb)
{
#pragma unroll
    for (int y = 0; y < kBH; ++y) {
#pragma unroll
        for (int x = 0; x < kBW; ++x) {
            float acc = bias;
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                const int yy = y + r - 1;
                if (yy < 0 || yy >= kBH) continue;
                const int edge = x == 0 ? 1 : (x == kBW - 1 ? 2 : 0);
                const uint32_t win = ((eb.rb[yy] << 1) >> x) & 7u; // bit dx = tile (x + dx - 1, yy)
                acc += tb.T[r][edge * 8 + win][lane];
            }
            zb[(y * kBW + x) * kCo + lane] = __float2bfloat16_rn(acc);
        }
    }
    for_each_object(eb, view, lane, [&](int c, int qx, int qy) {
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) {
            const int px = qx - (tap % 3 - 1), py = qy - (tap / 3 - 1); // out[p] sees in[p + tap]
            if ((unsigned)px < (unsigned)kBW && (unsigned)py < (unsigned)kBH) {
                __nv_bfloat16 *z = zb + (py * kBW + px) * kCo + lane;
                *z = __float2bfloat16_rn(__bfloat162float(*z) + tb.S[c][tap][lane]);
            }
        }
    });
}

__device__ __forceinline__ float2 unpack2(uint32_t u)
{
    return make_float2(__uint_as_float(u << 16), __uint_as_float(u & 0xFFFF0000u));
}
__device__ __forceinline__ uint32_t pack2(float a, float b)
{
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<const uint32_t *>(&h);
}
__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}

// ------------------------------------------------------------------------------------------------
// forward: y = relu(LN(conv1(obs(state)) + b1) * gamma + beta), channels-last bf16 [count][150][32]
__global__ void __launch_bounds__(kFwdWarps * 32)
encode_fwd_kernel(const uint32_t *__restrict__ planes, int64_t stride, int64_t count, int view,
                  const float *__restrict__ w1, const float *__restrict__ b1, const float2 *__restrict__ gamma,
                  const float2 *__restrict__ beta, float eps, uint32_t *__restrict__ y, float4 *__restrict__ extra,
                  float *__restrict__ mean_out, float *__restrict__ rstd_out)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Tables &tb = *reinterpret_cast<Tables *>(smem_raw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __nv_bfloat16 *zb = reinterpret_cast<__nv_bfloat16 *>(smem_raw + sizeof(Tables)) + (size_t)warp * kD;
    const uint32_t *z32 = reinterpret_cast<const uint32_t *>(zb);
    build_tables(tb, w1);
    __syncthreads();
    const float bias = b1[lane];
    for (int64_t s = (int64_t)blockIdx.x * kFwdWarps + warp; s < count; s += (int64_t)gridDim.x * kFwdWarps) {
        EnvBits eb;
        load_env_bits(planes, stride, s, lane, eb);
        if (lane == 0 && extra) extra[s] = extra_of(eb, view);
        conv1_to_smem(tb, eb, view, bias, lane, zb);
        __syncwarp();
        float sum = 0.f, sq = 0.f;
#pragma unroll 5
        for (int g = 0; g < kWords / 32; ++g) {
            const float2 z = unpack2(z32[g * 32 + lane]);
            sum += z.x + z.y;
            sq += z.x * z.x + z.y * z.y;
        }
        sum = warp_sum(sum);
        sq = warp_sum(sq);
        const float mean = sum * (1.0f / kD);
        const float var = fmaxf(sq * (1.0f / kD) - mean * mean, 0.f);
        const float rstd = rsqrtf(var + eps);
        if (lane == 0) {
            mean_out[s] = mean;
            rstd_out[s] = rstd;
        }
        uint32_t *out = y + s * kWords;
#pragma unroll 5
        for (int g = 0; g < kWords / 32; ++g) {
            const int j = g * 32 + lane;
            const float2 z = unpack2(z32[j]), ga = gamma[j], be = beta[j];
            out[j] = pack2(fmaxf((z.x - mean) * rstd * ga.x + be.x, 0.f), fmaxf((z.y - mean) * rstd * ga.y + be.y, 0.f));
        }
        __syncwarp(); // the next sample overwrites zb
    }
}

// ------------------------------------------------------------------------------------------------
// backward. Per-CTA partial sums, layout (floats): dgamma[4800] | dbeta[4800] | dense[18][32] |
// sparse[10][9][32]; encode_reduce_kernel sums the CTAs and assembles conv1's weight gradient.
constexpr int kDenseAcc = 18; // 9 white-tap sums, total, first/last row, first/last column, 4 corners
constexpr int kPartial = 2 * kD + kDenseAcc * kCo + kSparse * 9 * kCo;

__global__ void __launch_bounds__(kBwdWarps * 32, 1)
encode_bwd_kernel(const uint32_t *__restrict__ planes, int64_t stride, int64_t count, int view,
                  const float *__restrict__ w1, const float *__restrict__ b1, const float2 *__restrict__ gamma,
                  const float2 *__restrict__ beta, const float *__restrict__ mean_in, const float *__restrict__ rstd_in,
                  const uint32_t *__restrict__ dy, float *__restrict__ partials)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Tables &tb = *reinterpret_cast<Tables *>(smem_raw);
    __nv_bfloat16 *zall = reinterpret_cast<__nv_bfloat16 *>(smem_raw + sizeof(Tables));
    float *dws_all = reinterpret_cast<float *>(zall + (size_t)kBwdWarps * kD); // [warp][10][9][32]
    __shared__ float2 s_stat[kBwdWarps];   // mean, rstd of each warp's current sample
    __shared__ int64_t s_idx[kBwdWarps];   // its sample index, -1 = none
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __nv_bfloat16 *zb = zall + (size_t)warp * kD;
    uint32_t *z32 = reinterpret_cast<uint32_t *>(zb);
    float *dws = dws_all + (size_t)warp * (kSparse * 9 * kCo);
    build_tables(tb, w1);
    for (int i = lane; i < kSparse * 9 * kCo; i += 32) dws[i] = 0.f;
    const float bias = b1[lane];

    // this warp's slice of the LayerNorm affine gradient: bf16-pair indices [warp*300, warp*300+300)
    constexpr int kSlice = kWords / kBwdWarps, kIt = (kSlice + 31) / 32; // 300, 10
    float accg[kIt][2], accb[kIt][2];
#pragma unroll
    for (int it = 0; it < kIt; ++it) accg[it][0] = accg[it][1] = accb[it][0] = accb[it][1] = 0.f;
    float accw[9], tot = 0.f, rowf = 0.f, rowl = 0.f, colf = 0.f, coll = 0.f, k00 = 0.f, k10 = 0.f, k01 = 0.f, k11 = 0.f;
#pragma unroll
    for (int t = 0; t < 9; ++t) accw[t] = 0.f;

    const int64_t per_round = (int64_t)gridDim.x * kBwdWarps;
    const int64_t rounds = (count + per_round - 1) / per_round;
    for (int64_t rd = 0; rd < rounds; ++rd) {
        const int64_t s = rd * per_round + (int64_t)blockIdx.x * kBwdWarps + warp;
        const bool have = s < count;
        EnvBits eb;
        float mean = 0.f, rstd = 0.f;
        if (have) {
            load_env_bits(planes, stride, s, lane, eb);
            mean = mean_in[s];
            rstd = rstd_in[s];
            conv1_to_smem(tb, eb, view, bias, lane, zb);
        }
        if (lane == 0) {
            s_stat[warp] = make_float2(mean, rstd);
            s_idx[warp] = have ? s : -1;
        }
        __syncthreads(); // every warp's feature map is in shared memory

        // LayerNorm affine gradient: this warp's slice over all samples of the round
        for (int u = 0; u < kBwdWarps; ++u) {
            const int64_t su = s_idx[u];
            if (su < 0) continue;
            const float2 st = s_stat[u];
            const uint32_t *zu = reinterpret_cast<const uint32_t *>(zall + (size_t)u * kD);
            const uint32_t *du = dy + su * kWords;
#pragma unroll
            for (int it = 0; it < kIt; ++it) {
                const int k = it * 32 + lane;
                if (k < kSlice) {
                    const int j = warp * kSlice + k;
                    const float2 z = unpack2(zu[j]), d = unpack2(du[j]), ga = gamma[j], be = beta[j];
                    const float h0 = (z.x - st.x) * st.y, h1 = (z.y - st.x) * st.y;
                    const float g0 = (h0 * ga.x + be.x > 0.f) ? d.x : 0.f, g1 = (h1 * ga.y + be.y > 0.f) ? d.y : 0.f;
                    accg[it][0] += g0 * h0;
                    accg[it][1] += g1 * h1;
                    accb[it][0] += g0;
                    accb[it][1] += g1;
                }
            }
        }
        // own sample: the two LayerNorm row sums
        float s1 = 0.f, s2 = 0.f;
        if (have) {
            const uint32_t *dd = dy + s * kWords;
#pragma unroll 5
            for (int g = 0; g < kWords / 32; ++g) {
                const int j = g * 32 + lane;
                const float2 z = unpack2(z32[j]), d = unpack2(dd[j]), ga = gamma[j], be = beta[j];
                const float h0 = (z.x - mean) * rstd, h1 = (z.y - mean) * rstd;
                const float w0 = (h0 * ga.x + be.x > 0.f) ? d.x * ga.x : 0.f, w1v = (h1 * ga.y + be.y > 0.f) ? d.y * ga.y : 0.f;
                s1 += w0 + w1v;
                s2 += w0 * h0 + w1v * h1;
            }
        }
        s1 = warp_sum(s1);
        s2 = warp_sum(s2);
        const float m1 = s1 * (1.0f / kD), m2 = s2 * (1.0f / kD);
        __syncthreads(); // all slices have read every feature map; each warp may now overwrite its own

        if (have) {
            // gradient w.r.t. the conv output, in place (bf16, like the library path's dx)
            const uint32_t *dd = dy + s * kWords;
#pragma unroll 5
            for (int g = 0; g < kWords / 32; ++g) {
                const int j = g * 32 + lane;
                const float2 z = unpack2(z32[j]), d = unpack2(dd[j]), ga = gamma[j], be = beta[j];
                const float h0 = (z.x - mean) * rstd, h1 = (z.y - mean) * rstd;
                const float w0 = (h0 * ga.x + be.x > 0.f) ? d.x * ga.x : 0.f, w1v = (h1 * ga.y + be.y > 0.f) ? d.y * ga.y : 0.f;
                z32[j] = pack2(rstd * (w0 - m1 - h0 * m2), rstd * (w1v - m1 - h1 * m2));
            }
            __syncwarp();
            // conv1 weight gradient, dense planes: white-tap sums plus the border sums from which
            // the all-valid-tap sums (and so the black-tap sums) follow
#pragma unroll
            for (int y = 0; y < kBH; ++y) {
#pragma unroll
                for (int x = 0; x < kBW; ++x) {
                    const float dz = __bfloat162float(zb[(y * kBW + x) * kCo + lane]);
                    tot += dz;
                    if (y == 0) rowf += dz;
                    if (y == kBH - 1) rowl += dz;
                    if (x == 0) colf += dz;
                    if (x == kBW - 1) coll += dz;
                    if (x == 0 && y == 0) k00 += dz;
                    if (x == kBW - 1 && y == 0) k10 += dz;
                    if (x == 0 && y == kBH - 1) k01 += dz;
                    if (x == kBW - 1 && y == kBH - 1) k11 += dz;
#pragma unroll
                    for (int r = 0; r < 3; ++r) {
                        const int yy = y + r - 1;
                        if (yy < 0 || yy >= kBH) continue;
#pragma unroll
                        for (int dx = 0; dx < 3; ++dx) {
                            const int xx = x + dx - 1;
                            if (xx < 0 || xx >= kBW) continue;
                            if ((eb.rb[yy] >> xx) & 1u) accw[r * 3 + dx] += dz;
                        }
                    }
                }
            }
            // sparse planes
            for_each_object(eb, view, lane, [&](int c, int qx, int qy) {
#pragma unroll
                for (int tap = 0; tap < 9; ++tap) {
                    const int px = qx - (tap % 3 - 1), py = qy - (tap / 3 - 1);
                    if ((unsigned)px < (unsigned)kBW && (unsigned)py < (unsigned)kBH)
                        dws[(c * 9 + tap) * kCo + lane] += __bfloat162float(zb[(py * kBW + px) * kCo + lane]);
                }
            });
        }
        // the next round's conv writes only this warp's own buffer, which no other warp reads
        // before the next barrier
    }

    // ---- per-CTA partials
    float *out = partials + (size_t)blockIdx.x * kPartial;
#pragma unroll
    for (int it = 0; it < kIt; ++it) {
        const int k = it * 32 + lane;
        if (k < kSlice) {
            const int j = warp * kSlice + k;
            out[2 * j] = accg[it][0];
            out[2 * j + 1] = accg[it][1];
            out[kD + 2 * j] = accb[it][0];
            out[kD + 2 * j + 1] = accb[it][1];
        }
    }
    __syncthreads();
    float *scratch = reinterpret_cast<float *>(zall); // [warp][18][32], the feature maps are dead now
    {
        float *m = scratch + (size_t)warp * kDenseAcc * kCo;
#pragma unroll
        for (int t = 0; t < 9; ++t) m[t * kCo + lane] = accw[t];
        m[9 * kCo + lane] = tot;
        m[10 * kCo + lane] = rowf;
        m[11 * kCo + lane] = rowl;
        m[12 * kCo + lane] = colf;
        m[13 * kCo + lane] = coll;
        m[14 * kCo + lane] = k00;
        m[15 * kCo + lane] = k10;
        m[16 * kCo + lane] = k01;
        m[17 * kCo + lane] = k11;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kDenseAcc * kCo; i += blockDim.x) {
        float a = 0.f;
        for (int w = 0; w < kBwdWarps; ++w) a += scratch[(size_t)w * kDenseAcc * kCo + i];
        out[2 * kD + i] = a;
    }
    for (int i = threadIdx.x; i < kSparse * 9 * kCo; i += blockDim.x) {
        float a = 0.f;
        for (int w = 0; w < kBwdWarps; ++w) a += dws_all[(size_t)w * (kSparse * 9 * kCo) + i];
        out[2 * kD + kDenseAcc * kCo + i] = a;
    }
}

// Stage 1 of the reduction: red[i] = sum over CTAs of partials[cta][i]. 32 outputs x 8 part groups per
// block (a thread per output alone would walk the 148 partials one latency at a time).
__global__ void __launch_bounds__(256) encode_sum_partials_kernel(const float *__restrict__ partials, int nparts,
                                                                   float *__restrict__ red)
{
    __shared__ float s[8][33];
    const int i = blockIdx.x * 32 + threadIdx.x;
    float a = 0.f;
    if (i < kPartial)
        for (int p = threadIdx.y; p < nparts; p += 8) a += partials[(size_t)p * kPartial + i];
    s[threadIdx.y][threadIdx.x] = a;
    __syncthreads();
    if (threadIdx.y == 0 && i < kPartial) {
        float t = 0.f;
#pragma unroll
        for (int y = 0; y < 8; ++y) t += s[y][threadIdx.x];
        red[i] = t;
    }
}

// Stage 2, one thread per OUTPUT element: dgamma[4800], dbeta[4800], dw1[32*12*9], db1[32].
__global__ void encode_reduce_kernel(const float *__restrict__ red, float *__restrict__ dw1, float *__restrict__ db1,
                                     float *__restrict__ dgamma, float *__restrict__ dbeta)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    auto total = [&](int off) { return red[off]; };
    if (i < kD) { dgamma[i] = total(i); return; }
    if (i < 2 * kD) { dbeta[i - kD] = total(i); return; }
    int k = i - 2 * kD;
    const int dense0 = 2 * kD, sparse0 = dense0 + kDenseAcc * kCo;
    if (k < kCo * kCi * 9) {
        const int tap = k % 9, ci = (k / 9) % kCi, co = k / (9 * kCi);
        if (ci >= 2) { dw1[k] = total(sparse0 + ((ci - 2) * 9 + tap) * kCo + co); return; }
        const int r = tap / 3, dx = tap % 3;
        const float white = total(dense0 + tap * kCo + co);
        if (ci == 1) { dw1[k] = white; return; }
        // sum of dz over every position where this tap is inside the board
        float all = total(dense0 + 9 * kCo + co);
        if (r == 0) all -= total(dense0 + 10 * kCo + co);
        if (r == 2) all -= total(dense0 + 11 * kCo + co);
        if (dx == 0) all -= total(dense0 + 12 * kCo + co);
        if (dx == 2) all -= total(dense0 + 13 * kCo + co);
        if (r == 0 && dx == 0) all += total(dense0 + 14 * kCo + co);
        if (r == 0 && dx == 2) all += total(dense0 + 15 * kCo + co);
        if (r == 2 && dx == 0) all += total(dense0 + 16 * kCo + co);
        if (r == 2 && dx == 2) all += total(dense0 + 17 * kCo + co);
        dw1[k] = all - white;
        return;
    }
    k -= kCo * kCi * 9;
    if (k < kCo) db1[k] = total(dense0 + 9 * kCo + k);
}

constexpr size_t kFwdSmem = sizeof(Tables) + (size_t)kFwdWarps * kD * 2;
constexpr size_t kBwdSmem = sizeof(Tables) + (size_t)kBwdWarps * kD * 2 + (size_t)kBwdWarps * kSparse * 9 * kCo * 4;
constexpr const char *kBadArg = "null pointer, count or stride out of range, or view not 0 or 1";

} // namespace

extern "C" {

int inv_encode_partials_floats(void) { return (inv_host::sm_count() + 1) * kPartial; } // per-CTA partials + their sum

int inv_encode_fwd(const void *packed_dev, int64_t stride, int64_t count, int view, const float *w1, const float *b1,
                   const float *gamma_hwc, const float *beta_hwc, float eps, void *y_out, float *extra_out,
                   float *mean_out, float *rstd_out, void *stream)
{
    const char *who = "inv_encode_fwd";
    if (int rc = inv_host::require_sm100(who)) return rc;
    if (!packed_dev || !w1 || !b1 || !gamma_hwc || !beta_hwc || !y_out || !mean_out || !rstd_out || count < 0 ||
        stride < count || (view != 0 && view != 1))
        return inv_host::set_error(INV_ERR_INVALID_ARG, who, kBadArg);
    if (count == 0) return INV_OK;
    if (inv_host::allow_dynamic_smem((const void *)encode_fwd_kernel, kFwdSmem) != cudaSuccess) return inv_host::launch_status(who);
    const int64_t want = (count + kFwdWarps - 1) / kFwdWarps, nsm = inv_host::sm_count();
    const unsigned grid = (unsigned)(want < nsm ? want : nsm);
    encode_fwd_kernel<<<grid, kFwdWarps * 32, kFwdSmem, (cudaStream_t)stream>>>(
        static_cast<const uint32_t *>(packed_dev), stride, count, view, w1, b1, reinterpret_cast<const float2 *>(gamma_hwc),
        reinterpret_cast<const float2 *>(beta_hwc), eps, static_cast<uint32_t *>(y_out),
        reinterpret_cast<float4 *>(extra_out), mean_out, rstd_out);
    return inv_host::launch_status(who);
}

int inv_encode_bwd(const void *packed_dev, int64_t stride, int64_t count, int view, const float *w1, const float *b1,
                   const float *gamma_hwc, const float *beta_hwc, const float *mean, const float *rstd, const void *dy,
                   float *dw1, float *db1, float *dgamma_hwc, float *dbeta_hwc, float *partials, void *stream)
{
    const char *who = "inv_encode_bwd";
    if (int rc = inv_host::require_sm100(who)) return rc;
    if (!packed_dev || !w1 || !b1 || !gamma_hwc || !beta_hwc || !mean || !rstd || !dy || !dw1 || !db1 || !dgamma_hwc ||
        !dbeta_hwc || !partials || count <= 0 || stride < count || (view != 0 && view != 1))
        return inv_host::set_error(INV_ERR_INVALID_ARG, who, kBadArg);
    if (inv_host::allow_dynamic_smem((const void *)encode_bwd_kernel, kBwdSmem) != cudaSuccess) return inv_host::launch_status(who);
    const int64_t want = (count + kBwdWarps - 1) / kBwdWarps, nsm = inv_host::sm_count();
    const int grid = (int)(want < nsm ? want : nsm);
    cudaStream_t st = (cudaStream_t)stream;
    encode_bwd_kernel<<<grid, kBwdWarps * 32, kBwdSmem, st>>>(
        static_cast<const uint32_t *>(packed_dev), stride, count, view, w1, b1, reinterpret_cast<const float2 *>(gamma_hwc),
        reinterpret_cast<const float2 *>(beta_hwc), mean, rstd, static_cast<const uint32_t *>(dy), partials);
    if (int rc = inv_host::launch_status(who)) return rc;
    float *red = partials + (size_t)nsm * kPartial;
    encode_sum_partials_kernel<<<(kPartial + 31) / 32, dim3(32, 8), 0, st>>>(partials, grid, red);
    const int outputs = 2 * kD + kCo * kCi * 9 + kCo;
    encode_reduce_kernel<<<(outputs + 127) / 128, 128, 0, st>>>(red, dw1, db1, dgamma_hwc, dbeta_hwc);
    return inv_host::launch_status(who);
}

} // extern "C"
