// inversus_b200.cu -- host side of the C ABI declared in include/inversus_b200.h.
//
// The handle owns all device memory (packed state planes + every output buffer); callers see raw
// device pointers through inv_get_buffer and may wrap them without copies. No torch, no
// third-party code: CUDA runtime only. There is deliberately no CPU fallback -- every entry point
// fails with INV_ERR_NO_DEVICE / INV_ERR_CUDA when no sm_100 device is usable.
#include "inversus_kernels.cuh"

#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <thread>
#include <vector>

using namespace inv;

namespace inv_host { // host_expand.cpp
void expand_f32(const uint32_t *bits, float *dst, int64_t lo, int64_t hi, int nthreads);
int hardware_threads();
bool stage_action_ids(int8_t *dst, const int8_t *src, int64_t n);
bool check_action_ids(const int8_t *src, int64_t n);
} // namespace inv_host

struct inv_sim {
    inv_config cfg;
    int64_t n;
    uint4 *state;
    void *obs1, *obs2;
    float *extra1, *extra2, *reward;
    uint8_t *done, *info, *dbg;
    int32_t *ep_steps;
    double *ep_return, *reward64;
    uint32_t *status;
    const uint32_t *table;
    int sm_count;
    int64_t launches;
    bool was_reset;
    // staging for the *_host calls: pinned host + device copies of the action ids
    int8_t *h_a1, *h_a2, *d_a1, *d_a2;
    uint32_t *h_status;
    cudaStream_t host_stream, copy_stream; // *_host calls: kernels on host_stream, D2H copies on copy_stream
    // ordering of the *_host calls after launches the caller enqueued on its own streams
    cudaEvent_t ev_last;
    bool ev_last_valid, need_device_sync;
    cudaEvent_t ev_kernel[8], ev_bits[8], ev_t0, ev_t1;
    // the small per-env outputs live in ONE device block (extra1, extra2, reward, episode_steps,
    // episode_return, done, info) so that the *_host calls can fetch them with a single copy
    char *d_small, *h_small;
    size_t small_bytes, off_extra1, off_extra2, off_reward, off_steps, off_return, off_done, off_info;
    // host-expand path of inv_step_host (f32 obs only): packed rows device + pinned host staging
    int host_threads;   // 0 = plain DMA of the f32 observation
    double dma_frac;    // share of the envs whose f32 observation is copied directly (rest expanded)
    bool dma_frac_auto;
    uint4 *d_bits[2];
    uint32_t *h_bits[2];
    double last_dma_s, last_expand_s;
    // inv_step_host_events: compact list of the episodes that ended in the step
    char *d_events;         // [16-byte header: int64 count][n records of inv_episode_event]
    int32_t *d_ev_counts;   // finished episodes per block of kEvBlockEnvs envs
    int64_t *h_ev_count;    // pinned landing slot of the header
    int64_t ev_guess;       // records fetched together with the header (1.5 x the last count)
    cudaEvent_t ev_events;
};

static thread_local char g_err[512] = "";

static int fail(int code, const char *fmt, const char *a = "", const char *b = "")
{
    snprintf(g_err, sizeof(g_err), fmt, a, b);
    return code;
}

#define CUDA_TRY(expr)                                                                      \
    do {                                                                                    \
        cudaError_t e_ = (expr);                                                            \
        if (e_ != cudaSuccess) return fail(INV_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(e_)); \
    } while (0)

namespace {

__global__ void init_episode_kernel(uint4 *plane2, int64_t n)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) plane2[i] = make_uint4(0xFFFFFFFFu, 0u, 0u, 0u); // episode = "none yet", return = 0.0
}

// Generalised advantage estimation over a [T][N] rollout, one thread per env, walking time
// backwards (ppo_agent.py:127-157). float32 arithmetic in the reference's operation order
// (numpy 2 keeps python-float constants "weak", so every product/sum there is float32); _rn
// intrinsics forbid fma contraction so the result is bit-identical to the numpy loop.
// N = 1, T = len(buffer) reproduces the reference's flat-list quirk (values[t+1] of the NEXT
// list element, whatever env it belongs to).
__global__ void gae_kernel(const float *__restrict__ reward, const float *__restrict__ value,
                           const uint8_t *__restrict__ done, const float *__restrict__ last_value, float gamma,
                           float gamma_lam, int T, int64_t N, float *__restrict__ adv, float *__restrict__ ret)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    float next_v = last_value ? last_value[i] : 0.0f;
    float last = 0.0f;
    for (int t = T - 1; t >= 0; --t) {
        const int64_t k = (int64_t)t * N + i;
        const float r = reward[k], v = value[k];
        if (done[k]) {
            last = __fsub_rn(r, v);                                            // :146-147
        } else {
            const float delta = __fsub_rn(__fadd_rn(r, __fmul_rn(gamma, next_v)), v); // :149
            last = __fadd_rn(delta, __fmul_rn(gamma_lam, last));               // :150
        }
        adv[k] = last;                                                         // :151
        ret[k] = __fadd_rn(last, v);                                           // :154
        next_v = v;
    }
}

// ---- finished-episode list (inv_step_host_events) -----------------------------------------------
// Two small launches over the done flags, deterministic and in env order: blocks of kEvBlockEnvs envs
// count their finished episodes, then every block sums the counts before it, scans its own threads
// and writes its records. 16 done bytes per thread and load.
constexpr int kEvThreads = 256, kEvPerThread = 16, kEvBlockEnvs = kEvThreads * kEvPerThread;
constexpr size_t kEvHeaderBytes = 16;
static_assert(sizeof(inv_episode_event) == 24, "inv_episode_event is 24 bytes in the ABI");

__device__ __forceinline__ uint32_t done_mask16(const uint8_t *__restrict__ done, int64_t i, int64_t n)
{
    uint32_t m = 0;
    if (i + kEvPerThread <= n) {
        const uint4 v = *reinterpret_cast<const uint4 *>(done + i);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int q = 0; q < 4; ++q)
#pragma unroll
            for (int b = 0; b < 4; ++b) m |= ((w[q] >> (8 * b)) & 0xFFu) ? 1u << (4 * q + b) : 0u;
    } else {
        for (int k = 0; k < kEvPerThread; ++k)
            if (i + k < n && done[i + k]) m |= 1u << k;
    }
    return m;
}

__global__ void __launch_bounds__(kEvThreads) episode_count_kernel(const uint8_t *__restrict__ done, int64_t n,
                                                                    int32_t *__restrict__ block_counts)
{
    const int64_t i = (int64_t)blockIdx.x * kEvBlockEnvs + (int64_t)threadIdx.x * kEvPerThread;
    int c = i < n ? __popc(done_mask16(done, i, n)) : 0;
    c = __reduce_add_sync(0xffffffffu, c);
    __shared__ int s_c[kEvThreads / 32];
    if ((threadIdx.x & 31) == 0) s_c[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int w = 0; w < kEvThreads / 32; ++w) t += s_c[w];
        block_counts[blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(kEvThreads)
episode_write_kernel(const uint8_t *__restrict__ done, const uint8_t *__restrict__ info,
                     const int32_t *__restrict__ ep_steps, const double *__restrict__ ep_return, int64_t n,
                     const int32_t *__restrict__ block_counts, int64_t *__restrict__ header,
                     inv_episode_event *__restrict__ events)
{
    __shared__ long long s_part[kEvThreads / 32];
    __shared__ int s_w[kEvThreads / 32];
    __shared__ long long s_base;
    // records of the blocks before this one (and, in the last block, the grand total for the header)
    long long before = 0, total = 0;
    for (int b = threadIdx.x; b < (int)gridDim.x; b += kEvThreads) {
        const int c = block_counts[b];
        total += c;
        if (b < (int)blockIdx.x) before += c;
    }
    for (int o = 16; o > 0; o >>= 1) {
        before += __shfl_xor_sync(0xffffffffu, before, o);
        total += __shfl_xor_sync(0xffffffffu, total, o);
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) s_part[warp] = before;
    __syncthreads();
    if (threadIdx.x == 0) {
        long long t = 0;
        for (int w = 0; w < kEvThreads / 32; ++w) t += s_part[w];
        s_base = t;
    }
    __syncthreads();
    if (blockIdx.x == gridDim.x - 1) { // total: same reduction once more, by the last block only
        if (lane == 0) s_part[warp] = total;
        __syncthreads();
        if (threadIdx.x == 0) {
            long long t = 0;
            for (int w = 0; w < kEvThreads / 32; ++w) t += s_part[w];
            header[0] = t;
        }
    }
    const int64_t i = (int64_t)blockIdx.x * kEvBlockEnvs + (int64_t)threadIdx.x * kEvPerThread;
    const uint32_t m = i < n ? done_mask16(done, i, n) : 0u;
    const int c = __popc(m);
    int incl = c; // inclusive scan of the per-thread counts: warp, then across the block's warps
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    int woff = 0;
    for (int w = 0; w < warp; ++w) woff += s_w[w];
    long long pos = s_base + woff + incl - c;
    for (uint32_t mm = m; mm; mm &= mm - 1) {
        const int64_t e = i + (__ffs(mm) - 1);
        inv_episode_event r;
        r.env = e;
        r.episode_return = ep_return[e];
        r.episode_steps = ep_steps[e];
        r.info = info[e];
        events[pos++] = r;
    }
}

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) cudaSetDevice(dev);
        else prev = -1;
    }
    ~DeviceGuard()
    {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

size_t obs_elem_bytes(int dt) { return dt == INV_OBS_F32 ? 4 : dt == INV_OBS_BF16 ? 2 : dt == INV_OBS_U8 ? 1 : 0; }
size_t obs_env_bytes(int dt) { return (size_t)INV_OBS_ELEMS * obs_elem_bytes(dt); }

Params base_params(const inv_sim *s)
{
    Params p;
    memset(&p, 0, sizeof(p));
    p.state = s->state;
    p.stride = s->n;
    p.count = s->n;
    p.table = s->table;
    p.obs1 = s->obs1; p.obs2 = s->obs2;
    p.bits1 = nullptr; p.bits2 = nullptr;
    p.extra1 = s->extra1; p.extra2 = s->extra2;
    p.reward = s->reward; p.reward64 = s->reward64; p.done = s->done; p.info = s->info; p.dbg = s->dbg;
    p.ep_steps = s->ep_steps; p.ep_return = s->ep_return;
    p.status = s->status;
    p.seed_lo = (uint32_t)s->cfg.seed;
    p.seed_hi = (uint32_t)(s->cfg.seed >> 32);
    p.env_id_base = (uint32_t)s->cfg.env_id_base;
    p.mode = s->cfg.mode;
    p.difficulty = s->cfg.difficulty;
    p.max_steps = s->cfg.max_episode_steps;
    p.auto_reset = (s->cfg.flags & INV_FLAG_AUTO_RESET) ? 1 : 0;
    return p;
}

// Launch shape (measured, profiles/r1_tile_grid_sweep.txt): 128-thread CTAs, a tile of E envs per
// CTA (E/32 warps run the game logic, all four stream the observations) and ONE CTA PER TILE.
// Letting the hardware block scheduler hand out tiles keeps CTAs desynchronised, so logic phases
// of some overlap store phases of others: 0.99 of the measured HBM peak at 1M-4M envs for fp32
// observations with E = 32, versus 0.94 for a persistent grid-stride loop (whose CTAs drift into
// lock-step). The narrower the observation, the more logic per stored byte, so bf16/u8 step
// kernels use more logic warps per CTA: E = 64 (bf16, one view) or 128 (bf16 two views, u8).
constexpr int kTileEnvs = 32;
// fp32 observations, large batches (round 2, profiles/r2_variants_f32*.txt): 32-byte stores plus
// more store warps per CTA lift the step kernel from 6.39 to 6.93 TB/s (a pure store stream in
// the same shape reaches 7.1-7.5 TB/s, profiles/r2_store_ceiling.txt). Small batches keep the
// 32-env / 128-thread shape (more CTAs, shorter critical path).
#ifndef INV_BF16_E   // bf16 one-view step: tile envs / threads per CTA
#define INV_BF16_E 64
#endif
#ifndef INV_BF16_T
#define INV_BF16_T 128
#endif
#ifndef INV_NARROW_E // u8 and two-view bf16 steps
#define INV_NARROW_E 128
#endif
#ifndef INV_NARROW_T
#define INV_NARROW_T 128
#endif
#ifndef INV_WIDE_MIN_ENVS
#define INV_WIDE_MIN_ENVS 131072
#endif

template <int OP, int DT, bool P2V, bool INDEXED, int E, int T = kThreads>
cudaError_t launch_one(const Params &p, int sm_count, cudaStream_t st)
{
    (void)sm_count;
    auto kern = inv_kernel<OP, DT, P2V, INDEXED, E, T>;
    constexpr size_t smem = smem_bytes<E, P2V, INDEXED, DT>();
    static bool configured[64] = {}; // per instantiation and per device (function attributes are per device)
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64) configured[dev] = true;
    }
    const int64_t ntiles = (p.count + E - 1) / E;
    if (ntiles <= 0) return cudaSuccess;
    const unsigned grid = (unsigned)(ntiles < (int64_t)0x7FFFFFFF ? ntiles : (int64_t)0x7FFFFFFF);
    kern<<<grid, T, smem, st>>>(p);
    return cudaGetLastError();
}

template <int OP, int DT, bool P2V, bool INDEXED>
cudaError_t launch_e(const Params &p, int sm_count, cudaStream_t st)
{
    if constexpr (DT == INV_OBS_NONE && !INDEXED && OP != OP_DEBUG) {
        return launch_one<OP, DT, P2V, false, 128, 128>(p, sm_count, st); // pure thread-per-env, no store phase
    } else if constexpr (OP == OP_STEP && !INDEXED && DT != INV_OBS_F32) {
        constexpr int E = (DT == INV_OBS_BF16 && !P2V) ? INV_BF16_E : INV_NARROW_E;
        constexpr int T = (DT == INV_OBS_BF16 && !P2V) ? INV_BF16_T : INV_NARROW_T;
        return launch_one<OP_STEP, DT, P2V, false, E, T>(p, sm_count, st);
    } else if constexpr (DT == INV_OBS_F32 && !INDEXED && OP != OP_DEBUG) {
        if (p.count >= INV_WIDE_MIN_ENVS) {
            if constexpr (OP == OP_STEP && !P2V) return launch_one<OP, DT, P2V, false, 64, 256>(p, sm_count, st);
            else if constexpr (OP == OP_STEP) return launch_one<OP, DT, P2V, false, 64, 384>(p, sm_count, st);
            else return launch_one<OP, DT, P2V, false, 128, 512>(p, sm_count, st);
        }
        return launch_one<OP, DT, P2V, INDEXED, kTileEnvs>(p, sm_count, st);
    } else {
        return launch_one<OP, DT, P2V, INDEXED, kTileEnvs>(p, sm_count, st);
    }
}

template <int OP, bool INDEXED>
cudaError_t launch(const Params &p, int dt, bool p2v, int sm_count, cudaStream_t st)
{
#define INV_CASE(DTV)                                                                   \
    case DTV:                                                                           \
        return p2v ? launch_e<OP, DTV, true, INDEXED>(p, sm_count, st)                  \
                   : launch_e<OP, DTV, false, INDEXED>(p, sm_count, st);
    switch (dt) {
        INV_CASE(INV_OBS_F32)
        INV_CASE(INV_OBS_BF16)
        INV_CASE(INV_OBS_U8)
        INV_CASE(INV_OBS_NONE)
    default:
        return cudaErrorInvalidValue;
    }
#undef INV_CASE
}

} // namespace

extern "C" {

int inv_abi_version(void) { return INV_ABI_VERSION; }
const char *inv_last_error(void) { return g_err; }

int inv_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int inv_create(const inv_config *cfg, inv_sim **out)
{
    if (!cfg || !out) return fail(INV_ERR_INVALID_ARG, "inv_create: null argument");
    *out = nullptr;
    if (cfg->n_envs <= 0) return fail(INV_ERR_INVALID_ARG, "inv_create: n_envs must be positive");
    if (cfg->mode != INV_MODE_DUMMY && cfg->mode != INV_MODE_SELFPLAY)
        return fail(INV_ERR_INVALID_ARG, "Unknown opponent_type"); // env_wrappers.py:316
    if (cfg->difficulty != INV_DIFFICULTY_EASY && cfg->difficulty != INV_DIFFICULTY_HARD)
        return fail(INV_ERR_INVALID_ARG, "inv_create: difficulty must be easy(0) or hard(1)");
    if (cfg->obs_dtype < INV_OBS_F32 || cfg->obs_dtype > INV_OBS_NONE)
        return fail(INV_ERR_INVALID_ARG, "inv_create: unknown obs_dtype");
    if (cfg->max_episode_steps <= 0) return fail(INV_ERR_INVALID_ARG, "inv_create: max_episode_steps must be positive");
    if (cfg->env_id_base < 0 || cfg->env_id_base + cfg->n_envs > 0xFFFFFFFFll)
        return fail(INV_ERR_INVALID_ARG, "inv_create: global env ids must fit 32 bits");
    int ndev = inv_device_count();
    if (ndev <= 0) return fail(INV_ERR_NO_DEVICE, "no CUDA device: this simulator has no CPU fallback");
    if (cfg->device < 0 || cfg->device >= ndev) return fail(INV_ERR_INVALID_ARG, "inv_create: bad device ordinal");
    DeviceGuard g(cfg->device);
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, cfg->device));
    if (prop.major != 10)
        return fail(INV_ERR_NO_DEVICE, "device is not sm_100 (B200): kernels are built for sm_100a only");

    inv_sim *s = new (std::nothrow) inv_sim();
    if (!s) return fail(INV_ERR_INVALID_ARG, "out of host memory");
    memset(s, 0, sizeof(*s));
    s->cfg = *cfg;
    if (cfg->mode == INV_MODE_SELFPLAY) s->cfg.flags |= INV_FLAG_P2_VIEW; // env_wrappers.py:311
    s->n = cfg->n_envs;
    s->sm_count = prop.multiProcessorCount;
    s->host_threads = inv_host::hardware_threads() > 32 ? 32 : inv_host::hardware_threads();
    s->dma_frac = 0.35;
    s->dma_frac_auto = true;
    const int64_t n = s->n;
    const bool p2v = (s->cfg.flags & INV_FLAG_P2_VIEW) != 0;
    const size_t obs_bytes = (size_t)n * INV_OBS_ELEMS * obs_elem_bytes(cfg->obs_dtype);
#define ALLOC(ptr, bytes)                                                        \
    do {                                                                         \
        cudaError_t e_ = cudaMalloc((void **)&(ptr), (bytes));                   \
        if (e_ != cudaSuccess) {                                                 \
            fail(INV_ERR_CUDA, "cudaMalloc(%s): %s", #ptr, cudaGetErrorString(e_)); \
            inv_destroy(s);                                                      \
            return INV_ERR_CUDA;                                                 \
        }                                                                        \
    } while (0)
    ALLOC(s->state, (size_t)n * INV_PACKED_STATE_BYTES);
    if (obs_bytes) {
        ALLOC(s->obs1, obs_bytes);
        if (p2v) ALLOC(s->obs2, obs_bytes);
    }
    {
        auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
        size_t o = 0;
        s->off_extra1 = o; o = up(o + (size_t)n * 16);
        s->off_extra2 = o; o = up(o + (p2v ? (size_t)n * 16 : 0));
        s->off_reward = o; o = up(o + (size_t)n * 4);
        s->off_steps = o; o = up(o + (size_t)n * 4);
        s->off_return = o; o = up(o + (size_t)n * 8);
        s->off_done = o; o = up(o + (size_t)n);
        s->off_info = o; o = up(o + (size_t)n);
        s->small_bytes = o;
        ALLOC(s->d_small, s->small_bytes);
        s->extra1 = reinterpret_cast<float *>(s->d_small + s->off_extra1);
        s->extra2 = p2v ? reinterpret_cast<float *>(s->d_small + s->off_extra2) : nullptr;
        s->reward = reinterpret_cast<float *>(s->d_small + s->off_reward);
        s->ep_steps = reinterpret_cast<int32_t *>(s->d_small + s->off_steps);
        s->ep_return = reinterpret_cast<double *>(s->d_small + s->off_return);
        s->done = reinterpret_cast<uint8_t *>(s->d_small + s->off_done);
        s->info = reinterpret_cast<uint8_t *>(s->d_small + s->off_info);
    }
    ALLOC(s->dbg, (size_t)n);
    if (cfg->flags & INV_FLAG_REWARD_F64) ALLOC(s->reward64, (size_t)n * 8);
    ALLOC(s->status, 4);
    ALLOC(s->d_a1, (size_t)n);
    ALLOC(s->d_a2, (size_t)n);
#undef ALLOC
    // "no episode yet": zero state with episode = 0xFFFFFFFF so that the first reset starts episode 0
    cudaMemset(s->state, 0, (size_t)n * INV_PACKED_STATE_BYTES);
    init_episode_kernel<<<(unsigned)((n + 255) / 256), 256>>>(s->state + 2 * n, n);
    cudaMemset(s->status, 0, 4);
    cudaMemset(s->d_small, 0, s->small_bytes);
    cudaMemset(s->dbg, 0, (size_t)n);
    bool ok = cudaMallocHost((void **)&s->h_status, 4) == cudaSuccess &&
              cudaStreamCreateWithFlags(&s->host_stream, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&s->copy_stream, cudaStreamNonBlocking) == cudaSuccess &&
              cudaEventCreateWithFlags(&s->ev_last, cudaEventDisableTiming) == cudaSuccess &&
              cudaEventCreate(&s->ev_t0) == cudaSuccess && cudaEventCreate(&s->ev_t1) == cudaSuccess;
    for (int c = 0; ok && c < 8; ++c)
        ok = cudaEventCreateWithFlags(&s->ev_kernel[c], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&s->ev_bits[c], cudaEventDisableTiming) == cudaSuccess;
    if (!ok) {
        fail(INV_ERR_CUDA, "pinned staging / stream allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
        inv_destroy(s);
        return INV_ERR_CUDA;
    }
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        fail(INV_ERR_CUDA, "inv_create: %s", cudaGetErrorString(e));
        inv_destroy(s);
        return INV_ERR_CUDA;
    }
    *out = s;
    return INV_OK;
}

int inv_destroy(inv_sim *s)
{
    if (!s) return INV_OK;
    DeviceGuard g(s->cfg.device);
    cudaDeviceSynchronize();
    void *dev[] = {s->state, s->obs1, s->obs2, s->d_small, s->dbg, s->status, s->d_a1, s->d_a2, s->reward64};
    for (void *p : dev)
        if (p) cudaFree(p);
    if (s->h_small) cudaFreeHost(s->h_small);
    if (s->h_a1) cudaFreeHost(s->h_a1);
    if (s->h_a2) cudaFreeHost(s->h_a2);
    if (s->h_status) cudaFreeHost(s->h_status);
    if (s->ev_last) cudaEventDestroy(s->ev_last);
    if (s->ev_t0) cudaEventDestroy(s->ev_t0);
    if (s->ev_t1) cudaEventDestroy(s->ev_t1);
    for (int c = 0; c < 8; ++c) {
        if (s->ev_kernel[c]) cudaEventDestroy(s->ev_kernel[c]);
        if (s->ev_bits[c]) cudaEventDestroy(s->ev_bits[c]);
    }
    if (s->copy_stream) cudaStreamDestroy(s->copy_stream);
    for (int v = 0; v < 2; ++v) {
        if (s->d_bits[v]) cudaFree(s->d_bits[v]);
        if (s->h_bits[v]) cudaFreeHost(s->h_bits[v]);
    }
    if (s->d_events) cudaFree(s->d_events);
    if (s->d_ev_counts) cudaFree(s->d_ev_counts);
    if (s->h_ev_count) cudaFreeHost(s->h_ev_count);
    if (s->ev_events) cudaEventDestroy(s->ev_events);
    if (s->host_stream) cudaStreamDestroy(s->host_stream);
    delete s;
    return INV_OK;
}

int inv_get_config(const inv_sim *s, inv_config *out)
{
    if (!s || !out) return fail(INV_ERR_INVALID_ARG, "inv_get_config: null argument");
    *out = s->cfg;
    return INV_OK;
}

// Launches enqueued on the caller's streams are remembered through one event, so that the
// synchronous *_host calls (which run on the handle's own streams) can order themselves after them
// without a device-wide synchronisation. A launch recorded into a CUDA graph cannot be tracked this
// way; from then on the *_host calls fall back to cudaDeviceSynchronize.
static void note_launch(inv_sim *s, cudaStream_t st)
{
    s->launches += 1;
    if (st == s->host_stream) return;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cap) != cudaSuccess || cap != cudaStreamCaptureStatusNone ||
        cudaEventRecord(s->ev_last, st) != cudaSuccess) {
        cudaGetLastError();
        s->need_device_sync = true;
        return;
    }
    s->ev_last_valid = true;
}

static int order_host_stream(inv_sim *s)
{
    if (s->need_device_sync) CUDA_TRY(cudaDeviceSynchronize());
    else if (s->ev_last_valid) CUDA_TRY(cudaStreamWaitEvent(s->host_stream, s->ev_last, 0));
    return INV_OK;
}

// The same launch restricted to envs [first, first + count): every per-env pointer moves, the plane
// stride and the global-id base keep describing the whole handle.
static Params chunk_params(const Params &b, int64_t first, int64_t count, size_t env_bytes)
{
    Params p = b;
    p.state = b.state + first;
    p.count = count;
    if (b.a1) p.a1 = b.a1 + first;
    if (b.a2) p.a2 = b.a2 + first;
    if (b.table) p.table = b.table + first * INV_TABLE_STRIDE;
    p.obs1 = static_cast<char *>(b.obs1) + (size_t)first * env_bytes;
    if (b.obs2) p.obs2 = static_cast<char *>(b.obs2) + (size_t)first * env_bytes;
    if (b.bits1) p.bits1 = b.bits1 + first * 16;
    if (b.bits2) p.bits2 = b.bits2 + first * 16;
    p.extra1 = b.extra1 + first * 4;
    if (b.extra2) p.extra2 = b.extra2 + first * 4;
    p.reward = b.reward + first;
    if (b.reward64) p.reward64 = b.reward64 + first;
    p.done = b.done + first;
    p.info = b.info + first;
    p.dbg = b.dbg + first;
    p.ep_steps = b.ep_steps + first;
    p.ep_return = b.ep_return + first;
    p.env_id_base = b.env_id_base + (uint32_t)first;
    return p;
}

int inv_reset(inv_sim *s, void *stream)
{
    if (!s) return fail(INV_ERR_INVALID_ARG, "inv_reset: null handle");
    DeviceGuard g(s->cfg.device);
    Params p = base_params(s);
    CUDA_TRY((launch<OP_RESET, false>(p, s->cfg.obs_dtype, (s->cfg.flags & INV_FLAG_P2_VIEW) != 0, s->sm_count,
                                      (cudaStream_t)stream)));
    note_launch(s, (cudaStream_t)stream);
    s->was_reset = true;
    return INV_OK;
}

int inv_reset_envs(inv_sim *s, const int64_t *idx_dev, int64_t count, void *stream)
{
    if (!s || (!idx_dev && count > 0)) return fail(INV_ERR_INVALID_ARG, "inv_reset_envs: null argument");
    if (count < 0 || count > s->n) return fail(INV_ERR_INVALID_ARG, "inv_reset_envs: bad count");
    if (count == 0) return INV_OK;
    DeviceGuard g(s->cfg.device);
    Params p = base_params(s);
    p.idx = idx_dev;
    p.count = count;
    CUDA_TRY((launch<OP_RESET, true>(p, s->cfg.obs_dtype, (s->cfg.flags & INV_FLAG_P2_VIEW) != 0, s->sm_count,
                                     (cudaStream_t)stream)));
    note_launch(s, (cudaStream_t)stream);
    return INV_OK;
}

// One fused step launch over envs [first, first + count).
static int step_impl(inv_sim *s, const int8_t *a1, const int8_t *a2, void *stream, uint4 *bits1, uint4 *bits2,
                     int64_t first, int64_t count)
{
    if (!s || !a1) return fail(INV_ERR_INVALID_ARG, "inv_step: null argument");
    if (!s->was_reset) return fail(INV_ERR_NOT_RESET, "inv_step before inv_reset");
    if (s->cfg.mode == INV_MODE_SELFPLAY && !a2)
        return fail(INV_ERR_INVALID_ARG, "opponent_policy required for selfplay mode"); // env_wrappers.py:309
    DeviceGuard g(s->cfg.device);
    Params p = base_params(s);
    p.a1 = a1;
    p.a2 = a2;
    p.bits1 = bits1;
    p.bits2 = bits2;
    if (first != 0 || count != s->n) p = chunk_params(p, first, count, obs_env_bytes(s->cfg.obs_dtype));
    CUDA_TRY((launch<OP_STEP, false>(p, s->cfg.obs_dtype, (s->cfg.flags & INV_FLAG_P2_VIEW) != 0, s->sm_count,
                                     (cudaStream_t)stream)));
    note_launch(s, (cudaStream_t)stream);
    return INV_OK;
}

int inv_step(inv_sim *s, const int8_t *a1, const int8_t *a2, void *stream)
{
    return step_impl(s, a1, a2, stream, nullptr, nullptr, 0, s ? s->n : 0);
}

// ------------------------------------------------------------------------------------------------
// Host-buffer calls (the numpy contract of MultiEnvRunner.step). The batch is cut into up to 8 env
// chunks; chunk c's kernel runs on host_stream while copy_stream brings chunk c-1's outputs to the
// host, and the host threads expand the packed observation rows of chunk c-2.
constexpr int kMaxHostChunks = 8;
constexpr int64_t kHostChunkMinEnvs = 131072;  // chunks keep the wide launch shape
constexpr size_t kStagedSmallMax = 8u << 20;   // small outputs: one staged copy up to 8 MB, direct copies above

struct SmallOut {
    float *extra_p1, *extra_p2, *reward;
    uint8_t *done, *info;
    int32_t *episode_steps;
    double *episode_return;
};

static int ensure_host_staging(inv_sim *s)
{
    const size_t n = (size_t)s->n;
    if (!s->h_a1) CUDA_TRY(cudaMallocHost((void **)&s->h_a1, n));
    if (!s->h_a2) CUDA_TRY(cudaMallocHost((void **)&s->h_a2, n));
    size_t staged_max = kStagedSmallMax;
    if (const char *e = getenv("INV_HOST_STAGED_MAX")) staged_max = (size_t)atoll(e); // tests: force the direct-copy path
    if (!s->h_small && s->small_bytes <= staged_max) CUDA_TRY(cudaMallocHost((void **)&s->h_small, s->small_bytes));
    return INV_OK;
}

// After the copies have landed: scatter the staged small-output block to the caller.
static void scatter_small_outputs(inv_sim *s, const SmallOut &o)
{
    if (!s->h_small) return;
    const size_t n = (size_t)s->n;
    if (o.extra_p1) memcpy(o.extra_p1, s->h_small + s->off_extra1, n * 16);
    if (o.extra_p2 && s->extra2) memcpy(o.extra_p2, s->h_small + s->off_extra2, n * 16);
    if (o.reward) memcpy(o.reward, s->h_small + s->off_reward, n * 4);
    if (o.episode_steps) memcpy(o.episode_steps, s->h_small + s->off_steps, n * 4);
    if (o.episode_return) memcpy(o.episode_return, s->h_small + s->off_return, n * 8);
    if (o.done) memcpy(o.done, s->h_small + s->off_done, n);
    if (o.info) memcpy(o.info, s->h_small + s->off_info, n);
}

// Small outputs of envs [first, first + count) to the host: the whole block into the staging buffer
// (small batches, one copy), or straight into the caller's arrays.
static int copy_small_outputs(inv_sim *s, cudaStream_t st, const SmallOut &o, int64_t first, int64_t count)
{
    if (s->h_small) {
        if (first == 0) CUDA_TRY(cudaMemcpyAsync(s->h_small, s->d_small, s->small_bytes, cudaMemcpyDeviceToHost, st));
        return INV_OK;
    }
    const size_t f = (size_t)first, c = (size_t)count;
    if (o.extra_p1) CUDA_TRY(cudaMemcpyAsync(o.extra_p1 + f * 4, s->extra1 + f * 4, c * 16, cudaMemcpyDeviceToHost, st));
    if (o.extra_p2) CUDA_TRY(cudaMemcpyAsync(o.extra_p2 + f * 4, s->extra2 + f * 4, c * 16, cudaMemcpyDeviceToHost, st));
    if (o.reward) CUDA_TRY(cudaMemcpyAsync(o.reward + f, s->reward + f, c * 4, cudaMemcpyDeviceToHost, st));
    if (o.done) CUDA_TRY(cudaMemcpyAsync(o.done + f, s->done + f, c, cudaMemcpyDeviceToHost, st));
    if (o.info) CUDA_TRY(cudaMemcpyAsync(o.info + f, s->info + f, c, cudaMemcpyDeviceToHost, st));
    if (o.episode_steps) CUDA_TRY(cudaMemcpyAsync(o.episode_steps + f, s->ep_steps + f, c * 4, cudaMemcpyDeviceToHost, st));
    if (o.episode_return) CUDA_TRY(cudaMemcpyAsync(o.episode_return + f, s->ep_return + f, c * 8, cudaMemcpyDeviceToHost, st));
    return INV_OK;
}

static bool use_host_expand(const inv_sim *s, const void *obs_p1, const void *obs_p2)
{
    return s->host_threads > 0 && s->cfg.obs_dtype == INV_OBS_F32 && (obs_p1 || obs_p2) && s->n >= 4096;
}

static int ensure_bits_staging(inv_sim *s, bool p2)
{
    for (int v = 0; v < (p2 ? 2 : 1); ++v) {
        if (!s->d_bits[v]) CUDA_TRY(cudaMalloc((void **)&s->d_bits[v], (size_t)s->n * 256));
        if (!s->h_bits[v]) CUDA_TRY(cudaMallocHost((void **)&s->h_bits[v], (size_t)s->n * 256));
    }
    return INV_OK;
}

// What every host-buffer step starts with: the reference's argument errors, then the action ids
// host -> pinned staging -> device on the handle's own stream.
static int begin_host_step(inv_sim *s, const int8_t *a1, const int8_t *a2, const char *who)
{
    if (!s || !a1) return fail(INV_ERR_INVALID_ARG, "%s: null argument", who);
    if (!s->was_reset) return fail(INV_ERR_NOT_RESET, "%s before inv_reset", who);
    const bool selfplay = s->cfg.mode == INV_MODE_SELFPLAY;
    if (selfplay && !a2) return fail(INV_ERR_INVALID_ARG, "opponent_policy required for selfplay mode");
    const int64_t n = s->n;
    int rc = ensure_host_staging(s);
    if (rc != INV_OK) return rc;
    // discrete_to_action raises before anything is stepped (env_wrappers.py:302, :66): the ids are
    // checked in the same pass that moves them into the pinned staging buffer, and nothing has been
    // enqueued when the error is reported
    // Ids the caller already keeps in page-locked memory are only checked and go up from where they
    // are (the call synchronises before it returns, so the caller cannot change them under the copy).
    auto page_locked = [](const void *p) {
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
            cudaGetLastError();
            return false;
        }
        return at.type == cudaMemoryTypeHost;
    };
    const int8_t *src1 = s->h_a1, *src2 = s->h_a2;
    bool bad;
    if (page_locked(a1)) { bad = inv_host::check_action_ids(a1, n); src1 = a1; }
    else bad = inv_host::stage_action_ids(s->h_a1, a1, n);
    if (selfplay) {
        if (page_locked(a2)) { bad |= inv_host::check_action_ids(a2, n); src2 = a2; }
        else bad |= inv_host::stage_action_ids(s->h_a2, a2, n);
    }
    if (bad) return fail(INV_ERR_INVALID_ACTION, "Invalid action_id: must be 0-12");
    if ((rc = order_host_stream(s)) != INV_OK) return rc;
    CUDA_TRY(cudaMemcpyAsync(s->d_a1, src1, (size_t)n, cudaMemcpyHostToDevice, s->host_stream));
    if (selfplay) CUDA_TRY(cudaMemcpyAsync(s->d_a2, src2, (size_t)n, cudaMemcpyHostToDevice, s->host_stream));
    return INV_OK;
}

// Env ranges of the pipelined host step; returns the number of chunks, bounds[0 .. chunks] filled.
static int host_chunk_bounds(int64_t n, bool with_obs, bool single, int64_t *bounds)
{
    int nchunks = (int)(n / kHostChunkMinEnvs);
    nchunks = nchunks < 1 ? 1 : (nchunks > kMaxHostChunks ? kMaxHostChunks : nchunks);
    if (!with_obs && nchunks > 4) nchunks = 4; // small outputs only: fewer, larger copies
    if (const char *e = getenv("INV_HOST_CHUNKS")) { // experiments (profiles/)
        const int v = atoi(e);
        if (v >= 1 && v <= kMaxHostChunks && (int64_t)v <= n / 256) nchunks = v;
    }
    if (single) nchunks = 1;
    const int64_t per = ((n + nchunks - 1) / nchunks + 255) & ~(int64_t)255;
    // small outputs only: what is not overlapped is the LAST chunk's copy, so the chunks shrink
    // towards the end (3 : 3 : 1 : 1)
    const bool tapered = !with_obs && nchunks == 4;
    for (int c = 0; c <= nchunks; ++c) {
        int64_t b = tapered ? (n * (c == 0 ? 0 : c == 1 ? 3 : c == 2 ? 6 : c == 3 ? 7 : 8) / 8) & ~(int64_t)255
                            : (int64_t)c * per;
        bounds[c] = (c == nchunks || b > n) ? n : b;
    }
    return nchunks;
}

int inv_step_host(inv_sim *s, const int8_t *a1, const int8_t *a2, void *obs_p1, float *extra_p1, void *obs_p2,
                  float *extra_p2, float *reward, uint8_t *done, uint8_t *info, int32_t *episode_steps,
                  double *episode_return)
{
    if (!s) return fail(INV_ERR_INVALID_ARG, "inv_step_host: null argument");
    if (obs_p1 && !s->obs1) return fail(INV_ERR_INVALID_ARG, "this handle keeps no observation tensor (INV_OBS_NONE)");
    if (obs_p2 && !s->obs2) return fail(INV_ERR_INVALID_ARG, "P2 view was not enabled (INV_FLAG_P2_VIEW)");
    if (extra_p2 && !s->extra2) return fail(INV_ERR_INVALID_ARG, "P2 view was not enabled (INV_FLAG_P2_VIEW)");
    DeviceGuard g(s->cfg.device);
    int rc = begin_host_step(s, a1, a2, "inv_step_host");
    if (rc != INV_OK) return rc;
    const int64_t n = s->n;
    const bool selfplay = s->cfg.mode == INV_MODE_SELFPLAY;
    const bool expand = use_host_expand(s, obs_p1, obs_p2);
    if (expand && (rc = ensure_bits_staging(s, obs_p2 != nullptr)) != INV_OK) return rc;
    cudaStream_t ks = s->host_stream, cs = s->copy_stream;
    int64_t bounds[kMaxHostChunks + 1];
    const int nchunks = host_chunk_bounds(n, obs_p1 || obs_p2, s->h_small != nullptr, bounds);
    const SmallOut so = {extra_p1, extra_p2, reward, done, info, episode_steps, episode_return};
    const size_t env_bytes = (size_t)INV_OBS_ELEMS * obs_elem_bytes(s->cfg.obs_dtype);
    void *dst[2] = {obs_p1, obs_p2};
    const void *src[2] = {s->obs1, s->obs2};
    const double frac = expand ? s->dma_frac : 1.0; // share of each chunk's envs whose f32 data is copied directly
    int64_t lo[kMaxHostChunks], mid[kMaxHostChunks], hi[kMaxHostChunks];

    // all kernels are enqueued first (the launch stream never waits for the host to issue copies) ...
    int used = 0;
    for (int c = 0; c < nchunks; ++c) {
        const int64_t first = bounds[c];
        if (first >= n) break;
        const int64_t count = bounds[c + 1] - first;
        if (count <= 0) break;
        lo[c] = first;
        hi[c] = first + count;
        mid[c] = expand ? first + ((int64_t)((double)count * frac) & ~(int64_t)255) : first + count;
        rc = step_impl(s, s->d_a1, selfplay ? s->d_a2 : nullptr, ks, expand ? s->d_bits[0] : nullptr,
                       expand && obs_p2 ? s->d_bits[1] : nullptr, first, count);
        if (rc != INV_OK) return rc;
        CUDA_TRY(cudaEventRecord(s->ev_kernel[c], ks));
        used = c + 1;
    }
    // ... then the copy stream follows chunk by chunk
    CUDA_TRY(cudaEventRecord(s->ev_t0, cs));
    for (int c = 0; c < used; ++c) {
        CUDA_TRY(cudaStreamWaitEvent(cs, s->ev_kernel[c], 0));
        if ((rc = copy_small_outputs(s, cs, so, lo[c], hi[c] - lo[c])) != INV_OK) return rc;
        if (expand) { // packed rows of the envs the host will expand
            for (int v = 0; v < 2; ++v)
                if (dst[v] && hi[c] > mid[c])
                    CUDA_TRY(cudaMemcpyAsync(s->h_bits[v] + (size_t)mid[c] * 64, s->d_bits[v] + (size_t)mid[c] * 16,
                                             (size_t)(hi[c] - mid[c]) * 256, cudaMemcpyDeviceToHost, cs));
            CUDA_TRY(cudaEventRecord(s->ev_bits[c], cs));
        }
        for (int v = 0; v < 2; ++v) // the directly copied observations
            if (dst[v] && mid[c] > lo[c])
                CUDA_TRY(cudaMemcpyAsync(static_cast<char *>(dst[v]) + (size_t)lo[c] * env_bytes,
                                         static_cast<const char *>(src[v]) + (size_t)lo[c] * env_bytes,
                                         (size_t)(mid[c] - lo[c]) * env_bytes, cudaMemcpyDeviceToHost, cs));
    }
    CUDA_TRY(cudaEventRecord(s->ev_t1, cs));

    double expand_s = 0.0;
    if (expand) { // host side: expand chunk c as soon as its packed rows have landed
        using clk = std::chrono::steady_clock;
        for (int c = 0; c < used; ++c) {
            CUDA_TRY(cudaEventSynchronize(s->ev_bits[c]));
            const auto t0 = clk::now();
            for (int v = 0; v < 2; ++v)
                if (dst[v] && hi[c] > mid[c])
                    inv_host::expand_f32(s->h_bits[v], static_cast<float *>(dst[v]), mid[c], hi[c], s->host_threads);
            expand_s += std::chrono::duration<double>(clk::now() - t0).count();
        }
    }
    CUDA_TRY(cudaStreamSynchronize(cs));
    scatter_small_outputs(s, so);
    if (expand) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, s->ev_t0, s->ev_t1);
        const double dma_s = ms * 1e-3;
        s->last_dma_s = dma_s;
        s->last_expand_s = expand_s;
        if (s->dma_frac_auto && expand_s > 0.0 && dma_s > 0.0) { // balance the two legs from their measured rates
            const double r_exp = (1.0 - frac) / expand_s;
            const double r_dma = frac > 0.0 ? frac / dma_s : r_exp * 0.5;
            double f = r_dma / (r_dma + r_exp);
            f = f < 0.0 ? 0.0 : (f > 0.9 ? 0.9 : f);
            s->dma_frac = 0.5 * s->dma_frac + 0.5 * f;
        }
    }
    return INV_OK;
}

// The trainer's view of a step (training.py:140-151): observations -- grid AND extra -- are consumed on
// the GPU; the host wants reward / done / info per env and the statistics of the episodes that just
// ended. Dense: 6 bytes per env. Sparse: one 24-byte record per finished episode, in env order,
// fetched together with its count (1.5 x the previous step's count travels with the header; a second
// copy follows only if more episodes ended than that).
static int ensure_event_buffers(inv_sim *s)
{
    if (s->d_events) return INV_OK;
    const size_t nblocks = ((size_t)s->n + kEvBlockEnvs - 1) / kEvBlockEnvs;
    const size_t ev_bytes = kEvHeaderBytes + (size_t)s->n * sizeof(inv_episode_event);
    CUDA_TRY(cudaMalloc((void **)&s->d_events, ev_bytes));
    CUDA_TRY(cudaMemsetAsync(s->d_events, 0, ev_bytes, s->host_stream)); // the prefix copy may read past the count
    CUDA_TRY(cudaMalloc((void **)&s->d_ev_counts, nblocks * sizeof(int32_t)));
    CUDA_TRY(cudaMallocHost((void **)&s->h_ev_count, sizeof(int64_t)));
    CUDA_TRY(cudaEventCreateWithFlags(&s->ev_events, cudaEventDisableTiming));
    s->ev_guess = 1024;
    return INV_OK;
}

int inv_step_host_events(inv_sim *s, const int8_t *a1, const int8_t *a2, float *reward, uint8_t *done,
                         uint8_t *info, inv_episode_event *events, int64_t capacity, int64_t *n_events)
{
    if (!s || !events || !n_events || capacity < 0)
        return fail(INV_ERR_INVALID_ARG, "inv_step_host_events: null handle, events or n_events, or negative capacity");
    DeviceGuard g(s->cfg.device);
    static const bool trace = getenv("INV_HOST_TRACE") != nullptr; // stderr: where a call's wall time goes
    const auto t_in = std::chrono::steady_clock::now();
    auto lap = [&](const char *what) {
        if (trace)
            fprintf(stderr, "[inv_step_host_events] %-22s %8.1f us\n", what,
                    std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t_in).count());
    };
    int rc = begin_host_step(s, a1, a2, "inv_step_host_events");
    if (rc != INV_OK) return rc;
    lap("ids checked + staged");
    if ((rc = ensure_event_buffers(s)) != INV_OK) return rc;
    const int64_t n = s->n;
    const bool selfplay = s->cfg.mode == INV_MODE_SELFPLAY;
    cudaStream_t ks = s->host_stream, cs = s->copy_stream;
    int64_t bounds[kMaxHostChunks + 1];
    const int nchunks = host_chunk_bounds(n, false, false, bounds);
    int used = 0;
    for (int c = 0; c < nchunks; ++c) {
        const int64_t first = bounds[c], count = bounds[c + 1] - first;
        if (first >= n || count <= 0) break;
        if ((rc = step_impl(s, s->d_a1, selfplay ? s->d_a2 : nullptr, ks, nullptr, nullptr, first, count)) != INV_OK) return rc;
        CUDA_TRY(cudaEventRecord(s->ev_kernel[c], ks));
        used = c + 1;
    }
    {   // the finished-episode list, once the whole done array is in place
        const unsigned nblocks = (unsigned)((n + kEvBlockEnvs - 1) / kEvBlockEnvs);
        int64_t *header = reinterpret_cast<int64_t *>(s->d_events);
        inv_episode_event *recs = reinterpret_cast<inv_episode_event *>(s->d_events + kEvHeaderBytes);
        episode_count_kernel<<<nblocks, kEvThreads, 0, ks>>>(s->done, n, s->d_ev_counts);
        episode_write_kernel<<<nblocks, kEvThreads, 0, ks>>>(s->done, s->info, s->ep_steps, s->ep_return, n,
                                                             s->d_ev_counts, header, recs);
        CUDA_TRY(cudaGetLastError());
        s->launches += 2;
        CUDA_TRY(cudaEventRecord(s->ev_events, ks));
    }
    for (int c = 0; c < used; ++c) { // dense outputs follow chunk by chunk on the copy stream
        const size_t f = (size_t)bounds[c], cnt = (size_t)(bounds[c + 1] - bounds[c]);
        CUDA_TRY(cudaStreamWaitEvent(cs, s->ev_kernel[c], 0));
        if (reward) CUDA_TRY(cudaMemcpyAsync(reward + f, s->reward + f, cnt * 4, cudaMemcpyDeviceToHost, cs));
        if (done) CUDA_TRY(cudaMemcpyAsync(done + f, s->done + f, cnt, cudaMemcpyDeviceToHost, cs));
        if (info) CUDA_TRY(cudaMemcpyAsync(info + f, s->info + f, cnt, cudaMemcpyDeviceToHost, cs));
    }
    const char *recs = s->d_events + kEvHeaderBytes;
    const int64_t guess = s->ev_guess < capacity ? s->ev_guess : capacity;
    CUDA_TRY(cudaStreamWaitEvent(cs, s->ev_events, 0));
    CUDA_TRY(cudaMemcpyAsync(s->h_ev_count, s->d_events, sizeof(int64_t), cudaMemcpyDeviceToHost, cs));
    if (guess > 0)
        CUDA_TRY(cudaMemcpyAsync(events, recs, (size_t)guess * sizeof(inv_episode_event), cudaMemcpyDeviceToHost, cs));
    lap("all work enqueued");
    if (trace) {
        for (int c = 0; c < used; ++c) {
            cudaEventSynchronize(s->ev_kernel[c]);
            lap("a chunk's kernel done");
        }
        cudaEventSynchronize(s->ev_events);
        lap("event list built");
    }
    CUDA_TRY(cudaStreamSynchronize(cs));
    lap("copies landed");
    const int64_t count = *s->h_ev_count;
    *n_events = count;
    s->ev_guess = count + count / 4 < 1024 ? 1024 : count + count / 4;
    if (count > capacity)
        return fail(INV_ERR_INVALID_ARG, "inv_step_host_events: more episodes ended than the events buffer holds "
                                         "(the step has been taken; capacity >= num_envs never overflows)");
    if (count > guess) {
        CUDA_TRY(cudaMemcpyAsync(events + guess, recs + (size_t)guess * sizeof(inv_episode_event),
                                 (size_t)(count - guess) * sizeof(inv_episode_event), cudaMemcpyDeviceToHost, cs));
        CUDA_TRY(cudaStreamSynchronize(cs));
    }
    return INV_OK;
}

int inv_set_host_path(inv_sim *s, int nthreads, double dma_fraction)
{
    if (!s || nthreads < 0 || nthreads > 256 || dma_fraction > 1.0) return fail(INV_ERR_INVALID_ARG, "inv_set_host_path: bad argument");
    s->host_threads = nthreads;
    if (dma_fraction < 0.0) { s->dma_frac_auto = true; }
    else { s->dma_frac_auto = false; s->dma_frac = dma_fraction; }
    return INV_OK;
}

int inv_get_host_path(const inv_sim *s, int *nthreads, double *dma_fraction, double *last_dma_s, double *last_expand_s)
{
    if (!s) return fail(INV_ERR_INVALID_ARG, "inv_get_host_path: null handle");
    if (nthreads) *nthreads = s->host_threads;
    if (dma_fraction) *dma_fraction = s->dma_frac;
    if (last_dma_s) *last_dma_s = s->last_dma_s;
    if (last_expand_s) *last_expand_s = s->last_expand_s;
    return INV_OK;
}

int inv_reset_host(inv_sim *s, void *obs_p1, float *extra_p1, void *obs_p2, float *extra_p2)
{
    if (!s) return fail(INV_ERR_INVALID_ARG, "inv_reset_host: null handle");
    if (obs_p1 && !s->obs1) return fail(INV_ERR_INVALID_ARG, "this handle keeps no observation tensor (INV_OBS_NONE)");
    if (obs_p2 && !s->obs2) return fail(INV_ERR_INVALID_ARG, "P2 view was not enabled (INV_FLAG_P2_VIEW)");
    if (extra_p2 && !s->extra2) return fail(INV_ERR_INVALID_ARG, "P2 view was not enabled (INV_FLAG_P2_VIEW)");
    DeviceGuard g(s->cfg.device);
    int rc = ensure_host_staging(s);
    if (rc != INV_OK) return rc;
    cudaStream_t st = s->host_stream;
    if ((rc = order_host_stream(s)) != INV_OK) return rc;
    if ((rc = inv_reset(s, st)) != INV_OK) return rc;
    const SmallOut so = {extra_p1, extra_p2, nullptr, nullptr, nullptr, nullptr, nullptr};
    if ((rc = copy_small_outputs(s, st, so, 0, s->n)) != INV_OK) return rc;
    const size_t ob = (size_t)s->n * INV_OBS_ELEMS * obs_elem_bytes(s->cfg.obs_dtype);
    if (obs_p1) CUDA_TRY(cudaMemcpyAsync(obs_p1, s->obs1, ob, cudaMemcpyDeviceToHost, st));
    if (obs_p2) CUDA_TRY(cudaMemcpyAsync(obs_p2, s->obs2, ob, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    scatter_small_outputs(s, so);
    return INV_OK;
}

int inv_host_alloc(void **out, int64_t nbytes)
{
    if (!out || nbytes <= 0) return fail(INV_ERR_INVALID_ARG, "inv_host_alloc: bad argument");
    CUDA_TRY(cudaMallocHost(out, (size_t)nbytes));
    return INV_OK;
}

int inv_host_free(void *p)
{
    if (p) CUDA_TRY(cudaFreeHost(p));
    return INV_OK;
}

int inv_get_buffer(inv_sim *s, int which, void **dev_ptr, int64_t *nbytes)
{
    if (!s || !dev_ptr) return fail(INV_ERR_INVALID_ARG, "inv_get_buffer: null argument");
    const int64_t n = s->n;
    const int64_t ob = n * INV_OBS_ELEMS * (int64_t)obs_elem_bytes(s->cfg.obs_dtype);
    void *p = nullptr;
    int64_t b = 0;
    switch (which) {
    case INV_BUF_OBS_P1: p = s->obs1; b = ob; break;
    case INV_BUF_EXTRA_P1: p = s->extra1; b = n * 16; break;
    case INV_BUF_OBS_P2: p = s->obs2; b = s->obs2 ? ob : 0; break;
    case INV_BUF_EXTRA_P2: p = s->extra2; b = s->extra2 ? n * 16 : 0; break;
    case INV_BUF_REWARD: p = s->reward; b = n * 4; break;
    case INV_BUF_DONE: p = s->done; b = n; break;
    case INV_BUF_INFO: p = s->info; b = n; break;
    case INV_BUF_EPISODE_STEPS: p = s->ep_steps; b = n * 4; break;
    case INV_BUF_EPISODE_RETURN: p = s->ep_return; b = n * 8; break;
    case INV_BUF_PACKED_STATE: p = s->state; b = n * INV_PACKED_STATE_BYTES; break;
    case INV_BUF_DEBUG_RESULT: p = s->dbg; b = n; break;
    case INV_BUF_REWARD_F64: p = s->reward64; b = s->reward64 ? n * 8 : 0; break;
    default: return fail(INV_ERR_INVALID_ARG, "inv_get_buffer: unknown buffer id");
    }
    if (!p) return fail(INV_ERR_INVALID_ARG, "inv_get_buffer: buffer not allocated for this configuration");
    *dev_ptr = p;
    if (nbytes) *nbytes = b;
    return INV_OK;
}

int inv_set_draw_table(inv_sim *s, const uint32_t *table_dev)
{
    if (!s) return fail(INV_ERR_INVALID_ARG, "inv_set_draw_table: null handle");
    s->table = table_dev;
    return INV_OK;
}

int inv_export_state(inv_sim *s, inv_env_state *out, int64_t first, int64_t count)
{
    if (!s || !out) return fail(INV_ERR_INVALID_ARG, "inv_export_state: null argument");
    if (first < 0 || count < 0 || first + count > s->n) return fail(INV_ERR_INVALID_ARG, "inv_export_state: bad range");
    if (count == 0) return INV_OK;
    DeviceGuard g(s->cfg.device);
    CUDA_TRY(cudaDeviceSynchronize());
    std::vector<uint4> buf((size_t)count * 5); // [5][count]: a plane set with stride count
    for (int k = 0; k < 5; ++k)
        CUDA_TRY(cudaMemcpy(buf.data() + (size_t)k * count, s->state + (size_t)k * s->n + first, (size_t)count * 16,
                            cudaMemcpyDeviceToHost));
    for (int64_t i = 0; i < count; ++i) {
        Env e;
        uint16_t sb[kSlots];
        load_env<1>(e, sb, buf.data(), count, i);
        env_to_canonical(e, sb, out[i]);
    }
    return INV_OK;
}

int inv_import_state(inv_sim *s, const inv_env_state *in, int64_t first, int64_t count)
{
    if (!s || !in) return fail(INV_ERR_INVALID_ARG, "inv_import_state: null argument");
    if (first < 0 || count < 0 || first + count > s->n) return fail(INV_ERR_INVALID_ARG, "inv_import_state: bad range");
    if (count == 0) return INV_OK;
    DeviceGuard g(s->cfg.device);
    std::vector<uint4> buf((size_t)count * 5); // [5][count]: a plane set with stride count
    for (int64_t i = 0; i < count; ++i) {
        Env e;
        uint16_t sb[kSlots];
        if (!env_from_canonical(in[i], e, sb)) return fail(INV_ERR_INVALID_ARG, "inv_import_state: field out of range");
        store_env<1>(e, sb, buf.data(), count, i);
    }
    CUDA_TRY(cudaDeviceSynchronize());
    for (int k = 0; k < 5; ++k)
        CUDA_TRY(cudaMemcpy(s->state + (size_t)k * s->n + first, buf.data() + (size_t)k * count, (size_t)count * 16,
                            cudaMemcpyHostToDevice));
    s->was_reset = true;
    return INV_OK;
}

int inv_load_packed_state(inv_sim *s, const void *packed_dev, void *stream)
{
    if (!s || !packed_dev) return fail(INV_ERR_INVALID_ARG, "inv_load_packed_state: null argument");
    DeviceGuard g(s->cfg.device);
    CUDA_TRY(cudaMemcpyAsync(s->state, packed_dev, (size_t)s->n * INV_PACKED_STATE_BYTES, cudaMemcpyDeviceToDevice,
                             (cudaStream_t)stream));
    s->was_reset = true;
    return INV_OK;
}

int inv_obs_from_packed(inv_sim *s, const void *packed_dev, int64_t stride, int64_t count, int view, int obs_dtype,
                        void *obs_out, float *extra_out, void *stream)
{
    if (!s || !packed_dev || !obs_out || !extra_out) return fail(INV_ERR_INVALID_ARG, "inv_obs_from_packed: null argument");
    if (count < 0 || stride < count || (view != 0 && view != 1)) return fail(INV_ERR_INVALID_ARG, "inv_obs_from_packed: bad argument");
    if (count == 0) return INV_OK;
    DeviceGuard g(s->cfg.device);
    Params p = base_params(s);
    p.state_in = static_cast<const uint4 *>(packed_dev);
    p.stride = stride;
    p.count = count;
    p.view = view;
    p.obs1 = obs_out;
    p.extra1 = extra_out;
    p.table = nullptr;
    cudaError_t ce;
    switch (obs_dtype) {
    case INV_OBS_F32: ce = launch_e<OP_OBS, INV_OBS_F32, false, false>(p, s->sm_count, (cudaStream_t)stream); break;
    case INV_OBS_BF16: ce = launch_e<OP_OBS, INV_OBS_BF16, false, false>(p, s->sm_count, (cudaStream_t)stream); break;
    case INV_OBS_U8: ce = launch_e<OP_OBS, INV_OBS_U8, false, false>(p, s->sm_count, (cudaStream_t)stream); break;
    default: return fail(INV_ERR_INVALID_ARG, "inv_obs_from_packed: unknown obs_dtype");
    }
    CUDA_TRY(ce);
    note_launch(s, (cudaStream_t)stream);
    return INV_OK;
}

int inv_debug_phase(inv_sim *s, int phase, int pid, int arg, int arg2, void *stream)
{
    if (!s) return fail(INV_ERR_INVALID_ARG, "inv_debug_phase: null handle");
    if (phase < 0 || phase > INV_PHASE_DUMMY_POLICY || (pid != 0 && pid != 1))
        return fail(INV_ERR_INVALID_ARG, "inv_debug_phase: bad phase or pid");
    if ((phase <= INV_PHASE_WIDE_SHOT) && (arg < 0 || arg > 3)) return fail(INV_ERR_INVALID_ARG, "inv_debug_phase: bad direction");
    if (phase == INV_PHASE_STEP_PLAYERS && (arg < 0 || arg > 12 || arg2 < 0 || arg2 > 12))
        return fail(INV_ERR_INVALID_ACTION, "Invalid action_id: must be 0-12");
    DeviceGuard g(s->cfg.device);
    Params p = base_params(s);
    p.phase = phase; p.pid = pid; p.arg = arg; p.arg2 = arg2;
    CUDA_TRY((launch_one<OP_DEBUG, INV_OBS_F32, false, false, 32>(p, s->sm_count, (cudaStream_t)stream)));
    note_launch(s, (cudaStream_t)stream);
    return INV_OK;
}

int inv_poll_status(inv_sim *s, void *stream, uint32_t *bits)
{
    if (!s || !bits) return fail(INV_ERR_INVALID_ARG, "inv_poll_status: null argument");
    DeviceGuard g(s->cfg.device);
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemcpyAsync(s->h_status, s->status, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemsetAsync(s->status, 0, 4, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    *bits = *s->h_status;
    return INV_OK;
}

int64_t inv_launch_count(const inv_sim *s) { return s ? s->launches : 0; }

int inv_gae(const float *reward_dev, const float *value_dev, const uint8_t *done_dev, const float *last_value_dev,
            double gamma, double lam, int32_t T, int64_t N, float *adv_dev, float *ret_dev, void *stream)
{
    if (!reward_dev || !value_dev || !done_dev || !adv_dev || !ret_dev || T < 0 || N < 0)
        return fail(INV_ERR_INVALID_ARG, "inv_gae: bad argument");
    if (T == 0 || N == 0) return INV_OK;
    const int threads = 128;
    gae_kernel<<<(unsigned)((N + threads - 1) / threads), threads, 0, (cudaStream_t)stream>>>(
        reward_dev, value_dev, done_dev, last_value_dev, (float)gamma, (float)(gamma * lam), T, N, adv_dev, ret_dev);
    CUDA_TRY(cudaGetLastError());
    return INV_OK;
}

} // extern "C"
