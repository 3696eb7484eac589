// eval_kernels.cu -- the two device steps of the evaluator (inversus_b200/evaluate.py) that the
// policy and the simulator do not already provide:
//
//   inv_select_actions  logits -> int8 action ids, greedy (first maximum) or sampled with one
//                       Philox4x32-10 draw per row whose counter is the env's global id and its
//                       (episode, step_count) words, so a draw is a pure function of the seed and
//                       the simulator state (DESIGN.md "evaluator").
//   inv_episode_tally   per-env wins / losses / draws / length sum / return sum of exactly the
//                       first `quota` episodes of every env, plus the number of envs still short
//                       of their quota.
//   inv_scripted_actions the scripted dummy as a player of either seat: one int8 action id per
//                       env, drawn from counters that are a pure function of the simulator state.
//
// They read the packed state through its codec (load_counters, load_board). Every value has one
// owner thread; the only atomic adds an integer count into `remaining`, whose sum does not depend
// on the order of the additions.
#include "inversus_kernels.cuh"
#include "launch_common.h"

using namespace inv;

namespace {

constexpr int kA = INV_NUM_ACTIONS;
constexpr int kSelThreads = 256;
constexpr int kTallyThreads = 256;
constexpr int kScriptThreads = 256;

// One thread per row. The block's rows are staged through shared memory so that the global reads
// are coalesced; a row's 13 floats then sit at an odd word stride, which is bank-conflict free.
__global__ void __launch_bounds__(kSelThreads)
select_actions_kernel(const float *__restrict__ logits, int64_t count, const uint4 *__restrict__ packed, int64_t stride,
                      uint32_t gid_base, uint32_t seed_lo, uint32_t seed_hi, uint32_t seat, int greedy,
                      int8_t *__restrict__ out)
{
    __shared__ float sl[kSelThreads * kA];
    const int64_t base = (int64_t)blockIdx.x * kSelThreads;
    const int rows = (int)min((int64_t)kSelThreads, count - base);
    const float *src = logits + base * kA;
    for (int k = threadIdx.x; k < rows * kA; k += kSelThreads) sl[k] = src[k];
    __syncthreads();
    if ((int)threadIdx.x >= rows) return;
    const int64_t i = base + threadIdx.x;
    const float *l = sl + threadIdx.x * kA;

    float m = l[0];
    int arg = 0;
    bool bad = false;
#pragma unroll
    for (int j = 0; j < kA; ++j) {
        const float v = l[j];
        bad = bad || isnan(v) || v == INFINITY;
        if (v > m) { m = v; arg = j; } // strict: the first maximum, like torch.argmax
    }
    bad = bad || m == -INFINITY;       // every logit -inf
    int a = arg;
    if (bad) {
        a = -1; // inv_step raises INV_STATUS_INVALID_ACTION
    } else if (!greedy) {
        const Counters c = load_counters(packed, stride, i);
        uint32_t r[4];
        philox4x32_10(gid_base + (uint32_t)i, c.episode, c.step, 0x80000000u | seat, seed_lo, seed_hi, r);
        float e[kA];
        float S = 0.0f;
#pragma unroll
        for (int j = 0; j < kA; ++j) {
            e[j] = expf(__fsub_rn(l[j], m));
            S = __fadd_rn(S, e[j]);
        }
        const float t = __fmul_rn(__fmul_rn(__uint2float_rn(r[0]), 0x1p-32f), S);
        float cum = 0.0f;
        int last = 0;
        a = -1;
#pragma unroll
        for (int j = 0; j < kA; ++j) {
            cum = __fadd_rn(cum, e[j]);
            if (e[j] > 0.0f) last = j;
            if (a < 0 && t < cum) a = j;
        }
        if (a < 0) a = last; // rounding put t at or past the total
    }
    out[i] = (int8_t)a;
}

__global__ void __launch_bounds__(kTallyThreads)
episode_tally_kernel(const uint8_t *__restrict__ done, const uint8_t *__restrict__ info,
                     const int32_t *__restrict__ ep_steps, const double *__restrict__ ep_return,
                     const uint4 *__restrict__ packed, int64_t stride, int64_t count, uint32_t quota,
                     int32_t *__restrict__ counts, double *__restrict__ return_sum, int32_t *__restrict__ remaining)
{
    const int64_t i = (int64_t)blockIdx.x * kTallyThreads + threadIdx.x;
    int short_of_quota = 0;
    if (i < count) {
        // post-step counter: an auto-reset has already advanced it past the episode that ended
        const uint32_t episode = load_counters(packed, stride, i).episode;
        short_of_quota = episode < quota;
        if (done[i] && episode - 1u < quota) {
            const uint32_t f = info[i];
            const int win = (f & INV_INFO_WIN) != 0, lose = (f & INV_INFO_LOSE) != 0;
            counts[i] += win;
            counts[count + i] += lose;
            counts[2 * count + i] += !win && !lose;
            counts[3 * count + i] += ep_steps[i];
            return_sum[i] = __dadd_rn(return_sum[i], ep_return[i]);
        }
    }
    const int n = __syncthreads_count(short_of_quota);
    if (threadIdx.x == 0 && n) atomicAdd(remaining, n);
}

// One thread per env: planes 0-2 in (48 B), one action id out.
__global__ void __launch_bounds__(kScriptThreads)
scripted_actions_kernel(const uint4 *__restrict__ packed, int64_t stride, int64_t count, uint32_t gid_base,
                        uint32_t seed_lo, uint32_t seed_hi, int seat, int difficulty, int8_t *__restrict__ out)
{
    const int64_t i = (int64_t)blockIdx.x * kScriptThreads + threadIdx.x;
    if (i >= count) return;
    Env s;
    load_board(s, packed, stride, i);
    Params p; // Draws reads only the key from it
    p.seed_lo = seed_lo;
    p.seed_hi = seed_hi;
    out[i] = (int8_t)scripted_action(s, p, gid_base + (uint32_t)i, seat, difficulty);
}

} // namespace

extern "C" {

int inv_select_actions(const float *logits, int64_t count, const void *packed_dev, int64_t stride, int64_t gid_base,
                       uint64_t seed, int seat, int greedy, int8_t *actions_out, void *stream)
{
    const char *who = "inv_select_actions";
    if (int rc = inv_host::require_sm100(who)) return rc;
    if (count < 0 || !logits || !actions_out || (!greedy && (!packed_dev || stride < count)) || (seat != 0 && seat != 1) ||
        gid_base < 0 || gid_base > 0x100000000ll - count)
        return inv_host::set_error(INV_ERR_INVALID_ARG, who, "bad argument");
    if (count == 0) return INV_OK;
    const int64_t blocks = (count + kSelThreads - 1) / kSelThreads;
    select_actions_kernel<<<(unsigned)blocks, kSelThreads, 0, (cudaStream_t)stream>>>(
        logits, count, static_cast<const uint4 *>(packed_dev), stride, (uint32_t)gid_base, (uint32_t)seed,
        (uint32_t)(seed >> 32), (uint32_t)seat, greedy, actions_out);
    return inv_host::launch_status(who);
}

int inv_episode_tally(const uint8_t *done, const uint8_t *info, const int32_t *episode_steps,
                      const double *episode_return, const void *packed_dev, int64_t stride, int64_t count, int64_t quota,
                      int32_t max_episode_steps, int32_t *counts_dev, double *return_sum_dev, int32_t *remaining_dev,
                      void *stream)
{
    const char *who = "inv_episode_tally";
    if (int rc = inv_host::require_sm100(who)) return rc;
    if (count < 0 || !done || !info || !episode_steps || !episode_return || !packed_dev || stride < count || !counts_dev ||
        !return_sum_dev || !remaining_dev || max_episode_steps <= 0)
        return inv_host::set_error(INV_ERR_INVALID_ARG, who, "bad argument");
    if (quota < 1 || quota >= (1ll << 31) || quota * (int64_t)max_episode_steps >= (1ll << 31))
        return inv_host::set_error(INV_ERR_INVALID_ARG, who,
                                   "quota * max_episode_steps must be below 2^31 (the per-env length sum is int32)");
    cudaStream_t st = (cudaStream_t)stream;
    if (cudaMemsetAsync(remaining_dev, 0, sizeof(int32_t), st) != cudaSuccess) return inv_host::launch_status(who);
    if (count == 0) return INV_OK;
    const int64_t blocks = (count + kTallyThreads - 1) / kTallyThreads;
    episode_tally_kernel<<<(unsigned)blocks, kTallyThreads, 0, st>>>(
        done, info, episode_steps, episode_return, static_cast<const uint4 *>(packed_dev), stride, count,
        (uint32_t)quota, counts_dev, return_sum_dev, remaining_dev);
    return inv_host::launch_status(who);
}

int inv_scripted_actions(const void *packed_dev, int64_t stride, int64_t count, int64_t gid_base, uint64_t seed,
                         int seat, int difficulty, int8_t *actions_out, void *stream)
{
    const char *who = "inv_scripted_actions";
    if (int rc = inv_host::require_sm100(who)) return rc;
    if (count < 0 || !packed_dev || !actions_out || stride < count || (seat != 0 && seat != 1) ||
        (difficulty != 0 && difficulty != 1) || gid_base < 0 || gid_base > 0x100000000ll - count)
        return inv_host::set_error(INV_ERR_INVALID_ARG, who, "bad argument");
    if (count == 0) return INV_OK;
    const int64_t blocks = (count + kScriptThreads - 1) / kScriptThreads;
    scripted_actions_kernel<<<(unsigned)blocks, kScriptThreads, 0, (cudaStream_t)stream>>>(
        static_cast<const uint4 *>(packed_dev), stride, count, (uint32_t)gid_base, (uint32_t)seed,
        (uint32_t)(seed >> 32), seat, difficulty, actions_out);
    return inv_host::launch_status(who);
}

} // extern "C"
