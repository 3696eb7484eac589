// harness.cpp -- TEST INFRASTRUCTURE. Drives the product's own device functions (load_env,
// rl_step, rl_reset, debug_phase, build_row, extra_vec, store_env of csrc/inversus_kernels.cuh) and
// its canonical-state conversions, compiled for the host through host_shim.h, over the same
// packed-state planes the GPU uses. One "thread" per env, tile size E = 1. See
// tests/test_host_kernel.py.
#define INV_HOST_BUILD 1
#include "../../inversus-reinforcement-learning_b200/csrc/inversus_kernels.cuh"

using namespace inv;

namespace {

void emit(const Env &s, const uint16_t *sb, int64_t i, float *obs1, float *extra1, float *obs2, float *extra2)
{
    uint32_t row[kRowWords];
    float *obs[2] = {obs1, obs2};
    float *extra[2] = {extra1, extra2};
    for (int v = 0; v < 2; ++v) {
        if (!obs[v]) continue;
        if (v == 0) build_row<1>(row, s, sb, 0);
        else build_row<1>(row, s, sb, 1);
        float *o = obs[v] + i * INV_OBS_ELEMS;
        for (int k = 0; k < INV_OBS_ELEMS; ++k) o[k] = ((row[k >> 5] >> (k & 31)) & 1u) ? 1.0f : 0.0f;
        const float4 x = v == 0 ? extra_vec(s, 0) : extra_vec(s, 1);
        float *e = extra[v] + i * 4;
        e[0] = x.x; e[1] = x.y; e[2] = x.z; e[3] = x.w;
    }
}

Params make_params(int mode, int difficulty, int max_steps, int auto_reset, uint64_t seed, uint32_t env_id_base,
                   const uint32_t *table, uint32_t *status)
{
    Params p;
    memset(&p, 0, sizeof(p));
    p.mode = mode; p.difficulty = difficulty; p.max_steps = max_steps; p.auto_reset = auto_reset;
    p.seed_lo = (uint32_t)seed; p.seed_hi = (uint32_t)(seed >> 32); p.env_id_base = env_id_base;
    p.table = table; p.status = status;
    return p;
}

} // namespace

extern "C" {

// planes: [5][n] uint4, exactly INV_BUF_PACKED_STATE
int hk_reset(uint32_t *planes, int64_t n, const int64_t *idx, int64_t count, uint64_t seed, uint32_t env_id_base,
             const uint32_t *table, float *obs1, float *extra1, float *obs2, float *extra2, uint32_t *status)
{
    uint4 *st = reinterpret_cast<uint4 *>(planes);
    Params p = make_params(0, 0, 0, 0, seed, env_id_base, table, status);
    const int64_t m = idx ? count : n;
    for (int64_t k = 0; k < m; ++k) {
        const int64_t i = idx ? idx[k] : k;
        Env s;
        uint16_t sb[kSlots] = {0};
        load_env<1>(s, sb, st, n, i);
        rl_reset(s, p, env_id_base + (uint32_t)i, table ? table + i * INV_TABLE_STRIDE : nullptr);
        store_env<1>(s, sb, st, n, i);
        emit(s, sb, i, obs1, extra1, obs2, extra2);
    }
    return 0;
}

int hk_step(uint32_t *planes, int64_t n, const int8_t *a1, const int8_t *a2, const uint32_t *table, int mode,
            int difficulty, int max_steps, int auto_reset, uint64_t seed, uint32_t env_id_base, float *obs1,
            float *extra1, float *obs2, float *extra2, float *reward, uint8_t *done, uint8_t *info,
            int32_t *ep_steps, double *ep_return, uint32_t *status)
{
    uint4 *st = reinterpret_cast<uint4 *>(planes);
    Params p = make_params(mode, difficulty, max_steps, auto_reset, seed, env_id_base, table, status);
    for (int64_t i = 0; i < n; ++i) {
        Env s;
        uint16_t sb[kSlots] = {0};
        load_env<1>(s, sb, st, n, i);
        const StepResult o = rl_step<1>(s, sb, a1[i], a2 ? a2[i] : 0, p, env_id_base + (uint32_t)i,
                                        table ? table + i * INV_TABLE_STRIDE : nullptr);
        reward[i] = o.reward; done[i] = o.done; info[i] = o.info; ep_steps[i] = o.ep_steps; ep_return[i] = o.ep_return;
        store_env<1>(s, sb, st, n, i);
        emit(s, sb, i, obs1, extra1, obs2, extra2);
    }
    return 0;
}

// One engine method of core.py on env 0..n-1, like inv_debug_phase (same dispatch, same device
// functions); result[i] = the method's return value.
int hk_debug(uint32_t *planes, int64_t n, int phase, int pid, int arg, int arg2, int difficulty, uint64_t seed,
             uint32_t env_id_base, uint8_t *result, uint32_t *status)
{
    if (phase < 0 || phase > INV_PHASE_DUMMY_POLICY) return -1;
    uint4 *st = reinterpret_cast<uint4 *>(planes);
    Params p = make_params(1, difficulty, 500, 0, seed, env_id_base, nullptr, status);
    p.phase = phase; p.pid = pid; p.arg = arg; p.arg2 = arg2;
    for (int64_t i = 0; i < n; ++i) {
        Env s;
        uint16_t sb[kSlots] = {0};
        load_env<1>(s, sb, st, n, i);
        result[i] = debug_phase<1>(s, sb, p, env_id_base + (uint32_t)i, nullptr);
        store_env<1>(s, sb, st, n, i);
    }
    return 0;
}

// Canonical state of envs [first, first+count) out of / into the planes, like inv_export_state /
// inv_import_state (same conversions). The import writes nothing unless every env is in range.
int hk_export_state(const uint32_t *planes, int64_t n, int64_t first, int64_t count, inv_env_state *out)
{
    for (int64_t k = 0; k < count; ++k) {
        Env s;
        uint16_t sb[kSlots];
        load_env<1>(s, sb, reinterpret_cast<const uint4 *>(planes), n, first + k);
        env_to_canonical(s, sb, out[k]);
    }
    return 0;
}

int hk_import_state(uint32_t *planes, int64_t n, int64_t first, int64_t count, const inv_env_state *in)
{
    Env s;
    uint16_t sb[kSlots];
    for (int64_t k = 0; k < count; ++k)
        if (!env_from_canonical(in[k], s, sb)) return -1;
    for (int64_t k = 0; k < count; ++k) {
        env_from_canonical(in[k], s, sb);
        store_env<1>(s, sb, reinterpret_cast<uint4 *>(planes), n, first + k);
    }
    return 0;
}

int hk_observation(const uint32_t *planes, int64_t n, int64_t i, int viewer, float *obs, float *extra)
{
    Env s;
    uint16_t sb[kSlots] = {0};
    load_env<1>(s, sb, reinterpret_cast<const uint4 *>(planes), n, i);
    if (viewer == 0) emit(s, sb, 0, obs, extra, nullptr, nullptr);
    else emit(s, sb, 0, nullptr, nullptr, obs, extra);
    return 0;
}

} // extern "C"

#ifdef HK_STANDALONE
// Sanitizer target: a self-contained random rollout (no reference involved), built with
// -fsanitize=address,undefined, exercising every branch family (both modes and difficulties,
// charge-heavy actions, auto-reset, timeouts) so that out-of-bounds indexing or UB in the shared
// game logic aborts the test. Every 20 steps all envs go through export and re-import, which must
// leave the planes byte-identical.
#include <cstdio>
#include <vector>
int main()
{
    const int64_t n = 257;
    uint64_t rng = 88172645463325252ull;
    auto next = [&]() { rng ^= rng << 13; rng ^= rng >> 7; rng ^= rng << 17; return (uint32_t)(rng >> 11); };
    long episodes = 0;
    for (int mode = 0; mode < 2; ++mode)
        for (int diff = 0; diff < 2; ++diff) {
            std::vector<uint32_t> planes((size_t)n * 20, 0u);
            std::vector<inv_env_state> states(n);
            for (auto &e : states) e.episode = 0xFFFFFFFFu; // no episode yet
            hk_import_state(planes.data(), n, 0, n, states.data());
            std::vector<float> obs1((size_t)n * INV_OBS_ELEMS), ex1((size_t)n * 4), obs2((size_t)n * INV_OBS_ELEMS), ex2((size_t)n * 4);
            std::vector<float> rew(n);
            std::vector<uint8_t> done(n), info(n);
            std::vector<int32_t> steps(n);
            std::vector<double> ret(n);
            std::vector<int8_t> a1(n), a2(n);
            std::vector<uint32_t> table((size_t)n * INV_TABLE_STRIDE);
            uint32_t status = 0;
            hk_reset(planes.data(), n, nullptr, 0, 7, 1000, nullptr, obs1.data(), ex1.data(), obs2.data(), ex2.data(), &status);
            for (int t = 0; t < 400; ++t) {
                const bool use_table = (t % 3) == 0;
                for (auto &v : table) v = (next() & 3) ? next() : next() >> 12;
                for (int64_t i = 0; i < n; ++i) {
                    a1[i] = (int8_t)((next() & 1) ? 5 + next() % 8 : next() % 13);
                    a2[i] = (int8_t)(next() % 13);
                }
                hk_step(planes.data(), n, a1.data(), a2.data(), use_table ? table.data() : nullptr, mode, diff, 37,
                        (t / 50) % 2, 7, 1000, obs1.data(), ex1.data(), obs2.data(), ex2.data(), rew.data(),
                        done.data(), info.data(), steps.data(), ret.data(), &status);
                for (int64_t i = 0; i < n; ++i) episodes += done[i];
                if (t % 20 == 19) {
                    const std::vector<uint32_t> before = planes;
                    hk_export_state(planes.data(), n, 0, n, states.data());
                    if (hk_import_state(planes.data(), n, 0, n, states.data()) != 0 || planes != before) {
                        std::printf("export/import round trip changed the planes at step %d\n", t);
                        return 1;
                    }
                }
                if (t % 50 == 49) { // manual resets of a scattered index list
                    std::vector<int64_t> idx;
                    for (int64_t i = 0; i < n; i += 3) idx.push_back(i);
                    hk_reset(planes.data(), n, idx.data(), (int64_t)idx.size(), 7, 1000, use_table ? table.data() : nullptr,
                             obs1.data(), ex1.data(), obs2.data(), ex2.data(), &status);
                }
            }
            if (status != 0) { std::printf("unexpected status %u\n", status); return 1; }
        }
    std::printf("host kernel sanitizer run ok: %ld episode ends\n", episodes);
    return 0;
}
#endif
