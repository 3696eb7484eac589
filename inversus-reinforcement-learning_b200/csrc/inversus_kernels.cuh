// inversus_kernels.cuh -- sm_100a device code of the batched INVERSUS simulator.
//
// One kernel template serves every operation of the rollout hot path (SURVEY.md section 8a):
//   OP_STEP       K1  fused step: scripted opponent (D1) + engine tick (S1-S7) + reward/done (W2)
//                     + trainer auto-reset (X1/R1) + observation write-out (O1)
//   OP_RESET      K2  reset of all envs / of an index list (R1, W1, MultiEnvRunner.reset)
//   OP_OBS        K3  observation rebuild from packed-state snapshots (O1)
//   OP_DEBUG          one engine method at a time (parity tests restating the reference's tests)
//
// Execution shape (DESIGN.md "kernel"): a 128-thread CTA owns a tile of E consecutive envs and the
// grid is one CTA per tile (E = 32 for fp32 observations: one logic warp, four store warps; 64/128
// for the narrower step variants -- see launch_e in inversus_b200.cu).
//   phase 1  thread-per-env: load the 80-byte packed state (5 coalesced 16 B plane loads), run the
//            integer game logic in registers (+ a private bullet column in shared memory), store
//            the state back, and leave each env's observation as an 1800-BIT string in shared
//            memory (12 planes x 150 tiles, exactly the reference's C-order element order).
//   phase 2  all threads: stream the tile's observations out as consecutive 16-byte stores --
//            each lane expands 4 (f32) or 8 (bf16/u8) bits of the shared string per store, so a
//            warp instruction writes 512 contiguous bytes. 97 % of the kernel's HBM traffic is
//            this store stream; the kernel is HBM-write bound by construction.
//
// Reference behaviour is cited as file:line of Jason-Hoford/inversus-reinforcement-learning.
#pragma once

#ifdef INV_HOST_BUILD
#include "host_shim.h" // tests/host_kernel: compiles the game logic below for the CPU (test harness only)
#else
#include <cuda_runtime.h>
#endif
#include <stdint.h>
#include <string.h>

#include "../../include/inversus_b200.h"

// The packed-state codec (Env, pack_*/unpack_*, load_env, store_env) is shared by the kernels and
// the host side of inv_export_state / inv_import_state.
#define INV_HD __host__ __device__ __forceinline__

namespace inv {

constexpr int kW = INV_BOARD_W;                 // config.py:7
constexpr int kH = INV_BOARD_H;                 // config.py:8
constexpr int kTiles = kW * kH;                 // 150
constexpr int kMaxAmmo = 6;                     // config.py:14
constexpr int kReloadTicks = 30;                // config.py:15
constexpr int kWideCost = 3;                    // config.py:16
constexpr int kSlots = INV_MAX_BULLETS;         // 16 ordered bullet slots (<= 14 live, SURVEY.md 7.1)
constexpr int kRowWords = 57;                   // ceil(1800 / 32); odd => conflict-free per-thread rows
constexpr int kThreads = 128;

// integer forms of the scripted opponent's float comparisons (env_wrappers.py:82-89,96,105,123);
// u = r / 2^32, so (u < p) <=> (r < ceil(p * 2^32)). Checked in tests/test_rng_spec.py.
constexpr uint32_t kThreshShootHard = 858993460u;    // u < 0.2
constexpr uint32_t kThreshRandMoveHard = 214748365u; // u < 0.05
constexpr uint32_t kThreshMoveEasy = 4294968u;       // !(u > 0.001)

enum : int { OP_STEP = 0, OP_RESET = 1, OP_OBS = 2, OP_DEBUG = 3 };

// Exact binary64 values of the proximity term 0.002 * (1.0 - dist / 25) (env_wrappers.py:378-382)
// for dist = 0..23, and exact binary32 values of (float)(ammo / 6) (env_wrappers.py:238-240):
// computed with the reference's own arithmetic (Python floats / numpy.float32) and written as hex
// literals, so the kernel needs no fp64 division. tests/test_rng_spec.py re-derives both tables.
__constant__ double kProximity[24] = {
    0x1.0624dd2f1a9fcp-9,  0x1.f75104d551d69p-10, 0x1.e2584f4c6e6dap-10, 0x1.cd5f99c38b04bp-10,
    0x1.b866e43aa79bcp-10, 0x1.a36e2eb1c432dp-10, 0x1.8e757928e0c9ep-10, 0x1.797cc39ffd60ep-10,
    0x1.64840e1719f7fp-10, 0x1.4f8b588e368f1p-10, 0x1.3a92a30553261p-10, 0x1.2599ed7c6fbd3p-10,
    0x1.10a137f38c544p-10, 0x1.f75104d551d69p-11, 0x1.cd5f99c38b04ap-11, 0x1.a36e2eb1c432dp-11,
    0x1.797cc39ffd60ep-11, 0x1.4f8b588e368f0p-11, 0x1.2599ed7c6fbd3p-11, 0x1.f75104d551d69p-12,
    0x1.a36e2eb1c432bp-12, 0x1.4f8b588e368f2p-12, 0x1.f75104d551d69p-13, 0x1.4f8b588e368eep-13};
__constant__ float kAmmoNorm[8] = {0x0.0p+0f, 0x1.555556p-3f, 0x1.555556p-2f, 0x1.0p-1f,
                                   0x1.555556p-1f, 0x1.aaaaaap-1f, 0x1.0p+0f, 0x1.2aaaaap+0f};

struct Params {
    uint4 *state;            // [5][stride] packed planes (read/write)
    const uint4 *state_in;   // OP_OBS: snapshot planes (read only)
    int64_t stride;          // plane stride in envs
    int64_t count;           // envs (or index entries) to process
    const int64_t *idx;      // INDEXED: local env index per entry
    const int8_t *a1, *a2;
    const uint32_t *table;   // draw table or nullptr (Philox)
    void *obs1, *obs2;
    uint4 *bits1, *bits2;    // optional: packed observation rows, 16 x 16 B per env (host-expand path)
    float *extra1, *extra2;
    float *reward;
    double *reward64;        // optional: the unrounded binary64 reward (INV_FLAG_REWARD_F64)
    uint8_t *done, *info, *dbg;
    int32_t *ep_steps;
    double *ep_return;
    uint32_t *status;
    uint32_t seed_lo, seed_hi, env_id_base;
    int mode, difficulty, max_steps, auto_reset;
    int view;                // OP_OBS: 0 = P1, 1 = P2
    int phase, pid, arg, arg2; // OP_DEBUG
};

// ------------------------------------------------------------------------------------------------
// Philox4x32-10 counter-based generator (Salmon et al., SC'11). Counter = (global env id, episode,
// stream, k/4), key = seed; stream = pre-step step_count for the opponent's draws,
// INV_STREAM_RESET for spawn draws. Replaces the reference's two Mersenne Twister streams
// (core.py:41, env_wrappers.py:5) -- the oracle and the live-reference harness inject the same.
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                              uint32_t k0, uint32_t k1, uint32_t (&out)[4])
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

struct Draws {
    uint32_t c0, c1, c2, k0, k1;
    const uint32_t *tab; // this env's table row (already offset), or nullptr
    uint32_t v[4];
    int k;
    __device__ __forceinline__ void init(const Params &p, uint32_t gid, uint32_t episode, uint32_t stream,
                                         const uint32_t *row)
    {
        c0 = gid; c1 = episode; c2 = stream; k0 = p.seed_lo; k1 = p.seed_hi; tab = row; k = 0;
    }
    __device__ __forceinline__ uint32_t next()
    {
        if (tab) return tab[k++];
        const int lane = k & 3;
        if (lane == 0) philox4x32_10(c0, c1, c2, (uint32_t)(k >> 2), k0, k1, v);
        ++k;
        return lane == 0 ? v[0] : lane == 1 ? v[1] : lane == 2 ? v[2] : v[3];
    }
    // random._randbelow stand-in: floor(r * n / 2^32)
    __device__ __forceinline__ int below(int n) { return (int)__umulhi(next(), (uint32_t)n); }
};

// ------------------------------------------------------------------------------------------------
// Per-env state in registers. Tiles: bit (y*15+x) set = WHITE (P1 walks on WHITE, P2 on BLACK;
// game_types.py:58, config.py:9,11).
struct Env {
    uint32_t t[5];
    int x[2], y[2], ammo[2], reload[2], alive[2];
    int nb;
    uint32_t step, episode;
    double ret;
};

INV_HD uint32_t pack_player(const Env &s, int i)
{
    return (uint32_t)s.x[i] | ((uint32_t)s.y[i] << 4) | ((uint32_t)s.ammo[i] << 8) |
           ((uint32_t)s.reload[i] << 11) | ((uint32_t)s.alive[i] << 16);
}
INV_HD void unpack_player(Env &s, int i, uint32_t w)
{
    s.x[i] = w & 15; s.y[i] = (w >> 4) & 15; s.ammo[i] = (w >> 8) & 7;
    s.reload[i] = (w >> 11) & 31; s.alive[i] = (w >> 16) & 1;
}

// bullets live in a private shared-memory column: sb[slot * E]; 16-bit x | y<<4 | dir<<8 | owner<<10
INV_HD uint32_t pack_bullet(int x, int y, int dir, int owner)
{
    return (uint32_t)x | ((uint32_t)y << 4) | ((uint32_t)dir << 8) | ((uint32_t)owner << 10);
}
INV_HD void unpack_bullet(uint32_t b, int8_t (&q)[4]) // x, y, dir, owner
{
    q[0] = (int8_t)(b & 15); q[1] = (int8_t)((b >> 4) & 15); q[2] = (int8_t)((b >> 8) & 3); q[3] = (int8_t)((b >> 10) & 1);
}

// the episode return is stored as its two 32-bit halves
INV_HD double double_from_words(uint32_t lo, uint32_t hi)
{
#ifdef __CUDA_ARCH__
    return __hiloint2double((int)hi, (int)lo);
#else
    const uint64_t bits = ((uint64_t)hi << 32) | lo;
    double d;
    memcpy(&d, &bits, 8);
    return d;
#endif
}
INV_HD uint32_t double_lo_word(double d)
{
#ifdef __CUDA_ARCH__
    return (uint32_t)__double2loint(d);
#else
    uint64_t bits;
    memcpy(&bits, &d, 8);
    return (uint32_t)bits;
#endif
}
INV_HD uint32_t double_hi_word(double d)
{
#ifdef __CUDA_ARCH__
    return (uint32_t)__double2hiint(d);
#else
    uint64_t bits;
    memcpy(&bits, &d, 8);
    return (uint32_t)(bits >> 32);
#endif
}

// The two RNG counter words of an env, (step_count, episode), from its planes 1 and 2. Consumers
// that need only the counters (the evaluator's action selector and episode tally) read them here.
struct Counters {
    uint32_t step, episode;
};
INV_HD Counters counters_from_planes(const uint4 &b, const uint4 &c) { return Counters{b.w, c.x}; }
INV_HD Counters load_counters(const uint4 *st, int64_t stride, int64_t i)
{
    return counters_from_planes(st[stride + i], st[2 * stride + i]);
}

// Everything but the bullet column, from planes 0-2.
INV_HD void board_from_planes(Env &s, const uint4 &a, const uint4 &b, const uint4 &c)
{
    s.t[0] = a.x; s.t[1] = a.y; s.t[2] = a.z; s.t[3] = a.w; s.t[4] = b.x;
    unpack_player(s, 0, b.y);
    s.nb = (int)(b.y >> 20) & 31;
    unpack_player(s, 1, b.z);
    const Counters k = counters_from_planes(b, c);
    s.step = k.step;
    s.episode = k.episode;
    s.ret = double_from_words(c.y, c.z);
}
// Planes 0-2 only (48 of the 80 bytes): tiles, players and counters, for consumers that never
// read a bullet (the scripted players of inv_scripted_actions).
INV_HD void load_board(Env &s, const uint4 *st, int64_t stride, int64_t i)
{
    board_from_planes(s, st[i], st[stride + i], st[2 * stride + i]);
}

template <int E>
INV_HD void load_env(Env &s, uint16_t *sb, const uint4 *st, int64_t stride, int64_t i)
{
    const uint4 a = st[i], b = st[stride + i], c = st[2 * stride + i];
    const uint4 d = st[3 * stride + i], e = st[4 * stride + i];
    board_from_planes(s, a, b, c);
    const uint32_t w[8] = {d.x, d.y, d.z, d.w, e.x, e.y, e.z, e.w};
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        if (2 * k < s.nb) { // slots >= nb hold zeros and are never read
            sb[(2 * k) * E] = (uint16_t)(w[k] & 0xFFFFu);
            sb[(2 * k + 1) * E] = (uint16_t)(w[k] >> 16);
        }
    }
}

template <int E>
INV_HD void store_env(const Env &s, const uint16_t *sb, uint4 *st, int64_t stride, int64_t i)
{
    st[i] = make_uint4(s.t[0], s.t[1], s.t[2], s.t[3]);
    st[stride + i] = make_uint4(s.t[4], pack_player(s, 0) | ((uint32_t)s.nb << 20), pack_player(s, 1), s.step);
    st[2 * stride + i] = make_uint4(s.episode, double_lo_word(s.ret), double_hi_word(s.ret), 0u);
    uint32_t w[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const uint32_t lo = (2 * k < s.nb) ? sb[(2 * k) * E] : 0u;     // slots >= nb are stored as 0
        const uint32_t hi = (2 * k + 1 < s.nb) ? sb[(2 * k + 1) * E] : 0u; // (canonical bytes)
        w[k] = lo | (hi << 16);
    }
    st[3 * stride + i] = make_uint4(w[0], w[1], w[2], w[3]);
    st[4 * stride + i] = make_uint4(w[4], w[5], w[6], w[7]);
}

// Env + its bullet column (E = 1) <-> the canonical inv_env_state of the C ABI (host only).
inline void env_to_canonical(const Env &s, const uint16_t *sb, inv_env_state &o)
{
    o = inv_env_state{};
    int32_t *pp[2] = {o.p1, o.p2};
    for (int k = 0; k < 5; ++k) o.tiles[k] = s.t[k];
    for (int i = 0; i < 2; ++i) {
        pp[i][0] = s.x[i]; pp[i][1] = s.y[i]; pp[i][2] = s.ammo[i]; pp[i][3] = s.reload[i]; pp[i][4] = s.alive[i];
    }
    o.n_bullets = s.nb;
    for (int k = 0; k < s.nb && k < kSlots; ++k) unpack_bullet(sb[k], o.bullets[k]);
    o.step_count = (int32_t)s.step;
    o.episode = s.episode;
    o.episode_return = s.ret;
}

// false if a field does not fit the packed layout (or the board)
inline bool env_from_canonical(const inv_env_state &in, Env &s, uint16_t *sb)
{
    if (in.tiles[4] >> (kTiles - 128)) return false; // bits beyond the 150 tiles
    if (in.n_bullets < 0 || in.n_bullets > kSlots) return false;
    const int32_t *pp[2] = {in.p1, in.p2};
    for (int k = 0; k < 5; ++k) s.t[k] = in.tiles[k];
    for (int i = 0; i < 2; ++i) {
        const int32_t *q = pp[i];
        if (q[0] < 0 || q[0] >= kW || q[1] < 0 || q[1] >= kH || q[2] < 0 || q[2] > 7 || q[3] < 0 || q[3] > 31 ||
            (q[4] != 0 && q[4] != 1))
            return false;
        s.x[i] = q[0]; s.y[i] = q[1]; s.ammo[i] = q[2]; s.reload[i] = q[3]; s.alive[i] = q[4];
    }
    s.nb = in.n_bullets;
    for (int k = 0; k < s.nb; ++k) {
        const int8_t *q = in.bullets[k];
        if (q[0] < 0 || q[0] >= kW || q[1] < 0 || q[1] >= kH || q[2] < 0 || q[2] > 3 || q[3] < 0 || q[3] > 1)
            return false;
        sb[k] = (uint16_t)pack_bullet(q[0], q[1], q[2], q[3]);
    }
    s.step = (uint32_t)in.step_count;
    s.episode = in.episode;
    s.ret = in.episode_return;
    return true;
}

// ---- tile bit access on the 5 register words (select chains: no local memory, no smem) ----
__device__ __forceinline__ uint32_t tile_white(const Env &s, int x, int y)
{
    const int idx = y * kW + x;
    const int w = idx >> 5;
    uint32_t v = s.t[0];
    v = (w == 1) ? s.t[1] : v;
    v = (w == 2) ? s.t[2] : v;
    v = (w == 3) ? s.t[3] : v;
    v = (w == 4) ? s.t[4] : v;
    return (v >> (idx & 31)) & 1u;
}
__device__ __forceinline__ void tile_flip(Env &s, int x, int y)
{
    const int idx = y * kW + x;
    const int w = idx >> 5;
    const uint32_t bit = 1u << (idx & 31);
#pragma unroll
    for (int k = 0; k < 5; ++k) s.t[k] ^= (w == k) ? bit : 0u;
}
__device__ __forceinline__ void tile_set(Env &s, int x, int y, uint32_t white)
{
    const int idx = y * kW + x;
    const int w = idx >> 5;
    const uint32_t bit = 1u << (idx & 31);
#pragma unroll
    for (int k = 0; k < 5; ++k)
        if (w == k) s.t[k] = white ? (s.t[k] | bit) : (s.t[k] & ~bit);
}
__device__ __forceinline__ bool in_bounds(int x, int y) // core.py:222-224
{
    return (unsigned)x < (unsigned)kW && (unsigned)y < (unsigned)kH;
}
__device__ __forceinline__ int dir_dx(int d) { return (d == 1) - (d == 3); } // UP,RIGHT,DOWN,LEFT
__device__ __forceinline__ int dir_dy(int d) { return (d == 2) - (d == 0); }
__device__ __forceinline__ int count_white(const Env &s)
{
    return __popc(s.t[0]) + __popc(s.t[1]) + __popc(s.t[2]) + __popc(s.t[3]) + __popc(s.t[4]);
}

// ---- engine: core.py ----

// core.py:249-296. A player stands only on the colour that is not its own: P1 (BLACK) on WHITE,
// P2 (WHITE) on BLACK. No player-player collision.
__device__ __forceinline__ int try_move(Env &s, int pid, int dir)
{
    if (!s.alive[pid]) return 0;
    const int nx = s.x[pid] + dir_dx(dir), ny = s.y[pid] + dir_dy(dir);
    if (!in_bounds(nx, ny)) return 0;
    if (tile_white(s, nx, ny) != (uint32_t)(pid == 0)) return 0;
    s.x[pid] = nx; s.y[pid] = ny;
    return 1;
}

template <int E>
__device__ __forceinline__ void append_bullet(Env &s, uint16_t *sb, int x, int y, int dir, int owner, uint32_t *status)
{
    if (s.nb < kSlots) {
        sb[s.nb * E] = (uint16_t)pack_bullet(x, y, dir, owner);
        ++s.nb;
    } else {
        atomicOr(status, INV_STATUS_BULLET_OVERFLOW);
    }
}

// core.py:298-326: the bullet is appended AT the shooter's tile; it moves in the same tick.
template <int E>
__device__ __forceinline__ int spawn_bullet(Env &s, uint16_t *sb, int pid, int dir, uint32_t *status)
{
    if (!s.alive[pid] || s.ammo[pid] <= 0) return 0;
    s.ammo[pid] -= 1;
    append_bullet<E>(s, sb, s.x[pid], s.y[pid], dir, pid, status);
    return 1;
}

// core.py:328-381: 3 ammo even when a side lane is clipped; lane order centre, -1, +1;
// vertical shots spread in x, horizontal shots in y.
template <int E>
__device__ __forceinline__ int spawn_wide_shot(Env &s, uint16_t *sb, int pid, int dir, uint32_t *status)
{
    if (!s.alive[pid] || s.ammo[pid] < kWideCost) return 0;
    s.ammo[pid] -= kWideCost;
    const int px = s.x[pid], py = s.y[pid];
    const int ox = (dir & 1) ? 0 : 1, oy = (dir & 1) ? 1 : 0;
    int spawned = 0;
#pragma unroll
    for (int l = 0; l < 3; ++l) {
        const int off = (l == 0) ? 0 : (l == 1 ? -1 : 1);
        const int bx = px + off * ox, by = py + off * oy;
        if (in_bounds(bx, by)) { append_bullet<E>(s, sb, bx, by, dir, pid, status); ++spawned; }
    }
    return spawned > 0;
}

// core.py:383-397: the counter only runs below full ammo and is not reset by firing.
__device__ __forceinline__ void reload_ammo(Env &s)
{
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        if (s.alive[i] && s.ammo[i] < kMaxAmmo) {
            s.reload[i] += 1;
            if (s.reload[i] >= kReloadTicks) { s.ammo[i] += 1; s.reload[i] = 0; }
        }
    }
}

// core.py:399-475. Pass 1 advances and drops off-board bullets (stable, in place). Pass 2 decides
// per bullet: it survives iff it is the FIRST bullet (list order) on its tile and no bullet of the
// other owner landed there; a survivor flips the tile if it shows its owner's colour and kills
// the other player standing on it. Survivors keep list order (= dict insertion order of the
// reference, since at most one bullet per tile survives). Pass 3 compacts.
template <int E>
__device__ __forceinline__ void update_bullets(Env &s, uint16_t *sb)
{
    int m = 0;
    for (int i = 0; i < s.nb; ++i) {
        const uint32_t b = sb[i * E];
        const int dir = (b >> 8) & 3;
        const int nx = (int)(b & 15) + dir_dx(dir), ny = (int)((b >> 4) & 15) + dir_dy(dir);
        if (in_bounds(nx, ny)) {
            sb[m * E] = (uint16_t)((b & 0xFF00u) | (uint32_t)nx | ((uint32_t)ny << 4));
            ++m;
        }
    }
    uint32_t keep = 0;
    for (int i = 0; i < m; ++i) {
        const uint32_t bi = sb[i * E];
        const uint32_t key = bi & 0xFFu, owner = (bi >> 10) & 1u;
        bool first = true, mixed = false;
        for (int j = 0; j < m; ++j) {
            const uint32_t bj = sb[j * E];
            if (j != i && (bj & 0xFFu) == key) {
                first = first && (j > i);
                mixed = mixed || (((bj >> 10) & 1u) != owner);
            }
        }
        if (first && !mixed) {
            keep |= 1u << i;
            const int x = key & 15, y = key >> 4;
            // owner 0 (P1, BLACK) flips BLACK->WHITE; owner 1 (P2, WHITE) flips WHITE->BLACK
            if (tile_white(s, x, y) == owner) tile_flip(s, x, y);
            // the other player standing on the tile dies; the bullet flies on (core.py:464-473)
            if (owner) { if (s.alive[0] && s.x[0] == x && s.y[0] == y) s.alive[0] = 0; }
            else       { if (s.alive[1] && s.x[1] == x && s.y[1] == y) s.alive[1] = 0; }
        }
    }
    int k = 0;
    for (int i = 0; i < m; ++i)
        if ((keep >> i) & 1u) { sb[k * E] = sb[i * E]; ++k; }
    s.nb = k;
}

// env_wrappers.py:20-66 + core.py:510-525
template <int E>
__device__ __forceinline__ void apply_action(Env &s, uint16_t *sb, int pid, int a, uint32_t *status)
{
    if (a >= 1 && a <= 4) try_move(s, pid, a - 1);
    else if (a >= 5 && a <= 8) spawn_bullet<E>(s, sb, pid, a - 5, status);
    else if (a >= 9 && a <= 12) spawn_wide_shot<E>(s, sb, pid, a - 9, status);
}

// core.py:497-531: P1, then P2, then reload, then bullets.
template <int E>
__device__ __forceinline__ void step_players(Env &s, uint16_t *sb, int a1, int a2, uint32_t *status)
{
    apply_action<E>(s, sb, 0, a1, status);
    apply_action<E>(s, sb, 1, a2, status);
    reload_ammo(s);
    update_bullets<E>(s, sb);
}

// core.py:55-154 on the fixed 15x10 board: spawns are in [1,13]x[1,8], so no plus is clipped.
__device__ __forceinline__ void paint_plus(Env &s, int cx, int cy, uint32_t white)
{
    tile_set(s, cx, cy, white);
    tile_set(s, cx + 1, cy, white);
    tile_set(s, cx - 1, cy, white);
    tile_set(s, cx, cy + 1, white);
    tile_set(s, cx, cy - 1, white);
}
__device__ __forceinline__ void engine_reset(Env &s, Draws &dr)
{
    const int p1x = 1 + dr.below(kW - 2), p1y = 1 + dr.below(kH - 2); // randint(1, W-2), randint(1, H-2)
    int p2x = 0, p2y = 0;
    for (int t = 0; t < 20; ++t) { // core.py:85-90: the 20th draw is kept whatever its distance
        p2x = 1 + dr.below(kW - 2);
        p2y = 1 + dr.below(kH - 2);
        if (abs(p2x - p1x) + abs(p2y - p1y) > 4) break;
    }
    // config.py:20-56: all BLACK with the legacy WHITE plus around (1,1): bits 1,15,16,17,31
    s.t[0] = (1u << 1) | (1u << 15) | (1u << 16) | (1u << 17) | (1u << 31);
    s.t[1] = s.t[2] = s.t[3] = s.t[4] = 0u;
    paint_plus(s, p2x, p2y, 1u); // core.py:96-108
    paint_plus(s, p1x, p1y, 1u); // core.py:112-121
    paint_plus(s, p2x, p2y, 0u); // core.py:136-146 wins every overlap
    s.x[0] = p1x; s.y[0] = p1y; s.x[1] = p2x; s.y[1] = p2y;
    s.ammo[0] = s.ammo[1] = kMaxAmmo;
    s.reload[0] = s.reload[1] = 0;
    s.alive[0] = s.alive[1] = 1;
    s.nb = 0;
}

// ---- wrapper: env_wrappers.py ----

// env_wrappers.py:115-119 for the player P: on the board and on the colour try_move lets P enter
// (WHITE for P1, BLACK for P2)
template <int P>
__device__ __forceinline__ bool can_step(const Env &s, int dir)
{
    const int nx = s.x[P] + dir_dx(dir), ny = s.y[P] + dir_dy(dir);
    return in_bounds(nx, ny) && tile_white(s, nx, ny) == (uint32_t)(P == 0);
}

// four 2-bit direction fields; random.shuffle = Fisher-Yates from the top (CPython Lib/random.py)
__device__ __forceinline__ uint32_t shuffle4(uint32_t d, Draws &dr)
{
#pragma unroll
    for (int i = 3; i >= 1; --i) {
        const int j = dr.below(i + 1);
        const uint32_t vi = (d >> (2 * i)) & 3u, vj = (d >> (2 * j)) & 3u;
        d &= ~((3u << (2 * i)) | (3u << (2 * j)));
        d |= (vj << (2 * i)) | (vi << (2 * j));
    }
    return d;
}

// env_wrappers.py:69-170 played by player P against player 1 - P. Returns P's action id; consumes
// 0..9 draws in the reference's order. P = 1 is the reference's dummy (the simulator's opponent);
// P = 0 is the same rule with the roles exchanged (inv_scripted_actions, seat 0).
template <int P>
__device__ __forceinline__ int dummy_policy(const Env &s, Draws &dr, int difficulty)
{
    constexpr int Q = 1 - P; // the player chased
    if (!s.alive[P]) return 0; // :77-78, no draw
    const bool hard = difficulty != 0;
    const bool x_al = s.x[P] == s.x[Q], y_al = s.y[P] == s.y[Q];
    const bool should_shoot = dr.next() < (hard ? kThreshShootHard : 0u); // :96
    if (should_shoot && s.ammo[P] > 0 && (x_al || y_al)) {
        if (x_al) return 5 + (s.y[Q] < s.y[P] ? 0 : 2);  // :98-99 UP / DOWN (DOWN on the same tile)
        return 5 + (s.x[Q] < s.x[P] ? 3 : 1);            // :100-101 LEFT / RIGHT
    }
    uint32_t dirs = 0u | (2u << 2) | (3u << 4) | (1u << 6); // [UP, DOWN, LEFT, RIGHT]  :104
    if (dr.next() < (hard ? kThreshRandMoveHard : 0u)) {    // :105
        dirs = shuffle4(dirs, dr);
        const int c = dirs & 3u;
        if (can_step<P>(s, c)) return 1 + c;
    }
    if (!hard) {                                            // :122-124
        if (!(dr.next() < kThreshMoveEasy)) return 0;
    }
    const int dx = s.x[Q] - s.x[P], dy = s.y[Q] - s.y[P];   // :127-136
    int c0 = -1, c1 = -1;
    if (dx != 0) c0 = dx > 0 ? 1 : 3;
    if (dy != 0) { const int v = dy > 0 ? 2 : 0; if (c0 < 0) c0 = v; else c1 = v; }
    if (c1 >= 0) { // shuffle of a 2-list: j = randbelow(2); swap(x[1], x[j])   :138
        if (dr.below(2) == 0) { const int t = c0; c0 = c1; c1 = t; }
    }
    if (c0 >= 0 && can_step<P>(s, c0)) return 1 + c0;
    if (c1 >= 0 && can_step<P>(s, c1)) return 1 + c1;
    dirs = shuffle4(dirs, dr);                              // :155 (possibly already permuted)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int c = (dirs >> (2 * i)) & 3u;
        if (can_step<P>(s, c)) return 1 + c;
    }
    return 0;
}

// The third counter word of the scripted draws of inv_scripted_actions for `seat`: the step's
// opponent stream (seat 1, what a dummy-mode step consumes) or 0x80000000 | step_count (seat 0),
// which no simulator stream (step_count < 2^31, INV_STREAM_RESET) can equal.
INV_HD uint32_t scripted_stream(int seat, uint32_t step) { return seat ? step : (INV_STREAM_SEAT0 | step); }

// inv_scripted_actions for one env: the scripted rule played by `seat` (0 = P1, 1 = P2) on the
// pre-step state, with the draws of counter (gid, episode, scripted_stream(seat, step_count), k/4).
__device__ __forceinline__ int scripted_action(const Env &s, const Params &p, uint32_t gid, int seat, int difficulty)
{
    Draws dr;
    dr.init(p, gid, s.episode, scripted_stream(seat, s.step), nullptr);
    return seat ? dummy_policy<1>(s, dr, difficulty) : dummy_policy<0>(s, dr, difficulty);
}

// (float)(k / 6.0) for the extra vector (env_wrappers.py:238-243)
__device__ __forceinline__ float ammo_norm(int k) { return kAmmoNorm[k & 7]; }
__device__ __forceinline__ float4 extra_vec(const Env &s, int viewer)
{
    const int e = 1 - viewer;
    return make_float4(s.alive[viewer] ? ammo_norm(s.ammo[viewer]) : 0.0f,
                       s.alive[e] ? ammo_norm(s.ammo[e]) : 0.0f,
                       s.alive[viewer] ? 1.0f : 0.0f, s.alive[e] ? 1.0f : 0.0f);
}

// The observation as a bit string in the reference's element order (env_wrappers.py:186-235):
// bit (ch*150 + y*15 + x). ch0 = BLACK, ch1 = WHITE (never swapped), ch2 = viewer, ch3 = enemy,
// ch4-7 = viewer's bullets by dir, ch8-11 = enemy's bullets by dir.
template <int E>
__device__ __forceinline__ void build_row(uint32_t *row, const Env &s, const uint16_t *sb, int viewer)
{
    const uint32_t *t = s.t;
    row[0] = ~t[0]; row[1] = ~t[1]; row[2] = ~t[2]; row[3] = ~t[3];
    row[4] = (~t[4] & 0x3FFFFFu) | (t[0] << 22);
    row[5] = (t[0] >> 10) | (t[1] << 22);
    row[6] = (t[1] >> 10) | (t[2] << 22);
    row[7] = (t[2] >> 10) | (t[3] << 22);
    row[8] = (t[3] >> 10) | (t[4] << 22);
    row[9] = (t[4] >> 10);
#pragma unroll
    for (int k = 10; k < kRowWords; ++k) row[k] = 0u;
    const int e = 1 - viewer;
    if (s.alive[viewer]) { const int b = 2 * kTiles + s.y[viewer] * kW + s.x[viewer]; row[b >> 5] |= 1u << (b & 31); }
    if (s.alive[e])      { const int b = 3 * kTiles + s.y[e] * kW + s.x[e];           row[b >> 5] |= 1u << (b & 31); }
    for (int i = 0; i < s.nb; ++i) {
        const uint32_t bl = sb[i * E];
        const int ch = ((((bl >> 10) & 1u) == (uint32_t)viewer) ? 4 : 8) + (int)((bl >> 8) & 3u);
        const int b = ch * kTiles + (int)((bl >> 4) & 15u) * kW + (int)(bl & 15u);
        row[b >> 5] |= 1u << (b & 31);
    }
}

// ---- the wrapper step as one function (also compiled for the host by tests/host_kernel) ----

struct StepResult {
    float reward;      // env_wrappers.py:525 (binary64 sum rounded to float32)
    double reward64;   // the sum itself (what SingleInversusRLEnv.step returns, env_wrappers.py:444)
    uint8_t done, info;
    int32_t ep_steps;  // info["episode_steps"], before any auto-reset
    double ep_return;  // info["episode_return"]
};

// env_wrappers.py:272-284 (+ core.py:55-154): a new episode in place.
__device__ __forceinline__ void rl_reset(Env &s, const Params &p, uint32_t gid, const uint32_t *trow)
{
    s.episode += 1u;
    Draws dr;
    dr.init(p, gid, s.episode, INV_STREAM_RESET, trow ? trow + INV_TABLE_RESET_OFF : nullptr);
    engine_reset(s, dr);
    s.step = 0u;
    s.ret = 0.0;
}

// env_wrappers.py:286-444 for one env: P2's action (scripted, or given in selfplay mode), engine tick,
// reward shaping, done/timeout, and -- with auto_reset -- the trainer's reset-on-done
// (training.py:148-151). Ids outside 0..12 raise the sticky status bit and act as NONE.
template <int E>
__device__ __forceinline__ StepResult rl_step(Env &s, uint16_t *sb, int a1, int a2, const Params &p, uint32_t gid,
                                              const uint32_t *trow)
{
    if ((unsigned)a1 > 12u) { atomicOr(p.status, INV_STATUS_INVALID_ACTION); a1 = 0; }
    if (p.mode == INV_MODE_DUMMY) { // env_wrappers.py:305-306
        Draws dr;
        dr.init(p, gid, s.episode, s.step, trow);
        a2 = dummy_policy<1>(s, dr, p.difficulty);
    } else if ((unsigned)a2 > 12u) { // :307-314, the caller ran opponent_policy
        atomicOr(p.status, INV_STATUS_INVALID_ACTION);
        a2 = 0;
    }
    const int prev_alive0 = s.alive[0], prev_alive1 = s.alive[1]; // :319-320
    const int white0 = count_white(s);                            // :328-329
    step_players<E>(s, sb, a1, a2, p.status);                     // :332
    s.step += 1u;                                                 // :333

    // reward shaping in binary64, in the reference's order (env_wrappers.py:343-438);
    // _rn intrinsics keep nvcc from contracting mul+add into fma.
    double r = 0.0;
    uint32_t info = 0u;
    const int diff = count_white(s) - white0;
    if (diff > 0) r = __dadd_rn(r, __dmul_rn((double)diff, 0.01));                          // :352-354
    if (prev_alive1 && !s.alive[1]) { r = __dadd_rn(r, 1.0); info |= INV_INFO_LANDED_HIT; } // :357-360
    if (prev_alive0 && !s.alive[0]) { r = __dadd_rn(r, -0.01); info |= INV_INFO_GOT_HIT; }  // :364-367
    if (s.alive[0] && s.ammo[0] == 0) r = __dadd_rn(r, -0.001);                             // :372-373
    if (s.alive[0] && s.alive[1]) {                                                         // :377-405
        const int dist = abs(s.x[0] - s.x[1]) + abs(s.y[0] - s.y[1]);
        r = __dadd_rn(r, kProximity[dist]); // 0.002 * (1 - dist / 25), dist <= 23
        const bool aligned = (s.x[0] == s.x[1]) || (s.y[0] == s.y[1]);
        if (aligned) r = __dadd_rn(r, 0.002);
        if (a1 >= 5 && aligned && s.ammo[0] > 0) {
            const int sd = (a1 - 5) & 3;
            bool aim = false;
            if (s.x[0] == s.x[1]) aim = (s.y[0] < s.y[1] && sd == 2) || (s.y[0] > s.y[1] && sd == 0);
            else                  aim = (s.x[0] < s.x[1] && sd == 1) || (s.x[0] > s.x[1] && sd == 3);
            if (aim) r = __dadd_rn(r, 0.05);
        }
    }
    bool done = false;
    const bool over = !(s.alive[0] && s.alive[1]);                                          // core.py:477-481
    if (over) {                                                                             // :408-422
        done = true;
        if (s.alive[0]) { r = __dadd_rn(r, 10.0); info |= INV_INFO_WIN; }
        else if (s.alive[1]) { r = __dadd_rn(r, -0.1); info |= INV_INFO_LOSE; }
    } else {
        r = __dadd_rn(r, -0.001);                                                           // :425
    }
    if (s.step >= (uint32_t)p.max_steps) {                                                  // :434-438
        done = true;
        if (!over) r = __dadd_rn(r, -2.0);
    }
    s.ret = __dadd_rn(s.ret, r);                                                            // :440
    StepResult o;
    o.reward = __double2float_rn(r);
    o.reward64 = r;
    o.done = done ? 1 : 0;
    o.info = (uint8_t)info;
    o.ep_steps = (int32_t)s.step;
    o.ep_return = s.ret;
    if (done && p.auto_reset) rl_reset(s, p, gid, trow);                                    // training.py:148-151
    return o;
}

// One engine method of core.py, selected by p.phase (inv_debug_phase); returns the method's result.
template <int E>
__device__ __forceinline__ uint8_t debug_phase(Env &s, uint16_t *sb, const Params &p, uint32_t gid, const uint32_t *trow)
{
    int res = 0;
    switch (p.phase) {
    case INV_PHASE_TRY_MOVE:
        res = p.pid ? try_move(s, 1, p.arg) : try_move(s, 0, p.arg);
        break;
    case INV_PHASE_SPAWN_BULLET:
        res = p.pid ? spawn_bullet<E>(s, sb, 1, p.arg, p.status) : spawn_bullet<E>(s, sb, 0, p.arg, p.status);
        break;
    case INV_PHASE_WIDE_SHOT:
        res = p.pid ? spawn_wide_shot<E>(s, sb, 1, p.arg, p.status) : spawn_wide_shot<E>(s, sb, 0, p.arg, p.status);
        break;
    case INV_PHASE_RELOAD: reload_ammo(s); break;
    case INV_PHASE_UPDATE_BULLETS: update_bullets<E>(s, sb); break;
    case INV_PHASE_STEP_PLAYERS: step_players<E>(s, sb, p.arg, p.arg2, p.status); break;
    case INV_PHASE_ENGINE_RESET: {
        s.episode += 1u;
        Draws dr;
        dr.init(p, gid, s.episode, INV_STREAM_RESET, trow ? trow + INV_TABLE_RESET_OFF : nullptr);
        engine_reset(s, dr);
        break;
    }
    case INV_PHASE_DUMMY_POLICY: {
        Draws dr;
        dr.init(p, gid, s.episode, s.step, trow);
        res = dummy_policy<1>(s, dr, p.difficulty);
        break;
    }
    default: break;
    }
    return (uint8_t)res;
}

#ifndef INV_HOST_BUILD
// ---- observation formats: how many store chunks per env and how a chunk is expanded ----
template <int DT> struct ObsFmt;
struct __align__(32) uint8v { uint4 lo, hi; }; // one 32-byte store (st.global.v8.b32, sm_100)
#ifndef INV_F32_STORE32
#define INV_F32_STORE32 1 // 32-byte stores: +5 % on the fp32 step kernel (profiles/r2_variants_f32.txt)
#endif
#if INV_F32_STORE32
template <> struct ObsFmt<INV_OBS_F32> {  // 1800 f32 = 225 x 32 B, 8 bits per chunk
    static constexpr int kChunks = 225, kBits = 8;
    typedef uint8v chunk_t;
    template <int K> static __device__ __forceinline__ uint32_t one(uint32_t b) { return (b & (1u << K)) * (0x3F800000u >> K); }
    static __device__ __forceinline__ chunk_t expand(uint32_t b)
    {
        chunk_t c; // bit k -> 1.0f or 0.0f in two instructions: isolate (LOP3), scale by 0x3F800000 >> k (IMAD, exact for k <= 23)
        c.lo = make_uint4(one<0>(b), one<1>(b), one<2>(b), one<3>(b));
        c.hi = make_uint4(one<4>(b), one<5>(b), one<6>(b), one<7>(b));
        return c;
    }
};
#else
template <> struct ObsFmt<INV_OBS_F32> {  // 1800 f32 = 450 x 16 B, 4 bits per chunk
    static constexpr int kChunks = 450, kBits = 4;
    typedef uint4 chunk_t;
    static __device__ __forceinline__ chunk_t expand(uint32_t b)
    {
        return make_uint4((b & 1u) ? 0x3F800000u : 0u, (b & 2u) ? 0x3F800000u : 0u,
                          (b & 4u) ? 0x3F800000u : 0u, (b & 8u) ? 0x3F800000u : 0u);
    }
};
#endif
template <> struct ObsFmt<INV_OBS_BF16> { // 1800 bf16 = 225 x 16 B, 8 bits per chunk
    static constexpr int kChunks = 225, kBits = 8;
    typedef uint4 chunk_t;
    static __device__ __forceinline__ uint32_t two(uint32_t b)
    {
        return ((b & 1u) ? 0x3F80u : 0u) | ((b & 2u) ? 0x3F800000u : 0u);
    }
    static __device__ __forceinline__ chunk_t expand(uint32_t b)
    {
        return make_uint4(two(b), two(b >> 2), two(b >> 4), two(b >> 6));
    }
};
template <> struct ObsFmt<INV_OBS_U8> {   // 1800 u8 = 225 x 8 B, 8 bits per chunk
    static constexpr int kChunks = 225, kBits = 8;
    typedef uint2 chunk_t;
    static __device__ __forceinline__ chunk_t expand(uint32_t b)
    {
        return make_uint2(((b & 15u) * 0x00204081u) & 0x01010101u, (((b >> 4) & 15u) * 0x00204081u) & 0x01010101u);
    }
};

#ifndef INV_ST_PLAIN
#define INV_ST_PLAIN 0
#endif
#if INV_ST_PLAIN
__device__ __forceinline__ void st_stream(uint4 *p, uint4 v) { *p = v; }
__device__ __forceinline__ void st_stream(uint2 *p, uint2 v) { *p = v; }
#else
__device__ __forceinline__ void st_stream(uint4 *p, uint4 v) { __stcs(p, v); }
__device__ __forceinline__ void st_stream(uint2 *p, uint2 v) { __stcs(p, v); }
#endif
template <> struct ObsFmt<INV_OBS_NONE> { // no observation tensor: the store phase is compiled out
    static constexpr int kChunks = 1, kBits = 0; // never used: the kernel leaves before phase 2
    typedef uint4 chunk_t;
    static __device__ __forceinline__ chunk_t expand(uint32_t) { return make_uint4(0u, 0u, 0u, 0u); }
};
__device__ __forceinline__ void st_stream(uint8v *p, uint8v v)
{
    asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(v.lo.x), "r"(v.lo.y), "r"(v.lo.z),
                 "r"(v.lo.w), "r"(v.hi.x), "r"(v.hi.y), "r"(v.hi.z), "r"(v.hi.w)
                 : "memory");
}

template <int E, bool P2V, bool INDEXED, int DT = INV_OBS_F32>
constexpr size_t smem_bytes()
{
    return (DT == INV_OBS_NONE ? 0 : (size_t)E * kRowWords * 4 * (P2V ? 2 : 1)) + (size_t)kSlots * E * 2 +
           (INDEXED ? (size_t)E * 8 : 0);
}

// ------------------------------------------------------------------------------------------------
// (A minimum-blocks hint was tried: (T, 5) and (T, 6) are slower, and even (T, 1) lets ptxas spend
// registers and costs 13 %: profiles/r2_variants_f32_b.txt. Plain __launch_bounds__(T) stays.)
template <int OP, int DT, bool P2V, bool INDEXED, int E, int T = kThreads>
__global__ void __launch_bounds__(T) inv_kernel(const Params p)
{
    static_assert(E <= T && E % 32 == 0 && T % 32 == 0, "tile must be whole warps");
    extern __shared__ __align__(16) uint32_t smem[];
    constexpr bool kObs = DT != INV_OBS_NONE;
    uint32_t *rows1 = smem;
    uint32_t *rows2 = rows1 + (P2V && kObs ? E * kRowWords : 0);
    uint16_t *sbul = reinterpret_cast<uint16_t *>(rows2 + (kObs ? E * kRowWords : 0));
    int64_t *s_env = reinterpret_cast<int64_t *>(sbul + kSlots * E); // INDEXED only
    typedef ObsFmt<DT> Fmt;
    typedef typename Fmt::chunk_t chunk_t;

    const int tid = threadIdx.x;
    const int64_t ntiles = (p.count + E - 1) / E;

    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t base = tile * E;
        const int nvalid = (int)min((int64_t)E, p.count - base);

        // ------------------------------------------------------------ phase 1: thread per env
        bool live = tid < nvalid;
        if (INDEXED && live) { // a bad index must not become an out-of-bounds write
            const int64_t cand = p.idx[base + tid];
            if ((uint64_t)cand >= (uint64_t)p.stride) {
                atomicOr(p.status, INV_STATUS_BAD_INDEX);
                s_env[tid] = -1;
                live = false;
            }
        }
        if (live) {
            const int64_t ei = INDEXED ? p.idx[base + tid] : base + tid;
            if (INDEXED) s_env[tid] = ei;
            uint16_t *sb = sbul + tid;
            uint32_t *row1 = rows1 + tid * kRowWords;
            Env s;
            load_env<E>(s, sb, OP == OP_OBS ? p.state_in : p.state, p.stride, ei);
            const uint32_t gid = p.env_id_base + (uint32_t)ei;
            const uint32_t *trow = p.table ? p.table + ei * INV_TABLE_STRIDE : nullptr;

            if (OP == OP_STEP) {
                const StepResult o = rl_step<E>(s, sb, p.a1[ei], p.mode == INV_MODE_DUMMY ? 0 : p.a2[ei], p, gid, trow);
                p.reward[ei] = o.reward;                                                           // env_wrappers.py:525
                if (p.reward64) p.reward64[ei] = o.reward64;
                p.done[ei] = o.done;
                p.info[ei] = o.info;
                p.ep_steps[ei] = o.ep_steps;
                p.ep_return[ei] = o.ep_return;
            } else if (OP == OP_RESET) { // env_wrappers.py:272-284
                rl_reset(s, p, gid, trow);
            } else if (OP == OP_DEBUG) {
                p.dbg[ei] = debug_phase<E>(s, sb, p, gid, trow);
            }

            if (OP != OP_OBS) store_env<E>(s, sb, p.state, p.stride, ei);

            if (OP != OP_DEBUG) {
                // extra vector: one coalesced 16 B store per env
                const int64_t eo = (OP == OP_OBS) ? base + tid : ei;
                if (OP == OP_OBS && p.view) { // viewer stays a compile-time constant in both arms
                    if (kObs) build_row<E>(row1, s, sb, 1);
                    reinterpret_cast<float4 *>(p.extra1)[eo] = extra_vec(s, 1);
                } else {
                    if (kObs) build_row<E>(row1, s, sb, 0);
                    reinterpret_cast<float4 *>(p.extra1)[eo] = extra_vec(s, 0);
                }
                if (P2V) {
                    if (kObs) build_row<E>(rows2 + tid * kRowWords, s, sb, 1);
                    reinterpret_cast<float4 *>(p.extra2)[eo] = extra_vec(s, 1);
                }
            }
        }
        if (OP == OP_DEBUG || !kObs) continue;
        __syncthreads();

        // ------------------------------------------------------------ phase 2: streaming obs store
#pragma unroll 1
        for (int v = 0; v < (P2V ? 2 : 1); ++v) {
            const uint32_t *rows = v ? rows2 : rows1;
            chunk_t *out = reinterpret_cast<chunk_t *>(v ? p.obs2 : p.obs1);
            const int total = nvalid * Fmt::kChunks;
            if (!INDEXED) {
                chunk_t *o = out + base * Fmt::kChunks;
#pragma unroll 4
                for (int g = tid; g < total; g += T) {
                    const int e = g / Fmt::kChunks;
                    const int bit = (g - e * Fmt::kChunks) * Fmt::kBits;
                    const uint32_t w = rows[e * kRowWords + (bit >> 5)] >> (bit & 31);
                    st_stream(o + g, Fmt::expand(w));
                }
            } else {
#pragma unroll 2
                for (int g = tid; g < total; g += T) {
                    const int e = g / Fmt::kChunks;
                    const int c = g - e * Fmt::kChunks;
                    const int bit = c * Fmt::kBits;
                    if (s_env[e] < 0) continue; // rejected index
                    const uint32_t w = rows[e * kRowWords + (bit >> 5)] >> (bit & 31);
                    st_stream(out + s_env[e] * Fmt::kChunks + c, Fmt::expand(w));
                }
            }
        }
        // optional packed copy of the same rows (1800 bits in 57 words, padded to 64 words = 256 B
        // per env): what inv_step_host ships over PCIe when the host expands the observation
        if (p.bits1) {
#pragma unroll 1
            for (int v = 0; v < (P2V ? 2 : 1); ++v) {
                const uint32_t *rows = v ? rows2 : rows1;
                uint4 *out = v ? p.bits2 : p.bits1;
                if (!out) continue;
                for (int g = tid; g < nvalid * 16; g += T) {
                    const int e = g >> 4, c = g & 15;
                    const uint32_t *r = rows + e * kRowWords + 4 * c;
                    uint4 w;
                    w.x = (4 * c + 0 < kRowWords) ? r[0] : 0u;
                    w.y = (4 * c + 1 < kRowWords) ? r[1] : 0u;
                    w.z = (4 * c + 2 < kRowWords) ? r[2] : 0u;
                    w.w = (4 * c + 3 < kRowWords) ? r[3] : 0u;
                    const int64_t eo = INDEXED ? s_env[e] : base + e;
                    if (INDEXED && eo < 0) continue;
                    out[eo * 16 + c] = w;
                }
            }
        }
        __syncthreads(); // the tile's shared rows are reused by the next iteration
    }
}

#endif // INV_HOST_BUILD

} // namespace inv
