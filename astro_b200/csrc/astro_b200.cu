// astro_b200.cu — kernels and C ABI (include/astro_b200.h) of the batched Astro game tick.
//
// Replaces, for N independent games at once:
//   astro/core.py:215-303  step            -> tick_kernel   (one fused launch per tick)
//   astro/core.py:306-327  roll_ships  }
//   astro/rl.py:43-99      get_features } -> observe_kernel
//                          to_batch     }
//   astro/core.py:86-135   create (host-built pool) -> reset inside tick_kernel / reset_kernel
//
// Thread-per-game over 32-game tiles: every global access is a coalesced 128-bit access across
// the warp (see the layout comment in the header).  HBM-bound; no tensor cores (no contraction).
#include "../../include/astro_b200.h"
#include "astro_device.cuh"
#include <cuda_fp16.h>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <type_traits>
#include <atomic>
#include <chrono>
#include <new>
#include <thread>
#include <vector>

using namespace astro;

namespace {

// One warp per CTA: a CTA holds its SM slot until its slowest warp ends, so the smallest CTA
// refills fastest (measured per 1M-game tick: 256 threads 111.3 us, 128: 96.0, 64: 94.0, 32: 93.3).
#ifndef ASTRO_PDL
#define ASTRO_PDL 1   /* programmatic dependent launch of the one-tick kernel: 69.8 -> 67.1 us per 1M-game tick */
#endif
#ifndef ASTRO_TICK_THREADS
#define ASTRO_TICK_THREADS 32
#endif
constexpr int kTickThreads = ASTRO_TICK_THREADS;
constexpr int kObserveWarps = 8;
constexpr int kStatReplicas = 64;   // copies of the 64-bit episode counters (16 words = one 128-byte line each), summed by astro_stats

struct TickParams {
    void* ships;
    void* ship_b;
    void* planets;
    void* bullets_in;   // the buffer holding the tiles' bullet lists, read by this tick
    void* bullets_out;  // the other buffer: receives the new lists
    uint32_t* meta;
    uint32_t* episode;
    const uint8_t* actions;
    float* reward;
    uint8_t* done;
    uint8_t* events;
    const uint32_t* fire_bits;
    const void* pool_ships;
    const void* pool_planets;
    const int32_t* pool_np;
    const float4* pool_rec;  // precision 32: the pool as one 128-byte record per entry (pack_pool_kernel)
    unsigned long long* stats;
    unsigned* stat_slots;  // u32 [n_tiles][16]: per-warp partial counters (tick_f32_kernel)
    int32_t n_games, K, timeout_tick, n_sched_ticks, pool_size, flags;
    uint32_t seed, step, first_game;
    int32_t n_fused;     // ticks per launch (tick_f32_kernel; 1 everywhere else)
    uint32_t act_stride, ev_stride;   // bytes from one tick's controls / events to the next tick's (0: no such array)
    uint32_t rw_stride, done_stride;  // the same for reward / done
    int32_t tile0, tiles;             // tick_f32_kernel: the launch covers tiles tile0 .. tile0 + tiles - 1
    float4* ring;                     // fresh-game mode (astro_fresh_games_enable): [n_tiles][quota] 128-byte records
    uint32_t* tile_used;              //   records of each tile consumed since the last refill
    uint32_t* game_pos;               //   [n_games] position in the generate_configs stream of each game's current episode
    int32_t quota, pad_;
    const uint32_t* step_base;        // captured launches (the bot loop as a CUDA graph): stream step = *step_base + step
    int32_t bot_modes, pad2_;         // bots evaluated inside the tick (tick_f32_kernel<..., BOT>): ASTRO_BOT_* of ship s in bits 4s..4s+3
    ScriptParams script;
    Consts c;
    // astro_rollout_device_record (tick_f32 kernels, non-FIX forms): the tick at stream step s stores its controls and event
    // byte into row s % rec_ticks.  Appended last so that no other parameter moves.
    uint8_t* rec_controls;            // u8 [rec_ticks][n_games][S], or NULL together with rec_events
    uint8_t* rec_events;              // u8 [rec_ticks][n_games]
    uint32_t rec_ticks, pad3_;
};


// Re-create game g from the reset pool (core.create, core.py:86-135, evaluated on the host):
// entry pick(seed, global game id, key) with key = 1 + the stream step of the tick that ended the
// game (0 for the initial fill) — no dependent load on the way; bullets cleared, tick 0.  The
// per-slot episode counter is bumped with a fire-and-forget RED.
template <typename R, int S, int PL>
__device__ __forceinline__ void recreate_from_pool(const TickParams& p, int g, uint32_t key, Body4<R>* ships,
                                                   R* ship_b, Body4<R>* planets) {
    using B4 = Body4<R>;
    atomicAdd(&p.episode[g], 1u);
    uint32_t k = pool_pick(p.seed, p.first_game + (uint32_t)g, key, (uint32_t)p.pool_size);
    const R* ps = reinterpret_cast<const R*>(p.pool_ships) + (size_t)k * (S * 5);
    const R* pp = reinterpret_cast<const R*>(p.pool_planets) + (size_t)k * (PL * 4);
    int np_new = p.pool_np[k];
#pragma unroll
    for (int s = 0; s < S; s++) {
        B4 o;
        o.x = ps[5 * s]; o.y = ps[5 * s + 1]; o.dx = ps[5 * s + 2]; o.dy = ps[5 * s + 3];
        ships[s * 32] = o;
        ship_b[s * 32] = ps[5 * s + 4];
    }
#pragma unroll
    for (int j = 0; j < PL; j++) {
        if (j < np_new) {
            B4 o;
            o.x = pp[4 * j]; o.y = pp[4 * j + 1]; o.dx = pp[4 * j + 2]; o.dy = pp[4 * j + 3];
            planets[j * 32] = o;
        }
    }
    p.meta[g] = meta_pack<PL>(0, np_new, 0, 0);
}

// The reset pool as one 128-byte record per entry, so that re-creating a game inside the tick is ONE
// round trip (the three pool arrays need the planet count first): floats 0 .. 5S-1 = ships
// (x, y, dx, dy, b each), word 10 = planet count, floats 16 .. 31 = planets.  8-slot batches: 256-byte
// records, planets in floats 16 .. 47.
template <int PL>
__host__ __device__ constexpr int pool_rec_float4s() { return PL > ASTRO_MAX_PLANETS ? 16 : 8; }
template <int S, int PL>
__global__ void pack_pool_kernel(const float* __restrict__ ships, const float* __restrict__ planets,
                                 const int32_t* __restrict__ np, float* __restrict__ rec, int m) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= m) return;
    float* r = rec + (size_t)k * (4 * pool_rec_float4s<PL>());
    for (int i = 0; i < 4 * pool_rec_float4s<PL>(); i++) r[i] = 0.f;
    for (int i = 0; i < 5 * S; i++) r[i] = ships[(size_t)k * (5 * S) + i];
    r[10] = __int_as_float(np[k]);
    for (int i = 0; i < 4 * PL; i++) r[16 + i] = planets[(size_t)k * (4 * PL) + i];
}

// Warp-level reduction of the per-game flags and counts into the block's shared counters:
// ballots / REDUX give warp-uniform totals, lane k keeps counter k, ONE shared atomic per warp.
// (32-bit shared counters: a block's per-tick totals are < 2^19.)
__device__ __forceinline__ unsigned warp_totals(int lane, int S, uint32_t ev, bool active, int spawned, int np,
                                               int nb, int m_out, bool have_nb_total = false, unsigned nb_total = 0u) {
    const unsigned full = 0xffffffffu;
    unsigned mine = 0;
    // most tiles, most ticks: nobody ended, overflowed or was skipped — the nine counters of those events (and the selects
    // that hand each to its lane) sit behind one ballot
    if (__ballot_sync(full, (ev & (ASTRO_EV_DONE_MASK | ASTRO_EV_OVERFLOW | ASTRO_EV_SKIPPED | ASTRO_EV_BAD_CONTROL | ASTRO_EV_AWAIT)) != 0)) {
        const bool coll = (ev & (ASTRO_EV_HIT0 | ASTRO_EV_HIT1)) != 0;
        const bool h0 = ev & ASTRO_EV_HIT0, h1 = ev & ASTRO_EV_HIT1;
        const unsigned v0 = __popc(__ballot_sync(full, (ev & ASTRO_EV_DONE_MASK) != 0));
        const unsigned v1 = __popc(__ballot_sync(full, S == 2 && coll && !h0));
        const unsigned v2 = __popc(__ballot_sync(full, S == 2 && coll && !h1));
        const unsigned v3 = __popc(__ballot_sync(full, coll && (S == 1 || (h0 && h1))));
        const unsigned v4 = __popc(__ballot_sync(full, (ev & ASTRO_EV_TIMEOUT) != 0));
        const unsigned v7 = __popc(__ballot_sync(full, (ev & ASTRO_EV_OVERFLOW) != 0));
        const unsigned v11 = __popc(__ballot_sync(full, (ev & ASTRO_EV_SKIPPED) != 0));
        const unsigned v12 = __popc(__ballot_sync(full, (ev & ASTRO_EV_BAD_CONTROL) != 0));
        const unsigned v13 = __popc(__ballot_sync(full, (ev & ASTRO_EV_AWAIT) != 0));
        mine = lane == 0 ? v0 : mine; mine = lane == 1 ? v1 : mine; mine = lane == 2 ? v2 : mine; mine = lane == 3 ? v3 : mine;
        mine = lane == 4 ? v4 : mine; mine = lane == 7 ? v7 : mine; mine = lane == 11 ? v11 : mine; mine = lane == 12 ? v12 : mine;
        mine = lane == 13 ? v13 : mine;
    }
    const unsigned v5 = __popc(__ballot_sync(full, active));
    const unsigned v6 = (unsigned)S * __popc(__ballot_sync(full, spawned != 0));
    const unsigned v8 = __reduce_add_sync(full, (unsigned)np);
    const unsigned v9 = have_nb_total ? nb_total : __reduce_add_sync(full, (unsigned)nb);     // (the tick has this sum already)
    const unsigned v10 = __reduce_add_sync(full, (unsigned)m_out);
    mine = lane == 5 ? v5 : mine; mine = lane == 6 ? v6 : mine; mine = lane == 8 ? v8 : mine; mine = lane == 9 ? v9 : mine;
    mine = lane == 10 ? v10 : mine;
    return mine;
}
__device__ __forceinline__ void warp_stats(unsigned* s_stats, int lane, int S, uint32_t ev, bool active,
                                           int spawned, int np, int nb, int m_out) {
    unsigned mine = warp_totals(lane, S, ev, active, spawned, np, nb, m_out);
    if (lane < ASTRO_N_STATS && mine) atomicAdd(&s_stats[lane], mine);
}

// Folds the per-warp slot rows of tick_f32_kernel into the 64-bit counters and clears them.
__global__ void fold_stats_kernel(unsigned* slots, int n_tiles, unsigned long long* stats) {
    __shared__ unsigned long long acc[ASTRO_N_STATS];
    if (threadIdx.x < ASTRO_N_STATS) acc[threadIdx.x] = 0ull;
    __syncthreads();
    const int k = threadIdx.x & 15;
    unsigned long long sum = 0;
    for (int tile = blockIdx.x * (blockDim.x >> 4) + (threadIdx.x >> 4); tile < n_tiles; tile += gridDim.x * (blockDim.x >> 4)) {
        unsigned* s = slots + (size_t)tile * 16 + k;
        unsigned v = *s;
        if (v) { sum += v; *s = 0u; }
    }
    if (k < ASTRO_N_STATS && sum) atomicAdd(&acc[k], sum);
    __syncthreads();
    if (threadIdx.x < ASTRO_N_STATS && acc[threadIdx.x]) atomicAdd(&stats[threadIdx.x], acc[threadIdx.x]);
}

// astro_stats: the kStatReplicas copies of the counters summed into `out` (and cleared).
__global__ void gather_stats_kernel(unsigned long long* stats, long long* out, int clear) {
    __shared__ unsigned long long acc[16];
    if (threadIdx.x < 16) acc[threadIdx.x] = 0ull;
    __syncthreads();
    unsigned long long sum = 0;
    for (int i = threadIdx.x; i < kStatReplicas * 16; i += blockDim.x) {
        const unsigned long long v = stats[i];
        if (v) { sum += v; if (clear) stats[i] = 0ull; }
    }
    if (sum) atomicAdd(&acc[threadIdx.x & 15], sum);     // (blockDim.x is a multiple of 16: a thread sees one counter)
    __syncthreads();
    if (threadIdx.x < ASTRO_N_STATS) out[threadIdx.x] = (long long)acc[threadIdx.x];
}

// astro_stats_allreduce: the episode counters of N processes (one GPU each, one node) summed in ONE kernel per rank over peer
// memory — no NCCL launch, no ring: every rank owns an exchange buffer [2][kPeerMax] rows of 16 words (14 counters, word 15 =
// the call number), mapped into every other process (CUDA IPC); call number n uses half n & 1.
//   1. this rank's counters = sum of the kStatReplicas copies (cleared on request)
//   2. thread r stores them into row `rank` of rank r's buffer — P2P stores through NVLink / NVSwitch — and, behind a
//      system-scope fence, the call number into the row's last word
//   3. thread r waits for row r of THIS rank's buffer to show the call number (the peers' stores land in local memory: the
//      poll never leaves the GPU), then the rows are summed into `out`.
// Two halves are enough: a rank can only be one call ahead of the slowest one (it needs that rank's row of the call to go on).
// A peer that never arrives (a rank died) ends the wait after ~2 s of polling with every counter set to -1.
constexpr int kPeerMax = 16;
struct PeerTable { unsigned long long* buf[kPeerMax]; };
__global__ void __launch_bounds__(256) stats_allreduce_kernel(unsigned long long* stats, long long* out, int clear, PeerTable peers,
                                                              int rank, int world, unsigned long long call) {
    __shared__ unsigned long long acc[16];
    __shared__ int failed;
    if (threadIdx.x < 16) acc[threadIdx.x] = 0ull;
    if (threadIdx.x == 0) failed = 0;
    __syncthreads();
    unsigned long long sum = 0;
    for (int i = threadIdx.x; i < kStatReplicas * 16; i += blockDim.x) {
        const unsigned long long v = stats[i];
        if (v) { sum += v; if (clear) stats[i] = 0ull; }
    }
    if (sum) atomicAdd(&acc[threadIdx.x & 15], sum);
    __syncthreads();
    const size_t half = (size_t)(call & 1ull) * kPeerMax * 16;
    if ((int)threadIdx.x < world) {
        volatile unsigned long long* row = peers.buf[threadIdx.x] + half + (size_t)rank * 16;
#pragma unroll
        for (int k = 0; k < ASTRO_N_STATS; k++) row[k] = acc[k];
        __threadfence_system();
        row[15] = call;
    }
    if ((int)threadIdx.x < world) {
        const volatile unsigned long long* row = peers.buf[rank] + half + (size_t)threadIdx.x * 16;
        const long long t0 = clock64();
        while (row[15] != call) {
            if (clock64() - t0 > (4ll << 30)) { failed = 1; break; }
        }
        __threadfence_system();
    }
    __syncthreads();
    if (threadIdx.x < ASTRO_N_STATS) {
        unsigned long long total = 0;
        const volatile unsigned long long* mine = peers.buf[rank] + half;
        for (int r = 0; r < world; r++) total += mine[(size_t)r * 16 + threadIdx.x];
        out[threadIdx.x] = failed ? -1ll : (long long)total;
    }
}

// First list item of game `gl` (0..31) of a tile: the bullet counts of the tile's lower games,
// summed by the warp (finished games own no items).  meta_tile = the tile's 32 meta words.
__device__ __forceinline__ unsigned tile_list_offset(const uint32_t* __restrict__ meta_tile, int gl, int lane) {
    const uint32_t m = meta_tile[lane];
    const unsigned nb = (lane < gl && !ASTRO_META_FINISHED(m)) ? ASTRO_META_NB(m) : 0u;
    return __reduce_add_sync(0xffffffffu, nb);
}
__device__ __forceinline__ unsigned warp_exclusive_sum(unsigned v, int lane) {
    unsigned incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        unsigned u = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += u;
    }
    return incl - v;
}

// ------------------------------------------------------------------------------------------
// tick_kernel<R, S, STATS>: one thread = one game, one launch = one core.step for all games.
//
// Phase order follows core.py:215-303: accelerations (old state) -> collisions (old state) ->
// collision terminal -> timeout terminal -> bullet despawn -> spawn -> integrate/cull.
// Bullets: a warp is a tile; each thread walks its game's run of the tile's list, compacting the
// survivors front to back inside that run (reference order: old survivors, then ship 0's and ship
// 1's newborn), then the runs move — dense again — to the tile's list in the other buffer.  When a
// game ends it owns no bullets (nb = 0); ships/planets keep the pre-step state unless AUTO_RESET
// re-initialises the slot from the pool.
// ------------------------------------------------------------------------------------------
template <typename R, int S, bool STATS, int PL>
__global__ void __launch_bounds__(kTickThreads) tick_kernel(const __grid_constant__ TickParams p) {
    using B4 = Body4<R>;
    __shared__ unsigned s_stats[ASTRO_N_STATS];
    if (STATS) {
        if (threadIdx.x < ASTRO_N_STATS) s_stats[threadIdx.x] = 0u;
        __syncthreads();
    }
    const int g = blockIdx.x * kTickThreads + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const bool in_range = g < p.n_games;  // whole warps: n_games % 32 == 0
    const Consts& c = p.c;

    uint32_t ev = 0;
    int np = 0, nb = 0, m_out = 0;
    bool active = false;
    int spawned = 0;

    if (in_range) {   // (warp-uniform)
        const size_t tile = (size_t)(g >> 5);
        B4* ships = reinterpret_cast<B4*>(p.ships) + tile * (S * 32) + lane;
        R* ship_b = reinterpret_cast<R*>(p.ship_b) + tile * (S * 32) + lane;
        B4* planets = reinterpret_cast<B4*>(p.planets) + tile * (PL * 32) + lane;

        const uint32_t meta = p.meta[g];
        // ships are loaded before meta is inspected: independent loads, one DRAM round trip
        B4 sh[S];
        R sb[S];
#pragma unroll
        for (int s = 0; s < S; s++) {
            sh[s] = ships[s * 32];
            sb[s] = ship_b[s * 32];
        }
        active = !ASTRO_META_FINISHED(meta);
        nb = active ? (int)ASTRO_META_NB(meta) : 0;
        np = active ? (int)meta_np<PL>(meta) : 0;
        const uint32_t tick = meta_tick<PL>(meta);
        // this game's run of the tile's list (read buffer); survivors are compacted inside it
        B4* const bullets = reinterpret_cast<B4*>(p.bullets_in) + tile * (size_t)(32 * p.K) + warp_exclusive_sum((unsigned)nb, lane);
        int m = 0, n_born = 0;
        B4 born[2];
        born[0] = born[1] = B4();
        float rw[S];
#pragma unroll
        for (int s = 0; s < S; s++) rw[s] = 0.0f;

        if (!active) {
            ev = ASTRO_EV_SKIPPED;
        } else {
            B4 pl[PL];
#pragma unroll
            for (int j = 0; j < PL; j++)
                if (j < np) pl[j] = planets[j * 32];

            // first group of bullets in flight while the ship/planet maths runs
            B4 bq[4];
#pragma unroll
            for (int u = 0; u < 4; u++)
                if (u < nb) bq[u] = bullets[u];

            // ---- controls (core.py:220-227,234-239)
            int ctl[S];
            bool bad_ctl = false;
            if (p.actions) {
                if (S == 2 && (p.flags & ASTRO_TICK_PACKED_CONTROLS)) {   // one byte per game: ship 0 bits 0-2, ship 1 bits 3-7
                    const uint8_t a = p.actions[g];
                    ctl[0] = a & 7;
                    ctl[S - 1] = a >> 3;
                } else if (S == 2) {
                    uint16_t a = reinterpret_cast<const uint16_t*>(p.actions)[g];
                    ctl[0] = a & 0xff;
                    ctl[S - 1] = a >> 8;
                } else {
                    ctl[0] = p.actions[g];
                }
#pragma unroll
                for (int s = 0; s < S; s++)   // codes above 5: outside the reference's table (core.py:220-227)
                    if (ctl[s] > 5) { ctl[s] = 2; bad_ctl = true; }
            } else {
                uint32_t h0 = game_key(p.seed, p.first_game + (uint32_t)g);
#pragma unroll
                for (int s = 0; s < S; s++) ctl[s] = action_from_key(h0, p.step, (uint32_t)s);
            }

            // ---- accelerations and ship collisions on the OLD state
            // (raw: the game holds core.create's float32 arrays — the reference's first-tick arithmetic, see the header)
            const bool raw = std::is_same<R, double>::value && nb == 0 &&
                             ((p.flags & ASTRO_TICK_ALL_CREATE_DTYPES) || ((p.flags & ASTRO_TICK_CREATE_DTYPES) && tick == 0));
            float dir0[S], dir1[S];
            R a0[S], a1[S];
            bool hit[S];
#pragma unroll
            for (int s = 0; s < S; s++) {
                np_sincos_f32((float)sb[s], dir0[s], dir1[s]);
                R g0 = 0, g1 = 0;
                bool h = false;
                if (raw) {
                    float f0 = 0.f, f1 = 0.f;
#pragma unroll
                    for (int j = 0; j < PL; j++) {
                        if (j < np) {
                            float t0, t1;
                            grav_term_np32((float)pl[j].x, (float)pl[j].y, (float)sh[s].x, (float)sh[s].y, c.gm_f, t0, t1);
                            if (j == 0) { f0 = t0; f1 = t1; } else { f0 = __fadd_rn(f0, t0); f1 = __fadd_rn(f1, t1); }
                            h |= collide_np32((float)sh[s].x, (float)sh[s].y, (float)pl[j].x, (float)pl[j].y, c.r2_sp);
                        }
                    }
                    g0 = (R)f0; g1 = (R)f1;
                } else {
#pragma unroll
                for (int j = 0; j < PL; j++) {
                    if (j < np) {
                        R t0, t1;
                        grav_term(pl[j].x, pl[j].y, sh[s].x, sh[s].y, c, t0, t1);
                        if (j == 0) { g0 = t0; g1 = t1; } else { g0 = add_rn(g0, t0); g1 = add_rn(g1, t1); }
                        h |= collide(sh[s].x, sh[s].y, pl[j].x, pl[j].y, c.r2_sp, c.r2f_sp);
                    }
                }
                }
                R th = mul_rn(Pick<R>::thrust(c), (R)(ctl[s] & 1));
                a0[s] = add_rn(mul_rn(th, (R)dir0[s]), g0);
                a1[s] = add_rn(mul_rn(th, (R)dir1[s]), g1);
                hit[s] = h;
            }
            if (S == 2) {
                bool h = raw ? collide_np32((float)sh[0].x, (float)sh[0].y, (float)sh[S - 1].x, (float)sh[S - 1].y, c.r2_ss)
                             : collide(sh[0].x, sh[0].y, sh[S - 1].x, sh[S - 1].y, c.r2_ss, c.r2f_ss);
                hit[0] |= h;
                hit[S - 1] |= h;
            }

            // ---- bullets: hit test on old positions, integrate, cull, compact inside the run
            for (int j0 = 0; j0 < nb; j0 += 4) {
                B4 cur[4];
#pragma unroll
                for (int u = 0; u < 4; u++) cur[u] = bq[u];
#pragma unroll
                for (int u = 0; u < 4; u++)
                    if (j0 + 4 + u < nb) bq[u] = bullets[j0 + 4 + u];
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    if (j0 + u < nb) {
                        B4 b = cur[u];
                        bool gone = false;
#pragma unroll
                        for (int s = 0; s < S; s++) {
                            bool h = collide(sh[s].x, sh[s].y, b.x, b.y, c.r2_sb, c.r2f_sb);
                            hit[s] |= h;
                            gone |= h;
                        }
#pragma unroll
                        for (int k = 0; k < PL; k++)
                            if (k < np) gone |= collide(pl[k].x, pl[k].y, b.x, b.y, c.r2_pb, c.r2f_pb);
                        bool keep = advance_bullet(b, c);
                        if (keep && !gone) {
                            bullets[m] = b;
                            m++;
                        }
                    }
                }
            }

            bool any_hit = hit[0];
            if (S == 2) any_hit |= hit[S - 1];
            const bool timeout = tick >= (uint32_t)p.timeout_tick;

            if (any_hit) {  // core.py:253-255
                ev = (hit[0] ? ASTRO_EV_HIT0 : 0);
                if (S == 2) ev |= (hit[S - 1] ? ASTRO_EV_HIT1 : 0);
#pragma unroll
                for (int s = 0; s < S; s++) rw[s] = hit[s] ? -1.0f : 1.0f;
                m = 0;
            } else if (timeout) {  // core.py:257-260
                ev = ASTRO_EV_TIMEOUT;
#pragma unroll
                for (int s = 0; s < S; s++) rw[s] = c.reward_timeout;
                m = 0;
            } else {
                // ---- spawn from the OLD ship state (core.py:267-280); float32 products
                const bool fire = tick < (uint32_t)p.n_sched_ticks && ((p.fire_bits[tick >> 5] >> (tick & 31)) & 1u);
                if (fire) {
                    ev |= ASTRO_EV_FIRED;
#pragma unroll
                    for (int s = 0; s < S; s++) {
                        Body4<double> nbl;
                        bool keep;
                        if (raw) {   // float32 ship state + float32 products, advanced in float32 (weak scalars)
                            const float x0 = __fadd_rn((float)sh[s].x, __fmul_rn(c.off_f, dir0[s]));
                            const float x1 = __fadd_rn((float)sh[s].y, __fmul_rn(c.off_f, dir1[s]));
                            const float w0 = __fadd_rn(__fadd_rn((float)sh[s].dx, __fmul_rn(c.spd_f, dir0[s])), (float)c.zero_dt);
                            const float w1 = __fadd_rn(__fadd_rn((float)sh[s].dy, __fmul_rn(c.spd_f, dir1[s])), (float)c.zero_dt);
                            nbl.x = (double)__fadd_rn(x0, __fmul_rn(c.dt_f, w0));
                            nbl.y = (double)__fadd_rn(x1, __fmul_rn(c.dt_f, w1));
                            nbl.dx = (double)w0;
                            nbl.dy = (double)w1;
                            keep = in_arena(nbl.x, nbl.y);
                        } else {
                        nbl.x = __dadd_rn((double)sh[s].x, (double)__fmul_rn(c.off_f, dir0[s]));
                        nbl.y = __dadd_rn((double)sh[s].y, (double)__fmul_rn(c.off_f, dir1[s]));
                        nbl.dx = __dadd_rn((double)sh[s].dx, (double)__fmul_rn(c.spd_f, dir0[s]));
                        nbl.dy = __dadd_rn((double)sh[s].dy, (double)__fmul_rn(c.spd_f, dir1[s]));
                        keep = advance_bullet(nbl, c);
                        }
                        if (keep) {
                            if (m + n_born < p.K) {
                                B4 o;
                                o.x = (R)nbl.x; o.y = (R)nbl.y; o.dx = (R)nbl.dx; o.dy = (R)nbl.dy;
                                if (n_born == 0) born[0] = o; else born[1] = o;
                                n_born++;
                            } else {
                                ev |= ASTRO_EV_OVERFLOW;
                            }
                        }
                    }
                    spawned = S;
                }
                // ---- planets (core.py:289-294): gravity of every planet on every planet, the
                // clamped self term included (f * 0 = 0)
                R q0[PL], q1[PL];
#pragma unroll
                for (int i = 0; i < PL; i++) {
                    q0[i] = 0; q1[i] = 0;
                    if (i < np) {
#pragma unroll
                        for (int j = 0; j < PL; j++) {
                            if (j < np) {
                                R t0, t1;
                                grav_term(pl[j].x, pl[j].y, pl[i].x, pl[i].y, c, t0, t1);
                                if (j == 0) { q0[i] = t0; q1[i] = t1; } else { q0[i] = add_rn(q0[i], t0); q1[i] = add_rn(q1[i], t1); }
                            }
                        }
                    }
                }
                if (raw) {   // float32 field, float32 a * dt (a float32 array times the weak scalar dt), then float64
                    float f0[PL], f1[PL];
#pragma unroll
                    for (int i = 0; i < PL; i++) {
                        f0[i] = f1[i] = 0.f;
                        if (i < np) {
#pragma unroll
                            for (int j = 0; j < PL; j++) {
                                if (j < np) {
                                    float t0, t1;
                                    grav_term_np32((float)pl[j].x, (float)pl[j].y, (float)pl[i].x, (float)pl[i].y, c.gm_f, t0, t1);
                                    if (j == 0) { f0[i] = t0; f1[i] = t1; } else { f0[i] = __fadd_rn(f0[i], t0); f1[i] = __fadd_rn(f1[i], t1); }
                                }
                            }
                        }
                    }
#pragma unroll
                    for (int i = 0; i < PL; i++) {
                        if (i < np) {
                            const double v0 = __dadd_rn((double)pl[i].dx, (double)__fmul_rn(f0[i], c.dt_f));
                            const double v1 = __dadd_rn((double)pl[i].dy, (double)__fmul_rn(f1[i], c.dt_f));
                            pl[i].x = (R)wrap_unit_f64(__dadd_rn((double)pl[i].x, __dmul_rn(c.dt, v0)));
                            pl[i].y = (R)wrap_unit_f64(__dadd_rn((double)pl[i].y, __dmul_rn(c.dt, v1)));
                            pl[i].dx = (R)v0; pl[i].dy = (R)v1;
                            planets[i * 32] = pl[i];
                        }
                    }
                } else {
#pragma unroll
                for (int i = 0; i < PL; i++) {
                    if (i < np) {
                        advance_body(pl[i], q0[i], q1[i], c);
                        planets[i * 32] = pl[i];
                    }
                }
                }
                // ---- ships (core.py:283-288)
#pragma unroll
                for (int s = 0; s < S; s++) {
                    advance_body(sh[s], a0[s], a1[s], c);
                    ships[s * 32] = sh[s];
                    R db = mul_rn(Pick<R>::db_unit(c), (R)((ctl[s] >> 1) - 1));
                    ship_b[s * 32] = add_rn(sb[s], db);
                }
                m_out = m + n_born;
                p.meta[g] = meta_pack<PL>(m_out, np, 0, tick + 1);
            }

            if (bad_ctl) ev |= ASTRO_EV_BAD_CONTROL;
            if (ev & ASTRO_EV_DONE_MASK) {
                if ((p.flags & ASTRO_TICK_AUTO_RESET) && p.pool_size > 0) {
                    recreate_from_pool<R, S, PL>(p, g, p.step + (p.step_base ? *p.step_base : 0u) + 1u, ships, ship_b, planets);
                } else {
                    p.meta[g] = meta_pack<PL>(0, np, 1, tick);
                }
            }
        }
        // ---- the new list of the tile: every game's survivors and newborn, dense, other buffer
        __syncwarp();
        B4* const out = reinterpret_cast<B4*>(p.bullets_out) + tile * (size_t)(32 * p.K) + warp_exclusive_sum((unsigned)m_out, lane);
        for (int k = 0; k < m; k++) out[k] = bullets[k];
        if (n_born > 0) out[m] = born[0];
        if (n_born > 1) out[m + 1] = born[1];

        if (p.reward) {
            if (S == 2) reinterpret_cast<float2*>(p.reward)[g] = make_float2(rw[0], rw[S - 1]);
            else p.reward[g] = rw[0];
        }
        if (p.events) {
            if (p.flags & ASTRO_TICK_EVENT_PLANES) {   // three bit planes u32 [3][n_tiles]: ended / ship 0 hit / ship 1 hit
                const unsigned b_done = __ballot_sync(0xffffffffu, (ev & ASTRO_EV_DONE_MASK) != 0);
                const unsigned b_h0 = __ballot_sync(0xffffffffu, (ev & ASTRO_EV_HIT0) != 0), b_h1 = __ballot_sync(0xffffffffu, (ev & ASTRO_EV_HIT1) != 0);
                if (lane < 3)
                    reinterpret_cast<uint32_t*>(p.events)[(size_t)lane * (p.n_games >> 5) + (g >> 5)] = lane == 0 ? b_done : (lane == 1 ? b_h0 : b_h1);
            } else {
                p.events[g] = (uint8_t)ev;
            }
        }
        if (p.done) p.done[g] = (uint8_t)((ev & (ASTRO_EV_DONE_MASK | ASTRO_EV_SKIPPED)) ? 1 : 0);
    }

    if (STATS) {
        warp_stats(s_stats, lane, S, ev, active, spawned, np, nb, m_out);
        __syncthreads();
        if (threadIdx.x < ASTRO_N_STATS && s_stats[threadIdx.x])
            atomicAdd(&p.stats[threadIdx.x], (unsigned long long)s_stats[threadIdx.x]);
    }
}


#include "tick_f32.cuh"

// ------------------------------------------------------------------------------------------
// reset_kernel: stand-alone form of AUTO_RESET — finished games are re-created from the pool.
// ------------------------------------------------------------------------------------------
template <typename R, int S, int PL>
__global__ void __launch_bounds__(kTickThreads) reset_kernel(const __grid_constant__ TickParams p) {
    using B4 = Body4<R>;
    const int g = blockIdx.x * kTickThreads + threadIdx.x;
    if (g >= p.n_games) return;
    const uint32_t meta = p.meta[g];
    if (!ASTRO_META_FINISHED(meta)) return;
    const size_t tile = (size_t)(g >> 5);
    const int lane = g & 31;
    B4* ships = reinterpret_cast<B4*>(p.ships) + tile * (S * 32) + lane;
    R* ship_b = reinterpret_cast<R*>(p.ship_b) + tile * (S * 32) + lane;
    B4* planets = reinterpret_cast<B4*>(p.planets) + tile * (PL * 32) + lane;
    recreate_from_pool<R, S, PL>(p, g, p.step, ships, ship_b, planets);
}

// ------------------------------------------------------------------------------------------
// observe_kernel<R, S, BOTH>: one warp = one game.  The warp builds the game's feature rows
// (rl.py:43-72: [flag | every ship's x,y,dx,dy,norm_angle(b)/pi | object x,y,dx,dy]) in shared
// memory — lane r builds row r, for ship 0's perspective and, with BOTH, for ship 1's
// (core.roll_ships: the ship column groups exchanged); rows beyond P+B are the -1 padding of
// to_batch (rl.py:91-98).  The finished block (both perspectives are adjacent in the output) then
// leaves as ONE bulk copy through the TMA engine (cp.async.bulk shared -> global): the kernel is a
// pure stream of writes, and this keeps the LSU out of it.
// ------------------------------------------------------------------------------------------
// per-warp staging: P perspectives x n_rows*D feature floats + 5*S ship features, padded to a 16-byte multiple
__host__ __device__ inline size_t observe_warp_floats(int n_rows, int D, int S, int P) {
    return (((size_t)P * n_rows * D + 5 * S) + 3) & ~(size_t)3;
}

template <typename R, int S, bool BOTH, int PL>
__global__ void __launch_bounds__(kObserveWarps * 32)
observe_kernel(const void* __restrict__ ships_, const void* __restrict__ ship_b_, const void* __restrict__ planets_,
               const void* __restrict__ bullets_, const uint32_t* __restrict__ meta_, float* __restrict__ obs,
               int n_games, int K, int n_rows, uint32_t ring_ticks, uint32_t step, const uint32_t* __restrict__ step_base) {
    using B4 = Body4<R>;
    constexpr int D = 1 + 5 * S + 4;
    constexpr int P = (BOTH && S == 2) ? 2 : 1;
    extern __shared__ float4 s_all4[];
    float* s_all = reinterpret_cast<float*>(s_all4);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.x * kObserveWarps + warp;
    if (g >= n_games) return;
    const int per = n_rows * D;  // % 4 == 0 (checked on the host)
    float* rows = s_all + (size_t)warp * observe_warp_floats(n_rows, D, S, P);
    float* sf = rows + (size_t)P * per;  // ship features, ship 0 first

    const size_t tile = (size_t)(g >> 5);
    const int gl = g & 31;
    const uint32_t meta = meta_[g];
    const bool fin = ASTRO_META_FINISHED(meta);
    const int np = fin ? 0 : (int)meta_np<PL>(meta);
    const int nb = fin ? 0 : (int)ASTRO_META_NB(meta);

    if (lane < S && !fin) {
        B4 s = reinterpret_cast<const B4*>(ships_)[tile * (S * 32) + lane * 32 + gl];
        R b = reinterpret_cast<const R*>(ship_b_)[tile * (S * 32) + lane * 32 + gl];
        sf[5 * lane + 0] = (float)s.x;
        sf[5 * lane + 1] = (float)s.y;
        sf[5 * lane + 2] = (float)s.dx;
        sf[5 * lane + 3] = (float)s.dy;
        sf[5 * lane + 4] = norm_angle_over_pi((double)b);
    }
    __syncwarp();
    const B4* planets = reinterpret_cast<const B4*>(planets_) + tile * (PL * 32) + gl;
    // the game's run of its tile's bullet list
    const B4* bullets = reinterpret_cast<const B4*>(bullets_) + tile * (size_t)(32 * K) + tile_list_offset(meta_ + tile * 32, gl, lane);
    for (int r = lane; r < n_rows; r += 32) {
        float* row = rows + r * D;
        if (r < np + nb) {
            B4 o = r < np ? planets[r * 32] : bullets[r - np];
            const float flag = r < np ? 0.0f : 1.0f;
#pragma unroll
            for (int q = 0; q < P; q++) {
                float* dst = row + q * per;
                dst[0] = flag;
#pragma unroll
                for (int s = 0; s < S; s++)
#pragma unroll
                    for (int k = 0; k < 5; k++) dst[1 + 5 * s + k] = sf[5 * ((s + q) % S) + k];
                dst[1 + 5 * S + 0] = (float)o.x;
                dst[1 + 5 * S + 1] = (float)o.y;
                dst[1 + 5 * S + 2] = (float)o.dx;
                dst[1 + 5 * S + 3] = (float)o.dy;
            }
        } else {
#pragma unroll
            for (int q = 0; q < P; q++)
#pragma unroll
                for (int k = 0; k < D; k++) row[q * per + k] = -1.0f;
        }
    }
    // hand the block to the TMA engine: generic-proxy writes -> async proxy, then one bulk store
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
    if (lane == 0) {
        float* out = obs + (size_t)g * P * per;
        // astro_rollout_device_record: obs is a ring of ring_ticks blocks, the block of stream step s in row s % ring_ticks
        // (inside a captured chunk of the bot loop the stream step is *step_base + step)
        if (ring_ticks) out += (size_t)((step + (step_base ? *step_base : 0u)) % ring_ticks) * n_games * P * per;
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(out),
                     "r"((unsigned)__cvta_generic_to_shared(rows)), "r"((unsigned)(P * per * 4))
                     : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // shared memory must outlive the read
    }
}

// ------------------------------------------------------------------------------------------
// script_kernel<R, S>: script.ScriptBot.__call__ (script.py:67-91) with _danger (:41-65) and
// _fly_to (:30-39) for every ship of every game — thread = game, both perspectives
// (core.roll_ships, core.py:306-327: ship `me` sees itself as ship 0, the other as ship 1).
// float64 throughout, the reference's operations in the reference's order (the bot reads a
// float64 State; float32 state converts exactly).  sqrt, division and fmod are IEEE-exact;
// atan2 is the device libm (<= 2 ulp) against glibc's (< 1 ulp), so a decision could differ from
// the reference only when an angle sits within an ulp of its threshold.
// Quirk kept: inside _danger the parameter `b` (my bearing) is shadowed by the quadratic
// coefficient (script.py:54), so `rotation` uses that coefficient.
// ------------------------------------------------------------------------------------------
// thread = one ship of one game (its own perspective).  The cheap part of _danger — two square
// roots, two divisions, the discriminant — runs for every planet without divergence and leaves a
// bit mask of the planets on a collision course; only those go through the atan2 / norm_angle
// test, in planet order (the first dangerous planet decides, script.py:69-76), so the warp executes
// that code as often as its worst lane needs it (usually once), from one copy of it.
#ifndef ASTRO_SCRIPT_MIN_BLOCKS
#define ASTRO_SCRIPT_MIN_BLOCKS 6   /* 80 registers: 41.1 -> 32.9 us per 262,144 games (the kernel waits on its loads: more warps) */
#endif
#ifndef ASTRO_SCRIPT_MIN_BLOCKS_WIDE
#define ASTRO_SCRIPT_MIN_BLOCKS_WIDE 2   /* 8 planet slots: five float64 candidates per planet stay in registers */
#endif
template <typename R, int S, int PL>
__global__ void __launch_bounds__(128, PL > ASTRO_MAX_PLANETS ? ASTRO_SCRIPT_MIN_BLOCKS_WIDE : ASTRO_SCRIPT_MIN_BLOCKS) script_kernel(const void* __restrict__ ships_, const void* __restrict__ ship_b_,
                                                     const void* __restrict__ planets_, const uint32_t* __restrict__ meta_,
                                                     uint8_t* __restrict__ actions, const __grid_constant__ ScriptParams q) {
    using B4 = Body4<R>;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int g = idx / S, me = idx % S;
    if (g >= q.n_games) return;
    const size_t tile = (size_t)(g >> 5);
    const int lane = g & 31;
    const uint32_t meta = meta_[g];
    if (ASTRO_META_FINISHED(meta)) {
        actions[idx] = 2;
        return;
    }
    const int np = (int)meta_np<PL>(meta);
    const B4 mv = reinterpret_cast<const B4*>(ships_)[tile * (S * 32) + me * 32 + lane];
    const R mb = reinterpret_cast<const R*>(ship_b_)[tile * (S * 32) + me * 32 + lane];
    B4 pl[PL];
#pragma unroll
    for (int j = 0; j < PL; j++) {
        pl[j] = B4();
        if (j < np) pl[j] = reinterpret_cast<const B4*>(planets_)[tile * (PL * 32) + j * 32 + lane];
    }
    B4 ev = B4();
    if (S == 2 && !q.solo) ev = reinterpret_cast<const B4*>(ships_)[tile * (S * 32) + ((me + 1) % S) * 32 + lane];
    actions[idx] = (uint8_t)script_decide<R, S, PL>(mv, mb, ev, pl, np, q);
}

// ------------------------------------------------------------------------------------------
// create_kernel<R, S>: core.create (core.py:86-135) for M seeds at once — thread = one new game.
//
// The reference draws from numpy's legacy RandomState(seed): MT19937 seeded by init_genrand, 32-bit
// words tempered in order.  A game needs fewer than kCreateWords words, and the first generation's
// word k depends only on the seeded state at k, k + 1 and k + 397, so the thread keeps those two
// short runs of the 624-word state while it walks the seeding recurrence once.
//   randint(lo, hi)   masked rejection on one word per try; no word when hi - lo == 1
//   rand()            ((w0 >> 5) * 2^26 + (w1 >> 6)) / 2^53
//   choice((-1, 1))   randint(0, 2)
// Arithmetic follows numpy >= 2 promotion (SURVEY 8c): ship positions / bearings and planet
// positions are float32 products, util.direction is the float32 sin/cos kernel, planet
// velocities are float64 (np.sqrt returns a float64 scalar).  Output is game-major, the layout of
// AstroResetPool: ships [M][S][5], planets [M][4][4] (dead slots zero), np [M].
// ------------------------------------------------------------------------------------------
constexpr int kCreateWords = 40;

struct CreateParams {
    double inner, outer, orbit, gravity, planet_mass;
    int32_t max_planets, solo, m, pad;
};

struct Mt19937Head {
    uint32_t lo[kCreateWords + 1], hi[kCreateWords];
    int k;
    __device__ void seed(uint32_t x) {
        // init_genrand: 436 dependent steps of three instructions (shift, xor, multiply-add).  Three loops, so that the
        // long middle stretch carries no store and no test (one loop with both predicates compiled to ~12 instructions per
        // step: 32 M warp-instructions per refill of 200,000 games, 57 us; now ~9 M).
        lo[0] = x;
#pragma unroll
        for (int j = 1; j <= kCreateWords; j++) {
            x = 1812433253u * (x ^ (x >> 30)) + (uint32_t)j;
            lo[j] = x;
        }
#pragma unroll 4
        for (int j = kCreateWords + 1; j < 397; j++) x = 1812433253u * (x ^ (x >> 30)) + (uint32_t)j;
#pragma unroll
        for (int j = 397; j < 397 + kCreateWords; j++) {
            x = 1812433253u * (x ^ (x >> 30)) + (uint32_t)j;
            hi[j - 397] = x;
        }
        k = 0;
    }
    __device__ uint32_t word() {
        const int i = k < kCreateWords ? k : kCreateWords - 1;  // (never reached: see the rejection bound below)
        k++;
        const uint32_t y = (lo[i] & 0x80000000u) | (lo[i + 1] & 0x7fffffffu);
        uint32_t v = hi[i] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
        v ^= v >> 11;
        v ^= (v << 7) & 0x9d2c5680u;
        v ^= (v << 15) & 0xefc60000u;
        v ^= v >> 18;
        return v;
    }
    __device__ double rand() {
        const uint32_t a = word() >> 5, b = word() >> 6;
        return __ddiv_rn(__dadd_rn(__dmul_rn((double)a, 67108864.0), (double)b), 9007199254740992.0);
    }
    __device__ uint32_t bounded(uint32_t rng) {  // value in [0, rng]
        if (rng == 0) return 0;
        uint32_t mask = rng;
        mask |= mask >> 1; mask |= mask >> 2; mask |= mask >> 4; mask |= mask >> 8; mask |= mask >> 16;
        uint32_t v;
        do v = word() & mask; while (v > rng && k < kCreateWords - 16);
        return v > rng ? rng : v;  // (a 2^-24 event cut short so that the word budget holds)
    }
};

// One created game in registers: float32 ship positions / bearings and planet positions, float64 planet velocities
// (the reference's dtypes under numpy >= 2).
template <int PL>
struct CreatedGameT {
    float sx[2][2], sb[2];
    float px[PL][2];
    double pv[PL][2];
    int n;
};
using CreatedGame = CreatedGameT<ASTRO_MAX_PLANETS>;
template <int S, int PL = ASTRO_MAX_PLANETS>
__device__ __forceinline__ void create_game(uint32_t seed, const CreateParams& q, CreatedGameT<PL>& o) {
    const double TWO_PI = 6.283185307179586, PI = 3.141592653589793;
    Mt19937Head mt;
    mt.seed(seed);
    const int n = 1 + (int)mt.bounded((uint32_t)(q.max_planets - 1));
    // 1. ships
    const float r0 = (float)mt.rand(), r1 = (float)mt.rand();
    const float d0 = __fsub_rn(r0, 0.5f), d1 = __fsub_rn(r1, 0.5f);
    const float outer_f = (float)q.outer, inner_f = (float)q.inner;
    const float o0 = __fmul_rn(outer_f, d0 > 0.f ? 1.f : (d0 < 0.f ? -1.f : 0.f));
    const float o1 = __fmul_rn(outer_f, d1 > 0.f ? 1.f : (d1 < 0.f ? -1.f : 0.f));
    float sn, cs;
    np_sincos_f32((float)__dmul_rn(TWO_PI, mt.rand()), sn, cs);
    const float i0 = __fmul_rn(inner_f, sn), i1 = __fmul_rn(inner_f, cs);
    if (n == 1) {
        o.sx[0][0] = o0; o.sx[0][1] = o1; o.sx[1][0] = -o0; o.sx[1][1] = -o1;
    } else {
        const bool first = mt.rand() < 0.5;
        if (S == 1) {
            o.sx[0][0] = first ? o0 : i0; o.sx[0][1] = first ? o1 : i1;
            o.sx[1][0] = o.sx[1][1] = 0.f;
        } else {
            o.sx[0][0] = first ? o0 : i0; o.sx[0][1] = first ? o1 : i1;
            o.sx[1][0] = first ? i0 : o0; o.sx[1][1] = first ? i1 : o1;
        }
    }
    const float two_pi_f = (float)TWO_PI;
    o.sb[1] = 0.f;
#pragma unroll
    for (int s = 0; s < S; s++) o.sb[s] = __fmul_rn(two_pi_f, (float)mt.rand());
    // 2. planets
#pragma unroll
    for (int j = 0; j < PL; j++) { o.px[j][0] = o.px[j][1] = 0.f; o.pv[j][0] = o.pv[j][1] = 0.0; }
    if (n > 1) {
        const double base = __dmul_rn(TWO_PI, mt.rand());
        const double step = __ddiv_rn(TWO_PI, (double)n);                    // np.linspace(0, 2 pi, n, endpoint=False)
        const double spin = mt.bounded(1u) ? 1.0 : -1.0;                     // random.choice((-1, 1))
        const double quarter = __ddiv_rn(__dmul_rn(spin, PI), 2.0);
        const double speed = sqrt(__ddiv_rn(__dmul_rn(__dmul_rn(q.gravity, q.planet_mass), (double)(n - 1)), 2.0));
        const float orbit_f = (float)q.orbit;
#pragma unroll
        for (int j = 0; j < PL; j++) {
            if (j < n) {
                const double phase = __dadd_rn(base, __dadd_rn(__dmul_rn((double)j, step), 0.0));
                float s0, c0, s1, c1;
                np_sincos_f32((float)phase, s0, c0);
                np_sincos_f32((float)__dadd_rn(phase, quarter), s1, c1);
                o.px[j][0] = __fmul_rn(orbit_f, s0);
                o.px[j][1] = __fmul_rn(orbit_f, c0);
                o.pv[j][0] = __dmul_rn(speed, (double)s1);
                o.pv[j][1] = __dmul_rn(speed, (double)c1);
            }
        }
    }
    o.n = n;
}

template <typename R, int S, int PL>
__global__ void __launch_bounds__(64) create_kernel(const uint32_t* __restrict__ seeds, R* __restrict__ ships,
                                                    R* __restrict__ planets, int32_t* __restrict__ np_out,
                                                    const __grid_constant__ CreateParams q) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= q.m) return;
    CreatedGameT<PL> o;
    create_game<S, PL>(seeds[i], q, o);
#pragma unroll
    for (int s = 0; s < S; s++) {
        R* d = ships + ((size_t)i * S + s) * 5;
        d[0] = (R)o.sx[s][0]; d[1] = (R)o.sx[s][1]; d[2] = (R)0; d[3] = (R)0;
        d[4] = (R)o.sb[s];
    }
    R* pl = planets + (size_t)i * (PL * 4);
#pragma unroll
    for (int j = 0; j < PL; j++) {
        pl[4 * j + 0] = (R)o.px[j][0];
        pl[4 * j + 1] = (R)o.px[j][1];
        pl[4 * j + 2] = (R)o.pv[j][0];
        pl[4 * j + 3] = (R)o.pv[j][1];
    }
    np_out[i] = o.n;
}

// ------------------------------------------------------------------------------------------
// Fresh games without a pool (core.generate_configs + core.create, core.py:77-135, for every re-creation): each tile
// owns `quota` pre-created games (128-byte records, the layout of pack_pool_kernel + word 11 = position in the
// generate_configs stream, word 12 = seed).  A game that ends takes the tile's next unused record — a warp-local
// counter, no atomics, no dependent address — and between launches the records that were used are re-created from the
// NEXT positions of the seed stream (host MT19937, uploaded ahead; positions handed out by a prefix sum in tile order,
// so a rollout is reproducible): every re-creation consumes a stream position exactly once.
//   refill_scan / refill_tasks   prefix sum of the tiles' used counts -> task list (record index), stream cursor
//   refill_create_kernel  thread = task: create_game(seed at cursor + task) -> record
//   fresh_fill_kernel     thread = game: (re)start every game of the batch from consecutive stream positions
// ------------------------------------------------------------------------------------------
struct FreshParams {
    float4* ring;                  // [n_tiles][quota][8]
    uint32_t* tile_used;           // [n_tiles] records of the tile consumed since the last refill
    uint32_t* tasks;               // [n_tiles * quota] record indices to re-create
    unsigned long long* cursor;    // [0] stream positions handed out so far, [1] refills completed, [2] tasks of the last plan
    const uint32_t* seeds;         // ring of uploaded seeds: position p at p & seed_mask
    uint32_t seed_mask;
    int32_t n_tiles, quota, n_games;
};

template <int S>
__device__ __forceinline__ void write_record(float4* rec, const CreatedGame& o, uint32_t pos, uint32_t seed) {
    float w[32];
#pragma unroll
    for (int i = 0; i < 32; i++) w[i] = 0.f;
#pragma unroll
    for (int s = 0; s < S; s++) {
        w[5 * s + 0] = o.sx[s][0]; w[5 * s + 1] = o.sx[s][1]; w[5 * s + 4] = o.sb[s];
    }
    w[10] = __int_as_float(o.n);
    w[11] = __uint_as_float(pos);
    w[12] = __uint_as_float(seed);
#pragma unroll
    for (int j = 0; j < ASTRO_MAX_PLANETS; j++) {
        w[16 + 4 * j + 0] = o.px[j][0]; w[16 + 4 * j + 1] = o.px[j][1];
        w[16 + 4 * j + 2] = (float)o.pv[j][0]; w[16 + 4 * j + 3] = (float)o.pv[j][1];
    }
#pragma unroll
    for (int i = 0; i < 8; i++) rec[i] = make_float4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
}

// Plan, in two small kernels (deterministic: task numbers follow the tile order).  Chunks of 32 tiles:
//   refill_scan_kernel   one CTA, thread = chunk: sums the chunk's used counts (one 128-byte run), block-wide exclusive scan
//                        -> chunk_base[chunk]; the total goes to cursor[2]
//   refill_tasks_kernel  warp = chunk, lane = tile: exclusive scan inside the chunk, the tile's used records are listed, its
//                        count cleared
__global__ void __launch_bounds__(1024) refill_scan_kernel(const __grid_constant__ FreshParams f, uint32_t* __restrict__ chunk_base) {
    __shared__ unsigned s_warp[32];
    const int n_chunks = (f.n_tiles + 31) / 32;
    unsigned running = 0;                                   // (batches beyond 32,768 tiles: several rounds of 1,024 chunks)
    for (int c0 = 0; c0 < n_chunks; c0 += 1024) {
        const int c = c0 + threadIdx.x;
        unsigned mine = 0;
        if (c < n_chunks) {
            const int t0 = c * 32, t1 = min(f.n_tiles, t0 + 32);
            if (t1 - t0 == 32) {                                  // a whole chunk: one 128-byte run, eight independent loads
                const uint4* u4 = reinterpret_cast<const uint4*>(f.tile_used + t0);
                uint4 v[8];
#pragma unroll
                for (int k = 0; k < 8; k++) v[k] = u4[k];
                const uint32_t q = (uint32_t)f.quota;
#pragma unroll
                for (int k = 0; k < 8; k++) mine += min(v[k].x, q) + min(v[k].y, q) + min(v[k].z, q) + min(v[k].w, q);
            } else {
                for (int t = t0; t < t1; t++) mine += min(f.tile_used[t], (uint32_t)f.quota);
            }
        }
        unsigned incl = mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned v = __shfl_up_sync(0xffffffffu, incl, d);
            if ((int)(threadIdx.x & 31) >= d) incl += v;
        }
        if ((threadIdx.x & 31) == 31) s_warp[threadIdx.x >> 5] = incl;
        __syncthreads();
        unsigned wsum = threadIdx.x < 32 ? s_warp[threadIdx.x] : 0u, wincl = wsum;
        if (threadIdx.x < 32) {
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const unsigned v = __shfl_up_sync(0xffffffffu, wincl, d);
                if ((int)threadIdx.x >= d) wincl += v;
            }
            s_warp[threadIdx.x] = wincl - wsum;             // exclusive warp offsets
        }
        __syncthreads();
        const unsigned base = running + s_warp[threadIdx.x >> 5] + incl - mine;
        if (c < n_chunks) chunk_base[c] = base;
        __syncthreads();
        if (threadIdx.x == 1023) s_warp[0] = base + mine;   // total so far
        __syncthreads();
        running = s_warp[0];
        __syncthreads();
    }
    if (threadIdx.x == 0) f.cursor[2] = running;
}
__global__ void __launch_bounds__(256) refill_tasks_kernel(const __grid_constant__ FreshParams f, const uint32_t* __restrict__ chunk_base) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;      // tile (whole warps run: the chunk scan needs every lane)
    const int lane = threadIdx.x & 31;
    const unsigned u = t < f.n_tiles ? min(f.tile_used[t], (uint32_t)f.quota) : 0u;
    unsigned at = chunk_base[min(t >> 5, (f.n_tiles + 31) / 32 - 1)] + warp_exclusive_sum(u, lane);
    for (unsigned j = 0; j < u; j++) f.tasks[at + j] = (uint32_t)t * (uint32_t)f.quota + j;
    if (u) f.tile_used[t] = 0u;
}

// (a grid that covers the device a few times over, striding over the tasks: the number of tasks is only known on the
// device, and a grid sized for the whole ring — 24,576 CTAs at 1M games, nearly all of them empty — cost 17 us by itself.
// The CTA that finishes last moves the cursor on: f.cursor[3] counts the finished CTAs.)
template <int S>
__global__ void __launch_bounds__(64) refill_create_kernel(const __grid_constant__ FreshParams f, const __grid_constant__ CreateParams q) {
    const unsigned n_tasks = (unsigned)f.cursor[2];
    const unsigned long long base = f.cursor[0];
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n_tasks; i += gridDim.x * blockDim.x) {
        const unsigned long long pos = base + i;
        const uint32_t seed = f.seeds[(uint32_t)pos & f.seed_mask];
        CreatedGame o;
        create_game<S>(seed, q, o);
        write_record<S>(f.ring + (size_t)f.tasks[i] * 8, o, (uint32_t)pos, seed);
    }
    __syncthreads();                       // every thread of the CTA has read the cursor and written its records
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(&f.cursor[3], 1ull) + 1ull == (unsigned long long)gridDim.x) {
            f.cursor[0] = base + n_tasks;
            f.cursor[1] += 1ull;
            f.cursor[2] = 0ull;
            f.cursor[3] = 0ull;
            __threadfence();
        }
    }
}

template <int S>
__global__ void __launch_bounds__(64) fresh_fill_kernel(const __grid_constant__ FreshParams f, const __grid_constant__ CreateParams q,
                                                        float4* __restrict__ ships, float* __restrict__ ship_b, float4* __restrict__ planets,
                                                        uint32_t* __restrict__ meta, uint32_t* __restrict__ episode, uint32_t* __restrict__ game_pos) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= f.n_games) return;
    const unsigned long long pos = f.cursor[0] + (unsigned)g;
    const uint32_t seed = f.seeds[(uint32_t)pos & f.seed_mask];
    CreatedGame o;
    create_game<S>(seed, q, o);
    const size_t tile = (size_t)(g >> 5);
    const int lane = g & 31;
#pragma unroll
    for (int s = 0; s < S; s++) {
        ships[tile * (S * 32) + s * 32 + lane] = make_float4(o.sx[s][0], o.sx[s][1], 0.f, 0.f);
        ship_b[tile * (S * 32) + s * 32 + lane] = o.sb[s];
    }
#pragma unroll
    for (int j = 0; j < ASTRO_MAX_PLANETS; j++)
        planets[tile * (ASTRO_MAX_PLANETS * 32) + j * 32 + lane] = make_float4(o.px[j][0], o.px[j][1], (float)o.pv[j][0], (float)o.pv[j][1]);
    meta[g] = ASTRO_META_PACK(0, o.n, 0, 0);
    episode[g] = 0u;
    game_pos[g] = (uint32_t)pos;
}
__global__ void fresh_fill_commit_kernel(const __grid_constant__ FreshParams f) { f.cursor[0] += (unsigned)f.n_games; }

// ------------------------------------------------------------------------------------------
// rl.ValueNetwork (rl.py:140-165): 32-wide layers, at most kPolMaxOut outputs
// ------------------------------------------------------------------------------------------
constexpr int kPolW = 32;           // layer width (rl.py:144)
constexpr int kPolMaxOut = 8;

// x / (1 + |x|) with the fast reciprocal (2 ulp): the network's outputs stay within ~1e-6 of PyTorch's
__device__ __forceinline__ float softsign(float x) { return div_fast_normal(x, 1.0f + fabsf(x)); }

// ------------------------------------------------------------------------------------------
// policy_mma_kernel<R, S, PL>: rl.ValueNetwork.forward (rl.py:140-165) on the features of rl.py:43-72, fused — the
// observation tensor never exists — for every game and both perspectives (core.roll_ships), then control = argmax q (the
// greedy policy of rl.QBot, rl.py:168-200).  The three per-object layers are batched GEMMs [row-vectors, 32] x [32, 32]:
// a warp takes a game's live rows eight objects at a time as ONE 16-row MMA tile — rows 0-7 the eight objects seen by
// ship 0, rows 8-15 the same objects seen by ship 1 — and runs f0, f[0], f[1] as mma.sync.m16n8k16 tiles with FP16
// operands and fp32 accumulators (HMMA.16816.F32).  An 11-bit operand alone would move the outputs by 1e-3 and flip
// near-tied argmaxes, so every product is taken as three: a = a_hi + a_lo, w = w_hi + w_lo (each part an FP16 number),
// a.w ~ a_lo.w_hi + a_hi.w_lo + a_hi.w_hi — fp32-level results (the outputs stay within 2e-6 of the PyTorch fp32
// network).  FP16's range (|x| < 65,504; lo parts below 6e-5 lose relative precision, 3e-8 absolute) is ample for this
// network: activations sit in (-1, 1), features and pre-activations within a few units.
//   * A fragments come straight from registers: the accumulator layout of one layer (columns 2t, 2t+1 of n-tiles 2k and
//     2k+1) IS the A layout of the next layer's k-step k — no shuffle, no shared memory between layers.  The first
//     layer's A fragment (15 features, K padded to 16: one k-step) is built per lane from the game's ship features and
//     one or two components of the row's object.
//   * B fragments (weights, split into hi / lo, fragment-ordered: one LDS.128 per k-step and n-tile) are built once by
//     astro_policy_set_weights and staged in shared memory once per CTA (20 KB).
//   * max-pool: a running maximum in the accumulator layout, reduced across the quads once per game; a warp pools 8
//     games and then runs the head (two 32 x 32 layers and 32 -> nout) for all of them as one 16-row tile.
// ------------------------------------------------------------------------------------------
constexpr int kMmaWarps = 4;
constexpr int kPoolStride = 36;      // floats per row of the pooled tile (32 + 4: the A-fragment loads hit 32 different banks)
constexpr int kKs0 = 1;              // k-steps of the first layer (16 input columns)
constexpr int kKs = 2;               // k-steps of a 32-wide layer
struct PolicyFragWeights {           // B fragments {b0_hi, b1_hi, b0_lo, b1_lo} per lane, built once by astro_policy_set_weights
    float4 f0[kKs0][4][32];          // [k-step][n-tile][lane]: per-object layers
    float4 f1[kKs][4][32];
    float4 f2[kKs][4][32];
    float4 v1[kKs][4][32];           // head
    float4 v2[kKs][4][32];
    float4 v0[kKs][32];              // head output: one n-tile (nout <= 8)
    float2 bias[5][4][4];            // [f0, f1, f2, v1, v2][n-tile][t] = bias of units 8 nt + 2t, 8 nt + 2t + 1
    float2 bias_v0[4];               // [t] = bias of outputs 2t, 2t + 1
};
struct PolicyFrags {                 // per CTA, in (dynamic) shared memory
    PolicyFragWeights w;             // copied from global memory, 16 bytes per thread and step
    float pool[kMmaWarps][16][kPoolStride];   // per warp: the pooled vectors of 8 games, rows 0-7 ship 0's view, 8-15 ship 1's
    float4 red[kMmaWarps][8][4][2];  // per warp: max-pool exchange, [quad][t][half of the 16 accumulators as 2 float4]
    float sf[kMmaWarps][8][12];      // per warp: the ship features of its 8 games, ship 0 then ship 1
};
// two fp32 values -> the FP16 pair (hi) and the FP16 pair of what that dropped (lo); lower half = the even column
__device__ __forceinline__ void split_f16x2(float xe, float xo, uint32_t& hi, uint32_t& lo) {
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(xo), "f"(xe));
    float he, ho;
    asm("{ .reg .f16 l, h; mov.b32 {l, h}, %2; cvt.f32.f16 %0, l; cvt.f32.f16 %1, h; }" : "=f"(he), "=f"(ho) : "r"(hi));
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(__fsub_rn(xo, ho)), "f"(__fsub_rn(xe, he)));
}
__device__ __forceinline__ void mma_f16(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
// one k-step (16 input columns) for NT n-tiles.  x = this lane's eight A values: (row g: columns 2t, 2t+1), (row g+8: same),
// (row g: columns 2t+8, 2t+9), (row g+8: same) — for a 32-wide layer exactly the accumulators of n-tiles 2 kk and 2 kk + 1.
template <int NT>
__device__ __forceinline__ void mma_kstep16(float (&acc)[NT][4], const float (&x)[8], const float4* __restrict__ bfrag, int lane) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; i++) split_f16x2(x[2 * i], x[2 * i + 1], h[i], l[i]);
#pragma unroll
    for (int nt = 0; nt < NT; nt++) {
        const float4 b = bfrag[nt * 32 + lane];
        const uint32_t bh0 = __float_as_uint(b.x), bh1 = __float_as_uint(b.y), bl0 = __float_as_uint(b.z), bl1 = __float_as_uint(b.w);
        mma_f16(acc[nt], l[0], l[1], l[2], l[3], bh0, bh1);      // small terms first
        mma_f16(acc[nt], h[0], h[1], h[2], h[3], bl0, bl1);
        mma_f16(acc[nt], h[0], h[1], h[2], h[3], bh0, bh1);
    }
}
// a 32-wide layer: out = bias + W act(in), in / out in the accumulator layout
template <int NT, bool ACT>
__device__ __forceinline__ void mma_layer(float (&out)[NT][4], const float (&in)[4][4], const float4* __restrict__ wf, int lane) {
#pragma unroll
    for (int kk = 0; kk < 2; kk++) {
        float x[8];
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const float v = in[2 * kk + (i >> 2)][i & 3];
            x[i] = ACT ? softsign(v) : v;
        }
        mma_kstep16<NT>(out, x, wf + kk * NT * 32, lane);
    }
}
template <int NT>
__device__ __forceinline__ void init_bias(float (&acc)[NT][4], const float2 (*bias)[4], int t) {
#pragma unroll
    for (int nt = 0; nt < NT; nt++) {
        const float2 b2 = bias[nt][t];
        acc[nt][0] = b2.x; acc[nt][1] = b2.y; acc[nt][2] = b2.x; acc[nt][3] = b2.y;
    }
}

#ifndef ASTRO_MMA_MIN_BLOCKS
#define ASTRO_MMA_MIN_BLOCKS 4
#endif
template <typename R, int S, int PL>
__global__ void __launch_bounds__(kMmaWarps * 32, ASTRO_MMA_MIN_BLOCKS)
policy_mma_kernel(const void* __restrict__ ships_, const void* __restrict__ ship_b_, const void* __restrict__ planets_,
                  const void* __restrict__ bullets_, const uint32_t* __restrict__ meta_, uint8_t* __restrict__ actions,
                  float* __restrict__ q_out, int n_games, int K, int nout, int ship_mask, const PolicyFragWeights* __restrict__ frags) {
    constexpr int DIN = 1 + 5 * S + 4;
    extern __shared__ float4 s_dyn[];
    PolicyFrags& s_all = *reinterpret_cast<PolicyFrags*>(s_dyn);
    const PolicyFragWeights& s_w = s_all.w;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gq = lane >> 2, t = lane & 3;                     // quad = object row of the tile / n column; t = k index
    // ---- the weights, already split and fragment-ordered (astro_policy_set_weights): one coalesced copy per CTA
    {
        const uint4* src = reinterpret_cast<const uint4*>(frags);
        uint4* dst = reinterpret_cast<uint4*>(&s_all.w);
        for (int i = threadIdx.x; i < (int)(sizeof(PolicyFragWeights) / 16); i += blockDim.x) dst[i] = src[i];
    }
    __syncthreads();
    // ---- what this lane's four feature slots (columns 2t, 2t + 1, 2t + 8, 2t + 9: one k-step of 16) are: flag / ship
    // feature / object component / zero
    int ship_idx[4], obj_idx[4];
    bool is_flag = false, any_obj = false;
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const int col = 2 * t + (j & 1) + 8 * (j >> 1);
        ship_idx[j] = obj_idx[j] = -1;
        if (col == 0) is_flag = true;                           // (slot 0 of lane t = 0)
        else if (col <= 5 * S) ship_idx[j] = col - 1;           // feature (col - 1) % 5 of ship (col - 1) / 5, ship 0's perspective
        else if (col < DIN) { obj_idx[j] = col - 1 - 5 * S; any_obj = true; }
    }
    float (*pool)[kPoolStride] = s_all.pool[warp];
    // a warp takes 8 consecutive games at a time (one quarter of a tile: n_games is a multiple of 32): their pooled vectors
    // make one 16-row tile for the head
    const int n_groups = n_games >> 3;
    for (int grp = blockIdx.x * kMmaWarps + warp; grp < n_groups; grp += gridDim.x * kMmaWarps) {
        // ---- everything the 8 games need that does not depend on the network, for all of them at once (one round of
        // loads per kind instead of one per game: a game's chain below starts with its rows already on their way)
        const size_t tile = (size_t)(grp >> 2);
        const int gl0 = (grp & 3) * 8;
        const uint32_t meta_l = meta_[tile * 32 + lane];                      // the tile's 32 meta words: list offsets, np, rows
        const bool fin_l = ASTRO_META_FINISHED(meta_l);
        const unsigned nb_l = fin_l ? 0u : ASTRO_META_NB(meta_l);
        unsigned incl = nb_l;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned v = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += v;
        }
        const unsigned off_l = incl - nb_l;                                  // first list item of lane's game (tile_list_offset)
        const int np_l = fin_l ? 0 : (int)meta_np<PL>(meta_l);
        const int rows_l = fin_l ? 0 : np_l + (int)nb_l;
        const unsigned live_mask = (__ballot_sync(0xffffffffu, rows_l > 0) >> gl0) & 0xffu;
        // ship features (x, y, dx, dy, norm_angle(b) / pi), ship 0 then ship 1, of the 8 games: the float64 bearings by
        // 8 S lanes in ONE pass, the 32 S plain components in S passes
        if (lane < 8 * S) {
            const int j8 = lane / S, s_ = lane % S;
            s_all.sf[warp][j8][5 * s_ + 4] = (float)__ddiv_rn(norm_angle_f64((double)reinterpret_cast<const R*>(ship_b_)[tile * (S * 32) + s_ * 32 + gl0 + j8]), 3.141592653589793);
        }
#pragma unroll
        for (int s_ = 0; s_ < S; s_++) {
            const int j8 = lane >> 2, c = lane & 3;
            s_all.sf[warp][j8][5 * s_ + c] = (float)reinterpret_cast<const R*>(ships_)[(tile * (S * 32) + s_ * 32 + gl0 + j8) * 4 + c];
        }
        __syncwarp();
        const Body4<R>* const pl_tile = reinterpret_cast<const Body4<R>*>(planets_) + tile * (PL * 32);
        const Body4<R>* const bl_tile = reinterpret_cast<const Body4<R>*>(bullets_) + tile * (size_t)(32 * K);
        // this lane's object component(s) of row gq of a game's first 8 rows (the quad covers the object's 16 bytes)
        auto load_first_rows = [&](int j8, float (&ov)[4]) {
            const int np = __shfl_sync(0xffffffffu, np_l, gl0 + j8), rows = __shfl_sync(0xffffffffu, rows_l, gl0 + j8);
            const unsigned off = __shfl_sync(0xffffffffu, off_l, gl0 + j8);
#pragma unroll
            for (int j = 0; j < 4; j++) ov[j] = 0.f;
            if (gq < rows && any_obj) {
                const R* o = reinterpret_cast<const R*>(gq < np ? &pl_tile[gq * 32 + gl0 + j8] : &bl_tile[off + (unsigned)(gq - np)]);
#pragma unroll
                for (int j = 0; j < 4; j++) if (obj_idx[j] >= 0) ov[j] = (float)o[obj_idx[j]];
            }
        };
        float ov_next[4];
        load_first_rows(0, ov_next);
#pragma unroll 1
        for (int j8 = 0; j8 < 8; j8++) {
            const int gl = gl0 + j8;
            const int np = __shfl_sync(0xffffffffu, np_l, gl), rows = __shfl_sync(0xffffffffu, rows_l, gl);
            const unsigned off = __shfl_sync(0xffffffffu, off_l, gl);
            float ov[4];
#pragma unroll
            for (int j = 0; j < 4; j++) ov[j] = ov_next[j];
            if (j8 < 7) load_first_rows(j8 + 1, ov_next);        // the next game's rows travel while this game's layers run
            float xa[4], xb[4];                                  // this lane's feature slots, perspective of ship 0 / ship 1
#pragma unroll
            for (int j = 0; j < 4; j++) {
                xa[j] = xb[j] = 0.f;
                if (ship_idx[j] >= 0) {
                    xa[j] = s_all.sf[warp][j8][ship_idx[j]];
                    xb[j] = s_all.sf[warp][j8][S == 2 ? (ship_idx[j] + 5) % 10 : ship_idx[j]];    // the ship column groups exchanged
                }
            }
            const Body4<R>* pl = pl_tile + gl;
            const Body4<R>* bl = bl_tile + off;
            float best[4][4];
#pragma unroll
            for (int nt = 0; nt < 4; nt++)
#pragma unroll
                for (int i = 0; i < 4; i++) best[nt][i] = -3.0e38f;
            for (int r0 = 0; r0 < rows; r0 += 8) {
                const int r = r0 + gq;
                const bool valid = r < rows;
                if (r0 == 0) {                                   // (loaded one game ahead)
#pragma unroll
                    for (int j = 0; j < 4; j++) if (obj_idx[j] >= 0) { xa[j] = ov[j]; xb[j] = ov[j]; }
                } else if (valid && any_obj) {                   // this lane's component(s) of the row's object: the quad covers its 16 bytes
                    const R* o = reinterpret_cast<const R*>(r < np ? &pl[r * 32] : &bl[r - np]);
#pragma unroll
                    for (int j = 0; j < 4; j++) if (obj_idx[j] >= 0) { const float v = (float)o[obj_idx[j]]; xa[j] = v; xb[j] = v; }
                }
                if (is_flag) xa[0] = xb[0] = (r < np) ? 0.0f : 1.0f;
                float acc[4][4], nxt[4][4];
                init_bias<4>(acc, s_w.bias[0], t);               // f0: K = 16 (15 features)
                {
                    const float x0[8] = {xa[0], xa[1], xb[0], xb[1], xa[2], xa[3], xb[2], xb[3]};
                    mma_kstep16<4>(acc, x0, &s_w.f0[0][0][0], lane);
                }
#pragma unroll
                for (int layer = 1; layer <= 2; layer++) {       // f[0], f[1]: h = W softsign(h) + b
                    const float4* wf = layer == 1 ? &s_w.f1[0][0][0] : &s_w.f2[0][0][0];
                    init_bias<4>(nxt, s_w.bias[layer], t);
                    mma_layer<4, true>(nxt, acc, wf, lane);
#pragma unroll
                    for (int nt = 0; nt < 4; nt++)
#pragma unroll
                        for (int i = 0; i < 4; i++) acc[nt][i] = nxt[nt][i];
                }
                if (valid) {
#pragma unroll
                    for (int nt = 0; nt < 4; nt++)
#pragma unroll
                        for (int i = 0; i < 4; i++) best[nt][i] = fmaxf(best[nt][i], acc[nt][i]);
                }
            }
            // max over the object rows = over the quads: through shared memory, transposed — lane u then holds unit u's
            // maximum for ship 0's view, and for ship 1's (two passes of 8 accumulators: 1 KB per warp)
            float pooled[2];
#pragma unroll
            for (int half = 0; half < 2; half++) {               // half 0: accumulator entries 0-1 (ship 0's view), 1: entries 2-3
                s_all.red[warp][gq][t][0] = make_float4(best[0][2 * half], best[0][2 * half + 1], best[1][2 * half], best[1][2 * half + 1]);
                s_all.red[warp][gq][t][1] = make_float4(best[2][2 * half], best[2][2 * half + 1], best[3][2 * half], best[3][2 * half + 1]);
                __syncwarp();
                // unit u = 8 nt + 2 t' + e sits at float index 2 nt + e of lane (quad, t')
                const int nt_u = lane >> 3, t_u = (lane >> 1) & 3, e_u = lane & 1;
                float m = -3.0e38f;
#pragma unroll
                for (int qd = 0; qd < 8; qd++) m = fmaxf(m, reinterpret_cast<const float*>(&s_all.red[warp][qd][t_u][0])[2 * nt_u + e_u]);
                pooled[half] = m;
                __syncwarp();
            }
            pool[j8][lane] = pooled[0];
            pool[8 + j8][lane] = pooled[1];
        }
        __syncwarp();
        // ---- head for the 8 games at once: v[0], v[1] (linear -> softsign) as 16 x 32 x 32 MMA tiles, v0 as 16 x 32 x 8
        float h1[4][4], h2[4][4], q4[1][4];
        init_bias<4>(h1, s_w.bias[3], t);
#pragma unroll
        for (int kk = 0; kk < 2; kk++) {
            const float2 p0 = *reinterpret_cast<const float2*>(&pool[gq][16 * kk + 2 * t]), p1 = *reinterpret_cast<const float2*>(&pool[gq + 8][16 * kk + 2 * t]);
            const float2 p2 = *reinterpret_cast<const float2*>(&pool[gq][16 * kk + 2 * t + 8]), p3 = *reinterpret_cast<const float2*>(&pool[gq + 8][16 * kk + 2 * t + 8]);
            const float x[8] = {p0.x, p0.y, p1.x, p1.y, p2.x, p2.y, p3.x, p3.y};
            mma_kstep16<4>(h1, x, &s_w.v1[kk][0][0], lane);
        }
        init_bias<4>(h2, s_w.bias[4], t);
        mma_layer<4, true>(h2, h1, &s_w.v2[0][0][0], lane);
        {
            const float2 b2 = s_w.bias_v0[t];
            q4[0][0] = b2.x; q4[0][1] = b2.y; q4[0][2] = b2.x; q4[0][3] = b2.y;
        }
        mma_layer<1, true>(q4, h2, &s_w.v0[0][0], lane);
        // this lane: game grp * 8 + gq, outputs 2t and 2t + 1, ship 0's view (entries 0-1) and ship 1's (2-3)
        const int g = grp * 8 + gq;
        const bool live = (live_mask >> gq) & 1u;
        float qv[4];
#pragma unroll
        for (int i = 0; i < 4; i++) qv[i] = (2 * t + (i & 1)) < nout ? tanhf(q4[0][i]) : -2.0f;    // outputs >= nout stay below any tanh value
        // argmax over the quad's 8 outputs, first maximum like torch.argmax
        float ma = qv[0], mb = qv[2];
        int ia = 2 * t, ib = 2 * t;
        if (qv[1] > ma) { ma = qv[1]; ia = 2 * t + 1; }
        if (qv[3] > mb) { mb = qv[3]; ib = 2 * t + 1; }
#pragma unroll
        for (int d = 1; d <= 2; d <<= 1) {
            const float oa = __shfl_xor_sync(0xffffffffu, ma, d), ob = __shfl_xor_sync(0xffffffffu, mb, d);
            const int ja = __shfl_xor_sync(0xffffffffu, ia, d), jb = __shfl_xor_sync(0xffffffffu, ib, d);
            if (oa > ma || (oa == ma && ja < ia)) { ma = oa; ia = ja; }
            if (ob > mb || (ob == mb && jb < ib)) { mb = ob; ib = jb; }
        }
        if (g < n_games) {
            if (t == 0 && (ship_mask & 1)) actions[(size_t)g * S] = (uint8_t)(live ? ia : 2);    // finished game: the no-op control
            if (S == 2 && t == 1 && (ship_mask & 2)) actions[(size_t)g * S + 1] = (uint8_t)(live ? ib : 2);
            if (q_out) {
#pragma unroll
                for (int e = 0; e < 2; e++) {
                    if (2 * t + e < nout) {
                        q_out[((size_t)g * S) * nout + 2 * t + e] = live ? qv[e] : 0.0f;
                        if (S == 2) q_out[((size_t)g * S + 1) * nout + 2 * t + e] = live ? qv[2 + e] : 0.0f;
                    }
                }
            }
        }
        __syncwarp();
    }  // groups of this warp
}

// ------------------------------------------------------------------------------------------
// value_forward_kernel<DIN>: rl.ValueNetwork.forward (rl.py:140-165) on a FEATURE batch — what astro.rl's own callers
// hold (get_features_batch / BatchedGames.observe() output) — for inference: features [n][rows][DIN] -> q [n][nout].
// The network of policy_mma_kernel, same weights (fragments), same three-product FP16 split, fed from the tensor instead
// of from the game state: a 16-row MMA tile = 8 consecutive rows of item A (tile rows 0-7) and of item B (rows 8-15); a
// warp takes 16 items at a time — pairs (j, j + 8) — so that their pooled vectors make the head's 16-row tile.
//   pooling = the reference's masked_max (rl.py:115-128): max over ALL rows of x - 1e9 * pad, pad = (features[row][0] < 0).
//   A chunk of 8 rows that is padding for both items is skipped once each item has shown a live row (its maximum can no
//   longer come from a padding row: pre-activations are far below 1e9); an item without any live row takes every chunk,
//   exactly the reference's arithmetic.
// ------------------------------------------------------------------------------------------
template <int DIN>
__global__ void __launch_bounds__(kMmaWarps * 32, ASTRO_MMA_MIN_BLOCKS)
value_forward_kernel(const float* __restrict__ features, float* __restrict__ q_out, int n_items, int rows, int nout,
                     const PolicyFragWeights* __restrict__ frags) {
    extern __shared__ float4 s_dyn[];
    PolicyFrags& s_all = *reinterpret_cast<PolicyFrags*>(s_dyn);
    const PolicyFragWeights& s_w = s_all.w;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gq = lane >> 2, t = lane & 3;
    {
        const uint4* src = reinterpret_cast<const uint4*>(frags);
        uint4* dst = reinterpret_cast<uint4*>(&s_all.w);
        for (int i = threadIdx.x; i < (int)(sizeof(PolicyFragWeights) / 16); i += blockDim.x) dst[i] = src[i];
    }
    __syncthreads();
    int col[4];                                   // this lane's feature columns: 2t, 2t + 1, 2t + 8, 2t + 9 (>= DIN: zero)
#pragma unroll
    for (int j = 0; j < 4; j++) col[j] = 2 * t + (j & 1) + 8 * (j >> 1);
    float (*pool)[kPoolStride] = s_all.pool[warp];
    const int n_groups = (n_items + 15) >> 4;
    const size_t item_stride = (size_t)rows * DIN;
    for (int grp = blockIdx.x * kMmaWarps + warp; grp < n_groups; grp += gridDim.x * kMmaWarps) {
#pragma unroll 1
        for (int j8 = 0; j8 < 8; j8++) {
            const int ia = grp * 16 + j8, ib = ia + 8;
            const bool has_a = ia < n_items, has_b = ib < n_items;       // (warp-uniform)
            const float* fa = features + (size_t)(has_a ? ia : 0) * item_stride;
            const float* fb = features + (size_t)(has_b ? ib : 0) * item_stride;
            float best[4][4];
#pragma unroll
            for (int nt = 0; nt < 4; nt++)
#pragma unroll
                for (int i = 0; i < 4; i++) best[nt][i] = -3.0e38f;
            bool seen_a = !has_a, seen_b = !has_b;
            for (int r0 = 0; r0 < rows; r0 += 8) {
                const int r = r0 + gq;
                const bool in_range = r < rows;
                // the type flags first (column 0: lanes t == 0), handed to the quad
                float flag_a = -1.f, flag_b = -1.f;
                if (t == 0 && in_range) {
                    if (has_a) flag_a = fa[(size_t)r * DIN];
                    if (has_b) flag_b = fb[(size_t)r * DIN];
                }
                flag_a = __shfl_sync(0xffffffffu, flag_a, lane & ~3);
                flag_b = __shfl_sync(0xffffffffu, flag_b, lane & ~3);
                const bool live_a = in_range && has_a && !(flag_a < 0.f), live_b = in_range && has_b && !(flag_b < 0.f);
                const bool any_live = __ballot_sync(0xffffffffu, live_a | live_b) != 0u;
                if (!any_live && seen_a && seen_b) continue;             // padding only, and nobody's maximum can be there
                seen_a |= __ballot_sync(0xffffffffu, live_a) != 0u;
                seen_b |= __ballot_sync(0xffffffffu, live_b) != 0u;
                float xa[4], xb[4];
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    xa[j] = xb[j] = 0.f;
                    if (col[j] < DIN && in_range) {
                        if (has_a) xa[j] = (col[j] == 0) ? flag_a : fa[(size_t)r * DIN + col[j]];
                        if (has_b) xb[j] = (col[j] == 0) ? flag_b : fb[(size_t)r * DIN + col[j]];
                    }
                }
                float acc[4][4], nxt[4][4];
                init_bias<4>(acc, s_w.bias[0], t);
                {
                    const float x0[8] = {xa[0], xa[1], xb[0], xb[1], xa[2], xa[3], xb[2], xb[3]};
                    mma_kstep16<4>(acc, x0, &s_w.f0[0][0][0], lane);
                }
#pragma unroll
                for (int layer = 1; layer <= 2; layer++) {
                    const float4* wf = layer == 1 ? &s_w.f1[0][0][0] : &s_w.f2[0][0][0];
                    init_bias<4>(nxt, s_w.bias[layer], t);
                    mma_layer<4, true>(nxt, acc, wf, lane);
#pragma unroll
                    for (int nt = 0; nt < 4; nt++)
#pragma unroll
                        for (int i = 0; i < 4; i++) acc[nt][i] = nxt[nt][i];
                }
                // masked_max: x - 1e9 * pad (float32, as torch computes it), rows past the tensor excluded
                const float pen_a = live_a ? 0.f : 1.0e9f, pen_b = live_b ? 0.f : 1.0e9f;
                if (in_range) {
#pragma unroll
                    for (int nt = 0; nt < 4; nt++) {
                        if (has_a) { best[nt][0] = fmaxf(best[nt][0], __fsub_rn(acc[nt][0], pen_a)); best[nt][1] = fmaxf(best[nt][1], __fsub_rn(acc[nt][1], pen_a)); }
                        if (has_b) { best[nt][2] = fmaxf(best[nt][2], __fsub_rn(acc[nt][2], pen_b)); best[nt][3] = fmaxf(best[nt][3], __fsub_rn(acc[nt][3], pen_b)); }
                    }
                }
            }
            float pooled[2];
#pragma unroll
            for (int half = 0; half < 2; half++) {
                s_all.red[warp][gq][t][0] = make_float4(best[0][2 * half], best[0][2 * half + 1], best[1][2 * half], best[1][2 * half + 1]);
                s_all.red[warp][gq][t][1] = make_float4(best[2][2 * half], best[2][2 * half + 1], best[3][2 * half], best[3][2 * half + 1]);
                __syncwarp();
                const int nt_u = lane >> 3, t_u = (lane >> 1) & 3, e_u = lane & 1;
                float m = -3.0e38f;
#pragma unroll
                for (int qd = 0; qd < 8; qd++) m = fmaxf(m, reinterpret_cast<const float*>(&s_all.red[warp][qd][t_u][0])[2 * nt_u + e_u]);
                pooled[half] = m;
                __syncwarp();
            }
            pool[j8][lane] = (has_a && rows > 0) ? pooled[0] : 0.f;
            pool[8 + j8][lane] = (has_b && rows > 0) ? pooled[1] : 0.f;
        }
        __syncwarp();
        // The pooled vector of an item WITHOUT a live row is the reference's x - 1e9 (masked_max): far outside FP16's range.
        // The first head layer is therefore taken per tile row on a power-of-two scaled copy of the row (exact), its
        // accumulators scaled back and the bias added last; rows of ordinary magnitude keep scale 1.
        float h1[4][4], h2[4][4], q4[1][4];
        float xs[2][8];
        float mx_a = 0.f, mx_b = 0.f;
#pragma unroll
        for (int kk = 0; kk < 2; kk++) {
            const float2 p0 = *reinterpret_cast<const float2*>(&pool[gq][16 * kk + 2 * t]), p1 = *reinterpret_cast<const float2*>(&pool[gq + 8][16 * kk + 2 * t]);
            const float2 p2 = *reinterpret_cast<const float2*>(&pool[gq][16 * kk + 2 * t + 8]), p3 = *reinterpret_cast<const float2*>(&pool[gq + 8][16 * kk + 2 * t + 8]);
            xs[kk][0] = p0.x; xs[kk][1] = p0.y; xs[kk][2] = p1.x; xs[kk][3] = p1.y; xs[kk][4] = p2.x; xs[kk][5] = p2.y; xs[kk][6] = p3.x; xs[kk][7] = p3.y;
            mx_a = fmaxf(mx_a, fmaxf(fmaxf(fabsf(p0.x), fabsf(p0.y)), fmaxf(fabsf(p2.x), fabsf(p2.y))));
            mx_b = fmaxf(mx_b, fmaxf(fmaxf(fabsf(p1.x), fabsf(p1.y)), fmaxf(fabsf(p3.x), fabsf(p3.y))));
        }
#pragma unroll
        for (int d = 1; d <= 2; d <<= 1) {
            mx_a = fmaxf(mx_a, __shfl_xor_sync(0xffffffffu, mx_a, d));
            mx_b = fmaxf(mx_b, __shfl_xor_sync(0xffffffffu, mx_b, d));
        }
        // scale 2^-e with 2^e the power of two above max / 1024 (1 for rows below 1024)
        // (max in [2^k, 2^(k+1)), biased exponent E = k + 127: scale 2^(9 - k) = bits (263 - E) << 23, its inverse (E - 9) << 23)
        const uint32_t ea = __float_as_uint(mx_a) >> 23, eb = __float_as_uint(mx_b) >> 23;
        const bool big_a = mx_a > 1024.f && mx_a < 3.0e38f, big_b = mx_b > 1024.f && mx_b < 3.0e38f;
        const float sc_a = big_a ? __uint_as_float((263u - ea) << 23) : 1.f, inv_a = big_a ? __uint_as_float((ea - 9u) << 23) : 1.f;
        const float sc_b = big_b ? __uint_as_float((263u - eb) << 23) : 1.f, inv_b = big_b ? __uint_as_float((eb - 9u) << 23) : 1.f;
#pragma unroll
        for (int nt = 0; nt < 4; nt++)
#pragma unroll
            for (int i = 0; i < 4; i++) h1[nt][i] = 0.f;
#pragma unroll
        for (int kk = 0; kk < 2; kk++) {
            const float x[8] = {xs[kk][0] * sc_a, xs[kk][1] * sc_a, xs[kk][2] * sc_b, xs[kk][3] * sc_b, xs[kk][4] * sc_a, xs[kk][5] * sc_a, xs[kk][6] * sc_b, xs[kk][7] * sc_b};
            mma_kstep16<4>(h1, x, &s_w.v1[kk][0][0], lane);
        }
        {
#pragma unroll
            for (int nt = 0; nt < 4; nt++) {
                const float2 b2 = s_w.bias[3][nt][t];
                h1[nt][0] = __fmaf_rn(h1[nt][0], inv_a, b2.x); h1[nt][1] = __fmaf_rn(h1[nt][1], inv_a, b2.y);
                h1[nt][2] = __fmaf_rn(h1[nt][2], inv_b, b2.x); h1[nt][3] = __fmaf_rn(h1[nt][3], inv_b, b2.y);
            }
        }
        // v[0], v[1]: h = softsign(W h + b) (rl.py:160-162) — the activation follows the layer here
        init_bias<4>(h2, s_w.bias[4], t);
        mma_layer<4, true>(h2, h1, &s_w.v2[0][0][0], lane);
        {
            const float2 b2 = s_w.bias_v0[t];
            q4[0][0] = b2.x; q4[0][1] = b2.y; q4[0][2] = b2.x; q4[0][3] = b2.y;
        }
        mma_layer<1, true>(q4, h2, &s_w.v0[0][0], lane);
        // this lane: outputs 2t, 2t + 1 of item grp * 16 + gq (entries 0-1) and of item grp * 16 + 8 + gq (entries 2-3)
#pragma unroll
        for (int e = 0; e < 2; e++) {
            if (2 * t + e < nout) {
                const int ia = grp * 16 + gq, ib = ia + 8;
                if (ia < n_items) q_out[(size_t)ia * nout + 2 * t + e] = tanhf(q4[0][e]);
                if (ib < n_items) q_out[(size_t)ib * nout + 2 * t + e] = tanhf(q4[0][2 + e]);
            }
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------
// explore_kernel: rl.EpsilonGreedy.__call__ (rl.py:10-30) for every ship — the random policy that
// rl.QBotTrainer lays over the greedy network (rl.py:249-258: action = greedy if greedy is not None
// else argmax q).  Per ship a two-state process: idle -> a random control 0..4 (randint(0, 5): never 5)
// when exp(-dt / t_in) < u, random control -> idle when exp(-dt / t_out) < u, one uniform u per call;
// dt = state.t - the t of the previous call, so the first call of a new game (t back to 0: dt < 0)
// never switches.  State per ship, caller-owned: (tick of the previous call) << 8 | (control + 1, 0 =
// idle).  The reference draws from a numpy RandomState per bot; here u and the control come from the
// counter stream keyed on (seed, global game, stream step, ship) — the same process, not the same
// sequence (host twin: astro_b200/rng.py explore_step).
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t explore_key(uint32_t seed, uint32_t game, uint32_t step, uint32_t ship) {
    return mix32(mix32(seed ^ 0x3C6EF372u ^ (game * 0x9E3779B1u)) ^ (step * 2u + ship));
}
template <int S, int PL>
__global__ void __launch_bounds__(128) explore_kernel(const uint32_t* __restrict__ meta_, int32_t* __restrict__ state,
                                                      uint8_t* __restrict__ actions, int n_games, int ship_mask, double dt,
                                                      double t_in, double t_out, uint32_t seed, uint32_t first_game, uint32_t step,
                                                      const uint32_t* __restrict__ step_base) {
    if (step_base) step += *step_base;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int g = idx / S, me = idx % S;
    if (g >= n_games || !((ship_mask >> me) & 1)) return;
    const uint32_t meta = meta_[g];
    if (ASTRO_META_FINISHED(meta)) return;
    const int tick = (int)meta_tick<PL>(meta);
    const int32_t st = state[idx];
    int policy = (st & 0xff) - 1;                     // -1 = idle
    const double gap = __dmul_rn(dt, (double)(tick - (st >> 8)));
    const uint32_t h = explore_key(seed, first_game + (uint32_t)g, step, (uint32_t)me);
    const double u = (double)(h >> 8) * (1.0 / 16777216.0);
    if (policy < 0) {
        if (exp(-gap / t_in) < u) policy = (int)__umulhi(mix32(h ^ 0x85EBCA6Bu), 5u);
    } else if (exp(-gap / t_out) < u) {
        policy = -1;
    }
    state[idx] = (tick << 8) | (policy + 1);
    if (policy >= 0) actions[idx] = (uint8_t)policy;
}

// ------------------------------------------------------------------------------------------
// export_kernel / import_kernel: the batch <-> game-major float64 arrays (AstroGameArrays), the
// form the host-side readers and writers of single games want: State conversion for the drop-in
// core.step / core.play (core.py:11-18, :215-303, :377-410), the JSONL logs (core.py:413-443),
// tests.  One kernel each instead of a chain of gathers: the tile lists are unpacked / packed on
// the device.
//   export: warp = one listed game; lane k copies bullet k, k + 32, ... of the game's run of its
//           tile's list; dead planet / bullet slots are written as zeros.
//   import: warp = one tile.  src[g] = the row of the arrays that replaces game g (-1: keep).  A
//           tile with a replaced game rebuilds its list — kept games' runs and the new games'
//           bullets, dense, in game order — in the tile's run of the OTHER buffer (dead between
//           ticks, so a free scratch area) and copies it back; then the rows and meta words of the
//           replaced games are written.
// ------------------------------------------------------------------------------------------
struct GameArrays {          // device pointers, see AstroGameArrays
    double* ships;
    double* planets;
    double* bullets;
    int32_t* n_planets;
    int32_t* n_bullets;
    int32_t* tick;
    uint8_t* finished;
    uint32_t* episode;
};

template <typename R, int S, int PL>
__global__ void __launch_bounds__(128) export_kernel(const void* __restrict__ ships_, const void* __restrict__ ship_b_,
                                                     const void* __restrict__ planets_, const void* __restrict__ bullets_,
                                                     const uint32_t* __restrict__ meta_, const uint32_t* __restrict__ episode_,
                                                     const int32_t* __restrict__ index, int m, int n_games, int K, int k_out,
                                                     const __grid_constant__ GameArrays a) {
    using B4 = Body4<R>;
    const int row = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= m) return;
    const int g = index ? index[row] : row;
    if (g < 0 || g >= n_games) return;   // (checked on the host for host-side indices)
    const size_t tile = (size_t)(g >> 5);
    const int gl = g & 31;
    const uint32_t meta = meta_[g];
    const bool fin = ASTRO_META_FINISHED(meta);
    const int np = (int)meta_np<PL>(meta), nb = fin ? 0 : (int)ASTRO_META_NB(meta);
    if (lane < S) {
        const B4 v = reinterpret_cast<const B4*>(ships_)[tile * (S * 32) + lane * 32 + gl];
        double* o = a.ships + ((size_t)row * S + lane) * 5;
        o[0] = (double)v.x; o[1] = (double)v.y; o[2] = (double)v.dx; o[3] = (double)v.dy;
        o[4] = (double)reinterpret_cast<const R*>(ship_b_)[tile * (S * 32) + lane * 32 + gl];
    }
    if (lane < PL) {
        B4 v = B4();
        if (lane < np) v = reinterpret_cast<const B4*>(planets_)[tile * (PL * 32) + lane * 32 + gl];
        double* o = a.planets + ((size_t)row * PL + lane) * 4;
        o[0] = (double)v.x; o[1] = (double)v.y; o[2] = (double)v.dx; o[3] = (double)v.dy;
    }
    const unsigned first = tile_list_offset(meta_ + tile * 32, gl, lane);
    const B4* run = reinterpret_cast<const B4*>(bullets_) + tile * (size_t)(32 * K) + first;
    for (int k = lane; k < k_out; k += 32) {
        B4 v = B4();
        if (k < nb) v = run[k];
        double* o = a.bullets + ((size_t)row * k_out + k) * 4;
        o[0] = (double)v.x; o[1] = (double)v.y; o[2] = (double)v.dx; o[3] = (double)v.dy;
    }
    if (lane == 0) {
        a.n_planets[row] = np;
        a.n_bullets[row] = nb;
        a.tick[row] = (int32_t)meta_tick<PL>(meta);
        a.finished[row] = fin ? 1 : 0;
        if (a.episode) a.episode[row] = episode_[g];
    }
}

__global__ void import_map_kernel(const int32_t* __restrict__ index, int m, int n_games, int32_t* __restrict__ src) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const int g = index[i];
    if (g >= 0 && g < n_games) src[g] = i;
}

template <typename R, int S, int PL>
__global__ void __launch_bounds__(128) import_kernel(void* __restrict__ ships_, void* __restrict__ ship_b_, void* __restrict__ planets_,
                                                     void* bullets_cur_, void* bullets_other_, uint32_t* __restrict__ meta_,
                                                     uint32_t* __restrict__ episode_, const int32_t* __restrict__ src, int m,
                                                     int n_games, int K, int k_in, const __grid_constant__ GameArrays a) {
    using B4 = Body4<R>;
    const unsigned full = 0xffffffffu;
    const int tile_i = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (tile_i * 32 >= n_games) return;
    const int g = tile_i * 32 + lane;
    const int row = src ? src[g] : (g < m ? g : -1);          // src == NULL: rows 0..m-1 replace games 0..m-1
    if (!__ballot_sync(full, row >= 0)) return;
    const size_t tile = (size_t)tile_i;
    const uint32_t meta = meta_[g];
    const unsigned old_nb = ASTRO_META_FINISHED(meta) ? 0u : ASTRO_META_NB(meta);
    unsigned new_nb = old_nb;
    bool fin = false;
    if (row >= 0) {
        fin = a.finished && a.finished[row];
        const int want = a.n_bullets ? a.n_bullets[row] : 0;
        new_nb = fin ? 0u : (unsigned)min(max(want, 0), min(K, k_in));
    }
    const unsigned old_first = warp_exclusive_sum(old_nb, lane), new_first = warp_exclusive_sum(new_nb, lane);
    const unsigned new_total = __reduce_add_sync(full, new_nb);
    B4* const cur = reinterpret_cast<B4*>(bullets_cur_) + tile * (size_t)(32 * K);
    B4* const scratch = reinterpret_cast<B4*>(bullets_other_) + tile * (size_t)(32 * K);
    if (row >= 0) {
        const double* bsrc = a.bullets + (size_t)row * k_in * 4;
        for (unsigned k = 0; k < new_nb; k++) {
            B4 v;
            v.x = (R)bsrc[4 * k]; v.y = (R)bsrc[4 * k + 1]; v.dx = (R)bsrc[4 * k + 2]; v.dy = (R)bsrc[4 * k + 3];
            scratch[new_first + k] = v;
        }
    } else {
        for (unsigned k = 0; k < new_nb; k++) scratch[new_first + k] = cur[old_first + k];
    }
    __syncwarp();
    for (unsigned j = lane; j < new_total; j += 32u) cur[j] = scratch[j];
    if (row >= 0) {
        const int np = min(max(a.n_planets[row], 0), PL);
#pragma unroll
        for (int s = 0; s < S; s++) {
            const double* o = a.ships + ((size_t)row * S + s) * 5;
            B4 v;
            v.x = (R)o[0]; v.y = (R)o[1]; v.dx = (R)o[2]; v.dy = (R)o[3];
            reinterpret_cast<B4*>(ships_)[tile * (S * 32) + s * 32 + lane] = v;
            reinterpret_cast<R*>(ship_b_)[tile * (S * 32) + s * 32 + lane] = (R)o[4];
        }
#pragma unroll
        for (int j = 0; j < PL; j++) {
            const double* o = a.planets + ((size_t)row * PL + j) * 4;
            B4 v = B4();
            if (j < np) { v.x = (R)o[0]; v.y = (R)o[1]; v.dx = (R)o[2]; v.dy = (R)o[3]; }
            reinterpret_cast<B4*>(planets_)[tile * (PL * 32) + j * 32 + lane] = v;
        }
        const uint32_t tick = a.tick ? (uint32_t)a.tick[row] : 0u;
        meta_[g] = meta_pack<PL>(new_nb, np, fin ? 1 : 0, tick);
        if (a.episode) episode_[g] = a.episode[row];
    }
}

// ------------------------------------------------------------------------------------------
// nstep_kernel: the n-step replay ingestion of rl.QBotTrainer.reward (rl.py:303-328) for every bot of every game over a
// window of T logged ticks — thread = one bot (game, ship).  The reference keeps, per bot, the (features, action) pairs
// since the last flush and, when the game ends or n_steps pairs are held, turns pair number n of L into
//     Experience(state_f, action, reward * d, discount * d, new_state_f)     d = discount ** (L - 1 - n)
// with `reward` the reward of the flushing tick (only terminal ticks have one) and new_state_f = None when the game
// ended.  Here an entry is identified by its tick (the observation taken before that tick); rows 0 .. H-1 of the outputs
// stand for the H = n_steps ticks before the window (entries a bot still held when the window began: `carry`), row
// H + t for tick t.  Per entry: reward * d, discount * d (float32) and `next` = the tick whose observation is the new
// state (window-relative, t_flush + 1), -1 = terminal (no new state), -2 = still held when the window ends (it comes
// back as a carried entry of the next window), -3 = no entry (the game was finished and skipped that tick).
// ------------------------------------------------------------------------------------------
template <int S>
__global__ void __launch_bounds__(128) nstep_kernel(const uint8_t* __restrict__ events, int T, int n_games, int n_steps, double discount,
                                                    float reward_timeout, int32_t* __restrict__ carry, float* __restrict__ out_reward,
                                                    float* __restrict__ out_discount, int32_t* __restrict__ out_next) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n_games * S) return;
    const int g = idx / S, me = idx % S;
    const int H = n_steps;
    const size_t stride = (size_t)n_games * S;
    int L = min(max(carry[idx], 0), n_steps - 1);
    int seg_start = -L;                                    // first held entry, as a window-relative tick
    for (int r = 0; r < H - L; r++) out_next[(size_t)r * stride + idx] = -3;       // history rows this bot does not hold
    for (int t = 0; t < T; t++) {
        const uint32_t ev = events[(size_t)t * n_games + g];
        if (ev & ASTRO_EV_SKIPPED) {                       // no step was taken: no entry; the bot holds nothing (its game is over)
            out_next[(size_t)(H + t) * stride + idx] = -3;
            seg_start = t + 1;
            continue;
        }
        L = t - seg_start + 1;
        const bool term = (ev & ASTRO_EV_DONE_MASK) != 0;
        if (term || L >= n_steps) {
            double reward = 0.0;
            if (ev & (ASTRO_EV_HIT0 | ASTRO_EV_HIT1)) reward = ((ev >> me) & 1u) ? -1.0 : 1.0;     // core.py:255
            else if (ev & ASTRO_EV_TIMEOUT) reward = (double)reward_timeout;                        // core.py:260
            for (int n = seg_start; n <= t; n++) {
                const double d = pow(discount, (double)(t - n));
                const size_t row = (size_t)(H + n) * stride + idx;
                out_reward[row] = (float)(reward * d);
                out_discount[row] = (float)(discount * d);
                out_next[row] = term ? -1 : t + 1;
            }
            seg_start = t + 1;
        }
    }
    for (int n = seg_start; n < T; n++) out_next[(size_t)(H + n) * stride + idx] = -2;
    carry[idx] = T - seg_start > 0 ? T - seg_start : 0;
    // (held entries that began before the window and are still held: the window was shorter than n_steps)
    for (int n = seg_start; n < 0; n++) out_next[(size_t)(H + n) * stride + idx] = -2;
}

// the device-resident stream step of captured bot-loop chunks (astro_rollout_device)
__global__ void step_base_set_kernel(uint32_t* p, uint32_t v) { *p = v; }
__global__ void step_base_add_kernel(uint32_t* p, uint32_t v) { *p += v; }

// ------------------------------------------------------------------------------------------
// host side of the C ABI
// ------------------------------------------------------------------------------------------
thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CUDA_TRY(expr)                                                                              \
    do {                                                                                            \
        cudaError_t e_ = (expr);                                                                    \
        if (e_ != cudaSuccess) return fail(ASTRO_E_CUDA, "%s: %s", #expr, cudaGetErrorString(e_)); \
    } while (0)

}  // namespace

// numpy's legacy RandomState(seed) word stream (MT19937, init_genrand seeding) on the host: core.generate_configs
// (core.py:77-83) draws one randint(2**30) per config = one 32-bit word masked to 30 bits (a power-of-two range: the
// masked rejection never rejects).
struct HostMt19937 {
    uint32_t mt[624];
    int idx;
    void seed(uint32_t s) {
        mt[0] = s;
        for (int i = 1; i < 624; i++) mt[i] = 1812433253u * (mt[i - 1] ^ (mt[i - 1] >> 30)) + (uint32_t)i;
        idx = 624;
    }
    static uint32_t twist(uint32_t a, uint32_t b, uint32_t far) {
        const uint32_t y = (a & 0x80000000u) | (b & 0x7fffffffu);
        return far ^ (y >> 1) ^ ((0u - (y & 1u)) & 0x9908b0dfu);
    }
    uint32_t next() {
        if (idx >= 624) {      // the three runs of the reference generator: no modulo in the loops
            int k = 0;
            for (; k < 624 - 397; k++) mt[k] = twist(mt[k], mt[k + 1], mt[k + 397]);
            for (; k < 623; k++) mt[k] = twist(mt[k], mt[k + 1], mt[k + 397 - 624]);
            mt[623] = twist(mt[623], mt[0], mt[396]);
            idx = 0;
        }
        uint32_t v = mt[idx++];
        v ^= v >> 11;
        v ^= (v << 7) & 0x9d2c5680u;
        v ^= (v << 15) & 0xefc60000u;
        v ^= v >> 18;
        return v;
    }
};

constexpr int kFreshLead = 3;     // refills the host may run ahead of the device
struct FreshState {
    FreshParams f;                // device pointers (ring, tile_used, tasks, cursor, seeds)
    CreateParams cq;
    uint32_t* game_pos;           // device [n_games]
    uint32_t* chunk_base;         // device [n_tiles / 32]: first task of each chunk of 32 tiles (refill plan)
    uint32_t* h_seeds;            // pinned mirror of the seed ring
    unsigned long long* h_cursor; // pinned: [0] stream positions handed out, [1] refills completed (lagging copies)
    HostMt19937 mt;               // (owned by the producer thread once it runs)
    // A producer thread keeps the pinned mirror topped up so that drawing seeds (a few ns each, ~10 k per tick and million
    // games) never sits in front of a launch: it draws positions [produced, target) in chunks; the caller raises
    // `target` one refill ahead and only ever waits when it has overtaken the forecast.
    std::thread* producer;
    std::atomic<unsigned long long> produced, target;
    std::atomic<int> stop;
    unsigned long long generated; // stream positions uploaded to the device so far
    unsigned long long refills;   // refills enqueued so far
    cudaEvent_t done[kFreshLead]; // refill k's completion = done[k % kFreshLead]
    cudaStream_t copy;            // seed uploads
    cudaEvent_t seeds_sent;
    int64_t ticks_since_refill;
    int64_t capacity;             // n_tiles * quota
};

struct LoopGraph {        // a captured chunk of the bot loop (astro_rollout_device)
    cudaGraphExec_t exec;
    int32_t modes[2], flags, cur;
    double avoid_distance, avoid_threshold;
    uint8_t* actions;
    uint8_t* events;
    AstroRecordRing rec;  // the recording ring the chunk writes (its row is read from the device step word, not captured)
    int64_t epoch;
    int32_t launches;     // kernels of one replay
};
constexpr int kLoopChunk = 16;   // ticks per captured chunk (even: the bullet buffers are back where they started)

struct SingleGraph {      // a captured single-game step (astro_step_single_host)
    cudaGraphExec_t exec;
    const void* in;
    void* out;
    int32_t flags;
};
constexpr int kSingleGraphs = 4;

struct AstroBatch {
    AstroConfig cfg;
    int32_t n_games, K, precision, device, S;
    int32_t PL;              // planet slots per game: ASTRO_MAX_PLANETS or ASTRO_MAX_PLANETS_WIDE (AstroConfig.planet_slots)
    bool bound;
    AstroBuffers bufs;
    AstroResetPool pool;
    uint32_t* d_fire_bits;
    int32_t n_sched_ticks, timeout_tick;
    int32_t sm_count;
    unsigned long long* d_stats;   // [kStatReplicas][16]
    // astro_stats_allreduce: this rank's exchange buffer, the peers' (IPC-mapped) and the call counter
    unsigned long long* d_peer_own;
    PeerTable peer_table;
    int32_t peer_rank, peer_world;
    bool peer_open;
    unsigned long long peer_calls;
    unsigned* d_stat_slots;  // per-warp partial counters, folded by astro_stats
    int32_t cur;             // which of the two bullet buffers holds the lists (flips every tick)
    float4* d_pool_rec;      // precision 32: packed copy of the reset pool (astro_set_reset_pool)
    int64_t ticks_since_fold;
    uint8_t* d_actions;  // staging for astro_tick_host
    uint8_t* d_events;
    // astro_rollout_host: double-buffered staging, copy streams and ordering events (created lazily)
    uint8_t* d_actions2[2];
    uint8_t* d_events2[2];
    cudaStream_t copy_in, copy_out;
    cudaEvent_t ev_in[2], ev_tick[2], ev_out[2];
    bool pipe_ready;
    // astro_tick_host: the tick cut into slices of tiles, one stream per slice (created lazily)
    // astro_rollout_device: the bot loop captured as a CUDA graph of kLoopChunk ticks (see there)
    LoopGraph loop_graph[2];
    uint32_t* d_step_base;        // device word: the stream step at the start of the chunk being replayed
    const uint32_t* step_base_now;// = d_step_base while a chunk is being captured, else NULL
    cudaStream_t loop_stream;
    cudaEvent_t loop_in, loop_out;
    int64_t config_epoch;         // bumped by every call that changes what a captured chunk depends on
    int32_t bot_modes_now;        // != 0 while astro_rollout_device runs ticks whose bots are evaluated inside the tick kernel
    AstroRecordRing rec_now;      // astro_rollout_device_record: the ring of the running call (events == NULL: none)
    ScriptParams script_now;
    // fresh-game mode (astro_fresh_games_enable): per-tile rings of pre-created games fed from the generate_configs stream
    FreshState* fresh;
    cudaEvent_t ev_host_done;   // astro_tick_host_begin / _end
    bool host_pending;
    cudaStream_t slice_stream[8];
    cudaEvent_t ev_slice_start;
    bool slice_ready;
    int32_t pipe_chunk;      // ticks per copy of astro_rollout_host
    uint8_t* d_done;
    float* d_reward;
    uint32_t seed, step;
    int64_t first_game;
    int64_t launches;
    int32_t policy_nout;  // > 0 once astro_policy_set_weights has been called
    PolicyFragWeights* d_pol_frags;   // this batch's network as tensor-core B fragments (astro_policy_set_weights)
    int32_t* d_src;       // astro_import_games: game -> row map
    char* d_single;       // astro_step_single_host: device staging, in record then out record
    int64_t single_bytes;
    cudaStream_t single_stream;
    cudaEvent_t single_event;
    SingleGraph single_graph[4];
    int32_t single_next;
    double explore_t_in, explore_t_out;   // astro_set_exploration (ASTRO_BOT_EXPLORE)
    uint32_t explore_seed;
    int32_t* explore_state;
    Consts c;
};

namespace {

void fill_consts(const AstroConfig& cfg, Consts& c) {
    // Python-float expressions of the reference, evaluated once in float64
    c.gm = cfg.gravity * cfg.planet_mass;
    c.dt = cfg.dt;
    c.thrust = cfg.ship_thrust;
    c.db_unit = cfg.dt * cfg.ship_rspeed;
    c.zero_dt = 0.0 * cfg.dt;
    const double rs = cfg.ship_radius, rp = cfg.planet_radius;
    c.r2_ss = (rs + rs) * (rs + rs);
    c.r2_sp = (rp + rs) * (rp + rs);
    c.r2_sb = (0.0 + rs) * (0.0 + rs);
    c.r2_pb = (0.0 + rp) * (0.0 + rp);
    c.off_f = (float)(1.001 * cfg.ship_radius);
    c.spd_f = (float)cfg.bullet_speed;
    c.gm_f = (float)c.gm;
    c.dt_f = (float)c.dt;
    c.thrust_f = (float)c.thrust;
    c.db_unit_f = (float)c.db_unit;
    c.r2f_ss = (float)c.r2_ss;
    c.r2f_sp = (float)c.r2_sp;
    c.r2f_sb = (float)c.r2_sb;
    c.r2f_pb = (float)c.r2_pb;
    c.reward_timeout = cfg.solo ? 1.0f : 0.0f;
}

int check(const AstroBatch* b, bool need_bound) {
    if (!b) return fail(ASTRO_E_INVALID, "null batch handle");
    if (need_bound && !b->bound) return fail(ASTRO_E_STATE, "astro_batch_bind has not been called");
    return ASTRO_OK;
}

// Bullet-list buffer `which` of the two: b->cur holds the lists, the other one is where the next tick writes them.
void* bullet_buffer(const AstroBatch* b, int which) {
    const size_t buf_bytes = (size_t)b->n_games * b->K * 4 * (b->precision == 32 ? sizeof(float) : sizeof(double));
    return (char*)b->bufs.bullets + (size_t)which * buf_bytes;
}

template <typename T> struct TypeTag { using type = T; };
template <int N> using IntTag = std::integral_constant<int, N>;

// The batch's layout as kernel template arguments: calls f(TypeTag<R>, IntTag<S>, IntTag<PL>) for the batch's precision,
// ships per game and planet slots, and returns what f returns.
template <typename F>
auto with_layout(const AstroBatch* b, F&& f) {
    auto by_pl = [&](auto r, auto s) {
        return b->PL == ASTRO_MAX_PLANETS_WIDE ? f(r, s, IntTag<ASTRO_MAX_PLANETS_WIDE>()) : f(r, s, IntTag<ASTRO_MAX_PLANETS>());
    };
    auto by_s = [&](auto r) { return b->S == 2 ? by_pl(r, IntTag<2>()) : by_pl(r, IntTag<1>()); };
    return b->precision == 32 ? by_s(TypeTag<float>()) : by_s(TypeTag<double>());
}

void fill_params(const AstroBatch* b, TickParams& p) {
    memset(&p, 0, sizeof(p));
    p.ships = b->bufs.ships;
    p.ship_b = b->bufs.ship_b;
    p.planets = b->bufs.planets;
    p.bullets_in = bullet_buffer(b, b->cur);
    p.bullets_out = bullet_buffer(b, b->cur ^ 1);
    p.meta = b->bufs.meta;
    p.episode = b->bufs.episode;
    p.fire_bits = b->d_fire_bits;
    p.pool_ships = b->pool.ships;
    p.pool_planets = b->pool.planets;
    p.pool_np = b->pool.np;
    p.pool_size = b->pool.size;
    p.pool_rec = b->d_pool_rec;
    p.stats = b->d_stats;
    p.stat_slots = b->d_stat_slots;
    p.n_games = b->n_games;
    p.K = b->K;
    p.timeout_tick = b->timeout_tick;
    p.n_sched_ticks = b->n_sched_ticks;
    if (b->fresh) {
        p.ring = b->fresh->f.ring;
        p.tile_used = b->fresh->f.tile_used;
        p.game_pos = b->fresh->game_pos;
        p.quota = b->fresh->f.quota;
    }
    p.seed = b->seed;
    p.step = b->step;
    p.step_base = b->step_base_now;
    p.first_game = (uint32_t)b->first_game;
    p.c = b->c;
    if (b->rec_now.events) {
        p.rec_controls = b->rec_now.controls;
        p.rec_events = b->rec_now.events;
        p.rec_ticks = (uint32_t)b->rec_now.ticks;
    }
}

template <typename R, int S, int PL>
cudaError_t launch_tick(const TickParams& p, cudaStream_t st) {
    const int grid = (p.n_games + kTickThreads - 1) / kTickThreads;
    if (p.flags & ASTRO_TICK_NO_STATS)
        tick_kernel<R, S, false, PL><<<grid, kTickThreads, 0, st>>>(p);
    else
        tick_kernel<R, S, true, PL><<<grid, kTickThreads, 0, st>>>(p);
    return cudaGetLastError();
}

template <int S>
cudaError_t launch_tick_f32(const TickParams& p, cudaStream_t st) {
    const int grid = (p.tiles * 32 + kTickThreads - 1) / kTickThreads;
    // experiment knob (tools/exp_tick.py): unused dynamic shared memory caps the resident CTAs per SM
    static const size_t extra = getenv("ASTRO_EXTRA_SMEM") ? (size_t)atoi(getenv("ASTRO_EXTRA_SMEM")) : 0;
    // The production rollout's options — duel games, packed controls in, event planes out, no reward / done arrays, auto-reset
    // from the pool — have instantiations of their own (tick_f32.cuh, FIX) in which those options are compile-time constants:
    // 56.4 against 60.8 us per tick at 20 ticks per launch (same box).  ASTRO_TICK_NO_FIX=1: the generic instantiations (A/B).
    static const bool no_fix = getenv("ASTRO_TICK_NO_FIX") && atoi(getenv("ASTRO_TICK_NO_FIX")) != 0;
    const bool fix = S == 2 && !no_fix && !p.bot_modes && p.actions && p.events && !p.reward && !p.done && !p.ring && !p.step_base && !p.game_pos && !p.rec_events && p.pool_size > 0 &&
                     (p.flags & (ASTRO_TICK_PACKED_CONTROLS | ASTRO_TICK_EVENT_PLANES | ASTRO_TICK_AUTO_RESET)) ==
                         (ASTRO_TICK_PACKED_CONTROLS | ASTRO_TICK_EVENT_PLANES | ASTRO_TICK_AUTO_RESET) && !(p.flags & 1024);
    if (p.bot_modes) {              // bots inside the tick: the many-tick form, whatever n_fused
        if (p.flags & ASTRO_TICK_NO_STATS) tick_f32_kernel<S, false, true, true><<<grid, kTickThreads, extra, st>>>(p);
        else tick_f32_kernel<S, true, true, true><<<grid, kTickThreads, extra, st>>>(p);
    } else if (p.n_fused > 1) {
        if (fix) {
            if (p.flags & ASTRO_TICK_NO_STATS) tick_f32_kernel<2, false, true, false, true><<<grid, kTickThreads, extra, st>>>(p);
            else tick_f32_kernel<2, true, true, false, true><<<grid, kTickThreads, extra, st>>>(p);
        } else if (p.flags & ASTRO_TICK_NO_STATS) tick_f32_kernel<S, false, true><<<grid, kTickThreads, extra, st>>>(p);
        else tick_f32_kernel<S, true, true><<<grid, kTickThreads, extra, st>>>(p);
    } else {
#if ASTRO_PDL
        // Programmatic dependent launch: the CTAs of this tick become resident while the previous kernel of the stream
        // drains and wait (griddepcontrol.wait, first thing in the kernel) for it to complete and flush.
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)grid);
        cfg.blockDim = dim3((unsigned)kTickThreads);
        cfg.dynamicSmemBytes = extra;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        if (fix) {
            if (p.flags & ASTRO_TICK_NO_STATS) return cudaLaunchKernelEx(&cfg, tick_f32_kernel<2, false, false, false, true>, p);
            return cudaLaunchKernelEx(&cfg, tick_f32_kernel<2, true, false, false, true>, p);
        }
        if (p.flags & ASTRO_TICK_NO_STATS) return cudaLaunchKernelEx(&cfg, tick_f32_kernel<S, false, false>, p);
        return cudaLaunchKernelEx(&cfg, tick_f32_kernel<S, true, false>, p);
#else
        if (fix) {
            if (p.flags & ASTRO_TICK_NO_STATS) tick_f32_kernel<2, false, false, false, true><<<grid, kTickThreads, extra, st>>>(p);
            else tick_f32_kernel<2, true, false, false, true><<<grid, kTickThreads, extra, st>>>(p);
        } else if (p.flags & ASTRO_TICK_NO_STATS) tick_f32_kernel<S, false, false><<<grid, kTickThreads, extra, st>>>(p);
        else tick_f32_kernel<S, true, false><<<grid, kTickThreads, extra, st>>>(p);
#endif
    }
    return cudaGetLastError();
}

// 8 planet slots: the generic instantiations, one tick or several per launch.  The FIX and BOT forms exist for 4 slots only
// (astro_rollout_device runs ScriptBots of 8-slot batches as bot kernel -> tick kernel).
template <int S>
cudaError_t launch_tick_f32_wide(const TickParams& p, cudaStream_t st) {
    const int grid = (p.tiles * 32 + kTickThreads - 1) / kTickThreads;
    if (p.n_fused > 1) {
        if (p.flags & ASTRO_TICK_NO_STATS) tick_f32_wide_kernel<S, false, true><<<grid, kTickThreads, 0, st>>>(p);
        else tick_f32_wide_kernel<S, true, true><<<grid, kTickThreads, 0, st>>>(p);
    } else {
        if (p.flags & ASTRO_TICK_NO_STATS) tick_f32_wide_kernel<S, false, false><<<grid, kTickThreads, 0, st>>>(p);
        else tick_f32_wide_kernel<S, true, false><<<grid, kTickThreads, 0, st>>>(p);
    }
    return cudaGetLastError();
}

cudaError_t fold_stats(AstroBatch* b, cudaStream_t st) {
    fold_stats_kernel<<<64, 256, 0, st>>>(b->d_stat_slots, b->n_games / ASTRO_TILE, b->d_stats);
    b->ticks_since_fold = 0;
    b->launches += 1;
    return cudaGetLastError();
}

// n_ticks consecutive ticks.  actions [n_ticks][n_games][S] (or NULL: counter stream), reward / done / events
// [n_ticks][...] (or NULL).  The production fp32 kernel runs up to kMaxFused of them per launch, each tile
// back to back (tick_f32_kernel); the generic / float64 kernels run one launch per tick.
constexpr int kMaxFused = 256;
constexpr int kMaxSlices = 8;
constexpr double kSinCosRange = 71476.0;   // np_sincos_f32 (astro_device.cuh)
// ---- fresh-game mode: the host side of the seed stream and the refill ---------------------------------------------
// Stream positions [generated, upto) are drawn from the host MT19937 into the pinned mirror ring and uploaded
// (stream-ordered) to the device ring.  A slot is overwritten ring-size positions later: the refill protocol keeps
// `generated` within kFreshLead + 1 capacities of the device's cursor, and the ring holds 2 (kFreshLead + 2) capacities.
void fresh_producer_main(FreshState* fs) {
    for (;;) {
        const unsigned long long want = fs->target.load(std::memory_order_acquire);
        unsigned long long have = fs->produced.load(std::memory_order_relaxed);
        if (fs->stop.load(std::memory_order_acquire)) return;
        if (have >= want) { std::this_thread::sleep_for(std::chrono::microseconds(50)); continue; }   // (works a refill ahead: no hurry)
        const unsigned long long n = want - have < 16384ull ? want - have : 16384ull;
        for (unsigned long long i = 0; i < n; i++) fs->h_seeds[(have + i) & fs->f.seed_mask] = fs->mt.next() & 0x3fffffffu;   // randint(2**30)
        fs->produced.store(have + n, std::memory_order_release);
    }
}

int fresh_upload_seeds(AstroBatch* b, unsigned long long upto, cudaStream_t st) {
    FreshState* fs = b->fresh;
    if (fs->generated >= upto) return ASTRO_OK;
    const unsigned long long ring = (unsigned long long)fs->f.seed_mask + 1ull;
    if (fs->target.load(std::memory_order_relaxed) < upto) fs->target.store(upto, std::memory_order_release);
    while (fs->produced.load(std::memory_order_acquire) < upto) std::this_thread::yield();    // (normally already there)
    while (fs->generated < upto) {
        const unsigned long long at = fs->generated & fs->f.seed_mask;
        unsigned long long n = upto - fs->generated;
        if (n > ring - at) n = ring - at;
        CUDA_TRY(cudaMemcpyAsync(const_cast<uint32_t*>(fs->f.seeds) + at, fs->h_seeds + at, (size_t)n * sizeof(uint32_t),
                                 cudaMemcpyHostToDevice, st));
        fs->generated += n;
    }
    return ASTRO_OK;
}

// One refill: every record used since the last one is re-created from the next positions of the stream.
int fresh_refill(AstroBatch* b, cudaStream_t st) {
    FreshState* fs = b->fresh;
    // the host runs at most kFreshLead refills ahead of the device: the cursor it reads below is then at most that stale
    if (fs->refills >= (unsigned long long)kFreshLead) CUDA_TRY(cudaEventSynchronize(fs->done[fs->refills % kFreshLead]));
    const unsigned long long cursor_seen = fs->h_cursor[0], refills_seen = fs->h_cursor[1];
    // every refill not yet seen hands out at most `capacity` positions, and so does this one
    const unsigned long long bound = cursor_seen + (fs->refills - refills_seen + 1ull) * (unsigned long long)fs->capacity;
    // The seeds travel on a copy stream of their own, ONE refill ahead of need (what this refill may use was sent during the
    // previous one), so the copy runs beside the tick launches instead of in front of the refill kernels.
    CUDA_TRY(cudaStreamWaitEvent(st, fs->seeds_sent, 0));                       // the previous upload (long complete)
    if (int r = fresh_upload_seeds(b, bound, st)) return r;                     // (only if the device got ahead of the forecast)
    if (int r = fresh_upload_seeds(b, bound + (unsigned long long)fs->capacity, fs->copy)) return r;
    CUDA_TRY(cudaEventRecord(fs->seeds_sent, fs->copy));
    // ... and the producer draws what the NEXT refill will upload while this launch runs
    fs->target.store(bound + 2ull * (unsigned long long)fs->capacity, std::memory_order_release);
    refill_scan_kernel<<<1, 1024, 0, st>>>(fs->f, fs->chunk_base);
    refill_tasks_kernel<<<(fs->f.n_tiles + 255) / 256, 256, 0, st>>>(fs->f, fs->chunk_base);
    const int grid = (int)std::min<int64_t>((fs->capacity + 63) / 64, (int64_t)b->sm_count * 32);
    if (b->S == 2) refill_create_kernel<2><<<grid, 64, 0, st>>>(fs->f, fs->cq);
    else refill_create_kernel<1><<<grid, 64, 0, st>>>(fs->f, fs->cq);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(fs->h_cursor, fs->f.cursor, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaEventRecord(fs->done[fs->refills % kFreshLead], st));
    fs->refills += 1;
    fs->ticks_since_refill = 0;
    b->launches += 3;
    return ASTRO_OK;
}

// bytes of one tick's controls / events in the form `flags` selects (include/astro_b200.h)
size_t actions_bytes(const AstroBatch* b, int32_t flags) {
    return (flags & ASTRO_TICK_PACKED_CONTROLS) && b->S == 2 ? (size_t)b->n_games : (size_t)b->n_games * b->S;
}
size_t events_bytes(const AstroBatch* b, int32_t flags) {
    return (flags & ASTRO_TICK_EVENT_PLANES) ? (size_t)(b->n_games / ASTRO_TILE) * 12 : (size_t)b->n_games;
}

// (tile0, tiles): the float32 kernel can run a launch over a sub-range of tiles (astro_tick_host slices a tick so that
// the copies of one slice overlap the kernel of another); tiles = 0: the whole batch.  A sliced call advances the
// stream step and flips the bullet buffers only with its LAST slice (`advance`).
int do_ticks(AstroBatch* b, const uint8_t* actions, float* reward, uint8_t* done, uint8_t* events, int32_t flags,
             cudaStream_t st, int32_t n_ticks, int32_t tile0 = 0, int32_t tiles = 0, bool advance = true) {
    if (b->n_sched_ticks <= 0) return fail(ASTRO_E_STATE, "astro_set_schedule has not been called");
    if ((flags & ASTRO_TICK_PACKED_CONTROLS) && b->S != 2) return fail(ASTRO_E_INVALID, "ASTRO_TICK_PACKED_CONTROLS is for duel games");
    if ((flags & ASTRO_TICK_AUTO_RESET) && b->pool.size <= 0 && !b->fresh)
        return fail(ASTRO_E_STATE, "ASTRO_TICK_AUTO_RESET needs astro_set_reset_pool or astro_fresh_games_enable");
    const bool fused = b->precision == 32 && !(flags & ASTRO_TICK_GENERIC_KERNEL);
    if (b->fresh && (flags & ASTRO_TICK_AUTO_RESET) && !fused)
        return fail(ASTRO_E_INVALID, "fresh-game mode re-creates games in the float32 production kernel only");
    const size_t n = (size_t)b->n_games;
    for (int32_t k0 = 0; k0 < n_ticks;) {
        const int32_t kc = fused ? (n_ticks - k0 < kMaxFused ? n_ticks - k0 : kMaxFused) : 1;
        if (b->fresh && (flags & ASTRO_TICK_AUTO_RESET) && advance && !b->step_base_now) {
            // top the tiles' rings up once the ticks since the last refill, plus this launch, exceed half a quota (a tile
            // loses ~0.3 games per tick under random play: ~15 % of its records by then)
            FreshState* fs = b->fresh;
            if (fs->ticks_since_refill > 0 && (fs->ticks_since_refill + kc) * 2 > fs->f.quota)
                if (int r = fresh_refill(b, st)) return r;
            fs->ticks_since_refill += kc;
        }
        TickParams p;
        fill_params(b, p);
        const uint32_t a_bytes = (uint32_t)actions_bytes(b, flags), e_bytes = (uint32_t)events_bytes(b, flags);
        p.actions = actions ? actions + (size_t)k0 * a_bytes : nullptr;
        p.reward = reward ? reward + (size_t)k0 * n * b->S : nullptr;
        p.done = done ? done + (size_t)k0 * n : nullptr;
        p.events = events ? events + (size_t)k0 * e_bytes : nullptr;
        p.act_stride = actions ? a_bytes : 0u;           // (a null array stays null when the kernel advances it)
        p.ev_stride = events ? e_bytes : 0u;
        p.rw_stride = reward ? (uint32_t)(n * b->S * sizeof(float)) : 0u;
        p.done_stride = done ? (uint32_t)n : 0u;
        p.flags = flags;
        p.n_fused = kc;
        p.tile0 = tile0;
        p.tiles = tiles > 0 ? tiles : b->n_games / ASTRO_TILE;
        if (fused && !actions && b->bot_modes_now) {
            p.bot_modes = b->bot_modes_now;
            p.script = b->script_now;
        }
        const cudaError_t e = with_layout(b, [&](auto r, auto s, auto pl) {
            if (fused) {                                     // (float32 batches only)
                if constexpr (pl == ASTRO_MAX_PLANETS) return launch_tick_f32<s>(p, st);
                else return launch_tick_f32_wide<s>(p, st);
            }
            return launch_tick<typename decltype(r)::type, s, pl>(p, st);
        });
        if (e != cudaSuccess) return fail(ASTRO_E_CUDA, "tick_kernel launch: %s", cudaGetErrorString(e));
        b->launches += 1;
        k0 += kc;
        if (!advance) continue;
        b->step += (uint32_t)kc;
        b->cur ^= kc & 1;   // the lists now live in the buffer the last tick wrote
        // 32-bit slot rows: fold long before a row can wrap (<= 32 * 1023 per tick)
        // (launches of >= 8 ticks add their totals straight to the 64-bit counters: nothing to fold)
        if (!(flags & ASTRO_TICK_NO_STATS) && !(fused && kc >= 8) && (b->ticks_since_fold += kc) >= 65536) {
            cudaError_t fe = fold_stats(b, st);
            if (fe != cudaSuccess) return fail(ASTRO_E_CUDA, "fold_stats_kernel launch: %s", cudaGetErrorString(fe));
        }
    }
    return ASTRO_OK;
}
int do_tick(AstroBatch* b, const uint8_t* actions, float* reward, uint8_t* done, uint8_t* events, int32_t flags,
            cudaStream_t st) {
    return do_ticks(b, actions, reward, done, events, flags, st, 1);
}

}  // namespace

extern "C" {

int astro_abi_version(void) { return ASTRO_ABI_VERSION; }

const char* astro_last_error(void) { return g_err; }

int astro_batch_create(const AstroConfig* cfg, int32_t n_games, int32_t bullet_cap, int32_t precision,
                       int32_t device, AstroBatch** out) {
    if (!cfg || !out) return fail(ASTRO_E_INVALID, "null argument");
    if (n_games <= 0 || n_games % ASTRO_TILE) return fail(ASTRO_E_INVALID, "n_games must be a positive multiple of %d", ASTRO_TILE);
    if (bullet_cap < 0 || bullet_cap > ASTRO_MAX_BULLET_CAP) return fail(ASTRO_E_INVALID, "bullet_cap out of range 0..%d", ASTRO_MAX_BULLET_CAP);
    if (precision != 32 && precision != 64) return fail(ASTRO_E_INVALID, "precision must be 32 or 64");
    if (cfg->planet_slots != 0 && cfg->planet_slots != ASTRO_MAX_PLANETS && cfg->planet_slots != ASTRO_MAX_PLANETS_WIDE)
        return fail(ASTRO_E_INVALID, "planet_slots must be 0 or %d (games of up to %d planets) or %d (up to %d planets), got %d",
                    ASTRO_MAX_PLANETS, ASTRO_MAX_PLANETS, ASTRO_MAX_PLANETS_WIDE, ASTRO_MAX_PLANETS_WIDE, cfg->planet_slots);
    if ((int64_t)n_games * bullet_cap >= (int64_t)1 << 31)
        return fail(ASTRO_E_INVALID, "n_games * bullet_cap must stay below 2^31 bullet slots per batch (32-bit slot indexing)");
    int count = 0;
    CUDA_TRY(cudaGetDeviceCount(&count));
    if (device < 0 || device >= count) return fail(ASTRO_E_INVALID, "device %d out of range (%d visible)", device, count);
    CUDA_TRY(cudaSetDevice(device));
    // The tick touches short runs (a game's live bullets, a tile row's live planet slots): ask L2
    // not to widen each miss to 64 bytes.  A hint; harmless where unsupported.
    if (const char* gran = getenv("ASTRO_L2_FETCH_GRANULARITY")) cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)atoi(gran));
    AstroBatch* b = new (std::nothrow) AstroBatch();
    if (!b) return fail(ASTRO_E_NOMEM, "out of host memory");
    memset(b, 0, sizeof(*b));
    b->cfg = *cfg;
    b->n_games = n_games;
    b->K = bullet_cap;
    b->precision = precision;
    b->device = device;
    b->S = cfg->solo ? 1 : 2;
    b->PL = cfg->planet_slots == ASTRO_MAX_PLANETS_WIDE ? ASTRO_MAX_PLANETS_WIDE : ASTRO_MAX_PLANETS;
    fill_consts(*cfg, b->c);
    if (cudaDeviceGetAttribute(&b->sm_count, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || b->sm_count <= 0) b->sm_count = 148;
    cudaError_t e = cudaMalloc(&b->d_stats, sizeof(unsigned long long) * 16 * kStatReplicas);
    if (e == cudaSuccess) e = cudaMemset(b->d_stats, 0, sizeof(unsigned long long) * 16 * kStatReplicas);
    const size_t slot_bytes = (size_t)(n_games / ASTRO_TILE) * 16 * sizeof(unsigned);
    if (e == cudaSuccess) e = cudaMalloc(&b->d_stat_slots, slot_bytes);
    if (e == cudaSuccess) e = cudaMemset(b->d_stat_slots, 0, slot_bytes);
    if (e == cudaSuccess) e = cudaMalloc(&b->d_actions, (size_t)n_games * b->S);
    if (e == cudaSuccess) e = cudaMalloc(&b->d_events, (size_t)n_games);
    if (e == cudaSuccess) e = cudaMalloc(&b->d_done, (size_t)n_games);
    if (e == cudaSuccess) e = cudaMalloc(&b->d_reward, sizeof(float) * (size_t)n_games * b->S);
    if (e != cudaSuccess) {
        astro_batch_destroy(b);
        return fail(ASTRO_E_CUDA, "cudaMalloc: %s", cudaGetErrorString(e));
    }
    *out = b;
    return ASTRO_OK;
}

static void fresh_free(AstroBatch* b);

int astro_batch_destroy(AstroBatch* b) {
    if (!b) return ASTRO_OK;
    cudaSetDevice(b->device);
    cudaFree(b->d_stats);
    if (b->peer_open)
        for (int r = 0; r < b->peer_world; r++)
            if (r != b->peer_rank && b->peer_table.buf[r]) cudaIpcCloseMemHandle(b->peer_table.buf[r]);
    cudaFree(b->d_peer_own);
    cudaFree(b->d_stat_slots);
    cudaFree(b->d_actions);
    cudaFree(b->d_events);
    cudaFree(b->d_done);
    cudaFree(b->d_reward);
    cudaFree(b->d_fire_bits);
    cudaFree(b->d_pool_rec);
    cudaFree(b->d_pol_frags);
    cudaFree(b->d_src);
    cudaFree(b->d_single);
    fresh_free(b);
    for (int i = 0; i < 2; i++) if (b->loop_graph[i].exec) cudaGraphExecDestroy(b->loop_graph[i].exec);
    if (b->d_step_base) { cudaFree(b->d_step_base); cudaStreamDestroy(b->loop_stream); cudaEventDestroy(b->loop_in); cudaEventDestroy(b->loop_out); }
    for (int i = 0; i < kSingleGraphs; i++)
        if (b->single_graph[i].exec) cudaGraphExecDestroy(b->single_graph[i].exec);
    if (b->single_stream) { cudaStreamDestroy(b->single_stream); cudaEventDestroy(b->single_event); }
    if (b->ev_host_done) cudaEventDestroy(b->ev_host_done);
    if (b->slice_ready) {
        for (int i = 0; i < 8; i++) cudaStreamDestroy(b->slice_stream[i]);
        cudaEventDestroy(b->ev_slice_start);
    }
    if (b->pipe_ready) {
        for (int i = 0; i < 2; i++) {
            cudaFree(b->d_actions2[i]);
            cudaFree(b->d_events2[i]);
            cudaEventDestroy(b->ev_in[i]);
            cudaEventDestroy(b->ev_tick[i]);
            cudaEventDestroy(b->ev_out[i]);
        }
        cudaStreamDestroy(b->copy_in);
        cudaStreamDestroy(b->copy_out);
    }
    delete b;
    return ASTRO_OK;
}

int astro_batch_bind(AstroBatch* b, const AstroBuffers* bufs) {
    if (int r = check(b, false)) return r;
    if (!bufs || !bufs->ships || !bufs->ship_b || !bufs->planets || !bufs->meta || !bufs->episode ||
        (b->K > 0 && !bufs->bullets))
        return fail(ASTRO_E_INVALID, "null buffer pointer");
    const uintptr_t al = (uintptr_t)(b->precision == 32 ? 16 : 32);
    if (((uintptr_t)bufs->ships | (uintptr_t)bufs->planets | (uintptr_t)bufs->bullets) & (al - 1))
        return fail(ASTRO_E_INVALID, "ships/planets/bullets must be %d-byte aligned", (int)al);
    b->bufs = *bufs;
    b->cur = 0;
    b->bound = true;
    b->config_epoch++;
    return ASTRO_OK;
}

int astro_set_schedule(AstroBatch* b, const uint32_t* fire_bits_host, int32_t n_ticks, int32_t timeout_tick) {
    if (int r = check(b, false)) return r;
    const int32_t max_ticks = b->PL == ASTRO_MAX_PLANETS_WIDE ? ASTRO_MAX_TICKS_WIDE : ASTRO_MAX_TICKS;
    if (!fire_bits_host || n_ticks <= 0 || n_ticks > max_ticks + 1 || timeout_tick < 0 || timeout_tick >= n_ticks)
        return fail(ASTRO_E_INVALID, "bad schedule (n_ticks %d, timeout_tick %d, max %d)", n_ticks, timeout_tick, max_ticks);
    // util.direction (util.py:87-92) is restated for |b| <= 71476 (np_sincos_f32); beyond that numpy takes another
    // reduction path and the results would silently differ.  Bearings start below 2 pi (core.py:113) and turn by at
    // most dt * ship_rspeed per tick.
    if (6.283185307179586 + (double)n_ticks * fabs(b->cfg.dt * b->cfg.ship_rspeed) > kSinCosRange)
        return fail(ASTRO_E_INVALID, "a bearing could reach %.0f rad within %d ticks (dt * ship_rspeed = %g): beyond the %.0f rad range "
                    "over which util.direction is reproduced", 6.283185307179586 + (double)n_ticks * fabs(b->cfg.dt * b->cfg.ship_rspeed),
                    n_ticks, b->cfg.dt * b->cfg.ship_rspeed, kSinCosRange);
    CUDA_TRY(cudaSetDevice(b->device));
    if (b->d_fire_bits) CUDA_TRY(cudaFree(b->d_fire_bits));
    b->d_fire_bits = nullptr;
    const size_t words = ((size_t)n_ticks + 31) / 32;
    CUDA_TRY(cudaMalloc(&b->d_fire_bits, words * sizeof(uint32_t)));
    CUDA_TRY(cudaMemcpy(b->d_fire_bits, fire_bits_host, words * sizeof(uint32_t), cudaMemcpyHostToDevice));
    b->n_sched_ticks = n_ticks;
    b->timeout_tick = timeout_tick;
    b->config_epoch++;
    return ASTRO_OK;
}

int astro_set_stream(AstroBatch* b, uint32_t seed, int64_t first_game, uint32_t step) {
    if (int r = check(b, false)) return r;
    b->seed = seed;
    b->first_game = first_game;
    b->step = step;
    b->config_epoch++;
    return ASTRO_OK;
}

int astro_set_reset_pool(AstroBatch* b, const AstroResetPool* pool) {
    if (int r = check(b, false)) return r;
    if (!pool || pool->size <= 0 || !pool->ships || !pool->planets || !pool->np)
        return fail(ASTRO_E_INVALID, "bad reset pool");
    if ((uintptr_t)pool->planets & 15) return fail(ASTRO_E_INVALID, "reset pool planets must be 16-byte aligned");
    b->pool = *pool;
    b->config_epoch++;
    if (b->precision == 32) {
        // the tick kernel reads a packed snapshot (one 128-byte record per entry; 256 bytes with 8 planet slots)
        CUDA_TRY(cudaSetDevice(b->device));
        CUDA_TRY(cudaDeviceSynchronize());   // the pool may just have been written on another stream
        if (b->d_pool_rec) CUDA_TRY(cudaFree(b->d_pool_rec));
        b->d_pool_rec = nullptr;
        const bool wide = b->PL == ASTRO_MAX_PLANETS_WIDE;
        CUDA_TRY(cudaMalloc(&b->d_pool_rec, (size_t)pool->size * (wide ? 256 : 128)));
        const int grid = (pool->size + 127) / 128;
        const float* ps = (const float*)pool->ships;
        const float* pp = (const float*)pool->planets;
        float* rec = (float*)b->d_pool_rec;
        with_layout(b, [&](auto, auto s, auto pl) { pack_pool_kernel<s, pl><<<grid, 128>>>(ps, pp, pool->np, rec, pool->size); });
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaDeviceSynchronize());
        b->launches += 1;
    }
    return ASTRO_OK;
}

int astro_tick(AstroBatch* b, const uint8_t* actions, float* reward, uint8_t* done, uint8_t* events,
               int32_t flags, void* stream) {
    if (int r = check(b, true)) return r;
    CUDA_TRY(cudaSetDevice(b->device));
    return do_tick(b, actions, reward, done, events, flags, (cudaStream_t)stream);
}

int astro_tick_many(AstroBatch* b, const uint8_t* actions, float* reward, uint8_t* done, uint8_t* events, int32_t n_ticks,
                    int32_t flags, void* stream) {
    if (int r = check(b, true)) return r;
    if (n_ticks < 0) return fail(ASTRO_E_INVALID, "n_ticks < 0");
    CUDA_TRY(cudaSetDevice(b->device));
    return do_ticks(b, actions, reward, done, events, flags, (cudaStream_t)stream, n_ticks);
}

int astro_tick_host(AstroBatch* b, const uint8_t* actions_host, float* reward_host, uint8_t* done_host,
                    uint8_t* events_host, int32_t flags, void* stream) {
    if (int r = check(b, true)) return r;
    CUDA_TRY(cudaSetDevice(b->device));
    cudaStream_t st = (cudaStream_t)stream;
    const size_t n = (size_t)b->n_games;
    // A closed loop (controls of tick k + 1 depend on the events of tick k) cannot overlap the copies of one tick with the
    // kernel of another — but games are independent, so the tick is cut into slices of tiles, each with its OWN stream:
    // copy in, kernel, copy out are stream-ordered inside a slice and overlap the other slices' (float32 kernel;
    // ASTRO_HOST_SLICES overrides, 1 = off).  (Three shared streams — copies in / kernels / copies out — ordered by
    // events were measured first and lost: every cross-stream dependency costs microseconds, 130 -> 147 us per tick.)
    const char* slices_str = getenv("ASTRO_HOST_SLICES");   // (read on every call: tests switch it)
    const int slices_env = slices_str ? atoi(slices_str) : 0;
    const int n_tiles = b->n_games / ASTRO_TILE;
    int slices = slices_env > 0 ? slices_env : (n_tiles >= 16384 ? 2 : 1);
    if (slices > kMaxSlices) slices = kMaxSlices;
    if (b->fresh) slices = 1;      // (the refill that a launch may trigger must not run beside other slices' kernels)
    if (slices > 1 && actions_host && events_host && !reward_host && !done_host && b->precision == 32 &&
        !(flags & ASTRO_TICK_GENERIC_KERNEL) && n_tiles >= slices) {
        if (!b->slice_ready) {
            for (int i = 0; i < kMaxSlices; i++) CUDA_TRY(cudaStreamCreateWithFlags(&b->slice_stream[i], cudaStreamNonBlocking));
            CUDA_TRY(cudaEventCreateWithFlags(&b->ev_slice_start, cudaEventDisableTiming));
            b->slice_ready = true;
        }
        const bool packed = (flags & ASTRO_TICK_PACKED_CONTROLS) != 0, planes = (flags & ASTRO_TICK_EVENT_PLANES) != 0;
        const size_t a_per_tile = (size_t)ASTRO_TILE * (packed ? 1 : b->S);
        CUDA_TRY(cudaEventRecord(b->ev_slice_start, st));               // earlier work of the caller's stream comes first
        for (int i = 0; i < slices; i++) {
            cudaStream_t ss = b->slice_stream[i];
            const int t0 = (int)((int64_t)n_tiles * i / slices), t1 = (int)((int64_t)n_tiles * (i + 1) / slices);
            CUDA_TRY(cudaStreamWaitEvent(ss, b->ev_slice_start, 0));
            CUDA_TRY(cudaMemcpyAsync(b->d_actions + t0 * a_per_tile, actions_host + t0 * a_per_tile, (size_t)(t1 - t0) * a_per_tile,
                                     cudaMemcpyHostToDevice, ss));
            if (int r = do_ticks(b, b->d_actions, nullptr, nullptr, b->d_events, flags, ss, 1, t0, t1 - t0, i == slices - 1)) return r;
            if (planes)
                CUDA_TRY(cudaMemcpy2DAsync(events_host + (size_t)t0 * 4, (size_t)n_tiles * 4, b->d_events + (size_t)t0 * 4, (size_t)n_tiles * 4,
                                           (size_t)(t1 - t0) * 4, 3, cudaMemcpyDeviceToHost, ss));
            else
                CUDA_TRY(cudaMemcpyAsync(events_host + (size_t)t0 * ASTRO_TILE, b->d_events + (size_t)t0 * ASTRO_TILE, (size_t)(t1 - t0) * ASTRO_TILE,
                                         cudaMemcpyDeviceToHost, ss));
        }
        for (int i = 0; i < slices; i++) CUDA_TRY(cudaStreamSynchronize(b->slice_stream[i]));
        return ASTRO_OK;
    }
    if (actions_host) CUDA_TRY(cudaMemcpyAsync(b->d_actions, actions_host, actions_bytes(b, flags), cudaMemcpyHostToDevice, st));
    if (int r = do_tick(b, actions_host ? b->d_actions : nullptr, reward_host ? b->d_reward : nullptr,
                        done_host ? b->d_done : nullptr, events_host ? b->d_events : nullptr, flags, st))
        return r;
    if (events_host) CUDA_TRY(cudaMemcpyAsync(events_host, b->d_events, events_bytes(b, flags), cudaMemcpyDeviceToHost, st));
    if (done_host) CUDA_TRY(cudaMemcpyAsync(done_host, b->d_done, n, cudaMemcpyDeviceToHost, st));
    if (reward_host) CUDA_TRY(cudaMemcpyAsync(reward_host, b->d_reward, n * b->S * sizeof(float), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return ASTRO_OK;
}

int astro_tick_host_begin(AstroBatch* b, const uint8_t* actions_host, uint8_t* events_host, int32_t flags, void* stream) {
    if (int r = check(b, true)) return r;
    if (!actions_host || !events_host) return fail(ASTRO_E_INVALID, "null host buffer");
    if (b->host_pending) return fail(ASTRO_E_STATE, "astro_tick_host_begin: the previous tick has not been ended (astro_tick_host_end)");
    CUDA_TRY(cudaSetDevice(b->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (!b->ev_host_done) CUDA_TRY(cudaEventCreateWithFlags(&b->ev_host_done, cudaEventDisableTiming));
    CUDA_TRY(cudaMemcpyAsync(b->d_actions, actions_host, actions_bytes(b, flags), cudaMemcpyHostToDevice, st));
    if (int r = do_tick(b, b->d_actions, nullptr, nullptr, b->d_events, flags, st)) return r;
    CUDA_TRY(cudaMemcpyAsync(events_host, b->d_events, events_bytes(b, flags), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaEventRecord(b->ev_host_done, st));
    b->host_pending = true;
    return ASTRO_OK;
}

int astro_tick_host_end(AstroBatch* b) {
    if (int r = check(b, true)) return r;
    if (!b->host_pending) return fail(ASTRO_E_STATE, "astro_tick_host_end without astro_tick_host_begin");
    b->host_pending = false;
    CUDA_TRY(cudaEventSynchronize(b->ev_host_done));
    return ASTRO_OK;
}

int astro_rollout_host(AstroBatch* b, const uint8_t* actions_host, uint8_t* events_host, int32_t n_ticks, int32_t flags,
                       void* stream) {
    if (int r = check(b, true)) return r;
    if (!actions_host || !events_host || n_ticks < 0) return fail(ASTRO_E_INVALID, "bad rollout arguments");
    CUDA_TRY(cudaSetDevice(b->device));
    cudaStream_t st = (cudaStream_t)stream;
    if ((flags & ASTRO_TICK_PACKED_CONTROLS) && b->S != 2) return fail(ASTRO_E_INVALID, "ASTRO_TICK_PACKED_CONTROLS is for duel games");
    const size_t n = events_bytes(b, flags), na = actions_bytes(b, flags);   // bytes per tick: events out, controls in
    // Ticks travel in chunks of C: the controls of C ticks are copied in (one copy per tick: 2 MB copies run at
    // 51 GB/s on the pool's boxes, 16 MB ones at 14 — tools/ubench/pcie.py), the C ticks run as ONE launch
    // (do_ticks: a tile's ticks back to back), their events are copied out.  1M games, 32 ticks per call, e2e
    // env-steps/s: C = 1 1.42e10, 4 1.48e10, 8 1.35e10, 16 1.13e10 (the pipeline is two chunks deep: large
    // chunks leave little to overlap within a call).  ASTRO_ROLLOUT_CHUNK overrides.
    static const int chunk_env = getenv("ASTRO_ROLLOUT_CHUNK") ? atoi(getenv("ASTRO_ROLLOUT_CHUNK")) : 0;
    // (round 2, 128 ticks per call, packed controls + event planes: C = 4 1.95e10, 8 2.00e10, 16 1.95e10, 32 1.84e10; byte forms:
    // 1.75e10 / 1.70e10 / 1.53e10 / 1.25e10 — half the bytes per tick move the optimum up one step)
    const int C = chunk_env > 0 ? chunk_env : ((flags & ASTRO_TICK_PACKED_CONTROLS) ? 8 : 4);
    if (b->pipe_ready && b->pipe_chunk != C) {
        for (int i = 0; i < 2; i++) {
            CUDA_TRY(cudaFree(b->d_actions2[i]));
            CUDA_TRY(cudaFree(b->d_events2[i]));
            CUDA_TRY(cudaMalloc(&b->d_actions2[i], (size_t)b->n_games * b->S * C));
            CUDA_TRY(cudaMalloc(&b->d_events2[i], (size_t)b->n_games * C));
        }
        b->pipe_chunk = C;
    }
    if (!b->pipe_ready) {
        CUDA_TRY(cudaStreamCreateWithFlags(&b->copy_in, cudaStreamNonBlocking));
        CUDA_TRY(cudaStreamCreateWithFlags(&b->copy_out, cudaStreamNonBlocking));
        for (int i = 0; i < 2; i++) {
            CUDA_TRY(cudaMalloc(&b->d_actions2[i], (size_t)b->n_games * b->S * C));
            CUDA_TRY(cudaMalloc(&b->d_events2[i], (size_t)b->n_games * C));
            CUDA_TRY(cudaEventCreateWithFlags(&b->ev_in[i], cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&b->ev_tick[i], cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&b->ev_out[i], cudaEventDisableTiming));
        }
        b->pipe_chunk = C;
        b->pipe_ready = true;
    }
    // Three queues: the controls of chunk c+1 travel host->device while the ticks of chunk c run and the
    // events of chunk c-1 travel device->host.  Buffer i = c % 2; an event per buffer and stage orders them.
    for (int c = 0, k0 = 0; k0 < n_ticks; c++, k0 += C) {
        const int i = c & 1, kc = n_ticks - k0 < C ? n_ticks - k0 : C;
        if (c >= 2) CUDA_TRY(cudaStreamWaitEvent(b->copy_in, b->ev_tick[i], 0));  // chunk c-2 has read buffer i
        for (int j = 0; j < kc; j++)   // (one copy per tick: 2 MB copies run at 51 GB/s on this pool, 16 MB ones at 14)
            CUDA_TRY(cudaMemcpyAsync(b->d_actions2[i] + (size_t)j * na, actions_host + (size_t)(k0 + j) * na, na, cudaMemcpyHostToDevice, b->copy_in));
        CUDA_TRY(cudaEventRecord(b->ev_in[i], b->copy_in));
        CUDA_TRY(cudaStreamWaitEvent(st, b->ev_in[i], 0));
        if (c >= 2) CUDA_TRY(cudaStreamWaitEvent(st, b->ev_out[i], 0));  // events of chunk c-2 have left buffer i
        if (int r = do_ticks(b, b->d_actions2[i], nullptr, nullptr, b->d_events2[i], flags, st, kc)) return r;
        CUDA_TRY(cudaEventRecord(b->ev_tick[i], st));
        CUDA_TRY(cudaStreamWaitEvent(b->copy_out, b->ev_tick[i], 0));
        for (int j = 0; j < kc; j++)
            CUDA_TRY(cudaMemcpyAsync(events_host + (size_t)(k0 + j) * n, b->d_events2[i] + (size_t)j * n, n, cudaMemcpyDeviceToHost, b->copy_out));
        CUDA_TRY(cudaEventRecord(b->ev_out[i], b->copy_out));
    }
    CUDA_TRY(cudaStreamSynchronize(b->copy_out));
    CUDA_TRY(cudaStreamSynchronize(st));
    return ASTRO_OK;
}

int astro_reset_done(AstroBatch* b, void* stream) {
    if (int r = check(b, true)) return r;
    if (b->pool.size <= 0) return fail(ASTRO_E_STATE, "astro_set_reset_pool has not been called");
    CUDA_TRY(cudaSetDevice(b->device));
    TickParams p;
    fill_params(b, p);
    const int grid = (p.n_games + kTickThreads - 1) / kTickThreads;
    cudaStream_t st = (cudaStream_t)stream;
    with_layout(b, [&](auto r, auto s, auto pl) { reset_kernel<typename decltype(r)::type, s, pl><<<grid, kTickThreads, 0, st>>>(p); });
    CUDA_TRY(cudaGetLastError());
    b->launches += 1;
    return ASTRO_OK;
}

static int observe_args(const AstroBatch* b, const float* obs, int32_t n_rows, bool both) {
    if (!obs) return fail(ASTRO_E_INVALID, "null obs");
    const int D = 1 + 5 * b->S + 4;
    if (n_rows < b->PL + b->K) return fail(ASTRO_E_INVALID, "n_rows %d < %d planet slots + bullet_cap %d", n_rows, b->PL, b->K);
    if ((n_rows * D) % 4) return fail(ASTRO_E_INVALID, "n_rows * %d must be a multiple of 4", D);
    if ((uintptr_t)obs & 15) return fail(ASTRO_E_INVALID, "obs must be 16-byte aligned");
    if ((size_t)kObserveWarps * observe_warp_floats(n_rows, D, b->S, (both && b->S == 2) ? 2 : 1) * sizeof(float) > 200 * 1024)
        return fail(ASTRO_E_INVALID, "n_rows %d too large for the staging buffer", n_rows);
    return ASTRO_OK;
}

// ring_ticks > 0: obs is a recording ring (AstroRecordRing.observations) and the block goes to the row of the current stream step
static int observe_impl(AstroBatch* b, float* obs, int32_t n_rows, bool both, void* stream, uint32_t ring_ticks = 0) {
    if (int r = check(b, true)) return r;
    if (int r = observe_args(b, obs, n_rows, both)) return r;
    CUDA_TRY(cudaSetDevice(b->device));
    const int D = 1 + 5 * b->S + 4;
    const size_t smem = (size_t)kObserveWarps * observe_warp_floats(n_rows, D, b->S, (both && b->S == 2) ? 2 : 1) * sizeof(float);
    const int grid = (b->n_games + kObserveWarps - 1) / kObserveWarps;
    cudaStream_t st = (cudaStream_t)stream;
    const AstroBuffers& u = b->bufs;
    auto launch = [&](auto kernel) {
        CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kernel<<<grid, kObserveWarps * 32, smem, st>>>(u.ships, u.ship_b, u.planets, bullet_buffer(b, b->cur), u.meta, obs, b->n_games,
                                                       b->K, n_rows, ring_ticks, b->step, b->step_base_now);
        return ASTRO_OK;
    };
    if (int r = with_layout(b, [&](auto tr, auto s, auto pl) {
            using R = typename decltype(tr)::type;
            if constexpr (s == 2) return both ? launch(observe_kernel<R, 2, true, pl>) : launch(observe_kernel<R, 2, false, pl>);
            else return launch(observe_kernel<R, 1, false, pl>);     // (both views of a solo game are the same)
        }))
        return r;
    CUDA_TRY(cudaGetLastError());
    b->launches += 1;
    return ASTRO_OK;
}

int astro_observe(AstroBatch* b, float* obs, int32_t n_rows, void* stream) { return observe_impl(b, obs, n_rows, true, stream); }

int astro_observe_shared(AstroBatch* b, float* obs, int32_t n_rows, void* stream) {
    return observe_impl(b, obs, n_rows, false, stream);
}

int astro_script_controls(AstroBatch* b, double avoid_distance, double avoid_threshold, uint8_t* actions, void* stream) {
    if (int r = check(b, true)) return r;
    if (!actions) return fail(ASTRO_E_INVALID, "null actions");
    CUDA_TRY(cudaSetDevice(b->device));
    ScriptParams q;
    q.radius = b->cfg.planet_radius + b->cfg.ship_radius;
    q.avoid_distance = avoid_distance;
    q.avoid_threshold = avoid_threshold;
    q.ship_thrust = b->cfg.ship_thrust;
    q.ship_rspeed = b->cfg.ship_rspeed;
    q.bullet_speed = b->cfg.bullet_speed;
    q.ship_radius = b->cfg.ship_radius;
    q.solo = b->cfg.solo;
    q.n_games = b->n_games;
    const int grid = (b->n_games * b->S + 127) / 128;
    cudaStream_t st = (cudaStream_t)stream;
    const AstroBuffers& u = b->bufs;
    with_layout(b, [&](auto r, auto s, auto pl) {
        script_kernel<typename decltype(r)::type, s, pl><<<grid, 128, 0, st>>>(u.ships, u.ship_b, u.planets, u.meta, actions, q);
    });
    CUDA_TRY(cudaGetLastError());
    b->launches += 1;
    return ASTRO_OK;
}

int astro_create_games(AstroBatch* b, const AstroCreateConfig* cc, const uint32_t* seeds, int32_t m, void* ships,
                       void* planets, int32_t* n_planets, void* stream) {
    if (int r = check(b, false)) return r;
    if (!cc || !seeds || !ships || !planets || !n_planets || m <= 0) return fail(ASTRO_E_INVALID, "bad create arguments");
    if (cc->max_planets < 1 || cc->max_planets > b->PL)
        return fail(ASTRO_E_INVALID, "max_planets must be 1..%d (the batch's planet slots; at most %d with planet_slots = %d)",
                    b->PL, ASTRO_MAX_PLANETS_WIDE, ASTRO_MAX_PLANETS_WIDE);
    CUDA_TRY(cudaSetDevice(b->device));
    CreateParams q;
    q.inner = cc->inner_ship_position;
    q.outer = cc->outer_ship_position;
    q.orbit = cc->planet_orbit;
    q.gravity = b->cfg.gravity;
    q.planet_mass = b->cfg.planet_mass;
    q.max_planets = cc->max_planets;
    q.solo = b->cfg.solo;
    q.m = m;
    q.pad = 0;
    const int grid = (m + 63) / 64;
    cudaStream_t st = (cudaStream_t)stream;
    with_layout(b, [&](auto tr, auto s, auto pl) {
        using R = typename decltype(tr)::type;
        create_kernel<R, s, pl><<<grid, 64, 0, st>>>(seeds, (R*)ships, (R*)planets, n_planets, q);
    });
    CUDA_TRY(cudaGetLastError());
    b->launches += 1;
    return ASTRO_OK;
}

int astro_policy_set_weights(AstroBatch* b, const float* weights_host, int32_t n_floats, int32_t nout) {
    if (int r = check(b, false)) return r;
    const int din = 1 + 5 * b->S + 4;
    if (nout < 1 || nout > kPolMaxOut) return fail(ASTRO_E_INVALID, "nout must be 1..%d", kPolMaxOut);
    const int expect = kPolW * din + kPolW + 4 * (kPolW * kPolW + kPolW) + nout * kPolW + nout;
    if (!weights_host || n_floats != expect)
        return fail(ASTRO_E_INVALID, "expected %d floats (f0, f[0], f[1], v[0], v[1], v0: weight then bias each), got %d", expect, n_floats);
    CUDA_TRY(cudaSetDevice(b->device));
    // weights_host: every layer's weight [out][in] (nn.Linear), then its bias
    const float* f0 = weights_host;
    const float* f1 = f0 + kPolW * din + kPolW;
    const float* f2 = f1 + kPolW * kPolW + kPolW;
    const float* v1 = f2 + kPolW * kPolW + kPolW;
    const float* v2 = v1 + kPolW * kPolW + kPolW;
    const float* v0 = v2 + kPolW * kPolW + kPolW;
    const float* v0b = v0 + nout * kPolW;
    // the weights as tensor-core B fragments for policy_mma_kernel / value_forward_kernel, input columns in the order the A
    // fragments arrive in (see the kernel)
    PolicyFragWeights* fw = new (std::nothrow) PolicyFragWeights();
    if (!fw) return fail(ASTRO_E_NOMEM, "out of host memory");
    memset(fw, 0, sizeof(*fw));
    {
        // FP16 pairs: a fragment register holds input columns (k, k + 1), the even one in the low half; hi = the weight rounded
        // to FP16, lo = what that dropped, rounded to FP16
        auto pair = [](float we, float wo, uint32_t& hi, uint32_t& lo) {
            const __half he = __float2half_rn(we), ho = __float2half_rn(wo);
            const __half le = __float2half_rn(we - __half2float(he)), lo_ = __float2half_rn(wo - __half2float(ho));
            hi = (uint32_t)__half_as_ushort(he) | ((uint32_t)__half_as_ushort(ho) << 16);
            lo = (uint32_t)__half_as_ushort(le) | ((uint32_t)__half_as_ushort(lo_) << 16);
        };
        auto entry16 = [&](auto&& weight, int k0) {             // b0: input columns k0, k0 + 1; b1: k0 + 8, k0 + 9
            uint32_t h0, l0, h1, l1;
            pair(weight(k0), weight(k0 + 1), h0, l0);
            pair(weight(k0 + 8), weight(k0 + 9), h1, l1);
            float4 r;
            memcpy(&r.x, &h0, 4); memcpy(&r.y, &h1, 4); memcpy(&r.z, &l0, 4); memcpy(&r.w, &l1, 4);
            return r;
        };
        for (int l = 0; l < 32; l++) {
            const int g_ = l >> 2, t_ = l & 3;
            for (int nt = 0; nt < 4; nt++) {
                const int n = nt * 8 + g_;
                fw->f0[0][nt][l] = entry16([&](int c) { return c < din ? f0[n * din + c] : 0.f; }, 2 * t_);
                for (int kk = 0; kk < 2; kk++) {
                    const int k0 = 16 * kk + 2 * t_;
                    fw->f1[kk][nt][l] = entry16([&](int c) { return f1[n * kPolW + c]; }, k0);
                    fw->f2[kk][nt][l] = entry16([&](int c) { return f2[n * kPolW + c]; }, k0);
                    fw->v1[kk][nt][l] = entry16([&](int c) { return v1[n * kPolW + c]; }, k0);
                    fw->v2[kk][nt][l] = entry16([&](int c) { return v2[n * kPolW + c]; }, k0);
                }
            }
            for (int kk = 0; kk < 2; kk++) fw->v0[kk][l] = entry16([&](int c) { return g_ < nout ? v0[g_ * kPolW + c] : 0.f; }, 16 * kk + 2 * t_);
        }
        const float* biases[5] = {f0 + kPolW * din, f1 + kPolW * kPolW, f2 + kPolW * kPolW, v1 + kPolW * kPolW, v2 + kPolW * kPolW};
        for (int layer = 0; layer < 5; layer++)
            for (int nt = 0; nt < 4; nt++)
                for (int t_ = 0; t_ < 4; t_++) fw->bias[layer][nt][t_] = make_float2(biases[layer][nt * 8 + 2 * t_], biases[layer][nt * 8 + 2 * t_ + 1]);
        for (int t_ = 0; t_ < 4; t_++) fw->bias_v0[t_] = make_float2(2 * t_ < nout ? v0b[2 * t_] : 0.f, 2 * t_ + 1 < nout ? v0b[2 * t_ + 1] : 0.f);
    }
    cudaError_t e = b->d_pol_frags ? cudaSuccess : cudaMalloc(&b->d_pol_frags, sizeof(PolicyFragWeights));
    // (pageable source: the copy has left `fw` when the call returns; stream-ordered before later launches)
    if (e == cudaSuccess) e = cudaMemcpy(b->d_pol_frags, fw, sizeof(*fw), cudaMemcpyHostToDevice);
    delete fw;
    if (e != cudaSuccess) return fail(ASTRO_E_CUDA, "policy weights upload: %s", cudaGetErrorString(e));
    b->policy_nout = nout;
    b->config_epoch++;
    return ASTRO_OK;
}

int astro_policy_controls(AstroBatch* b, uint8_t* actions, float* q_out, int32_t ship_mask, void* stream) {
    if (int r = check(b, true)) return r;
    if (b->policy_nout <= 0) return fail(ASTRO_E_STATE, "astro_policy_set_weights has not been called");
    if (!actions) return fail(ASTRO_E_INVALID, "null actions");
    CUDA_TRY(cudaSetDevice(b->device));
    cudaStream_t st = (cudaStream_t)stream;
    const AstroBuffers& u = b->bufs;
    int grid = ((b->n_games + 7) / 8 + kMmaWarps - 1) / kMmaWarps;      // a warp takes 8 games at a time
    if (grid > b->sm_count * ASTRO_MMA_MIN_BLOCKS) grid = b->sm_count * ASTRO_MMA_MIN_BLOCKS;
    const int smem = (int)sizeof(PolicyFrags);
    if (int r = with_layout(b, [&](auto tr, auto s, auto pl) {
            const auto kernel = policy_mma_kernel<typename decltype(tr)::type, s, pl>;
            CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
            kernel<<<grid, kMmaWarps * 32, smem, st>>>(u.ships, u.ship_b, u.planets, bullet_buffer(b, b->cur), u.meta, actions, q_out,
                                                       b->n_games, b->K, b->policy_nout, ship_mask, b->d_pol_frags);
            return ASTRO_OK;
        }))
        return r;
    CUDA_TRY(cudaGetLastError());
    b->launches += 1;
    return ASTRO_OK;
}

int astro_set_exploration(AstroBatch* b, double t_in, double t_out, uint32_t seed, int32_t* state) {
    if (int r = check(b, false)) return r;
    if (!state) return fail(ASTRO_E_INVALID, "null exploration state");
    if (!(t_in > 0.0) || !(t_out > 0.0)) return fail(ASTRO_E_INVALID, "t_in and t_out must be positive");
    b->explore_t_in = t_in;
    b->explore_t_out = t_out;
    b->explore_seed = seed;
    b->explore_state = state;
    b->config_epoch++;
    return ASTRO_OK;
}

int astro_explore_controls(AstroBatch* b, double t_in, double t_out, uint32_t seed, int32_t* state, uint8_t* actions,
                           int32_t ship_mask, void* stream) {
    if (int r = check(b, true)) return r;
    if (!state || !actions) return fail(ASTRO_E_INVALID, "null state / actions");
    if (!(t_in > 0.0) || !(t_out > 0.0)) return fail(ASTRO_E_INVALID, "t_in and t_out must be positive");
    CUDA_TRY(cudaSetDevice(b->device));
    const int grid = (b->n_games * b->S + 127) / 128;
    cudaStream_t st = (cudaStream_t)stream;
    with_layout(b, [&](auto, auto s, auto pl) {
        explore_kernel<s, pl><<<grid, 128, 0, st>>>(b->bufs.meta, state, actions, b->n_games, ship_mask, b->cfg.dt, t_in, t_out, seed,
                                                     (uint32_t)b->first_game, b->step, b->step_base_now);
    });
    CUDA_TRY(cudaGetLastError());
    b->launches += 1;
    return ASTRO_OK;
}

static int rollout_one_tick(AstroBatch* b, const int* modes, double avoid_distance, double avoid_threshold, uint8_t* actions, uint8_t* events,
                            int32_t flags, cudaStream_t st);

static int rollout_chunks(AstroBatch* b, int n_chunks, const int* modes, double avoid_distance, double avoid_threshold, uint8_t* actions,
                          uint8_t* events, int32_t flags, cudaStream_t st) {
    if (!b->d_step_base) {
        CUDA_TRY(cudaMalloc(&b->d_step_base, sizeof(uint32_t)));
        CUDA_TRY(cudaStreamCreateWithFlags(&b->loop_stream, cudaStreamNonBlocking));   // (a legacy default stream cannot be captured)
        CUDA_TRY(cudaEventCreateWithFlags(&b->loop_in, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&b->loop_out, cudaEventDisableTiming));
    }
    cudaStream_t ls = b->loop_stream;
    CUDA_TRY(cudaEventRecord(b->loop_in, st));                 // earlier work of the caller's stream comes first
    CUDA_TRY(cudaStreamWaitEvent(ls, b->loop_in, 0));
    step_base_set_kernel<<<1, 1, 0, ls>>>(b->d_step_base, b->step);
    for (int c = 0; c < n_chunks; c++) {
        if (b->fresh && (flags & ASTRO_TICK_AUTO_RESET)) {     // fresh-game mode: refills happen between chunks, outside the graph
            FreshState* fs = b->fresh;
            if (fs->ticks_since_refill > 0 && (fs->ticks_since_refill + kLoopChunk) * 2 > fs->f.quota)
                if (int r = fresh_refill(b, ls)) return r;
            fs->ticks_since_refill += kLoopChunk;
        }
        LoopGraph* g = nullptr;
        for (int i = 0; i < 2; i++) {
            LoopGraph& q = b->loop_graph[i];
            if (q.exec && q.epoch == b->config_epoch && q.cur == b->cur && q.flags == flags && q.modes[0] == modes[0] && q.modes[1] == modes[1] &&
                q.avoid_distance == avoid_distance && q.avoid_threshold == avoid_threshold && q.actions == actions && q.events == events &&
                q.rec.ticks == b->rec_now.ticks && q.rec.n_rows == b->rec_now.n_rows && q.rec.controls == b->rec_now.controls &&
                q.rec.events == b->rec_now.events && q.rec.observations == b->rec_now.observations)
                g = &q;
        }
        if (!g) {
            g = &b->loop_graph[b->cur & 1];
            if (g->exec) { cudaGraphExecDestroy(g->exec); g->exec = nullptr; }
            const uint32_t step_saved = b->step;
            const int32_t cur_saved = b->cur;
            const int64_t launches_saved = b->launches, fold_saved = b->ticks_since_fold;
            CUDA_TRY(cudaStreamBeginCapture(ls, cudaStreamCaptureModeThreadLocal));
            b->step_base_now = b->d_step_base;
            b->step = 0;                                       // steps inside a chunk are relative to the device word
            int rc = ASTRO_OK;
            for (int j = 0; j < kLoopChunk && !rc; j++) rc = rollout_one_tick(b, modes, avoid_distance, avoid_threshold, actions, events, flags, ls);
            if (!rc) step_base_add_kernel<<<1, 1, 0, ls>>>(b->d_step_base, (uint32_t)kLoopChunk);
            cudaGraph_t graph = nullptr;
            const cudaError_t e = cudaStreamEndCapture(ls, &graph);
            b->step_base_now = nullptr;
            b->step = step_saved;
            b->cur = cur_saved;
            g->launches = (int32_t)(b->launches - launches_saved) + 1;
            b->launches = launches_saved;
            b->ticks_since_fold = fold_saved;
            if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
            if (e != cudaSuccess) return fail(ASTRO_E_CUDA, "bot-loop capture: %s", cudaGetErrorString(e));
            const cudaError_t ei = cudaGraphInstantiate(&g->exec, graph, 0);
            cudaGraphDestroy(graph);
            if (ei != cudaSuccess) { g->exec = nullptr; return fail(ASTRO_E_CUDA, "bot-loop graph: %s", cudaGetErrorString(ei)); }
            g->epoch = b->config_epoch; g->cur = b->cur; g->flags = flags; g->modes[0] = modes[0]; g->modes[1] = modes[1];
            g->avoid_distance = avoid_distance; g->avoid_threshold = avoid_threshold; g->actions = actions; g->events = events;
            g->rec = b->rec_now;
        }
        CUDA_TRY(cudaGraphLaunch(g->exec, ls));
        b->step += (uint32_t)kLoopChunk;
        b->launches += g->launches;
        if (!(flags & ASTRO_TICK_NO_STATS)) b->ticks_since_fold += kLoopChunk;
    }
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(b->loop_out, ls));
    CUDA_TRY(cudaStreamWaitEvent(st, b->loop_out, 0));         // ... and the caller's stream carries on behind the chunks
    return ASTRO_OK;
}

// astro_rollout_device, recording into b->rec_now when its events array is set (astro_rollout_device_record)
static int rollout_device(AstroBatch* b, int32_t n_ticks, int32_t ship0_mode, int32_t ship1_mode, double avoid_distance,
                          double avoid_threshold, uint8_t* actions, uint8_t* events, int32_t flags, void* stream) {
    if (int r = check(b, true)) return r;
    if (n_ticks < 0) return fail(ASTRO_E_INVALID, "n_ticks < 0");
    const int modes[2] = {ship0_mode, b->S == 2 ? ship1_mode : ship0_mode};
    bool any_script = false, any_policy = false, any_stream = false, any_idle = false, any_explore = false;
    for (int k = 0; k < b->S; k++) {
        if (modes[k] < ASTRO_BOT_STREAM || modes[k] > ASTRO_BOT_EXPLORE) return fail(ASTRO_E_INVALID, "unknown bot mode %d", modes[k]);
        any_stream |= modes[k] == ASTRO_BOT_STREAM;
        any_script |= modes[k] == ASTRO_BOT_SCRIPT;
        any_policy |= modes[k] == ASTRO_BOT_POLICY || modes[k] == ASTRO_BOT_EXPLORE;
        any_explore |= modes[k] == ASTRO_BOT_EXPLORE;
        any_idle |= modes[k] == ASTRO_BOT_NOTHING;
    }
    const bool all_stream = any_stream && !any_script && !any_policy && !any_idle;
    if (any_stream && !all_stream) return fail(ASTRO_E_INVALID, "ASTRO_BOT_STREAM drives every ship or none");
    if (!all_stream && !actions) return fail(ASTRO_E_INVALID, "a scratch actions buffer [n_games][S] is needed for bot modes");
    if (any_policy && b->policy_nout <= 0) return fail(ASTRO_E_STATE, "astro_policy_set_weights has not been called");
    if (any_explore && !b->explore_state) return fail(ASTRO_E_STATE, "astro_set_exploration has not been called");
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(b->device));
    if (any_idle) CUDA_TRY(cudaMemsetAsync(actions, 2, (size_t)b->n_games * b->S, st));  // script.NothingBot: control 2
    // Recording: the tick kernel stores each tick's controls and events itself, so the two fast paths below keep their launches;
    // observations are taken by observe_kernel before every tick, which needs the per-tick loop at the end.
    float* const rec_obs = b->rec_now.observations;
    if (all_stream && !rec_obs) {
        // no bot between the ticks: the ticks of a tile run back to back inside the launches; `events` keeps the last tick's
        if (n_ticks > 1) if (int r = do_ticks(b, nullptr, nullptr, nullptr, nullptr, flags, st, n_ticks - 1)) return r;
        return n_ticks > 0 ? do_ticks(b, nullptr, nullptr, nullptr, events, flags, st, 1) : ASTRO_OK;
    }
    // ScriptBot / NothingBot on every ship (float32 build): the bots are evaluated INSIDE the tick kernel, from the rows a tile's
    // warp has just loaded, so the ticks of a tile run back to back within a launch — no launch, no control array between ticks
    // (`actions` is not written).  ASTRO_FUSED_BOTS=0 switches it off.  Batches with 8 planet slots have no such instantiation
    // and always take the bot kernel -> tick kernel loop below.
    {
        const char* fb = getenv("ASTRO_FUSED_BOTS");
        if (!any_policy && !rec_obs && b->precision == 32 && b->PL == ASTRO_MAX_PLANETS && !(flags & ASTRO_TICK_GENERIC_KERNEL) &&
            !(fb && atoi(fb) == 0) && n_ticks > 0) {
            b->bot_modes_now = modes[0] | (modes[1] << 4);
            ScriptParams& q = b->script_now;
            q.radius = b->cfg.planet_radius + b->cfg.ship_radius;
            q.avoid_distance = avoid_distance;
            q.avoid_threshold = avoid_threshold;
            q.ship_thrust = b->cfg.ship_thrust;
            q.ship_rspeed = b->cfg.ship_rspeed;
            q.bullet_speed = b->cfg.bullet_speed;
            q.ship_radius = b->cfg.ship_radius;
            q.solo = b->cfg.solo;
            q.n_games = b->n_games;
            int rc = ASTRO_OK;
            if (n_ticks > 1) rc = do_ticks(b, nullptr, nullptr, nullptr, nullptr, flags, st, n_ticks - 1);
            if (!rc) rc = do_ticks(b, nullptr, nullptr, nullptr, events, flags, st, 1);      // `events` keeps the last tick's
            b->bot_modes_now = 0;
            return rc;
        }
    }
    // One tick of the loop is 2-4 small launches; at 16,384 games the gaps between them cost as much as the kernels.  Whole
    // chunks of kLoopChunk ticks are therefore captured ONCE into a CUDA graph and replayed: one graph launch per chunk.
    // What changes from chunk to chunk — the stream step, which keys the pool picks and the exploration draws — is read
    // by the kernels from a device word (step_base) that a one-thread node advances at the end of every chunk; the rest
    // of a chunk's parameters are fixed (an even number of ticks leaves the bullet buffers where they started).
    // ASTRO_LOOP_GRAPH=0 switches it off.
    const char* lg = getenv("ASTRO_LOOP_GRAPH");
    int k_done = 0;
    if (n_ticks >= kLoopChunk && !(lg && atoi(lg) == 0)) {
        if (int r = rollout_chunks(b, n_ticks / kLoopChunk, modes, avoid_distance, avoid_threshold, actions, events, flags, st)) return r;
        k_done = (n_ticks / kLoopChunk) * kLoopChunk;
    }
    for (int k = k_done; k < n_ticks; k++) {
        if (int r = rollout_one_tick(b, modes, avoid_distance, avoid_threshold, actions, events, flags, st)) return r;
    }
    // the state after the last tick: the new state of the pairs that flush on it
    if (rec_obs) return observe_impl(b, rec_obs, b->rec_now.n_rows, false, stream, (uint32_t)b->rec_now.ticks);
    return ASTRO_OK;
}

int astro_rollout_device(AstroBatch* b, int32_t n_ticks, int32_t ship0_mode, int32_t ship1_mode, double avoid_distance,
                         double avoid_threshold, uint8_t* actions, uint8_t* events, int32_t flags, void* stream) {
    return rollout_device(b, n_ticks, ship0_mode, ship1_mode, avoid_distance, avoid_threshold, actions, events, flags, stream);
}

int astro_rollout_device_record(AstroBatch* b, int32_t n_ticks, int32_t ship0_mode, int32_t ship1_mode, double avoid_distance,
                                double avoid_threshold, uint8_t* actions, const AstroRecordRing* ring, int32_t flags,
                                void* stream) {
    if (int r = check(b, true)) return r;
    if (ring) {
        if (b->precision != 32)
            return fail(ASTRO_E_INVALID, "recording needs a float32 batch: the ring is written by the float32 tick kernel (precision %d)",
                        b->precision);
        if (flags & ASTRO_TICK_GENERIC_KERNEL)
            return fail(ASTRO_E_INVALID, "recording needs the float32 tick kernel: ASTRO_TICK_GENERIC_KERNEL runs the template kernel, which does not record");
        if (!ring->controls || !ring->events) return fail(ASTRO_E_INVALID, "the ring's controls and events arrays are required");
        if (b->S == 2 && ((uintptr_t)ring->controls & 1)) return fail(ASTRO_E_INVALID, "the ring's controls must be 2-byte aligned");
        if (ring->ticks < 2 || n_ticks >= ring->ticks)
            return fail(ASTRO_E_INVALID, "n_ticks %d needs a ring of at least n_ticks + 1 rows (ticks = %d): the state after the last "
                        "tick is recorded too", n_ticks, ring->ticks);
        if (ring->observations)
            if (int r = observe_args(b, ring->observations, ring->n_rows, false)) return r;
        b->rec_now = *ring;
    }
    const int rc = rollout_device(b, n_ticks, ship0_mode, ship1_mode, avoid_distance, avoid_threshold, actions, nullptr, flags, stream);
    b->rec_now = AstroRecordRing{};
    return rc;
}

// (the body of one tick of astro_rollout_device with bots, on stream st)
static int rollout_one_tick(AstroBatch* b, const int* modes, double avoid_distance, double avoid_threshold, uint8_t* actions, uint8_t* events,
                     int32_t flags, cudaStream_t st) {
    void* stream = (void*)st;
    bool any_script = false, any_policy = false, any_idle = false, any_explore = false;
    for (int k = 0; k < b->S; k++) {
        any_script |= modes[k] == ASTRO_BOT_SCRIPT;
        any_policy |= modes[k] == ASTRO_BOT_POLICY || modes[k] == ASTRO_BOT_EXPLORE;
        any_explore |= modes[k] == ASTRO_BOT_EXPLORE;
        any_idle |= modes[k] == ASTRO_BOT_NOTHING;
    }
    const bool all_stream = modes[0] == ASTRO_BOT_STREAM;   // (the counter stream drives every ship or none)
    if (b->rec_now.observations)                            // the recording ring: the state the bots are about to see
        if (int r = observe_impl(b, b->rec_now.observations, b->rec_now.n_rows, false, stream, (uint32_t)b->rec_now.ticks)) return r;
    {
        // a script bot writes every ship's control, the policy then overwrites the ships it drives
        if (any_script)
            if (int r = astro_script_controls(b, avoid_distance, avoid_threshold, actions, stream)) return r;
        if (any_idle && any_script) {
            // (NothingBot next to a ScriptBot: restore the idle column — one strided memset)
            for (int s = 0; s < b->S; s++)
                if (modes[s] == ASTRO_BOT_NOTHING)
                    CUDA_TRY(cudaMemset2DAsync(actions + s, b->S, 2, 1, (size_t)b->n_games, st));
        }
        if (any_policy) {
            int mask = 0;
            for (int s = 0; s < b->S; s++) mask |= (modes[s] == ASTRO_BOT_POLICY || modes[s] == ASTRO_BOT_EXPLORE) << s;
            if (int r = astro_policy_controls(b, actions, nullptr, mask, stream)) return r;
        }
        if (any_explore) {   // rl.QBotTrainer.__call__: the random policy, where active, replaces the greedy control
            int mask = 0;
            for (int s = 0; s < b->S; s++) mask |= (modes[s] == ASTRO_BOT_EXPLORE) << s;
            if (int r = astro_explore_controls(b, b->explore_t_in, b->explore_t_out, b->explore_seed, b->explore_state, actions, mask, stream)) return r;
        }
        if (int r = do_tick(b, all_stream ? nullptr : actions, nullptr, nullptr, events, flags, st)) return r;
    }
    return ASTRO_OK;
}

static GameArrays to_dev_arrays(const AstroGameArrays* a) {
    GameArrays d;
    d.ships = a->ships; d.planets = a->planets; d.bullets = a->bullets;
    d.n_planets = a->n_planets; d.n_bullets = a->n_bullets; d.tick = a->tick;
    d.finished = a->finished; d.episode = a->episode;
    return d;
}

int astro_export_games(AstroBatch* b, const int32_t* index, int32_t m, const AstroGameArrays* out, void* stream) {
    if (int r = check(b, true)) return r;
    if (!out || m < 0 || !out->ships || !out->planets || !out->n_planets || !out->n_bullets || !out->tick || !out->finished ||
        out->bullet_rows < 0 || (out->bullet_rows > 0 && !out->bullets))
        return fail(ASTRO_E_INVALID, "bad export arguments");
    if (!index && m > b->n_games) return fail(ASTRO_E_INVALID, "m %d > n_games %d", m, b->n_games);
    if (m == 0) return ASTRO_OK;
    CUDA_TRY(cudaSetDevice(b->device));
    const GameArrays a = to_dev_arrays(out);
    const AstroBuffers& u = b->bufs;
    const int grid = (m + 3) / 4;
    cudaStream_t st = (cudaStream_t)stream;
    with_layout(b, [&](auto r, auto s, auto pl) {
        export_kernel<typename decltype(r)::type, s, pl><<<grid, 128, 0, st>>>(u.ships, u.ship_b, u.planets, bullet_buffer(b, b->cur), u.meta,
                                                                                u.episode, index, m, b->n_games, b->K, out->bullet_rows, a);
    });
    CUDA_TRY(cudaGetLastError());
    b->launches += 1;
    return ASTRO_OK;
}

int astro_import_games(AstroBatch* b, const int32_t* index, int32_t m, const AstroGameArrays* in, void* stream) {
    if (int r = check(b, true)) return r;
    if (!in || m < 0 || !in->ships || !in->planets || !in->n_planets || in->bullet_rows < 0 ||
        (in->bullet_rows > 0 && in->n_bullets && !in->bullets))
        return fail(ASTRO_E_INVALID, "bad import arguments");
    if (!index && m > b->n_games) return fail(ASTRO_E_INVALID, "m %d > n_games %d", m, b->n_games);
    if (m == 0) return ASTRO_OK;
    CUDA_TRY(cudaSetDevice(b->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int32_t* src = nullptr;
    if (index) {
        if (!b->d_src) CUDA_TRY(cudaMalloc(&b->d_src, sizeof(int32_t) * (size_t)b->n_games));
        CUDA_TRY(cudaMemsetAsync(b->d_src, 0xff, sizeof(int32_t) * (size_t)b->n_games, st));
        import_map_kernel<<<(m + 255) / 256, 256, 0, st>>>(index, m, b->n_games, b->d_src);
        CUDA_TRY(cudaGetLastError());
        b->launches += 1;
        src = b->d_src;
    }
    const GameArrays a = to_dev_arrays(in);
    const AstroBuffers& u = b->bufs;
    void* cur = bullet_buffer(b, b->cur);
    void* other = bullet_buffer(b, b->cur ^ 1);
    const int grid = (b->n_games / ASTRO_TILE + 3) / 4;
    with_layout(b, [&](auto r, auto s, auto pl) {
        import_kernel<typename decltype(r)::type, s, pl><<<grid, 128, 0, st>>>(u.ships, u.ship_b, u.planets, cur, other, u.meta, u.episode,
                                                                                src, m, b->n_games, b->K, in->bullet_rows, a);
    });
    CUDA_TRY(cudaGetLastError());
    b->launches += 1;
    return ASTRO_OK;
}

int64_t astro_single_game_bytes(int32_t bullet_cap) {
    return (int64_t)sizeof(AstroSingleGame) + (int64_t)(bullet_cap > 0 ? bullet_cap : 0) * 4 * (int64_t)sizeof(double);
}

static AstroGameArrays single_arrays(char* rec, int32_t rows) {
    AstroSingleGame* g = reinterpret_cast<AstroSingleGame*>(rec);
    AstroGameArrays a;
    a.ships = &g->ships[0][0];
    a.planets = &g->planets[0][0];
    a.bullets = reinterpret_cast<double*>(rec + sizeof(AstroSingleGame));
    a.n_planets = &g->n_planets;
    a.n_bullets = &g->n_bullets;
    a.tick = &g->tick;
    a.finished = &g->finished[0];
    a.episode = &g->episode;
    a.bullet_rows = rows;
    a.reserved = 0;
    return a;
}

// The five operations of a single-game step (record in, import, tick, export, record out) are captured ONCE per
// (in, out, flags) into a CUDA graph and replayed: one graph launch per step instead of five API calls.  Every
// parameter of the sequence is fixed — the whole record travels, whatever the game's bullet count, and the lists are
// put back into bullet buffer 0 before every step.
static int single_graph_build(AstroBatch* b, const AstroSingleGame* in_host, AstroSingleGame* out_host, int32_t flags, SingleGraph* g) {
    const int64_t rec = b->single_bytes;
    char* d_in = b->d_single;
    char* d_out = b->d_single + rec;
    cudaStream_t st = b->single_stream;
    const size_t bytes = (size_t)astro_single_game_bytes(b->K);
    CUDA_TRY(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    int rc = ASTRO_OK;
    cudaError_t e = cudaMemcpyAsync(d_in, in_host, bytes, cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) rc = fail(ASTRO_E_CUDA, "record upload: %s", cudaGetErrorString(e));
    b->cur = 0;
    const AstroGameArrays ain = single_arrays(d_in, b->K);
    if (!rc) rc = astro_import_games(b, nullptr, 1, &ain, st);
    AstroSingleGame* g_in = reinterpret_cast<AstroSingleGame*>(d_in);
    AstroSingleGame* g_out = reinterpret_cast<AstroSingleGame*>(d_out);
    if (!rc) rc = do_tick(b, g_in->control, nullptr, nullptr, g_out->events, flags | ASTRO_TICK_NO_STATS, st);
    const AstroGameArrays aout = single_arrays(d_out, b->K);
    if (!rc) rc = astro_export_games(b, nullptr, 1, &aout, st);
    if (!rc) {
        e = cudaMemcpyAsync(out_host, d_out, bytes, cudaMemcpyDeviceToHost, st);
        if (e != cudaSuccess) rc = fail(ASTRO_E_CUDA, "record download: %s", cudaGetErrorString(e));
    }
    cudaGraph_t graph = nullptr;
    e = cudaStreamEndCapture(st, &graph);
    if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
    if (e != cudaSuccess) return fail(ASTRO_E_CUDA, "cudaStreamEndCapture: %s", cudaGetErrorString(e));
    e = cudaGraphInstantiate(&g->exec, graph, 0);
    cudaGraphDestroy(graph);
    if (e != cudaSuccess) return fail(ASTRO_E_CUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(e));
    g->in = in_host; g->out = out_host; g->flags = flags;
    return ASTRO_OK;
}

int astro_step_single_host(AstroBatch* b, const AstroSingleGame* in_host, AstroSingleGame* out_host, int32_t flags, void* stream) {
    if (int r = check(b, true)) return r;
    if (!in_host || !out_host) return fail(ASTRO_E_INVALID, "null record");
    if (b->n_games != ASTRO_TILE) return fail(ASTRO_E_INVALID, "astro_step_single_host needs a one-tile batch (n_games = %d)", ASTRO_TILE);
    const int32_t nb = in_host->n_bullets;
    if (nb < 0 || nb > b->K) return fail(ASTRO_E_INVALID, "the game holds %d bullets, bullet_cap is %d", nb, b->K);
    if (in_host->n_planets < 1 || in_host->n_planets > b->PL) return fail(ASTRO_E_INVALID, "a game needs 1..%d planets", b->PL);
    if (b->n_sched_ticks <= 0) return fail(ASTRO_E_STATE, "astro_set_schedule has not been called");
    if (in_host->tick < 0 || in_host->tick >= b->n_sched_ticks) return fail(ASTRO_E_INVALID, "tick %d is not on the schedule", in_host->tick);
    for (int s = 0; s < b->S; s++) {
        if (in_host->control[s] > 5) return fail(ASTRO_E_INVALID, "control code %d of ship %d is not one of 0..5", (int)in_host->control[s], s);
        if (!(fabs(in_host->ships[s][4]) <= kSinCosRange)) return fail(ASTRO_E_INVALID, "bearing %g of ship %d is beyond the range over which util.direction is reproduced", in_host->ships[s][4], s);
    }
    CUDA_TRY(cudaSetDevice(b->device));
    if (!b->d_single) {
        const int64_t rec = (astro_single_game_bytes(b->K) + 63) & ~(int64_t)63;
        CUDA_TRY(cudaMalloc(&b->d_single, (size_t)(2 * rec)));
        b->single_bytes = rec;
        CUDA_TRY(cudaStreamCreateWithFlags(&b->single_stream, cudaStreamNonBlocking));
        CUDA_TRY(cudaEventCreateWithFlags(&b->single_event, cudaEventDisableTiming));
    }
    SingleGraph* g = nullptr;
    for (int i = 0; i < kSingleGraphs; i++)
        if (b->single_graph[i].exec && b->single_graph[i].in == in_host && b->single_graph[i].out == out_host && b->single_graph[i].flags == flags)
            g = &b->single_graph[i];
    if (!g) {
        g = &b->single_graph[b->single_next++ % kSingleGraphs];
        if (g->exec) { cudaGraphExecDestroy(g->exec); g->exec = nullptr; }
        if (int r = single_graph_build(b, in_host, out_host, flags, g)) return r;
    }
    // earlier work of the caller's stream comes first; the step itself runs on the handle's own stream (a legacy
    // default stream cannot be captured) and is complete when the call returns
    CUDA_TRY(cudaEventRecord(b->single_event, (cudaStream_t)stream));
    CUDA_TRY(cudaStreamWaitEvent(b->single_stream, b->single_event, 0));
    b->cur = 0;
    CUDA_TRY(cudaGraphLaunch(g->exec, b->single_stream));
    CUDA_TRY(cudaStreamSynchronize(b->single_stream));
    b->cur = 1;          // the lists are where the tick wrote them
    b->launches += 3;
    return ASTRO_OK;
}

static void fresh_free(AstroBatch* b) {
    FreshState* fs = b->fresh;
    if (!fs) return;
    if (fs->producer) {
        fs->stop.store(1, std::memory_order_release);
        fs->producer->join();
        delete fs->producer;
    }
    cudaFree(fs->f.ring); cudaFree(fs->f.tile_used); cudaFree(fs->f.tasks); cudaFree(fs->f.cursor);
    cudaFree(const_cast<uint32_t*>(fs->f.seeds)); cudaFree(fs->game_pos); cudaFree(fs->chunk_base);
    cudaFreeHost(fs->h_seeds); cudaFreeHost(fs->h_cursor);
    for (int i = 0; i < kFreshLead; i++) if (fs->done[i]) cudaEventDestroy(fs->done[i]);
    if (fs->copy) cudaStreamDestroy(fs->copy);
    if (fs->seeds_sent) cudaEventDestroy(fs->seeds_sent);
    delete fs;
    b->fresh = nullptr;
}

int astro_fresh_games_enable(AstroBatch* b, const AstroCreateConfig* cc, uint32_t config_seed, int64_t skip, int32_t quota, void* stream) {
    if (int r = check(b, true)) return r;
    if (b->PL != ASTRO_MAX_PLANETS)
        return fail(ASTRO_E_INVALID, "fresh-game mode is not available in batches with %d planet slots (planet_slots = %d): use a reset pool",
                    b->PL, b->PL);
    if (!cc || cc->max_planets < 1 || cc->max_planets > ASTRO_MAX_PLANETS) return fail(ASTRO_E_INVALID, "bad create config");
    if (b->precision != 32) return fail(ASTRO_E_INVALID, "fresh-game mode needs the float32 build");
    if (quota < 1 || quota > 1024 || skip < 0) return fail(ASTRO_E_INVALID, "quota must be 1..1024, skip >= 0");
    CUDA_TRY(cudaSetDevice(b->device));
    cudaStream_t st = (cudaStream_t)stream;
    fresh_free(b);
    FreshState* fs = new (std::nothrow) FreshState();      // (value-initialised: every pointer / counter zero)
    if (!fs) return fail(ASTRO_E_NOMEM, "out of host memory");
    b->fresh = fs;
    const int n_tiles = b->n_games / ASTRO_TILE;
    fs->capacity = (int64_t)n_tiles * quota;
    fs->f.n_tiles = n_tiles; fs->f.quota = quota; fs->f.n_games = b->n_games;
    // seed ring: holds what the host may be ahead by (kFreshLead + 2 refills, or the initial fill of every game + every record), twice
    unsigned long long need = 2ull * (unsigned long long)(kFreshLead + 4) * (unsigned long long)fs->capacity;
    const unsigned long long first = 2ull * ((unsigned long long)b->n_games + (unsigned long long)fs->capacity);
    if (need < first) need = first;
    unsigned long long ring = 1024;
    while (ring < need) ring <<= 1;
    if (ring > (1ull << 31)) { fresh_free(b); return fail(ASTRO_E_INVALID, "batch too large for the seed ring"); }
    fs->f.seed_mask = (uint32_t)(ring - 1);
    fs->cq.inner = cc->inner_ship_position; fs->cq.outer = cc->outer_ship_position; fs->cq.orbit = cc->planet_orbit;
    fs->cq.gravity = b->cfg.gravity; fs->cq.planet_mass = b->cfg.planet_mass;
    fs->cq.max_planets = cc->max_planets; fs->cq.solo = b->cfg.solo; fs->cq.m = 0; fs->cq.pad = 0;
    cudaError_t e = cudaMalloc(&fs->f.ring, (size_t)fs->capacity * 128);
    if (e == cudaSuccess) e = cudaMalloc(&fs->f.tile_used, sizeof(uint32_t) * (size_t)n_tiles);
    if (e == cudaSuccess) e = cudaMalloc(&fs->f.tasks, sizeof(uint32_t) * (size_t)fs->capacity);
    if (e == cudaSuccess) e = cudaMalloc(&fs->f.cursor, 4 * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMalloc(const_cast<uint32_t**>(&fs->f.seeds), sizeof(uint32_t) * (size_t)ring);
    if (e == cudaSuccess) e = cudaMalloc(&fs->game_pos, sizeof(uint32_t) * (size_t)b->n_games);
    if (e == cudaSuccess) e = cudaMalloc(&fs->chunk_base, sizeof(uint32_t) * (size_t)((n_tiles + 31) / 32 + 1));
    if (e == cudaSuccess) e = cudaMallocHost(&fs->h_seeds, sizeof(uint32_t) * (size_t)ring);
    if (e == cudaSuccess) e = cudaMallocHost(&fs->h_cursor, 4 * sizeof(unsigned long long));
    for (int i = 0; i < kFreshLead && e == cudaSuccess; i++) e = cudaEventCreateWithFlags(&fs->done[i], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&fs->copy, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&fs->seeds_sent, cudaEventDisableTiming);
    if (e != cudaSuccess) { fresh_free(b); return fail(ASTRO_E_CUDA, "fresh-game buffers: %s", cudaGetErrorString(e)); }
    fs->mt.seed(config_seed);
    for (int64_t i = 0; i < skip; i++) fs->mt.next();
    // the stream positions count from `skip`: position p is generate_configs draw number p
    fs->generated = (unsigned long long)skip;
    fs->produced.store((unsigned long long)skip);
    fs->target.store((unsigned long long)skip);
    fs->stop.store(0);
    fs->producer = new (std::nothrow) std::thread(fresh_producer_main, fs);
    if (!fs->producer) { fresh_free(b); return fail(ASTRO_E_NOMEM, "out of host memory"); }
    const unsigned long long start[4] = {(unsigned long long)skip, 0ull, 0ull, 0ull};
    memcpy(fs->h_cursor, start, sizeof(start));
    CUDA_TRY(cudaMemcpyAsync(fs->f.cursor, fs->h_cursor, sizeof(start), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemsetAsync(fs->game_pos, 0xff, sizeof(uint32_t) * (size_t)b->n_games, st));
    // every record is "used": the first refill creates the whole ring
    std::vector<uint32_t> full((size_t)n_tiles, (uint32_t)quota);
    CUDA_TRY(cudaMemcpyAsync(fs->f.tile_used, full.data(), sizeof(uint32_t) * (size_t)n_tiles, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaStreamSynchronize(st));   // (`full` is pageable and leaves scope)
    return fresh_refill(b, st);
}

int astro_fresh_games_reset_all(AstroBatch* b, void* stream) {
    if (int r = check(b, true)) return r;
    FreshState* fs = b->fresh;
    if (!fs) return fail(ASTRO_E_STATE, "astro_fresh_games_enable has not been called");
    CUDA_TRY(cudaSetDevice(b->device));
    cudaStream_t st = (cudaStream_t)stream;
    // the device's cursor is read exactly (a rare call): the next n_games positions start there
    CUDA_TRY(cudaStreamSynchronize(st));
    unsigned long long cur[2];
    CUDA_TRY(cudaMemcpy(cur, fs->f.cursor, sizeof(cur), cudaMemcpyDeviceToHost));
    fs->h_cursor[0] = cur[0]; fs->h_cursor[1] = cur[1];
    if (int r = fresh_upload_seeds(b, cur[0] + (unsigned long long)b->n_games + (unsigned long long)fs->capacity, st)) return r;
    const AstroBuffers& u = b->bufs;
    const int grid = (b->n_games + 63) / 64;
    if (b->S == 2) fresh_fill_kernel<2><<<grid, 64, 0, st>>>(fs->f, fs->cq, (float4*)u.ships, (float*)u.ship_b, (float4*)u.planets, u.meta, u.episode, fs->game_pos);
    else fresh_fill_kernel<1><<<grid, 64, 0, st>>>(fs->f, fs->cq, (float4*)u.ships, (float*)u.ship_b, (float4*)u.planets, u.meta, u.episode, fs->game_pos);
    fresh_fill_commit_kernel<<<1, 1, 0, st>>>(fs->f);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(fs->h_cursor, fs->f.cursor, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    b->launches += 2;
    b->step = 0;
    return ASTRO_OK;
}

int astro_fresh_games_refill(AstroBatch* b, void* stream) {
    if (int r = check(b, true)) return r;
    if (!b->fresh) return fail(ASTRO_E_STATE, "astro_fresh_games_enable has not been called");
    CUDA_TRY(cudaSetDevice(b->device));
    return fresh_refill(b, (cudaStream_t)stream);
}

int astro_fresh_games_positions(AstroBatch* b, uint32_t* positions_dev, uint32_t* tile_used_dev, int64_t* cursor_host, void* stream) {
    if (int r = check(b, true)) return r;
    FreshState* fs = b->fresh;
    if (!fs) return fail(ASTRO_E_STATE, "astro_fresh_games_enable has not been called");
    CUDA_TRY(cudaSetDevice(b->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (positions_dev) CUDA_TRY(cudaMemcpyAsync(positions_dev, fs->game_pos, sizeof(uint32_t) * (size_t)b->n_games, cudaMemcpyDeviceToDevice, st));
    if (tile_used_dev) CUDA_TRY(cudaMemcpyAsync(tile_used_dev, fs->f.tile_used, sizeof(uint32_t) * (size_t)fs->f.n_tiles, cudaMemcpyDeviceToDevice, st));
    if (cursor_host) {
        CUDA_TRY(cudaStreamSynchronize(st));
        unsigned long long cur = 0;
        CUDA_TRY(cudaMemcpy(&cur, fs->f.cursor, sizeof(cur), cudaMemcpyDeviceToHost));
        *cursor_host = (int64_t)cur;
    }
    return ASTRO_OK;
}

int astro_config_seeds(uint32_t config_seed, int64_t skip, int64_t count, uint32_t* out_host) {
    if (!out_host || skip < 0 || count < 0) return fail(ASTRO_E_INVALID, "bad arguments");
    HostMt19937 mt;
    mt.seed(config_seed);
    for (int64_t i = 0; i < skip; i++) mt.next();
    for (int64_t i = 0; i < count; i++) out_host[i] = mt.next() & 0x3fffffffu;
    return ASTRO_OK;
}

int astro_nstep_experiences(AstroBatch* b, const uint8_t* events, int32_t n_ticks, int32_t n_steps, double discount, int32_t* carry,
                            float* out_reward, float* out_discount, int32_t* out_next, void* stream) {
    if (int r = check(b, false)) return r;
    if (!events || !carry || !out_reward || !out_discount || !out_next) return fail(ASTRO_E_INVALID, "null argument");
    if (n_ticks < 0 || n_steps < 1 || !(discount > 0.0)) return fail(ASTRO_E_INVALID, "bad n-step arguments");
    CUDA_TRY(cudaSetDevice(b->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = (b->n_games * b->S + 127) / 128;
    if (b->S == 2) nstep_kernel<2><<<grid, 128, 0, st>>>(events, n_ticks, b->n_games, n_steps, discount, b->c.reward_timeout, carry, out_reward, out_discount, out_next);
    else nstep_kernel<1><<<grid, 128, 0, st>>>(events, n_ticks, b->n_games, n_steps, discount, b->c.reward_timeout, carry, out_reward, out_discount, out_next);
    CUDA_TRY(cudaGetLastError());
    b->launches += 1;
    return ASTRO_OK;
}

int astro_stats(AstroBatch* b, int64_t* counters_dev, int32_t clear, void* stream) {
    if (int r = check(b, false)) return r;
    if (!counters_dev) return fail(ASTRO_E_INVALID, "null counters");
    CUDA_TRY(cudaSetDevice(b->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (b->ticks_since_fold > 0) CUDA_TRY(fold_stats(b, st));
    gather_stats_kernel<<<1, 256, 0, st>>>(b->d_stats, (long long*)counters_dev, clear ? 1 : 0);
    CUDA_TRY(cudaGetLastError());
    return ASTRO_OK;
}

int astro_value_forward(AstroBatch* b, const float* features, int32_t n_items, int32_t rows, float* q_out, void* stream) {
    if (int r = check(b, false)) return r;
    if (b->policy_nout <= 0 || !b->d_pol_frags) return fail(ASTRO_E_STATE, "astro_policy_set_weights has not been called");
    if (!features || !q_out) return fail(ASTRO_E_INVALID, "null argument");
    if (n_items < 0 || rows < 1) return fail(ASTRO_E_INVALID, "n_items >= 0 and rows >= 1");
    if (n_items == 0) return ASTRO_OK;
    CUDA_TRY(cudaSetDevice(b->device));
    cudaStream_t st = (cudaStream_t)stream;
    int grid = ((n_items + 15) / 16 + kMmaWarps - 1) / kMmaWarps;      // a warp takes 16 items at a time
    if (grid > b->sm_count * ASTRO_MMA_MIN_BLOCKS) grid = b->sm_count * ASTRO_MMA_MIN_BLOCKS;
    const int smem = (int)sizeof(PolicyFrags);
    if (b->S == 2) {
        CUDA_TRY(cudaFuncSetAttribute(value_forward_kernel<15>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        value_forward_kernel<15><<<grid, kMmaWarps * 32, smem, st>>>(features, q_out, n_items, rows, b->policy_nout, b->d_pol_frags);
    } else {
        CUDA_TRY(cudaFuncSetAttribute(value_forward_kernel<10>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        value_forward_kernel<10><<<grid, kMmaWarps * 32, smem, st>>>(features, q_out, n_items, rows, b->policy_nout, b->d_pol_frags);
    }
    CUDA_TRY(cudaGetLastError());
    b->launches += 1;
    return ASTRO_OK;
}

int astro_stats_peer_create(AstroBatch* b, int32_t rank, int32_t world, uint8_t* handle_out) {
    if (int r = check(b, false)) return r;
    if (!handle_out) return fail(ASTRO_E_INVALID, "null handle_out");
    if (world < 1 || world > kPeerMax || rank < 0 || rank >= world) return fail(ASTRO_E_INVALID, "rank %d of %d: 1..%d ranks", rank, world, kPeerMax);
    if (b->d_peer_own) return fail(ASTRO_E_STATE, "the exchange buffer of this batch exists already");
    static_assert(sizeof(cudaIpcMemHandle_t) == ASTRO_IPC_HANDLE_BYTES, "ASTRO_IPC_HANDLE_BYTES");
    CUDA_TRY(cudaSetDevice(b->device));
    const size_t bytes = sizeof(unsigned long long) * 2 * kPeerMax * 16;
    CUDA_TRY(cudaMalloc(&b->d_peer_own, bytes));
    CUDA_TRY(cudaMemset(b->d_peer_own, 0, bytes));
    CUDA_TRY(cudaDeviceSynchronize());
    cudaIpcMemHandle_t h;
    CUDA_TRY(cudaIpcGetMemHandle(&h, b->d_peer_own));
    memcpy(handle_out, &h, sizeof(h));
    b->peer_rank = rank;
    b->peer_world = world;
    b->peer_calls = 0;
    return ASTRO_OK;
}

int astro_stats_peer_open(AstroBatch* b, const uint8_t* handles) {
    if (int r = check(b, false)) return r;
    if (!handles) return fail(ASTRO_E_INVALID, "null handles");
    if (!b->d_peer_own) return fail(ASTRO_E_STATE, "astro_stats_peer_create has not been called");
    if (b->peer_open) return fail(ASTRO_E_STATE, "the peers' buffers are mapped already");
    CUDA_TRY(cudaSetDevice(b->device));
    memset(&b->peer_table, 0, sizeof(b->peer_table));
    for (int r = 0; r < b->peer_world; r++) {
        if (r == b->peer_rank) { b->peer_table.buf[r] = b->d_peer_own; continue; }
        cudaIpcMemHandle_t h;
        memcpy(&h, handles + (size_t)r * ASTRO_IPC_HANDLE_BYTES, sizeof(h));
        void* ptr = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            cudaGetLastError();
            for (int q = 0; q < r; q++)
                if (q != b->peer_rank && b->peer_table.buf[q]) cudaIpcCloseMemHandle(b->peer_table.buf[q]);
            memset(&b->peer_table, 0, sizeof(b->peer_table));
            return fail(ASTRO_E_CUDA, "cudaIpcOpenMemHandle (rank %d): %s", r, cudaGetErrorString(e));
        }
        b->peer_table.buf[r] = (unsigned long long*)ptr;
    }
    b->peer_open = true;
    return ASTRO_OK;
}

int astro_stats_allreduce(AstroBatch* b, int64_t* counters_dev, int32_t clear, void* stream) {
    if (int r = check(b, false)) return r;
    if (!counters_dev) return fail(ASTRO_E_INVALID, "null counters");
    if (!b->peer_open) return fail(ASTRO_E_STATE, "astro_stats_peer_open has not been called");
    CUDA_TRY(cudaSetDevice(b->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (b->ticks_since_fold > 0) CUDA_TRY(fold_stats(b, st));
    b->peer_calls += 1;
    stats_allreduce_kernel<<<1, 256, 0, st>>>(b->d_stats, (long long*)counters_dev, clear ? 1 : 0, b->peer_table, b->peer_rank, b->peer_world,
                                             b->peer_calls);
    CUDA_TRY(cudaGetLastError());
    return ASTRO_OK;
}

int64_t astro_launch_count(const AstroBatch* b) { return b ? b->launches : 0; }

int astro_bullet_buffer(const AstroBatch* b) { return b ? b->cur : ASTRO_E_INVALID; }

int astro_set_bullet_buffer(AstroBatch* b, int32_t which) {
    if (int r = check(b, false)) return r;
    if (which != 0 && which != 1) return fail(ASTRO_E_INVALID, "bullet buffer must be 0 or 1");
    b->cur = which;
    return ASTRO_OK;
}

#ifdef ASTRO_TIMELINE
// experiment builds only (tools/exp_timeline.py): device buffer of 8 clock stamps per tile
int astro_debug_set_timeline(long long* buf_dev) {
    return cudaMemcpyToSymbol(g_timeline, &buf_dev, sizeof(buf_dev)) == cudaSuccess ? 0 : -1;
}
#endif

}  // extern "C"
