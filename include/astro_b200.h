/*
 * astro_b200.h — C ABI of the B200-native batched Astro game tick.
 *
 * The reference (DouglasOrr/Astro) has no FFI layer: its boundary for this path is the
 * Python game API of astro/core.py (create/step/roll_ships/play) and
 * astro/rl.py ValueNetwork.get_features, get_features_batch and to_batch.  This header is the C-ABI a maintainer
 * would bind (ctypes, see INTEGRATION.md) to replace the bodies of those functions with the
 * CUDA path; each entry point cites the reference lines it replaces.
 *
 * Conventions
 *   - every function returns 0 on success or a negative ASTRO_E_* code; no C++ exception
 *     crosses the ABI; astro_last_error() gives the message of the calling thread's last
 *     failure.
 *   - all state memory is OWNED BY THE CALLER (PyTorch tensors in practice) and bound with
 *     astro_batch_bind(); pointers must stay valid while bound.
 *   - kernels are enqueued on the caller's CUDA stream (cudaStream_t passed as void*); calls
 *     are asynchronous unless the name ends in _host.  One handle per device; a handle is not
 *     re-entrant.
 *   - one Config per batch (the reference also passes one config per game loop).
 *
 * Device data layout ("tiles"): games are grouped in tiles of ASTRO_TILE = 32 consecutive
 * games (one warp).  R is float (precision 32) or double (precision 64); R4 = {x, y, dx, dy}.
 *     ships    R4  [n_tiles][S][32]      ship s of game g  -> ((g/32)*S + s)*32 + g%32
 *     ship_b   R   [n_tiles][S][32]      bearing
 *     planets  R4  [n_tiles][PL][32]     slots >= np are dead; PL = the batch's planet slots (4, or 8 for
 *                                        AstroConfig.planet_slots = 8: games of up to eight planets)
 *     bullets  R4  [2][n_tiles][32*K]    TILE LISTS, two buffers.  In the current buffer
 *                                        (astro_bullet_buffer()) tile t's run holds the bullets of its
 *                                        32 games back to back, no gaps: game g's bullets are items
 *                                        first(g) .. first(g)+nb(g)-1 with first(g) = sum of nb over
 *                                        the tile's lower games (finished games: nb = 0), in
 *                                        reference order; the rest of the run (capacity 32*K) is
 *                                        dead.  Every astro_tick reads the current buffer, writes
 *                                        the tile's new list into the other one and flips.
 *     meta     u32 [n_tiles*32]          nb (bits 0-9) | np (10-12) | finished (13) | tick (14-31)
 *                                        8-slot batches: np bit 3 in bit 31, tick in bits 14-30 (ASTRO_META_*_WIDE)
 *     episode  u32 [n_tiles*32]          games finished in this slot (a counter; bumped on reset)
 * Ships, planets and meta are accessed thread-per-game: every load/store is a fully coalesced
 * 128-bit (R=float) access across the warp.  A tile's bullets are one contiguous run in HBM (3 KB
 * on average instead of 32 runs of ~90 B): the warp reads it 512 B per step and writes the new
 * list the same way (see csrc/tick_f32.cuh).
 */
#ifndef ASTRO_B200_H
#define ASTRO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ASTRO_ABI_VERSION 5   /* 5: AstroConfig.planet_slots, AstroSingleGame.planets[ASTRO_MAX_PLANETS_WIDE] */
#define ASTRO_TILE 32
#define ASTRO_MAX_SHIPS 2
#define ASTRO_MAX_PLANETS 4
#define ASTRO_MAX_PLANETS_WIDE 8 /* AstroConfig.planet_slots = 8 */
#define ASTRO_MAX_BULLET_CAP 1023
#define ASTRO_MAX_TICKS 262143 /* 18-bit per-game tick counter */
#define ASTRO_MAX_TICKS_WIDE 131071 /* 17 bits in 8-slot batches */

/* meta word */
#define ASTRO_META_NB(m) ((m) & 1023u)
#define ASTRO_META_NP(m) (((m) >> 10) & 7u)
#define ASTRO_META_FINISHED(m) (((m) >> 13) & 1u)
#define ASTRO_META_TICK(m) ((m) >> 14)
#define ASTRO_META_PACK(nb, np, fin, tick) \
    ((uint32_t)(nb) | ((uint32_t)(np) << 10) | ((uint32_t)(fin) << 13) | ((uint32_t)(tick) << 14))
/* meta word of an 8-slot batch: np = 8 needs a fourth bit, which sits in bit 31; nb, the low three bits of np and the
 * finished bit stay where they are, and so does the tick's lowest bit (a tick still advances by + (1 << 14)) */
#define ASTRO_META_NP_WIDE(m) ((((m) >> 10) & 7u) | (((m) >> 28) & 8u))
#define ASTRO_META_TICK_WIDE(m) (((m) >> 14) & 0x1ffffu)
#define ASTRO_META_PACK_WIDE(nb, np, fin, tick)                                                                    \
    ((uint32_t)(nb) | (((uint32_t)(np) & 7u) << 10) | ((uint32_t)(fin) << 13) | ((uint32_t)(tick) << 14) |      \
     (((uint32_t)(np) & 8u) << 28))

/* per-game event bits written by astro_tick (u8 per game) */
#define ASTRO_EV_HIT0 1      /* ship 0 collided   (core.py:253-255) */
#define ASTRO_EV_HIT1 2      /* ship 1 collided */
#define ASTRO_EV_TIMEOUT 4   /* max_time reached  (core.py:257-260) */
#define ASTRO_EV_FIRED 8     /* ships fired this tick (core.py:267-280) */
#define ASTRO_EV_OVERFLOW 16 /* a newborn bullet was dropped: pool full */
#define ASTRO_EV_SKIPPED 32  /* game was already finished; nothing done */
#define ASTRO_EV_BAD_CONTROL 64 /* a control code above 5 was given (out of the reference's contract, core.py:220-227):
                                   the ship was flown with control 2 (no thrust, no turn) and the tick flagged */
#define ASTRO_EV_AWAIT 128 /* fresh-game mode: the game ended but its tile had no pre-created game left: it waits, frozen,
                              and is re-created by the first tick after the next refill (counted in astro_stats) */
#define ASTRO_EV_DONE_MASK 7

/* astro_tick flags */
#define ASTRO_TICK_AUTO_RESET 1 /* a game that ends is re-initialised from the reset pool in the same launch */
#define ASTRO_TICK_NO_STATS 2   /* skip the astro_stats counters for this tick */
#define ASTRO_TICK_GENERIC_KERNEL 4 /* precision 32 only: run the un-tuned template kernel (A/B checks) */
/* precision 64 only: a game on its tick 0 (bit 8) / every game of this call (bit 16) that owns no bullets is taken to
 * hold the arrays core.create returned (core.py:86-135: float32 ship / planet positions) and runs the reference's
 * first-tick arithmetic — _gravity, the squared distances of _collisions and the planets' a * dt in float32, bullets
 * born on that tick float32 throughout — so that a game played from create() equals the reference's core.play bit for
 * bit.  Without it tick 0 treats its inputs as float64 like every other tick (states canonicalised to float64). */
#define ASTRO_TICK_CREATE_DTYPES 8
#define ASTRO_TICK_ALL_CREATE_DTYPES 16
/* Compact host traffic (astro_tick, astro_tick_many and the _host forms; duel games, the float32 kernel):
 *   PACKED_CONTROLS  actions are u8 [n_games]: one byte per GAME, ship 0's code in bits 0-2, ship 1's in bits 3-5
 *                    (the two codes of core.py:220-227 need 6 bits) — half the bytes of [n_games][2].
 *   EVENT_PLANES     events are u32 [3][n_games / 32] per tick, three bit planes: bit g % 32 of word g / 32 of plane 0 =
 *                    game g ended this tick, plane 1 = ship 0 was hit, plane 2 = ship 1 was hit (ended with neither:
 *                    timeout) — everything core.step's (state is None, reward) carries (core.py:253-260), in 12 bytes
 *                    per 32 games instead of 32.  ASTRO_EV_FIRED is a function of the schedule; overflow / skipped /
 *                    bad-control ticks are counted by astro_stats. */
#define ASTRO_TICK_PACKED_CONTROLS 32
#define ASTRO_TICK_EVENT_PLANES 64

/* error codes */
#define ASTRO_OK 0
#define ASTRO_E_INVALID (-1)
#define ASTRO_E_CUDA (-2)
#define ASTRO_E_STATE (-3)
#define ASTRO_E_NOMEM (-4)

/* World part of the reference Config (core.py:20-41; defaults core.py:52-74). */
typedef struct AstroConfig {
    double gravity, dt, max_time, reload_time, bullet_speed, ship_thrust, ship_rspeed, ship_radius,
        planet_mass, planet_radius;
    int32_t solo; /* 1 -> one ship per game */
    int32_t planet_slots; /* planet slots per game: 0 or 4 (ASTRO_MAX_PLANETS), or 8 (ASTRO_MAX_PLANETS_WIDE) for games of
                             up to eight planets.  The game-major arrays of the batch (AstroResetPool, astro_create_games,
                             AstroGameArrays) then hold that many planet rows per game. */
} AstroConfig;

/* Device pointers of the caller-owned state (layout above; bullets = both buffers, contiguous). */
typedef struct AstroBuffers {
    void* ships;
    void* ship_b;
    void* planets;
    void* bullets;
    uint32_t* meta;
    uint32_t* episode;
} AstroBuffers;

/* Reset pool: M initial states built by create() (core.py:86-135) on the host, in device
 * memory, game-major: ships R [M][S][5] = x,y,dx,dy,b ; planets R [M][PL][4] ; np i32 [M]. */
typedef struct AstroResetPool {
    const void* ships;
    const void* planets;
    const int32_t* np;
    int32_t size;
    int32_t reserved;
} AstroResetPool;

/* Creation part of the reference Config (core.py:30-41; defaults core.py:64-71); gravity,
 * planet_mass and solo come from the batch's AstroConfig, the seed is per game. */
typedef struct AstroCreateConfig {
    double inner_ship_position, outer_ship_position, planet_orbit;
    int32_t max_planets;
    int32_t reserved;
} AstroCreateConfig;

#define ASTRO_N_STATS 14
/* astro_stats counters (int64 each), summed over every astro_tick since the last clear:
 *  0 episodes  1 wins0  2 wins1  3 both_lost (or solo crash)  4 timeouts  5 env_steps
 *  6 bullets_spawned  7 overflow  8 planets_live (sum of np over env-steps)
 *  9 bullets_in (sum of nb read)  10 bullets_out (sum of nb written)  11 skipped
 *  12 bad_controls (env-steps that saw a control code above 5)
 *  13 awaiting (fresh-game mode: games that ended with their tile's ring of pre-created games empty)  */

typedef struct AstroBatch AstroBatch;

int astro_abi_version(void);
const char* astro_last_error(void);

/* Batch lifetime.  n_games is rounded up to whole tiles by the caller: n_games % 32 == 0.
 * precision: 32 (float state; predicates exact via fp64 fallback) or 64 (double state, the
 * validation build: bit-identical to the reference's float64 arithmetic). */
int astro_batch_create(const AstroConfig* cfg, int32_t n_games, int32_t bullet_cap, int32_t precision,
                       int32_t device, AstroBatch** out);
int astro_batch_destroy(AstroBatch* b);
int astro_batch_bind(AstroBatch* b, const AstroBuffers* bufs);   /* the lists are in bullet buffer 0 after a bind */

/* Which of the two bullet buffers holds the tile lists right now (0 or 1): what a host-side reader or
 * writer of `bullets` (to_state, set_states) must index with.  astro_set_bullet_buffer declares where
 * the caller has put them (e.g. after restoring a saved batch). */
int astro_bullet_buffer(const AstroBatch* b);
int astro_set_bullet_buffer(AstroBatch* b, int32_t which);

/* reload / t are Python-float accumulators in the reference (core.py:257-280,302): a pure
 * function of the tick index.  The host evaluates them once, in the reference's arithmetic,
 * and hands over: bit k of fire_bits = "ships fire on a game's k-th tick", and the tick index
 * on which the timeout terminal fires.  n_ticks = timeout_tick + 1. */
int astro_set_schedule(AstroBatch* b, const uint32_t* fire_bits_host, int32_t n_ticks, int32_t timeout_tick);

/* Counter-stream keys (astro_b200/rng.py): controls when actions == NULL, reset-pool picks. */
int astro_set_stream(AstroBatch* b, uint32_t seed, int64_t first_game, uint32_t step);
/* The pool is SNAPSHOT by this call (precision 32: repacked into one 128-byte record per entry — 256 bytes in 8-slot
 * batches — which the tick kernel reads); call it again after changing the pool's contents.  Synchronises the device. */
int astro_set_reset_pool(AstroBatch* b, const AstroResetPool* pool);

/* core.step (core.py:215-303) for every game of the batch: one fused kernel.
 *   actions  u8 [n_games][S] device, control codes 0..5 (core.py:220-227); NULL -> counter stream
 *   reward   f32 [n_games][S] device or NULL   (core.py:255,260,303)
 *   done     u8 [n_games] device or NULL       (reference returns state None)
 *   events   u8 [n_games] device or NULL       (ASTRO_EV_*)
 * Each call advances the batch's stream step by one. */
int astro_tick(AstroBatch* b, const uint8_t* actions, float* reward, uint8_t* done, uint8_t* events,
               int32_t flags, void* stream);

/* n_ticks consecutive astro_tick calls in as few launches as possible: actions u8 [n_ticks][n_games][S] (NULL ->
 * counter stream), reward f32 [n_ticks][n_games][S], done / events u8 [n_ticks][n_games] (each may be NULL), all on
 * the device.  Games do not interact, so the production kernel (precision 32) runs up to 256 ticks of a tile back to
 * back inside one launch: what tick k wrote is what tick k+1 reads, from L2 instead of HBM, and there is no launch
 * boundary between them.  Results are identical to n_ticks separate astro_tick calls.  This is the loop of core.play /
 * rl.train (core.py:388-404) whenever the controls of a block of ticks do not depend on the states inside the block
 * (replays, random or pre-computed exploration, the counter stream). */
int astro_tick_many(AstroBatch* b, const uint8_t* actions, float* reward, uint8_t* done, uint8_t* events, int32_t n_ticks,
                    int32_t flags, void* stream);

/* Same call with HOST buffers (pinned for full speed): H2D actions, tick, D2H events (and
 * reward/done when not NULL), then synchronises the stream.  Large float32 batches asked for events only run the tick as
 * two slices of tiles on internal streams, so that one slice's copies overlap the other's kernel. */
int astro_tick_host(AstroBatch* b, const uint8_t* actions_host, float* reward_host, uint8_t* done_host,
                    uint8_t* events_host, int32_t flags, void* stream);

/* astro_tick_host in two halves, for a closed loop over SEVERAL batches: _begin enqueues the copy in, the tick and the copy
 * of the events out on `stream` and returns at once; _end blocks until those events are on the host.  Games are
 * independent, so a host policy can hold the games as two (or more) batches on their own streams and alternate —
 * while batch A's tick runs, batch B's events travel back, its policy is evaluated and its next controls travel in
 * (every batch still sees its tick k events before it gives its tick k + 1 controls: the loop of core.play /
 * rl.train, core.py:388-404, per batch).  One tick may be pending per handle. */
int astro_tick_host_begin(AstroBatch* b, const uint8_t* actions_host, uint8_t* events_host, int32_t flags, void* stream);
int astro_tick_host_end(AstroBatch* b);

/* n_ticks consecutive astro_tick_host calls as one pipelined stream: actions_host u8
 * [n_ticks][n_games][S], events_host u8 [n_ticks][n_games] (pinned).  Ticks travel in chunks of 4: the
 * controls of the next chunk are copied in while this chunk runs as one launch (astro_tick_many) and the events of
 * the previous chunk are copied out (two internal copy streams, double-buffered staging; ASTRO_ROLLOUT_CHUNK overrides).  Returns when every event byte is on the host.  This is
 * the rollout loop of core.play / rl.train (core.py:388-404) for a host-side policy whose controls
 * for a block of ticks are known up front (replays, scripted or random play). */
int astro_rollout_host(AstroBatch* b, const uint8_t* actions_host, uint8_t* events_host, int32_t n_ticks,
                       int32_t flags, void* stream);

/* Re-initialise finished games from the reset pool (the stand-alone form of AUTO_RESET).
 * Pool entry = pick(seed, global game id, key): key = 0 for the initial fill, 1 + the stream step of
 * the tick that ended the game for AUTO_RESET, the current stream step here. */
int astro_reset_done(AstroBatch* b, void* stream);

/* rl.ValueNetwork.get_features + to_batch (rl.py:43-99) with core.roll_ships (core.py:306-327)
 * for both perspectives: obs f32 [n_games][S][n_rows][1+5S+4] device; rows = planets then
 * bullets, the rest filled with -1; n_rows >= PL + bullet_cap.  Finished games: all -1. */
int astro_observe(AstroBatch* b, float* obs, int32_t n_rows, void* stream);

/* The same features written ONCE: obs f32 [n_games][n_rows][1+5S+4], ship 0's perspective only.
 * Ship 1's view of the same game (core.roll_ships, core.py:306-327, then rl.py:62-70) is this block
 * with the two ship column groups exchanged (columns 1..5 <-> 6..10), every other column and the
 * -1 padding being perspective-free — a consumer applies the exchange to its first-layer weights
 * instead of reading a second tensor (astro_b200/rl.py ValueNetwork.forward_both): half the
 * observation bytes written and read. */
int astro_observe_shared(AstroBatch* b, float* obs, int32_t n_rows, void* stream);

/* core.create (core.py:86-135) for m seeds at once, on the device: numpy RandomState(seed) (MT19937,
 * legacy randint / rand / choice draws in the reference's order) and the reference's float32 /
 * float64 arithmetic, bit for bit.  seeds u32 [m] device (core.generate_configs, core.py:77-83, is
 * RandomState(config.seed).randint(2**30) per game: astro_b200/rng.py config_seeds).  Output in
 * the AstroResetPool layout, batch precision R: ships R [m][S][5], planets R [m][PL][4] (dead slots
 * zero), max_planets <= PL, n_planets i32 [m] — pass it to astro_set_reset_pool, or refresh it between rollouts so
 * that re-created games never repeat. */
int astro_create_games(AstroBatch* b, const AstroCreateConfig* cc, const uint32_t* seeds, int32_t m, void* ships,
                       void* planets, int32_t* n_planets, void* stream);

/* Fresh games without a pool: core.generate_configs + core.create (core.py:77-135) for EVERY re-creation, the way
 * core.play / rl.train start every episode from the next config of the stream (rl.py:350,374).  float32 build.
 *   _enable     every tile of 32 games gets a ring of `quota` pre-created games; ASTRO_TICK_AUTO_RESET then re-creates a game
 *               that ends from its tile's next unused record (a warp-local count: no atomics, no dependent address), and
 *               between launches the used records are re-created from the NEXT positions of the stream — positions handed
 *               out by a prefix sum in tile order (reproducible), seeds drawn on the host exactly like
 *               numpy.random.RandomState(config_seed).randint(2**30) and uploaded ahead of the device.  Every position of
 *               the stream (from `skip`) is consumed exactly once: no initial state repeats unless the stream itself does.
 *               A tile that uses its whole quota between two refills (quota 48 covers 64-tick launches of random play)
 *               leaves the game frozen (ASTRO_EV_AWAIT) until the next refill; nothing is ever re-used.
 *   _reset_all  (re)starts every game of the batch from the next n_games positions (synchronises the stream).
 *   _refill     an explicit refill (astro_tick / astro_tick_many refill by themselves, about every quota / 2 ticks).
 *   _positions  positions_dev u32 [n_games] <- stream position of each game's current episode; tile_used_dev u32 [n_tiles]
 *               <- records used since the last refill; *cursor_host <- positions handed out so far (synchronises). */
int astro_fresh_games_enable(AstroBatch* b, const AstroCreateConfig* cc, uint32_t config_seed, int64_t skip, int32_t quota, void* stream);
int astro_fresh_games_reset_all(AstroBatch* b, void* stream);
int astro_fresh_games_refill(AstroBatch* b, void* stream);
int astro_fresh_games_positions(AstroBatch* b, uint32_t* positions_dev, uint32_t* tile_used_dev, int64_t* cursor_host, void* stream);
/* The seeds of core.generate_configs (core.py:77-83) on the host: RandomState(config_seed).randint(2**30), draws number
 * skip .. skip + count - 1 (the library's own MT19937; pinned against numpy in the tests). */
int astro_config_seeds(uint32_t config_seed, int64_t skip, int64_t count, uint32_t* out_host);

/* script.ScriptBot.__call__ (script.py:13-91: _danger, _fly_to) for every ship of every game, each
 * seeing the game from its own perspective (core.roll_ships, core.py:306-327):
 * actions u8 [n_games][S] device, control codes 0..5; finished games get 2 (no-op).  The
 * reference's tuned arguments are avoid_distance 0.1, avoid_threshold 0.45 (script.py:16-20).
 * The output is directly the `actions` input of astro_tick: scripted games run without the host. */
int astro_script_controls(AstroBatch* b, double avoid_distance, double avoid_threshold, uint8_t* actions, void* stream);

/* rl.ValueNetwork.forward (rl.py:140-165) over the features of rl.py:43-72 for every game and both
 * ship perspectives, fused: no observation tensor is written.  Weights: the reference network's
 * state_dict flattened in order — f0, f[0], f[1], v[0], v[1], v0, weight [out][in] then bias
 * each; width 32, inputs 15 (10 solo), nout <= 8 outputs — copied to device
 * memory owned by the handle (every batch has its own network).
 *   actions  u8 [n_games][S] device: argmax_q per ship (the greedy control of rl.QBot, rl.py:168-200);
 *            written only for the ships whose bit is set in ship_mask (bit k = ship k), so another
 *            bot can fill the rest; finished games get 2 (no-op)
 *   q_out    f32 [n_games][S][nout] device or NULL: the network outputs (tanh) */
int astro_policy_set_weights(AstroBatch* b, const float* weights_host, int32_t n_floats, int32_t nout);
int astro_policy_controls(AstroBatch* b, uint8_t* actions, float* q_out, int32_t ship_mask, void* stream);

/* rl.EpsilonGreedy.__call__ (rl.py:10-30) for every ship whose bit is set in ship_mask: the random policy that
 * rl.QBotTrainer lays over the greedy network (rl.py:249-258).  Per ship a two-state process — idle -> a random
 * control 0..4 when exp(-dt / t_in) < u, random control -> idle when exp(-dt / t_out) < u, dt = the game time since
 * the previous call — whose draws come from the counter stream (seed, global game, stream step, ship) instead of a
 * numpy RandomState per bot: the same process, not the same sequence.
 *   state    i32 [n_games][S] device, caller-owned, zero-initialised: (tick of the previous call) << 8 | (control + 1)
 *   actions  u8 [n_games][S] device: overwritten with the random control where a ship's random policy is active
 * Call it after astro_policy_controls and before astro_tick (the reference's t_in = 1.0, t_out = 0.1). */
int astro_explore_controls(AstroBatch* b, double t_in, double t_out, uint32_t seed, int32_t* state, uint8_t* actions,
                           int32_t ship_mask, void* stream);
/* The same parameters and state buffer for ASTRO_BOT_EXPLORE ships of astro_rollout_device. */
int astro_set_exploration(AstroBatch* b, double t_in, double t_out, uint32_t seed, int32_t* state);

/* n_ticks of a whole game loop without the host between ticks (core.play, core.py:377-410, and the
 * evaluation games of rl.train, rl.py:350-374, for N games at once): every tick the chosen bot of
 * each ship writes its control, then astro_tick runs.  Asynchronous; episode outcomes accumulate in
 * the astro_stats counters (wins0 / wins1 / both_lost / timeouts).
 *   shipK_mode  ASTRO_BOT_STREAM  counter-stream random controls (both ships or none)
 *               ASTRO_BOT_SCRIPT  script.ScriptBot        (astro_script_controls)
 *               ASTRO_BOT_POLICY  greedy rl.ValueNetwork  (astro_policy_controls)
 *               ASTRO_BOT_NOTHING script.NothingBot: control 2
 *               ASTRO_BOT_EXPLORE the greedy network with rl.EpsilonGreedy laid over it, like rl.QBotTrainer
 *                                 (astro_policy_controls, then astro_explore_controls; needs astro_set_exploration)
 *   actions     u8 [n_games][S] device scratch (may be NULL for ASTRO_BOT_STREAM); holds the last tick's controls, EXCEPT when
 *               every ship is SCRIPT or NOTHING on a float32 batch: those bots are evaluated inside the tick kernel from
 *               the rows it has just loaded (many ticks per launch, no control array) and `actions` is left untouched
 *               (ASTRO_FUSED_BOTS=0 in the environment restores the bot-kernel -> tick-kernel loop)
 *   events      u8 [n_games] device or NULL: the last tick's events */
#define ASTRO_BOT_STREAM 0
#define ASTRO_BOT_SCRIPT 1
#define ASTRO_BOT_POLICY 2
#define ASTRO_BOT_NOTHING 3
#define ASTRO_BOT_EXPLORE 4
int astro_rollout_device(AstroBatch* b, int32_t n_ticks, int32_t ship0_mode, int32_t ship1_mode, double avoid_distance,
                         double avoid_threshold, uint8_t* actions, uint8_t* events, int32_t flags, void* stream);

/* A per-tick recording ring for astro_rollout_device_record: what every game's ships flew, what came of it and (optionally)
 * what ship 0 saw, for each tick of a rollout — the log that rl.QBotTrainer keeps per bot (Experience, rl.py:212-228) and
 * that astro_nstep_experiences turns into n-step replay pairs.  Device pointers, caller-owned; row r of every array holds
 * the tick run at stream step s with s % ticks == r. */
typedef struct AstroRecordRing {
    int32_t ticks;        /* R rows; the tick run at stream step s is recorded in row s % R */
    int32_t n_rows;       /* observation rows per game (as astro_observe_shared); ignored when observations is NULL */
    uint8_t* controls;    /* u8 [R][n_games][S]: the control each ship flew on that tick (required) */
    uint8_t* events;      /* u8 [R][n_games]: that tick's ASTRO_EV_* byte, exactly what astro_tick writes (required) */
    float* observations;  /* f32 [R][n_games][n_rows][1+5S+4] or NULL: ship 0's view of the state BEFORE the tick */
} AstroRecordRing;
/* astro_rollout_device (same arguments but `events`, same results: recording changes no state and no counter) that also
 * records every tick into `ring` (NULL: astro_rollout_device without events).  A call of n_ticks from stream
 * step s0 fills rows s0 .. s0 + n_ticks - 1 (mod R) and, with observations, writes the observation of the state after its
 * last tick into row (s0 + n_ticks) % R, so that the new state of every pair a window yields is in the ring: n_ticks <= R - 1.
 * Float32 batches only (not precision 64, not ASTRO_TICK_GENERIC_KERNEL); observations 16-byte aligned, n_rows >= the
 * planet slots + bullet_cap.  Controls and events are stored by the tick kernel itself, so the counter stream keeps its
 * many-tick launches and ScriptBot / NothingBot games keep the bots inside the tick; with observations every tick is
 * observe -> bots -> tick. */
int astro_rollout_device_record(AstroBatch* b, int32_t n_ticks, int32_t ship0_mode, int32_t ship1_mode, double avoid_distance,
                                double avoid_threshold, uint8_t* actions, const AstroRecordRing* ring, int32_t flags,
                                void* stream);

/* Game-major float64 view of games, the layout host-side code wants (State conversion for the drop-in core.step /
 * core.play, core.py:11-18 and :377-410; JSONL logs, core.py:413-443): row i describes one game.  DEVICE pointers.
 *   ships R [m][S][5] = x, y, dx, dy, b    planets [m][PL][4] (dead slots zero)    bullets [m][k][4] (dead slots zero)
 *   n_planets / n_bullets / tick i32 [m]   finished u8 [m]   episode u32 [m] (may be NULL) */
typedef struct AstroGameArrays {
    double* ships;
    double* planets;
    double* bullets;
    int32_t* n_planets;
    int32_t* n_bullets;
    int32_t* tick;
    uint8_t* finished;
    uint32_t* episode;
    int32_t bullet_rows; /* k: rows per game of `bullets` (export: >= the largest live count wanted; import: <= bullet_cap) */
    int32_t reserved;
} AstroGameArrays;

/* Games index[0..m-1] (device i32; NULL: games 0..m-1) -> rows 0..m-1 of `out`, one kernel: the tile lists are unpacked
 * on the device.  Float32 state converts exactly.  A finished game exports finished = 1, n_bullets = 0. */
int astro_export_games(AstroBatch* b, const int32_t* index, int32_t m, const AstroGameArrays* out, void* stream);
/* The inverse: rows 0..m-1 of `in` replace games index[0..m-1] (NULL: games 0..m-1; an index must not repeat), every
 * other game — including the bullets of the other games of a touched tile — is kept.  Float32 batches round the values
 * to float32.  n_bullets is clipped to bullet_cap.  `tick` = the game's index on the batch's schedule (astro_set_schedule). */
int astro_import_games(AstroBatch* b, const int32_t* index, int32_t m, const AstroGameArrays* in, void* stream);

/* core.step (core.py:215-303) for ONE game with HOST buffers — the body of the drop-in astro_b200.core.step: one pinned
 * record in, import -> tick -> export on the stream, one record out, then a stream synchronise.  The batch must hold
 * exactly one tile (n_games = 32); game 0 is used.  The record is followed in memory by double bullets[bullet_cap][4]
 * (astro_single_game_bytes); only the live rows travel.
 *   in:  ships / planets / bullets / n_planets / n_bullets, control[s], tick = where the game stands on the batch's
 *        schedule (the host evaluates the reload / timeout predicates of core.py:257-267 in Python floats and picks
 *        the index of a schedule entry with that outcome)
 *   out: the new state (tick + 1), events[0] = ASTRO_EV_* of the tick, finished = 1 when the game ended */
typedef struct AstroSingleGame {
    double ships[ASTRO_MAX_SHIPS][5];
    double planets[ASTRO_MAX_PLANETS_WIDE][4]; /* rows >= the batch's planet slots are ignored */
    int32_t n_planets, n_bullets, tick, reserved;
    uint32_t episode;
    uint8_t finished[4];
    uint8_t control[ASTRO_TILE * ASTRO_MAX_SHIPS]; /* [0..S-1] are read; the rest belongs to the tile's empty slots */
    uint8_t events[ASTRO_TILE];                    /* [0] is the game's */
} AstroSingleGame;
int64_t astro_single_game_bytes(int32_t bullet_cap);
int astro_step_single_host(AstroBatch* b, const AstroSingleGame* in_host, AstroSingleGame* out_host, int32_t flags, void* stream);

/* The n-step replay ingestion of rl.QBotTrainer.reward (rl.py:303-328) for every bot (game, ship) over a window of n_ticks
 * logged ticks: which (state, action) pairs are flushed into the replay buffer when, with which discounted reward, discount
 * and new state — from the ticks' event bytes alone (an Experience is identified by its tick; the actions and observations
 * of the ticks are in the AstroRecordRing that astro_rollout_device_record filled, or wherever the caller logged them).
 * Device pointers:
 *   events     u8 [n_ticks][n_games]            the ticks' ASTRO_EV_* bytes (astro_tick_many / astro_rollout_*, a ring's rows)
 *   carry      i32 [n_games][S]  in/out         pairs a bot still holds (before the window / after it); zero-initialised
 *   out_reward / out_discount f32, out_next i32 [n_steps + n_ticks][n_games][S]: row n_steps + t = the pair of tick t, rows
 *              below n_steps = the ticks before the window (carried pairs that flush now).  reward = r * d and discount =
 *              discount * d with d = discount ** (pairs held after this one), r the flushing tick's reward (core.py:255,260);
 *              next = window-relative tick whose observation is the new state (flush tick + 1), -1 terminal (new state None),
 *              -2 still held at the end of the window, -3 no pair (the game was finished and skipped the tick). */
int astro_nstep_experiences(AstroBatch* b, const uint8_t* events, int32_t n_ticks, int32_t n_steps, double discount, int32_t* carry,
                            float* out_reward, float* out_discount, int32_t* out_next, void* stream);

/* Copies the ASTRO_N_STATS device counters into counters_dev (device pointer, e.g. the input of
 * an NCCL all-reduce) on the stream; clear != 0 zeroes them afterwards. */
int astro_stats(AstroBatch* b, int64_t* counters_dev, int32_t clear, void* stream);

/* rl.ValueNetwork.forward (rl.py:140-165) on a feature batch — the tensor astro.rl's own callers hold (get_features_batch,
 * rl.py:101-112, or astro_observe's output) — for inference, with the batch's network (astro_policy_set_weights): the three
 * per-object layers, masked_max over the rows (rl.py:115-128: max of x - 1e9 * (features[row][0] < 0)), the head, tanh.
 *   features f32 [n_items][rows][din] device, din = 15 (duel) / 10 (solo), contiguous
 *   q_out    f32 [n_items][nout] device
 * Tensor-core kernel (FP16 three-product split, fp32 accumulation): within 2e-6 of the PyTorch fp32 network. */
int astro_value_forward(AstroBatch* b, const float* features, int32_t n_items, int32_t rows, float* q_out, void* stream);

/* The same counters summed over the N processes of one node (one GPU each; "NCCL used only for the optional episode-stats
 * reduction" in the north star — this is that reduction without NCCL): ONE kernel per rank that stores the rank's counters
 * into every rank's exchange buffer through peer memory (NVLink / NVSwitch, buffers mapped by CUDA IPC), waits for the other
 * ranks' rows and writes the total to counters_dev — the latency of one P2P store instead of a collective launch.
 *   astro_stats_peer_create  allocates this rank's exchange buffer; handle_out receives its ASTRO_IPC_HANDLE_BYTES-byte IPC
 *                            handle, which the caller hands to every rank (e.g. torch.distributed.all_gather)
 *   astro_stats_peer_open    handles = world x ASTRO_IPC_HANDLE_BYTES bytes in rank order: maps the peers' buffers
 *   astro_stats_allreduce    collective: every rank calls it the same number of times.  counters_dev as in astro_stats; a
 *                            peer that does not arrive within ~2 s of polling leaves every counter at -1. */
#define ASTRO_IPC_HANDLE_BYTES 64
int astro_stats_peer_create(AstroBatch* b, int32_t rank, int32_t world, uint8_t* handle_out);
int astro_stats_peer_open(AstroBatch* b, const uint8_t* handles);
int astro_stats_allreduce(AstroBatch* b, int64_t* counters_dev, int32_t clear, void* stream);

/* Environment knobs of the library (A/B switches; none changes results, every form is covered by the parity tests):
 *   ASTRO_TICK_NO_FIX=1        the generic tick instantiations instead of the ones with the rollout options fixed at compile time
 *   ASTRO_FUSED_BOTS=0         astro_rollout_device: bot kernel -> tick kernel per tick instead of the ScriptBot inside the tick
 *   ASTRO_LOOP_GRAPH=0         astro_rollout_device: plain launches instead of CUDA graphs of 16 ticks
 *   ASTRO_ROLLOUT_CHUNK=n      astro_rollout_host: ticks per copy / launch (default 8 with packed controls, else 4)
 *   ASTRO_HOST_SLICES=n        astro_tick_host: slices of tiles on internal streams (copies of one overlap the kernel of another)
 *   ASTRO_L2_FETCH_GRANULARITY, ASTRO_EXTRA_SMEM   experiment knobs (tools/experiments) */

/* Launch bookkeeping for bench.py: kernels launched by this handle since creation. */
int64_t astro_launch_count(const AstroBatch* b);

#ifdef __cplusplus
}
#endif
#endif
