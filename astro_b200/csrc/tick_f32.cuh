// tick_f32.cuh — the production tick kernel (included by astro_b200.cu inside its anonymous
// namespace, after TickParams / recreate_from_pool / warp_stats).
//
// One warp owns one 32-game tile.  Two phases:
//
//  A. BULLETS, warp-cooperative.  Each lane stages its game's ships and planets in shared
//     memory, the per-game bullet counts are prefix-summed across the warp, and the tile's
//     bullets are processed as ONE flat list, 32 per iteration, whatever game they belong to —
//     a warp with bullet counts (0, 17, 3, ...) runs ceil(sum/32) iterations, not max = 17.
//     Per bullet: squared distances to both ships and four planet slots (dead slots hold a
//     far-away sentinel) reduced with min, the advance, and ONE band test deciding whether the
//     fp32 comparisons provably equal the reference's float64 results; only a bullet inside a
//     band (|d2 - R2| <= 1e-6 R2, or |x'| within 4e-6 of the arena bound — ~1e-5 of bullets),
//     and every ship hit, takes the float64 path.  Survivors are compacted with a warp ballot:
//     rank inside the game's segment = popc(ballot & segment mask), so the reference order
//     (stable) is kept.  In HBM the flat list IS the storage order (one dense run per tile, see
//     the header): a window of 32 list items is one contiguous 512-byte read, and the new list —
//     survivors and newborn, dense again — is written to the tile's run in the other buffer.  (The
//     production rollout's fused form keeps the list in shared memory from tick to tick instead and
//     writes it once per launch: the resident pool, section 6 of tick_tile.)
//  B. SHIPS AND PLANETS, thread-per-game from the staged copies: direction, gravity, collisions,
//     terminal logic, spawn, integration, reset — all coalesced 128-bit accesses.
//
// Instantiations, tick_f32_kernel<S, STATS, MANY, BOT, FIX> (4 planet slots) and tick_f32_wide_kernel<S, STATS, MANY> (8):
//   MANY  several ticks of a tile per launch (astro_tick_many): meta / ships / bearings handed from tick to tick in registers,
//         7 staging windows and 28 one-warp CTAs per SM (the one-tick launch: 8 and 26) — this form is bound by instruction issue
//   BOT   script.ScriptBot / NothingBot evaluated inside the tick (astro_rollout_device)
//   FIX   the production rollout's options fixed at compile time: packed controls given, event planes written, no reward / done
//         arrays, auto-reset from the pool, no recording ring.  launch_tick_f32 (astro_b200.cu) picks it when the launch's
//         options match.  Every other form stores each tick's controls and event byte into the recording ring of
//         astro_rollout_device_record when one is given (TickParams::rec_*).
// What the issue-bound form paid for, and no longer does (profiles/r2_ab_diet.md): option tests and the address arithmetic of
// absent arrays (FIX); a test and a round loop around the common bullet loop (duplicated per value of `multi`); values ptxas
// re-derived instead of keeping — the shared-memory base behind every rare float64 block, the tile index, the lane id — which now
// go through a shuffle once (a shuffle's result cannot be re-materialised).
#pragma once

// Dead planet slots sit at kFar: the squared distance overflows to +inf, so a dead slot is never
// a minimum, never inside a band, and its gravity G*M/inf is exactly 0 — no predication on np.
constexpr float kFar = 1.0e20f;
constexpr int kTickWarps = kTickThreads / 32;
#ifndef ASTRO_PREFETCH_PLANETS
#define ASTRO_PREFETCH_PLANETS 4
#endif

// Bullets staged per round: W windows x 32 (512 bytes each).  The launch of several ticks is bound by issue slots and takes every
// warp it can get: 7 windows (224 bullets, 7,216 bytes per warp) let 28 one-warp CTAs share an SM's shared memory — also what the
// registers allow (72 x 32 x 28) — against 26 with 8; the one-tick launch is bound by HBM and is slower with more address streams
// open at once (A/B at 1,048,576 games, 7 windows + 28 CTAs against 8 + 26: several ticks per launch 59.7 -> 59.2 us per tick,
// 131,072 games — 4,096 tiles, ONE wave of 4,144 resident CTAs instead of 3,848 + 248 — 12.6 -> 11.4; one launch per tick
// 67.8 -> 70.2), so each form keeps its own.  (A tile with more bullets than a round holds takes a second round: correct, rare.)
#ifndef ASTRO_STAGE_WINDOWS
#define ASTRO_STAGE_WINDOWS 8
#endif
#ifndef ASTRO_STAGE_WINDOWS_MANY
#define ASTRO_STAGE_WINDOWS_MANY 7
#endif
#ifndef ASTRO_TICK_MIN_BLOCKS_MANY
#define ASTRO_TICK_MIN_BLOCKS_MANY 28
#endif
#ifndef ASTRO_TICK_MIN_BLOCKS_BOT
#define ASTRO_TICK_MIN_BLOCKS_BOT 12    /* the instantiation with the ScriptBot inside: float64 chains, 160 registers */
#endif
// 8 planet slots (PL = 8): eight float4 planets, their pairs and forces live in registers, and the staged frame holds two
// more planet pairs per game (1 KB more shared memory per warp)
#ifndef ASTRO_TICK_MIN_BLOCKS_WIDE
#define ASTRO_TICK_MIN_BLOCKS_WIDE 16
#endif
#ifndef ASTRO_TICK_MIN_BLOCKS_WIDE_MANY
#define ASTRO_TICK_MIN_BLOCKS_WIDE_MANY 16
#endif
// Round 2, instruction diet of the fused form (issue-bound; ncu dynamic instruction counts in profiles/r2_ab_diet.md):
#ifndef ASTRO_OPT_STAGE
#define ASTRO_OPT_STAGE 1     /* several ticks per launch: staging requests unrolled and predicated, 2-3 instructions per window instead of ~14 */
#endif
#ifndef ASTRO_OPT_PTRS
#define ASTRO_OPT_PTRS 1      /* per-tick pointers = base + tick * stride (stride 0 for an absent array): no null tests, no 64-bit products */
#endif

// Per-game entries used by the bullet loop are indexed by the game's rank among the tile's games
// that own bullets (`cid`): item -> cid comes out of one ballot per window, no lookup table.
template <int W, int PL>
struct TileScratchT {              // per warp
    float4 bul[W * 32];            // the tile's bullet list, staged by cp.async; survivors are compacted here
    float4 fsxy[32];               // [cid] OLD ship0.xy, ship1.xy                } what the bullet loop reads
    float4 fpxy[PL / 2][32];       // [cid] OLD planet0.xy planet1.xy / 2,3 / ... } (transposed pairs)
    float4 sxy[32];                // [lane] OLD ship positions  }
    float4 svel[32];               // [lane] OLD ship velocities } for the newborn bullets
    float4 dir[32];                // [lane] sin/cos of both bearings
    uint32_t hits[32];             // [cid] bits 0-1: ship hits found by the bullet loop; bits 8+: np
    union {
        int32_t shift[32];         // [cid] new list: item j of the compacted list moves to j + shift (kDrop: game over)
        uint32_t gcount[32];       // resident pool: [lane] items the bullet loop removed, then the game's next list slot
    };
    uint16_t gstart[34];           // [cid] first survivor of the game in the compacted list; [n] = survivors of the tile
    uint8_t ref[W * 32];               // compacted item -> cid (resident pool: item -> tag, lane | generation << 5)
    uint32_t used;                     // fresh-game mode: records of the tile's ring consumed since the last refill
};
constexpr int kDrop = 0x40000000;

// Shared-memory accesses of the bullet loop through explicit 32-bit addresses off ONE base register (ASTRO_SMEM_ASM): ptxas
// otherwise re-derives the base (S2R SR_CgaCtaId + MOV + LEA, predicated, twice per window) behind the loop's rare float64
// block, which clobbers it.  The base goes through a shuffle, which cannot be re-materialised.
#ifndef ASTRO_SMEM_ASM
#define ASTRO_SMEM_ASM 1
#endif
#ifndef ASTRO_OPAQUE_LANE
#define ASTRO_OPAQUE_LANE 1
#endif
#ifndef ASTRO_OPAQUE_TILE
#define ASTRO_OPAQUE_TILE 1
#endif
__device__ __forceinline__ float4 lds128(unsigned a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void sts128(unsigned a, float4 v) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ unsigned lds32(unsigned a) { unsigned v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ unsigned lds16(unsigned a) { unsigned v; asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ unsigned lds8(unsigned a) { unsigned v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ void sts32(unsigned a, unsigned v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts8(unsigned a, unsigned v) { asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts16(unsigned a, unsigned v) { asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void reds_add(unsigned a, unsigned v) { asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void reds_or(unsigned a, unsigned v) { asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
// Resident bullet pool (tick_tile, MANY && FIX): the pool size, or kNotResident when the next tick stages its list from HBM.
constexpr unsigned kNotResident = 0xffffffffu;
// Tag of a pool item: owning lane in bits 0-4, the game's generation in bit 5 (0xff: past the end, never live).  An item is
// live iff its generation bit equals bit `lane` of the warp's generation mask.
__device__ __forceinline__ bool tag_live(unsigned tag, unsigned genmask) {
    return (tag >> 5) == (__funnelshift_r(genmask, genmask, tag) & 1u);   // (funnel shift: the amount is taken mod 32)
}

__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// Exact (reference float64) evaluation of one bullet against the OLD ship / planet positions:
// despawn flags, per-ship hit bits, advance + cull.  Taken by ~1e-5 of bullets.
struct ExactResult {
    float x, y;
    unsigned flags;  // bit 0 keep, bits 1-2 ship hits
};
// p[k] = planets 2k and 2k + 1: (x, y) of each.
template <int PL>
__device__ __forceinline__ ExactResult bullet_exact(float bx, float by, float bdx, float bdy, float4 sxy, const float4 (&p)[PL / 2],
                                                    int n_ships, int np, const Consts& c) {
    unsigned ship_hits = 0;
    if (collide_exact((double)sxy.x, (double)sxy.y, (double)bx, (double)by, c.r2_sb)) ship_hits |= 1u;
    if (n_ships > 1 && collide_exact((double)sxy.z, (double)sxy.w, (double)bx, (double)by, c.r2_sb)) ship_hits |= 2u;
    bool gone = ship_hits != 0;
    gone |= collide_exact((double)p[0].x, (double)p[0].y, (double)bx, (double)by, c.r2_pb);  // np >= 1
    if (np > 1) gone |= collide_exact((double)p[0].z, (double)p[0].w, (double)bx, (double)by, c.r2_pb);
    if (np > 2) gone |= collide_exact((double)p[1].x, (double)p[1].y, (double)bx, (double)by, c.r2_pb);
    if (np > 3) gone |= collide_exact((double)p[1].z, (double)p[1].w, (double)bx, (double)by, c.r2_pb);
#pragma unroll
    for (int k = 2; k < PL / 2; k++) {
        if (np > 2 * k) gone |= collide_exact((double)p[k].x, (double)p[k].y, (double)bx, (double)by, c.r2_pb);
        if (np > 2 * k + 1) gone |= collide_exact((double)p[k].z, (double)p[k].w, (double)bx, (double)by, c.r2_pb);
    }
    double v0 = __dadd_rn((double)bdx, c.zero_dt), v1 = __dadd_rn((double)bdy, c.zero_dt);
    double e0 = __dadd_rn((double)bx, __dmul_rn(c.dt, v0)), e1 = __dadd_rn((double)by, __dmul_rn(c.dt, v1));
    ExactResult r;
    r.x = (float)e0;
    r.y = (float)e1;
    r.flags = ((in_arena(e0, e1) && !gone) ? 1u : 0u) | (ship_hits << 1);
    return r;
}

// ---- packed fp32 pairs ------------------------------------------------------------------------
// sm_100a issues FADD2 / FMUL2 / FFMA2: one issue slot, two IEEE fp32 operations, each half rounded
// exactly like the scalar instruction.  The tick is bound by instruction issue as much as by HBM,
// so the x/y halves of a body (the natural register pairs of its float4) and pairs of staged
// objects go through them.
#ifndef ASTRO_PACKED_F32
#define ASTRO_PACKED_F32 1
#endif
#if ASTRO_PACKED_F32
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pk2(float lo, float hi) {
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void upk2(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b) {
    f32x2 d;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
    f32x2 d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
    f32x2 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
#else
// Scalar twin (same roundings), -DASTRO_PACKED_F32=0.  FADD2/FMUL2/FFMA2 hold the FMA pipe for two
// cycles (tools/ubench/f32x2.cu), which made them neutral while the tick waited on scattered HBM
// runs; with the tile lists the tick is a chain of dependent instructions per warp and the ~150
// saved issue slots per tile are worth 10 % (88.3 -> 79.0 us per 1M-game tick).
struct f32x2 {
    float lo, hi;
};
__device__ __forceinline__ f32x2 pk2(float lo, float hi) { return f32x2{lo, hi}; }
__device__ __forceinline__ void upk2(f32x2 v, float& lo, float& hi) { lo = v.lo; hi = v.hi; }
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b) { return f32x2{__fsub_rn(a.lo, b.lo), __fsub_rn(a.hi, b.hi)}; }
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) { return f32x2{__fmul_rn(a.lo, b.lo), __fmul_rn(a.hi, b.hi)}; }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
    return f32x2{__fmaf_rn(a.lo, b.lo, c.lo), __fmaf_rn(a.hi, b.hi, c.hi)};
}
#endif
__device__ __forceinline__ f32x2 bc2(float v) { return pk2(v, v); }
__device__ __forceinline__ float min2(f32x2 v) {
    float a, b;
    upk2(v, a, b);
    return fminf(a, b);
}

// Squared distances of one point (bx, by) to two staged objects held TRANSPOSED, o = (x0, x1, y0, y1):
// d^2 = fma(dy, dy, dx * dx) per object (one subtraction per axis, one product, one FMA).
__device__ __forceinline__ f32x2 dist2_pair(float4 o, f32x2 bx, f32x2 by) {
    f32x2 dx = sub2(pk2(o.x, o.y), bx), dy = sub2(pk2(o.z, o.w), by);
    return fma2(dy, dy, mul2(dx, dx));
}

// bullet_exact() for the transposed staging.
template <int PL>
__device__ __forceinline__ ExactResult bullet_exact_t(float4 bv, float4 sT, const float4 (&pT)[PL / 2], int n_ships, int np,
                                                      const Consts& c) {
    float4 p[PL / 2];
#pragma unroll
    for (int k = 0; k < PL / 2; k++) p[k] = make_float4(pT[k].x, pT[k].z, pT[k].y, pT[k].w);
    return bullet_exact<PL>(bv.x, bv.y, bv.z, bv.w, make_float4(sT.x, sT.z, sT.y, sT.w), p, n_ships, np, c);
}

// One bullet bv = (x, y, dx, dy) against its game's staged frame (transposed pairs: both ships,
// planets 0/1, planets 2/3, ...).  Returns keep; bv.x / bv.y advanced; ship_hits receives bits 0/1 when
// the bullet touches ship 0/1 (always decided in float64).  Arena test: keep iff (|x'| <= 1) or
// (|y'| <= 1)  <=>  min(|x'|, |y'|) <= 1, so only the smaller magnitude can sit in the band.
template <int S, int PL>
__device__ __forceinline__ bool bullet_step_t(float4& bv, float4 sT, const float4 (&pT)[PL / 2], const uint32_t* np_of,
                                              unsigned gi, const Consts& c, unsigned& ship_hits) {
    const f32x2 bx = bc2(bv.x), by = bc2(bv.y);
    const float ds = min2(dist2_pair(sT, bx, by));  // S == 1: both halves hold ship 0
    float dp = fminf(min2(dist2_pair(pT[0], bx, by)), min2(dist2_pair(pT[1], bx, by)));
#pragma unroll
    for (int k = 2; k < PL / 2; k++) dp = fminf(dp, min2(dist2_pair(pT[k], bx, by)));
    float x0, x1;
    upk2(fma2(bc2(c.dt_f), pk2(bv.z, bv.w), pk2(bv.x, bv.y)), x0, x1);
    const float mn = fminf(fabsf(x0), fabsf(x1));
    const bool sure = (ds >= c.r2f_sb * 1.000001f) & (fabsf(dp - c.r2f_pb) > c.r2f_pb * 1e-6f) & (fabsf(mn - 1.0f) > 4e-6f);
    bool keep = (mn <= 1.0f) & (dp >= c.r2f_pb);
    if (__builtin_expect(!sure, 0)) {
        ExactResult r = bullet_exact_t<PL>(bv, sT, pT, S, (int)(np_of[gi] >> 8), c);
        x0 = r.x;
        x1 = r.y;
        keep = r.flags & 1u;
        ship_hits = r.flags >> 1;
    }
    bv.x = x0;
    bv.y = x1;
    return keep;
}

// np_sincos_f32 for two bearings at once (same operations, same bits).
__device__ __forceinline__ void np_sincos_f32x2(float xa, float xb, float& sna, float& csa, float& snb, float& csb) {
    const f32x2 x = pk2(xa, xb), magic = bc2(12582912.0f);
    const f32x2 q = sub2(fma2(x, bc2(0x1.45f306p-1f), magic), magic);
    f32x2 r = fma2(q, bc2(-0x1.921fb0p+00f), x);
    r = fma2(q, bc2(-0x1.5110b4p-22f), r);
    r = fma2(q, bc2(-0x1.846988p-48f), r);
    const f32x2 r2 = mul2(r, r);
    f32x2 cc = fma2(bc2(0x1.98e616p-16f), r2, bc2(-0x1.6c06dcp-10f));
    cc = fma2(cc, r2, bc2(0x1.55553cp-5f));
    cc = fma2(cc, r2, bc2(-0x1.000000p-1f));
    cc = fma2(cc, r2, bc2(0x1.000000p+0f));
    f32x2 ss = fma2(bc2(0x1.7d3bbcp-19f), r2, bc2(-0x1.a06bbap-13f));
    ss = fma2(ss, r2, bc2(0x1.11119ap-7f));
    ss = fma2(ss, r2, bc2(-0x1.555556p-3f));
    ss = fma2(ss, r2, bc2(0.0f));
    ss = fma2(ss, r, r);
    float qa, qb, ca, cb, sa, sb_;
    upk2(q, qa, qb);
    upk2(cc, ca, cb);
    upk2(ss, sa, sb_);
    {
        const int iq = (int)qa, ic = iq + 1;
        const float vs = (iq & 1) ? ca : sa, vc = (ic & 1) ? ca : sa;
        sna = (iq & 2) ? -vs : vs;
        csa = (ic & 2) ? -vc : vc;
    }
    {
        const int iq = (int)qb, ic = iq + 1;
        const float vs = (iq & 1) ? cb : sb_, vc = (ic & 1) ? cb : sb_;
        snb = (iq & 2) ? -vs : vs;
        csb = (ic & 2) ? -vc : vc;
    }
}

// Symplectic Euler step of one body held as pairs xy = (x, y), v = (dx, dy) (core.py:189-197);
// the wrap is evaluated only by a body that actually left the square (rare).
__device__ __forceinline__ float4 advance_body2(f32x2 xy, f32x2 v, f32x2 acc, const Consts& c) {
    const f32x2 dt2 = bc2(c.dt_f);
    const f32x2 vn = fma2(acc, dt2, v);
    const f32x2 xn = fma2(dt2, vn, xy);
    float x0, x1, v0, v1;
    upk2(xn, x0, x1);
    upk2(vn, v0, v1);
    if (__builtin_expect(fmaxf(fabsf(x0), fabsf(x1)) >= 1.0f, 0)) {
        if (fabsf(x0) >= 1.0f) x0 = wrap_unit_f32(x0);
        if (fabsf(x1) >= 1.0f) x1 = wrap_unit_f32(x1);
    }
    return make_float4(x0, x1, v0, v1);
}

// Gravity of a body at o on a body at xy (core.py:138-153): rx = o - xy, f = G*M / max(1e-12, |rx|^2),
// acc += f * rx; returns |rx|^2 (for the collision test of the same pair).  A dead planet slot sits
// at kFar: |rx|^2 = +inf, f = 0, no predication.
__device__ __forceinline__ float grav_pair(f32x2 o, f32x2 xy, f32x2& acc, const Consts& c) {
    const f32x2 q = sub2(o, xy);
    float s0, s1;
    upk2(mul2(q, q), s0, s1);
    const float d2 = __fadd_rn(s0, s1);
    const float f = div_fast_normal(c.gm_f, fmaxf(1e-12f, d2));
    acc = fma2(bc2(f), q, acc);
    return d2;
}

// -DASTRO_TIMELINE: every warp records clock64() at its phase boundaries (tools/exp_timeline.py)
#ifdef ASTRO_TIMELINE
__device__ long long* g_timeline = nullptr;
#define TL(k) do { if (g_timeline && lane == 0) g_timeline[(size_t)(g >> 5) * 8 + (k)] = clock64(); } while (0)
#else
#define TL(k) do { } while (0)
#endif
#ifndef ASTRO_BOUSTROPHEDON
#define ASTRO_BOUSTROPHEDON 1   /* A/B: 1M games 77.2 -> 76.0 us, 512k 43.5 -> 41.0, 2M 141.6 -> 143.8 */
#endif
#ifndef ASTRO_TICK_MIN_BLOCKS
#define ASTRO_TICK_MIN_BLOCKS 26  /* shared memory admits 26 one-warp CTAs per SM: 72 registers */
#endif
// Cache hints for the once-per-tick streams (A/B: ASTRO_STREAM_HINTS = 1 -> ld.global.cs / st.global.cs)
#ifndef ASTRO_STREAM_HINTS
#define ASTRO_STREAM_HINTS 0
#endif
#if ASTRO_STREAM_HINTS
#define LD_STREAM(ptr) __ldcs(ptr)
#define ST_STREAM(ptr, v) __stcs(ptr, v)
#else
#define LD_STREAM(ptr) (*(ptr))
#define ST_STREAM(ptr, v) (*(ptr) = (v))
#endif

// What a tile's first round trip to HBM brings: the fixed-size rows that do not depend on meta.
// What changes from one tick to the next inside a launch that runs several ticks (astro_tick_many):
// the stream step, the per-tick inputs / outputs, and which bullet buffer is read.
struct TickVar {
    uint32_t step;
    const uint8_t* actions;
    float* reward;
    uint8_t* done;
    uint8_t* events;
    float4* bullets_in;
    float4* bullets_out;
};
template <int S>
__device__ __forceinline__ TickVar tick_var(const TickParams& p, unsigned k) {
    TickVar v;
    v.step = p.step + k;
#if ASTRO_OPT_PTRS
    // base + tick * stride in 32 x 32 -> 64-bit products; the stride of an absent (null) array is 0
    v.actions = p.actions + (size_t)k * p.act_stride;     // [n][S] bytes, or [n] packed
    v.reward = reinterpret_cast<float*>(reinterpret_cast<char*>(p.reward) + (size_t)k * p.rw_stride);
    v.done = p.done + (size_t)k * p.done_stride;
    v.events = p.events + (size_t)k * p.ev_stride;        // [n] bytes, or three bit planes
#else
    const size_t n = (size_t)p.n_games;
    v.actions = p.actions ? p.actions + k * (size_t)p.act_stride : nullptr;
    v.reward = p.reward ? p.reward + k * n * S : nullptr;
    v.done = p.done ? p.done + k * n : nullptr;
    v.events = p.events ? p.events + k * (size_t)p.ev_stride : nullptr;
#endif
    v.bullets_in = reinterpret_cast<float4*>((k & 1u) ? p.bullets_out : p.bullets_in);
    v.bullets_out = reinterpret_cast<float4*>((k & 1u) ? p.bullets_in : p.bullets_out);
    return v;
}
// The control bytes of game g: two bytes (one per ship), or — ASTRO_TICK_PACKED_CONTROLS — one byte holding both
// codes (ship 0 in bits 0-2, ship 1 in bits 3-5), expanded to the two-byte form (bits 6-7 land in ship 1's byte and
// flag the control as bad, like any code above 5).
template <int S>
__device__ __forceinline__ uint32_t load_controls(const uint8_t* a, size_t g, bool packed) {
    if (S == 2 && !packed) return (uint32_t)reinterpret_cast<const uint16_t*>(a)[g];
    const uint32_t b = (uint32_t)a[g];
    if (S == 2) return (b & 7u) | ((b & 0xf8u) << 5);
    return b;
}
struct TileIn {
    uint32_t meta;
    float4 shv[2];
    float sb[2];
    uint32_t ctl_raw;   // the tile's control bytes of this lane's game (S bytes), when actions are given
    uint32_t fire_word; // (several ticks per launch) the fire-schedule word of this game's tick, requested at the top
};
template <int S, int PL, bool FIX = false, bool WARM_PLANETS = true>
__device__ __forceinline__ void load_tile_in(const TickParams& p, const TickVar& v, unsigned tile, unsigned lane, TileIn& in) {
    const size_t g = (size_t)tile * 32 + lane;
    in.meta = LD_STREAM(&p.meta[g]);
    const float4* ships = reinterpret_cast<const float4*>(p.ships) + (size_t)tile * (S * 32) + lane;
    const float* ship_b = reinterpret_cast<const float*>(p.ship_b) + (size_t)tile * (S * 32) + lane;
    // The planet slots to load depend on meta (np).  Warm L2 with the tile's planet rows meanwhile:
    // the dependent loads then take an L2 round trip instead of an HBM one (measured:
    // 93.4 -> 91.4 us per 1M-game tick; sectors without a live lane are the price).
    const float4* planets = reinterpret_cast<const float4*>(p.planets) + (size_t)tile * (PL * 32) + lane;
    if (WARM_PLANETS) {
#pragma unroll
        for (int j = 0; j < ASTRO_PREFETCH_PLANETS; j++) asm volatile("prefetch.global.L2 [%0];" ::"l"(&planets[j * 32]));
    }
#pragma unroll
    for (int s = 0; s < S; s++) {
        in.shv[s] = LD_STREAM(&ships[s * 32]);
        in.sb[s] = LD_STREAM(&ship_b[s * 32]);
    }
    if (S == 1) { in.shv[1] = in.shv[0]; in.sb[1] = in.sb[0]; }  // S == 1: the second half of every ship pair mirrors ship 0
    in.ctl_raw = 0;
    if (FIX || v.actions) in.ctl_raw = load_controls<S>(v.actions, g, FIX || (p.flags & ASTRO_TICK_PACKED_CONTROLS) != 0);
    // Everything above is ONE round trip to HBM only if it is requested before the first use of meta.
    // ptxas is free to hoist meta-dependent code (it drags a later load and its address arithmetic up)
    // above these requests, which then leave a whole round trip late — seen at random from build to
    // build, 10 % of the tick (profiles/r1_ab_v6_experiments.md, session 4).  A warp barrier pins them.
    __syncwarp();
}

// One core.step for the 32 games of one tile, by one warp.
// `next` receives what the following tick of the same tile would load from the rows this tick wrote (meta, ships,
// bearings): inside a launch that runs several ticks they are handed on in registers.
// FIX = the launch's options are the production rollout's, known at compile time (launch_tick_f32 checks them): duel games,
// packed controls given, event planes written, no reward / done arrays, auto-reset from the pool (no ring, no captured
// step base) — the tests of those options and the address arithmetic of the absent arrays fold away.
template <int S, bool STATS, bool MANY, bool BOT, bool FIX, int PL>
// `last` = no further tick of this tile follows in this launch: only then do meta, ships and bearings go to memory
// (planets and the bullet list always do), and the tile's statistics (`stat_acc`, summed over the launch's ticks).
__device__ __forceinline__ void tick_tile(const TickParams& p, const TickVar& v, TileScratchT<MANY ? ASTRO_STAGE_WINDOWS_MANY : ASTRO_STAGE_WINDOWS, PL>& t, const unsigned lane,
                                          const unsigned tile_index, const TileIn& in, TileIn& next, const bool last,
                                          unsigned& stat_acc, const bool have_fire_word, unsigned& pool, unsigned& genmask,
                                          const unsigned rec_row) {
    using B4 = Body4<float>;
    constexpr int kStageWindows = MANY ? ASTRO_STAGE_WINDOWS_MANY : ASTRO_STAGE_WINDOWS;
    // `pool` / `genmask` (warp-uniform, kept by the caller from tick to tick): the resident bullet pool of section 6
    constexpr bool RES = ASTRO_SMEM_ASM && MANY && FIX && !BOT;
    const bool resident = RES && pool != kNotResident;
    const unsigned full = 0xffffffffu;
    const int g = (int)(tile_index * 32u + lane);
    const Consts& c = p.c;
    const size_t tile = (size_t)tile_index;
    float4* ships = reinterpret_cast<float4*>(p.ships) + tile * (S * 32) + lane;
    float* ship_b = reinterpret_cast<float*>(p.ship_b) + tile * (S * 32) + lane;
    float4* planets = reinterpret_cast<float4*>(p.planets) + tile * (PL * 32) + lane;
    // The tile's bullet list: a dense run of capacity 32 K in the buffer being read, rewritten dense
    // into the same run of the other buffer.  32-bit indexing (astro_batch_create checks
    // n_games * K < 2^31): one IMAD.WIDE per address.
    const unsigned K = (unsigned)p.K;
    const unsigned tile_off = (unsigned)(g >> 5) * 32u * K;
    float4* const list_in = v.bullets_in + tile_off;
    float4* const list_out = v.bullets_out + tile_off;

    // ================= 1. this lane's game (rows already loaded: TileIn) ========================
    TL(0);
    const uint32_t meta = in.meta;
    float4 shv[2] = {in.shv[0], in.shv[1]};
    float sb[2] = {in.sb[0], in.sb[1]};
    int ctl[2];
    bool bad_ctl = false;
    const bool has_ring = !FIX && p.ring != nullptr;
    const uint32_t step_base = FIX ? 0u : (p.step_base ? *p.step_base : 0u);
    if (FIX || v.actions) {
        ctl[0] = (int)(in.ctl_raw & 0xffu);
        ctl[1] = S == 2 ? (int)(in.ctl_raw >> 8) : ctl[0];
        // codes above 5 are outside the reference's table (core.py:220-227): no-op control, tick flagged.
        // (a byte is 0..5 iff neither it nor it + 2 has a bit above the low three)
        bad_ctl = ((in.ctl_raw | (in.ctl_raw + 0x0202u)) & 0xf8f8u) != 0u;
        if (__builtin_expect(bad_ctl, 0)) {
            if (ctl[0] > 5) ctl[0] = 2;
            if (ctl[1] > 5) ctl[1] = 2;
        }
    } else if (!BOT) {
        // (the stream step: in a captured chunk of astro_rollout_device's loop — the counter stream with a recording ring of
        // observations — it is relative to the device step word)
        uint32_t h0 = game_key(p.seed, p.first_game + (uint32_t)g);
        ctl[0] = action_from_key(h0, v.step + step_base, 0u);
        ctl[1] = S == 2 ? action_from_key(h0, v.step + step_base, 1u) : ctl[0];
    } else {
        ctl[0] = ctl[1] = 2;      // (bots decide below, once the planets are here)
    }
    // What the END of the tick will need from memory is requested now, off the critical path: the
    // fire-schedule word of this game's tick and, with auto-reset, the planet count of the pool
    // entry that would replace the game (the pick is keyed on the stream step, not on state).
    const bool auto_reset = FIX || ((p.flags & ASTRO_TICK_AUTO_RESET) && (p.pool_size > 0 || p.ring != nullptr));
    const bool active = !ASTRO_META_FINISHED(meta);
    const int nb = active ? (int)ASTRO_META_NB(meta) : 0;
    const int np = active ? (int)meta_np<PL>(meta) : 0;
    const uint32_t tick = meta_tick<PL>(meta);
    float4 plv[PL];
#pragma unroll
    for (int j = 0; j < PL; j++) {
        plv[j] = make_float4(kFar, kFar, 0.f, 0.f);
        if (j < np) plv[j] = LD_STREAM(&planets[j * 32]);
    }

    if (BOT && !FIX && !v.actions) {
        // The bots of astro_rollout_device evaluated here, from the rows this lane has just loaded: script.ScriptBot
        // (script_decide: script.py:67-91, each ship from its own perspective) or script.NothingBot (control 2) per ship —
        // so that scripted games need no launch between ticks and run many ticks per launch like the counter-stream ones.
        if (active) {
            Body4<float> pl4[PL];
#pragma unroll
            for (int j = 0; j < PL; j++) { pl4[j].x = plv[j].x; pl4[j].y = plv[j].y; pl4[j].dx = plv[j].z; pl4[j].dy = plv[j].w; }
#pragma unroll
            for (int s = 0; s < S; s++) {
                if (((p.bot_modes >> (4 * s)) & 15) == ASTRO_BOT_SCRIPT) {
                    Body4<float> me, en;
                    me.x = shv[s].x; me.y = shv[s].y; me.dx = shv[s].z; me.dy = shv[s].w;
                    en.x = shv[S - 1 - s].x; en.y = shv[S - 1 - s].y; en.dx = shv[S - 1 - s].z; en.dy = shv[S - 1 - s].w;
                    ctl[s] = script_decide<float, S, PL>(me, sb[s], en, pl4, np, p.script);
                }
            }
        }
    }
    // The recording ring (astro_rollout_device_record): whatever the source of this tick's controls — the actions array, the
    // counter stream or the bots above — they are final here.  Row = the tick's stream step mod the ring's rows.
    const bool recording = !FIX && p.rec_events != nullptr;
    if (recording) {
        const size_t at = (size_t)rec_row * (unsigned)p.n_games + (unsigned)g;
        if (S == 2) ST_STREAM(reinterpret_cast<unsigned short*>(p.rec_controls) + at, (unsigned short)(ctl[0] | (ctl[1] << 8)));
        else ST_STREAM(p.rec_controls + at, (unsigned char)ctl[0]);
    }

    // ================= 2. flat bullet list of the tile; stage it with cp.async =================
#ifdef ASTRO_TIMELINE
    if (__shfl_xor_sync(full, meta, 1) == 0xdeadbeefu) return;  // consume meta: stamp 1 = meta has arrived
    TL(1);
#endif
    const unsigned total = __reduce_add_sync(full, (unsigned)nb);   // all the requests need; the prefix sums follow them
    const unsigned lt_mask = (1u << lane) - 1u, le_mask = full >> (31u - lane);
    const bool nonempty = nb > 0;
    const unsigned ne = __ballot_sync(full, nonempty);
    const unsigned cid = __popc(ne & lt_mask);                    // this game's rank among the games with bullets
    // a tile whose list does not fit the staging buffer (more than kStageWindows * 32 bullets, rare) takes several rounds
    const bool multi = !resident && total > (unsigned)kStageWindows * 32u;
    // the resident pool's per-game rows are indexed by lane (every lane writes its own), except in a tick of several rounds
    const bool by_lane = RES && !multi;
    const unsigned fi = by_lane ? lane : cid;
    using Scratch = TileScratchT<kStageWindows, PL>;
#if ASTRO_SMEM_ASM
    // every hot shared-memory access of the tick goes off this one base register (see lds128 above)
    const unsigned sbase = __shfl_sync(full, (unsigned)__cvta_generic_to_shared(&t), 0);
#define SOFF(field) (sbase + (unsigned)offsetof(Scratch, field))
    if (by_lane || nonempty) sts32(SOFF(hits) + fi * 4u, (unsigned)np << 8);
    if (RES) sts32(SOFF(gcount) + lane * 4u, 0u);
#else
    if (nonempty) t.hits[cid] = (unsigned)np << 8;
#endif
    // One window = 32 consecutive list items = 512 contiguous bytes; a round = up to kStageWindows
    // windows, all requested at once (16-byte cp.async each) and as early as possible — nothing
    // else sits between the arrival of meta and these requests (measured: working out the item ->
    // game labels here instead of in the bullet loop costs 10 % of the tick).  Lanes past the end of
    // the list stage a bullet that is certainly culled (no `valid` flag in the loop below).
#if ASTRO_SMEM_ASM
    const unsigned bul_s = SOFF(bul) + lane * 16u;
#else
    const unsigned bul_s = (unsigned)__cvta_generic_to_shared(&t.bul[lane]);
#endif
    auto stage_round = [&](unsigned round_base) {
        const unsigned left = total - round_base;
#if ASTRO_OPT_STAGE
        if (MANY) {
        // every window that holds a list item is requested, unrolled and predicated (one compare + one request each);
        // the lanes past the end of the list in the last window stage the sentinel.  (Fewer instructions; the one-tick
        // launch, which waits on HBM rather than on issue slots, is faster with the rolled loop below.)
        const float4* const src = list_in + round_base + lane;
#pragma unroll
        for (unsigned w = 0; w < (unsigned)kStageWindows; w++) {
            if (w * 32u + lane < left)
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(bul_s + w * 512u), "l"(src + w * 32u) : "memory");
        }
        const unsigned items = left < (unsigned)kStageWindows * 32u ? left : (unsigned)kStageWindows * 32u;
#if ASTRO_SMEM_ASM
        if ((items & 31u) != 0u && lane >= (items & 31u)) sts128(bul_s + (items & ~31u) * 16u, make_float4(4.0f, 4.0f, 0.0f, 0.0f));
#else
        if ((items & 31u) != 0u && lane >= (items & 31u)) t.bul[(items & ~31u) + lane] = make_float4(4.0f, 4.0f, 0.0f, 0.0f);
#endif
        cp_async_commit();
        return;
        }
#endif
        const unsigned n_win = left >= (unsigned)kStageWindows * 32u ? (unsigned)kStageWindows : (left + 31u) >> 5;
#pragma unroll 1
        for (unsigned w = 0; w < n_win; w++) {
            const unsigned item = round_base + w * 32u + lane;
            if (item < total) {
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(bul_s + w * 512u), "l"(list_in + item)
                             : "memory");
            } else {
                t.bul[w * 32u + lane] = make_float4(4.0f, 4.0f, 0.0f, 0.0f);
            }
        }
        cp_async_commit();
    };
    unsigned my_excl = 0;   // (the resident pool stages nothing and needs no prefix sum)
    if (!resident) {
        stage_round(0u);
        unsigned incl = (unsigned)nb;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            unsigned v = __shfl_up_sync(full, incl, d);
            if ((int)lane >= d) incl += v;
        }
        my_excl = incl - (unsigned)nb;
    }
    const unsigned start_key = nonempty ? my_excl : 0x80000000u;  // empty games never "start"
#if ASTRO_SMEM_ASM
    if (RES && !resident && !multi) {
        // the staged list becomes the pool: every item tagged with its game's lane (generation 0), the tail never live
        genmask = 0u;
        for (unsigned i = 0; i < (unsigned)nb; i++) sts8(SOFF(ref) + my_excl + i, lane);
        if ((total & 31u) != 0u && lane >= (total & 31u)) sts8(SOFF(ref) + (total & ~31u) + lane, 0xffu);
    }
#endif
    TL(2);

    // ================= 3. ships and planets while the bullets fly ===============================
    // OLD positions are staged for the bullet loop (addressed by game, transposed into the pairs
    // the packed distance code wants); the new ship / planet state goes straight to HBM.  (A
    // game that ends is re-created below; without auto-reset its ships and planets are left in
    // this post-step state: the state of a finished game is unspecified, the reference has none.)
#if ASTRO_SMEM_ASM
    sts128(SOFF(sxy) + lane * 16u, make_float4(shv[0].x, shv[1].x, shv[0].y, shv[1].y));
    sts128(SOFF(svel) + lane * 16u, make_float4(shv[0].z, shv[0].w, shv[1].z, shv[1].w));
    if (by_lane || nonempty) {
        sts128(SOFF(fsxy) + fi * 16u, make_float4(shv[0].x, shv[1].x, shv[0].y, shv[1].y));
#pragma unroll
        for (int k = 0; k < PL / 2; k++)
            sts128(SOFF(fpxy) + (unsigned)k * 512u + fi * 16u, make_float4(plv[2 * k].x, plv[2 * k + 1].x, plv[2 * k].y, plv[2 * k + 1].y));
    }
#else
    t.sxy[lane] = make_float4(shv[0].x, shv[1].x, shv[0].y, shv[1].y);
    t.svel[lane] = make_float4(shv[0].z, shv[0].w, shv[1].z, shv[1].w);
    if (nonempty) {
        t.fsxy[cid] = make_float4(shv[0].x, shv[1].x, shv[0].y, shv[1].y);
#pragma unroll
        for (int k = 0; k < PL / 2; k++) t.fpxy[k][cid] = make_float4(plv[2 * k].x, plv[2 * k + 1].x, plv[2 * k].y, plv[2 * k + 1].y);
    }
#endif
#ifdef ASTRO_TIMELINE
    if (__shfl_xor_sync(full, __float_as_uint(shv[0].x) ^ __float_as_uint(sb[1]) ^ __float_as_uint(plv[0].x) ^ __float_as_uint(plv[3].x), 1) == 0xdeadbeefu) return;
    TL(3);  // ships and planets have arrived
#endif
    unsigned hits = 0;
    next.shv[0] = shv[0]; next.shv[1] = shv[1];   // (finished games: rows untouched)
    next.sb[0] = sb[0]; next.sb[1] = sb[1];
#ifdef ASTRO_EXPERIMENTS
    // experiment builds only (flag 1024): the tick's memory traffic without its arithmetic — every load
    // and store of a tick whose games neither move nor end (tools/ab_repeat.sh, DESIGN.md section 5)
    const bool freeze = (p.flags & 1024) != 0;
    if (freeze && active) {
#pragma unroll
        for (int s = 0; s < S; s++) {
            ST_STREAM(&ships[s * 32], shv[s]);
            ST_STREAM(&ship_b[s * 32], sb[s]);
        }
#pragma unroll
        for (int i = 0; i < PL; i++)
            if (i < np) ST_STREAM(&planets[i * 32], plv[i]);
    }
    if (active && !freeze) {
#else
    if (active) {
#endif
        f32x2 pxy[PL];
#pragma unroll
        for (int j = 0; j < PL; j++) pxy[j] = pk2(plv[j].x, plv[j].y);
        float dirs[4];
        if (S == 2) np_sincos_f32x2(sb[0], sb[1], dirs[0], dirs[1], dirs[2], dirs[3]);
        else { np_sincos_f32(sb[0], dirs[0], dirs[1]); dirs[2] = dirs[0]; dirs[3] = dirs[1]; }
#if ASTRO_SMEM_ASM
        sts128(SOFF(dir) + lane * 16u, make_float4(dirs[0], dirs[1], dirs[2], dirs[3]));
#else
        t.dir[lane] = make_float4(dirs[0], dirs[1], dirs[2], dirs[3]);
#endif
        // direction, gravity, ship-planet and ship-ship collisions on the old state
#pragma unroll
        for (int s = 0; s < S; s++) {
            const f32x2 sxy = pk2(shv[s].x, shv[s].y);
            f32x2 acc = bc2(0.0f);
            float dmin = 3.0e38f;
#pragma unroll
            for (int j = 0; j < PL; j++) dmin = fminf(dmin, grav_pair(pxy[j], sxy, acc, c));
            bool h = dmin < c.r2f_sp;
            if (__builtin_expect(fabsf(dmin - c.r2f_sp) <= c.r2f_sp * 1e-6f, 0)) {
                h = false;
#pragma unroll
                for (int j = 0; j < PL; j++)
                    if (j < np)
                        h |= collide_exact((double)shv[s].x, (double)shv[s].y, (double)plv[j].x, (double)plv[j].y, c.r2_sp);
            }
            hits |= h ? (1u << s) : 0u;
            const float th = (ctl[s] & 1) ? c.thrust_f : 0.f;
            acc = fma2(bc2(th), pk2(dirs[2 * s], dirs[2 * s + 1]), acc);
            next.shv[s] = advance_body2(sxy, pk2(shv[s].z, shv[s].w), acc, c);  // core.py:283-288
            next.sb[s] = __fmaf_rn(c.db_unit_f, (float)((ctl[s] >> 1) - 1), sb[s]);
            if (last | !auto_reset) {   // (without auto-reset a game may end — and freeze — on any tick of the launch)
                ST_STREAM(&ships[s * 32], next.shv[s]);
                ST_STREAM(&ship_b[s * 32], next.sb[s]);
            }
        }
        if (S == 2) {
            if (collide(shv[0].x, shv[0].y, shv[1].x, shv[1].y, c.r2_ss, c.r2f_ss)) hits |= 3u;
        }
        // planets (core.py:289-294): pair forces are antisymmetric, the clamped self term is zero
        f32x2 q[PL];
#pragma unroll
        for (int i = 0; i < PL; i++) q[i] = bc2(0.0f);
#pragma unroll
        for (int i = 0; i < PL; i++) {
#pragma unroll
            for (int j = i + 1; j < PL; j++) {
                const f32x2 e = sub2(pxy[j], pxy[i]);
                float s0, s1;
                upk2(mul2(e, e), s0, s1);
                const float fj = div_fast_normal(c.gm_f, fmaxf(1e-12f, __fadd_rn(s0, s1)));  // dead: 0, or e = 0
                q[i] = fma2(bc2(fj), e, q[i]);
                q[j] = fma2(bc2(-fj), e, q[j]);
            }
        }
#pragma unroll
        for (int i = 0; i < PL; i++)
            if (i < np) ST_STREAM(&planets[i * 32], advance_body2(pxy[i], pk2(plv[i].z, plv[i].w), q[i], c));
    }

    // A game that ends here and now (ship hit a planet / the other ship, or timeout) will be re-created
    // from its pool record at the end: pull the record towards L2 while the bullet loop runs.
    // (the pick is a few dozen integer instructions: only the rare lanes that need it work it out)
    if (auto_reset && active && (hits || tick >= (uint32_t)p.timeout_tick)) {
        if (!has_ring) {
            const uint32_t k = pool_pick(p.seed, p.first_game + (uint32_t)g, v.step + step_base + 1u, (uint32_t)p.pool_size);
            const float4* const r = p.pool_rec + (size_t)k * pool_rec_float4s<PL>();
            asm volatile("prefetch.global.L2 [%0];" ::"l"(r));
            if (PL > ASTRO_MAX_PLANETS) asm volatile("prefetch.global.L2 [%0];" ::"l"(r + 8));   // (a 256-byte record: two lines)
        } else {
            // fresh-game mode: which record the game will get depends on who else ends this tick; the tile's next
            // record is the likely one
            asm volatile("prefetch.global.L2 [%0];" ::"l"(p.ring + ((size_t)tile_index * (unsigned)p.quota + min(t.used, (unsigned)p.quota - 1u)) * 8));
        }
    }

    // ================= 4. the bullet loop, from shared memory =======================================
    // Survivors are compacted over the WHOLE staged list, in list order (stable), labels along with
    // them: survivor number `pos` of the tile = survivors before the window (`carry`, warp-uniform) +
    // popc of the keep ballot below the lane.  Each game's first item records where the game's
    // survivors begin (and the previous game's end).  A tile whose list does not fit the staging
    // buffer (`multi`: more than kStageWindows * 32 bullets, rare) compacts into the list it is
    // reading instead — writes only land on items already consumed — and copies from there.
    unsigned carry = 0, c0 = 0;

    TL(4);  // physics done, new ship / planet state stored
    // (two copies of the loops, one per value of `multi`: the common one — a single round, survivors into shared memory —
    // carries neither the test nor the round loop)
    auto bullet_rounds = [&](auto multi_c) {
        constexpr bool MULTI = decltype(multi_c)::value;
        for (unsigned round_base = 0; round_base < (MULTI ? total : 1u); round_base += (unsigned)kStageWindows * 32u) {
            if (MULTI && round_base) {
                __syncwarp();
                stage_round(round_base);
            }
            cp_async_wait_all();
            __syncwarp();
            if (round_base == 0) TL(5);  // bullets have arrived
            const unsigned left = total - round_base;
            const unsigned n_win = (MULTI && left >= (unsigned)kStageWindows * 32u) ? (unsigned)kStageWindows : (left + 31u) >> 5;
#pragma unroll 1
            for (unsigned w = 0; w < n_win; w++) {
                // item -> game: bit r of `starts` = a game's first bullet is item r of this window; c0 =
                // games that started before it (warp-uniform)
                const unsigned rel = start_key - (round_base + w * 32u);   // >= 32 unless this lane's game starts here
                unsigned start_bit;      // 1 << rel, 0 for rel >= 32: PTX shl clamps the shift amount (C++ needs a test and a select)
                asm("shl.b32 %0, 1, %1;" : "=r"(start_bit) : "r"(rel));
                const unsigned starts = __reduce_or_sync(full, start_bit);
                const unsigned gi = c0 + __popc(starts & le_mask) - 1u;    // (items past the end: the last game)
                c0 += __popc(starts);
#if ASTRO_SMEM_ASM
                float4 bv = lds128(bul_s + w * 512u);
                const unsigned fr = sbase + gi * 16u;
                const float4 sT = lds128(fr + (unsigned)offsetof(Scratch, fsxy));
                float4 pT[PL / 2];
#pragma unroll
                for (int k = 0; k < PL / 2; k++) pT[k] = lds128(fr + (unsigned)offsetof(Scratch, fpxy) + (unsigned)k * 512u);
#else
                float4 bv = t.bul[w * 32u + lane];
                const float4 sT = t.fsxy[gi];
                float4 pT[PL / 2];
#pragma unroll
                for (int k = 0; k < PL / 2; k++) pT[k] = t.fpxy[k][gi];
#endif
                unsigned sh_hits = 0;
#ifdef ASTRO_EXPERIMENTS
                const bool keep = freeze ? (bv.x + sT.x + pT[0].x + pT[1].x != 123456.0f) : bullet_step_t<S, PL>(bv, sT, pT, t.hits, gi, c, sh_hits);
#else
                const bool keep = bullet_step_t<S, PL>(bv, sT, pT, t.hits, gi, c, sh_hits);
#endif
                if (sh_hits) atomicOr(&t.hits[gi], sh_hits);
                const unsigned kb = __ballot_sync(full, keep);   // (every lane has loaded its window item by now)
                const unsigned pos = carry + __popc(kb & lt_mask);
                if (keep) {
                    if (!MULTI) {
#if ASTRO_SMEM_ASM
                        sts128(sbase + (unsigned)offsetof(Scratch, bul) + pos * 16u, bv);
                        sts8(sbase + (unsigned)offsetof(Scratch, ref) + pos, gi);
#else
                        t.bul[pos] = bv;
                        t.ref[pos] = (uint8_t)gi;
#endif
                    } else {
                        list_in[pos] = bv;
                    }
                }
#if ASTRO_SMEM_ASM
                if ((starts >> lane) & 1u) sts16(sbase + (unsigned)offsetof(Scratch, gstart) + gi * 2u, pos);
#else
                if ((starts >> lane) & 1u) t.gstart[gi] = (uint16_t)pos;
#endif
                carry += __popc(kb);
            }
        }
    };
#if ASTRO_SMEM_ASM
    if (by_lane) {
        // The resident pool (section 6): item j's game comes from its tag; an item of a game that ended on the previous
        // tick (generation bit out of date) or past the end is dropped and counted nowhere.  The game's live items that
        // go (culled or hit a ship) are counted per game: survivors = nb - removed.
        cp_async_wait_all();
        __syncwarp();
        TL(5);
        const unsigned n_win = ((resident ? pool : total) + 31u) >> 5;
#pragma unroll 1
        for (unsigned w = 0; w < n_win; w++) {
            const unsigned tag = lds8(SOFF(ref) + w * 32u + lane);
            float4 bv = lds128(bul_s + w * 512u);
            const unsigned gl = tag & 31u;
            const bool live = tag_live(tag, genmask);
            const unsigned fr = sbase + gl * 16u;
            const float4 sT = lds128(fr + (unsigned)offsetof(Scratch, fsxy));
            float4 pT[PL / 2];
#pragma unroll
            for (int k = 0; k < PL / 2; k++) pT[k] = lds128(fr + (unsigned)offsetof(Scratch, fpxy) + (unsigned)k * 512u);
            unsigned sh_hits = 0;
#ifdef ASTRO_EXPERIMENTS
            bool keep = freeze ? (bv.x + sT.x + pT[0].x + pT[1].x != 123456.0f) : bullet_step_t<S, PL>(bv, sT, pT, t.hits, gl, c, sh_hits);
#else
            bool keep = bullet_step_t<S, PL>(bv, sT, pT, t.hits, gl, c, sh_hits);
#endif
            if (live && !keep) {   // (a ship hit is never kept)
                reds_add(SOFF(gcount) + gl * 4u, 1u);
                if (sh_hits) reds_or(SOFF(hits) + gl * 4u, sh_hits);
            }
            keep = keep && live;
            const unsigned kb = __ballot_sync(full, keep);   // (every lane has loaded its window item by now)
            const unsigned pos = carry + __popc(kb & lt_mask);
            if (keep) {
                sts128(SOFF(bul) + pos * 16u, bv);
                sts8(SOFF(ref) + pos, tag);
            }
            carry += __popc(kb);
        }
    } else
#endif
    if (total != 0u) {
        if (__builtin_expect(multi, 0)) bullet_rounds(std::true_type{});
        else bullet_rounds(std::false_type{});
    }
#if ASTRO_SMEM_ASM
    if (!by_lane && lane == 0) sts16(SOFF(gstart) + (unsigned)__popc(ne) * 2u, carry);
    __syncwarp();
    // first survivor of this lane's game in the compacted list, and one past its last
    const bool in_gstart = !by_lane && nonempty;
    const unsigned g_first = in_gstart ? lds16(SOFF(gstart) + cid * 2u) : 0u, g_end = in_gstart ? lds16(SOFF(gstart) + cid * 2u + 2u) : 0u;
#else
    if (lane == 0) t.gstart[__popc(ne)] = (uint16_t)carry;
    __syncwarp();
    // first survivor of this lane's game in the compacted list, and one past its last
    const unsigned g_first = nonempty ? (unsigned)t.gstart[cid] : 0u, g_end = nonempty ? (unsigned)t.gstart[cid + 1u] : 0u;
#endif
    TL(6);

    // ================= 5. terminal logic, spawn, bookkeeping ==========================================
    uint32_t ev = 0;
    next.meta = meta;
    int m_out = 0, spawned = 0;
    unsigned surv = 0, n_born = 0;      // what this game contributes to the new list: survivors, then newborn
    float4 born[2];
    born[0] = born[1] = make_float4(0.f, 0.f, 0.f, 0.f);
    float rw[2] = {0.0f, 0.0f};
    if (!active) {
        ev = ASTRO_EV_SKIPPED;
    } else {
        int m = 0;   // survivors of this game
#if ASTRO_SMEM_ASM
        if (by_lane) {
            m = nb - (int)lds32(SOFF(gcount) + lane * 4u);
            hits |= lds32(SOFF(hits) + lane * 4u) & 3u;
        } else
#endif
        if (nonempty) {
            m = (int)(g_end - g_first);
#if ASTRO_SMEM_ASM
            hits |= lds32(SOFF(hits) + cid * 4u) & 3u;
#else
            hits |= t.hits[cid] & 3u;
#endif
        }
#ifdef ASTRO_EXPERIMENTS
        const bool timeout = !freeze && tick >= (uint32_t)p.timeout_tick;
#else
        const bool timeout = tick >= (uint32_t)p.timeout_tick;
#endif
        if (hits) {  // core.py:253-255
            ev = hits;  // ASTRO_EV_HIT0 | ASTRO_EV_HIT1 are bits 0 and 1
#pragma unroll
            for (int s = 0; s < S; s++) rw[s] = ((hits >> s) & 1u) ? -1.0f : 1.0f;
        } else if (timeout) {  // core.py:257-260
            ev = ASTRO_EV_TIMEOUT;
#pragma unroll
            for (int s = 0; s < S; s++) rw[s] = c.reward_timeout;
        } else {
            surv = (unsigned)m;
            const uint32_t fire_word = have_fire_word ? in.fire_word : p.fire_bits[min(tick, (uint32_t)p.n_sched_ticks - 1u) >> 5];
#ifdef ASTRO_EXPERIMENTS
            const bool fire = !freeze && tick < (uint32_t)p.n_sched_ticks && ((fire_word >> (tick & 31)) & 1u);
#else
            const bool fire = tick < (uint32_t)p.n_sched_ticks && ((fire_word >> (tick & 31)) & 1u);
#endif
            if (fire) {  // core.py:267-280, from the OLD ship state
                ev |= ASTRO_EV_FIRED;
#if ASTRO_SMEM_ASM
                const float4 dv = lds128(SOFF(dir) + lane * 16u), oxy = lds128(SOFF(sxy) + lane * 16u), ov = lds128(SOFF(svel) + lane * 16u);
#else
                const float4 dv = t.dir[lane], oxy = t.sxy[lane], ov = t.svel[lane];
#endif
#pragma unroll
                for (int s = 0; s < S; s++) {
                    const float d0 = s == 0 ? dv.x : dv.z, d1 = s == 0 ? dv.y : dv.w;
                    const float sx = s == 0 ? oxy.x : oxy.y, sy = s == 0 ? oxy.z : oxy.w;
                    const float vx = s == 0 ? ov.x : ov.z, vy = s == 0 ? ov.y : ov.w;
                    // fp32 products as in the reference; the sums and the advance in fp32 too,
                    // unless the newborn lands within the band of the arena bound
                    float o0 = __fmul_rn(c.off_f, d0), o1 = __fmul_rn(c.off_f, d1);
                    float w0 = __fmul_rn(c.spd_f, d0), w1 = __fmul_rn(c.spd_f, d1);
                    float4 o;
                    o.z = __fadd_rn(vx, w0);
                    o.w = __fadd_rn(vy, w1);
                    o.x = __fmaf_rn(c.dt_f, o.z, __fadd_rn(sx, o0));
                    o.y = __fmaf_rn(c.dt_f, o.w, __fadd_rn(sy, o1));
                    float mn = fminf(fabsf(o.x), fabsf(o.y));
                    bool keep = mn <= 1.0f;
                    if (__builtin_expect(fabsf(mn - 1.0f) <= 8e-6f, 0)) {
                        Body4<double> nbl;
                        nbl.x = __dadd_rn((double)sx, (double)o0);
                        nbl.y = __dadd_rn((double)sy, (double)o1);
                        nbl.dx = __dadd_rn((double)vx, (double)w0);
                        nbl.dy = __dadd_rn((double)vy, (double)w1);
                        keep = advance_bullet(nbl, c);
                        o = make_float4((float)nbl.x, (float)nbl.y, (float)nbl.dx, (float)nbl.dy);
                    }
                    if (keep) {
                        if (m < (int)K) {
                            if (n_born == 0) born[0] = o; else born[1] = o;
                            n_born++;
                            m++;
                        } else {
                            ev |= ASTRO_EV_OVERFLOW;
                        }
                    }
                }
                spawned = S;
            }
            next.meta = meta_pack<PL>(m, np, 0, tick + 1);
            if (last) ST_STREAM(&p.meta[g], next.meta);
            m_out = m;
        }
        if (__builtin_expect(bad_ctl, 0)) ev |= ASTRO_EV_BAD_CONTROL;
    }
    // ---- a game that ended is re-created in the same launch (auto-reset) or frozen
    const bool ended = (ev & ASTRO_EV_DONE_MASK) != 0;       // (a skipped game: no)
    if (auto_reset) {
        // Where the new game comes from (core.create, core.py:86-135): a 128-byte record — ships (5 floats each), planet
        // count (word 10), planets (floats 16..31; 8-slot batches: 256 bytes, floats 16..47) — of the reset pool, picked by a hash of (game, stream step); or, in
        // fresh-game mode, the tile's next unused record of its ring (words 11 / 12: position in the generate_configs
        // stream, seed): a warp-local count, so every record — every stream position — is consumed exactly once.  A game
        // that finds the tile's ring empty waits, frozen (tick field = ASTRO_MAX_TICKS), and asks again every tick.
        const float4* rec = nullptr;
        if (has_ring) {
            const bool want = ended | (!active && meta_tick<PL>(meta) == max_ticks<PL>());
            const unsigned wants = __ballot_sync(full, want);
            if (wants) {
                const unsigned used = t.used;
                const unsigned idx = used + __popc(wants & lt_mask);
                __syncwarp();
                if (lane == 0) t.used = min(used + (unsigned)__popc(wants), (unsigned)p.quota);
                if (want && idx < (unsigned)p.quota) rec = p.ring + ((size_t)tile_index * (unsigned)p.quota + idx) * 8;
            }
        } else if (ended) {
            rec = p.pool_rec + (size_t)pool_pick(p.seed, p.first_game + (uint32_t)g, v.step + step_base + 1u, (uint32_t)p.pool_size) * pool_rec_float4s<PL>();
        }
        if (ended) atomicAdd(&p.episode[g], 1u);      // the per-slot episode counter: a fire-and-forget RED
        if (rec) {
            float4 r[4 + PL];
#pragma unroll
            for (int j = 0; j < 4 + PL; j++) r[j] = __ldg(&rec[j]);
            const int np_new = __float_as_int(r[2].z);
            next.shv[0] = r[0];
            next.sb[0] = r[1].x;
            if (last) {
                ships[0] = r[0];
                ship_b[0] = r[1].x;
            }
            if (S == 2) {
                next.shv[1] = make_float4(r[1].y, r[1].z, r[1].w, r[2].x);
                next.sb[1] = r[2].y;
                if (last) {
                    ships[32] = next.shv[1];
                    ship_b[32] = next.sb[1];
                }
            }
#pragma unroll
            for (int j = 0; j < PL; j++)
                if (j < np_new) planets[j * 32] = r[4 + j];
            next.meta = meta_pack<PL>(0, np_new, 0, 0);
            if (last) p.meta[g] = next.meta;
            if (!FIX && p.game_pos) p.game_pos[g] = __float_as_uint(r[2].w);
        } else if (ended) {
            ev |= ASTRO_EV_AWAIT;
            next.meta = meta_pack<PL>(0, np, 1, max_ticks<PL>());
            p.meta[g] = next.meta;
        }
    } else if (ended) {
        // Frozen from here on: the later ticks of this launch skip the game without touching its rows,
        // so the finished word goes to memory now, whichever tick of the launch this is (the ships were
        // stored by the physics above: without auto-reset every tick stores them) — identical to
        // separate astro_tick calls.
        next.meta = meta_pack<PL>(0, np, 1, tick);
        p.meta[g] = next.meta;
    }

    // ================= 6. the new list: survivors and newborn =======================================
    // In HBM: dense, into the other buffer, in game order, the game's survivors (reference order) then
    // its newborn.  The compacted list in shared memory is already that, except for the survivors of
    // games that just ended (dropped) and the newborn (inserted after their game): when the tile has
    // neither, the compacted list is copied out as it is; otherwise every survivor moves by its game's
    // shift.  Either way a step stores (nearly) contiguous 512 bytes.
    // The production rollout's fused form (RES) keeps the list in shared memory instead, as a resident
    // pool, and writes the dense list once per launch (below).
    const unsigned n_surv = carry;
#if ASTRO_SMEM_ASM
    if (RES) {
        // The resident pool: the compacted survivors stay in `bul`, each with its tag in `ref`, the newborn are appended
        // after them, and a game that ended flips its generation bit — its items die in the next tick's loop.  Nothing
        // goes to HBM: inside the launch only this warp reads the tile's list, so the pool need not be dense nor in game
        // order.  Each game's items stay in reference order among themselves (stable compaction, newborn after the
        // survivors).  The canonical list — dense, game order — is written once, on the launch's last tick, or when
        // survivors and newborn would not fit the staging buffer; the next tick then stages from HBM again.
        genmask ^= __ballot_sync(full, (ev & ASTRO_EV_DONE_MASK) != 0);
        bool write_out = true;
        if (!multi) {
            const unsigned b1 = __ballot_sync(full, n_born >= 1u), b2 = __ballot_sync(full, n_born >= 2u);
            const unsigned n_new = n_surv + (unsigned)(__popc(b1) + __popc(b2));
            if (!last && n_new <= (unsigned)kStageWindows * 32u) {
                write_out = false;
                const unsigned at = n_surv + (unsigned)(__popc(b1 & lt_mask) + __popc(b2 & lt_mask));
                const unsigned tag = lane | (((genmask >> lane) & 1u) << 5);
                if (n_born > 0) { sts128(SOFF(bul) + at * 16u, born[0]); sts8(SOFF(ref) + at, tag); }
                if (n_born > 1) { sts128(SOFF(bul) + at * 16u + 16u, born[1]); sts8(SOFF(ref) + at + 1u, tag); }
                if ((n_new & 31u) != 0u && lane >= (n_new & 31u)) {
                    sts128(SOFF(bul) + ((n_new & ~31u) + lane) * 16u, make_float4(4.0f, 4.0f, 0.0f, 0.0f));   // (certainly culled)
                    sts8(SOFF(ref) + (n_new & ~31u) + lane, 0xffu);
                }
                pool = n_new;
            }
        }
        if (write_out) {
            pool = kNotResident;
            unsigned oincl = (unsigned)m_out;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                unsigned v = __shfl_up_sync(full, oincl, d);
                if ((int)lane >= d) oincl += v;
            }
            const unsigned oexcl = oincl - (unsigned)m_out;
            if (n_born > 0) ST_STREAM(&list_out[oexcl + surv], born[0]);
            if (n_born > 1) ST_STREAM(&list_out[oexcl + surv + 1u], born[1]);
            if (!multi) {
                // a stable counting sort by game: item -> first(game) + rank among the game's earlier live items
                sts32(SOFF(gcount) + lane * 4u, oexcl);
                __syncwarp();
#pragma unroll 1
                for (unsigned j0 = 0; j0 < n_surv; j0 += 32u) {
                    const unsigned j = j0 + lane, tag = lds8(SOFF(ref) + j), gl = tag & 31u;
                    const bool live = j < n_surv && tag_live(tag, genmask);     // (games that ended on this tick: dropped)
                    const unsigned grp = __match_any_sync(full, live ? gl : 32u + lane);
                    unsigned at = 0;
                    if (live) {
                        at = lds32(SOFF(gcount) + gl * 4u);
                        ST_STREAM(&list_out[at + (unsigned)__popc(grp & lt_mask)], lds128(SOFF(bul) + j * 16u));
                    }
                    __syncwarp();
                    if (live && (grp >> lane) == 1u) sts32(SOFF(gcount) + gl * 4u, at + (unsigned)__popc(grp));
                    __syncwarp();
                }
            } else {
                // (rare) the survivors sit compacted in the list that was read: every lane copies its game's run
                for (unsigned k = 0; k < surv; k++) list_out[oexcl + k] = list_in[g_first + k];
            }
        }
    } else
#endif
    {
        const bool moves = __ballot_sync(full, (ev & ASTRO_EV_DONE_MASK) != 0 || n_born != 0) != 0;
        if (!moves && !multi) {
#pragma unroll 1
#if ASTRO_SMEM_ASM
            for (unsigned j = lane; j < n_surv; j += 32u) ST_STREAM(&list_out[j], lds128(SOFF(bul) + j * 16u));
#else
            for (unsigned j = lane; j < n_surv; j += 32u) ST_STREAM(&list_out[j], t.bul[j]);
#endif
        } else {
            unsigned oincl = (unsigned)m_out;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                unsigned v = __shfl_up_sync(full, oincl, d);
                if ((int)lane >= d) oincl += v;
            }
            const unsigned oexcl = oincl - (unsigned)m_out;
            if (n_born > 0) ST_STREAM(&list_out[oexcl + surv], born[0]);
            if (n_born > 1) ST_STREAM(&list_out[oexcl + surv + 1u], born[1]);
            if (!multi) {
#if ASTRO_SMEM_ASM
                if (nonempty) sts32(SOFF(shift) + cid * 4u, (unsigned)((ev & ASTRO_EV_DONE_MASK) ? kDrop : (int)oexcl - (int)g_first));
#else
                if (nonempty) t.shift[cid] = (ev & ASTRO_EV_DONE_MASK) ? kDrop : (int)oexcl - (int)g_first;
#endif
                __syncwarp();
                // (byte offsets from the two shared arrays and the list base: 9 instructions per step)
                const char* const bul_b = reinterpret_cast<const char*>(t.bul);
                char* const out_b = reinterpret_cast<char*>(list_out);
#pragma unroll 1
                for (unsigned j = lane; j < n_surv; j += 32u) {
#if ASTRO_SMEM_ASM
                    const int sh = (int)lds32(SOFF(shift) + lds8(SOFF(ref) + j) * 4u);
                    const float4 bv = lds128(SOFF(bul) + j * 16u);
#else
                    const int sh = t.shift[t.ref[j]];
                    const float4 bv = *reinterpret_cast<const float4*>(bul_b + j * 16u);
#endif
                    if (sh != kDrop) ST_STREAM(reinterpret_cast<float4*>(out_b + (size_t)((j + (unsigned)sh) * 16u)), bv);
                }
            } else {
                // (rare) the survivors sit compacted in the list that was read: every lane copies its game's run
                const unsigned from = g_first;
                for (unsigned k = 0; k < surv; k++) list_out[oexcl + k] = list_in[from + k];
            }
        }
    }
    if (!FIX && v.reward) {
        if (S == 2) reinterpret_cast<float2*>(v.reward)[g] = make_float2(rw[0], rw[1]);
        else v.reward[g] = rw[0];
    }
    if (FIX || v.events) {
        if (FIX || (p.flags & ASTRO_TICK_EVENT_PLANES)) {
            // three bit planes per tick, u32 [3][n_tiles]: bit g % 32 of word g / 32 = game g ended / ship 0 was hit /
            // ship 1 was hit (a timeout: ended and nobody hit) — 12 bytes per tile instead of 32
            const unsigned b_done = __ballot_sync(full, (ev & ASTRO_EV_DONE_MASK) != 0);
            const unsigned b_h0 = __ballot_sync(full, (ev & ASTRO_EV_HIT0) != 0), b_h1 = __ballot_sync(full, (ev & ASTRO_EV_HIT1) != 0);
            if (lane < 3u)
                reinterpret_cast<uint32_t*>(v.events)[(size_t)lane * ((unsigned)p.n_games >> 5) + tile_index] = lane == 0u ? b_done : (lane == 1u ? b_h0 : b_h1);
        } else {
            ST_STREAM(&v.events[g], (uint8_t)ev);
        }
    }
    if (!FIX && v.done) v.done[g] = (uint8_t)((ev & (ASTRO_EV_DONE_MASK | ASTRO_EV_SKIPPED)) ? 1 : 0);
    if (recording) ST_STREAM(&p.rec_events[(size_t)rec_row * (unsigned)p.n_games + (unsigned)g], (uint8_t)ev);

    if (STATS) {
        // warp totals -> this warp's private slot row in HBM (no block barrier, no contention);
        // astro_stats() folds the rows
        stat_acc += warp_totals((int)lane, S, ev, active, spawned, np, nb, m_out, true, total);
        if (last) {
            if (MANY && p.n_fused >= 8) {
                // a launch of many ticks: the tile's totals of the whole launch go straight to the 64-bit counters —
                // one RED per counter and tile per LAUNCH is cheap, and astro_stats needs no fold pass afterwards.  The
                // counters are kept kStatReplicas times (one 128-byte line each, picked by the tile), so that the REDs of
                // all the tiles do not queue on a single L2 line.
                if (lane < ASTRO_N_STATS && stat_acc) atomicAdd(&p.stats[(blockIdx.x & (unsigned)(kStatReplicas - 1)) * 16u + lane], (unsigned long long)stat_acc);   // (blockIdx: no live register)
            } else {
                unsigned* slot = p.stat_slots + ((size_t)(g >> 5) * 16u + lane);
                if (lane < ASTRO_N_STATS && stat_acc) atomicAdd(slot, stat_acc);  // RED: fire and forget
            }
        }
    }
    TL(7);
}

// ---- the launchable form ----------------------------------------------------------------------
// One warp (= one CTA) per tile; the block scheduler balances the load.  (Persistent forms — static
// tile striding, a device-side tile queue with the next tile's rows prefetched, a fully staged
// software pipeline — were built and measured 12-48 % slower: profiles/r1_ab_v6_experiments.md.)
// (BOT: the instantiation with the ScriptBot inside — float64 arithmetic of its own, far more registers: fewer CTAs per SM)
template <int S, bool STATS, bool MANY, bool BOT = false, bool FIX = false>
__global__ void __launch_bounds__(kTickThreads, BOT ? ASTRO_TICK_MIN_BLOCKS_BOT : (MANY ? ASTRO_TICK_MIN_BLOCKS_MANY : ASTRO_TICK_MIN_BLOCKS)) tick_f32_kernel(const __grid_constant__ TickParams p) {
    constexpr int PL = ASTRO_MAX_PLANETS;
    using TileScratch = TileScratchT<MANY ? ASTRO_STAGE_WINDOWS_MANY : ASTRO_STAGE_WINDOWS, PL>;
    __shared__ TileScratch s_tiles[kTickWarps];
    unsigned tile = (blockIdx.x * kTickThreads + threadIdx.x) >> 5;   // among the p.tiles tiles of this launch, from p.tile0
#if ASTRO_PDL
    if (!MANY) {
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // the next kernel's CTAs may take the slots this grid frees
        asm volatile("griddepcontrol.wait;" ::: "memory");                // ... and the previous kernel's stores are visible from here
    }
#endif
    if (tile >= (unsigned)p.tiles) return;  // whole warps: n_games % 32 == 0
#if ASTRO_BOUSTROPHEDON
    // Odd launches walk the tiles backwards: what the previous launch wrote last — still in the 126 MB L2 —
    // is read first, and rewritten there before it ever went to HBM.
    if ((!MANY || ASTRO_OPAQUE_TILE) && (p.step & 1u)) tile = (unsigned)p.tiles - 1u - tile;
#endif
    tile += (unsigned)p.tile0;
#if ASTRO_OPAQUE_TILE
    // A launch of several ticks: ptxas re-derives the tile index from %ctaid every tick (five instructions) rather than keep
    // it; the result of a shuffle it has to keep.  (A/B at 20 ticks per launch: 52.7 -> 50.8 us per tick together with the
    // cheaper statistics; without the backwards walk at all: 51.7.)
    if (MANY) tile = __shfl_sync(0xffffffffu, tile, 0);
#endif
#if ASTRO_OPAQUE_LANE
    // (several ticks per launch: ptxas re-reads %tid.x a dozen times per tick instead of keeping the lane id; a value that came
    // through a shuffle it keeps)
    const unsigned lane = MANY ? __shfl_sync(0xffffffffu, threadIdx.x & 31u, threadIdx.x & 31u) : (threadIdx.x & 31u);
#else
    const unsigned lane = threadIdx.x & 31u;
#endif
    // n_fused consecutive ticks of this tile, back to back (astro_tick_many): games do not interact, so a
    // tile can run ahead of the others; what tick k wrote is what tick k + 1 reads — from L2, not from HBM.
    // The rows are lane-private; the bullet list is written by some lanes and read by others: the warp
    // barrier orders those accesses.
    // (MANY = false: the one-tick launch, without the loop around it — the loop form costs a single tick 6 %)
    TileIn in, next;
    unsigned stat_acc = 0;
    unsigned pool = kNotResident, genmask = 0u;   // (the resident bullet pool of tick_tile, section 6: MANY && FIX only)
    TileScratch& scratch = s_tiles[kTickWarps == 1 ? 0 : (threadIdx.x >> 5)];
    // fresh-game mode: how many of the tile's pre-created games have been used since the last refill — requested with the
    // tile's rows, parked in shared memory once they are all on their way (a wait here would cost a round trip)
    unsigned used0 = 0;
    const bool has_ring = !FIX && p.ring != nullptr;
    if (has_ring && lane == 0) used0 = p.tile_used[tile];
    load_tile_in<S, PL, FIX>(p, tick_var<S>(p, 0u), tile, lane, in);
    if (has_ring && lane == 0) scratch.used = used0;
    // the recording ring's row of this launch's first tick (then one row further per tick, wrapping)
    unsigned rec_row = 0;
    if (!FIX && p.rec_events) rec_row = (p.step + (p.step_base ? *p.step_base : 0u)) % p.rec_ticks;
#pragma unroll 1
    for (unsigned k = 0; k < (MANY ? (unsigned)p.n_fused : 1u); k++) {
        const TickVar v = tick_var<S>(p, MANY ? k : 0u);
        // (several ticks per launch) the NEXT tick's controls are requested now — a different array every tick,
        // straight from HBM — so that they have arrived when this tick is done
        uint32_t ctl_next = 0;
        if (MANY && (FIX || p.actions) && k + 1u < (unsigned)p.n_fused) {
            const size_t g = (size_t)tile * 32 + lane;
            ctl_next = load_controls<S>(v.actions + p.act_stride, g, FIX || (p.flags & ASTRO_TICK_PACKED_CONTROLS) != 0);
        }
        if (MANY) in.fire_word = p.fire_bits[min(meta_tick<PL>(in.meta), (uint32_t)p.n_sched_ticks - 1u) >> 5];
        // (one-warp CTAs: the scratch is s_tiles[0], every shared address a compile-time constant — no base register)
        tick_tile<S, STATS, MANY, BOT, FIX, PL>(p, v, scratch, lane, tile, in, next, !MANY || k + 1u == (unsigned)p.n_fused, stat_acc, MANY, pool, genmask, rec_row);
        if (MANY) {
            if (++rec_row == p.rec_ticks) rec_row = 0;
            // The next tick of this tile: meta, ships and bearings are handed on in registers (they were stored as
            // well), so it starts its prefix sums and list requests at once; only the planet rows are loaded.  The
            // warp barrier orders this tick's list stores before the next tick's requests (no fence: a fence would
            // hold the warp until its last stores are acknowledged).
            in = next;
            in.ctl_raw = ctl_next;
            if (S == 1) { in.shv[1] = in.shv[0]; in.sb[1] = in.sb[0]; }
            __syncwarp();
        }
    }
    if (has_ring) {
        __syncwarp();
        if (lane == 0) p.tile_used[tile] = scratch.used;
    }
}

// The same shell for 8 planet slots, generic options only (no BOT / FIX forms): a kernel of its own name, so that the
// 4-slot kernels above are compiled exactly as before.
template <int S, bool STATS, bool MANY, bool BOT, bool FIX, int PL>
__device__ __forceinline__ void tick_f32_body(const TickParams& p) {
    using TileScratch = TileScratchT<MANY ? ASTRO_STAGE_WINDOWS_MANY : ASTRO_STAGE_WINDOWS, PL>;
    __shared__ TileScratch s_tiles[kTickWarps];
    unsigned tile = (blockIdx.x * kTickThreads + threadIdx.x) >> 5;   // among the p.tiles tiles of this launch, from p.tile0
#if ASTRO_PDL
    if (!MANY) {
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // the next kernel's CTAs may take the slots this grid frees
        asm volatile("griddepcontrol.wait;" ::: "memory");                // ... and the previous kernel's stores are visible from here
    }
#endif
    if (tile >= (unsigned)p.tiles) return;  // whole warps: n_games % 32 == 0
#if ASTRO_BOUSTROPHEDON
    // Odd launches walk the tiles backwards: what the previous launch wrote last — still in the 126 MB L2 —
    // is read first, and rewritten there before it ever went to HBM.
    if ((!MANY || ASTRO_OPAQUE_TILE) && (p.step & 1u)) tile = (unsigned)p.tiles - 1u - tile;
#endif
    tile += (unsigned)p.tile0;
#if ASTRO_OPAQUE_TILE
    // A launch of several ticks: ptxas re-derives the tile index from %ctaid every tick (five instructions) rather than keep
    // it; the result of a shuffle it has to keep.  (A/B at 20 ticks per launch: 52.7 -> 50.8 us per tick together with the
    // cheaper statistics; without the backwards walk at all: 51.7.)
    if (MANY) tile = __shfl_sync(0xffffffffu, tile, 0);
#endif
#if ASTRO_OPAQUE_LANE
    // (several ticks per launch: ptxas re-reads %tid.x a dozen times per tick instead of keeping the lane id; a value that came
    // through a shuffle it keeps)
    const unsigned lane = MANY ? __shfl_sync(0xffffffffu, threadIdx.x & 31u, threadIdx.x & 31u) : (threadIdx.x & 31u);
#else
    const unsigned lane = threadIdx.x & 31u;
#endif
    // n_fused consecutive ticks of this tile, back to back (astro_tick_many): games do not interact, so a
    // tile can run ahead of the others; what tick k wrote is what tick k + 1 reads — from L2, not from HBM.
    // The rows are lane-private; the bullet list is written by some lanes and read by others: the warp
    // barrier orders those accesses.
    // (MANY = false: the one-tick launch, without the loop around it — the loop form costs a single tick 6 %)
    TileIn in, next;
    unsigned stat_acc = 0;
    unsigned pool = kNotResident, genmask = 0u;   // (the resident bullet pool of tick_tile, section 6: MANY && FIX only)
    TileScratch& scratch = s_tiles[kTickWarps == 1 ? 0 : (threadIdx.x >> 5)];
    // fresh-game mode: how many of the tile's pre-created games have been used since the last refill — requested with the
    // tile's rows, parked in shared memory once they are all on their way (a wait here would cost a round trip)
    unsigned used0 = 0;
    const bool has_ring = !FIX && p.ring != nullptr;
    if (has_ring && lane == 0) used0 = p.tile_used[tile];
    load_tile_in<S, PL, FIX>(p, tick_var<S>(p, 0u), tile, lane, in);
    if (has_ring && lane == 0) scratch.used = used0;
    // the recording ring's row of this launch's first tick (then one row further per tick, wrapping)
    unsigned rec_row = 0;
    if (!FIX && p.rec_events) rec_row = (p.step + (p.step_base ? *p.step_base : 0u)) % p.rec_ticks;
#pragma unroll 1
    for (unsigned k = 0; k < (MANY ? (unsigned)p.n_fused : 1u); k++) {
        const TickVar v = tick_var<S>(p, MANY ? k : 0u);
        // (several ticks per launch) the NEXT tick's controls are requested now — a different array every tick,
        // straight from HBM — so that they have arrived when this tick is done
        uint32_t ctl_next = 0;
        if (MANY && (FIX || p.actions) && k + 1u < (unsigned)p.n_fused) {
            const size_t g = (size_t)tile * 32 + lane;
            ctl_next = load_controls<S>(v.actions + p.act_stride, g, FIX || (p.flags & ASTRO_TICK_PACKED_CONTROLS) != 0);
        }
        if (MANY) in.fire_word = p.fire_bits[min(meta_tick<PL>(in.meta), (uint32_t)p.n_sched_ticks - 1u) >> 5];
        // (one-warp CTAs: the scratch is s_tiles[0], every shared address a compile-time constant — no base register)
        tick_tile<S, STATS, MANY, BOT, FIX, PL>(p, v, scratch, lane, tile, in, next, !MANY || k + 1u == (unsigned)p.n_fused, stat_acc, MANY, pool, genmask, rec_row);
        if (MANY) {
            if (++rec_row == p.rec_ticks) rec_row = 0;
            // The next tick of this tile: meta, ships and bearings are handed on in registers (they were stored as
            // well), so it starts its prefix sums and list requests at once; only the planet rows are loaded.  The
            // warp barrier orders this tick's list stores before the next tick's requests (no fence: a fence would
            // hold the warp until its last stores are acknowledged).
            in = next;
            in.ctl_raw = ctl_next;
            if (S == 1) { in.shv[1] = in.shv[0]; in.sb[1] = in.sb[0]; }
            __syncwarp();
        }
    }
    if (has_ring) {
        __syncwarp();
        if (lane == 0) p.tile_used[tile] = scratch.used;
    }
}

template <int S, bool STATS, bool MANY>
__global__ void __launch_bounds__(kTickThreads, MANY ? ASTRO_TICK_MIN_BLOCKS_WIDE_MANY : ASTRO_TICK_MIN_BLOCKS_WIDE) tick_f32_wide_kernel(const __grid_constant__ TickParams p) {
    tick_f32_body<S, STATS, MANY, false, false, ASTRO_MAX_PLANETS_WIDE>(p);
}
