// astro_device.cuh — device-side arithmetic of the batched Astro tick (sm_100a).
//
// Two arithmetic policies behind one template parameter R:
//   R = double  the validation build: every operation is the reference's float64 numpy op, in
//               the reference's order, one rounding each (__dadd_rn/__dmul_rn/__ddiv_rn never
//               contract to FMA) — bit-identical to astro/core.py on float64 inputs.
//   R = float   the production build: state is stored and integrated in fp32 (HBM-bound, the
//               FP64 pipe stays idle), but every DISCRETE predicate (collision, bullet cull) is
//               decided exactly as the reference's float64 arithmetic would on the same inputs:
//               a fp32 evaluation with a proven error bound decides unless the value falls in
//               the uncertainty band, where the reference's float64 expression is evaluated.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace astro {

template <typename R>
struct alignas(4 * sizeof(R)) Body4 {
    R x, y, dx, dy;
};

// ---- the meta word (include/astro_b200.h) of a batch with PL planet slots ---------------------
// PL = 4 reads and writes today's fields; PL = 8 keeps np's fourth bit in bit 31 (ASTRO_META_*_WIDE).
template <int PL>
__host__ __device__ __forceinline__ uint32_t meta_np(uint32_t m) {
    return PL > ASTRO_MAX_PLANETS ? ASTRO_META_NP_WIDE(m) : ASTRO_META_NP(m);
}
template <int PL>
__host__ __device__ __forceinline__ uint32_t meta_tick(uint32_t m) {
    return PL > ASTRO_MAX_PLANETS ? ASTRO_META_TICK_WIDE(m) : ASTRO_META_TICK(m);
}
template <int PL>
__host__ __device__ __forceinline__ uint32_t meta_pack(uint32_t nb, uint32_t np, uint32_t fin, uint32_t tick) {
    return PL > ASTRO_MAX_PLANETS ? ASTRO_META_PACK_WIDE(nb, np, fin, tick) : ASTRO_META_PACK(nb, np, fin, tick);
}
template <int PL>
__host__ __device__ constexpr uint32_t max_ticks() { return PL > ASTRO_MAX_PLANETS ? ASTRO_MAX_TICKS_WIDE : ASTRO_MAX_TICKS; }

// ---- counter-based streams (host twin: astro_b200/rng.py) -------------------------------
__device__ __forceinline__ uint32_t mix32(uint32_t x) {
    x ^= x >> 16; x *= 0x7FEB352Du; x ^= x >> 15; x *= 0x846CA68Bu; x ^= x >> 16;
    return x;
}
__device__ __forceinline__ uint32_t game_key(uint32_t seed, uint32_t game) {
    return mix32(seed ^ (game * 0x9E3779B1u));
}
__device__ __forceinline__ int action_from_key(uint32_t h0, uint32_t step, uint32_t ship) {
    return (int)__umulhi(mix32(h0 ^ (step * 2u + ship)), 6u);
}
__device__ __forceinline__ uint32_t pool_pick(uint32_t seed, uint32_t game, uint32_t key, uint32_t pool_size) {
    uint32_t h0 = mix32(seed ^ 0xA5A5A5A5u ^ (game * 0x9E3779B1u));
    return __umulhi(mix32(h0 ^ key), pool_size);
}

// ---- util.direction (util.py:87-92) -----------------------------------------------------
// numpy evaluates sin/cos of float32 input with its SIMD kernel: 3-constant Cody-Waite
// reduction (FMA) and degree-8/9 polynomials.  Restated operation for operation so the result
// is the same float32 bit pattern (|x| <= 71476; bearings stay below ~250).
__device__ __forceinline__ void np_sincos_f32(float x, float& sn, float& cs) {
    const float magic = 12582912.0f;  // 0x1.8p+23
    float q = __fsub_rn(__fmaf_rn(x, 0x1.45f306p-1f, magic), magic);
    float r = __fmaf_rn(q, -0x1.921fb0p+00f, x);
    r = __fmaf_rn(q, -0x1.5110b4p-22f, r);
    r = __fmaf_rn(q, -0x1.846988p-48f, r);
    float r2 = __fmul_rn(r, r);
    float c = __fmaf_rn(0x1.98e616p-16f, r2, -0x1.6c06dcp-10f);
    c = __fmaf_rn(c, r2, 0x1.55553cp-5f);
    c = __fmaf_rn(c, r2, -0x1.000000p-1f);
    c = __fmaf_rn(c, r2, 0x1.000000p+0f);
    float s = __fmaf_rn(0x1.7d3bbcp-19f, r2, -0x1.a06bbap-13f);
    s = __fmaf_rn(s, r2, 0x1.11119ap-7f);
    s = __fmaf_rn(s, r2, -0x1.555556p-3f);
    s = __fmaf_rn(s, r2, 0.0f);
    s = __fmaf_rn(s, r, r);
    int iq = (int)q;
    float vs = (iq & 1) ? c : s;
    sn = (iq & 2) ? -vs : vs;
    int ic = iq + 1;
    float vc = (ic & 1) ? c : s;
    cs = (ic & 2) ? -vc : vc;
}

// ---- numpy floored remainder / util.wrap_unit_square (util.py:145-148) -------------------
__device__ __forceinline__ double np_remainder(double a, double b) {
    double m = fmod(a, b);
    if (m != 0.0) {
        if ((b < 0) != (m < 0)) m = __dadd_rn(m, b);
    } else {
        m = copysign(0.0, b);
    }
    return m;
}
// ((x + 1) % 2) - 1 in float64.  (y mod 2) = y - 2*floor(y/2) is exact for a power-of-two
// modulus, including numpy's "+0 when the remainder is zero" and the rounding of tiny
// negative y up to 2.0.
__device__ __forceinline__ double wrap_unit_f64(double x) {
    double y = __dadd_rn(x, 1.0);
    double r = __dsub_rn(y, __dmul_rn(2.0, floor(__dmul_rn(y, 0.5))));
    return __dsub_rn(r, 1.0);
}
// fp32 state: inside (-1, 1) the reference's wrap is the identity up to 1e-16, so only a body
// that actually left the square (rare) evaluates it.
__device__ __forceinline__ float wrap_unit_f32(float x) {
    float y = __fadd_rn(x, 1.0f);
    float r = __fsub_rn(y, __fmul_rn(2.0f, floorf(__fmul_rn(y, 0.5f))));
    return __fsub_rn(r, 1.0f);
}
// util.norm_angle(b) / pi (util.py:125-132, rl.py:58): float64, then stored as float32.
__device__ __forceinline__ float norm_angle_over_pi(double b) {
    const double PI = 3.141592653589793;
    double a = __dsub_rn(np_remainder(__dadd_rn(b, PI), __dmul_rn(2.0, PI)), PI);
    return (float)__ddiv_rn(a, PI);
}

// ---- constants of one batch (host-computed in float64, the reference's Python floats) -----
struct Consts {
    double gm;       // gravity * planet_mass                       core.py:149
    double dt;
    double thrust;   // ship_thrust                                  core.py:238
    double db_unit;  // dt * ship_rspeed                             core.py:239
    double zero_dt;  // 0 * dt: bullets integrate with a = 0         core.py:297
    double r2_ss, r2_sp, r2_sb, r2_pb;  // (r_i + r_j)^2             core.py:211
    float off_f, spd_f;                 // f32(1.001*ship_radius), f32(bullet_speed)  core.py:273,277
    float gm_f, dt_f, thrust_f, db_unit_f;
    float r2f_ss, r2f_sp, r2f_sb, r2f_pb;
    float reward_timeout;               // 1 solo / 0 duel           core.py:259-260
};

// ---- the discrete predicates -------------------------------------------------------------
// core._collisions (core.py:200-212): |x_j - x_i|^2 < (r_i + r_j)^2, strict.
__device__ __forceinline__ bool collide_exact(double ax, double ay, double bx, double by, double r2) {
    double d0 = __dsub_rn(bx, ax), d1 = __dsub_rn(by, ay);
    return __dadd_rn(__dmul_rn(d0, d0), __dmul_rn(d1, d1)) < r2;
}
__device__ __forceinline__ bool collide(double ax, double ay, double bx, double by, double r2, float) {
    return collide_exact(ax, ay, bx, by, r2);
}
// fp32 filter: d2 carries a relative error <= 4u (u = 2^-24: one subtraction per axis, one
// product, one FMA; no cancellation in a sum of squares), r2f <= u.  Outside a 16u band the
// fp32 comparison provably equals the reference's float64 one; inside, evaluate that.
__device__ __forceinline__ bool collide(float ax, float ay, float bx, float by, double r2, float r2f) {
    float d0 = __fsub_rn(bx, ax), d1 = __fsub_rn(by, ay);
    float d2 = __fmaf_rn(d1, d1, __fmul_rn(d0, d0));
    bool h = d2 < r2f;
    if (fabsf(d2 - r2f) <= r2f * 1e-6f) h = collide_exact((double)ax, (double)ay, (double)bx, (double)by, r2);
    return h;
}
// core._update_bodies cull (core.py:192-195): keep iff (-1<=x'<=1) or (-1<=y'<=1).
__device__ __forceinline__ bool in_arena(double x0, double x1) {
    return ((-1.0 <= x0) & (x0 <= 1.0)) | ((-1.0 <= x1) & (x1 <= 1.0));
}

// One bullet: dx' = dx + 0*dt ; x' = x + dt*dx' ; returns keep flag; b updated in place.
__device__ __forceinline__ bool advance_bullet(Body4<double>& b, const Consts& c) {
    double v0 = __dadd_rn(b.dx, c.zero_dt), v1 = __dadd_rn(b.dy, c.zero_dt);
    double x0 = __dadd_rn(b.x, __dmul_rn(c.dt, v0)), x1 = __dadd_rn(b.y, __dmul_rn(c.dt, v1));
    b.x = x0; b.y = x1; b.dx = v0; b.dy = v1;
    return in_arena(x0, x1);
}
// fp32: x' = fma(dt_f, v, x) is within (|v| dt + |x'|) u of the float64 value; only when |x'|
// is that close to 1 can the inclusive bound test differ — then evaluate the reference's.
__device__ __forceinline__ bool advance_bullet(Body4<float>& b, const Consts& c) {
    float x0 = __fmaf_rn(c.dt_f, b.dx, b.x), x1 = __fmaf_rn(c.dt_f, b.dy, b.y);
    bool in0 = fabsf(x0) <= 1.0f, in1 = fabsf(x1) <= 1.0f;
    bool near0 = fabsf(fabsf(x0) - 1.0f) <= 2e-6f * (1.0f + fabsf(b.dx));
    bool near1 = fabsf(fabsf(x1) - 1.0f) <= 2e-6f * (1.0f + fabsf(b.dy));
    bool keep = in0 | in1;
    if (near0 | near1) {
        double v0 = __dadd_rn((double)b.dx, c.zero_dt), v1 = __dadd_rn((double)b.dy, c.zero_dt);
        double e0 = __dadd_rn((double)b.x, __dmul_rn(c.dt, v0)), e1 = __dadd_rn((double)b.y, __dmul_rn(c.dt, v1));
        keep = in_arena(e0, e1);
        x0 = (float)e0; x1 = (float)e1;
    }
    b.x = x0; b.y = x1;
    return keep;
}

// x / y for a NORMAL y (never subnormal): one MUFU.RCP and one multiply, the same bits as __fdividef,
// which spends four more instructions per call on subnormal denominators (no -ftz build here).
__device__ __forceinline__ float div_fast_normal(float x, float y) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(y));
    return __fmul_rn(x, r);
}

// ---- gravity (core.py:138-153) -------------------------------------------------------------
// One term f * rx with f = G*M / max(1e-12, |rx|^2); also reports |rx|^2 for the collision test
// of the same pair.
__device__ __forceinline__ void grav_term(double px, double py, double x, double y, const Consts& c,
                                          double& t0, double& t1) {
    double r0 = __dsub_rn(px, x), r1 = __dsub_rn(py, y);
    double d2 = __dadd_rn(__dmul_rn(r0, r0), __dmul_rn(r1, r1));
    double f = __ddiv_rn(c.gm, fmax(1e-12, d2));
    t0 = __dmul_rn(f, r0);
    t1 = __dmul_rn(f, r1);
}
__device__ __forceinline__ void grav_term(float px, float py, float x, float y, const Consts& c,
                                          float& t0, float& t1) {
    float r0 = __fsub_rn(px, x), r1 = __fsub_rn(py, y);
    float d2 = __fmaf_rn(r1, r1, __fmul_rn(r0, r0));
    float f = div_fast_normal(c.gm_f, fmaxf(1e-12f, d2));
    t0 = __fmul_rn(f, r0);
    t1 = __fmul_rn(f, r1);
}

// ---- the first tick after core.create (validation build) -----------------------------------
// core.create (core.py:86-135) returns float32 ship and planet positions, so on a game's first tick numpy
// evaluates _gravity and the squared distances of _collisions in float32 — one rounding per operation, no FMA,
// IEEE division — before everything promotes to float64 (ASTRO_TICK_CREATE_DTYPES).
__device__ __forceinline__ void grav_term_np32(float px, float py, float x, float y, float gm_f, float& t0, float& t1) {
    const float r0 = __fsub_rn(px, x), r1 = __fsub_rn(py, y);
    const float d2 = __fadd_rn(__fmul_rn(r0, r0), __fmul_rn(r1, r1));
    const float f = __fdiv_rn(gm_f, fmaxf(1e-12f, d2));
    t0 = __fmul_rn(f, r0);
    t1 = __fmul_rn(f, r1);
}
__device__ __forceinline__ bool collide_np32(float ax, float ay, float bx, float by, double r2) {
    const float d0 = __fsub_rn(bx, ax), d1 = __fsub_rn(by, ay);
    return (double)__fadd_rn(__fmul_rn(d0, d0), __fmul_rn(d1, d1)) < r2;   // float32 < float64: promoted exactly
}

// ---- symplectic Euler (core.py:189-197) -----------------------------------------------------
__device__ __forceinline__ void advance_body(Body4<double>& s, double a0, double a1, const Consts& c) {
    double v0 = __dadd_rn(s.dx, __dmul_rn(a0, c.dt)), v1 = __dadd_rn(s.dy, __dmul_rn(a1, c.dt));
    s.x = wrap_unit_f64(__dadd_rn(s.x, __dmul_rn(c.dt, v0)));
    s.y = wrap_unit_f64(__dadd_rn(s.y, __dmul_rn(c.dt, v1)));
    s.dx = v0; s.dy = v1;
}
__device__ __forceinline__ void advance_body(Body4<float>& s, float a0, float a1, const Consts& c) {
    float v0 = __fmaf_rn(a0, c.dt_f, s.dx), v1 = __fmaf_rn(a1, c.dt_f, s.dy);
    float x0 = __fmaf_rn(c.dt_f, v0, s.x), x1 = __fmaf_rn(c.dt_f, v1, s.y);
    if (__builtin_expect(fmaxf(fabsf(x0), fabsf(x1)) >= 1.0f, 0)) {
        if (fabsf(x0) >= 1.0f) x0 = wrap_unit_f32(x0);
        if (fabsf(x1) >= 1.0f) x1 = wrap_unit_f32(x1);
    }
    s.x = x0; s.y = x1;
    s.dx = v0; s.dy = v1;
}

__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }

template <typename R> struct Pick;
template <> struct Pick<double> {
    static __device__ __forceinline__ double thrust(const Consts& c) { return c.thrust; }
    static __device__ __forceinline__ double db_unit(const Consts& c) { return c.db_unit; }
};
template <> struct Pick<float> {
    static __device__ __forceinline__ float thrust(const Consts& c) { return c.thrust_f; }
    static __device__ __forceinline__ float db_unit(const Consts& c) { return c.db_unit_f; }
};


// ---- script.ScriptBot (script.py:13-91) ---------------------------------------------------------
struct ScriptParams {
    double radius;           // planet_radius + ship_radius                  script.py:53
    double avoid_distance, avoid_threshold;
    double ship_thrust, ship_rspeed, bullet_speed, ship_radius;
    int32_t solo, n_games;
};

// fmod(a, m) for m > 0 and |a / m| < 2^52, exact like the library routine but in a few operations: with
// the right integer quotient q, a - q m is representable (it is the result) and fma(-q, m, a) rounds
// once, i.e. not at all; a quotient off by one after the division's rounding is corrected and redone.
__device__ __forceinline__ double fmod_small(double a, double m) {
    const double x = fabs(a);
    double q = floor(__ddiv_rn(x, m));
    double r = fma(-q, m, x);
    if (r < 0.0) { q -= 1.0; r = fma(-q, m, x); }
    else if (r >= m) { q += 1.0; r = fma(-q, m, x); }
    return copysign(r, a);   // sign of the dividend (C fmod), -0.0 kept
}
__device__ __forceinline__ double norm_angle_f64(double b) {  // util.norm_angle, util.py:125-132
    const double PI = 3.141592653589793, TWO_PI = 6.283185307179586;
    const double a = __dadd_rn(b, PI);
    double m = fmod_small(a, TWO_PI);          // numpy's floored remainder (divisor > 0)
    if (m != 0.0) { if (m < 0.0) m = __dadd_rn(m, TWO_PI); } else m = 0.0;
    return __dsub_rn(m, PI);
}
__device__ __forceinline__ int fly_to(double target, double my_b, double t, bool fwd) {  // script.py:30-39
    const double angle = norm_angle_f64(__dsub_rn(target, my_b));
    if (angle < -t) return 0;
    if (t < angle) return 4;
    return fwd ? 3 : 2;
}


// script.ScriptBot.__call__ (script.py:67-91) for one ship seen from its own perspective (core.roll_ships, core.py:306-327):
// mv / mb = my ship (x, y, dx, dy) and bearing, ev = the other ship, pl[0..np-1] = the planets.  float64 throughout, the
// reference's operations in its order.  The cheap part of _danger (:41-65) — two square roots, two divisions, the
// discriminant — runs for every planet without divergence and leaves a bit mask of the planets on a collision course;
// only those go through the atan2 / norm_angle test, in planet order (the first dangerous planet decides, script.py:69-76).
// Quirk kept: inside _danger the parameter `b` (my bearing) is shadowed by the quadratic coefficient (script.py:54).
template <typename R, int S, int PL>
__device__ __forceinline__ int script_decide(const Body4<R>& mv, R mb, const Body4<R>& ev, const Body4<R> (&pl)[PL], int np,
                                             const ScriptParams& q) {
    const double my[5] = {(double)mv.x, (double)mv.y, (double)mv.dx, (double)mv.dy, (double)mb};
    unsigned cand = 0;
    double cx0[PL], cx1[PL], cb[PL], csd[PL], cspeed[PL];
    const double ra = __dadd_rn(q.radius, q.avoid_distance);
    const double ra2 = __dmul_rn(ra, ra);
#pragma unroll
    for (int j = 0; j < PL; j++) {
        cx0[j] = cx1[j] = cb[j] = csd[j] = cspeed[j] = 0.0;
        if (j < np) {
            const Body4<R> v = pl[j];
            const double x0 = __dsub_rn(my[0], (double)v.x), x1 = __dsub_rn(my[1], (double)v.y);
            const double v0 = __dsub_rn(my[2], (double)v.dx), v1 = __dsub_rn(my[3], (double)v.dy);
            const double speed = sqrt(__dadd_rn(__dmul_rn(v0, v0), __dmul_rn(v1, v1)));   // util.mag(dx)
            const double den = __dadd_rn(speed, 1e-12);
            const double n0 = __ddiv_rn(v0, den), n1 = __ddiv_rn(v1, den);                   // util.norm(dx)
            const double b = __dmul_rn(2.0, __dadd_rn(__dmul_rn(n0, x0), __dmul_rn(n1, x1)));
            const double mx = sqrt(__dadd_rn(__dmul_rn(x0, x0), __dmul_rn(x1, x1)));
            const double cc = __dsub_rn(__dmul_rn(mx, mx), ra2);
            const double det = __dsub_rn(__dmul_rn(b, b), __dmul_rn(4.0, cc));
            if (0.0 < det) {
                const double sd = sqrt(det);
                if (0.0 <= __dadd_rn(-b, sd)) {       // real roots, at least one positive (script.py:57)
                    cand |= 1u << j;
                    cx0[j] = x0; cx1[j] = x1; cb[j] = b; csd[j] = sd; cspeed[j] = speed;
                }
            }
        }
    }
    int ctl = -1;
    while (cand && ctl < 0) {
        const int j = __ffs(cand) - 1;
        cand &= cand - 1u;
        double x0 = cx0[0], x1 = cx1[0], b = cb[0], sd = csd[0], speed = cspeed[0];
#pragma unroll
        for (int k = 1; k < PL; k++)
            if (j == k) { x0 = cx0[k]; x1 = cx1[k]; b = cb[k]; sd = csd[k]; speed = cspeed[k]; }
        const double distance = __dsub_rn(-b, sd);
        const double bear = atan2(x0, x1);                                        // util.bearing(x)
        const double rotation = fabs(norm_angle_f64(__dsub_rn(bear, b)));         // (`b` shadowed: script.py:54)
        const double lim = __dmul_rn(__dadd_rn(__ddiv_rn(speed, q.ship_thrust), __ddiv_rn(q.ship_rspeed, rotation)), speed);
        if (distance < lim) ctl = fly_to(bear, my[4], q.avoid_threshold, true);
    }
    if (ctl < 0) {
        if (q.solo || S < 2) {
            ctl = 2;
        } else {
            const double en[4] = {(double)ev.x, (double)ev.y, (double)ev.dx, (double)ev.dy};
            const double e0 = __dsub_rn(en[0], my[0]), e1 = __dsub_rn(en[1], my[1]);
            const double enemy_distance = sqrt(__dadd_rn(__dmul_rn(e0, e0), __dmul_rn(e1, e1)));
            const double bullet_time = __ddiv_rn(enemy_distance, q.bullet_speed);
            const double f0 = __dadd_rn(en[0], __dmul_rn(bullet_time, __dsub_rn(en[2], my[2])));
            const double f1 = __dadd_rn(en[1], __dmul_rn(bullet_time, __dsub_rn(en[3], my[3])));
            ctl = fly_to(atan2(__dsub_rn(f0, my[0]), __dsub_rn(f1, my[1])), my[4], __ddiv_rn(q.ship_radius, enemy_distance), false);
        }
    }
    return ctl;
}

}  // namespace astro
