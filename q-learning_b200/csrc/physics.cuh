// physics.cuh — device-side Breakout mechanics for sm_100a (one thread advances one env).
//
// B200-first restructuring of the reference's AoS / Vec<Brick> / recursive code
// (/root/reference/src/breakout-game/src/mechanics.rs:119-214,257-444,485-649 and algebra_2d.rs:46-75):
//   * bricks are a 60-bit mask (bit 20*row + k) and a closed-form grid, so the <= 4 bricks that can possibly
//     touch the ball are enumerated by index arithmetic instead of testing all 60 AABBs;
//   * the recursion of proceed_ball_with / binary_search_first_contact becomes bounded loops with sticky
//     error flags instead of panics / unbounded stack;
//   * acos() is removed: |acos(d)| > FRAC_PI_2 holds for exactly the f32 set -1 <= d <= -1.03316033e-07
//     with glibc 2.39 acosf (exhaustive sweep over all 2^32 inputs, see DESIGN.md), so the acceptance test
//     (mechanics.rs:327) is two compares;
//   * f32::hypot (glibc hypotf) is reproduced bit-exactly as (float)sqrt((double)x*x + (double)y*y).
// Everything is compiled with -fmad=false: Rust never contracts a*b+c, and one ulp eventually flips a brick hit.
#pragma once
#include <stdint.h>
#include <cuda_runtime.h>

namespace qlc {

constexpr uint32_t ENVERR_WALL_DISTANCE = 1u, ENVERR_APPROX_RANGE = 2u, ENVERR_RECURSION = 4u,
                   ENVERR_BISECTION = 8u, ENVERR_DEGENERATE = 16u, ENVERR_ACTION = 32u;
constexpr int MAX_REFLECTIONS = 16;   // proceed_ball_with recursion bound
constexpr int MAX_BISECTION = 40;     // binary_search_first_contact bound

// mechanics.rs:12-44
constexpr float GRID_X = 600.0f, GRID_Y = 600.0f;
constexpr float SPACE_GRANULARITY = 0.001f;
constexpr float DT = 0.02f;                    // Duration::from_millis(20).as_secs_f32()
constexpr float PAD_MIN_Y = 565.0f, PAD_MAX_Y = 575.0f, PAD_INIT_MIN_X = 270.0f, PAD_INIT_MAX_X = 330.0f;
constexpr float PAD_VMAX = 160.0f, PAD_ACCEL = 20.0f, PAD_BRAKE = 7.0f;
constexpr float BALL_R = 10.0f, BALL_SPEED = 200.0f;
constexpr float CONTACT_PREDICTION = 0.8f;
constexpr float F32_EPS = 1.1920929e-7f;
constexpr uint64_t ALL_BRICKS = 0x0FFFFFFFFFFFFFFFull;   // 3 rows x 20

struct Surface { float way, approx, nx, ny; };
struct Contact { bool some; float dist, nx, ny; };        // (nx, ny) = box-side normal; ball-side normal = -(nx, ny)

// Vec2::length = f32::hypot -> glibc hypotf: double-precision sum of exact squares, one sqrt, one narrowing.
__device__ __forceinline__ float length2(float x, float y) {
    double dx = (double)x, dy = (double)y;
    return (float)sqrt(dx * dx + dy * dy);
}
// Vec2::normalized (emath 0.22): zero vector stays, otherwise component-wise division by the length.
__device__ __forceinline__ void normalize2(float& x, float& y) {
    float len = length2(x, y);
    if (len > 0.0f) { x = x / len; y = y / len; }
}
// f32::round (half away from zero), exact for |x| < 2^23 and the identity above.
__device__ __forceinline__ float round_half_away(float x) {
    float t = truncf(x);
    if (fabsf(x - t) >= 0.5f) t += copysignf(1.0f, x);
    return t;
}
__device__ __forceinline__ float granulate(float v) { return round_half_away(v * 1000.0f) / 1000.0f; }

// parry2d query::contact(ball, cuboid, prediction = 0.8) for axis-aligned translations.
// (acx, acy) box centre, (hex, hey) half extents.
__device__ __noinline__ Contact contact_degenerate(float px, float py, float qx, float qy, float sx, float sy,
                                                   float hex, float hey, float r, uint32_t& err) {
    // ball centre on the box boundary (|proj - centre| <= eps). Unreachable in play; kept so that the device code
    // answers the reference's own vector mechanics.rs:721 like parry2d does: feature normal, else the direction
    // box-centre -> projection, else +y.
    (void)px; (void)py;
    err |= ENVERR_DEGENERATE;
    Contact c; c.some = false; c.dist = -r; c.nx = 0.0f; c.ny = 0.0f;
    const bool zx = (sx == 0.0f), zy = (sy == 0.0f);
    bool have = false;
    if (zx && zy) {
        if (qx > hex - F32_EPS)        { c.nx = 1.0f;  have = true; }
        else if (qx <= -hex + F32_EPS) { c.nx = -1.0f; have = true; }
        else if (qy > hey - F32_EPS)   { c.ny = 1.0f;  have = true; }
        else if (qy <= -hey + F32_EPS) { c.ny = -1.0f; have = true; }
    } else if (zx != zy) {
        if (!zx) c.nx = (qx < (-hex + hex) / 2.0f) ? -1.0f : 1.0f;
        else     c.ny = (qy < (-hey + hey) / 2.0f) ? -1.0f : 1.0f;
        have = true;
    } else {
        float vx = (qx < (-hex + hex) / 2.0f) ? -1.0f : 1.0f, vy = (qy < (-hey + hey) / 2.0f) ? -1.0f : 1.0f;
        float n = sqrtf(vx * vx + vy * vy);
        c.nx = vx / n; c.ny = vy / n; have = true;
    }
    if (!have) {
        float psq = qx * qx + qy * qy;
        if (psq > F32_EPS * F32_EPS) { float n = sqrtf(psq); c.nx = qx / n; c.ny = qy / n; }
        else { c.nx = 0.0f; c.ny = 1.0f; }
    }
    c.some = (c.dist <= CONTACT_PREDICTION);
    return c;
}

__device__ __forceinline__ Contact contact_ball_box(float bx, float by, float r, float acx, float acy,
                                                    float hex, float hey, uint32_t& err) {
    // ball centre in the box frame
    const float px = -(acx - bx), py = -(acy - by);
    const float lox = -hex - px, hix = px - hex;      // mins - pt, pt - maxs
    const float loy = -hey - py, hiy = py - hey;
    const float sx = (lox > 0.0f ? lox : 0.0f) - (hix > 0.0f ? hix : 0.0f);
    const float sy = (loy > 0.0f ? loy : 0.0f) - (hiy > 0.0f ? hiy : 0.0f);
    const bool inside = (sx == 0.0f) && (sy == 0.0f);
    float fx = sx, fy = sy;                            // shift actually applied
    if (inside) {
        // hollow projection: move to the nearest face
        float best = -3.40282347e+38f; int axis = 0; bool is_min = false;
        if (lox < hix) { if (hix > best) { axis = 0; is_min = false; best = hix; } }
        else if (lox > best) { axis = 0; is_min = true; best = lox; }
        if (loy < hiy) { if (hiy > best) { axis = 1; is_min = false; best = hiy; } }
        else if (loy > best) { axis = 1; is_min = true; best = loy; }
        const float s = is_min ? best : -best;
        fx = (axis == 0) ? s : 0.0f;
        fy = (axis == 1) ? s : 0.0f;
    }
    const float qx = px + fx, qy = py + fy;            // projection
    const float vx = qx - px, vy = qy - py;
    const float sq = vx * vx + vy * vy;
    if (!(sq > F32_EPS * F32_EPS)) return contact_degenerate(px, py, qx, qy, fx, fy, hex, hey, r, err);
    const float len = sqrtf(sq);
    const float ux = vx / len, uy = vy / len;          // ball centre -> box
    Contact c;
    if (inside) { c.dist = -len - r; c.nx = ux;  c.ny = uy; }
    else        { c.dist =  len - r; c.nx = -ux; c.ny = -uy; }
    c.some = (c.dist <= CONTACT_PREDICTION);
    return c;
}

// Ball::collision_check_with_rectangle (mechanics.rs:318-443) as a loop.
__device__ __forceinline__ bool sweep_ball_box(float cx, float cy, float r, float mvx, float mvy, float len_mv,
                                               float acx, float acy, float hex, float hey,
                                               Surface& out, uint32_t& err) {
    Contact c = contact_ball_box(cx + mvx, cy + mvy, r, acx, acy, hex, hey, err);
    if (!c.some) return false;
    float way, approx, nx, ny;
    if (c.dist < 0.0f) {
        // penetrating at the end of the move: closed-form back-off, then bisection if the estimate misses
        const float cosang = ((-c.nx) * mvx + (-c.ny) * mvy) / len_mv;
        const float back = fabsf(c.dist) / cosang;
        const float p = 1.0f - back / len_mv;
        Contact c2 = contact_ball_box(cx + mvx * p, cy + mvy * p, r, acx, acy, hex, hey, err);
        if (c2.some && !(c2.dist < 0.0f)) {
            way = len_mv * p; approx = c2.dist; nx = c2.nx; ny = c2.ny;
        } else {
            float lo = c2.some ? 0.0f : p;
            float hi = c2.some ? p : 1.0f;
            int depth = 0;
            for (;;) {
                const float m = (lo + hi) / 2.0f;
                Contact cm = contact_ball_box(cx + mvx * m, cy + mvy * m, r, acx, acy, hex, hey, err);
                if (depth >= MAX_BISECTION) {
                    err |= ENVERR_BISECTION;
                    way = len_mv * m; approx = 0.0f;
                    nx = cm.some ? cm.nx : 0.0f; ny = cm.some ? cm.ny : 1.0f;
                    break;
                }
                if (!cm.some) lo = m;
                else if (cm.dist < 0.0f) hi = m;
                else { way = len_mv * m; approx = cm.dist; nx = cm.nx; ny = cm.ny; break; }
                ++depth;
            }
        }
    } else {
        way = len_mv; approx = c.dist; nx = c.nx; ny = c.ny;
    }
    // accept only surfaces facing the motion: |acos(mv^ . n^)| > pi/2  <=>  -1 <= d <= -1.03316033e-07 (NaN rejects)
    float ax = mvx, ay = mvy; normalize2(ax, ay);
    float bx = nx, by = ny;   normalize2(bx, by);
    const float d = ax * bx + ay * by;
    if (!(d >= -1.0f && d <= __uint_as_float(0xB3DDDE97u))) return false;
    out.way = way; out.approx = approx; out.nx = nx; out.ny = ny;
    return true;
}

// One env's mechanics registers.
struct Env {
    float cx, cy, dx, dy;          // ball centre, direction (un-normalised until the first bounce: mechanics.rs:103,166)
    float pmin, pmax, pspeed;      // paddle min.x, max.x (kept separately: :571-587), speed
    uint64_t bricks;
    uint32_t score;
    uint32_t err;
    bool finished;
};

__device__ __forceinline__ void env_init(Env& e, float dir_x) {           // mechanics.rs:57-116
    e.cx = GRID_X * 0.5f; e.cy = GRID_Y * 0.5f; e.dx = dir_x; e.dy = -1.0f;
    e.pmin = PAD_INIT_MIN_X; e.pmax = PAD_INIT_MAX_X; e.pspeed = 0.0f;
    e.bricks = ALL_BRICKS; e.score = 0u; e.finished = false;
}

struct Candidates {
    static constexpr int CAP = 8;                 // 3 walls + paddle + at most 2x2 bricks near the ball
    float way[CAP], approx[CAP], nx[CAP], ny[CAP];
    int brick[CAP];
    int n;
    __device__ __forceinline__ void push(const Surface& s, int b, uint32_t& err) {
        if (!(s.approx >= 0.0f && s.approx <= CONTACT_PREDICTION)) err |= ENVERR_APPROX_RANGE;   // mechanics.rs:511
        if (n < CAP) { way[n] = s.way; approx[n] = s.approx; nx[n] = s.nx; ny[n] = s.ny; brick[n] = b; ++n; }
    }
};

// proceed_ball_with (mechanics.rs:137-184) without recursion. len0 = |mv| of the first leg (cached by the caller:
// it is a pure function of the direction). Returns true when the direction changed (a reflection happened).
__device__ __forceinline__ bool advance_ball(Env& e, float mvx, float mvy, float len0) {
    bool bounced = false;
    for (int bounce = 0;; ++bounce) {
        const float len_mv = bounce == 0 ? len0 : length2(mvx, mvy);
        if (len_mv < SPACE_GRANULARITY) return bounced;
        Candidates cs; cs.n = 0;
        Surface s;
        // walls (mechanics.rs:260-315), insertion order left, right, top
        {
            const float d = e.cx - BALL_R;
            if (!(d >= 0.0f)) e.err |= ENVERR_WALL_DISTANCE;
            if (!(d + mvx > 0.0f)) {
                const float f = d / fabsf(mvx);
                s.way = length2(mvx * f, mvy * f); s.approx = 0.0f; s.nx = 1.0f; s.ny = 0.0f; cs.push(s, -1, e.err);
            }
        }
        {
            const float d = GRID_X - e.cx - BALL_R;
            if (!(d >= 0.0f)) e.err |= ENVERR_WALL_DISTANCE;
            if (!(mvx < d)) {
                const float f = d / fabsf(mvx);
                s.way = length2(mvx * f, mvy * f); s.approx = 0.0f; s.nx = -1.0f; s.ny = 0.0f; cs.push(s, -1, e.err);
            }
        }
        {
            const float d = e.cy - BALL_R - 0.0f;
            if (!(d >= 0.0f)) e.err |= ENVERR_WALL_DISTANCE;
            if (!(d + mvy > 0.0f)) {
                const float f = d / fabsf(mvy);
                s.way = length2(mvx * f, mvy * f); s.approx = 0.0f; s.nx = 0.0f; s.ny = 1.0f; cs.push(s, -1, e.err);
            }
        }
        // paddle: the sweep starts with a contact query at the end point, which answers None unless that point is
        // within r + prediction (10.8) of the box — skip the query when it is not even within 11.5
        {
            const float ex = e.cx + mvx, ey = e.cy + mvy;
            if (ey > PAD_MIN_Y - 11.5f && ey < PAD_MAX_Y + 11.5f && ex > e.pmin - 11.5f && ex < e.pmax + 11.5f) {
                if (sweep_ball_box(e.cx, e.cy, BALL_R, mvx, mvy, len_mv, (e.pmin + e.pmax) / 2.0f, (PAD_MIN_Y + PAD_MAX_Y) / 2.0f,
                                   (e.pmax - e.pmin) / 2.0f, (PAD_MAX_Y - PAD_MIN_Y) / 2.0f, s, e.err))
                    cs.push(s, -1, e.err);
            }
        }
        // bricks: only the grid cells whose box, grown by r + prediction (+ slack), contains the end point can
        // return a contact at all; every other brick answers None in the reference too.
        if (e.cy + mvy < 126.0f) {     // lowest brick edge 114 + 11.x
            const float ex = e.cx + mvx, ey = e.cy + mvy;
            int k0 = (int)ceilf((ex - 66.0f) / 27.0f), k1 = (int)floorf((ex - 19.0f) / 27.0f);
            int r0 = (int)ceilf((ey - 71.0f) / 27.0f), r1 = (int)floorf((ey - 24.0f) / 27.0f);
            k0 = k0 < 0 ? 0 : k0; k1 = k1 > 19 ? 19 : k1; r0 = r0 < 0 ? 0 : r0; r1 = r1 > 2 ? 2 : r1;
            for (int r = r0; r <= r1; ++r)
                for (int k = k0; k <= k1; ++k) {
                    const int b = 20 * r + k;
                    if ((e.bricks >> b) & 1ull) {
                        if (sweep_ball_box(e.cx, e.cy, BALL_R, mvx, mvy, len_mv, 42.5f + 27.0f * (float)k, 47.5f + 27.0f * (float)r,
                                           12.5f, 12.5f, s, e.err))
                            cs.push(s, b, e.err);
                    }
                }
        }
        if (cs.n == 0) { e.cx = e.cx + mvx; e.cy = e.cy + mvy; return bounced; }

        // ContactCandidates::consider (:496-516): the surviving set is {way+approx <= min + 0.001}, insertion order kept
        float way, nx, ny;
        if (cs.n == 1) {
            way = cs.way[0]; nx = cs.nx[0]; ny = cs.ny[0];
            if (cs.brick[0] >= 0) { e.bricks &= ~(1ull << cs.brick[0]); e.score += 1u; }
        } else {
            float best = __int_as_float(0x7f800000);
            for (int i = 0; i < cs.n; ++i) { const float p = cs.way[i] + cs.approx[i]; if (p < best) best = p; }
            const float limit = best + SPACE_GRANULARITY;
            float sx = 0.0f, sy = 0.0f, sw = 0.0f; int kept = 0; int first = -1;
            for (int i = 0; i < cs.n; ++i) {
                if (cs.way[i] + cs.approx[i] <= limit) {
                    if (first < 0) first = i;
                    sx = sx + cs.nx[i]; sy = sy + cs.ny[i]; sw = sw + cs.way[i]; ++kept;
                    if (cs.brick[i] >= 0) { e.bricks &= ~(1ull << cs.brick[i]); e.score += 1u; }
                }
            }
            if (kept == 1) { way = cs.way[first]; nx = cs.nx[first]; ny = cs.ny[first]; }
            else { normalize2(sx, sy); nx = sx; ny = sy; way = sw / (float)kept; }      // :519-538
        }
        // reflect (:165-171)
        const float ncx = e.cx + e.dx * way, ncy = e.cy + e.dy * way;
        const float remaining = len_mv - way;
        const float f = 2.0f * (e.dx * nx + e.dy * ny);
        float rx = e.dx - nx * f, ry = e.dy - ny * f;
        normalize2(rx, ry);
        e.cx = ncx; e.cy = ncy; e.dx = rx; e.dy = ry;
        bounced = true;
        mvx = rx * remaining; mvy = ry * remaining;
        if (!(length2(mvx, mvy) > 0.0f)) return bounced;
        if (bounce >= MAX_REFLECTIONS) { e.err |= ENVERR_RECURSION; return bounced; }
    }
}

// Ball::move_vector (:258): ((normalized(dir) * speed) * dt) and its length — pure functions of the direction, so they
// are cached in registers and recomputed only after a reflection or a reset (bit-identical to recomputing each step).
struct MoveCache { float mvx, mvy, len; };
__device__ __forceinline__ void move_cache_update(MoveCache& m, const Env& e) {
    float ux = e.dx, uy = e.dy; normalize2(ux, uy);
    m.mvx = ux * BALL_SPEED * DT; m.mvy = uy * BALL_SPEED * DT;
    m.len = length2(m.mvx, m.mvy);
}

// BreakoutMechanics::time_step (mechanics.rs:119-129)
__device__ __forceinline__ void time_step(Env& e, uint32_t action, MoveCache& mc) {
    // Panel::proceed (:571-587) with the speed chosen on the previous step
    {
        const float d = e.pspeed * DT;
        const float nmin = e.pmin + d, nmax = e.pmax + d;
        if (nmin <= 0.0f)        { const float s = -nmin;        e.pmin = nmin + s; e.pmax = nmax + s; e.pspeed = 0.0f; }
        else if (nmax >= GRID_X) { const float s = GRID_X - nmax; e.pmin = nmin + s; e.pmax = nmax + s; e.pspeed = 0.0f; }
        else { e.pmin = nmin; e.pmax = nmax; }
    }
    if (advance_ball(e, mc.mvx, mc.mvy, mc.len)) move_cache_update(mc, e);
    if (e.cy >= PAD_MAX_Y || e.bricks == 0ull) e.finished = true;               // :131-135
    if (!e.finished) {                                                           // Panel::process_input :553-566
        const float v = e.pspeed;
        if (action == 1u || action == 2u) {                                      // accelerate :631-649
            const float t = v + (action == 1u ? -PAD_ACCEL : PAD_ACCEL);
            const float lim = fabsf(t) > PAD_VMAX ? (signbit(t) ? -PAD_VMAX : PAD_VMAX) : t;
            e.pspeed = granulate(lim);
        } else {                                                                 // decrease_speed :616-628 (brakes a negative speed to 0 at once)
            float g = 0.0f;
            if (v > 0.0f) g = granulate(v - PAD_BRAKE);
            else if (v < 0.0f) g = granulate(v + PAD_BRAKE);
            e.pspeed = g > 0.0f ? g : 0.0f;
        }
    }
}

// ---- Philox-4x32-10 (Salmon et al., SC'11) and the random inputs derived from it ----
constexpr uint32_t STREAM_RESET = 0x52455345u, STREAM_SAMPLE = 0x53414D50u, STREAM_ACTION = 0x41435449u, STREAM_PRIORITY = 0x5052494Fu;

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
    #pragma unroll
    for (int i = 0; i < 10; ++i) {
        const uint32_t h0 = __umulhi(0xD2511F53u, c.x), l0 = 0xD2511F53u * c.x;
        const uint32_t h1 = __umulhi(0xCD9E8D57u, c.z), l1 = 0xCD9E8D57u * c.z;
        c = make_uint4(h1 ^ c.y ^ k.x, l1, h0 ^ c.w ^ k.y, l0);
        k.x += 0x9E3779B9u; k.y += 0xBB67AE85u;
    }
    return c;
}
// The learner's pure-random phase (self_driving_tf_q_learner.rs:153-157: rng.gen_range(0..ACTION_SPACE) while
// step_count < epsilon_pure_random_steps) with the draw made on the device: uniform in {0, 1, 2} from word 0 of
// philox({env_global_id, t, 0, 'ACTI'}) by multiply-shift (the synthetic action stream of bench.py and the oracle).
__device__ __forceinline__ uint32_t policy_action(uint64_t seed, uint32_t env_global_id, uint32_t t) {
    const uint4 r = philox4x32_10(make_uint4(env_global_id, t, 0u, STREAM_ACTION), make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    return (uint32_t)(((uint64_t)r.x * 3ull) >> 32);
}
// rand 0.8.5 gen_range(-0.35f32..-0.15) from 32 random bits (mechanics.rs:103)
__device__ __forceinline__ float reset_dir_x(uint64_t seed, uint32_t env_global_id, uint32_t episode) {
    const uint4 r = philox4x32_10(make_uint4(env_global_id, episode, 0u, STREAM_RESET), make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const float low = -0.35f, high = -0.15f;
    const float scale = high - low;
    const float v01 = __uint_as_float(0x3F800000u | (r.x >> 9)) - 1.0f;
    return v01 * scale + low;
}

}  // namespace qlc
