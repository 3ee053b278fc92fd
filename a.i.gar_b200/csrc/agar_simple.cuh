/*
 * agar_simple.cuh — register-resident kernel for single-cell pellet-collection envs (BASELINE configs[1], [4]):
 * K = 1 NN agent, one cell, no viruses / split / eject, pellet channel only.
 *
 * Why a second kernel: in k_main the per-frame work of such an env is ~1000 dependent lane-0 instructions that
 * go through shared-memory structs (profiles/r01_k_main_W32_*), and sub-warp tiles fall out of lockstep at
 * every tile-level barrier.  Here
 *   - an env is owned by W adjacent lanes (W = 1, 2, 4, 8); its whole scalar state is REPLICATED in the registers
 *     of those lanes, which all execute the same scalar arithmetic (no broadcast, no lane-0 sections);
 *   - control flow is warp-uniform: every data-dependent loop runs until no tile of the warp needs another
 *     iteration, collectives always use the full mask, so the 32/W envs of a warp advance per instruction;
 *   - only the pellet pool (packed u32) sits in shared memory; the O(pool) loops are strided over the W lanes:
 *     an integer window pre-filter builds a per-lane candidate bitmask, the exact float64 tests then run on the few
 *     candidates in slot order (tile-min), which keeps the reference's sequential eat chain exact;
 *   - observations are accumulated straight into the caller's buffer with fire-and-forget float REDs (pellet
 *     masses are small integers: exact and order-free).
 * Semantics and arithmetic are those of k_main<W,false> (same helpers, same operation order): the two kernels are
 * bit-identical, and both equal the portable-math oracle.
 */
#pragma once
#include "agar_bots.cuh"
#include "agar_dev.cuh"

#define S_FULL 0xffffffffu
#define S_NONE 0x7fffffff

struct SReg {
    /* header */
    uint32_t rng_field, frame;
    int32_t n_pellets, n_events;
    uint64_t event_hash;
    /* player */
    double cmd_x, cmd_y, fov_x, fov_y, fov_size;
    int32_t fov_valid;
    /* the cell */
    double x, y, mass, radius, svx, svy, merge_time;
    int32_t counter;
    uint32_t uid, flags;
    /* bot */
    int32_t has_action, has_last_action, skip_frames, has_last_mass, has_old_state, time, skipping, turn_begun, need_action,
        exp_valid, exp_done;
    double a0, a1, a2, a3, l0, l1, l2, l3;
    double cum_reward, last_reward, last_mass, fov_size_feat, stat_mass_sum, stat_mass_max, stat_frames;
};

struct SPtr {
    AgarEnvHeader* h; /* global memory: scalar part of the record (touched at launch start / end only) */
    AgarPlayer* p;
    AgarCell* c;
    uint32_t* pel;    /* shared memory: pellet slots */
    AgarEvent* ev;    /* shared memory: event ring   */
    uint32_t* grid;   /* shared memory: G x G mass sums of the observation being built (nullptr: accumulate in the caller's row) */
};

DEV void s_load(SReg& r, const SPtr& q) {
    r.rng_field = q.h->rng_field, r.frame = q.h->frame, r.n_pellets = q.h->n_pellets, r.n_events = q.h->n_events;
    r.event_hash = q.h->event_hash;
    r.cmd_x = q.p->cmd_x, r.cmd_y = q.p->cmd_y, r.fov_x = q.p->fov_x, r.fov_y = q.p->fov_y, r.fov_size = q.p->fov_size;
    r.fov_valid = q.p->fov_valid;
    r.x = q.c->x, r.y = q.c->y, r.mass = q.c->mass, r.radius = q.c->radius, r.svx = q.c->svx, r.svy = q.c->svy;
    r.merge_time = q.c->merge_time, r.counter = q.c->counter, r.uid = q.c->uid, r.flags = q.c->flags;
    const AgarBot* B = &q.p->bot;
    r.has_action = B->has_action, r.has_last_action = B->has_last_action, r.skip_frames = B->skip_frames;
    r.has_last_mass = B->has_last_mass, r.has_old_state = B->has_old_state, r.time = B->time, r.skipping = B->skipping;
    r.turn_begun = B->turn_begun, r.need_action = B->need_action, r.exp_valid = B->exp_valid, r.exp_done = B->exp_done;
    r.a0 = B->cur_action[0], r.a1 = B->cur_action[1], r.a2 = B->cur_action[2], r.a3 = B->cur_action[3];
    r.l0 = B->last_action[0], r.l1 = B->last_action[1], r.l2 = B->last_action[2], r.l3 = B->last_action[3];
    r.cum_reward = B->cum_reward, r.last_reward = B->last_reward, r.last_mass = B->last_mass;
    r.fov_size_feat = B->fov_size_feat, r.stat_mass_sum = B->stat_mass_sum, r.stat_mass_max = B->stat_mass_max;
    r.stat_frames = B->stat_frames;
}
DEV void s_store(const SReg& r, const SPtr& q) {
    q.h->rng_field = r.rng_field, q.h->frame = r.frame, q.h->n_pellets = r.n_pellets, q.h->n_events = r.n_events;
    q.h->event_hash = r.event_hash;
    q.p->cmd_x = r.cmd_x, q.p->cmd_y = r.cmd_y, q.p->fov_x = r.fov_x, q.p->fov_y = r.fov_y, q.p->fov_size = r.fov_size;
    q.p->fov_valid = r.fov_valid;
    q.p->do_split = 0, q.p->do_eject = 0;
    q.c->x = r.x, q.c->y = r.y, q.c->mass = r.mass, q.c->radius = r.radius, q.c->svx = r.svx, q.c->svy = r.svy;
    q.c->merge_time = r.merge_time, q.c->counter = r.counter, q.c->flags = r.flags;
    AgarBot* B = &q.p->bot;
    B->has_action = r.has_action, B->has_last_action = r.has_last_action, B->skip_frames = r.skip_frames;
    B->has_last_mass = r.has_last_mass, B->has_old_state = r.has_old_state, B->time = r.time, B->skipping = r.skipping;
    B->turn_begun = r.turn_begun, B->need_action = r.need_action, B->exp_valid = r.exp_valid, B->exp_done = r.exp_done;
    B->cur_action[0] = r.a0, B->cur_action[1] = r.a1, B->cur_action[2] = r.a2, B->cur_action[3] = r.a3;
    B->last_action[0] = r.l0, B->last_action[1] = r.l1, B->last_action[2] = r.l2, B->last_action[3] = r.l3;
    B->cum_reward = r.cum_reward, B->last_reward = r.last_reward, B->last_mass = r.last_mass;
    B->fov_size_feat = r.fov_size_feat, B->stat_mass_sum = r.stat_mass_sum, B->stat_mass_max = r.stat_mass_max;
    B->stat_frames = r.stat_frames;
}

/* warp-uniform predicates: every data-dependent loop runs until no lane of the WARP needs another iteration.  Also
 * for W == 1 — measured: letting 32 single-lane envs leave loops independently is 4x slower (they never reconverge) */
template <int W>
DEV bool s_any(bool p) {
    return __any_sync(S_FULL, p);
}
template <int W>
DEV void s_sync() {
    __syncwarp();
}
template <int W>
DEV int tile_min(int v) {
#pragma unroll
    for (int off = W / 2; off > 0; off >>= 1) v = min(v, __shfl_xor_sync(S_FULL, v, off));
    return v;
}

/* replicated in every lane of the tile; the ring write is lane sub == 0's */
DEV void s_log(SReg& r, const SPtr& q, const DevParams& P, bool writer, int type, int a, int b, int cc, int d) {
    if (writer && r.n_events < P.L.event_cap) {
        AgarEvent* ev = &q.ev[r.n_events];
        ev->type = type, ev->a = a, ev->b = b, ev->c = cc, ev->d = d;
    }
    r.n_events += 1;
    uint64_t hh = r.event_hash;
    hh = (hh ^ (uint64_t)(uint32_t)type) * 0x100000001B3ULL;
    hh = (hh ^ (uint64_t)(uint32_t)a) * 0x100000001B3ULL;
    hh = (hh ^ (uint64_t)(uint32_t)b) * 0x100000001B3ULL;
    hh = (hh ^ (uint64_t)(uint32_t)cc) * 0x100000001B3ULL;
    hh = (hh ^ (uint64_t)(uint32_t)d) * 0x100000001B3ULL;
    r.event_hash = hh;
}
DEV int s_randint(SReg& r, const DevParams& P, uint32_t env_id, int lo, int hi) {
    uint32_t w[4];
    philox(r.rng_field, 0u, env_id, 0, (uint32_t)P.seed, (uint32_t)(P.seed >> 32), w);
    r.rng_field += 1;
    return lo + (int)(((unsigned long long)w[0] * (unsigned long long)(hi - lo)) >> 32);
}
/* Player.getFovPos / getFovSize for one cell (player.py:156-167); numpy.sum of one element is 0.0 + v */
DEV void s_update_fov(SReg& r, const DevParams& P) {
    double tm = 0.0 + r.mass;
    if (tm != 0) {
        r.fov_x = (0.0 + r.x * r.mass) / tm;
        r.fov_y = (0.0 + r.y * r.mass) / tm;
        r.fov_valid = 1;
    }
    r.fov_size = agar_pow(r.radius, 0.475) * P.pow_n[1] * 35;
}
/* The two pow() of a frame — fov size (radius ^ 0.475, player.py:163-167) and speed (mass' ^ -0.35 with the mass as
 * it will be after this frame's decay, cell.py:123-126,246-248) — have independent inputs.  With W >= 2 lanes per env
 * the even lanes evaluate one and the odd lanes the other in the SAME instruction stream, then swap: one pow per
 * frame instead of two (same function, same inputs: bit-identical results). */
template <int W>
DEV void s_dual_pow(double x0, double y0, double x1, double y1, int sub, double& p0, double& p1) {
    if (W == 1) {
        p0 = agar_pow(x0, y0);
        p1 = agar_pow(x1, y1);
        return;
    }
    const bool odd = (sub & 1) != 0;
    const double mine = agar_pow(odd ? x1 : x0, odd ? y1 : y0);
    const double other = __shfl_xor_sync(S_FULL, mine, 1);
    p0 = odd ? other : mine;
    p1 = odd ? mine : other;
}
/* a / b and c / d for the price of one division: even lanes divide one pair, odd lanes the other, then they swap */
template <int W>
DEV void s_dual_div(double a, double b, double c, double d, int sub, double& q0, double& q1) {
    if (W == 1) {
        q0 = a / b;
        q1 = c / d;
        return;
    }
    const bool odd = (sub & 1) != 0;
    const double mine = (odd ? c : a) / (odd ? d : b);
    const double other = __shfl_xor_sync(S_FULL, mine, 1);
    q0 = odd ? other : mine;
    q1 = odd ? mine : other;
}
/* bot.py:550-577 + the speed factor of the coming frame */
template <int W>
DEV void s_set_command_point(SReg& r, const DevParams& P, double a0, double a1, int sub, double& speed_pow) {
    double tm = 0.0 + r.mass; /* s_update_fov, with the pow and the divisions shared across the lane pair */
    {
        double fx, fy;
        s_dual_div<W>(0.0 + r.x * r.mass, tm, 0.0 + r.y * r.mass, tm, sub, fx, fy);
        if (tm != 0) {
            r.fov_x = fx;
            r.fov_y = fy;
            r.fov_valid = 1;
        }
    }
    const double mass_next = r.mass >= 4 ? r.mass * P.decay_rate : r.mass;
    double fov_pow;
    s_dual_pow<W>(r.radius, 0.475, mass_next, -0.35, sub, fov_pow, speed_pow);
    r.fov_size = fov_pow * P.pow_n[1] * 35;
    int x = (int)r.fov_x, y = (int)r.fov_y;
    int left = x - (int)(r.fov_size / 2), top = y - (int)(r.fov_size / 2);
    int size = (int)r.fov_size;
    r.cmd_x = left + a0 * size;
    r.cmd_y = top + a1 * size;
}

/* Candidate masks of the two pellet loops (observation, eating): bit j of word 0 / word 1 <-> slot sub + W * j / sub + W * (MB + j).
 * Tiles of >= 4 lanes hold at most 64 slots per lane (agar_set_tile_width checks pellet_cap <= 64 W) and keep 32-bit words — the
 * 64-bit shifts / find-first-set of the wide form were 9 % of k_simple<8>'s instructions; 1- and 2-lane tiles keep 64-bit words. */
template <int W>
struct SMask {
    typedef uint32_t T;
    static constexpr int MB = 32;
};
template <>
struct SMask<1> {
    typedef unsigned long long T;
    static constexpr int MB = 64;
};
template <>
struct SMask<2> {
    typedef unsigned long long T;
    static constexpr int MB = 64;
};
DEV int s_ffs(uint32_t m) { return __ffs((int)m); }
DEV int s_ffs(unsigned long long m) { return __ffsll((long long)m); }

/* The state change of an observation (player.py:156-167, bot.py:326): the fov caches advance; s_encode reads them. */
DEV void s_observe_state(SReg& r, const DevParams& P) {
    s_update_fov(r, P);
    r.fov_size_feat = P.cfg.use_fovsize ? r.fov_size : r.fov_size_feat;
}

/* bot.py:326-497 for the pellet channel: bins q.pel into row.  Reads r.fov_x, r.fov_y, r.fov_size and r.mass only, and
 * writes nothing but q.grid and row — so it can run on a snapshot of the pool and of those four values (observer warps,
 * k_simple).  Warp-uniform: every lane calls it; out = this tile stores a row. */
template <int W>
DEV void s_encode(const SReg& r, const SPtr& q, const DevParams& P, bool out, float* row, int sub) {
    const int G = P.L.grid_squares, GG = G * G, SL = P.L.state_len;
    const double S = (double)P.S;
    if (!s_any<W>(out)) return;
    const bool staged = q.grid != nullptr;
    if (out) { /* clear the row; extras: [fov size], [total mass] (bot.py:302-323) */
        if (staged)
            for (int i = sub; i < GG; i += W) q.grid[i] = 0u;
        else
            for (int i = sub; i < GG; i += W) row[i] = 0.f;
        if (sub == 0) {
            int n = GG;
            if (P.cfg.use_fovsize) row[n++] = (float)r.fov_size;
            if (P.cfg.use_totalmass) row[n++] = (float)(0.0 + r.mass);
            (void)SL;
        }
    }
    s_sync<W>(); /* orders the clearing stores before the REDs below (same warp) */
    if (out) {
        const double fov = r.fov_size, fx = r.fov_x, fy = r.fov_y;
        const double left = fx - fov / 2, top = fy - fov / 2;
        const double gs = fov / G, inv = 1.0 / gs;
        const bool canon = P.cfg.obs_mode == AGAR_OBS_CANONICAL;
        const int cols = canon ? G : (int)ceil(fov / gs);
        /* squares entirely outside the field show nothing (bot.py:392-393); mid points accumulate like the reference */
        double mx = left + gs / 2, my = top + gs / 2;
        unsigned col_bad = 0, row_bad = 0;
        for (int i = 0; i < G; ++i) {
            if (mx + gs / 2 < 0 || mx - gs / 2 > S) col_bad |= 1u << i;
            if (my + gs / 2 < 0 || my - gs / 2 > S) row_bad |= 1u << i;
            mx += gs;
            my += gs;
        }
        const Rect ra = rect_of(P.S, fx, fy, fov / 2);
        const double h = fov / 2;
        const double xmin = fx - h, xmax = fx + h, ymin = fy - h, ymax = fy + h;
        /* integer window that contains every pellet in_fov() can accept (radius < 1) */
        const int wx0 = (int)floor(xmin) - 1, wx1 = (int)ceil(xmax) + 1, wy0 = (int)floor(ymin) - 1, wy1 = (int)ceil(ymax) + 1;
        /* phase 1: integer window -> candidate bitmask over this lane's slots (converged, cheap) */
        typedef typename SMask<W>::T MT;
        constexpr int MB = SMask<W>::MB;
        MT m0 = 0, m1 = 0;
        {
            const int cap = P.L.pellet_cap, split = min(cap, sub + MB * W);
            int j = 0;
            for (int s = sub; s < split; s += W, ++j) { /* branch-free accumulation, two plain loops */
                uint32_t pk = q.pel[s];
                int px = AGAR_PELLET_X(pk), py = AGAR_PELLET_Y(pk);
                bool in = px >= wx0 && px <= wx1 && py >= wy0 && py <= wy1 && pk != 0;
                m0 |= (MT)in << j;
            }
            j = 0;
            for (int s = sub + MB * W; s < cap; s += W, ++j) {
                uint32_t pk = q.pel[s];
                int px = AGAR_PELLET_X(pk), py = AGAR_PELLET_Y(pk);
                bool in = px >= wx0 && px <= wx1 && py >= wy0 && py <= wy1 && pk != 0;
                m1 |= (MT)in << j;
            }
        }
        /* phase 2: every lane bins its own next candidate per iteration.  The body is straight-line (predicated REDs,
         * two-bucket axis form), so the lanes of a warp stay converged until the longest list ends. */
        const bool sheared = cols != G;
        const bool use_bits = W <= 2 && !canon && G <= 15; /* 2 (G + 1) edge evaluations per observation instead of 4 per pellet */
        const unsigned edges = use_bits ? edge_bits(gs, inv, G) : 0u;
        while (m0 | m1) {
            int j;
            if (m0) {
                j = s_ffs(m0) - 1;
                m0 &= m0 - 1;
            } else {
                j = MB + s_ffs(m1) - 1;
                m1 &= m1 - 1;
            }
            uint32_t pk = q.pel[sub + W * j];
            int px = AGAR_PELLET_X(pk), py = AGAR_PELLET_Y(pk), pm = AGAR_PELLET_M(pk);
            double pr = P.pellet_r[pm & 3];
            double dx = (double)px, dy = (double)py;
            bool ok = rect_hit(ra, pellet_rect(px, py)) && !(dx + pr < xmin || dx - pr > xmax || dy + pr < ymin || dy - pr > ymax);
            int c0, c1, r0, r1;
            if (use_bits) {
                axis_buckets2_bits(dx - left, pr, fov, gs, inv, edges, c0, c1);
                axis_buckets2_bits(dy - top, pr, fov, gs, inv, edges, r0, r1);
            } else {
                axis_buckets2(dx - left, pr, fov, gs, inv, canon, c0, c1);
                axis_buckets2(dy - top, pr, fov, gs, inv, canon, r0, r1);
            }
            float fm = (float)pm;
            auto put = [&](int cc, int rr) {
                /* bucket id = cc + rr * cols is read by square (id / G, id % G).  cols == G: that is (rr, cc); cols == G + 1
                 * (the reference's shear): id = (cc + rr) + rr * G — no integer division either way */
                int sr = sheared ? cc + rr : cc, sc = rr;
                if (sr >= G) sr -= G, sc += 1;
                int id = sr + sc * G;
                if (ok && cc >= 0 && rr >= 0 && sc < G && !((row_bad >> sc & 1) || (col_bad >> sr & 1))) {
                    if (staged)
                        atomicAdd(&q.grid[id], (unsigned)pm); /* pellet masses are small integers: the float sum is this integer, in any order */
                    else
                        atomicAdd(&row[id], fm);
                }
            };
            put(c0, r0);
            put(c1, r0);
            put(c0, r1);
            put(c1, r1);
        }
    }
    if (staged) { /* the finished grid leaves shared memory once, as consecutive floats of the env's row */
        s_sync<W>();
        if (out)
            for (int i = sub; i < GG; i += W) row[i] = (float)q.grid[i];
    }
}

/* Warp-uniform: every lane calls it; `mine` = this tile observes now.  row: this env's observation row in the caller's
 * buffer (nullptr: a decision inside a multi-frame step, nobody reads the grid — only the fov caches advance, as in the
 * reference). */
template <int W>
DEV void s_observe(SReg& r, const SPtr& q, const DevParams& P, bool mine, float* row, int sub) {
    if (mine) s_observe_state(r, P);
    s_encode<W>(r, q, P, mine && row != nullptr, row, sub);
}

/* one frame of Field.update for a single-cell env (field.py:85-92); warp-uniform, state replicated per tile */
template <int W>
DEV void s_field_update(SReg& r, const SPtr& q, const DevParams& P, uint32_t env_id, int sub, double speed_pow) {
    const double S = (double)P.S;
    /* Player.update (player.py:30-36) */
    double mass = r.mass, radius = r.radius;
    if (mass >= 4) {
        mass = mass * P.decay_rate;
        radius = radius_of(mass);
    }
    update_momentum(r.svx, r.svy, r.counter);
    if (r.merge_time > 0) r.merge_time = r.merge_time - 1;
    double xd = r.cmd_x - r.x, yd = r.cmd_y - r.y;
    double h2 = xd * xd + yd * yd, r2 = radius * radius;
    double sm = (h2 < r2 ? h2 : r2) / r2;
    double cs, sn;
    agar_dir(yd, xd, &cs, &sn); /* cell.py:49-57: cos / sin of the ROUNDED angle atan2 returns, bit-identical to libm */
    double rs = P.move_speed * speed_pow; /* = agar_pow(mass, -0.35), evaluated next to the fov pow in s_turn_end */
    double vx = rs * sm * cs, vy = rs * sm * sn;
    update_pos(r.x, r.y, vx, vy, r.svx, r.svy, r.counter, S);
    r.flags |= AGAR_CF_INHASH;
    /* playerPelletOverlap (field.py:207-213): slot order, the cell grows as it eats.
     * Phase 1: candidate filter around the cell -> bitmask over this lane's slots. */
    /* The candidate rectangle is fixed before the cell grows (field.py:207).  While the cell has not grown this frame the
     * rectangle test is implied by the eat test — overlap with the cell as the bigger one puts the pellet's integer centre
     * strictly inside (x - r, x + r), i.e. inside the coordinates [bucket_left, limit - 1] the cell's buckets cover
     * (axis_range), and the pellet's own bucket px / 20 is one of its rectangle's — so it is only evaluated, from the
     * pre-growth radius, for pellets met after the first one eaten in the frame. */
    const double radius0 = radius;
    const double cx = r.x, cy = r.y;
    const int cap = P.L.pellet_cap;
    /* Candidate filter.  Tiles of <= 2 lanes (one conversion pipe for many slots per lane: the float form below costs 15 % at
     * one lane per env): the integer window |p - floor(c)| <= (int)r + 1 per axis — a pellet that passes the eat test has
     * d^2 * 1.1 < r^2, so |px - cx| <= d < 0.954 r and |px - icx| < 0.954 r + 1, an integer: <= (int)r + 1; the bound depends on
     * (int)r only, so the masks stay valid while the cell grows inside the same integer radius.
     * Tiles of >= 4 lanes: the eat test itself in float32 with slack.  The exact test needs d^2 <= 0.90910 r^2; the float32
     * distance (px - (float)cx)^2 + (py - (float)cy)^2 differs from d^2 by less than 3e-3 for coordinates below 128 and d < 110
     * (|dx| is off by <= 6e-6, three roundings of 2^-24), so "d2f <= 0.9101 (float)(r^2) + 0.1" admits every pellet the exact test
     * can accept and almost nothing else (the window admits 0.9-1.8 candidates per env and frame, each one more trip of the
     * ordered loop).  That bound follows the radius: the slots after an eaten pellet are always re-scanned. */
    constexpr bool DISC = W >= 4;
    const int icx = (int)cx, icy = (int)cy;
    int reach = (int)radius + 1;
    const float cxf = (float)cx, cyf = (float)cy;
    float thr = 0.9101f * (float)(radius * radius) + 0.1f;
    /* When the pool is full (the steady state: cap == refill target) the free slots after eating are exactly the
     * eaten ones, in ascending order — remember up to four and skip the free-slot search when respawning. */
    const bool pool_full = r.n_pellets == cap;
    int eaten0 = S_NONE, eaten1 = S_NONE, eaten2 = S_NONE, eaten3 = S_NONE, n_eaten = 0;
    typedef typename SMask<W>::T MT;
    constexpr int MB = SMask<W>::MB;
    MT m0 = 0, m1 = 0; /* bit j <-> slot sub + W * j (m0), sub + W * (MB + j) (m1) */
    auto scan = [&](int first_slot) {
        m0 = m1 = 0;
        const int split = min(cap, sub + MB * W);
        const unsigned r2 = (unsigned)(2 * reach);
        auto test = [&](uint32_t pk, int s) {
            if (DISC) {
                const float dx = (float)AGAR_PELLET_X(pk) - cxf, dy = (float)AGAR_PELLET_Y(pk) - cyf;
                return dx * dx + dy * dy <= thr && pk != 0 && s >= first_slot;
            }
            const int px = AGAR_PELLET_X(pk), py = AGAR_PELLET_Y(pk);
            return (unsigned)(px - icx + reach) <= r2 && (unsigned)(py - icy + reach) <= r2 && pk != 0 && s >= first_slot;
        };
        int j = 0;
        for (int s = sub; s < split; s += W, ++j) m0 |= (MT)test(q.pel[s], s) << j; /* branch-free accumulation, two plain loops */
        j = 0;
        for (int s = sub + MB * W; s < cap; s += W, ++j) m1 |= (MT)test(q.pel[s], s) << j;
    };
    scan(0);
    while (s_any<W>((m0 | m1) != 0)) { /* one vote decides the (usual) frame without candidates: no find-first-set, no tile minimum */
        int mine = m0 ? sub + W * (s_ffs(m0) - 1) : (m1 ? sub + W * (MB + s_ffs(m1) - 1) : S_NONE);
        int first = tile_min<W>(mine);
        if (first != S_NONE && mine == first) { /* owner lane drops the candidate */
            int j = (first - sub) / W;
            if (j < MB)
                m0 &= ~((MT)1 << j);
            else
                m1 &= ~((MT)1 << (j - MB));
        }
        const uint32_t pk = q.pel[first != S_NONE ? first : 0];
        s_sync<W>(); /* every lane has read its tile's candidate before lane sub == 0 may clear the slot */
        if (first != S_NONE) {
            int px = AGAR_PELLET_X(pk), py = AGAR_PELLET_Y(pk), pm = AGAR_PELLET_M(pk);
            if (overlap(cx, cy, mass, radius, (double)px, (double)py, (double)pm, P.pellet_r[pm & 3]) && mass > 1.25 * (double)pm &&
                (n_eaten == 0 || rect_hit(rect_of(P.S, cx, cy, radius0), pellet_rect(px, py)))) {
                s_log(r, q, P, sub == 0, AGAR_EV_EAT_PELLET, 0, (int)r.uid, first, 0);
                double nm = mass + (double)pm;
                if (!(nm < AG_MAX_MASS)) nm = AG_MAX_MASS;
                mass = nm;
                radius = radius_of(nm);
                if (sub == 0) q.pel[first] = 0;
                r.n_pellets -= 1;
                if (n_eaten == 0) eaten0 = first;
                else if (n_eaten == 1) eaten1 = first;
                else if (n_eaten == 2) eaten2 = first;
                else if (n_eaten == 3) eaten3 = first;
                n_eaten += 1;
                if (DISC) { /* the grown cell reaches farther: re-scan the slots after this one */
                    thr = 0.9101f * (float)(radius * radius) + 0.1f;
                    scan(first + 1);
                } else if ((int)radius + 1 > reach) {
                    reach = (int)radius + 1;
                    scan(first + 1);
                }
            }
        }
    }
    r.mass = mass, r.radius = radius;
    s_sync<W>(); /* eaten slots are visible to the tile before the free-slot search */
    /* spawnPellets (field.py:303-313) */
    int from = 0;
    while (s_any<W>((double)r.n_pellets < P.L.max_pellets)) {
        const bool need = (double)r.n_pellets < P.L.max_pellets;
        int mine = S_NONE;
        const bool known = pool_full && n_eaten <= 4;
        if (need && known) {
            mine = eaten0; /* the lowest free slot is the earliest eaten one */
            eaten0 = eaten1, eaten1 = eaten2, eaten2 = eaten3, eaten3 = S_NONE;
        } else if (need) {
            int s = from + ((sub - from) % W + W) % W; /* first slot >= from owned by this lane */
            for (; s < cap; s += W)
                if (q.pel[s] == 0) {
                    mine = s;
                    break;
                }
        }
        int slot = tile_min<W>(mine);
        if (need) {
            if (slot == S_NONE) {
                r.n_pellets = (int)P.L.max_pellets + 1; /* cannot happen: n_pellets < max <= cap */
            } else {
                int x = s_randint(r, P, env_id, 0, P.S), y = s_randint(r, P, env_id, 0, P.S);
                int v = s_randint(r, P, env_id, 0, 50);
                int m = v > 46 ? 50 - v : 1;
                s_log(r, q, P, sub == 0, AGAR_EV_SPAWN_PELLET, slot, x, y, m);
                if (sub == 0) q.pel[slot] = AGAR_PELLET_PACK(x, y, m);
                r.n_pellets += 1;
                from = slot + 1;
            }
        }
        s_sync<W>();
    }
    r.frame += 1;
}

/* first half of move_NN (bot.py:195-217).  Returns 1 if this env observes now. */
DEV int s_turn_begin(SReg& r, const DevParams& P) {
    int do_obs = 0;
    if (!r.turn_begun) {
        double tm = 0.0 + r.mass;
        r.stat_mass_sum += tm;
        if (tm > r.stat_mass_max) r.stat_mass_max = tm;
        r.stat_frames += 1;
        r.skipping = 0;
        r.need_action = r.exp_valid = r.exp_done = 0;
        if (r.has_action) {
            if (r.has_last_mass && r.last_mass != 0) {
                double rew = P.cfg.mass_as_reward ? tm - P.cfg.reward_term : (tm - r.last_mass) * P.cfg.reward_scale - P.cfg.reward_term;
                r.cum_reward += rew;
            }
            r.last_reward = r.cum_reward;
            if (r.skip_frames > 0) {
                r.skip_frames -= 1;
                r.skipping = 1;
            }
        }
        if (!r.skipping) {
            if (r.has_old_state) {
                r.time += 1;
                r.exp_valid = 1;
            }
            r.need_action = 1;
            do_obs = 1;
        }
        r.turn_begun = 1;
    }
    return do_obs;
}
/* second half of move_NN + tail of makeMove (bot.py:223-232,256-270) */
template <int W>
DEV void s_turn_end(SReg& r, const DevParams& P, const float* act, int sub, double& speed_pow) {
    if (r.need_action) {
        r.cum_reward = 0;
        r.skip_frames = P.cfg.frame_skip;
        r.has_old_state = 1;
        r.l0 = r.a0, r.l1 = r.a1, r.l2 = r.a2, r.l3 = r.a3;
        r.has_last_action = r.has_action;
        r.a0 = (double)act[0], r.a1 = (double)act[1], r.a2 = 0.0, r.a3 = 0.0; /* action_len == 2 */
        r.has_action = 1;
    }
    if (!r.skipping) {
        r.last_mass = 0.0 + r.mass;
        r.has_last_mass = 1;
    }
    r.turn_begun = 0;
    s_set_command_point<W>(r, P, r.a0, r.a1, sub, speed_pow);
}
