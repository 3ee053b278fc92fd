/*
 * agar_dev.cuh — device side of the B200-native batched agar.io step.
 *
 * Execution model: one env per TILE of W lanes (W = 1..32, a cooperative-groups tile of a warp).  The env
 * record (include/agar_b200.h) is staged from HBM into shared memory by the whole CTA with coalesced 16-byte
 * accesses, stepped there for every frame of the launch, and written back once.  Inside a tile, lane 0 is
 * the "scalar processor" that executes the order-dependent parts of the reference exactly as a sequential
 * program (SEQ sections); the other lanes are the vector assist for the O(pool) loops: the pellet overlap
 * scan (ballot + ordered eat chain), free-slot search, field-of-view binning, candidate pre-checks.
 *
 * All fp64 arithmetic is IEEE basic operations + include/agar_math.h, compiled with -fmad=false, so that
 * the state is BIT-IDENTICAL to oracle/agar_oracle.c built with -DAGAR_PORTABLE_MATH.
 *
 * Every function cites the reference lines it replaces (paths relative to /root/reference/src/model/).
 */
#pragma once
#include <cooperative_groups.h>
#include <cooperative_groups/reduce.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/agar_b200.h"
#include "../../include/agar_math.h"

namespace cg = cooperative_groups;

#define DEV __device__ __forceinline__
#define DEVN __device__ __noinline__

#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif

/* parameters.py:10-35 */
#define AG_BUCKET 20
#define AG_MAX_MASS 22500.0

struct DevParams {
    AgarConfig cfg;
    AgarLayout L;
    int S, nb, n_envs, rec_stride; /* rec_stride: bytes between staged records in shared memory */
    int scratch_bytes, full;
    double move_speed, decay_rate, blob_mass, virus_split_mass, start_radius, virus_radius;
    double pellet_r[4];
    double pow_n[17];
    const double* deg_tab; /* cos(d*pi/180)[360], sin(...)[360] — host libm, exactly the oracle's table */
    uint64_t seed, first_env;
    int pel_index; /* 1: multi-agent configs with a large pellet pool build the per-env bucket index every frame (agar_dev.cuh) */
    int hot_a, live_off; /* live_off: offset of the live-cell list in a tile's scratch (multi-agent configs) */ /* hot_a: 0 or off_blobs; FULL kernels cache bytes [0, hot_a) of a record (header, players, cells, viruses) in shared memory too */
    /* optional per-launch outputs of the last bot turn ([E][A]); NULL = use agar_get */
    float* turn_reward;
    uint8_t* turn_done;
    int cap_shift;               /* cell_cap is 1 or 16 (agar_layout.h): slot index -> (player, cell) by shift and mask           */
    uint32_t g_magic;            /* floor(2^32 / G) + 1: idx / G == __umulhi(idx, g_magic) for idx < 2^16, G >= 2 (checked at create) */
    /* agar_step_host with pinned caller buffers: every CTA of the step launch exports its own envs' rows over PCIe as soon as
     * it has finished them (export_tail below); the last CTA raises a flag in host memory the caller polls */
    float* host_obs;             /* device-visible address of the caller's pinned observation buffer, or NULL           */
    uint32_t* host_turn;         /* device-visible address of the pinned packed block: float reward[EA] | uint8 done[EA] */
    unsigned int* export_count;  /* device counter of CTAs that have exported                                          */
    volatile uint32_t* host_flag;
    uint32_t flag_value;
};

/* flags of k_main */
enum { KF_OBS_BEFORE = 1, KF_OBS_AFTER = 2, KF_RANDOM_ACTIONS = 4 };

template <int W>
struct Ctx {
    cg::thread_block_tile<W> t;
    int lane;
    uint32_t env_id; /* global env id: Philox counter word 2 */
    uint8_t* rec;
    AgarEnvHeader* h;
    AgarPlayer* pl;
    AgarCell* cells;
    AgarMote* vir;
    AgarMote* blob;
    AgarFatPellet* fat;
    uint32_t* pel;
    float* hist;
    AgarEvent* ev;
    uint8_t* scratch;
#ifdef AGAR_PHASE_CLOCKS
    long long clk_t;
    int clk_env;
#endif
    bool fov_done; /* this frame's fields of view were computed up front for every player (update_all_fovs) */
    int n_live;    /* >= 0: live_cells() lists the (player * cell_cap + cell) indices of all live cells, canonical order */
    __device__ Ctx(cg::thread_block_tile<W> tile) : t(tile), fov_done(false), n_live(-1) {}
};

#ifdef AGAR_PHASE_CLOCKS
__device__ unsigned long long g_clk[32768 * 16];
template <int W>
__device__ __forceinline__ void clk_mark(Ctx<W>& c, int slot) {
    if (c.lane == 0 && c.clk_env < 32768) {
        const long long now = clock64();
        g_clk[(size_t)c.clk_env * 16 + slot] += (unsigned long long)(now - c.clk_t);
        c.clk_t = now;
    }
}
#define CLK_IN(c, slot) clk_mark(c, slot)
#else
#define CLK_IN(c, slot) do { } while (0)
#endif

#define CELLP(c, P, k, i) (&(c).cells[(k) * (P).L.cell_cap + (i)])

/* Tail of a step launch issued by agar_step_host (every thread of the CTA calls it): the observation rows and the reward /
 * done words of this CTA's envs [env0, env0 + n_here) go from the device staging buffers (just written by this CTA's own
 * threads; read back through L2, where the observation REDs landed) to the caller's pinned buffers with 16-byte stores.
 * No second kernel, no grid-wide wait: a CTA's rows leave while other CTAs still step.  __threadfence_system orders the
 * PCIe writes before the CTA's count; the CTA that counts last writes the flag the host polls. */
__device__ __forceinline__ void export_tail(const DevParams& P, const float* obs_dev, int env0, int n_here) {
    if (!P.host_turn) return;
    __syncthreads();
    const int A = P.L.n_agents > 0 ? P.L.n_agents : 1;
    const size_t tid = threadIdx.x, nt = blockDim.x;
    if (P.host_obs && obs_dev) {
        const size_t w0 = (size_t)env0 * A * P.L.state_len, w1 = w0 + (size_t)n_here * A * P.L.state_len; /* float indices */
        size_t a0 = (w0 + 3) & ~(size_t)3;
        if (a0 > w1) a0 = w1;
        const size_t a1 = a0 + ((w1 - a0) & ~(size_t)3);
        for (size_t i = w0 + tid; i < a0; i += nt) P.host_obs[i] = __ldcg(obs_dev + i);
        for (size_t i = a0 / 4 + tid; i < a1 / 4; i += nt) ((uint4*)P.host_obs)[i] = __ldcg((const uint4*)obs_dev + i);
        for (size_t i = a1 + tid; i < w1; i += nt) P.host_obs[i] = __ldcg(obs_dev + i);
    }
    {
        const size_t EA = (size_t)P.n_envs * A, t0 = (size_t)env0 * A, t1 = t0 + (size_t)n_here * A;
        float* hr = (float*)P.host_turn;
        uint8_t* hd = (uint8_t*)P.host_turn + EA * 4;
        for (size_t i = t0 + tid; i < t1; i += nt) {
            hr[i] = __ldcg(P.turn_reward + i);
            hd[i] = __ldcg(P.turn_done + i);
        }
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int c = atomicAdd(P.export_count, 1u);
        if (c == gridDim.x - 1) {
            *P.export_count = 0; /* every other CTA has counted: ready for the next launch */
            __threadfence_system();
            *P.host_flag = P.flag_value;
        }
    }
}

/* ------------------------------------------------------------------ small exact helpers */
DEV double py_max0(double v) { return v > 0 ? v : 0.0; }
DEV double py_minS(double S, double v) { return v < S ? v : S; }
DEV double clampS(double v, double S) { return py_minS(S, py_max0(v)); }
DEV double radius_of(double m) { return m > 0 ? sqrt(m / M_PI) : 0.0; } /* cell.py:210-212 */

struct Rect {
    int x0, x1, y0, y1;
};
/* spatialHashTable.py:70-83 getIdsForArea, one axis */
DEV void axis_range(double p, double radius, int S, int& b0, int& b1) {
    double cl = py_max0(p - radius);
    /* int(cl - cl % 20) == 20 * floor(cl / 20) exactly (fmod is exact); in integers: floor(floor(cl) / 20) */
    int bucket_left = ((int)cl / AG_BUCKET) * AG_BUCKET;
    int limit = (int)py_minS((double)S, p + radius + 1);
    b0 = bucket_left / AG_BUCKET;
    b1 = limit > bucket_left ? b0 + (limit - bucket_left - 1) / AG_BUCKET : b0 - 1;
}
DEV Rect rect_of(int S, double x, double y, double r) {
    Rect q;
    axis_range(x, r, S, q.x0, q.x1);
    axis_range(y, r, S, q.y0, q.y1);
    return q;
}
DEV bool rect_hit(const Rect& a, const Rect& b) {
    if (a.x1 < a.x0 || a.y1 < a.y0 || b.x1 < b.x0 || b.y1 < b.y0) return false;
    return a.x0 <= b.x1 && b.x0 <= a.x1 && a.y0 <= b.y1 && b.y0 <= a.y1;
}
/* integer pellet at (px, py), radius < 1: its hash rectangle in closed form (tests/test_layout.py proves it
 * equal to axis_range for every coordinate and mass) */
DEV Rect pellet_rect(int px, int py) {
    Rect q;
    q.x0 = (px > 0 ? px - 1 : 0) / AG_BUCKET, q.x1 = px / AG_BUCKET;
    q.y0 = (py > 0 ? py - 1 : 0) / AG_BUCKET, q.y1 = py / AG_BUCKET;
    return q;
}
/* cell.py:143-152 */
DEV bool overlap(double ax, double ay, double am, double ar, double bx, double by, double bm, double br) {
    double bigx, bigy, bigr, smx, smy;
    if (am > bm)
        bigx = ax, bigy = ay, bigr = ar, smx = bx, smy = by;
    else
        bigx = bx, bigy = by, bigr = br, smx = ax, smy = ay;
    double d2 = (bigx - smx) * (bigx - smx) + (bigy - smy) * (bigy - smy);
    return d2 * 1.1 < bigr * bigr;
}
DEV bool in_fov(double x, double y, double r, double fx, double fy, double fov) { /* cell.py:169-177 */
    double h = fov / 2;
    double xmin = fx - h, xmax = fx + h, ymin = fy - h, ymax = fy + h;
    return !(x + r < xmin || x - r > xmax || y + r < ymin || y - r > ymax);
}
DEV void grow(AgarCell* c, double food) { /* cell.py:119-121 */
    double nm = c->mass + food;
    if (!(nm < AG_MAX_MASS)) nm = AG_MAX_MASS;
    c->mass = nm;
    c->radius = radius_of(nm);
}
DEV void grow_mote(AgarMote* c, double food) {
    double nm = c->mass + food;
    if (!(nm < AG_MAX_MASS)) nm = AG_MAX_MASS;
    c->mass = nm;
    c->radius = radius_of(nm);
}
DEV double merge_time_for(double factor, double mass) { /* cell.py:154-155 */
    return factor * (25 + mass * 0.0233) * 30 / 2 / 1;
}

/* Out-of-line leaves for the multi-agent kernel.  Its frame body is ~13 000 hot SASS instructions (~200 KB, more than the SM's
 * instruction cache: `stall_no_inst` was 20 % of the samples of the steady-state arena profile) and these three were inlined at
 * 15 / 29 / 20+ places.  Scalar arguments and results only: nothing is forced into local memory at the call. */
DEVN double radius_of_call(double m) { return radius_of(m); }
DEVN uint32_t rect_of_packed(int S, double x, double y, double r) { /* bucket indices are -1 .. 52: one byte each, biased by 1 */
    const Rect q = rect_of(S, x, y, r);
    return (uint32_t)(q.x0 + 1) | (uint32_t)(q.x1 + 1) << 8 | (uint32_t)(q.y0 + 1) << 16 | (uint32_t)(q.y1 + 1) << 24;
}
DEV Rect rect_of_call(int S, double x, double y, double r) {
    const uint32_t w = rect_of_packed(S, x, y, r);
    Rect q;
    q.x0 = (int)(w & 0xffu) - 1, q.x1 = (int)(w >> 8 & 0xffu) - 1, q.y0 = (int)(w >> 16 & 0xffu) - 1, q.y1 = (int)(w >> 24) - 1;
    return q;
}
/* numpy pairwise summation order for n <= 16 (oracle np_sum) */
template <class F>
DEV double np_sum(F get, int n) {
    if (n < 8) {
        double r = 0.0;
        for (int i = 0; i < n; ++i) r += get(i);
        return r;
    }
    double r0 = get(0), r1 = get(1), r2 = get(2), r3 = get(3), r4 = get(4), r5 = get(5), r6 = get(6), r7 = get(7);
    int i = 8;
    if (n == 16) {
        r0 += get(8), r1 += get(9), r2 += get(10), r3 += get(11), r4 += get(12), r5 += get(13), r6 += get(14),
            r7 += get(15);
        i = 16;
    }
    double res = ((r0 + r1) + (r2 + r3)) + ((r4 + r5) + (r6 + r7));
    for (; i < n; ++i) res += get(i);
    return res;
}

/* the three sums over a player's cells (total mass, mass-weighted x / y: player.py:129-161), out of line — see above */
DEVN double cells_np_sum(const AgarCell* base, int n, int what) {
    if (what == 0) return np_sum([&](int i) { return base[i].mass; }, n);
    if (what == 1) return np_sum([&](int i) { return base[i].x * base[i].mass; }, n);
    return np_sum([&](int i) { return base[i].y * base[i].mass; }, n);
}

/* ------------------------------------------------------------------ Philox4x32-10 (oracle/philox.py) */
DEV void philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t out[4]) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0, c1 = n1, c2 = n2, c3 = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0, out[1] = c1, out[2] = c2, out[3] = c3;
}
/* the draw_* functions are called by lane 0 only (they advance the serial in the record) */
template <int W>
DEV void draw_words(Ctx<W>& c, const DevParams& P, int stream, uint32_t out[4]) {
    uint32_t* serial = stream == 0 ? &c.h->rng_field : &c.h->rng_bot;
    philox(*serial, (uint32_t)stream, c.env_id, 0, (uint32_t)P.seed, (uint32_t)(P.seed >> 32), out);
    *serial += 1;
}
template <int W>
DEV int draw_randint(Ctx<W>& c, const DevParams& P, int stream, double lo, double hi) {
    long long l = (long long)lo, h = (long long)hi; /* numpy truncates float bounds toward zero */
    uint32_t w[4];
    draw_words(c, P, stream, w);
    return (int)(l + (long long)(((unsigned long long)w[0] * (unsigned long long)(h - l)) >> 32));
}
template <int W>
DEV double draw_random(Ctx<W>& c, const DevParams& P, int stream) {
    uint32_t w[4];
    draw_words(c, P, stream, w);
    return ((double)(w[0] >> 5) * 67108864.0 + (double)(w[1] >> 6)) / 9007199254740992.0;
}

/* lane 0 only */
template <int W>
DEV void log_ev(Ctx<W>& c, const DevParams& P, int type, int a, int b, int cc, int d) {
    int n = c.h->n_events;
    if (n < P.L.event_cap) {
        AgarEvent* ev = &c.ev[n];
        ev->type = type, ev->a = a, ev->b = b, ev->c = cc, ev->d = d;
    }
    c.h->n_events = n + 1;
    if (type == AGAR_EV_COLLIDE) return; /* logged, not hashed (see oracle log_ev) */
    uint64_t hh = c.h->event_hash;
    hh = (hh ^ (uint64_t)(uint32_t)type) * 0x100000001B3ULL;
    hh = (hh ^ (uint64_t)(uint32_t)a) * 0x100000001B3ULL;
    hh = (hh ^ (uint64_t)(uint32_t)b) * 0x100000001B3ULL;
    hh = (hh ^ (uint64_t)(uint32_t)cc) * 0x100000001B3ULL;
    hh = (hh ^ (uint64_t)(uint32_t)d) * 0x100000001B3ULL;
    c.h->event_hash = hh;
}

/* ------------------------------------------------------------------ player helpers (player.py:129-167); any lane */
template <int W>
DEV double total_mass(const Ctx<W>& c, const DevParams& P, int k) {
    int n = c.pl[k].n_cells;
    if (n == 0) return 0.0;
    const AgarCell* base = CELLP(c, P, k, 0);
    return cells_np_sum(base, n, 0);
}
/* lane 0: getFovPos + getFovSize, caches in the player */
template <int W>
DEV void update_fov(Ctx<W>& c, const DevParams& P, int k) {
    AgarPlayer* p = &c.pl[k];
    if (!p->alive) return;
    int n = p->n_cells;
    const AgarCell* base = CELLP(c, P, k, 0);
    double tm = total_mass(c, P, k);
    if (tm != 0) {
        p->fov_x = cells_np_sum(base, n, 1) / tm;
        p->fov_y = cells_np_sum(base, n, 2) / tm;
        p->fov_valid = 1;
    }
    double rmax = base[0].radius;
    for (int i = 1; i < n; ++i)
        if (base[i].radius > rmax) rmax = base[i].radius;
    p->fov_size = agar_pow(rmax, 0.475) * P.pow_n[n] * 35;
}
/* cooperative: the fields of view of ALL players at once, lane k for player k.  Every alive player's bot turn computes
 * them from the same cells (bot turns only set command points and split / eject flags), so K sequential lane-0 passes
 * — a `pow`, two pairwise sums and a mass total each — become one pass with K lanes busy. */
template <int W>
DEV void update_all_fovs(Ctx<W>& c, const DevParams& P) {
    for (int k = c.lane; k < P.L.n_players; k += W) update_fov(c, P, k);
    c.t.sync();
}
/* cooperative: compact list of the live cells (of 16 x 16 slots, ~24 are live in the arena), valid while no cell is
 * created or removed — the bot phase.  Loops over "every cell of every player" then run one or two full-width
 * iterations instead of eight nearly empty ones. */
template <int W>
DEV const uint16_t* live_cells(const Ctx<W>& c, const DevParams& P) { return (const uint16_t*)(c.scratch + P.live_off); }
template <int W>
DEV void build_live_cells(Ctx<W>& c, const DevParams& P) {
    uint16_t* live = (uint16_t*)(c.scratch + P.live_off);
    const int cap = P.L.cell_cap, total = P.L.n_players * cap;
    int n = 0;
    for (int base = 0; base < total; base += W) {
        int idx = base + c.lane, k2 = idx >> P.cap_shift, j = idx - (k2 << P.cap_shift);
        bool on = idx < total && j < c.pl[k2].n_cells;
        unsigned b = c.t.ballot(on);
        if (on) live[n + __popc(b & ((1u << c.lane) - 1))] = (uint16_t)idx;
        n += __popc(b);
    }
    c.n_live = n;
    c.t.sync();
}
template <int W>
DEV void cell_remove(Ctx<W>& c, const DevParams& P, int k, int i) {
    AgarPlayer* p = &c.pl[k];
    AgarCell* base = CELLP(c, P, k, 0);
    for (int j = i; j + 1 < p->n_cells; ++j) base[j] = base[j + 1];
    p->n_cells -= 1;
    AgarCell z = {};
    base[p->n_cells] = z;
}
template <int W>
DEV AgarCell* cell_append(Ctx<W>& c, const DevParams& P, int k, double x, double y, double mass) {
    AgarPlayer* p = &c.pl[k];
    AgarCell* nc = CELLP(c, P, k, p->n_cells);
    AgarCell z = {};
    *nc = z;
    nc->x = x, nc->y = y, nc->mass = mass, nc->radius = radius_of_call(mass);
    nc->uid = c.h->next_uid++;
    p->n_cells += 1;
    return nc;
}
template <int W>
DEV void delete_player_cell(Ctx<W>& c, const DevParams& P, int k, int i) { /* field.py:382-388 */
    cell_remove(c, P, k, i);
    AgarPlayer* p = &c.pl[k];
    if (p->n_cells == 0) {
        c.h->dead_order[c.h->n_dead++] = k;
        p->alive = 0;
        p->respawn_time = 1;
        log_ev(c, P, AGAR_EV_PLAYER_DIED, k, 0, 0, 0);
        p->bot.stat_deaths += 1;
    }
}

/* ------------------------------------------------------------------ momentum / movement (cell.py:96-141) */
DEV void add_momentum(double S, double x, double y, double px, double py, double orig_radius, double* svx, double* svy,
                      int32_t* counter) {
    double cx = py_max0(py_minS(S, px)), cy = py_max0(py_minS(S, py));
    double cs, sn;
    agar_dir(cy - y, cx - x, &cs, &sn);
    double speed = 2 + orig_radius * 0.05;
    *svx = cs * speed;
    *svy = sn * speed;
    *counter = 15;
}
DEV void update_momentum(double& svx, double& svy, int32_t& counter) {
    if (counter == -1) return;
    if (counter > 0) {
        counter -= 1;
        double ratio = (double)counter / 15;
        if (ratio < 0.1) {
            svx *= (1 - ratio);
            svy *= (1 - ratio);
        }
    } else {
        svx = 0, svy = 0;
        counter = -1;
    }
}
DEV void update_pos(double& x, double& y, double vx, double vy, double& svx, double& svy, int counter, double S) {
    double xs = vx + svx, ys = vy + svy;
    x = clampS(x + xs, S);
    y = clampS(y + ys, S);
    if ((counter && x == S) || x == 0) svx *= -1;
    if ((counter && y == S) || y == 0) svy *= -1;
}

/* ------------------------------------------------------------------ spawning (field.py:262-313) */
/* lane 0 */
template <int W>
DEV bool player_bucket_occupied(const Ctx<W>& c, const DevParams& P, int bx, int by) {
    for (int k = 0; k < P.L.n_players; ++k)
        for (int i = 0; i < c.pl[k].n_cells; ++i) {
            const AgarCell* q = CELLP(c, P, k, i);
            if (!(q->flags & AGAR_CF_INHASH)) continue;
            Rect r = rect_of_call(P.S, q->x, q->y, q->radius);
            if (r.x1 < r.x0 || r.y1 < r.y0) continue;
            if (bx >= r.x0 && bx <= r.x1 && by >= r.y0 && by <= r.y1) return true;
        }
    return false;
}
template <int W>
DEV void get_spawn_pos(Ctx<W>& c, const DevParams& P, double radius, double& ox, double& oy) { /* :283-301 */
    int cols = P.nb, total = cols * cols;
    int b = draw_randint(c, P, 0, 0, total), count = 0;
    while (count < total && player_bucket_occupied(c, P, b % cols, b / cols)) {
        b = (b + 1) % total;
        count++;
    }
    if (count == total) {
        ox = (double)draw_randint(c, P, 0, 0, P.S);
        oy = (double)draw_randint(c, P, 0, 0, P.S);
    } else {
        int x = b % cols;
        double y = (double)(b - x) / cols;
        double left = (double)((x - 1) * AG_BUCKET), top = y * AG_BUCKET;
        ox = (double)draw_randint(c, P, 0, left + radius, left + AG_BUCKET - radius);
        oy = (double)draw_randint(c, P, 0, top + radius, top + AG_BUCKET - radius);
    }
}
template <int W>
DEV void initialize_player(Ctx<W>& c, const DevParams& P, int k) { /* :49-55, lane 0 */
    AgarPlayer* p = &c.pl[k];
    AgarCell z = {};
    for (int i = 0; i < P.L.cell_cap; ++i) *CELLP(c, P, k, i) = z;
    p->n_cells = 0;
    double x, y;
    get_spawn_pos(c, P, P.start_radius, x, y);
    AgarCell* nc = cell_append(c, P, k, x, y, 10.0);
    p->alive = 1;
    p->respawn_time = 0;
    log_ev(c, P, AGAR_EV_SPAWN_PLAYER, k, (int)nc->uid, (int)x, (int)y);
}
/* cooperative: every lane of the tile calls it.  field.py:303-313, :20-26 */
template <int W>
DEV void spawn_pellets(Ctx<W>& c, const DevParams& P) {
    int from = 0;
    const int cap = P.L.pellet_cap;
    while (true) {
        bool need = (double)(c.h->n_pellets + c.h->n_fat) < P.L.max_pellets;
        if (!need) break;
        int slot = -1;
        for (int base = from; base < cap; base += W) {
            int s = base + c.lane;
            bool fr = s < cap && c.pel[s] == 0;
            unsigned b = c.t.ballot(fr);
            if (b) {
                slot = base + __ffs(b) - 1;
                break;
            }
        }
        if (slot < 0) break; /* cannot happen: n_pellets < max <= cap */
        if (c.lane == 0) {
            int x = draw_randint(c, P, 0, 0, P.S), y = draw_randint(c, P, 0, 0, P.S);
            int v = draw_randint(c, P, 0, 0, 50);
            int m = v > 46 ? 50 - v : 1;
            log_ev(c, P, AGAR_EV_SPAWN_PELLET, slot, x, y, m);
            c.pel[slot] = AGAR_PELLET_PACK(x, y, m);
            c.h->n_pellets += 1;
        }
        from = slot + 1;
        c.t.sync();
    }
}
template <int W>
DEV void spawn_viruses(Ctx<W>& c, const DevParams& P) { /* lane 0; :262-275 */
    while ((double)c.h->n_viruses < P.L.max_viruses) {
        if (c.h->n_viruses >= P.L.virus_cap) {
            c.h->overflow |= AGAR_OVF_VIRUS;
            break;
        }
        double x, y;
        get_spawn_pos(c, P, P.virus_radius, x, y);
        double acc = AG_BUCKET - P.virus_radius;
        x += (double)draw_randint(c, P, 0, (-1) * acc / 2, acc / 2);
        y += (double)draw_randint(c, P, 0, (-1) * acc / 2, acc / 2);
        AgarMote* v = &c.vir[c.h->n_viruses];
        AgarMote z = {};
        *v = z;
        v->x = x, v->y = y, v->mass = 100.0, v->radius = radius_of_call(100.0);
        log_ev(c, P, AGAR_EV_SPAWN_VIRUS, c.h->n_viruses, (int)x, (int)y, 0);
        c.h->n_viruses += 1;
    }
}
template <int W>
DEV void spawn_players(Ctx<W>& c, const DevParams& P) { /* lane 0; :277-281 */
    int n = c.h->n_dead, w = 0;
    int order[AGAR_MAX_PLAYERS];
    for (int i = 0; i < n; ++i) order[i] = c.h->dead_order[i];
    for (int i = 0; i < n; ++i) {
        int k = order[i];
        if (c.pl[k].respawn_time == 0)
            initialize_player(c, P, k);
        else
            c.h->dead_order[w++] = k;
    }
    c.h->n_dead = w;
    for (int i = w; i < n; ++i) c.h->dead_order[i] = 0;
}
template <int W, bool FULL>
DEV void spawn_stuff(Ctx<W>& c, const DevParams& P) { /* cooperative; :256-260 */
    spawn_pellets(c, P);
    if (FULL) {
        if (c.lane == 0) {
            if (P.cfg.virus_enabled) spawn_viruses(c, P);
            if (c.h->n_dead) spawn_players(c, P);
        }
        c.t.sync();
    }
}

/* ------------------------------------------------------------------ Field.update phases */
template <int W>
DEV void blob_remove(Ctx<W>& c, int i) {
    for (int j = i; j + 1 < c.h->n_blobs; ++j) c.blob[j] = c.blob[j + 1];
    c.h->n_blobs -= 1;
    AgarMote z = {};
    c.blob[c.h->n_blobs] = z;
}
template <int W>
DEV void virus_remove(Ctx<W>& c, int i) {
    for (int j = i; j + 1 < c.h->n_viruses; ++j) c.vir[j] = c.vir[j + 1];
    c.h->n_viruses -= 1;
    AgarMote z = {};
    c.vir[c.h->n_viruses] = z;
}
/* cooperative; field.py:94-110 */
template <int W>
DEV void update_viruses_blobs(Ctx<W>& c, const DevParams& P) {
    const double S = (double)P.S;
    int nv = c.h->n_viruses, nb = c.h->n_blobs;
    for (int i = c.lane; i < nv; i += W) {
        AgarMote* v = &c.vir[i];
        double svx = v->svx, svy = v->svy, x = v->x, y = v->y;
        int32_t cnt = v->counter;
        update_momentum(svx, svy, cnt);
        update_pos(x, y, 0, 0, svx, svy, cnt, S);
        v->svx = svx, v->svy = svy, v->x = x, v->y = y, v->counter = cnt;
    }
    bool any_still = false;
    for (int i = c.lane; i < nb; i += W) {
        AgarMote* b = &c.blob[i];
        if (b->counter == 0) {
            any_still = true;
            continue;
        }
        double svx = b->svx, svy = b->svy, x = b->x, y = b->y;
        int32_t cnt = b->counter;
        update_momentum(svx, svy, cnt);
        update_pos(x, y, 0, 0, svx, svy, cnt, S);
        /* a blob whose counter reaches 0 here stays a blob until the next frame; mark it with counter 0 */
        b->svx = svx, b->svy = svy, b->x = x, b->y = y, b->counter = cnt;
        if (cnt == 0) b->aux |= 0x80000000u; /* "reached zero this frame" (cleared below) */
    }
    c.t.sync();
    if (nb && c.t.any(any_still)) {
        if (c.lane == 0) { /* blobs that were already still become float-position pellets, in list order */
            int i = 0;
            while (i < c.h->n_blobs) {
                AgarMote b = c.blob[i];
                if (b.counter != 0 || (b.aux & 0x80000000u)) {
                    ++i;
                    continue;
                }
                blob_remove(c, i);
                int slot = 0;
                while (slot < P.L.fat_cap && c.fat[slot].mass != 0) ++slot;
                if (slot == P.L.fat_cap) {
                    c.h->overflow |= AGAR_OVF_FAT;
                    continue;
                }
                AgarFatPellet* f = &c.fat[slot];
                f->x = b.x, f->y = b.y, f->mass = b.mass, f->radius = b.radius;
                c.h->n_fat += 1;
                log_ev(c, P, AGAR_EV_BLOB_TO_PELLET, slot, 0, 0, 0);
            }
        }
        c.t.sync();
    }
    if (nb) {
        for (int i = c.lane; i < c.h->n_blobs; i += W) c.blob[i].aux &= 0x7fffffffu;
        c.t.sync();
    }
}

/* lane 0: split / eject flag / movement / ejections / collisions of one player.  vel = scratch [cells][2]. */
template <int W>
DEVN void player_split_and_flags(Ctx<W>& c, const DevParams& P, int k, double* vel) { /* lane 0; before the cells move */
    AgarPlayer* p = &c.pl[k];
    AgarCell* base = CELLP(c, P, k, 0);
    const double S = (double)P.S;
    double* vx = vel + (size_t)k * P.L.cell_cap * 2;
    double* vy = vx + P.L.cell_cap;
    if (p->do_split) { /* player.py:53-61 */
        for (int i = 1; i < p->n_cells; ++i) {
            AgarCell t = base[i];
            double tvx = vx[i], tvy = vy[i];
            int j = i - 1;
            while (j >= 0 && base[j].mass < t.mass) {
                base[j + 1] = base[j];
                vx[j + 1] = vx[j], vy[j + 1] = vy[j];
                --j;
            }
            base[j + 1] = t;
            vx[j + 1] = tvx, vy[j + 1] = tvy;
        }
        int n0 = p->n_cells;
        for (int i = 0; i < n0; ++i) {
            AgarCell* q = &base[i];
            if (q->mass > 36 && p->n_cells < 16) { /* cell.py:72-85 */
                double parent_radius = q->radius;
                int ni = p->n_cells;
                AgarCell* nc = cell_append(c, P, k, q->x, q->y, q->mass / 2);
                vx[ni] = 0, vy[ni] = 0;
                double cs, sn;
                agar_dir(p->cmd_y - nc->y, p->cmd_x - nc->x, &cs, &sn);
                double xp = cs * nc->radius * 4.5 + q->x, yp = sn * nc->radius * 4.5 + q->y;
                add_momentum(S, nc->x, nc->y, xp, yp, parent_radius, &nc->svx, &nc->svy, &nc->counter);
                nc->merge_time = merge_time_for(1, nc->mass);
                q->mass = q->mass / 2;
                q->radius = radius_of_call(q->mass);
                log_ev(c, P, AGAR_EV_SPLIT, k, (int)q->uid, (int)nc->uid, 0);
            }
        }
    }
    if (p->do_eject) /* player.py:63-68 */
        for (int i = 0; i < p->n_cells; ++i)
            if (base[i].mass >= 35) base[i].flags |= AGAR_CF_EJECT;
}

/* lane 0; after the player's cells have moved, before their self-collisions (field.py:134-146) */
template <int W>
DEVN void player_ejections(Ctx<W>& c, const DevParams& P, int k) {
    AgarPlayer* p = &c.pl[k];
    AgarCell* base = CELLP(c, P, k, 0);
    const double S = (double)P.S;
    if (p->do_eject) /* field.py:134-146, cell.py:90-94 */
        for (int i = 0; i < p->n_cells; ++i) {
            AgarCell* q = &base[i];
            if (!(q->flags & AGAR_CF_EJECT)) continue;
            q->mass -= 18;
            q->flags &= ~AGAR_CF_EJECT;
            if (c.h->n_blobs >= P.L.blob_cap) {
                c.h->overflow |= AGAR_OVF_BLOB;
                continue;
            }
            AgarMote* b = &c.blob[c.h->n_blobs];
            AgarMote z = {};
            *b = z;
            b->x = q->x, b->y = q->y, b->mass = P.blob_mass, b->radius = radius_of_call(P.blob_mass);
            add_momentum(S, b->x, b->y, p->cmd_x, p->cmd_y, q->radius, &b->svx, &b->svy, &b->counter);
            b->aux = q->uid;
            log_ev(c, P, AGAR_EV_EJECT, k, (int)q->uid, c.h->n_blobs, 0);
            c.h->n_blobs += 1;
        }
}

/* cooperative: handlePlayerCollisions (field.py:149-181) — the same-player push-apart, a Gauss-Seidel sweep over the ORDERED
 * pairs (i, j), j != i, with immediate position updates.  At steady state a split player holds up to 16 cells that sit exactly
 * touching one another, so the reference's 240 sequential pair tests (a sqrt each) with ~10 adjustments per player and frame
 * were the largest single-lane loop of the multi-agent kernel (27 % of all instructions of the 1-vs-greedy config, and the
 * main source of CTA-barrier imbalance).  Exact parallel form: every lane tests its share of the 16 x 16 pair slots on the
 * current positions; the tile takes the FIRST hit in pair order, lane 0 applies the adjustment with the reference's arithmetic,
 * and only the pairs after it that involve one of the two moved cells are re-tested (a test depends on nothing else).  Pairs
 * before the current one are never revisited, exactly as in the sequential sweep.  The sqrt is only evaluated inside the
 * rounding band of `dist < sum` (d2 against sum^2 with a 1e-12 margin decides everything else identically). */
DEV bool self_collision_test(const AgarCell* base, int n, int i, int j) {
    if (i >= n || j >= n || i == j) return false;
    const AgarCell* a = &base[i];
    const AgarCell* b = &base[j];
    if (a->counter > 0 || b->counter > 0 || (a->merge_time <= 0 && b->merge_time <= 0)) return false;
    const double d2 = (a->x - b->x) * (a->x - b->x) + (a->y - b->y) * (a->y - b->y);
    const double sum = a->radius + b->radius, s2 = sum * sum;
    if (d2 > s2 * (1.0 + 1e-12) || d2 == 0.0) return false;
    if (d2 < s2 * (1.0 - 1e-12)) return true;
    const double dist = sqrt(d2);
    return dist < sum && dist != 0;
}
/* lane 0: the sequential sweep (tiles narrower than a warp, where the cooperative form below does not fit) */
template <int W>
DEV void self_collisions_seq(Ctx<W>& c, const DevParams& P, int k) {
    AgarPlayer* p = &c.pl[k];
    AgarCell* base = CELLP(c, P, k, 0);
    const double S = (double)P.S;
    for (int i = 0; i < p->n_cells; ++i) {
        AgarCell* a = &base[i];
        if (a->counter > 0) continue;
        for (int j = 0; j < p->n_cells; ++j) {
            AgarCell* b = &base[j];
            if (i == j || b->counter > 0 || (a->merge_time <= 0 && b->merge_time <= 0)) continue;
            double d2 = (a->x - b->x) * (a->x - b->x) + (a->y - b->y) * (a->y - b->y);
            double dist = sqrt(d2), sum = a->radius + b->radius;
            if (dist < sum && dist != 0) {
                log_ev(c, P, AGAR_EV_COLLIDE, k, (int)a->uid, (int)b->uid, 0);
                AgarCell *big, *sm;
                if (a->mass > b->mass)
                    big = a, sm = b;
                else
                    big = b, sm = a;
                double ds = (sum - dist) / dist, q = sm->mass / big->mass;
                double xs = (big->x - sm->x) * ds, ys = (big->y - sm->y) * ds;
                double nbx = big->x + xs * q, nby = big->y + ys * q;
                double nsx = sm->x - xs * (1 - q), nsy = sm->y - ys * (1 - q);
                big->x = clampS(nbx, S), big->y = clampS(nby, S);
                sm->x = clampS(nsx, S), sm->y = clampS(nsy, S);
            }
        }
    }
}
/* W == 32.  Lane r < 16 keeps row r of the 16 x 16 hit matrix (bit j: the ordered pair (r, j) collides on the current
 * positions).  After an adjustment of (i, j) only rows i, j and columns i, j can change: lanes 0..15 re-test row i, lanes
 * 16..31 row j (one test each, gathered with a ballot), then the same for the two columns (each lane folds its own bit in). */
template <int W>
DEV void player_self_collisions(Ctx<W>& c, const DevParams& P, int k) {
    AgarPlayer* p = &c.pl[k];
    const int n = p->n_cells;
    if (n < 2) return;
    if (W != 32) {
        if (c.lane == 0) self_collisions_seq(c, P, k);
        return;
    }
    AgarCell* base = CELLP(c, P, k, 0);
    const double S = (double)P.S;
    const int r = c.lane & 15, half = c.lane >> 4;
    unsigned row = 0;
    { /* initial matrix: lane (r, half) tests columns [8 half, 8 half + 8) of row r */
        unsigned part = 0;
        const int j0 = half * 8, j1 = min(n, j0 + 8);
        if (r < n)
            for (int j = j0; j < j1; ++j)
                if (self_collision_test(base, n, r, j)) part |= 1u << j;
        row = part | c.t.shfl_xor(part, 16);
    }
    int ci = -1, cj = -1; /* the pair processed last: everything up to it in (i, j) order is done */
    while (true) {
        unsigned m = row;
        if (r < ci) m = 0;
        else if (r == ci) m &= ~((2u << cj) - 1u);
        const int mine = (half == 0 && m) ? r * 16 + __ffs((int)m) - 1 : 0x7fffffff;
        const int first = cg::reduce(c.t, mine, cg::less<int>());
        if (first == 0x7fffffff) break;
        const int i = first >> 4, j = first & 15;
        if (c.lane == 0) {
            AgarCell *a = &base[i], *b = &base[j];
            double d2 = (a->x - b->x) * (a->x - b->x) + (a->y - b->y) * (a->y - b->y);
            double dist = sqrt(d2), sum = a->radius + b->radius;
            log_ev(c, P, AGAR_EV_COLLIDE, k, (int)a->uid, (int)b->uid, 0);
            AgarCell *big, *sm;
            if (a->mass > b->mass)
                big = a, sm = b;
            else
                big = b, sm = a;
            double ds = (sum - dist) / dist, q = sm->mass / big->mass;
            double xs = (big->x - sm->x) * ds, ys = (big->y - sm->y) * ds;
            double nbx = big->x + xs * q, nby = big->y + ys * q;
            double nsx = sm->x - xs * (1 - q), nsy = sm->y - ys * (1 - q);
            big->x = clampS(nbx, S), big->y = clampS(nby, S);
            sm->x = clampS(nsx, S), sm->y = clampS(nsy, S);
        }
        c.t.sync();
        ci = i, cj = j;
        { /* rows i (lanes 0..15) and j (lanes 16..31) */
            const bool h = self_collision_test(base, n, half ? j : i, r);
            const unsigned bal = c.t.ballot(h);
            if (r == i) row = bal & 0xffffu;
            if (r == j) row = bal >> 16;
        }
        { /* columns i (lanes 0..15 test (r, i)) and j (lanes 16..31 test (r, j)): lane r folds both bits into its row */
            const bool h = self_collision_test(base, n, r, half ? j : i);
            const unsigned bal = c.t.ballot(h);
            const unsigned bi = (bal >> r) & 1u, bj = (bal >> (16 + r)) & 1u;
            row = (row & ~((1u << i) | (1u << j))) | (bi << i) | (bj << j);
        }
    }
}

/* per-cell kinematics of one cell: decay, momentum, merge timer, velocity (player.py:43-51; cell.py:47-57,105-130) */
DEV void cell_kinematics(const DevParams& P, AgarCell* q, double cmd_x, double cmd_y, double& vx, double& vy) {
    double mass = q->mass, radius = q->radius;
    if (mass >= 4) {
        mass = mass * P.decay_rate;
        radius = radius_of_call(mass);
        q->mass = mass, q->radius = radius;
    }
    double svx = q->svx, svy = q->svy;
    int32_t cnt = q->counter;
    update_momentum(svx, svy, cnt);
    q->svx = svx, q->svy = svy, q->counter = cnt;
    double mt = q->merge_time;
    if (mt > 0) q->merge_time = mt - 1;
    double xd = cmd_x - q->x, yd = cmd_y - q->y;
    double h2 = xd * xd + yd * yd, r2 = radius * radius;
    double sm = (h2 < r2 ? h2 : r2) / r2;
    double cs, sn;
    agar_dir(yd, xd, &cs, &sn);
    double rs = P.move_speed * agar_pow(mass, -0.35);
    vx = rs * sm * cs;
    vy = rs * sm * sn;
}

/* cooperative; field.py:112-132 (updatePlayers + updateHashTables) */
template <int W, bool FULL>
DEV void update_players(Ctx<W>& c, const DevParams& P) {
    const double S = (double)P.S;
    if (!FULL) { /* K == 1, one cell, no split / eject / virus: everything is lane 0's */
        if (c.lane == 0) {
            AgarPlayer* p = &c.pl[0];
            AgarCell* q = &c.cells[0];
            double vx, vy;
            cell_kinematics(P, q, p->cmd_x, p->cmd_y, vx, vy);
            update_pos(q->x, q->y, vx, vy, q->svx, q->svy, q->counter, S);
            q->flags |= AGAR_CF_INHASH;
        }
        c.t.sync();
        return;
    }
    const int K = P.L.n_players, cap = P.L.cell_cap;
    double* vel = (double*)c.scratch; /* [K][2][cap] */
    /* phase A: every live cell of every live player, lane-parallel */
    for (int idx = c.lane; idx < K * cap; idx += W) {
        int k = idx >> P.cap_shift, i = idx - (k << P.cap_shift);
        const AgarPlayer* p = &c.pl[k];
        if (!p->alive || i >= p->n_cells) continue;
        double vx, vy;
        cell_kinematics(P, CELLP(c, P, k, i), p->cmd_x, p->cmd_y, vx, vy);
        vel[(size_t)k * cap * 2 + i] = vx;
        vel[(size_t)k * cap * 2 + cap + i] = vy;
    }
    c.t.sync();
    /* phase B (updatePlayers, field.py:112-119 + player.py:30-36), per player in player order — the event log and the blob list are
     * ordered by player: split and eject flags (lane 0, rare: only on decision frames with a split / eject bit), then the player's
     * cells move, ONE LANE PER CELL (round 1 moved them one after the other on lane 0: in the arena, whose cells live in HBM, a
     * chain of dependent global round trips), then ejections (lane 0), then the cooperative self-collision sweep. */
    for (int k = 0; k < K; ++k) {
        AgarPlayer* p = &c.pl[k];
        if (!p->alive) {
            if (c.lane == 0) p->respawn_time -= 1;
            continue;
        }
        if (p->do_split || p->do_eject) {
            if (c.lane == 0) player_split_and_flags(c, P, k, vel);
            c.t.sync();
        }
        const int n = p->n_cells;
        for (int i = c.lane; i < n; i += W) {
            AgarCell* q = CELLP(c, P, k, i);
            update_pos(q->x, q->y, vel[(size_t)k * cap * 2 + i], vel[(size_t)k * cap * 2 + cap + i], q->svx, q->svy, q->counter, S);
        }
        if (p->do_eject) {
            c.t.sync();
            if (c.lane == 0) player_ejections(c, P, k);
        }
        if (n > 1) {
            c.t.sync();
            player_self_collisions<W>(c, P, k);
        }
    }
    c.t.sync();
    /* updateHashTables: every live cell / virus is (re)inserted */
    for (int idx = c.lane; idx < K * cap; idx += W) {
        int k = idx >> P.cap_shift, i = idx - (k << P.cap_shift);
        if (i < c.pl[k].n_cells) CELLP(c, P, k, i)->flags |= AGAR_CF_INHASH;
    }
    for (int i = c.lane; i < c.h->n_viruses; i += W) c.vir[i].aux = AGAR_CF_INHASH;
    c.t.sync();
}

/* lane 0; field.py:183-198, :372-380 */
template <int W>
DEVN void merge_player_cells_seq(Ctx<W>& c, const DevParams& P, int k) {
    AgarPlayer* p = &c.pl[k];
    AgarCell* base = CELLP(c, P, k, 0);
    uint32_t uid[AGAR_MAX_CELLS];
    double mass[AGAR_MAX_CELLS];
    int n = 0;
    for (int i = 0; i < p->n_cells; ++i)
        if (base[i].merge_time <= 0) uid[n] = base[i].uid, mass[n] = base[i].mass, ++n;
    if (n <= 1) return;
    for (int a = 1; a < n; ++a) {
        uint32_t tu = uid[a];
        double tm = mass[a];
        int j = a - 1;
        while (j >= 0 && mass[j] < tm) {
            uid[j + 1] = uid[j], mass[j + 1] = mass[j];
            --j;
        }
        uid[j + 1] = tu, mass[j + 1] = tm;
    }
    unsigned alive = (1u << n) - 1;
    for (int a = 0; a < n; ++a) {
        if (!(alive >> a & 1)) continue;
        for (int b = 0; b < n; ++b) {
            if (!(alive >> b & 1) || b == a) continue;
            int ia = -1, ib = -1;
            for (int i = 0; i < p->n_cells; ++i) {
                if (base[i].uid == uid[a]) ia = i;
                if (base[i].uid == uid[b]) ib = i;
            }
            AgarCell *c1 = &base[ia], *c2 = &base[ib];
            if (overlap(c1->x, c1->y, c1->mass, c1->radius, c2->x, c2->y, c2->mass, c2->radius)) {
                bool first_big = c1->mass > c2->mass;
                AgarCell *cb = first_big ? c1 : c2, *cs = first_big ? c2 : c1;
                int sm = first_big ? b : a;
                log_ev(c, P, AGAR_EV_MERGE, k, (int)cb->uid, (int)cs->uid, 0);
                grow(cb, cs->mass);
                alive &= ~(1u << sm);
                delete_player_cell(c, P, k, first_big ? ib : ia);
                if (!(alive >> a & 1)) break;
            }
        }
    }
}

/* lane 0; field.py:246-253, :316-325 */
template <int W>
DEVN void virus_blob_overlap_seq(Ctx<W>& c, const DevParams& P) {
    const double S = (double)P.S;
    for (int vi = 0; vi < c.h->n_viruses; ++vi) {
        AgarMote* v = &c.vir[vi];
        Rect rv = rect_of_call(P.S, v->x, v->y, v->radius);
        /* candidates are the blobs sharing a bucket with the virus BEFORE it eats; kept as a bitmask walk */
        int nb0 = c.h->n_blobs;
        int removed_before = 0;
        for (int b0 = 0; b0 < nb0; ++b0) {
            int b = b0 - removed_before;
            AgarMote* bl = &c.blob[b];
            /* rect test uses the virus rectangle at the start of its pass (rv) */
            if (!rect_hit(rv, rect_of_call(P.S, bl->x, bl->y, bl->radius))) continue;
            if (!overlap(v->x, v->y, v->mass, v->radius, bl->x, bl->y, bl->mass, bl->radius)) continue;
            double bx = bl->x, by = bl->y;
            grow_mote(v, bl->mass);
            blob_remove(c, b);
            removed_before += 1;
            int split = 0;
            if (v->mass >= P.virus_split_mass) {
                if (c.h->n_viruses >= P.L.virus_cap)
                    c.h->overflow |= AGAR_OVF_VIRUS;
                else {
                    double ox = 2 * v->x - bx, oy = 2 * v->y - by;
                    AgarMote* nv = &c.vir[c.h->n_viruses];
                    AgarMote z = {};
                    *nv = z;
                    nv->x = v->x, nv->y = v->y, nv->mass = v->mass / 2, nv->radius = radius_of_call(nv->mass);
                    double cs, sn;
                    agar_dir(oy - nv->y, ox - nv->x, &cs, &sn);
                    double xp = cs * nv->radius * 4.5 + v->x, yp = sn * nv->radius * 4.5 + v->y;
                    add_momentum(S, nv->x, nv->y, xp, yp, v->radius, &nv->svx, &nv->svy, &nv->counter);
                    v->mass = v->mass / 2;
                    v->radius = radius_of_call(v->mass);
                    c.h->n_viruses += 1;
                    split = 1;
                }
            }
            log_ev(c, P, AGAR_EV_VIRUS_EAT_BLOB, vi, b, split, 0);
        }
    }
}

/* lane 0; field.py:350-370 */
template <int W>
DEV void player_cell_ate_virus(Ctx<W>& c, const DevParams& P, int k, int ci) {
    const double S = (double)P.S;
    AgarPlayer* p = &c.pl[k];
    int n_new = 16 - p->n_cells;
    if (n_new == 0) return;
    AgarCell* q = CELLP(c, P, k, ci);
    double distributed = q->mass * 0.6;
    double per = distributed / n_new;
    q->merge_time = merge_time_for(0.85, q->mass);
    grow(q, -1 * per * n_new);
    for (int j = 0; j < n_new; ++j) {
        AgarCell* nc = cell_append(c, P, k, q->x, q->y, per);
        int deg = draw_randint(c, P, 0, 0, 360);
        double cs = P.deg_tab[deg], sn = P.deg_tab[360 + deg];
        double xp = cs * q->radius * 12 + q->x, yp = sn * q->radius * 12 + q->y;
        add_momentum(S, nc->x, nc->y, xp, yp, q->radius, &nc->svx, &nc->svy, &nc->counter);
        nc->merge_time = merge_time_for(0.8, nc->mass);
        nc->flags |= AGAR_CF_INHASH;
    }
}
/* lane 0; field.py:225-231, :333-335 */
template <int W>
DEVN void player_virus_overlap_seq(Ctx<W>& c, const DevParams& P) {
    for (int k = 0; k < P.L.n_players; ++k) {
        AgarPlayer* p = &c.pl[k];
        if (!p->alive) continue;
        for (int ci = 0; ci < p->n_cells; ++ci) {
            AgarCell* q = CELLP(c, P, k, ci);
            Rect rc = rect_of_call(P.S, q->x, q->y, q->radius);
            /* candidate set fixed at the start of the cell's pass: bit v0 of a 64-bit mask over the virus list */
            unsigned long long cand = 0;
            int nv0 = c.h->n_viruses;
            for (int v = 0; v < nv0 && v < 64; ++v)
                if ((c.vir[v].aux & AGAR_CF_INHASH) &&
                    rect_hit(rc, rect_of_call(P.S, c.vir[v].x, c.vir[v].y, c.vir[v].radius)))
                    cand |= 1ull << v;
            int removed = 0;
            for (int v0 = 0; v0 < nv0 && v0 < 64; ++v0) {
                if (!(cand >> v0 & 1)) continue;
                int vi = v0 - removed;
                AgarMote* v = &c.vir[vi];
                if (overlap(q->x, q->y, q->mass, q->radius, v->x, v->y, v->mass, v->radius) && q->mass > 1.25 * v->mass) {
                    log_ev(c, P, AGAR_EV_EAT_VIRUS, k, (int)q->uid, vi, 16 - p->n_cells);
                    grow(q, v->mass * 0.5);
                    virus_remove(c, vi);
                    removed += 1;
                    player_cell_ate_virus(c, P, k, ci);
                }
            }
        }
    }
}

/* ---- per-env pellet index (north star (3): a per-env uniform grid built by a shared-memory counting sort).  The INTEGER
 * pellet pool is bucketed by the pellet's own point on a 10-unit grid — finer than the reference's 20-unit hash table
 * (spatialHashTable.py:49-83): the reference's table only decides which pairs get TESTED, and a pair that fails the overlap
 * test has no effect whatsoever, so any index that returns a superset of the pellets a cell can actually eat is equivalent
 * (the exact bucket-rectangle condition of the reference's candidate list is still applied per pellet, and eaten pellets are
 * taken in canonical slot order).  Rebuilt once per frame in the tile's scratch: count (shared-memory atomics on packed uint16
 * pairs) -> exclusive scan over the gb x gb buckets -> scatter.  Layout: uint16 cnt[gb2 + 2] (after the scatter cnt[b] = END of
 * bucket b, so bucket b = [b ? cnt[b - 1] : 0, cnt[b])), uint16 ent[pellet_cap] (pool slots), uint16 tmp[64]. */
#define AG_IDX_CELL 10
DEV int pel_index_gb(const DevParams& P) { return (P.S + AG_IDX_CELL - 1) / AG_IDX_CELL; }
DEV int pel_index_cnt_len(const DevParams& P) { return (pel_index_gb(P) * pel_index_gb(P) + 2 + 1) & ~1; }
DEV bool pel_index_enabled(const DevParams& P) { return P.full && P.pel_index; }
template <int W>
DEV void build_pellet_index(Ctx<W>& c, const DevParams& P) {
    const int gb = pel_index_gb(P), gb2 = gb * gb, cap = P.L.pellet_cap, nc = pel_index_cnt_len(P);
    uint16_t* cnt = (uint16_t*)c.scratch;
    uint32_t* cnt32 = (uint32_t*)c.scratch; /* two counters per word: counts stay below 65536, the halves never carry */
    uint16_t* ent = cnt + nc;
    for (int i = c.lane; i < nc / 2; i += W) cnt32[i] = 0;
    c.t.sync();
    for (int s = c.lane; s < cap; s += W) {
        const uint32_t pk = c.pel[s];
        if (!pk) continue;
        const int b = (AGAR_PELLET_Y(pk) / AG_IDX_CELL) * gb + AGAR_PELLET_X(pk) / AG_IDX_CELL;
        atomicAdd(&cnt32[b >> 1], (b & 1) ? 0x10000u : 1u);
    }
    c.t.sync();
    /* exclusive scan: lane l owns the consecutive buckets [l * per, l * per + per) */
    const int per = (gb2 + W - 1) / W;
    uint32_t local = 0;
    for (int i = 0; i < per; ++i) {
        const int b = c.lane * per + i;
        if (b < gb2) local += cnt[b];
    }
    uint32_t incl = local;
    for (int off = 1; off < W; off <<= 1) {
        const uint32_t v = c.t.shfl_up(incl, off);
        if (c.lane >= off) incl += v;
    }
    uint32_t run = incl - local;
    for (int i = 0; i < per; ++i) {
        const int b = c.lane * per + i;
        if (b < gb2) {
            const uint32_t n = cnt[b];
            cnt[b] = (uint16_t)run;
            run += n;
        }
    }
    c.t.sync();
    for (int s = c.lane; s < cap; s += W) {
        const uint32_t pk = c.pel[s];
        if (!pk) continue;
        const int b = (AGAR_PELLET_Y(pk) / AG_IDX_CELL) * gb + AGAR_PELLET_X(pk) / AG_IDX_CELL;
        const uint32_t old = atomicAdd(&cnt32[b >> 1], (b & 1) ? 0x10000u : 1u);
        ent[(b & 1) ? (old >> 16) : (old & 0xffffu)] = (uint16_t)s;
    }
    c.t.sync();
}

/* cooperative, W == 32: one cell's pellet eating through the index.  Returns false (nothing done) if the candidate set is too
 * large for the scratch list — the caller then runs the full scan, which is always correct.
 *   1. window: every pellet the chain can eat lies within R >= r_final + 1 of the centre, r_final <= radius(mass + 3 x pellets in
 *      the window); R starts at radius + 2 and is widened until that bound holds (almost always at once);
 *   2. the window's entries (a contiguous range per bucket row) are filtered with the reference's candidate condition and a
 *      CONSERVATIVE overlap test against the largest radius the cell can reach; survivors (usually 0-3) go to a short list;
 *   3. the list is consumed in ascending slot order (tile-min), each pellet tested against the cell as grown so far: the
 *      reference's sequential eat chain, exactly. */
template <int W>
DEV bool cell_eats_pellets_indexed(Ctx<W>& c, const DevParams& P, int k, int ci, const Rect& rc, double& cm, double& cr, uint32_t uid) {
    const int gb = pel_index_gb(P), nc = pel_index_cnt_len(P);
    const uint16_t* cnt = (const uint16_t*)c.scratch;
    const uint16_t* ent = cnt + nc;
    uint16_t* tmp = (uint16_t*)(ent + P.L.pellet_cap);
    const double cx = CELLP(c, P, k, ci)->x, cy = CELLP(c, P, k, ci)->y;
    int R = (int)cr + 2, bx0, bx1, by0, by1, total;
    double m_max, r_max;
    for (int pass = 0;; ++pass) {
        if (pass == 4) return false;
        bx0 = max(0, ((int)floor(cx) - R) / AG_IDX_CELL), bx1 = min(gb - 1, ((int)floor(cx) + R + 1) / AG_IDX_CELL);
        by0 = max(0, ((int)floor(cy) - R) / AG_IDX_CELL), by1 = min(gb - 1, ((int)floor(cy) + R + 1) / AG_IDX_CELL);
        if ((int)floor(cx) - R < 0) bx0 = 0;
        if ((int)floor(cy) - R < 0) by0 = 0;
        total = 0;
        for (int by = by0 + c.lane; by <= by1; by += W) {
            const int b0 = by * gb + bx0, b1 = by * gb + bx1;
            total += (int)cnt[b1] - (b0 ? (int)cnt[b0 - 1] : 0);
        }
        total = cg::reduce(c.t, total, cg::plus<int>());
        m_max = cm + 3.0 * total;
        if (!(m_max < AG_MAX_MASS)) m_max = AG_MAX_MASS;
        r_max = radius_of_call(m_max);
        if (r_max < cr) r_max = cr; /* after an eject the stored radius is STALE (larger than sqrt(mass / pi), cell.py:92) until the
                                     * next decay; the first tests of the chain use it as it is */
        if ((int)r_max + 2 <= R) break;
        R = (int)r_max + 2;
    }
    if (total == 0) return true;
    /* 2. filter into the short list */
    const double rr = r_max > 1.0 ? r_max * r_max : 1.0;
    int n_list = 0;
    for (int by = by0; by <= by1; ++by) {
        const int b0 = by * gb + bx0, b1 = by * gb + bx1;
        const int beg = b0 ? (int)cnt[b0 - 1] : 0, end = (int)cnt[b1];
        for (int base = beg; base < end; base += W) {
            const int e = base + c.lane;
            const int slot = e < end ? (int)ent[e] : -1;
            const uint32_t pk = slot >= 0 ? c.pel[slot] : 0u;
            const int px = AGAR_PELLET_X(pk), py = AGAR_PELLET_Y(pk), pm = AGAR_PELLET_M(pk);
            const double dx = cx - (double)px, dy = cy - (double)py;
            const bool poss = pk != 0 && rect_hit(rc, pellet_rect(px, py)) && (dx * dx + dy * dy) * 1.1 < rr * (1.0 + 1e-9) &&
                              m_max > 1.25 * (double)pm;
            const unsigned bal = c.t.ballot(poss);
            if (bal) {
                const int pos = n_list + __popc(bal & ((1u << c.lane) - 1u));
                if (poss && pos < 64) tmp[pos] = (uint16_t)slot;
                n_list += __popc(bal);
            }
        }
    }
    if (n_list == 0) return true;
    if (n_list > 64) return false;
    c.t.sync();
    /* 3. ordered chain over the short list: lane l holds entries l and l + 32 */
    int s0 = c.lane < n_list ? (int)tmp[c.lane] : 0x7fffffff, s1 = c.lane + 32 < n_list ? (int)tmp[c.lane + 32] : 0x7fffffff;
    while (true) {
        const int first = cg::reduce(c.t, min(s0, s1), cg::less<int>());
        if (first == 0x7fffffff) break;
        if (s0 == first) s0 = 0x7fffffff;
        if (s1 == first) s1 = 0x7fffffff;
        const uint32_t pk = c.pel[first];
        const int px = AGAR_PELLET_X(pk), py = AGAR_PELLET_Y(pk), pm = AGAR_PELLET_M(pk);
        if (overlap(cx, cy, cm, cr, (double)px, (double)py, (double)pm, P.pellet_r[pm & 3]) && cm > 1.25 * (double)pm) {
            double nm = cm + (double)pm;
            if (!(nm < AG_MAX_MASS)) nm = AG_MAX_MASS;
            cm = nm;
            cr = radius_of_call(nm);
            c.t.sync(); /* every lane has read the slot */
            if (c.lane == 0) {
                log_ev(c, P, AGAR_EV_EAT_PELLET, k, (int)uid, first, 0);
                c.pel[first] = 0;
                c.h->n_pellets -= 1;
            }
        }
    }
    return true;
}

/* ONE LANE, one cell: can this cell eat anything this frame?  Conservative (a superset of what the exact ordered chain can eat):
 * the window / largest-radius bound of cell_eats_pellets_indexed, with every live ex-blob pellet counted into the mass bound.
 * Used to pre-filter 32 cells at a time: most cells of a frame have no edible pellet in reach and skip the cooperative pass. */
template <int W>
DEV bool cell_may_eat(const Ctx<W>& c, const DevParams& P, int k, int ci, const uint16_t* fatlist, int n_fatl, bool fat_unknown) {
    const int gb = pel_index_gb(P), nc = pel_index_cnt_len(P);
    const uint16_t* cnt = (const uint16_t*)c.scratch;
    const uint16_t* ent = cnt + nc;
    const AgarCell* q = CELLP(c, P, k, ci);
    const double cx = q->x, cy = q->y, cm = q->mass, cr = q->radius;
    if (fat_unknown) return true;
    const Rect rc = rect_of_call(P.S, cx, cy, cr);
    const double fat_mass = (double)n_fatl * P.blob_mass * 1.000001;
    int R = (int)cr + 2, bx0, bx1, by0, by1;
    double m_max, r_max;
    for (int pass = 0;; ++pass) {
        if (pass == 4) return true;
        const int fx = (int)floor(cx), fy = (int)floor(cy);
        bx0 = fx - R < 0 ? 0 : (fx - R) / AG_IDX_CELL, bx1 = min(gb - 1, (fx + R + 1) / AG_IDX_CELL);
        by0 = fy - R < 0 ? 0 : (fy - R) / AG_IDX_CELL, by1 = min(gb - 1, (fy + R + 1) / AG_IDX_CELL);
        int total = 0;
        for (int by = by0; by <= by1; ++by) {
            const int b0 = by * gb + bx0, b1 = by * gb + bx1;
            total += (int)cnt[b1] - (b0 ? (int)cnt[b0 - 1] : 0);
        }
        m_max = cm + 3.0 * total + fat_mass;
        if (!(m_max < AG_MAX_MASS)) m_max = AG_MAX_MASS;
        r_max = radius_of_call(m_max);
        if (r_max < cr) r_max = cr;
        if ((int)r_max + 2 <= R) break;
        R = (int)r_max + 2;
    }
    const double rr = (r_max > 1.0 ? r_max * r_max : 1.0) * (1.0 + 1e-9);
    for (int by = by0; by <= by1; ++by) {
        const int b0 = by * gb + bx0, b1 = by * gb + bx1;
        const int beg = b0 ? (int)cnt[b0 - 1] : 0, end = (int)cnt[b1];
        for (int e = beg; e < end; ++e) {
            const uint32_t pk = c.pel[ent[e]];
            if (!pk) continue;
            const int px = AGAR_PELLET_X(pk), py = AGAR_PELLET_Y(pk), pm = AGAR_PELLET_M(pk);
            const double dx = cx - (double)px, dy = cy - (double)py;
            if ((dx * dx + dy * dy) * 1.1 < rr && m_max > 1.25 * (double)pm && rect_hit(rc, pellet_rect(px, py))) return true;
        }
    }
    for (int t = 0; t < n_fatl; ++t) {
        const AgarFatPellet* f = &c.fat[fatlist[t]];
        const double fm = f->mass, fr = f->radius;
        if (fm == 0) continue;
        const double dx = cx - f->x, dy = cy - f->y;
        const double reach2 = (fr * fr > rr ? fr * fr * (1.0 + 1e-9) : rr);
        if ((dx * dx + dy * dy) * 1.1 < reach2 && m_max > 1.25 * fm && rect_hit(rc, rect_of_call(P.S, f->x, f->y, fr))) return true;
    }
    return false;
}

/* cooperative: the hot loop.  field.py:207-213 + eatPellet :327-344.  For one cell (k, ci): integer pellets in slot
 * order, then float ("fat") pellets in slot order; the eat chain is sequential — a pellet is tested against the
 * cell as grown by every earlier eat — but hits are found 32 pellets at a time with a ballot. */
template <int W>
DEV void cell_eats_pellets(Ctx<W>& c, const DevParams& P, int k, int ci, bool fat_too, bool indexed = false) {
    AgarCell* q = CELLP(c, P, k, ci);
    double cx = q->x, cy = q->y, cm = q->mass, cr = q->radius;
    const Rect rc = rect_of_call(P.S, cx, cy, cr); /* candidates are fixed before the cell grows */
    const bool by_index = W == 32 && indexed && cell_eats_pellets_indexed(c, P, k, ci, rc, cm, cr, q->uid);
    const int cap = by_index ? 0 : P.L.pellet_cap; /* the index served this cell: no scan of the pool */
    /* Integer window: a pellet can only be eaten if it lies within the cell's radius, and within one chunk of W
     * pellets the cell gains at most 3 W mass — so nothing outside |d| <= radius(mass + 3 W) + 2 matters for the
     * chunk at hand.  The window only skips chunks; hits are decided by the exact tests below.  It is
     * re-derived after every eat. */
    const int icx = (int)cx, icy = (int)cy;
    const bool windowed = cap > 8 * W; /* small pools: the window costs more than the chunks it skips (measured) */
    int reach = windowed ? (int)sqrt((cm + 3.0 * W) / M_PI) + 2 : 4096;
    for (int base = 0; base < cap; base += W) {
        int s = base + c.lane;
        uint32_t pk = s < cap ? c.pel[s] : 0u;
        int px = AGAR_PELLET_X(pk), py = AGAR_PELLET_Y(pk);
        bool win = pk != 0 && (unsigned)(px - icx + reach) <= (unsigned)(2 * reach) &&
                   (unsigned)(py - icy + reach) <= (unsigned)(2 * reach);
        if (windowed && !c.t.any(win)) continue;
        int pm = AGAR_PELLET_M(pk);
        bool cand = win && rect_hit(rc, pellet_rect(px, py));
        double pr = P.pellet_r[pm & 3];
        unsigned done_mask = 0; /* lanes at or below the last eaten one */
        while (true) {
            bool hit = cand && overlap(cx, cy, cm, cr, (double)px, (double)py, (double)pm, pr) && cm > 1.25 * (double)pm;
            unsigned b = c.t.ballot(hit) & ~done_mask;
            if (!b) break;
            int l = __ffs(b) - 1;
            int em = c.t.shfl(pm, l);
            /* every lane tracks the grown cell identically (grow(): cell.py:119-121) */
            double nm = cm + (double)em;
            if (!(nm < AG_MAX_MASS)) nm = AG_MAX_MASS;
            cm = nm;
            cr = radius_of_call(nm);
            if (c.lane == 0) {
                log_ev(c, P, AGAR_EV_EAT_PELLET, k, (int)q->uid, base + l, 0);
                c.pel[base + l] = 0;
                c.h->n_pellets -= 1;
            }
            done_mask |= (l == 31) ? 0xffffffffu : ((2u << l) - 1);
            if (windowed) reach = (int)sqrt((cm + 3.0 * W) / M_PI) + 2;
        }
    }
    if (fat_too) {
        const int fcap = P.L.fat_cap;
        for (int base = 0; base < fcap; base += W) {
            int s = base + c.lane;
            double fx = 0, fy = 0, fm = 0, fr = 0;
            if (s < fcap) fx = c.fat[s].x, fy = c.fat[s].y, fm = c.fat[s].mass, fr = c.fat[s].radius;
            bool cand = fm != 0 && rect_hit(rc, rect_of_call(P.S, fx, fy, fr));
            unsigned done_mask = 0;
            while (true) {
                bool hit = cand && overlap(cx, cy, cm, cr, fx, fy, fm, fr) && cm > 1.25 * fm;
                unsigned b = c.t.ballot(hit) & ~done_mask;
                if (!b) break;
                int l = __ffs(b) - 1;
                double em = c.t.shfl(fm, l);
                double nm = cm + em;
                if (!(nm < AG_MAX_MASS)) nm = AG_MAX_MASS;
                cm = nm;
                cr = radius_of_call(nm);
                if (c.lane == 0) {
                    log_ev(c, P, AGAR_EV_EAT_PELLET, k, (int)q->uid, (base + l) | 0x10000, 0);
                    AgarFatPellet z = {};
                    c.fat[base + l] = z;
                    c.h->n_fat -= 1;
                }
                done_mask |= (l == 31) ? 0xffffffffu : ((2u << l) - 1);
            }
        }
    }
    if (c.lane == 0 && cm != q->mass) q->mass = cm, q->radius = cr;
    c.t.sync();
}

/* lane 0; field.py:215-222 */
template <int W>
DEVN void player_blob_overlap_seq(Ctx<W>& c, const DevParams& P) {
    for (int k = 0; k < P.L.n_players; ++k) {
        AgarPlayer* p = &c.pl[k];
        if (!p->alive) continue;
        for (int ci = 0; ci < p->n_cells; ++ci) {
            AgarCell* q = CELLP(c, P, k, ci);
            Rect rc = rect_of_call(P.S, q->x, q->y, q->radius);
            int nb0 = c.h->n_blobs, removed = 0;
            for (int b0 = 0; b0 < nb0; ++b0) {
                int bi = b0 - removed;
                AgarMote* b = &c.blob[bi];
                if (!rect_hit(rc, rect_of_call(P.S, b->x, b->y, b->radius))) continue;
                if (overlap(q->x, q->y, q->mass, q->radius, b->x, b->y, b->mass, b->radius) && b->aux != q->uid &&
                    q->mass > 1.25 * b->mass) {
                    log_ev(c, P, AGAR_EV_EAT_BLOB, k, (int)q->uid, bi, (int)b->aux);
                    grow(q, b->mass);
                    blob_remove(c, bi);
                    removed += 1;
                }
            }
        }
    }
}

/* lane 0; field.py:233-244, :346-348 */
template <int W>
DEVN bool player_player_one_cell(Ctx<W>& c, const DevParams& P, int k, int ci) {
    /* lane 0: the reference's inner loops for ONE iterated cell (field.py:236-244).  Returns true if that cell was eaten (the
     * caller's ++ci then skips the cell that moved into its slot: Python's list iterator does the same). */
    const int K = P.L.n_players;
    AgarCell* q = CELLP(c, P, k, ci);
    uint32_t my_uid = q->uid;
    Rect rc = rect_of_call(P.S, q->x, q->y, q->radius);
    /* candidate snapshot: per enemy player a 16-bit mask over its cell list, taken before any eating;
     * enemy lists only shrink by this cell's own eating, tracked with `removed` per player */
    for (int k2 = 0; k2 < K; ++k2) {
        if (k2 == k) continue;
        AgarPlayer* p2 = &c.pl[k2];
        int n2 = p2->n_cells;
        unsigned cand = 0;
        for (int j = 0; j < n2; ++j) {
            const AgarCell* o = CELLP(c, P, k2, j);
            if ((o->flags & AGAR_CF_INHASH) && rect_hit(rc, rect_of_call(P.S, o->x, o->y, o->radius))) cand |= 1u << j;
        }
        int removed = 0;
        for (int j0 = 0; j0 < n2; ++j0) {
            if (!(cand >> j0 & 1)) continue;
            int j = j0 - removed;
            AgarCell* o = CELLP(c, P, k2, j);
            if (!overlap(q->x, q->y, q->mass, q->radius, o->x, o->y, o->mass, o->radius)) continue;
            if (q->mass > 1.25 * o->mass) {
                log_ev(c, P, AGAR_EV_EAT_CELL, k, (int)q->uid, k2, (int)o->uid);
                grow(q, o->mass);
                delete_player_cell(c, P, k2, j);
                removed += 1;
            } else if (o->mass > 1.25 * q->mass) {
                log_ev(c, P, AGAR_EV_EAT_CELL, k2, (int)o->uid, k, (int)my_uid);
                grow(o, q->mass);
                delete_player_cell(c, P, k, ci);
                return true;
            }
        }
    }
    return false;
}
/* cooperative; field.py:233-244.  The reference visits every cell of every player and tests it against its enemy candidates;
 * a visit changes nothing unless the cell OVERLAPS a candidate at that moment.  So the tile tests the visited cell against all
 * enemy cells at once (32 per step, the reference's own candidate + overlap predicates) and only hands the visit to the
 * sequential lane-0 body when some lane sees an overlap — a handful of visits per frame instead of cells x enemy cells
 * rectangle tests on one lane (the arena's largest lane-0 pass: up to 2 M cycles in the frames where it ran). */
template <int W>
DEV void player_player_overlap_seq(Ctx<W>& c, const DevParams& P) {
    const int K = P.L.n_players, cap = P.L.cell_cap;
    const bool use_live = K * cap > W;
    for (int k = 0; k < K; ++k) {
        if (!c.pl[k].alive) continue;
        for (int ci = 0; ci < c.pl[k].n_cells; ++ci) {
            const AgarCell* q = CELLP(c, P, k, ci);
            const double qx = q->x, qy = q->y, qm = q->mass, qr = q->radius;
            const Rect rc = rect_of_call(P.S, qx, qy, qr);
            const uint16_t* live = live_cells(c, P);
            const int n_it = c.n_live >= 0 ? c.n_live : K * cap;
            bool hit = false;
            for (int t = c.lane; t < n_it && !hit; t += W) {
                const int idx = c.n_live >= 0 ? (int)live[t] : t;
                const int k2 = idx >> P.cap_shift, j = idx - (k2 << P.cap_shift);
                if (k2 == k || j >= c.pl[k2].n_cells) continue;
                const AgarCell* o = CELLP(c, P, k2, j);
                if ((o->flags & AGAR_CF_INHASH) && rect_hit(rc, rect_of_call(P.S, o->x, o->y, o->radius)) &&
                    overlap(qx, qy, qm, qr, o->x, o->y, o->mass, o->radius))
                    hit = true;
            }
            if (!c.t.any(hit)) continue;
            int eaten = 0;
            if (c.lane == 0) eaten = player_player_one_cell(c, P, k, ci) ? 1 : 0;
            c.t.sync();
            if (use_live) build_live_cells(c, P); /* cells may have been removed */
            (void)eaten; /* an eaten cell left its slot: ++ci skips the one that moved in, exactly like the list iterator */
        }
    }
}

/* cooperative pre-checks: does ANY (cell, object) pair satisfy the eat predicate on the current state?  If not,
 * the sequential pass would change nothing (state only changes through a first hit) and is skipped. */
template <int W>
DEV bool any_player_mote_hit(Ctx<W>& c, const DevParams& P, const AgarMote* motes, int n, bool is_virus) {
    const int K = P.L.n_players, cap = P.L.cell_cap;
    bool hit = false;
    const uint16_t* live = live_cells(c, P);
    const int n_it = c.n_live >= 0 ? c.n_live : K * cap;
    if (n > 0)
        for (int t = c.lane; t < n_it && !hit; t += W) {
            int idx = c.n_live >= 0 ? (int)live[t] : t;
            int k = idx >> P.cap_shift, i = idx - (k << P.cap_shift);
            if (!c.pl[k].alive || i >= c.pl[k].n_cells) continue;
            const AgarCell* q = CELLP(c, P, k, i);
            for (int v = 0; v < n; ++v) {
                const AgarMote* m = &motes[v];
                if (overlap(q->x, q->y, q->mass, q->radius, m->x, m->y, m->mass, m->radius) && q->mass > 1.25 * m->mass &&
                    (is_virus || m->aux != q->uid)) {
                    hit = true;
                    break;
                }
            }
        }
    return c.t.any(hit);
}
template <int W>
DEV bool any_player_player_hit(Ctx<W>& c, const DevParams& P) {
    const int K = P.L.n_players, cap = P.L.cell_cap;
    bool hit = false;
    const uint16_t* live = live_cells(c, P);
    const int n_it = c.n_live >= 0 ? c.n_live : K * cap;
    for (int t = c.lane; t < n_it && !hit; t += W) {
        int idx = c.n_live >= 0 ? (int)live[t] : t;
        int k = idx >> P.cap_shift, i = idx - (k << P.cap_shift);
        if (!c.pl[k].alive || i >= c.pl[k].n_cells) continue;
        const AgarCell* q = CELLP(c, P, k, i);
        for (int k2 = k + 1; k2 < K && !hit; ++k2) {
            int n2 = c.pl[k2].n_cells;
            for (int j = 0; j < n2; ++j) {
                const AgarCell* o = CELLP(c, P, k2, j);
                if (overlap(q->x, q->y, q->mass, q->radius, o->x, o->y, o->mass, o->radius)) {
                    hit = true;
                    break;
                }
            }
        }
    }
    return c.t.any(hit);
}
template <int W>
DEV bool any_virus_blob_hit(Ctx<W>& c, const DevParams& P) {
    int nv = c.h->n_viruses, nb = c.h->n_blobs;
    bool hit = false;
    for (int idx = c.lane; idx < nv * nb && !hit; idx += W) {
        const AgarMote *v = &c.vir[idx / nb], *b = &c.blob[idx % nb];
        if (overlap(v->x, v->y, v->mass, v->radius, b->x, b->y, b->mass, b->radius)) hit = true;
    }
    return c.t.any(hit);
}

/* cooperative; field.py:85-92 */
template <int W, bool FULL>
DEV void field_update_phase(Ctx<W>& c, const DevParams& P, int phase) {
    /* the frame in AGAR_FIELD_PHASES pieces, so that the caller can put CTA barriers between them (the warps of a CTA
     * then fetch the same instructions together; see k_main) */
    if (phase == 0) {
        if (FULL) update_viruses_blobs(c, P);
        update_players<W, FULL>(c, P);
    } else if (phase == 1) {
        if (FULL) {
            /* mergePlayerCells: only players with >= 2 cells can merge */
            for (int k = 0; k < P.L.n_players; ++k) {
                /* any() is also the barrier that keeps lane 0's writes away from the other lanes' reads of n_cells */
                if (c.t.any(c.pl[k].alive && c.pl[k].n_cells > 1)) {
                    if (c.lane == 0) merge_player_cells_seq(c, P, k);
                    c.t.sync();
                }
            }
            if (c.h->n_viruses && c.h->n_blobs && any_virus_blob_hit(c, P)) {
                if (c.lane == 0) virus_blob_overlap_seq(c, P);
                c.t.sync();
            }
            const bool use_live = P.L.n_players * P.L.cell_cap > W; /* cells are stable from here to the seq passes */
            if (use_live && c.h->n_viruses > 0) build_live_cells(c, P);
            bool vh = any_player_mote_hit(c, P, c.vir, c.h->n_viruses, true);
            c.n_live = -1;
            if (vh) {
                if (c.lane == 0) player_virus_overlap_seq(c, P);
                c.t.sync();
            }
        }
    } else if (phase == 2) {
        /* playerPelletOverlap */
        if (!FULL) {
            cell_eats_pellets(c, P, 0, 0, false);
        } else {
            bool fat_too = P.L.fat_cap > 0;
            const bool indexed = W == 32 && pel_index_enabled(P);
            if (indexed) { /* index + a lane-per-cell pre-filter: only cells that may eat something run the cooperative ordered pass */
                build_pellet_index(c, P);
                build_live_cells(c, P);
                const uint16_t* live = live_cells(c, P);
                const int cap_c = P.L.cell_cap, n_live = c.n_live;
                uint16_t* fatlist = (uint16_t*)c.scratch + pel_index_cnt_len(P) + P.L.pellet_cap + 64;
                int n_fatl = 0;
                if (fat_too && c.h->n_fat > 0) { /* compact list of the live ex-blob pellets (few) */
                    for (int base = 0; base < P.L.fat_cap; base += W) {
                        const int sl = base + c.lane;
                        const bool on = sl < P.L.fat_cap && c.fat[sl].mass != 0;
                        const unsigned bal = c.t.ballot(on);
                        const int pos = n_fatl + __popc(bal & ((1u << c.lane) - 1u));
                        if (on && pos < 32) fatlist[pos] = (uint16_t)sl;
                        n_fatl += __popc(bal);
                    }
                    c.t.sync();
                }
                const bool fat_unknown = n_fatl > 32;
                for (int base = 0; base < n_live; base += W) {
                    const int t = base + c.lane;
                    const int idx = t < n_live ? (int)live[t] : 0;
                    const bool may = t < n_live && cell_may_eat(c, P, idx >> P.cap_shift, idx & (cap_c - 1), fatlist, fat_unknown ? 0 : n_fatl, fat_unknown);
                    unsigned todo = c.t.ballot(may);
                    while (todo) { /* canonical order: ascending (player, cell) */
                        const int l = __ffs(todo) - 1;
                        todo &= todo - 1;
                        const int id = c.t.shfl(idx, l);
                        cell_eats_pellets(c, P, id >> P.cap_shift, id & (cap_c - 1), fat_too && c.h->n_fat > 0, true);
                    }
                }
                c.n_live = -1;
            } else {
                for (int k = 0; k < P.L.n_players; ++k) {
                    if (!c.pl[k].alive) continue;
                    for (int ci = 0; ci < c.pl[k].n_cells; ++ci) cell_eats_pellets(c, P, k, ci, fat_too && c.h->n_fat > 0, false);
                }
            }
        }
    } else {
        if (FULL) {
            /* pellet and blob eating change masses, not the set of cells: one live list serves both pre-checks */
            if (P.L.n_players * P.L.cell_cap > W && (c.h->n_blobs > 0 || P.L.n_players > 1)) build_live_cells(c, P);
            if (any_player_mote_hit(c, P, c.blob, c.h->n_blobs, false)) {
                if (c.lane == 0) player_blob_overlap_seq(c, P);
                c.t.sync();
            }
            bool ph = P.L.n_players > 1 && any_player_player_hit(c, P);
            if (ph) {
                player_player_overlap_seq(c, P); /* keeps the live-cell list current while cells are eaten */
                c.t.sync();
            }
            c.n_live = -1;
        }
        spawn_stuff<W, FULL>(c, P);
    }
}
#define AGAR_FIELD_PHASES 4
