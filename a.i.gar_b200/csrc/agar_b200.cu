/*
 * agar_b200.cu — kernels + the C ABI (include/agar_b200.h) of the B200-native batched agar.io step.
 * Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -fmad=false -shared -Xcompiler -fPIC
 * No torch, no CPU fallback: every entry point runs CUDA kernels on the handle's device or fails.
 */
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/agar_b200.h"
#include "../../include/agar_layout.h"
#include "agar_bots.cuh"
#include "agar_dev.cuh"
#include "agar_simple.cuh"

extern __shared__ __align__(16) uint8_t g_smem[];

/* ------------------------------------------------------------------ staging: HBM <-> shared memory, whole CTA */
__device__ __forceinline__ void stage_in(const DevParams& P, const uint8_t* state, int env0, int n_here, bool zero) {
    const int chunks = (int)(P.L.record_bytes / 8);
    const int total = n_here * chunks;
    const uint2* src = (const uint2*)(state + (size_t)env0 * P.L.record_bytes);
    for (int i = threadIdx.x; i < total; i += blockDim.x) {
        int e = i / chunks, w = i - e * chunks;
        uint2 v = zero ? make_uint2(0u, 0u) : src[i];
        ((uint2*)(g_smem + (size_t)e * P.rec_stride))[w] = v;
    }
    __syncthreads();
}
__device__ __forceinline__ void stage_out(const DevParams& P, uint8_t* state, int env0, int n_here) {
    __syncthreads();
    const int chunks = (int)(P.L.record_bytes / 8);
    const int total = n_here * chunks;
    uint2* dst = (uint2*)(state + (size_t)env0 * P.L.record_bytes);
    for (int i = threadIdx.x; i < total; i += blockDim.x) {
        int e = i / chunks, w = i - e * chunks;
        dst[i] = ((const uint2*)(g_smem + (size_t)e * P.rec_stride))[w];
    }
}
/* FULL kernels ("hot sections"): big records stay in HBM / L2; what every scan and every lane-0 step reads is cached in
 * shared memory — the pellet pool, and with hot_a > 0 also bytes [0, hot_a) = header, players, cells, viruses */
__device__ __forceinline__ int hot_a_bytes(const DevParams& P) { return (P.hot_a + 15) / 16 * 16; }
__device__ __forceinline__ int pel_cache_bytes(const DevParams& P) { return hot_a_bytes(P) + (P.L.pellet_cap * 4 + 15) / 16 * 16; }
__device__ __forceinline__ void pel_cache_copy(const DevParams& P, uint8_t* state, int env0, int n_here, int tiles, bool in) {
    const int wa = P.hot_a / 4, words = wa + P.L.pellet_cap;
    for (int i = threadIdx.x; i < n_here * words; i += blockDim.x) {
        int e = i / words, w = i - e * words;
        uint8_t* rec = state + (size_t)(env0 + e) * P.L.record_bytes;
        uint8_t* hot = g_smem + (size_t)tiles * P.scratch_bytes + (size_t)e * pel_cache_bytes(P);
        uint32_t* g = w < wa ? (uint32_t*)rec + w : (uint32_t*)(rec + P.L.off_pellets) + (w - wa);
        uint32_t* s = w < wa ? (uint32_t*)hot + w : (uint32_t*)(hot + hot_a_bytes(P)) + (w - wa);
        if (in) *s = *g; else *g = *s;
    }
    __syncthreads();
}
/* where a record lives during a launch: !FULL (the single-cell general kernel) stages the whole record in shared memory
 * (stage_in / stage_out); FULL keeps it in HBM / L2 and caches the hot sections (pel_cache_copy) */
template <int W, bool FULL>
__device__ __forceinline__ void bind_ctx(Ctx<W>& c, const DevParams& P, int tile_id, int tiles, int env, uint8_t* state) {
    c.lane = c.t.thread_rank();
    c.env_id = (uint32_t)(P.first_env + (uint64_t)env);
    c.rec = FULL ? state + (size_t)env * P.L.record_bytes : g_smem + (size_t)tile_id * P.rec_stride;
    c.h = (AgarEnvHeader*)(c.rec + P.L.off_header);
    c.pl = (AgarPlayer*)(c.rec + P.L.off_players);
    c.cells = (AgarCell*)(c.rec + P.L.off_cells);
    c.vir = (AgarMote*)(c.rec + P.L.off_viruses);
    c.blob = (AgarMote*)(c.rec + P.L.off_blobs);
    c.fat = (AgarFatPellet*)(c.rec + P.L.off_fat);
    c.pel = (uint32_t*)(c.rec + P.L.off_pellets);
    c.hist = (float*)(c.rec + P.L.off_hist);
    c.ev = (AgarEvent*)(c.rec + P.L.off_events);
    c.scratch = g_smem + (FULL ? 0 : (size_t)tiles * P.rec_stride) + (size_t)tile_id * P.scratch_bytes;
    if (FULL) {
        uint8_t* hot = g_smem + (size_t)tiles * P.scratch_bytes + (size_t)tile_id * pel_cache_bytes(P);
        c.pel = (uint32_t*)(hot + hot_a_bytes(P));
        if (P.hot_a) { /* hot_a = off_blobs: header, players, cells, viruses are contiguous from byte 0 of the record */
            c.h = (AgarEnvHeader*)(hot + P.L.off_header);
            c.pl = (AgarPlayer*)(hot + P.L.off_players);
            c.cells = (AgarCell*)(hot + P.L.off_cells);
            c.vir = (AgarMote*)(hot + P.L.off_viruses);
        }
    }
}

#ifdef AGAR_PHASE_CLOCKS
/* debug build only (tools/phase_clocks.py): cycles each env's tile spent per frame phase, summed over the launch */

#define CLK_MARK(slot)                                                      \
    do {                                                                    \
        if (active) clk_mark(c, slot);                                      \
    } while (0)
extern "C" int agar_debug_read_clocks(unsigned long long* host, int n_envs, int reset) {
    if (cudaMemcpyFromSymbol(host, g_clk, (size_t)n_envs * 16 * 8) != cudaSuccess) return -1;
    if (reset) {
        void* p = nullptr;
        cudaGetSymbolAddress(&p, g_clk);
        cudaMemset(p, 0, sizeof(unsigned long long) * 32768 * 16);
    }
    return 0;
}
#else
#define CLK_MARK(slot) do { } while (0)
#endif

/* ------------------------------------------------------------------ the step kernel */
template <int W, bool FULL, int MAXT>
/* minBlocks = 1 matters for the multi-agent kernels: with maxThreads alone ptxas budgets for two 512-thread CTAs per SM
 * (64 registers, 540 bytes of spills); one CTA per SM is what their shared memory allows anyway -> 112-116 registers, no
 * spills (measured +11 % config 3, +7 % config 4).  The single-cell general kernel runs many small CTAs per SM and keeps
 * the 64-register budget (measured -13 % at 65536 envs with 125 registers).  MAXT = 1024: 32 envs per CTA when their hot
 * sections fit (1-vs-greedy config): twice the warps walking the frame body in lock-step is worth more (+26 %) than the
 * registers (64, with spills). */
__global__ void __launch_bounds__(MAXT, (FULL || MAXT > 512) ? 1 : 2)
k_main(const __grid_constant__ DevParams P, uint8_t* __restrict__ state, const float* __restrict__ actions,
       float* __restrict__ obs, int n_frames, int n_dec, int flags, uint32_t dec_base) {
    const int tiles = blockDim.x / W;
    const int env0 = blockIdx.x * tiles;
    const int n_here = min(tiles, P.n_envs - env0);
    if (FULL) pel_cache_copy(P, state, env0, n_here, tiles, true);
    else stage_in(P, state, env0, n_here, false);
    const int tile_id = threadIdx.x / W;
    const bool active = tile_id < n_here;
    {
        Ctx<W> c(cg::tiled_partition<W>(cg::this_thread_block()));
        const int env = env0 + (active ? tile_id : 0);
        bind_ctx<W, FULL>(c, P, active ? tile_id : 0, tiles, env, state);
        const int A = P.L.n_agents, K = P.L.n_players, SL = P.L.state_len;
        float* obs_env = obs ? obs + (size_t)env * A * SL : nullptr;
        /* One loop with ONE call site per helper: the multi-agent frame is ~22 k SASS instructions and instruction
         * fetch is its top stall (profiles/r01_k_main_cfg3_*), so nothing big may be inlined twice.  Iteration `it` is
         * frame f of decision d; the trailing observation (KF_OBS_AFTER) is one extra iteration without a frame.
         * FULL: CTA barriers at frame start and before the field update keep all warps of the CTA in the same code
         * region, so the instruction cache serves them together (idle tiles of a partly filled CTA only hit the
         * barriers; measured 2.5x, DESIGN §4). */
        const int total = n_dec * n_frames;
        for (int it = 0; it <= total; ++it) {
            const bool last = it == total;
            if (last && !(flags & KF_OBS_AFTER)) break;
#ifdef AGAR_PHASE_CLOCKS
            c.clk_t = clock64(), c.clk_env = env;
#endif
            if (FULL) __syncthreads();
            CLK_MARK(0); /* (ptxas hoists this clock read above the barrier: the wait lands in the NEXT slot, the fov pass) */
            const int f = n_frames > 0 ? it % n_frames : 0, d = n_frames > 0 ? it / n_frames : 0;
            const bool emit = last || (f == 0 && (flags & KF_OBS_BEFORE)); /* observations leave the kernel here */
            if (active && !last && c.lane == 0) c.h->n_events = 0;
            if (FULL && K > 1 && active && !last) { /* every alive player's turn below would compute its own, on lane 0 */
                update_all_fovs(c, P);
                c.fov_done = true;
                CLK_MARK(8); /* fov pass */
                if (K * P.L.cell_cap > W) build_live_cells(c, P); /* one iteration covers all slots otherwise */
                CLK_MARK(11); /* live-cell list */
            }
            for (int k = 0; k < K; ++k) {
                if (active) {
                    if (!FULL || P.cfg.bot_type[k] == AGAR_BOT_NN) {
                        nn_turn_begin<W, FULL>(c, P, k, (emit && obs_env) ? obs_env + (size_t)k * SL : nullptr);
                        if (last) continue;
                        if (c.lane == 0) {
                            float act[4] = {0.f, 0.f, 0.f, 0.f};
                            if (c.pl[k].bot.need_action) {
                                if (flags & KF_RANDOM_ACTIONS) { /* random-action driver (SURVEY §8d config 2) */
                                    uint32_t w[4];
                                    philox(dec_base + (uint32_t)d, 7u, c.env_id, (uint32_t)k, (uint32_t)P.seed,
                                           (uint32_t)(P.seed >> 32), w);
                                    for (int i = 0; i < 4; ++i) act[i] = (float)(w[i] >> 8) * (1.0f / 16777216.0f);
                                } else {
                                    const float* ap = actions + ((size_t)env * A + k) * 4;
                                    for (int i = 0; i < 4; ++i) act[i] = ap[i];
                                }
                            }
                            nn_turn_end(c, P, k, act);
                        }
                        c.t.sync();
                    } else if (FULL && !last) {
                        CLK_MARK(1); /* NN turns so far */
                        scripted_turn(c, P, k);
                        CLK_MARK(7); /* scripted (greedy / random) turns */
                    }
                }
            }
            if (last) break;
            CLK_MARK(1); /* bot turns */
            c.fov_done = false, c.n_live = -1;
            for (int ph = 0; ph < AGAR_FIELD_PHASES; ++ph) {
                if (FULL && ph == 0) __syncthreads();
                if (ph == 0) CLK_MARK(2); /* wait at the field barrier */
                if (active) field_update_phase<W, FULL>(c, P, ph);
                CLK_MARK(3 + ph); /* 3: viruses / blobs / players  4: merge, virus overlaps  5: pellets  6: blobs, player-player, spawn */
            }
            if (active) {
                if (c.lane == 0) c.h->frame += 1;
                c.t.sync();
            }
            CLK_MARK(12); /* frame tail */
        }
        if (active && c.lane == 0 && (P.turn_reward || P.turn_done))
            for (int a = 0; a < A; ++a) {
                if (P.turn_reward) P.turn_reward[(size_t)env * A + a] = (float)c.pl[a].bot.last_reward;
                if (P.turn_done) P.turn_done[(size_t)env * A + a] = (uint8_t)c.pl[a].bot.exp_done;
            }
    }
    if (FULL) {
        __syncthreads();
        pel_cache_copy(P, state, env0, n_here, tiles, false);
    } else
        stage_out(P, state, env0, n_here);
    export_tail(P, obs, env0, n_here);
}


/* ------------------------------------------------------------------ register-resident kernel (agar_simple.cuh) */
struct SimplePlan {
    int strideB; /* bytes between the staged [pellets .. end of record] regions of consecutive envs */
    int grid_off; /* byte offset of the env's G x G observation accumulator inside its region; 0: accumulate in the caller's row */
    int obs_warps; /* observer warps at the end of the CTA (0: every warp steps envs and encodes its own observations) */
    int snap_off; /* byte offset of the two snapshot buffers (observer launches): after the envs' regions */
    int snap_stride; /* bytes per env in one snapshot buffer: SimpleSnap + the pellet pool */
};

/* Observer warps (launches that hand decision observations off, see plan_observers): at each decision the physics warps
 * copy the env's pellet pool and the four values s_encode reads into a snapshot slot and go straight on to the frames;
 * the observer warps bin the snapshot into the env's row meanwhile.  Nothing the frames read depends on the grid, and the
 * pool changes only in s_field_update, so the row is the one the inline encoder would have written at that moment.
 * Two snapshot buffers (decision d uses buffer d & 1), each with a FULL / EMPTY named-barrier pair:
 *   physics:  [d >= 2: bar.sync EMPTY[b]]  fill b  bar.arrive FULL[b]
 *   observer: bar.sync FULL[b]  encode b  [d + 2 < n_dec: bar.arrive EMPTY[b]]
 * so every barrier instance gets exactly (physics + observer threads) arrivals.  ID 0 stays __syncthreads. */
enum { SB_PHYS = 1, SB_FULL = 2, SB_EMPTY = 4 }; /* named barrier IDs: SB_FULL + b, SB_EMPTY + b for buffer b */
struct SimpleSnap {
    double fov_x, fov_y, fov_size, mass;
    int32_t out; /* a row is stored (the env observes at this decision and is not a spare slot) */
    int32_t pad;
};
/* CTA size bound of k_simple<W, true>: the physics warps plus the observers.  W = 8: 11 warps, one CTA per SM
 * (ptxas budgets the bound rounded up to 12 warps: 168 registers; CUDA 12.9 allocates 167, no spills — 176 without the
 * bound).  W = 4 needs 188-192 registers and spills under that budget, so it keeps 8 warps (4 + 4, 255 registers). */
__host__ __device__ constexpr int simple_max_threads(int W) { return W == 8 ? 352 : 256; }
constexpr int SIMPLE_OBS_MIN_FRAMES = 4; /* frames per handed-off observation below which the inline encoder stays (measured) */
constexpr int SIMPLE_OBS_LANES = 4;      /* lanes per env of the observer warps */
constexpr int SIMPLE_OBS_WARPS = 4;      /* observer warps per CTA */

/* immediate IDs: ptxas then reserves the barriers used, not all 16 */
template <int ID>
DEV void named_bar_sync(int n) { asm volatile("bar.sync %0, %1;" ::"n"(ID), "r"(n) : "memory"); }
template <int ID>
DEV void named_bar_arrive(int n) { asm volatile("bar.arrive %0, %1;" ::"n"(ID), "r"(n) : "memory"); }

/* one lane per env is throughput-bound: cap registers at 128 for 8 CTAs / SM (measured +10..50 % at >= 64k envs);
 * wider tiles are latency-bound at small env counts and prefer the uncapped allocation (measured) */
template <int W, bool OBSW> /* OBSW: the observer-warp launch (plan_observers); false: the inline encoder, CTA barrier per frame */
__global__ void __launch_bounds__(OBSW ? simple_max_threads(W) : 256, W == 1 ? 2 : 1)
k_simple(const __grid_constant__ DevParams P, const SimplePlan SP, uint8_t* __restrict__ state, const float* __restrict__ actions,
         float* __restrict__ obs, int n_frames, int n_dec, int flags, uint32_t dec_base) {
    const int phys_threads = blockDim.x - 32 * SP.obs_warps; /* the one place the barrier counts come from */
    const int per = phys_threads / W; /* envs per CTA */
    const int env0 = blockIdx.x * per;
    const int n_here = min(per, P.n_envs - env0);
    const int rec_words = (int)(P.L.record_bytes / 4), pel_word = (int)(P.L.off_pellets / 4);
    const int tail_words = rec_words - pel_word;
    {   /* stage the pellet pool (+ event ring) in: coalesced 4-byte words; spare slots replicate the last env so that
         * every lane of a partly filled warp runs well-defined work */
        for (int i = threadIdx.x; i < per * tail_words; i += blockDim.x) {
            int e = i / tail_words, w = i - e * tail_words;
            int es = e < n_here ? e : n_here - 1;
            const uint32_t* src = (const uint32_t*)(state + (size_t)(env0 + es) * P.L.record_bytes) + pel_word;
            *(uint32_t*)(g_smem + (size_t)e * SP.strideB + w * 4) = src[w];
        }
    }
    __syncthreads();
    auto snap = [&](int buf, int e) { return g_smem + SP.snap_off + (size_t)(buf * per + e) * SP.snap_stride; };
    if (OBSW && (int)threadIdx.x >= phys_threads) { /* observer warps */
        constexpr int WO = SIMPLE_OBS_LANES;
        const int ot = ((int)threadIdx.x - phys_threads) / WO, osub = threadIdx.x % WO, n_ot = 32 * SP.obs_warps / WO;
        for (int d = 0; d < n_dec; ++d) {
            const int buf = d & 1;
            if (buf) named_bar_sync<SB_FULL + 1>(blockDim.x);
            else named_bar_sync<SB_FULL>(blockDim.x);
            /* static env -> observer tile map: each env's rows are stored by one tile, in decision order, and its G x G
             * accumulator has one user */
            for (int base = 0; base < per; base += n_ot) { /* warp-uniform trip count */
                const int e = min(base + ot, per - 1);
                const SimpleSnap* sn = (const SimpleSnap*)snap(buf, e);
                SReg r;
                r.fov_x = sn->fov_x, r.fov_y = sn->fov_y, r.fov_size = sn->fov_size, r.mass = sn->mass;
                SPtr q;
                q.pel = (uint32_t*)(sn + 1);
                q.grid = (uint32_t*)(g_smem + (size_t)e * SP.strideB + SP.grid_off);
                const bool out = base + ot < per && sn->out != 0;
                s_encode<WO>(r, q, P, out, out ? obs + (size_t)(env0 + e) * P.L.state_len : nullptr, osub);
            }
            if (d + 2 < n_dec) {
                if (buf) named_bar_arrive<SB_EMPTY + 1>(blockDim.x);
                else named_bar_arrive<SB_EMPTY>(blockDim.x);
            }
        }
        if (flags & KF_OBS_AFTER) __syncthreads(); /* drained: the physics warps' trailing observation may use the grids */
    } else { /* physics warps */
        const int slot = threadIdx.x / W, sub = threadIdx.x % W;
        const bool valid = slot < n_here;
        const int env = env0 + (valid ? slot : n_here - 1);
        const uint32_t env_id = (uint32_t)(P.first_env + (uint64_t)env);
        uint8_t* rec = state + (size_t)env * P.L.record_bytes;
        uint8_t* b = g_smem + (size_t)slot * SP.strideB;
        SPtr q;
        q.h = (AgarEnvHeader*)(rec + P.L.off_header);
        q.p = (AgarPlayer*)(rec + P.L.off_players);
        q.c = (AgarCell*)(rec + P.L.off_cells);
        q.pel = (uint32_t*)b;
        q.ev = (AgarEvent*)(b + (P.L.off_events - P.L.off_pellets));
        q.grid = SP.grid_off ? (uint32_t*)(b + SP.grid_off) : nullptr;
        SReg r;
        s_load(r, q);
        float* row = (obs != nullptr && valid) ? obs + (size_t)env * P.L.state_len : nullptr;
        /* one barrier per frame: the warps of a CTA walk the ~5000-instruction frame body together (measured 1.9x at 1M envs
         * and 2.3x at 4096); the physics warps only, observers keep their own pace */
        auto frame_bar = [&]() {
            if (OBSW) named_bar_sync<SB_PHYS>(phys_threads);
            else __syncthreads();
        };
        for (int d = 0; d < n_dec; ++d) {
            if (OBSW && SP.obs_warps) { /* hand the observation off (the host sets obs_warps only with KF_OBS_BEFORE and a row buffer) */
                const int d_o = s_turn_begin(r, P);
                if (d_o) s_observe_state(r, P);
                const int buf = d & 1;
                if (d >= 2) {
                    if (buf) named_bar_sync<SB_EMPTY + 1>(blockDim.x);
                    else named_bar_sync<SB_EMPTY>(blockDim.x);
                }
                uint8_t* sn = snap(buf, slot);
                uint32_t* pool = (uint32_t*)(sn + sizeof(SimpleSnap));
                for (int i = sub; i < P.L.pellet_cap; i += W) pool[i] = q.pel[i];
                if (sub == 0) {
                    SimpleSnap* h = (SimpleSnap*)sn;
                    h->fov_x = r.fov_x, h->fov_y = r.fov_y, h->fov_size = r.fov_size, h->mass = r.mass;
                    h->out = d_o != 0 && row != nullptr;
                }
                if (buf) named_bar_arrive<SB_FULL + 1>(blockDim.x);
                else named_bar_arrive<SB_FULL>(blockDim.x);
            } else if (flags & KF_OBS_BEFORE) {
                int d_o = s_turn_begin(r, P);
                s_observe<W>(r, q, P, d_o != 0, row, sub);
            }
            for (int f = 0; f < n_frames; ++f) {
                frame_bar();
                r.n_events = 0;
                int d_o = s_turn_begin(r, P);
                s_observe<W>(r, q, P, d_o != 0, nullptr, sub);
                float act[4] = {0.f, 0.f, 0.f, 0.f};
                if (r.need_action) {
                    if (flags & KF_RANDOM_ACTIONS) {
                        uint32_t w[4];
                        philox(dec_base + (uint32_t)d, 7u, env_id, 0u, (uint32_t)P.seed, (uint32_t)(P.seed >> 32), w);
                        for (int i = 0; i < 4; ++i) act[i] = (float)(w[i] >> 8) * (1.0f / 16777216.0f);
                    } else {
                        const float* ap = actions + (size_t)env * 4;
                        for (int i = 0; i < 4; ++i) act[i] = ap[i];
                    }
                }
                double speed_pow;
                s_turn_end<W>(r, P, act, sub, speed_pow);
                s_field_update<W>(r, q, P, env_id, sub, speed_pow);
            }
        }
        if (flags & KF_OBS_AFTER) {
            if (OBSW) __syncthreads(); /* the observers have stored every handed-off row and left the grid accumulators */
            int d_o = s_turn_begin(r, P);
            s_observe<W>(r, q, P, d_o != 0, row, sub);
        }
        if (valid && sub == 0) {
            s_store(r, q);
            if (P.turn_reward) P.turn_reward[env] = (float)r.last_reward; /* Bot.getLastReward / done of this turn, fused */
            if (P.turn_done) P.turn_done[env] = (uint8_t)r.exp_done;
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n_here * tail_words; i += blockDim.x) { /* stage the pools out */
        int e = i / tail_words, w = i - e * tail_words;
        uint32_t* dst = (uint32_t*)(state + (size_t)(env0 + e) * P.L.record_bytes) + pel_word;
        dst[w] = *(const uint32_t*)(g_smem + (size_t)e * SP.strideB + w * 4);
    }
    export_tail(P, obs, env0, n_here);
}

/* mode 0: Model(...) + createBot*K + Model.initialize (model.py:51,154-162,90-94; field.py:57-67)
 * mode 1: Model.resetModel -> Field.reset (field.py:69-83)      mode 2: Model.resetBots (bot.py:125-164) */
template <int W, bool FULL>
__global__ void __launch_bounds__(1024)
k_init(const __grid_constant__ DevParams P, uint8_t* __restrict__ state, const uint8_t* __restrict__ mask, int mode) {
    const int tiles = blockDim.x / W;
    const int env0 = blockIdx.x * tiles;
    const int n_here = min(tiles, P.n_envs - env0);
    if (FULL) {
        if (mode == 0) { /* records stay in HBM: clear them in place */
            const int chunks = (int)(P.L.record_bytes / 8);
            uint2* dst = (uint2*)(state + (size_t)env0 * P.L.record_bytes);
            for (int i = threadIdx.x; i < n_here * chunks; i += blockDim.x) dst[i] = make_uint2(0u, 0u);
            __syncthreads();
        }
        pel_cache_copy(P, state, env0, n_here, tiles, true);
    } else
        stage_in(P, state, env0, n_here, mode == 0);
    const int tile_id = threadIdx.x / W;
    if (tile_id < n_here && (mask == nullptr || mode == 0 || mask[env0 + tile_id])) {
        Ctx<W> c(cg::tiled_partition<W>(cg::this_thread_block()));
        bind_ctx<W, FULL>(c, P, tile_id, tiles, env0 + tile_id, state);
        const int K = P.L.n_players;
        if (mode == 0 || mode == 1) {
            if (mode == 1) { /* clear pools cooperatively: fresh lists and hash tables */
                for (int i = c.lane; i < P.L.pellet_cap; i += W) c.pel[i] = 0;
                AgarFatPellet zf = {};
                for (int i = c.lane; i < P.L.fat_cap; i += W) c.fat[i] = zf;
                AgarMote zm = {};
                for (int i = c.lane; i < P.L.blob_cap; i += W) c.blob[i] = zm;
                for (int i = c.lane; i < P.L.virus_cap; i += W) c.vir[i] = zm;
                c.t.sync();
            }
            if (c.lane == 0) {
                if (mode == 0) {
                    for (int k = 0; k < K; ++k) {
                        AgarPlayer* p = &c.pl[k];
                        p->alive = 1;
                        p->cmd_x = p->cmd_y = -1;
                        p->bot.type = P.cfg.bot_type[k];
                    }
                } else {
                    c.h->n_events = 0;
                    c.h->n_pellets = c.h->n_fat = c.h->n_blobs = c.h->n_viruses = 0;
                    c.h->n_dead = 0;
                    for (int i = 0; i < AGAR_MAX_PLAYERS; ++i) c.h->dead_order[i] = 0;
                    for (int k = 0; k < K; ++k)
                        for (int i = 0; i < c.pl[k].n_cells; ++i) CELLP(c, P, k, i)->flags &= ~AGAR_CF_INHASH;
                    c.h->frame = 0;
                }
                c.h->event_hash = 0xCBF29CE484222325ULL;
                for (int k = 0; k < K; ++k) initialize_player(c, P, k);
            }
            c.t.sync();
            spawn_pellets(c, P);
            if (c.lane == 0) {
                if (P.cfg.virus_enabled) spawn_viruses(c, P);
                if (c.h->n_dead) spawn_players(c, P);
            }
            c.t.sync();
        }
        if (mode == 0 || mode == 2) {
            if (c.lane == 0)
                for (int k = 0; k < K; ++k) bot_reset(c, P, k);
            const int nh = P.L.n_agents * P.L.n_hist * P.L.grid_squares * P.L.grid_squares;
            for (int i = c.lane; i < nh; i += W) c.hist[i] = 0.f;
            c.t.sync();
        }
    }
    if (FULL) {
        __syncthreads();
        pel_cache_copy(P, state, env0, n_here, tiles, false);
    } else
        stage_out(P, state, env0, n_here);
}

/* agar_get: one thread per (env, agent) or per env, straight from HBM */
__global__ void k_get(const __grid_constant__ DevParams P, const uint8_t* __restrict__ state, int which, void* out) {
    const int A = P.L.n_agents;
    const int per_env = (which == AGAR_GET_OVERFLOW || which == AGAR_GET_EVENT_HASH);
    const int n = per_env ? P.n_envs : P.n_envs * A;
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int env = per_env ? i : i / A, a = per_env ? 0 : i - env * A;
    const uint8_t* rec = state + (size_t)env * P.L.record_bytes;
    const AgarEnvHeader* h = (const AgarEnvHeader*)(rec + P.L.off_header);
    const AgarPlayer* p = (const AgarPlayer*)(rec + P.L.off_players) + a;
    const AgarCell* cells = (const AgarCell*)(rec + P.L.off_cells) + (size_t)a * P.L.cell_cap;
    switch (which) {
    case AGAR_GET_REWARD: ((float*)out)[i] = (float)p->bot.last_reward; break;
    case AGAR_GET_DONE: ((uint8_t*)out)[i] = (uint8_t)p->bot.exp_done; break;
    case AGAR_GET_VALID: ((uint8_t*)out)[i] = (uint8_t)p->bot.exp_valid; break;
    case AGAR_GET_NEED_ACTION: ((uint8_t*)out)[i] = (uint8_t)p->bot.need_action; break;
    case AGAR_GET_MASS: {
        int nc = p->n_cells;
        ((float*)out)[i] = nc ? (float)np_sum([&](int j) { return cells[j].mass; }, nc) : 0.f;
        break;
    }
    case AGAR_GET_FOV: ((float*)out)[i] = (float)p->fov_size; break;
    case AGAR_GET_NCELLS: ((int32_t*)out)[i] = p->n_cells; break;
    case AGAR_GET_ALIVE: ((uint8_t*)out)[i] = (uint8_t)p->alive; break;
    case AGAR_GET_STATS: {
        double* o = (double*)out + (size_t)i * 4;
        o[0] = p->bot.stat_mass_sum, o[1] = p->bot.stat_mass_max, o[2] = p->bot.stat_frames, o[3] = p->bot.stat_deaths;
        break;
    }
    case AGAR_GET_OVERFLOW: ((uint32_t*)out)[i] = h->overflow; break;
    case AGAR_GET_EVENT_HASH: ((uint64_t*)out)[i] = h->event_hash; break;
    }
}

/* ------------------------------------------------------------------ host side */
struct LaunchShape {
    int W;       /* lanes per env */
    int tiles;   /* envs per CTA (0: the shape does not fit) */
    int threads; /* CTA size; k_simple with observer warps: tiles * W physics threads + the observers */
    size_t smem; /* dynamic shared memory */
};
struct AgarEnv {
    AgarConfig cfg;
    AgarLayout L;
    DevParams P;
    uint8_t* state;
    double* deg_tab;
    int n_envs, device, full;
    LaunchShape init; /* k_init<32, FULL> */
    LaunchShape step; /* k_simple<W, false> if `simple`, else k_main<W, FULL> */
    int simple;
    SimplePlan sp;
    SimplePlan sp_obs; /* observer launches of k_simple (plan_observers); obs.threads == 0: none */
    LaunchShape obs;
    int64_t launches;
    int64_t observer_launches; /* launches of k_simple<W, true> */
    char err[256];
    /* step_host staging */
    float *d_actions, *d_obs, *d_reward;
    uint8_t* d_done;
    void* h_turn; /* pinned: float reward[EA] | uint8 done[EA], then (64-byte aligned) the completion flag word */
    volatile uint32_t* h_flag; /* inside h_turn's allocation; the last CTA of a zero-copy step launch writes flag_seq there */
    unsigned int* d_export_count;
    uint32_t flag_seq;
    int host_polling; /* the pending step raises h_flag (zero-copy path) */
    int host_pending; /* agar_step_host_begin issued, _end not yet */
};
static char g_create_err[256] = "";

static int fail(AgarEnv* e, int code, const char* fmt, const char* detail) {
    char* dst = e ? e->err : g_create_err;
    snprintf(dst, 256, fmt, detail);
    return code;
}
#define CU(call)                                                                 \
    do {                                                                         \
        cudaError_t _e = (call);                                                 \
        if (_e != cudaSuccess) return fail(env, AGAR_E_CUDA, "CUDA error: %s", cudaGetErrorString(_e)); \
    } while (0)

extern "C" int agar_layout_for_config(const AgarConfig* cfg, AgarLayout* out) {
    if (!cfg || !out) return AGAR_E_INVALID;
    return agar_layout_compute(cfg, out);
}

static bool config_is_simple(const AgarConfig& c, const AgarLayout& L) {
    return c.n_players == 1 && c.bot_type[0] == AGAR_BOT_NN && !c.virus_enabled && !c.enable_split && !c.enable_eject &&
           c.pellet_grid && /* s_encode always writes the G x G pellet grid in front of the extras */
           L.cell_cap == 1 && !c.self_grid && !c.wall_grid && !c.enemy_grid && !c.virus_grid && !c.self_grid_lf &&
           !c.self_grid_slf && !c.enemy_grid_lf && !c.enemy_grid_slf && !c.use_last_action && !c.use_second_last_action &&
           !c.use_last_fovsize && L.n_hist == 0 && !c.all_player_grid && !c.simple_state && /* the 12-value representation lives in the general kernel */
           L.field_size < 128; /* the float32 candidate filter of k_simple's eat chain is analysed for coordinates below 128 (one player: 75) */
}

/* launch shape of k_init / k_main for tile width W (bind_ctx's shared-memory layout); tiles == 0: one record does not fit */
static LaunchShape plan_launch(const AgarEnv* e, int W) {
    const size_t budget = 200 * 1024;
    const size_t per_tile = (size_t)e->P.scratch_bytes +
                            (e->full ? (size_t)((e->P.hot_a + 15) / 16 * 16) + (size_t)((e->L.pellet_cap * 4 + 15) / 16 * 16)
                                     : (size_t)e->P.rec_stride);
    const int max_threads = (e->full && W == 32) ? 1024 : 512; /* k_main<32, true, 1024> exists for 32-lane tiles only */
    int tiles = e->full ? max_threads / W : 128 / W; /* as many envs per CTA as fit: the barriers then align more warps */
    while (tiles > 1 && per_tile * tiles > budget) tiles -= 1;
    if (W == 32 && tiles > 4) tiles -= tiles % 4; /* warps spread evenly over the four schedulers of an SM */
    if (per_tile * tiles > budget) return LaunchShape{W, 0, 0, 0};
    if (e->full && W == 32 && tiles > 8) {
        /* one CTA per SM and all CTAs take about as long: fewer envs per CTA can fill the last wave better.  Cost model
         * waves x envs-per-CTA (measured, config 3 at 16384 envs: 32 -> 1.01e8, 28 -> 1.05e8, 24 -> 0.97e8, 20 -> 0.89e8) */
        int sms = 148;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->device);
        long long best_cost = -1;
        int best = tiles;
        for (int t = tiles; t >= 8 && t >= tiles - 4; t -= 4) { /* one step: smaller CTAs lose lock-step efficiency */
            long long ctas = (e->n_envs + t - 1) / t, waves = (ctas + sms - 1) / sms;
            long long cost = waves * t;
            if (best_cost < 0 || cost < best_cost) best_cost = cost, best = t;
        }
        tiles = best;
    }
    return LaunchShape{W, tiles, tiles * W, per_tile * tiles};
}

/* cudaFuncSetAttribute is per kernel FUNCTION and process-wide, not per handle: two handles with different shared-memory
 * needs (a training batch and an evaluation batch of the same config) must not lower each other's limit.  Every
 * instantiation is therefore raised ONCE per device to the device's opt-in maximum (the launch itself still requests only
 * what it needs, so occupancy is unaffected).  `done` is a per-instantiation static; setting twice is harmless. */
template <typename K>
static cudaError_t ensure_max_smem(K kernel, int device, unsigned char* done) {
    if (device >= 0 && device < 64 && done[device]) return cudaSuccess;
    int optin = 0;
    cudaError_t err = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    if (err != cudaSuccess) return err;
    err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, optin);
    if (err == cudaSuccess && device >= 0 && device < 64) done[device] = 1;
    return err;
}

template <int W, bool FULL, int MAXT>
static cudaError_t launch_main_k(AgarEnv* e, const float* actions, float* obs, int n_frames, int n_dec, int flags,
                                 uint32_t dec_base, cudaStream_t s) {
    static unsigned char done[64];
    cudaError_t err = ensure_max_smem(k_main<W, FULL, MAXT>, e->device, done);
    if (err != cudaSuccess) return err;
    int blocks = (e->n_envs + e->step.tiles - 1) / e->step.tiles;
    k_main<W, FULL, MAXT><<<blocks, e->step.threads, e->step.smem, s>>>(e->P, e->state, actions, obs, n_frames, n_dec, flags, dec_base);
    return cudaGetLastError();
}
template <int W, bool FULL>
static cudaError_t launch_main_t(AgarEnv* e, const float* actions, float* obs, int n_frames, int n_dec, int flags,
                                 uint32_t dec_base, cudaStream_t s) {
    if (W == 32 && FULL && e->step.threads > 768) return launch_main_k<32, true, 1024>(e, actions, obs, n_frames, n_dec, flags, dec_base, s);
    if (W == 32 && FULL && e->step.threads > 512) return launch_main_k<32, true, 768>(e, actions, obs, n_frames, n_dec, flags, dec_base, s);
    return launch_main_k<W, FULL, 512>(e, actions, obs, n_frames, n_dec, flags, dec_base, s);
}
template <bool FULL>
static cudaError_t launch_init_t(AgarEnv* e, const uint8_t* mask, int mode, cudaStream_t s) {
    static unsigned char done[64];
    cudaError_t err = ensure_max_smem(k_init<32, FULL>, e->device, done);
    if (err != cudaSuccess) return err;
    int blocks = (e->n_envs + e->init.tiles - 1) / e->init.tiles;
    k_init<32, FULL><<<blocks, e->init.threads, e->init.smem, s>>>(e->P, e->state, mask, mode);
    return cudaGetLastError();
}

static int launch_main(AgarEnv* e, const float* actions, float* obs, int n_frames, int n_dec, int flags, uint32_t dec_base,
                       void* stream) {
    AgarEnv* env = e;
    CU(cudaSetDevice(e->device));
    cudaError_t err;
    if (e->simple) {
        /* observer warps encode the observations a launch hands off before its frames (KF_OBS_BEFORE), when enough frames
         * follow each one to hide the encoder; a trailing observation (KF_OBS_AFTER) stays with the physics warps */
        const bool handoff = e->obs.threads && (flags & KF_OBS_BEFORE) && obs != nullptr && n_frames >= SIMPLE_OBS_MIN_FRAMES;
        const SimplePlan& sp = handoff ? e->sp_obs : e->sp;
        const LaunchShape& sh = handoff ? e->obs : e->step;
        const int per = (sh.threads - 32 * sp.obs_warps) / sh.W; /* what k_simple derives from blockDim */
        if (sh.threads % 32 || sh.threads > (handoff ? simple_max_threads(sh.W) : 256) || per < 1 || per != sh.tiles ||
            per * sh.W % 32 || (sp.obs_warps && (!sp.grid_off || 32 * sp.obs_warps % SIMPLE_OBS_LANES)))
            return fail(e, AGAR_E_INVALID, "inconsistent k_simple launch shape%s", "");
        int blocks = (e->n_envs + per - 1) / per;
#define LAUNCH_SIMPLE(WW, OB)                                                                                                 \
    do {                                                                                                                      \
        static unsigned char done_##WW##OB[64];                                                                               \
        err = ensure_max_smem(k_simple<WW, OB>, e->device, done_##WW##OB);                                                    \
        if (err == cudaSuccess) {                                                                                             \
            k_simple<WW, OB><<<blocks, sh.threads, sh.smem, (cudaStream_t)stream>>>(e->P, sp, e->state, actions, obs,         \
                                                                                    n_frames, n_dec, flags, dec_base);        \
            err = cudaGetLastError();                                                                                         \
        }                                                                                                                     \
    } while (0)
        if (handoff && sh.W == 4) LAUNCH_SIMPLE(4, true);
        else if (handoff) LAUNCH_SIMPLE(8, true);
        else if (sh.W == 1) LAUNCH_SIMPLE(1, false);
        else if (sh.W == 2) LAUNCH_SIMPLE(2, false);
        else if (sh.W == 4) LAUNCH_SIMPLE(4, false);
        else if (sh.W == 8) LAUNCH_SIMPLE(8, false);
        else if (sh.W == 16) LAUNCH_SIMPLE(16, false);
        else LAUNCH_SIMPLE(32, false);
#undef LAUNCH_SIMPLE
        if (handoff && err == cudaSuccess) e->observer_launches += 1;
    } else {
        const int W = e->step.W;
        cudaStream_t s = (cudaStream_t)stream;
        err = !e->full ? launch_main_t<32, false>(e, actions, obs, n_frames, n_dec, flags, dec_base, s)
              : W == 32 ? launch_main_t<32, true>(e, actions, obs, n_frames, n_dec, flags, dec_base, s)
              : W == 16 ? launch_main_t<16, true>(e, actions, obs, n_frames, n_dec, flags, dec_base, s)
              : W == 8  ? launch_main_t<8, true>(e, actions, obs, n_frames, n_dec, flags, dec_base, s)
                        : launch_main_t<4, true>(e, actions, obs, n_frames, n_dec, flags, dec_base, s);
    }
    if (err != cudaSuccess) return fail(e, AGAR_E_CUDA, "kernel launch failed: %s", cudaGetErrorString(err));
    e->launches += 1;
    return AGAR_OK;
}
static int launch_init(AgarEnv* e, const uint8_t* mask, int mode, void* stream) {
    AgarEnv* env = e;
    CU(cudaSetDevice(e->device));
    cudaError_t err = e->full ? launch_init_t<true>(e, mask, mode, (cudaStream_t)stream)
                              : launch_init_t<false>(e, mask, mode, (cudaStream_t)stream);
    if (err != cudaSuccess) return fail(e, AGAR_E_CUDA, "kernel launch failed: %s", cudaGetErrorString(err));
    e->launches += 1;
    return AGAR_OK;
}

/* resident CTAs per SM of k_simple<W, OBSW> at this CTA size and shared memory (0: cannot run, or the query failed) */
template <int W, bool OBSW>
static int simple_ctas_per_sm(int device, int threads, size_t smem) {
    static unsigned char done[64];
    int n = 0;
    if (ensure_max_smem(k_simple<W, OBSW>, device, done) != cudaSuccess ||
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_simple<W, OBSW>, threads, smem) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

/* Launch shape of k_simple with observer warps: one CTA per SM, ceil(envs / SMs) envs rounded up to whole physics warps
 * (4096 envs at W = 8: 7 warps, 28 envs, 147 CTAs), plus SIMPLE_OBS_WARPS observers, within the registers of one SM
 * (simple_max_threads).  Latency-bound tile widths (4 and 8 lanes) only: at 1 and 2 lanes the kernel is throughput-bound
 * and the encoder's work costs the same wherever it runs.  Wave-aware: past the physics-warp cap one CTA holds at most 28
 * (W = 8) or 32 (W = 4) envs and an SM holds one such CTA, while the inline shape fits two CTAs of 16 / 32 envs per SM —
 * the observers are used only where their launch needs no more waves than the inline one (4096 envs at W = 8: one wave
 * each; 4608: two against one). */
static void plan_observers(AgarEnv* e) {
    e->obs = LaunchShape{};
    e->sp_obs = e->sp;
    const int W = e->step.W;
    if ((W != 4 && W != 8) || !e->sp.grid_off || e->L.pellet_cap > 64 * SIMPLE_OBS_LANES) return; /* SMask<SIMPLE_OBS_LANES> */
    if (cudaSetDevice(e->device) != cudaSuccess) {
        cudaGetLastError();
        return;
    }
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->device);
    const int per_warp = 32 / W;
    const int K = SIMPLE_OBS_WARPS;
    int warps = ((e->n_envs + sms - 1) / sms + per_warp - 1) / per_warp;
    if (warps > simple_max_threads(W) / 32 - K) warps = simple_max_threads(W) / 32 - K;
    const int per = warps * per_warp;
    const size_t env_bytes = ((size_t)per * e->sp.strideB + 15) / 16 * 16;
    const int snap_stride = (int)((sizeof(SimpleSnap) + (size_t)e->L.pellet_cap * 4 + 15) / 16 * 16);
    const size_t smem = env_bytes + 2 * (size_t)per * snap_stride;
    if (smem > 200 * 1024) return;
    const int threads = (warps + K) * 32;
    const int occ = W == 8 ? simple_ctas_per_sm<8, true>(e->device, threads, smem) : simple_ctas_per_sm<4, true>(e->device, threads, smem);
    const int occ_in = W == 8 ? simple_ctas_per_sm<8, false>(e->device, e->step.threads, e->step.smem)
                              : simple_ctas_per_sm<4, false>(e->device, e->step.threads, e->step.smem);
    if (occ < 1 || occ_in < 1) return;
    const long long per_in = e->step.tiles;
    const long long waves = ((e->n_envs + per - 1) / per + (long long)sms * occ - 1) / ((long long)sms * occ);
    const long long waves_in = ((e->n_envs + per_in - 1) / per_in + (long long)sms * occ_in - 1) / ((long long)sms * occ_in);
    if (waves > waves_in) return;
    e->sp_obs.obs_warps = K;
    e->sp_obs.snap_off = (int)env_bytes;
    e->sp_obs.snap_stride = snap_stride;
    e->obs = LaunchShape{W, per, threads, smem};
}

/* Lanes per env.  Single-cell pellet-collection configs (config_is_simple) with G <= 16: 1, 2, 4, 8, 16, 32 select the
 * register-resident kernel (agar_simple.cuh, k_simple<W>); they run the general kernel (k_main<32, false>, 32 lanes only)
 * with G > 16 or under AGAR_GENERAL_KERNEL=1.  Every other config: 4, 8, 16, 32 (general kernel). */
extern "C" int agar_set_tile_width(AgarEnv* e, int W) {
    if (!e) return AGAR_E_INVALID;
    /* the register-resident kernel bins a pellet into at most two squares per axis: 2 * radius < fov / G needs G <= 16 */
    if (!e->full && e->L.grid_squares <= 16 && (W == 1 || W == 2 || W == 4 || W == 8 || W == 16 || W == 32) &&
        !getenv("AGAR_GENERAL_KERNEL")) {
        const int tail_words = (int)((e->L.record_bytes - e->L.off_pellets) / 4);
        SimplePlan sp = {};
        sp.strideB = (tail_words | 1) * 4;
        /* the observation's G x G sums are accumulated in shared memory and leave once, as consecutive floats of the row
         * (measured: 4096 envs W=8 +1.2 %, 65536 envs W=2 +8 %).  Not at one lane per env: 484 more bytes per env halve the
         * resident envs per SM there (1M envs: 3.28e9 -> 1.52e9), and a lone lane's stores are strided either way. */
        if (W >= 2) {
            const int gg = e->L.grid_squares * e->L.grid_squares;
            sp.grid_off = tail_words * 4;
            sp.strideB = ((tail_words + gg) | 1) * 4;
        }
        if (e->L.pellet_cap > (W >= 4 ? 64 : 128) * W) /* two mask words per lane: SMask<W>, agar_simple.cuh */
            return fail(e, AGAR_E_UNSUPPORTED, "pellet pool too large for this tile width%s", "");
        int threads = 128; /* measured (round 2, exact libm arithmetic): four warps per CTA beat two at every batch size (4096 envs: 7.7e8 vs 7.0e8) */
        const size_t per_env = (size_t)sp.strideB;
        while (threads > 32 && per_env * (threads / W) > 200 * 1024) threads -= 32;
        if (per_env * (threads / W) > 200 * 1024)
            return fail(e, AGAR_E_NOMEM, "pellet pool + event ring of %s do not fit in shared memory at this tile width", "the envs of one CTA");
        e->simple = 1;
        e->sp = sp;
        e->step = LaunchShape{W, threads / W, threads, per_env * (threads / W)};
        plan_observers(e);
        return AGAR_OK;
    }
    bool ok = W == 32 || (e->full && (W == 4 || W == 8 || W == 16));
    if (!ok) return fail(e, AGAR_E_INVALID, "unsupported tile width%s", "");
    const LaunchShape s = plan_launch(e, W);
    if (!s.tiles) return fail(e, AGAR_E_NOMEM, "env record does not fit in shared memory%s", "");
    e->simple = 0;
    e->step = s;
    return AGAR_OK;
}
extern "C" int agar_get_tile_width(const AgarEnv* e) { return e ? e->step.W : 0; }

extern "C" int agar_create(const AgarConfig* cfg, int n_envs, int device, uint64_t seed, uint64_t first_env_id, void* stream,
                           AgarEnv** out) {
    AgarEnv* env = nullptr;
    if (!cfg || !out || n_envs < 1) return fail(nullptr, AGAR_E_INVALID, "bad arguments to agar_create%s", "");
    AgarLayout L;
    int rc = agar_layout_compute(cfg, &L);
    if (rc != AGAR_OK) return fail(nullptr, rc, "config rejected by agar_layout_compute%s", "");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev)
        return fail(nullptr, AGAR_E_CUDA, "no such CUDA device%s", "");
    CU(cudaSetDevice(device));
    AgarEnv* e = (AgarEnv*)calloc(1, sizeof(AgarEnv));
    env = e;
    e->cfg = *cfg;
    e->L = L;
    e->n_envs = n_envs;
    e->device = device;
    e->full = config_is_simple(*cfg, L) ? 0 : 1;
    DevParams& P = e->P;
    memset(&P, 0, sizeof P);
    P.cfg = *cfg;
    P.L = L;
    P.S = L.field_size;
    P.nb = (int)ceil((double)P.S / AG_BUCKET);
    P.n_envs = n_envs;
    P.rec_stride = (int)L.record_bytes + 8;
    P.full = e->full;
    static_assert(AGAR_MAX_CELLS == 16, "cap_shift assumes cell_cap in {1, 16} (agar_layout.h)");
    P.cap_shift = L.cell_cap == AGAR_MAX_CELLS ? 4 : 0;
    P.g_magic = L.grid_squares > 1 ? (uint32_t)((1ull << 32) / (unsigned)L.grid_squares) + 1u : 0u;
    int vel_bytes = e->full ? L.n_players * L.cell_cap * 2 * 8 : 0;
    int obs_bytes = obs_scratch_bytes(L.grid_squares, e->full != 0);
    /* the pellet index (agar_dev.cuh) lives in the same scratch: it is built after the players have moved (velocities dead)
     * and before the next bot phase (observation tables dead); pools of <= 8 chunks are scanned directly */
    P.pel_index = e->full && L.pellet_cap > 256;
    const int gb_idx = (P.S + 9) / 10; /* AG_IDX_CELL */
    int idx_bytes = P.pel_index ? ((gb_idx * gb_idx + 3) & ~1) * 2 + L.pellet_cap * 2 + 128 + 64 + 16 : 0; /* counters, entries, sort list, ex-blob list */
    if (idx_bytes > vel_bytes) vel_bytes = idx_bytes;
    P.scratch_bytes = ((vel_bytes > obs_bytes ? vel_bytes : obs_bytes) + 15) / 16 * 16 + 8;
    P.live_off = P.scratch_bytes; /* live-cell list: uint16 per cell slot, after the observation / velocity scratch */
    if (e->full) P.scratch_bytes += (L.n_players * L.cell_cap * 2 + 15) / 16 * 16;
    /* Where a record lives during a launch (bind_ctx).  The single-cell general kernel stages the whole record in shared
     * memory.  Multi-agent configs keep the record in HBM / L2 and cache on chip what every scan and lane-0 step reads:
     * header + players + cells + viruses (hot_a = off_blobs) + pellet pool if at least 12 envs per CTA still fit, else the
     * pellet pool only (the 16-player arena: 23 KB of cells).  Measured when the policy was chosen (16 envs per CTA):
     * config 3 6.3e7 / 7.3e7 / 7.7e7 env-steps/s for whole record / pool / hot sections; config 4 0.75e6 (whole record, 3
     * warps per SM) / 3.3e6 (pool) / 1.6e6 (hot sections); with 32 envs per CTA (profiles/r01_sweep.txt) config 3 does
     * 9.1e7 (pool) / 9.6e7 (hot sections). */
    if (e->full) {
        size_t hot = (size_t)((L.off_blobs + 15) / 16 * 16) + (size_t)((L.pellet_cap * 4 + 15) / 16 * 16) + P.scratch_bytes;
        P.hot_a = hot * 12 <= 200 * 1024 ? (int)L.off_blobs : 0;
    }
    double speed_modifier = 1.0 / 30;
    P.move_speed = 90 * speed_modifier;
    P.decay_rate = 1 - (0.01 * speed_modifier);
    P.blob_mass = 18 * 0.8;
    P.virus_split_mass = 100.0 + 7 * 18 * 0.8;
    P.start_radius = sqrt(10.0 / M_PI);
    P.virus_radius = sqrt(100.0 / M_PI);
    for (int m = 0; m < 4; ++m) P.pellet_r[m] = m ? sqrt((double)m / M_PI) : 0.0;
    for (int n = 1; n <= 16; ++n) P.pow_n[n] = pow((double)n, 0.32);
    P.seed = seed;
    P.first_env = first_env_id;
    double tab[720];
    for (int d = 0; d < 360; ++d) {
        double a = d * (M_PI / 180.0);
        tab[d] = cos(a), tab[360 + d] = sin(a);
    }
    if (cudaMalloc(&e->deg_tab, sizeof tab) != cudaSuccess || cudaMalloc(&e->state, (size_t)n_envs * L.record_bytes) != cudaSuccess) {
        cudaGetLastError();
        if (e->deg_tab) cudaFree(e->deg_tab);
        free(e);
        return fail(nullptr, AGAR_E_NOMEM, "cudaMalloc of the env state failed%s", "");
    }
    CU(cudaMemcpyAsync(e->deg_tab, tab, sizeof tab, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    CU(cudaStreamSynchronize((cudaStream_t)stream)); /* tab is a stack buffer */
    P.deg_tab = e->deg_tab;
    e->init = plan_launch(e, 32); /* k_init always runs with 32-lane tiles */
    if (!e->init.tiles) {
        cudaFree(e->state), cudaFree(e->deg_tab), free(e);
        return fail(nullptr, AGAR_E_NOMEM, "env record does not fit in shared memory%s", "");
    }
    int W = e->full ? 32 : (n_envs <= 8192 ? 8 : (n_envs <= 32768 ? 2 : 1)); /* tools/sweep.py, profiles/r01_sweep.txt */
    if (agar_set_tile_width(e, W) != AGAR_OK && agar_set_tile_width(e, 8) != AGAR_OK && agar_set_tile_width(e, 32) != AGAR_OK) {
        snprintf(g_create_err, sizeof g_create_err, "%s", e->err);
        cudaFree(e->state), cudaFree(e->deg_tab), free(e);
        return AGAR_E_NOMEM;
    }
    rc = launch_init(e, nullptr, 0, stream);
    if (rc != AGAR_OK) {
        snprintf(g_create_err, sizeof g_create_err, "%s", e->err);
        cudaFree(e->state), cudaFree(e->deg_tab), free(e);
        return rc;
    }
    *out = e;
    return AGAR_OK;
}
extern "C" int agar_destroy(AgarEnv* e) {
    if (!e) return AGAR_E_INVALID;
    cudaSetDevice(e->device);
    cudaFree(e->state);
    cudaFree(e->deg_tab);
    if (e->d_actions) cudaFree(e->d_actions);
    if (e->d_obs) cudaFree(e->d_obs);
    if (e->d_reward) cudaFree(e->d_reward);
    if (e->h_turn) cudaFreeHost(e->h_turn);
    if (e->d_export_count) cudaFree(e->d_export_count);
    free(e);
    return AGAR_OK;
}
extern "C" const char* agar_last_error(const AgarEnv* e) { return e ? e->err : g_create_err; }
extern "C" int agar_get_layout(const AgarEnv* e, AgarLayout* out) {
    if (!e || !out) return AGAR_E_INVALID;
    *out = e->L;
    return AGAR_OK;
}
extern "C" int agar_num_envs(const AgarEnv* e) { return e ? e->n_envs : AGAR_E_INVALID; }
extern "C" int64_t agar_launch_count(const AgarEnv* e) { return e ? e->launches : 0; }
extern "C" int64_t agar_observer_launch_count(const AgarEnv* e) { return e ? e->observer_launches : 0; }
extern "C" void* agar_state_ptr(const AgarEnv* e) { return e ? e->state : nullptr; }

extern "C" int agar_reset(AgarEnv* e, const uint8_t* env_mask_dev, void* stream) {
    if (!e) return AGAR_E_INVALID;
    return launch_init(e, env_mask_dev, 1, stream);
}
extern "C" int agar_reset_bots(AgarEnv* e, const uint8_t* env_mask_dev, void* stream) {
    if (!e) return AGAR_E_INVALID;
    return launch_init(e, env_mask_dev, 2, stream);
}
extern "C" int agar_observe(AgarEnv* e, float* obs_dev, void* stream) {
    if (!e) return AGAR_E_INVALID;
    return launch_main(e, nullptr, obs_dev, 0, 0, KF_OBS_AFTER, 0, stream);
}
extern "C" int agar_step(AgarEnv* e, const float* actions_dev, int n_frames, void* stream) {
    if (!e || n_frames < 0) return AGAR_E_INVALID;
    if (!actions_dev && e->L.n_agents > 0) return fail(e, AGAR_E_INVALID, "actions_dev is NULL%s", "");
    return launch_main(e, actions_dev, nullptr, n_frames, 1, 0, 0, stream);
}
extern "C" int agar_step_observe(AgarEnv* e, const float* actions_dev, int n_frames, float* obs_dev, void* stream) {
    if (!e || n_frames < 0) return AGAR_E_INVALID;
    if (!actions_dev && e->L.n_agents > 0) return fail(e, AGAR_E_INVALID, "actions_dev is NULL%s", "");
    return launch_main(e, actions_dev, obs_dev, n_frames, 1, KF_OBS_AFTER, 0, stream);
}
/* n_decisions x (observe -> uniform random action from Philox stream 7 -> n_frames frames), one launch.
 * The random-action driver of BASELINE config 2; obs_dev (nullable) receives every decision's observation. */
extern "C" int agar_rollout_random(AgarEnv* e, int n_decisions, int n_frames, uint32_t decision_base, float* obs_dev,
                                   void* stream) {
    if (!e || n_decisions < 0 || n_frames < 0) return AGAR_E_INVALID;
    return launch_main(e, nullptr, obs_dev, n_frames, n_decisions, KF_OBS_BEFORE | KF_RANDOM_ACTIONS, decision_base, stream);
}
extern "C" int agar_get(AgarEnv* e, AgarField which, void* out_dev, void* stream) {
    AgarEnv* env = e;
    if (!e || !out_dev || (int)which < 0 || (int)which > AGAR_GET_EVENT_HASH) return AGAR_E_INVALID;
    CU(cudaSetDevice(e->device));
    int per_env = (which == AGAR_GET_OVERFLOW || which == AGAR_GET_EVENT_HASH);
    int n = per_env ? e->n_envs : e->n_envs * e->L.n_agents;
    if (n == 0) return AGAR_OK;
    k_get<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(e->P, e->state, (int)which, out_dev);
    CU(cudaGetLastError());
    e->launches += 1;
    return AGAR_OK;
}
extern "C" int agar_debug_dump(AgarEnv* e, int env_index, void* record_host, size_t bytes, void* stream) {
    AgarEnv* env = e;
    if (!e || !record_host || env_index < 0 || env_index >= e->n_envs || bytes != e->L.record_bytes) return AGAR_E_INVALID;
    CU(cudaSetDevice(e->device));
    CU(cudaMemcpyAsync(record_host, e->state + (size_t)env_index * e->L.record_bytes, bytes, cudaMemcpyDeviceToHost,
                       (cudaStream_t)stream));
    CU(cudaStreamSynchronize((cudaStream_t)stream));
    return AGAR_OK;
}
extern "C" int agar_debug_load(AgarEnv* e, int env_index, const void* record_host, size_t bytes, void* stream) {
    AgarEnv* env = e;
    if (!e || !record_host || env_index < 0 || env_index >= e->n_envs || bytes != e->L.record_bytes) return AGAR_E_INVALID;
    CU(cudaSetDevice(e->device));
    CU(cudaMemcpyAsync(e->state + (size_t)env_index * e->L.record_bytes, record_host, bytes, cudaMemcpyHostToDevice,
                       (cudaStream_t)stream));
    CU(cudaStreamSynchronize((cudaStream_t)stream));
    return AGAR_OK;
}
/* device-visible address of a pinned host buffer, or nullptr for pageable memory */
static void* pinned_dev_ptr(const void* p) {
    if (!p) return nullptr;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return at.type == cudaMemoryTypeHost ? at.devicePointer : nullptr;
}

extern "C" int agar_step_host_begin(AgarEnv* e, const float* actions_host, int n_frames, float* obs_host, void* stream) {
    AgarEnv* env = e;
    if (!e || !actions_host || n_frames < 0) return AGAR_E_INVALID;
    CU(cudaSetDevice(e->device));
    cudaStream_t s = (cudaStream_t)stream;
    const size_t EA = (size_t)e->n_envs * (e->L.n_agents ? e->L.n_agents : 1);
    const size_t turn_words = (EA * 5 + 3) / 4;
    if (!e->d_actions) {
        CU(cudaMalloc(&e->d_actions, EA * 4 * sizeof(float)));
        CU(cudaMalloc(&e->d_obs, EA * e->L.state_len * sizeof(float)));
        CU(cudaMalloc(&e->d_reward, turn_words * 4)); /* packed: float reward[EA] | uint8 done[EA] -> one copy back */
        const size_t flag_off = (turn_words * 4 + 63) / 64 * 64;
        CU(cudaMallocHost(&e->h_turn, flag_off + 64));
        e->h_flag = (volatile uint32_t*)((uint8_t*)e->h_turn + flag_off);
        *e->h_flag = 0;
        e->flag_seq = 0;
        CU(cudaMalloc(&e->d_export_count, sizeof(unsigned int)));
        CU(cudaMemsetAsync(e->d_export_count, 0, sizeof(unsigned int), s));
        e->d_done = (uint8_t*)e->d_reward + EA * 4;
        CU(cudaMemsetAsync(e->d_obs, 0, EA * e->L.state_len * sizeof(float), s));
        CU(cudaMemsetAsync(e->d_reward, 0, turn_words * 4, s));
    }
    /* Pinned caller buffers (cudaHostAlloc / cudaHostRegister / torch pin_memory) are visible to the device: the step
     * kernel reads the actions in place and its CTAs store the results straight into them (export_tail).  Pageable buffers take the
     * copy-engine path. */
    const float* act_dev = (const float*)pinned_dev_ptr(actions_host);
    float* obs_dev_host = (float*)pinned_dev_ptr(obs_host);
    const bool zero_copy = act_dev && (!obs_host || (obs_dev_host && ((uintptr_t)obs_dev_host & 15) == 0));
    if (!zero_copy) CU(cudaMemcpyAsync(e->d_actions, actions_host, EA * 4 * sizeof(float), cudaMemcpyHostToDevice, s));
    e->P.turn_reward = e->d_reward, e->P.turn_done = e->d_done; /* reward / done written by the step kernel itself */
    e->host_polling = 0;
    if (zero_copy) { /* ONE launch: each CTA exports its own rows over PCIe and the last one raises the flag (export_tail) */
        void* turn_dev_host = nullptr;
        void* flag_dev_host = nullptr;
        CU(cudaHostGetDevicePointer(&turn_dev_host, e->h_turn, 0));
        CU(cudaHostGetDevicePointer(&flag_dev_host, (void*)e->h_flag, 0));
        e->flag_seq += 1;
        if (e->flag_seq == 0) e->flag_seq = 1;
        e->P.host_obs = obs_dev_host, e->P.host_turn = (uint32_t*)turn_dev_host, e->P.export_count = e->d_export_count;
        e->P.host_flag = (volatile uint32_t*)flag_dev_host, e->P.flag_value = e->flag_seq;
        e->host_polling = 1;
    }
    int rc = launch_main(e, zero_copy ? act_dev : e->d_actions, e->d_obs, n_frames, 1, KF_OBS_AFTER, 0, s);
    e->P.turn_reward = nullptr, e->P.turn_done = nullptr;
    e->P.host_obs = nullptr, e->P.host_turn = nullptr, e->P.export_count = nullptr, e->P.host_flag = nullptr;
    if (rc != AGAR_OK) {
        e->host_polling = 0;
        return rc;
    }
    if (!zero_copy) {
        const size_t obs_bytes = EA * e->L.state_len * sizeof(float);
        if (obs_host) CU(cudaMemcpyAsync(obs_host, e->d_obs, obs_bytes, cudaMemcpyDeviceToHost, s));
        CU(cudaMemcpyAsync(e->h_turn, e->d_reward, EA * 5, cudaMemcpyDeviceToHost, s));
    }
    e->host_pending = 1;
    return AGAR_OK;
}

extern "C" int agar_step_host_end(AgarEnv* e, float* reward_host, uint8_t* done_host, void* stream) {
    AgarEnv* env = e;
    if (!e) return AGAR_E_INVALID;
    if (!e->host_pending) return fail(env, AGAR_E_INVALID, "%s", "agar_step_host_end without agar_step_host_begin");
    CU(cudaSetDevice(e->device));
    if (e->host_polling) {
        /* the launch's last CTA writes flag_seq into pinned memory after every row has been made visible system-wide: poll it
         * (a few hundred ns of latency instead of a driver wake-up); cudaStreamQuery now and then catches a failed launch */
        const uint32_t want = e->flag_seq;
        unsigned spins = 0;
        while (*e->h_flag != want) {
            if ((++spins & 0xfff) == 0) {
                cudaError_t q = cudaStreamQuery((cudaStream_t)stream);
                if (q == cudaSuccess) break;
                if (q != cudaErrorNotReady) return fail(env, AGAR_E_CUDA, "CUDA error: %s", cudaGetErrorString(q));
            }
#if defined(__x86_64__) || defined(__i386__)
            __builtin_ia32_pause();
#endif
        }
        if (*e->h_flag != want) CU(cudaStreamSynchronize((cudaStream_t)stream)); /* the stream drained without the flag: surface the error */
        e->host_polling = 0;
    } else {
        CU(cudaStreamSynchronize((cudaStream_t)stream));
    }
    e->host_pending = 0;
    const size_t EA = (size_t)e->n_envs * (e->L.n_agents ? e->L.n_agents : 1);
    if (reward_host) memcpy(reward_host, e->h_turn, EA * 4);
    if (done_host) memcpy(done_host, (uint8_t*)e->h_turn + EA * 4, EA);
    return AGAR_OK;
}

extern "C" int agar_step_host(AgarEnv* e, const float* actions_host, int n_frames, float* obs_host, float* reward_host,
                              uint8_t* done_host, void* stream) {
    int rc = agar_step_host_begin(e, actions_host, n_frames, obs_host, stream);
    return rc != AGAR_OK ? rc : agar_step_host_end(e, reward_host, done_host, stream);
}
