/*
 * agar_replay.cu — GPU replay buffer (uniform ring + prioritized with sum / min segment trees).
 * Replaces src/model/replay_buffer.py and src/model/common/segment_tree.py; C ABI in include/agar_replay.h.
 * HBM-bound: add / gather move 2 * state_len + action_len + 2 floats per transition with coalesced row copies;
 * the trees are float64 arrays of 2 * it_capacity nodes rebuilt level by level (a node is op(left, right), so the
 * tree is a function of the leaves only and batched updates commute).
 */
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/agar_b200.h"
#include "../../include/agar_math.h"
#include "../../include/agar_replay.h"

struct ReplayDev {
    float *obs_t, *obs_tp1, *action, *reward;
    uint8_t* done;
    double *sum, *mn;    /* segment trees, 2 * itcap each (node 1 = root) */
    int32_t* counters;   /* [0] next_idx  [1] size  [2] n_valid of the last add  [3] error flags  [4] verdict of the last load */
    double* max_priority;
    int32_t* pos;        /* scratch: ring position per candidate of the last add (-1 = not stored) */
    int cap, itcap, L, AL, prioritized;
    double alpha, beta;
};
struct AgarReplay {
    ReplayDev d;
    int device, pos_cap;
    int64_t launches;
    char err[256];
};
constexpr size_t RP_COUNTER_BYTES = 32; /* int32 counters[8]; [5..7] unused */
static char g_rp_err[256] = "";

static int rp_fail(AgarReplay* rp, int code, const char* msg) {
    snprintf(rp ? rp->err : g_rp_err, 256, "%s", msg);
    return code;
}
#define RCU(call)                                                                       \
    do {                                                                                \
        cudaError_t _e = (call);                                                        \
        if (_e != cudaSuccess) return rp_fail(rp, AGAR_E_CUDA, cudaGetErrorString(_e)); \
    } while (0)

/* ---- add: ranks of the valid candidates (one CTA, chunked block scan), then one warp per stored transition */
__global__ void k_rp_scan(ReplayDev d, const uint8_t* __restrict__ valid, int n) {
    __shared__ int warp_tot[32];
    __shared__ int running;
    if (threadIdx.x == 0) running = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    /* pass 1: count */
    int total = 0;
    for (int base = 0; base < n; base += blockDim.x) {
        int i = base + threadIdx.x;
        int v = i < n && (valid == nullptr || valid[i]);
        unsigned b = __ballot_sync(0xffffffffu, v);
        if (lane == 0) warp_tot[wid] = __popc(b);
        __syncthreads();
        if (threadIdx.x == 0) {
            int s = 0;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += warp_tot[w];
            running += s;
        }
        __syncthreads();
    }
    total = running;
    __syncthreads();
    const int next0 = d.counters[0], size0 = d.counters[1];
    const int skip = total > d.cap ? total - d.cap : 0; /* later adds of the same batch would overwrite these */
    if (threadIdx.x == 0) running = 0;
    __syncthreads();
    /* pass 2: positions */
    for (int base = 0; base < n; base += blockDim.x) {
        int i = base + threadIdx.x;
        int v = i < n && (valid == nullptr || valid[i]);
        unsigned b = __ballot_sync(0xffffffffu, v);
        if (lane == 0) warp_tot[wid] = __popc(b);
        __syncthreads();
        int before = running;
        for (int w = 0; w < wid; ++w) before += warp_tot[w];
        int rank = before + __popc(b & ((1u << lane) - 1));
        if (i < n) d.pos[i] = (v && rank >= skip) ? (int)(((long long)next0 + rank) % d.cap) : -1;
        __syncthreads();
        if (threadIdx.x == 0) {
            int s = 0;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += warp_tot[w];
            running += s;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        d.counters[0] = (int)(((long long)next0 + total) % d.cap);
        long long sz = (long long)size0 + total;
        d.counters[1] = sz > d.cap ? d.cap : (int)sz;
        d.counters[2] = total;
    }
}
__global__ void k_rp_store(ReplayDev d, const float* __restrict__ obs_t, const float* __restrict__ action,
                           const float* __restrict__ reward, const float* __restrict__ obs_tp1,
                           const uint8_t* __restrict__ done, int n) {
    int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= n) return;
    int p = d.pos[w];
    if (p < 0) return;
    const float* s0 = obs_t + (size_t)w * d.L;
    const float* s1 = obs_tp1 + (size_t)w * d.L;
    float* d0 = d.obs_t + (size_t)p * d.L;
    float* d1 = d.obs_tp1 + (size_t)p * d.L;
    for (int i = lane; i < d.L; i += 32) {
        d0[i] = s0[i];
        d1[i] = s1[i];
    }
    if (lane < d.AL) d.action[(size_t)p * d.AL + lane] = action[(size_t)w * d.AL + lane];
    if (lane == 0) {
        d.reward[p] = reward[w];
        d.done[p] = done[w];
        if (d.prioritized) { /* leaf = max_priority ** alpha (replay_buffer.py:111-112) */
            double v = agar_pow(*d.max_priority, d.alpha);
            d.sum[d.itcap + p] = v;
            d.mn[d.itcap + p] = v;
        }
    }
}
__global__ void k_rp_init(ReplayDev d) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 2 * d.itcap) {
        d.sum[i] = 0.0;
        d.mn[i] = INFINITY;
    }
    if (i == 0) {
        d.counters[0] = d.counters[1] = d.counters[2] = d.counters[3] = 0;
        *d.max_priority = 1.0;
    }
}
__global__ void k_rp_gather(ReplayDev d, const int32_t* __restrict__ idx, int batch, float* obs_t, float* action, float* reward,
                            float* obs_tp1, uint8_t* done) {
    int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= batch) return;
    int p = idx[w];
    if (p < 0 || p >= d.counters[1]) { /* the reference asserts 0 <= idx < len(storage); here: flag, read slot 0 */
        if (lane == 0) atomicOr(&d.counters[3], AGAR_RP_ERR_INDEX);
        p = 0;
    }
    const float* s0 = d.obs_t + (size_t)p * d.L;
    const float* s1 = d.obs_tp1 + (size_t)p * d.L;
    for (int i = lane; i < d.L; i += 32) {
        if (obs_t) obs_t[(size_t)w * d.L + i] = s0[i];
        if (obs_tp1) obs_tp1[(size_t)w * d.L + i] = s1[i];
    }
    if (action && lane < d.AL) action[(size_t)w * d.AL + lane] = d.action[(size_t)p * d.AL + lane];
    if (lane == 0) {
        if (reward) reward[w] = d.reward[p];
        if (done) done[w] = d.done[p];
    }
}
__global__ void k_rp_uniform_idx(ReplayDev d, const double* __restrict__ u, int batch, int32_t* idx) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= batch) return;
    int len = d.counters[1];
    if (len < 1) { /* random.randint(0, -1) raises in the reference; here: index 0 and a sticky error flag */
        atomicOr(&d.counters[3], AGAR_RP_ERR_EMPTY);
        idx[i] = 0;
        return;
    }
    int v = (int)(u[i] * (double)len); /* random.randint(0, len - 1) */
    idx[i] = v >= len ? len - 1 : v;
}
/* SegmentTree._reduce_helper for the prefix [0, end] (segment_tree.py:38-53): value[left child] + helper(right), i.e.
 * v1 + (v2 + (v3 + ...)) over the maximal nodes of the prefix */
__device__ double rp_prefix_sum(const ReplayDev& d, int end) {
    double parts[40];
    int np = 0;
    int node = 1, ns = 0, ne = d.itcap - 1;
    if (end < 0) return 0.0; /* callers guard len < 2; never descend with an end the loop cannot reach */
    if (end > ne) end = ne;
    while (true) {
        if (end == ne) {
            parts[np++] = d.sum[node];
            break;
        }
        int mid = (ns + ne) / 2;
        if (end <= mid) {
            node = 2 * node, ne = mid;
        } else {
            parts[np++] = d.sum[2 * node];
            node = 2 * node + 1, ns = mid + 1;
        }
    }
    double acc = parts[np - 1];
    for (int i = np - 2; i >= 0; --i) acc = parts[i] + acc;
    return acc;
}
__global__ void k_rp_per_sample(ReplayDev d, const double* __restrict__ u, int batch, int32_t* idx, double* weights) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= batch) return;
    const int len = d.counters[1];
    if (len < 2) { /* the reference recurses without end here (sum(0, len - 1) over an empty prefix); flag and return slot 0 */
        atomicOr(&d.counters[3], AGAR_RP_ERR_EMPTY);
        idx[i] = 0;
        if (weights) weights[i] = 0.0;
        return;
    }
    /* _sample_proportional (:113-120): sum(0, len - 1) reduces over [0, len - 2] (reduce() decrements `end`) */
    double total = rp_prefix_sum(d, len - 2);
    double mass = u[i] * total;
    int node = 1;
    while (node < d.itcap) { /* find_prefixsum_idx (segment_tree.py:107-126) */
        double l = d.sum[2 * node];
        if (l > mass)
            node = 2 * node;
        else {
            mass -= l;
            node = 2 * node + 1;
        }
    }
    int p = node - d.itcap;
    idx[i] = p;
    if (weights) { /* :157-166 */
        double root = d.sum[1];
        double p_min = d.mn[1] / root;
        double max_weight = agar_pow(p_min * len, -d.beta);
        double p_sample = d.sum[d.itcap + p] / root;
        weights[i] = agar_pow(p_sample * len, -d.beta) / max_weight;
    }
}
/* staged != 0: the launch carries batch * 4 bytes of dynamic shared memory and every CTA keeps a copy of idx there — the
 * "does a later entry name the same leaf" scan then runs on shared memory without an early exit (consecutive threads read
 * consecutive words): 2048 entries 123 us -> a few us */
__global__ void k_rp_set_priorities(ReplayDev d, const int32_t* __restrict__ idx, const double* __restrict__ prio, int batch, int staged) {
    extern __shared__ int32_t sh_idx[];
    if (staged) {
        for (int j = threadIdx.x; j < batch; j += blockDim.x) sh_idx[j] = idx[j];
        __syncthreads();
    }
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= batch) return;
    /* duplicates in idx: the reference applies them in order, the last one wins */
    if (staged) {
        const int32_t mine = sh_idx[i];
        bool later = false;
        for (int j = i + 1; j < batch; ++j) later |= sh_idx[j] == mine;
        if (later) return;
    } else {
        for (int j = i + 1; j < batch; ++j)
            if (idx[j] == idx[i]) return;
    }
    /* replay_buffer.py:203-204 asserts priority > 0 and 0 <= idx < len(storage): skip and flag instead of poisoning the trees */
    if (idx[i] < 0 || idx[i] >= d.counters[1]) {
        atomicOr(&d.counters[3], AGAR_RP_ERR_INDEX);
        return;
    }
    if (!(prio[i] > 0.0) || prio[i] > 1.7e308) {
        atomicOr(&d.counters[3], AGAR_RP_ERR_PRIORITY);
        return;
    }
    double v = agar_pow(prio[i], d.alpha);
    d.sum[d.itcap + idx[i]] = v;
    d.mn[d.itcap + idx[i]] = v;
}
/* _max_priority = max(_max_priority, priority) over the batch (replay_buffer.py:188): a maximum, so any order — one CTA, strided
 * loads and a shared-memory tree (a lone thread walking 2048 priorities took 190 us of a 750 us learner tick) */
__global__ void __launch_bounds__(256) k_rp_max_priority(ReplayDev d, const double* __restrict__ prio, int batch) {
    __shared__ double sm[256];
    double m = 0.0; /* priorities are > 0 (guarded by k_rp_set_priorities) */
    for (int i = threadIdx.x; i < batch; i += 256) {
        const double v = prio[i];
        if (v > m && v <= 1.7e308) m = v;
    }
    sm[threadIdx.x] = m;
    __syncthreads();
    for (int off = 128; off > 0; off >>= 1) {
        if (threadIdx.x < off && sm[threadIdx.x + off] > sm[threadIdx.x]) sm[threadIdx.x] = sm[threadIdx.x + off];
        __syncthreads();
    }
    if (threadIdx.x == 0 && sm[0] > *d.max_priority) *d.max_priority = sm[0];
}

/* Repair the sum / min trees above the n leaves idx[0..n) (entries < 0 are skipped) in ONE launch: a node is
 * op(left child, right child) (segment_tree.py:76-87), so only the ancestors of touched leaves change, level by level.  One
 * CTA walks the levels with a barrier in between; threads that reach the same parent recompute the same value from the same
 * finished children (a benign duplicate).  Replaces 20 level-wide launches per add / priority update (the learner tick is
 * launch-bound: ~150 small kernels). */
__global__ void __launch_bounds__(1024) k_rp_fix_paths(ReplayDev d, const int32_t* __restrict__ idx, int n) {
    int levels = 0;
    while ((1 << levels) < d.itcap) ++levels;
    for (int lv = 1; lv <= levels; ++lv) {
        const int width = d.itcap >> lv; /* nodes on this level */
        if (width <= n) { /* near the root there are fewer nodes than touched leaves: recompute the level (same values, fewer loads) */
            for (int i = threadIdx.x; i < width; i += blockDim.x) {
                const int node = width + i;
                d.sum[node] = d.sum[2 * node] + d.sum[2 * node + 1];
                const double a = d.mn[2 * node], b = d.mn[2 * node + 1];
                d.mn[node] = b < a ? b : a;
            }
        } else {
            for (int i = threadIdx.x; i < n; i += blockDim.x) {
                const int p = idx[i];
                if (p < 0 || p >= d.cap) continue;
                const int node = (d.itcap + p) >> lv;
                d.sum[node] = d.sum[2 * node] + d.sum[2 * node + 1];
                const double a = d.mn[2 * node], b = d.mn[2 * node + 1];
                d.mn[node] = b < a ? b : a; /* Python min(a, b): b only if b < a */
            }
        }
        __syncthreads();
    }
}
/* all nodes of one tree level: value[node] = op(value[2 node], value[2 node + 1]) (segment_tree.py:76-87) */
__global__ void k_rp_level(ReplayDev d, int first, int count) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    int node = first + i;
    d.sum[node] = d.sum[2 * node] + d.sum[2 * node + 1];
    double a = d.mn[2 * node], b = d.mn[2 * node + 1];
    d.mn[node] = b < a ? b : a;
}
/* few touched leaves (a learner's batch, a tick of a few thousand envs): one launch that walks their ancestors; many (a tick of
 * 65k envs touches a large part of every level anyway): one grid-wide launch per level */
static int rp_fix_paths(AgarReplay* rp, const int32_t* idx_dev, int n, cudaStream_t s) {
    if (n <= 8192) {
        k_rp_fix_paths<<<1, 1024, 0, s>>>(rp->d, idx_dev, n);
        rp->launches += 1;
    } else {
        for (int count = rp->d.itcap / 2; count >= 1; count /= 2) {
            k_rp_level<<<(count + 255) / 256, 256, 0, s>>>(rp->d, count, count);
            rp->launches += 1;
        }
    }
    RCU(cudaGetLastError());
    return AGAR_OK;
}

/* ---- state snapshots (agar_replay_save / agar_replay_load; bank layout in agar_replay.h) */
constexpr int RP_SECTIONS = 6; /* obs_t, obs_tp1, action, reward, done, leaf */
constexpr int RP_LEAF = 5;
struct RpStateLayout {
    int64_t off[RP_SECTIONS + 1]; /* section s spans bytes [off[s], off[s + 1]) of the bank; off[RP_SECTIONS] = bank bytes */
    int64_t row[RP_SECTIONS];     /* bytes per ring slot (0 for the leaves of a uniform buffer: an empty section) */
};
static RpStateLayout rp_state_layout(const ReplayDev& d) {
    const int64_t row[RP_SECTIONS] = {4ll * d.L, 4ll * d.L, 4ll * d.AL, 4, 1, d.prioritized ? 8 : 0};
    RpStateLayout s;
    int64_t at = 256; /* the header */
    for (int i = 0; i < RP_SECTIONS; ++i) {
        s.row[i] = row[i];
        s.off[i] = at;
        at = (at + (int64_t)d.cap * row[i] + 255) & ~(int64_t)255;
    }
    s.off[RP_SECTIONS] = at;
    return s;
}
__device__ uint8_t* rp_ring(const ReplayDev& d, int s) {
    return s == 0 ? (uint8_t*)d.obs_t : s == 1 ? (uint8_t*)d.obs_tp1 : s == 2 ? (uint8_t*)d.action : s == 3 ? (uint8_t*)d.reward : d.done;
}
union RpWord {
    uint4 v;
    uint8_t b[16];
};
/* 16-byte word i of a ring allocation whose first `live` bytes are live; bytes past `live` read as zero (and are not read:
 * the allocation need not extend to a whole word) */
__device__ uint4 rp_fetch(const uint8_t* a, int64_t i, int64_t live) {
    const int64_t o = i * 16;
    if (o + 16 <= live) return *(const uint4*)(a + o);
    RpWord w;
    w.v = make_uint4(0, 0, 0, 0);
    for (int k = 0; o + k < live; ++k) w.b[k] = a[o + k];
    return w.v;
}
__device__ void rp_put(uint8_t* a, int64_t i, int64_t live, uint4 v) {
    const int64_t o = i * 16;
    if (o + 16 <= live) {
        *(uint4*)(a + o) = v;
        return;
    }
    RpWord w;
    w.v = v;
    for (int k = 0; o + k < live; ++k) a[o + k] = w.b[k];
}
__device__ bool rp_leaf_bad(double v, int64_t k, int64_t size) {
    return k >= size ? __double_as_longlong(v) != 0 : !(v >= 0.0); /* +0.0 past size; below it neither NaN nor negative */
}
/* Load, step 1: the verdict (counters[4], zeroed by the host's memset) is set when the bank fails any check listed at
 * agar_replay_load.  Thread 0 checks the header, the grid the leaves. */
__global__ void __launch_bounds__(256) k_rp_validate(ReplayDev d, RpStateLayout s, const uint8_t* __restrict__ bank) {
    const AgarReplayStateHeader* h = (const AgarReplayStateHeader*)bank;
    const int64_t size = h->size;
    bool bad = false;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        const double mp = h->max_priority;
        bad = h->capacity != d.cap || h->state_len != d.L || h->action_len != d.AL || h->prioritized != (d.prioritized != 0) ||
              h->alpha_bits != (uint64_t)__double_as_longlong(d.alpha) || h->beta_bits != (uint64_t)__double_as_longlong(d.beta) ||
              h->next_idx < 0 || h->next_idx >= d.cap || size < 0 || size > d.cap || (size < d.cap && h->next_idx != size) ||
              !(mp >= 1.0 && mp <= 1.7e308);
    }
    if (d.prioritized) {
        const double2* leaf = (const double2*)(bank + s.off[RP_LEAF]);
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; 2 * i < d.cap; i += (int64_t)gridDim.x * blockDim.x) {
            const double2 v = leaf[i];
            bad |= rp_leaf_bad(v.x, 2 * i, size) || (2 * i + 1 < d.cap && rp_leaf_bad(v.y, 2 * i + 1, size));
        }
    }
    if (bad) {
        d.counters[4] = 1;
        atomicOr(&d.counters[3], AGAR_RP_ERR_STATE);
    }
}
/* Save (load = 0): bank <- buffer, zeros for ring rows and leaves at index >= size and for padding.  Load, step 2: buffer <-
 * bank if the verdict is good, ring rows below the bank's size and every leaf (sum / min: the leaf below size, 0 / +inf at
 * and above it).  blockIdx.y is the section; the grid strides over its 16-byte words with RP_COPY_U loads in flight. */
constexpr int RP_COPY_U = 4;
__global__ void __launch_bounds__(256) k_rp_state(ReplayDev d, RpStateLayout s, uint8_t* bank, int load) {
    if (load && d.counters[4] != 0) return;
    const AgarReplayStateHeader* hb = (const AgarReplayStateHeader*)bank;
    const int64_t size = load ? hb->size : d.counters[1];
    const int sec = blockIdx.y;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x, t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nw = (s.off[sec + 1] - s.off[sec]) / 16;
    uint4* b = (uint4*)(bank + s.off[sec]);
    if (sec == 0 && t0 == 0) {
        if (load) {
            d.counters[0] = (int32_t)hb->next_idx;
            d.counters[1] = (int32_t)size;
            *d.max_priority = hb->max_priority;
        } else {
            union {
                AgarReplayStateHeader h;
                uint4 w[16];
            } u;
            for (int k = 0; k < 16; ++k) u.w[k] = make_uint4(0, 0, 0, 0);
            u.h.capacity = d.cap, u.h.state_len = d.L, u.h.action_len = d.AL, u.h.prioritized = d.prioritized != 0;
            u.h.alpha_bits = (uint64_t)__double_as_longlong(d.alpha), u.h.beta_bits = (uint64_t)__double_as_longlong(d.beta);
            u.h.next_idx = d.counters[0], u.h.size = size, u.h.max_priority = *d.max_priority;
            for (int k = 0; k < 16; ++k) ((uint4*)bank)[k] = u.w[k];
        }
    }
    if (sec == RP_LEAF) {
        double2* leaf = (double2*)b;
        for (int64_t i = t0; i < nw; i += stride) {
            const int64_t k = 2 * i;
            if (load) {
                const double2 v = leaf[i];
                if (k < d.cap) d.sum[d.itcap + k] = k < size ? v.x : 0.0, d.mn[d.itcap + k] = k < size ? v.x : INFINITY;
                if (k + 1 < d.cap) d.sum[d.itcap + k + 1] = k + 1 < size ? v.y : 0.0, d.mn[d.itcap + k + 1] = k + 1 < size ? v.y : INFINITY;
            } else {
                leaf[i] = make_double2(k < size ? d.sum[d.itcap + k] : 0.0, k + 1 < size ? d.sum[d.itcap + k + 1] : 0.0);
            }
        }
        return;
    }
    uint8_t* a = rp_ring(d, sec);
    const int64_t live = size * s.row[sec];
    for (int64_t base = t0; base < nw; base += RP_COPY_U * stride) {
        uint4 v[RP_COPY_U];
#pragma unroll
        for (int u = 0; u < RP_COPY_U; ++u) {
            const int64_t i = base + u * stride;
            if (i < nw) v[u] = load ? b[i] : rp_fetch(a, i, live);
        }
#pragma unroll
        for (int u = 0; u < RP_COPY_U; ++u) {
            const int64_t i = base + u * stride;
            if (i < nw) {
                if (load)
                    rp_put(a, i, live, v[u]);
                else
                    b[i] = v[u];
            }
        }
    }
}

/* Load, step 3: both trees from their leaves, RP_REBUILD_LEVELS levels per launch.  CTA b owns the subtree above nodes
 * [first + b 2^RP_REBUILD_LEVELS, first + (b + 1) 2^RP_REBUILD_LEVELS) of the starting level, with a barrier between levels: 2
 * launches for 2^20 slots where the per-level kernel k_rp_level takes 20, whose launch gaps made a restore of a 1 GB bank 15 %
 * slower (DESIGN §9).  Same op as k_rp_level per node, so the same nodes bit for bit. */
constexpr int RP_REBUILD_LEVELS = 11;
__global__ void __launch_bounds__(1024) k_rp_rebuild(ReplayDev d, int first, int levels) {
    for (int lv = 1; lv <= levels; ++lv) {
        const int width = first >> lv, per = (1 << RP_REBUILD_LEVELS) >> lv;
        for (int i = threadIdx.x; i < per && blockIdx.x * per + i < width; i += blockDim.x) {
            const int node = width + blockIdx.x * per + i;
            d.sum[node] = d.sum[2 * node] + d.sum[2 * node + 1];
            const double a = d.mn[2 * node], b = d.mn[2 * node + 1];
            d.mn[node] = b < a ? b : a;
        }
        __syncthreads();
    }
}
static int rp_rebuild(AgarReplay* rp, cudaStream_t s) {
    for (int first = rp->d.itcap; first > 1;) {
        int levels = 0;
        while (levels < RP_REBUILD_LEVELS && (first >> levels) > 1) ++levels;
        k_rp_rebuild<<<first > (1 << RP_REBUILD_LEVELS) ? first >> RP_REBUILD_LEVELS : 1, 1024, 0, s>>>(rp->d, first, levels);
        rp->launches += 1;
        first >>= levels;
    }
    RCU(cudaGetLastError());
    return AGAR_OK;
}

extern "C" int agar_replay_create(int capacity, int state_len, int action_len, int prioritized, double alpha, double beta,
                                  int device, AgarReplay** out) {
    AgarReplay* rp = nullptr;
    if (!out || capacity < 1 || state_len < 1 || action_len < 1 || action_len > 32) return rp_fail(nullptr, AGAR_E_INVALID, "bad arguments");
    if (prioritized && (alpha < 0 || beta <= 0)) return rp_fail(nullptr, AGAR_E_INVALID, "alpha >= 0 and beta > 0 required");
    RCU(cudaSetDevice(device));
    rp = (AgarReplay*)calloc(1, sizeof(AgarReplay));
    ReplayDev& d = rp->d;
    d.cap = capacity, d.L = state_len, d.AL = action_len, d.prioritized = prioritized, d.alpha = alpha, d.beta = beta;
    d.itcap = 1;
    while (d.itcap < capacity) d.itcap *= 2;
    rp->device = device;
    size_t cap = (size_t)capacity;
    if (cudaMalloc(&d.obs_t, cap * state_len * 4) != cudaSuccess || cudaMalloc(&d.obs_tp1, cap * state_len * 4) != cudaSuccess ||
        cudaMalloc(&d.action, cap * action_len * 4) != cudaSuccess || cudaMalloc(&d.reward, cap * 4) != cudaSuccess ||
        cudaMalloc(&d.done, cap) != cudaSuccess || cudaMalloc(&d.sum, (size_t)2 * d.itcap * 8) != cudaSuccess ||
        cudaMalloc(&d.mn, (size_t)2 * d.itcap * 8) != cudaSuccess || cudaMalloc(&d.counters, RP_COUNTER_BYTES) != cudaSuccess ||
        cudaMalloc(&d.max_priority, 8) != cudaSuccess) {
        cudaGetLastError();
        free(rp);
        return rp_fail(nullptr, AGAR_E_NOMEM, "cudaMalloc of the replay storage failed");
    }
    k_rp_init<<<(2 * d.itcap + 255) / 256, 256>>>(d);
    RCU(cudaDeviceSynchronize());
    rp->launches = 1;
    *out = rp;
    return AGAR_OK;
}
extern "C" int agar_replay_destroy(AgarReplay* rp) {
    if (!rp) return AGAR_E_INVALID;
    cudaSetDevice(rp->device);
    ReplayDev& d = rp->d;
    cudaFree(d.obs_t), cudaFree(d.obs_tp1), cudaFree(d.action), cudaFree(d.reward), cudaFree(d.done);
    cudaFree(d.sum), cudaFree(d.mn), cudaFree(d.counters), cudaFree(d.max_priority);
    if (d.pos) cudaFree(d.pos);
    free(rp);
    return AGAR_OK;
}
extern "C" const char* agar_replay_last_error(const AgarReplay* rp) { return rp ? rp->err : g_rp_err; }
extern "C" int64_t agar_replay_launch_count(const AgarReplay* rp) { return rp ? rp->launches : 0; }
static int rp_counter(AgarReplay* rp, int which, void* stream) {
    int v = 0;
    if (cudaSetDevice(rp->device) != cudaSuccess) return AGAR_E_CUDA;
    if (cudaMemcpyAsync(&v, rp->d.counters + which, 4, cudaMemcpyDeviceToHost, (cudaStream_t)stream) != cudaSuccess) return AGAR_E_CUDA;
    if (cudaStreamSynchronize((cudaStream_t)stream) != cudaSuccess) return AGAR_E_CUDA;
    return v;
}
/* sticky AGAR_RP_ERR_* bits raised on the device since create (sampling from a buffer that is too small, an index outside
 * [0, size), a priority <= 0): where the reference raises / asserts, the kernels skip the offending element and flag it */
extern "C" int agar_replay_error_flags(AgarReplay* rp, void* stream) { return rp ? rp_counter(rp, 3, stream) : AGAR_E_INVALID; }
extern "C" int agar_replay_size(AgarReplay* rp, void* stream) { return rp ? rp_counter(rp, 1, stream) : AGAR_E_INVALID; }
extern "C" int agar_replay_next_idx(AgarReplay* rp, void* stream) { return rp ? rp_counter(rp, 0, stream) : AGAR_E_INVALID; }

extern "C" int agar_replay_add_batch(AgarReplay* rp, const float* obs_t, const float* action, const float* reward,
                                     const float* obs_tp1, const uint8_t* done, const uint8_t* valid, int n, void* stream) {
    if (!rp || !obs_t || !action || !reward || !obs_tp1 || !done || n < 0) return AGAR_E_INVALID;
    if (n == 0) return AGAR_OK;
    RCU(cudaSetDevice(rp->device));
    cudaStream_t s = (cudaStream_t)stream;
    if (n > rp->pos_cap) {
        if (rp->d.pos) RCU(cudaFree(rp->d.pos));
        RCU(cudaMalloc(&rp->d.pos, (size_t)n * 4));
        rp->pos_cap = n;
    }
    k_rp_scan<<<1, 1024, 0, s>>>(rp->d, valid, n);
    k_rp_store<<<(int)(((size_t)n * 32 + 255) / 256), 256, 0, s>>>(rp->d, obs_t, action, reward, obs_tp1, done, n);
    RCU(cudaGetLastError());
    rp->launches += 2;
    if (rp->d.prioritized) return rp_fix_paths(rp, rp->d.pos, n, s);
    return AGAR_OK;
}
extern "C" int agar_replay_gather(AgarReplay* rp, const int32_t* idx_dev, int batch, float* obs_t, float* action, float* reward,
                                  float* obs_tp1, uint8_t* done, void* stream) {
    if (!rp || !idx_dev || batch < 0) return AGAR_E_INVALID;
    if (batch == 0) return AGAR_OK;
    RCU(cudaSetDevice(rp->device));
    k_rp_gather<<<(int)(((size_t)batch * 32 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(rp->d, idx_dev, batch, obs_t, action, reward,
                                                                                            obs_tp1, done);
    RCU(cudaGetLastError());
    rp->launches += 1;
    return AGAR_OK;
}
extern "C" int agar_replay_sample_uniform(AgarReplay* rp, const double* u_dev, int batch, int32_t* idx_out, float* obs_t,
                                          float* action, float* reward, float* obs_tp1, uint8_t* done, void* stream) {
    if (!rp || !u_dev || !idx_out || batch < 0) return AGAR_E_INVALID;
    if (batch == 0) return AGAR_OK;
    RCU(cudaSetDevice(rp->device));
    k_rp_uniform_idx<<<(batch + 255) / 256, 256, 0, (cudaStream_t)stream>>>(rp->d, u_dev, batch, idx_out);
    RCU(cudaGetLastError());
    rp->launches += 1;
    return agar_replay_gather(rp, idx_out, batch, obs_t, action, reward, obs_tp1, done, stream);
}
extern "C" int agar_replay_sample_prioritized(AgarReplay* rp, const double* u_dev, int batch, int32_t* idx_out, double* weights_out,
                                              float* obs_t, float* action, float* reward, float* obs_tp1, uint8_t* done,
                                              void* stream) {
    if (!rp || !u_dev || !idx_out || batch < 0) return AGAR_E_INVALID;
    if (!rp->d.prioritized) return rp_fail(rp, AGAR_E_UNSUPPORTED, "buffer was created without priorities");
    if (batch == 0) return AGAR_OK;
    RCU(cudaSetDevice(rp->device));
    k_rp_per_sample<<<(batch + 127) / 128, 128, 0, (cudaStream_t)stream>>>(rp->d, u_dev, batch, idx_out, weights_out);
    RCU(cudaGetLastError());
    rp->launches += 1;
    return agar_replay_gather(rp, idx_out, batch, obs_t, action, reward, obs_tp1, done, stream);
}
extern "C" int agar_replay_update_priorities(AgarReplay* rp, const int32_t* idx_dev, const double* priorities_dev, int batch,
                                             void* stream) {
    if (!rp || !idx_dev || !priorities_dev || batch < 0) return AGAR_E_INVALID;
    if (!rp->d.prioritized || batch == 0) return AGAR_OK; /* ReplayBuffer.update_priorities is a no-op (:69-70) */
    RCU(cudaSetDevice(rp->device));
    cudaStream_t s = (cudaStream_t)stream;
    const int staged = batch <= 12288; /* 48 KB of shared memory */
    k_rp_set_priorities<<<(batch + 127) / 128, 128, staged ? (size_t)batch * 4 : 0, s>>>(rp->d, idx_dev, priorities_dev, batch, staged);
    k_rp_max_priority<<<1, 256, 0, s>>>(rp->d, priorities_dev, batch);
    RCU(cudaGetLastError());
    rp->launches += 2;
    return rp_fix_paths(rp, idx_dev, batch, s);
}

extern "C" int64_t agar_replay_state_bytes(const AgarReplay* rp) { return rp ? rp_state_layout(rp->d).off[RP_SECTIONS] : AGAR_E_INVALID; }
/* a bank must be 16-byte aligned (the copy moves 16-byte words) and must not overlap any allocation of the buffer */
static int rp_bank_check(AgarReplay* rp, const void* bank, const char* what) {
    char msg[160];
    const ReplayDev& d = rp->d;
    const char* why = nullptr;
    const uintptr_t b0 = (uintptr_t)bank, b1 = b0 + (uintptr_t)rp_state_layout(d).off[RP_SECTIONS];
    const size_t cap = (size_t)d.cap;
    const struct {
        const void* p;
        size_t n;
    } own[] = {{d.obs_t, cap * d.L * 4},         {d.obs_tp1, cap * d.L * 4},         {d.action, cap * d.AL * 4},
               {d.reward, cap * 4},              {d.done, cap},                      {d.sum, (size_t)2 * d.itcap * 8},
               {d.mn, (size_t)2 * d.itcap * 8}, {d.counters, RP_COUNTER_BYTES},   {d.max_priority, 8},
               {d.pos, (size_t)rp->pos_cap * 4}};
    if (!bank)
        why = "bank is NULL";
    else if (b0 % 16)
        why = "bank is not 16-byte aligned";
    for (const auto& o : own)
        if (!why && o.p && b0 < (uintptr_t)o.p + o.n && (uintptr_t)o.p < b1) why = "bank overlaps the buffer's own allocations";
    if (!why) return AGAR_OK;
    snprintf(msg, sizeof msg, "%s: %s", what, why);
    return rp_fail(rp, AGAR_E_INVALID, msg);
}
static dim3 rp_state_grid(const RpStateLayout& s) {
    int64_t most = 0;
    for (int i = 0; i < RP_SECTIONS; ++i) most = s.off[i + 1] - s.off[i] > most ? s.off[i + 1] - s.off[i] : most;
    const int64_t blocks = (most / 16 + 256 * RP_COPY_U - 1) / (256 * RP_COPY_U);
    return dim3((unsigned)(blocks < 1 ? 1 : blocks > 1024 ? 1024 : blocks), RP_SECTIONS);
}
extern "C" int agar_replay_save(AgarReplay* rp, void* bank_dev, void* stream) {
    if (!rp) return AGAR_E_INVALID;
    const int rc = rp_bank_check(rp, bank_dev, "agar_replay_save");
    if (rc != AGAR_OK) return rc;
    RCU(cudaSetDevice(rp->device));
    const RpStateLayout s = rp_state_layout(rp->d);
    k_rp_state<<<rp_state_grid(s), 256, 0, (cudaStream_t)stream>>>(rp->d, s, (uint8_t*)bank_dev, 0);
    RCU(cudaGetLastError());
    rp->launches += 1;
    return AGAR_OK;
}
/* validate, then install (a refused bank installs nothing), then rebuild the trees from their leaves: a rebuild after a refusal
 * recomputes the same nodes from the same leaves, so the buffer stays as it was without a host synchronisation */
extern "C" int agar_replay_load(AgarReplay* rp, const void* bank_dev, void* stream) {
    if (!rp) return AGAR_E_INVALID;
    const int rc = rp_bank_check(rp, bank_dev, "agar_replay_load");
    if (rc != AGAR_OK) return rc;
    RCU(cudaSetDevice(rp->device));
    cudaStream_t s = (cudaStream_t)stream;
    const RpStateLayout lay = rp_state_layout(rp->d);
    const int64_t pairs = rp->d.prioritized ? ((int64_t)rp->d.cap + 1) / 2 : 1;
    const int vblocks = (int)((pairs + 255) / 256 > 1024 ? 1024 : (pairs + 255) / 256);
    RCU(cudaMemsetAsync(rp->d.counters + 4, 0, 4, s));
    k_rp_validate<<<vblocks, 256, 0, s>>>(rp->d, lay, (const uint8_t*)bank_dev);
    k_rp_state<<<rp_state_grid(lay), 256, 0, s>>>(rp->d, lay, (uint8_t*)bank_dev, 1);
    RCU(cudaGetLastError());
    rp->launches += 2;
    return rp->d.prioritized ? rp_rebuild(rp, s) : AGAR_OK;
}
