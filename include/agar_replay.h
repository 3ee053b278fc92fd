/*
 * agar_replay.h — C ABI of the GPU replay buffer (SURVEY.md §8f rank 1: the step right after the env path).
 *
 * Replaces src/model/replay_buffer.py (ReplayBuffer :7-73, PrioritizedReplayBuffer :76-209) and
 * src/model/common/segment_tree.py for batches of transitions that never leave the GPU: the env's observation /
 * reward / done buffers (agar_b200.h) are appended straight into the ring.  Same conventions as agar_b200.h.
 *
 * Randomness is the caller's: every sampling entry takes uniforms in [0, 1) (the reference draws them with the
 * stdlib `random` module, replay_buffer.py:66,116), so results are reproducible and comparable with the reference.
 */
#ifndef AGAR_REPLAY_H
#define AGAR_REPLAY_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct AgarReplay AgarReplay; /* opaque */

/* ReplayBuffer(size) / PrioritizedReplayBuffer(size, alpha, beta) — replay_buffer.py:8-19,77-106 */
int agar_replay_create(int capacity, int state_len, int action_len, int prioritized, double alpha, double beta, int device,
                       AgarReplay** out);
int agar_replay_destroy(AgarReplay* rp);
const char* agar_replay_last_error(const AgarReplay* rp);
/* len(buffer) and _next_idx (synchronise `stream`) */
int agar_replay_size(AgarReplay* rp, void* stream);
int agar_replay_next_idx(AgarReplay* rp, void* stream);

/* ReplayBuffer.add (:24-31) / PrioritizedReplayBuffer.add (:108-113) for the n candidate transitions of one tick:
 * those with valid[i] != 0 (an experience was emitted, bot.py:204-217) are appended in index order.  All pointers
 * are device pointers: obs_t, obs_tp1 float[n][state_len], action float[n][action_len], reward float[n],
 * done uint8[n], valid uint8[n] (NULL = all valid). */
int agar_replay_add_batch(AgarReplay* rp, const float* obs_t, const float* action, const float* reward,
                          const float* obs_tp1, const uint8_t* done, const uint8_t* valid, int n, void* stream);

/* ReplayBuffer._encode_sample (:33-44): gather the transitions idx[0..batch) */
int agar_replay_gather(AgarReplay* rp, const int32_t* idx_dev, int batch, float* obs_t, float* action, float* reward,
                       float* obs_tp1, uint8_t* done, void* stream);
/* ReplayBuffer.sample (:46-67): idx[i] = randint(0, len - 1) drawn as floor(u[i] * len), then gather */
int agar_replay_sample_uniform(AgarReplay* rp, const double* u_dev, int batch, int32_t* idx_out, float* obs_t, float* action,
                               float* reward, float* obs_tp1, uint8_t* done, void* stream);
/* PrioritizedReplayBuffer.sample (:113-171): mass = u[i] * sum(0, len - 1), idx = find_prefixsum_idx(mass);
 * weights[i] = ((p_i * len) ** -beta) / max_weight */
int agar_replay_sample_prioritized(AgarReplay* rp, const double* u_dev, int batch, int32_t* idx_out, double* weights_out,
                                   float* obs_t, float* action, float* reward, float* obs_tp1, uint8_t* done, void* stream);
/* PrioritizedReplayBuffer.update_priorities (:173-195) */
int agar_replay_update_priorities(AgarReplay* rp, const int32_t* idx_dev, const double* priorities_dev, int batch, void* stream);
/* Sticky error bits raised ON THE DEVICE since create (synchronises `stream`).  Where the reference raises — sampling an empty
 * buffer (random.randint(0, -1), replay_buffer.py:66; the prioritized path recurses without end for len < 2, :116) — or asserts
 * (0 <= idx < len(storage), priority > 0, :203-204), the kernels skip the offending element (index 0 / weight 0 is returned,
 * trees are left untouched) and set a bit here instead of hanging or corrupting memory.  AGAR_RP_ERR_STATE: a bank refused by
 * agar_replay_load (below). */
enum { AGAR_RP_ERR_EMPTY = 1, AGAR_RP_ERR_INDEX = 2, AGAR_RP_ERR_PRIORITY = 4, AGAR_RP_ERR_STATE = 8 };
int agar_replay_error_flags(AgarReplay* rp, void* stream);
/* number of kernels launched so far */
int64_t agar_replay_launch_count(const AgarReplay* rp);

/* ---- state snapshots: the whole observable state of a buffer in one caller-owned device bank (checkpoint, resume, clone).
 *
 * Bank layout (every offset 64-bit; each section starts on a 256-byte boundary, the bank is padded to one):
 *   [0, 256)   AgarReplayStateHeader below, zero-padded
 *   obs_t      float [cap][state_len]
 *   obs_tp1    float [cap][state_len]
 *   action     float [cap][action_len]
 *   reward     float [cap]
 *   done       uint8 [cap]
 *   leaf       double [cap]   prioritized buffers only: the common leaf of the sum and min trees
 * The trees' internal nodes are not stored: a node is op(left child, right child), so a load installs the leaves and
 * rebuilds both trees.  Below `size` the sum and min leaves are equal; at and above it they are 0 and +inf.
 *
 * Banks are canonical: a save writes zeros for every ring row and leaf at index >= size and for all padding, so two buffers
 * with the same observable state give byte-identical banks.
 *
 * Not state, and left as they are by a load: the sticky error flags, the n_valid of the last add and the add scratch.
 * A load copies into the buffer's existing allocations, so a CUDA graph that captured this buffer's kernels sees the restored
 * contents on its next replay. */
typedef struct AgarReplayStateHeader {
    int64_t capacity, state_len, action_len, prioritized; /* prioritized: 0 or 1 */
    uint64_t alpha_bits, beta_bits;                       /* the float64 bits of alpha and beta */
    int64_t next_idx, size;
    double max_priority;
} AgarReplayStateHeader;

/* bytes of one bank of this buffer (< 0: an AGAR_E_* code) */
int64_t agar_replay_state_bytes(const AgarReplay* rp);
/* Write the buffer's state into bank_dev (agar_replay_state_bytes bytes, 16-byte aligned, on the buffer's device, not
 * overlapping any of its allocations).  One kernel launch on `stream`; no host synchronisation, no allocation. */
int agar_replay_save(AgarReplay* rp, void* bank_dev, void* stream);
/* Install a bank written by agar_replay_save of a buffer created with the same capacity, state_len, action_len, prioritized,
 * alpha and beta.  Enqueued on `stream` without host synchronisation or allocation: a 4-byte memset of the verdict word, a
 * validation kernel, an install kernel that copies only if the verdict is good, and for prioritized buffers the rebuild of
 * both trees from their leaves, 11 tree levels per launch: ceil(log2(capacity rounded up to a power of two) / 11) launches
 * (1 up to 2048 slots, 2 up to 4M).  So 2 launches, plus the rebuild's.
 *
 * The device refuses the bank, sets AGAR_RP_ERR_STATE and leaves the buffer unchanged bit for bit when: a header shape field
 * (capacity, state_len, action_len, prioritized, alpha or beta bits) differs from the buffer's; next_idx is outside [0, cap)
 * or size outside [0, cap]; size < cap and next_idx != size; max_priority is NaN or outside [1, 1.7e308]; or, for a
 * prioritized buffer, a leaf at index >= size is not +0.0 or a leaf below size is NaN or negative (0 and +inf are reachable
 * leaves below size: agar_pow underflows and overflows for alpha >= 1).
 * The host refuses (AGAR_E_INVALID) a NULL bank, a bank that is not 16-byte aligned or one that overlaps the buffer's own
 * allocations; agar_replay_save does the same. */
int agar_replay_load(AgarReplay* rp, const void* bank_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AGAR_REPLAY_H */
