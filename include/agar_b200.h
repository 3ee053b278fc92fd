/*
 * agar_b200.h — C ABI of the B200-native batched agar.io env step.
 *
 * The reference (NILOIDE/A.I.gar) has no FFI layer: its boundary is the Python
 * object API of src/model/{model,field,player,cell,bot}.py.  Every entry point
 * below names the reference call(s) it replaces (file:line under
 * /root/reference/src).  Plain pointers and sizes only; no torch / C++ types.
 *
 * Conventions
 *   - every function returns AGAR_OK (0) or a negative AGAR_E_* code;
 *     agar_last_error() returns a human readable message for the last failure
 *     on that handle (or the last create failure when env == NULL).
 *   - pointers suffixed _dev are device pointers on the handle's GPU; pointers
 *     suffixed _host are ordinary host pointers.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default
 *     stream).  All device work is enqueued on it; nothing synchronises the
 *     host unless the function says so.
 *   - a handle is bound to one device and is not thread-safe.
 *
 * The same structs describe the per-env state RECORD (one contiguous block per
 * env in HBM, see DESIGN.md §3).  The CPU oracle (oracle/agar_oracle.c, test
 * infrastructure) uses the identical record so that state can be moved between
 * the two for parity checks (agar_debug_dump / agar_debug_load).
 */
#ifndef AGAR_B200_H
#define AGAR_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AGAR_ABI_VERSION 1

#define AGAR_MAX_PLAYERS 16  /* K: bots per field (config 4 uses 16)                  */
#define AGAR_MAX_CELLS   16  /* cells per player, src/model/player.py:59, field.py:353 */
#define AGAR_ACTION_DIM  4   /* x, y, split, eject — src/model/bot.py:550-577          */

enum { AGAR_OK = 0, AGAR_E_INVALID = -1, AGAR_E_CUDA = -2, AGAR_E_NOMEM = -3, AGAR_E_UNSUPPORTED = -4,
       AGAR_E_RANGE = -5 };

/* bot kinds, creation order NN.., Greedy.., Random.. as src/aigar.py:778-780 */
enum { AGAR_BOT_NN = 0, AGAR_BOT_GREEDY = 1, AGAR_BOT_RANDOM = 2 };

/* grid-vision binning: reproduce src/model/spatialHashTable.py:19,91-112 operation by operation
 * (including the ceil()/int() rounding artefacts), or the canonical G-column binning */
enum { AGAR_OBS_REFERENCE = 0, AGAR_OBS_CANONICAL = 1 };
/* length of Bot.getSimpleStateRepresentation: 3 (own cell) + 3 (closest enemy) + 2 (closest pellet) + 4 (field edges) */
#define AGAR_SIMPLE_STATE_LEN 12

/* ------------------------------------------------------------------ config */
/* Mirrors the flag subset of src/model/networkParameters.py that the env path reads
 * (SURVEY.md §2 rows 6-7) plus pool capacities. */
typedef struct AgarConfig {
    int32_t n_players;                    /* NUM_NN_BOTS + NUM_GREEDY_BOTS + NUM_RANDOM_BOTS        */
    int32_t bot_type[AGAR_MAX_PLAYERS];   /* AGAR_BOT_* per player slot                              */
    int32_t virus_enabled;                /* VIRUS_SPAWN              networkParameters.py:11        */
    int32_t enable_split;                 /* ENABLE_SPLIT             :37                            */
    int32_t enable_eject;                 /* ENABLE_EJECT             :38                            */
    int32_t enable_greedy_split;          /* ENABLE_GREEDY_SPLIT      :17 (only 0 supported)         */
    int32_t pellet_spawn;                 /* PELLET_SPAWN             :10                            */
    int32_t grid_squares;                 /* GRID_SQUARES_PER_FOV     :97                            */
    int32_t frame_skip;                   /* FRAME_SKIP_RATE          :33                            */
    int32_t pellet_grid, self_grid, wall_grid, enemy_grid, virus_grid;      /* :78-84               */
    int32_t self_grid_lf, self_grid_slf, enemy_grid_lf, enemy_grid_slf;     /* :80-86               */
    int32_t use_fovsize, use_last_fovsize, use_totalmass;                   /* :92-94               */
    int32_t use_last_action, use_second_last_action;                        /* :95-96               */
    int32_t mass_as_reward;               /* MASS_AS_REWARD           :50                            */
    int32_t obs_mode;                     /* AGAR_OBS_*                                              */
    int32_t fat_cap;                      /* ex-blob pellet pool (0 = default)                       */
    int32_t virus_cap;                    /* virus pool          (0 = default)                       */
    int32_t blob_cap;                     /* ejected-blob pool   (0 = default)                       */
    int32_t event_cap;                    /* per-frame event log entries per env (0 = no log)        */
    int32_t pellet_cap;                   /* integer-pellet slots; 0 = default (the refill target, field.py:65) */
    int32_t all_player_grid;              /* ALL_PLAYER_GRID :88-91 — one channel with the biggest cell of ANY player per square,
                                           * instead of the self / enemy channels (which must then be off)      */
    int32_t normalize_grid_by_max_mass;   /* NORMALIZE_GRID_BY_MAX_MASS :76-77 as the RUN's parameters module carries it (bot.py:365,412,
                                           * 422,430): the own / enemy / all-player channels are divided by the mass of the biggest
                                           * player cell in view.  (bot.py:402,439 — pellet and virus channels — read the package-
                                           * global flag instead, which the reference's driver never rewrites: not modelled.)      */
    int32_t simple_state;                 /* GRID_VIEW_ENABLED = False (networkParameters.py:119): observations are the 12 values of
                                           * Bot.getSimpleStateRepresentation (bot.py:511-548) — first own cell, closest enemy cell,
                                           * closest pellet (relative to the integer field of view), distances to the visible field
                                           * edges — instead of the grids; state_len = 12, the channel / extra flags are ignored */
    int32_t reserved[3];
    double reward_scale;                  /* REWARD_SCALE :70 */
    double reward_term;                   /* REWARD_TERM  :69 */
    double death_term;                    /* DEATH_TERM   :71 */
    double death_factor;                  /* DEATH_FACTOR :72 */
} AgarConfig;

/* ------------------------------------------------------- per-env state record */
/* A player cell — src/model/cell.py:21-45 (only the attributes the step reads) */
typedef struct AgarCell {
    double x, y;
    double mass, radius;   /* radius is NOT always sqrt(mass/pi): Cell.eject() leaves it stale (cell.py:92) */
    double svx, svy;       /* splitVelocity                                                               */
    double merge_time;     /* mergeTime                                                                   */
    int32_t counter;       /* splitVelocityCounter (15..0, -1 = none; a fresh Cell has 0)                 */
    uint32_t uid;          /* creation serial within the env (object identity for blob.ejecterCell)       */
    uint32_t flags;        /* AGAR_CF_*                                                                   */
    uint32_t pad;
} AgarCell;
enum { AGAR_CF_EJECT = 1u,   /* blobToBeEjected                                             */
       AGAR_CF_INHASH = 2u   /* present in field.playerHashTable (field.py:121-126,402-404) */ };

/* virus / ejected blob — both are player-less Cells with momentum */
typedef struct AgarMote {
    double x, y, mass, radius, svx, svy;
    int32_t counter;
    uint32_t aux;          /* virus: AGAR_CF_INHASH flag; blob: uid of the ejecting cell */
} AgarMote;

/* a blob that lost its momentum and became a pellet with float position (field.py:107-110) */
typedef struct AgarFatPellet {
    double x, y, mass, radius;   /* mass == 0 marks a free slot */
} AgarFatPellet;

/* Bot bookkeeping — src/model/bot.py:125-232 */
typedef struct AgarBot {
    int32_t type;              /* AGAR_BOT_*                                               */
    int32_t has_action;        /* currentAction is not None                                */
    int32_t has_last_action;   /* lastAction is not None                                   */
    int32_t skip_frames;       /* skipFrames                                               */
    int32_t has_last_mass;     /* lastMass is not None                                     */
    int32_t has_old_state;     /* oldState is not None                                     */
    int32_t time;              /* Bot.time (random bot action clock, bot.py:243-249)       */
    int32_t skipping;          /* currentlySkipping of the current bot turn                */
    int32_t turn_begun;        /* agar_observe already ran the first half of this turn     */
    int32_t need_action;       /* alive and not skipping: decideMove() would be called     */
    int32_t exp_valid;         /* an experience tuple was emitted this turn                */
    int32_t exp_done;          /* ... and its new state is None (player dead)              */
    double cur_action[4];      /* currentAction                                            */
    double last_action[4];     /* lastAction                                               */
    double cum_reward;         /* cumulativeReward                                         */
    double last_reward;        /* lastReward                                               */
    double last_mass;          /* lastMass                                                 */
    double fov_size_feat;      /* Bot.fovSize (extra feature memory, bot.py:304-309)       */
    double last_fov_size_feat; /* Bot.lastFovSize                                          */
    double stat_mass_sum;      /* sum of totalMasses (bot.py:253)                          */
    double stat_mass_max;      /* max of totalMasses                                       */
    double stat_frames;        /* len(totalMasses)                                         */
    double stat_deaths;        /* number of deaths of this player                          */
} AgarBot;

/* Player — src/model/player.py:11-28 */
typedef struct AgarPlayer {
    int32_t alive;             /* isAlive                 */
    int32_t respawn_time;      /* respawnTime             */
    int32_t n_cells;           /* len(cells)              */
    int32_t do_split;          /* doSplit                 */
    int32_t do_eject;          /* doEject                 */
    int32_t fov_valid;         /* fovPos / fovSize have been computed at least once */
    double cmd_x, cmd_y;       /* commandPoint            */
    double fov_x, fov_y;       /* fovPos (kept while dead, player.py:156-161) */
    double fov_size;           /* fovSize                 */
    AgarBot bot;
} AgarPlayer;

typedef struct AgarEnvHeader {
    uint32_t rng_field;        /* next serial of Philox stream 0 (field.py draws)   */
    uint32_t rng_bot;          /* next serial of Philox stream 1 (bot.py draws)     */
    uint32_t next_uid;         /* next player-cell creation serial                  */
    uint32_t frame;            /* frames stepped since create/reset                 */
    int32_t n_viruses;         /* len(field.viruses)                                */
    int32_t n_blobs;           /* len(field.blobs)                                  */
    int32_t n_fat;             /* live ex-blob pellets                              */
    int32_t n_pellets;         /* live integer pellets                              */
    int32_t n_dead;            /* len(field.deadPlayers)                            */
    int32_t n_events;          /* events logged for the last stepped frame          */
    uint32_t overflow;         /* AGAR_OVF_* bits, sticky                           */
    uint32_t pad0;
    uint64_t event_hash;       /* order-sensitive running hash of all events since reset except COLLIDE */
    int32_t dead_order[AGAR_MAX_PLAYERS];   /* field.deadPlayers as player indices  */
} AgarEnvHeader;
enum { AGAR_OVF_FAT = 1u, AGAR_OVF_VIRUS = 2u, AGAR_OVF_BLOB = 4u,
       AGAR_OVF_EVENT = 8u /* reserved, never set: a full event ring just stops recording — n_events keeps counting (compare it
                            * with event_cap) and the running event_hash covers every event.  The bit is not raised because the
                            * overflow word is part of the state the parity tests compare with the reference. */ };

/* One logged event.  Parity tests compare these bit for bit against the oracle. */
typedef struct AgarEvent { int32_t type, a, b, c, d; } AgarEvent;
enum {
    AGAR_EV_EAT_PELLET = 1,     /* a=player b=cell uid c=slot (|0x10000 for ex-blob pellets) d=0 — field.py:207-213 */
    AGAR_EV_EAT_BLOB = 2,       /* a=player b=cell uid c=blob index d=ejecter uid                — field.py:215-222 */
    AGAR_EV_EAT_VIRUS = 3,      /* a=player b=cell uid c=virus index d=new cells                 — field.py:225-231,350-370 */
    AGAR_EV_VIRUS_EAT_BLOB = 4, /* a=virus index b=blob index c=1 if the virus split             — field.py:246-253,316-325 */
    AGAR_EV_EAT_CELL = 5,       /* a=eater player b=eater uid c=eaten player d=eaten uid         — field.py:233-244,346-348 */
    AGAR_EV_MERGE = 6,          /* a=player b=bigger uid c=smaller uid                           — field.py:183-198,372-380 */
    AGAR_EV_COLLIDE = 7,        /* a=player b=uid cell c=uid otherCell                           — field.py:149-181 */
    AGAR_EV_SPAWN_PELLET = 8,   /* a=slot b=x c=y d=mass                                          — field.py:303-313 */
    AGAR_EV_SPAWN_VIRUS = 9,    /* a=virus index b=trunc(x) c=trunc(y)                            — field.py:262-275 */
    AGAR_EV_SPAWN_PLAYER = 10,  /* a=player b=uid c=x d=y                                         — field.py:49-55,277-301 */
    AGAR_EV_SPLIT = 11,         /* a=player b=parent uid c=twin uid                               — player.py:53-61 */
    AGAR_EV_EJECT = 12,         /* a=player b=cell uid c=blob index                               — field.py:134-146 */
    AGAR_EV_BLOB_TO_PELLET = 13,/* a=fat slot                                                     — field.py:99-110 */
    AGAR_EV_PLAYER_DIED = 14    /* a=player                                                       — field.py:382-388 */
};

/* Byte layout of one env record (all offsets from the record start).  Filled by
 * agar_layout_for_config(); identical for the oracle and the GPU library. */
typedef struct AgarLayout {
    int32_t field_size;        /* S = int(75*sqrt(K))            field.py:58            */
    int32_t n_players;         /* K                                                     */
    int32_t cell_cap;          /* cells stored per player (16, or 1 when nothing can split) */
    int32_t pellet_cap;        /* P = number of integer pellet slots (field.py:65,303-305) */
    int32_t fat_cap, virus_cap, blob_cap, event_cap;
    int32_t grid_squares;      /* G                                                     */
    int32_t n_grids;           /* NUM_OF_GRIDS             networkParameters.py:98-100  */
    int32_t n_extra;           /* EXTRA_INPUT              :101                         */
    int32_t state_len;         /* L = STATE_REPR_LEN       :102                         */
    int32_t n_agents;          /* number of NN bots (always the first player slots)     */
    int32_t action_len;        /* 2, 3 or 4 — len(action) the reference learner emits   */
    int32_t n_hist;            /* history grids kept per agent (4)                      */
    int32_t pad;
    double max_pellets;        /* maxCollectibleCount (float) field.py:65               */
    double max_viruses;        /* maxVirusCount       (float) field.py:66               */
    uint64_t off_header, off_players, off_cells, off_viruses, off_blobs, off_fat, off_pellets, off_hist,
        off_events;
    uint64_t record_bytes;     /* multiple of 128                                       */
} AgarLayout;

/* integer pellet slot: x | y<<10 | mass<<20 ; 0 = free slot.  x,y in [0,S) from
 * randint(0,S), mass in {1,2,3} from randomSize() (field.py:20-26,307-313). */
#define AGAR_PELLET_PACK(x, y, m) ((uint32_t)(x) | ((uint32_t)(y) << 10) | ((uint32_t)(m) << 20))
#define AGAR_PELLET_X(p) ((int)((p) & 1023u))
#define AGAR_PELLET_Y(p) ((int)(((p) >> 10) & 1023u))
#define AGAR_PELLET_M(p) ((int)((p) >> 20))

/* which per-agent quantity agar_get() copies out ([E][A] row-major, A = n_agents) */
typedef enum AgarField {
    AGAR_GET_REWARD = 0,      /* float  — Bot.getLastReward()           bot.py:645        */
    AGAR_GET_DONE = 1,        /* uint8  — emitted next state is None    bot.py:202,217    */
    AGAR_GET_VALID = 2,       /* uint8  — an experience was emitted     bot.py:204-216    */
    AGAR_GET_NEED_ACTION = 3, /* uint8  — decideMove() is due           bot.py:223-226    */
    AGAR_GET_MASS = 4,        /* float  — Player.getTotalMass()         player.py:129     */
    AGAR_GET_FOV = 5,         /* float  — Player.getFovSize()           player.py:163     */
    AGAR_GET_NCELLS = 6,      /* int32  — len(player.cells)                               */
    AGAR_GET_ALIVE = 7,       /* uint8  — Player.getIsAlive()           player.py:180     */
    AGAR_GET_STATS = 8,       /* double[4] per agent: sum, max, count of totalMasses, deaths (bot.py:253) */
    AGAR_GET_OVERFLOW = 9,    /* uint32 per ENV ([E]) — sticky AGAR_OVF_* bits            */
    AGAR_GET_EVENT_HASH = 10  /* uint64 per ENV ([E]) — running event hash                */
} AgarField;

typedef struct AgarEnv AgarEnv; /* opaque */

/* Fill `out` with the record layout a config implies.  Pure host arithmetic, no GPU. */
int agar_layout_for_config(const AgarConfig* cfg, AgarLayout* out);

/* Model(...) + createBot(...)*K + Model.initialize()  — src/model/model.py:51,154-162,90-94;
 * src/model/field.py:57-67.  Allocates n_envs records on `device`, seeds env e with the Philox key
 * (seed, first_env_id + e) and runs the initial spawn on `stream`. */
int agar_create(const AgarConfig* cfg, int n_envs, int device, uint64_t seed, uint64_t first_env_id, void* stream,
                AgarEnv** out);
int agar_destroy(AgarEnv* env);
const char* agar_last_error(const AgarEnv* env);
int agar_get_layout(const AgarEnv* env, AgarLayout* out);
int agar_num_envs(const AgarEnv* env);

/* Model.resetModel()  — model.py:96-98, field.py:69-83.  env_mask_dev: uint8[E] or NULL (= all). */
int agar_reset(AgarEnv* env, const uint8_t* env_mask_dev, void* stream);
/* Model.resetBots()   — model.py:118-120, bot.py:125-164 */
int agar_reset_bots(AgarEnv* env, const uint8_t* env_mask_dev, void* stream);

/* First half of every NN bot's turn (bot.py:195-217): accumulate reward, frame-skip bookkeeping and,
 * for agents that are not skipping, the state representation (bot.py:272-299, 326-497).
 * obs_dev: float[E][A][L] (rows of skipping / dead agents are left untouched).  Results of the
 * turn (reward, done, valid, need_action) are read with agar_get().  Idempotent within a frame. */
int agar_observe(AgarEnv* env, float* obs_dev, void* stream);

/* Second half of the bot turns + n_frames x Field.update()  (model.py:100-112, bot.py:223-232,252-270,
 * field.py:85-92).  actions_dev: float[E][A][4] in [0,1]; an agent whose decideMove() is due in any of the
 * n_frames frames takes its row.  Scripted bots (Greedy/Random) are advanced inside. */
int agar_step(AgarEnv* env, const float* actions_dev, int n_frames, void* stream);

/* Fused rollout primitive for lock-stepped agents: agar_step(actions, n_frames) followed by agar_observe(obs)
 * in one launch (one decision period = FRAME_SKIP_RATE+1 frames, aigar.py:844-849). */
int agar_step_observe(AgarEnv* env, const float* actions_dev, int n_frames, float* obs_dev, void* stream);

/* The random-action driver of BASELINE.json configs[1] ("random-action driver, 1000-step rollouts") in ONE launch:
 * n_decisions x ( agar_observe -> action = 4 uniforms of Philox(counter = (decision_base + d, 7, env id, agent),
 * key = seed) -> n_frames frames ).  Replaces the collector loop src/aigar.py:844-849 driven by a random
 * learner.  obs_dev (nullable) is rewritten with every decision's observation. */
int agar_rollout_random(AgarEnv* env, int n_decisions, int n_frames, uint32_t decision_base, float* obs_dev,
                        void* stream);

int agar_get(AgarEnv* env, AgarField which, void* out_dev, void* stream);

/* lanes of a warp that cooperate on one env (1, 2, 4, 8, 16, 32; multi-cell configs: 4..32).  A tuning knob:
 * results are identical for every width. */
int agar_set_tile_width(AgarEnv* env, int lanes);
int agar_get_tile_width(const AgarEnv* env);
/* device pointer of the env records ([n_envs][record_bytes]); read-only use (checksums, DLPack export) */
void* agar_state_ptr(const AgarEnv* env);

/* parity / debugging: copy one env record device->host (synchronises `stream`) or host->device. */
int agar_debug_dump(AgarEnv* env, int env_index, void* record_host, size_t bytes, void* stream);
int agar_debug_load(AgarEnv* env, int env_index, const void* record_host, size_t bytes, void* stream);

/* number of kernels this handle has launched so far (bench.py's gpu_launches) */
int64_t agar_launch_count(const AgarEnv* env);
/* how many of them handed their observations to observer warps (single-cell rollouts at 4 / 8 lanes per env) */
int64_t agar_observer_launch_count(const AgarEnv* env);

/* ---- host-buffer convenience path (the e2e call: host arrays in, host arrays out) ----
 * actions_host float[E][A][4] -> H2D, n_frames frames, observe, D2H of obs/reward/done.
 * Buffers should be pinned for full PCIe speed: pinned (device-visible) actions_host / obs_host are read and written in
 * place by the kernels, pageable ones go through staging copies.  Synchronises `stream` before returning. */
int agar_step_host(AgarEnv* env, const float* actions_host, int n_frames, float* obs_host, float* reward_host,
                   uint8_t* done_host, void* stream);
/* The same call in two halves, so that a caller can keep several groups of envs (one handle + one stream each) in
 * flight: _begin enqueues H2D + frames + observe + D2H and returns at once; _end waits for that group and fills
 * reward / done.  obs_host and actions_host must stay valid (and should be pinned) until _end returns.
 * agar_step_host == _begin followed by _end. */
int agar_step_host_begin(AgarEnv* env, const float* actions_host, int n_frames, float* obs_host, void* stream);
int agar_step_host_end(AgarEnv* env, float* reward_host, uint8_t* done_host, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AGAR_B200_H */
