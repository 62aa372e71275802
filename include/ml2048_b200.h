/*
 * ml2048_b200.h -- C ABI of the B200-native VecGame hot path (libml2048_b200.so).
 *
 * The reference (tsangwpx/ml2048) has no FFI layer: its boundary for this path is the Python class
 * `VecGame` plus the Numba-jitted functions it calls (reference: src/ml2048/game_numba.py).  Every
 * entry point below replaces one of those jitted functions / host loops; the citation says which.
 * The Python shim `ml2048_b200.VecGame` keeps the reference's class surface and calls these through
 * ctypes (see INTEGRATION.md for the binding a maintainer would add on the reference side).
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless named host_*;
 *   - the library never allocates, frees or retains memory (except ml2048_alloc_compressible / ml2048_free_compressible,
 *     which do nothing else);  all work is enqueued on `stream`
 *     (a cudaStream_t passed as void*) and the call returns immediately: no hidden synchronisation,
 *     CUDA-graph capturable;
 *   - return value: 0 = ok, negative = argument error (ML2048_E_*), positive = cudaError_t of the launch;
 *   - boards are 16 bytes per game (exponents, 0 = empty, cell = row*4+col, game_numba.py:13-20),
 *     16-byte aligned;  masks are 4 bytes per game (left,right,up,down; game.py:14-17), 4-byte aligned;
 *   - "slot" = index of a game inside this shard; global slot = slot_base + slot (multi-GPU sharding:
 *     table rows and Philox counters use the GLOBAL slot so results do not depend on the shard count).
 */
#ifndef ML2048_B200_H
#define ML2048_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* 12 also covers ml2048_alloc_compressible / ml2048_free_compressible, added without a bump (unlike earlier additions):
 * they change no existing struct or signature, and a loader that binds them by name fails on a library without them. */
#define ML2048_ABI_VERSION 12

#if defined(__GNUC__)
#define ML2048_API __attribute__((visibility("default")))
#else
#define ML2048_API
#endif

/* error codes (negative) */
#define ML2048_E_NULL (-1)    /* required pointer is null */
#define ML2048_E_ALIGN (-2)   /* pointer not aligned as documented */
#define ML2048_E_SIZE (-3)    /* num_games <= 0 or capacity too small */
#define ML2048_E_ENUM (-4)    /* bad enum value */
#define ML2048_E_STRUCT (-5)  /* struct_size does not match this library */
#define ML2048_E_UNSUPPORTED (-6) /* no CUDA driver or device, or the device lacks the feature */

/* reward_fn, selected by identity on the Python side (game_numba.py:408-504) */
enum { ML2048_REWARD_NORMAL = 0, ML2048_REWARD_IMPROVED = 1, ML2048_REWARD_RANK = 2, ML2048_REWARD_MAXCELL = 3 };

/* where spawn randomness comes from */
enum {
    ML2048_RNG_REPLAY = 0, /* the reference's pre-drawn tables: bit-exact (game_numba.py:172-212) */
    ML2048_RNG_PHILOX = 1  /* counter-based: Philox2x32-10 blocks keyed by the seed, counter = (global slot >> 1, step counter);
                              a block's two words serve the two slots of a pair (even slot: word 0, odd slot: word 1).  Separate
                              streams (key ^ tag) for the policy's words, the spawn cells and the auto-reset's cells */
};

/* element type of the `actions` array */
enum { ML2048_ACT_U8 = 0, ML2048_ACT_I32 = 1, ML2048_ACT_I64 = 2 };

/* where actions come from */
enum {
    ML2048_ACTIONS_GIVEN = 0,       /* read `actions` */
    ML2048_ACTIONS_RANDOM_VALID = 1, /* uniform over valid actions, Philox (policy/random.py:17-27);
                                        the chosen action is written to `actions_out` when not null */
    ML2048_ACTIONS_FROM_LOGITS = 2   /* masked categorical sample from the policy head's logits
                                        (_sample_action, policy/actor_critic.py:56-76): invalid actions get
                                        finfo.min, softmax, one Philox uniform picks the action; the action goes to
                                        `actions_out`, its log-probability to `log_prob_out` (when not null) */
};

/* fused observation encoding (policy/_network.py:86-95): out[g][k][c] = (board[g][c] == k), k < 16 */
enum { ML2048_ONEHOT_NONE = 0, ML2048_ONEHOT_F32 = 1, ML2048_ONEHOT_BF16 = 2, ML2048_ONEHOT_U8 = 3 };

/* Episode statistics accumulated on the device (RunnerStats, runner.py:139-189, plus score/step moments).
 * `replicas` copies of this struct are laid out back to back to spread atomics; sum them to read. */
typedef struct {
    unsigned long long max_tile_hist[20]; /* runner.py:150-166: counts[max exponent] of finished games */
    unsigned long long episodes;          /* runner.py:166 terminated_count */
    unsigned long long score_sum;         /* sum of final scores (scores are integers) */
    unsigned long long step_sum;          /* sum of final step counts */
    unsigned long long score_max;         /* max final score */
} ml2048_stats;

#define ML2048_STATS_REPLICAS 64

/* One pre-drawn runner step of the host random schedule, kept on the device so that a CUDA graph can replay
 * many steps without host work.  The reference draws these numbers on the host in every prepare()/step()
 * (game_numba.py:622-626, :670); none depends on game state, so they can be drawn ahead (ml2048_b200/vecgame.py
 * draws them from the same generator in the same order).  When `sched` is set in the argument structs the
 * kernels read entry sched[*sched_cursor] INSTEAD of the scalar fields rand_base / rand_seed / two_mask /
 * philox_counter, and the random tables of slot `table` of the table ring. */
typedef struct {
    int64_t rand_base;        /* prepare: _rand_step + rand_offset (:651) */
    int64_t rand_seed;        /* step:    _rand_step + rand_offset (:681) */
    uint64_t philox_counter;  /* prepare uses this value, step uses this value + 1 */
    uint32_t two_mask;        /* 2-vs-4 mask of the tables in force */
    uint32_t table;           /* slot of the table ring holding the tables in force */
} ml2048_sched_entry;

/* Arguments of one environment step.  Replaces VecGame.step + _vec_step
 * (game_numba.py:660-698, 701-738) including the prev_state / prev_valid_actions copies (:672-673):
 * boards and masks are ping-pong buffers, so board_in / valid_in ARE the "prev" arrays afterwards. */
typedef struct {
    uint32_t struct_size;  /* sizeof(ml2048_step_args) */
    int32_t reward_kind;   /* ML2048_REWARD_* */
    int32_t rng_mode;      /* ML2048_RNG_* */
    int32_t action_dtype;  /* ML2048_ACT_* */
    int32_t action_mode;   /* ML2048_ACTIONS_* */
    int32_t onehot_dtype;  /* ML2048_ONEHOT_* */
    int64_t num_games;     /* games in this shard */
    int64_t slot_base;     /* global slot of game 0 of this shard */

    const void *board_in;  /* [num_games][16] u8 */
    void *board_out;       /* [num_games][16] u8, must not alias board_in */
    const void *valid_in;  /* [num_games][4] u8; read when action_mode is RANDOM_VALID or FROM_LOGITS or tr_valid_actions
                              is set; may be null otherwise (the move itself decides validity) */
    void *valid_out;       /* [num_games][4] u8 */
    const void *actions;   /* [num_games] of action_dtype, values 0..3 (others count as invalid moves) */
    void *actions_out;     /* [num_games] u8 or null: the action chosen in-kernel (RANDOM_VALID, FROM_LOGITS) */

    int32_t *step;         /* in place; += 1 on a valid move            (game_numba.py:719).  `step` and `score` are the halves of ONE
                              array of 8-byte {int32 step, float score} records, [num_games][2] words: step[2*g] and
                              score[2*g] belong to game g, score == (float *)step + 1, step 8-byte aligned (else ML2048_E_ALIGN).
                              One load and one store per game instead of two of each: a write-dominated kernel pays for
                              every separate read stream (profiles/README.md). */
    float *score;          /* in place; += normal reward on a valid move (:729-731); see `step` */
    float *reward;         /* in place; written on a valid move only: stays stale otherwise (:730, :737-738) */
    uint8_t *terminated;   /* in place; written on a valid move only (:735) */
    uint8_t *invalid;      /* always written (:736, :738) */
    uint8_t *merged;       /* [num_games][16] or null; written on a valid move only (:723) */

    void *onehot_out;      /* [num_games][16][16] of onehot_dtype, or null */

    /* replay mode (game_numba.py:733, 172-212) */
    const uint8_t *randperm_keys; /* [1024][16]: the reference's randperm table in inverse form,
                                     keys[row][cell] = 16*rank(cell)+cell (ml2048_pack_randperm_keys) */
    int64_t rand_seed;       /* _rand_step + rand_offset (:681); row = (rand_seed + global slot) mod 1024 */
    uint32_t two_mask;       /* bit c set <=> a tile spawned on CELL c is a 2 (else a 4).  Replay mode: (double)randfloat[c] <
                                two_prob (ml2048_two_mask).  Philox mode: the same per-cell, per-table-epoch law drawn from the
                                Philox stream on the host (ml2048_philox_epoch_draws) -- the reference ties the 2-vs-4 choice to
                                the cell for a whole table epoch (game_numba.py:207), and that is part of its episode statistics */

    /* philox mode */
    uint32_t two_threshold;  /* host-side only (Bernoulli threshold of ml2048_philox_epoch_draws); the kernels ignore it */
    uint64_t philox_seed;
    uint64_t philox_counter; /* caller increments once per step */

    ml2048_stats *stats;     /* [ML2048_STATS_REPLICAS] or null: finished-episode statistics */

    /* device-resident schedule (or null: use the scalar fields above) */
    const ml2048_sched_entry *sched;
    const int64_t *sched_cursor;   /* device scalar: index of the entry to use */
    int64_t *sched_cursor_next;    /* device scalar (not aliasing sched_cursor) or null: receives *sched_cursor + 1 */
    int64_t table_stride;          /* bytes between consecutive slots of the table ring (randperm_keys = slot 0) */

    /* per-episode record keyed by GAME ID (or null): when the game with id in [episode_id_base,
     * episode_id_base + episode_capacity) finishes, its final step count, score and max tile exponent are stored
     * at index id - episode_id_base.  This is what eval_perf.py gathers through ReplayRecorder for the games
     * with `buffer.id < rounds` (eval_perf.py:80-102, replay.py:110-232) without any per-step host loop. */
    int32_t *id;                   /* [num_games] game ids (the array ml2048_prepare maintains; written by the fused auto-reset) */
    int64_t episode_id_base;
    int64_t episode_capacity;
    int32_t *episode_steps;        /* [episode_capacity] */
    float *episode_score;          /* [episode_capacity] */
    uint8_t *episode_max_tile;     /* [episode_capacity]; 0 = not finished yet */

    /* ML2048_ACTIONS_FROM_LOGITS */
    const float *logits;           /* [num_games][4] f32, 16-byte aligned */
    float *log_prob_out;           /* [num_games] or null */

    /* Transition record (each pointer nullable): one row of the caller's (use, step, game) rollout buffers with
     * the REPLAY_SPEC dtypes (replay.py:10-20), written by the kernel instead of the seven host copies of
     * Trainer.on_stepped (run_train3.py:138-149).  Stale fields of invalid moves are copied stale, as there. */
    int8_t *tr_state;              /* [num_games][16] = prev_state */
    uint8_t *tr_valid_actions;     /* [num_games][4]  = prev_valid_actions (bool bytes) */
    int8_t *tr_action;             /* [num_games] */
    float *tr_reward;              /* [num_games] */
    int8_t *tr_next_state;         /* [num_games][16] */
    uint8_t *tr_next_valid_actions;/* [num_games][4] */
    int32_t *tr_step;              /* [num_games] */
    uint8_t *tr_terminated;        /* [num_games] (bool bytes) */

    /* Whole-episode capture keyed by GAME ID (or null), the device form of ReplayRecorder (replay.py:110-232): every
     * runner step of a game with id in [traj_id_base, traj_id_base + traj_capacity) appends the row
     * (prev_state, action, score) -- invalid moves included, like replay.py:178-189 -- and the step that finishes the game
     * appends a last row (final state, 0, score) (:191-201).  Rows beyond traj_max_rows are dropped (the count saturates). */
    int32_t *age;                  /* [num_games]: runner steps since the slot's game started; cleared by ml2048_prepare */
    int64_t traj_id_base;
    int64_t traj_capacity;
    int64_t traj_max_rows;
    int8_t *traj_state;            /* [traj_capacity][traj_max_rows][16] */
    int8_t *traj_action;           /* [traj_capacity][traj_max_rows] */
    float *traj_score;             /* [traj_capacity][traj_max_rows] */
    int32_t *traj_rows;            /* [traj_capacity]: rows written (= steps + 1 once the game is over) */

    /* Fused auto-reset (ML2048_ACTIONS_RANDOM_VALID only; null = off): the games that are over when the step starts are
     * first reset exactly as ml2048_prepare resets them -- record cleared, id = *reset_id_base + rank of the slot among
     * the finished slots (slot-ordered, game_numba.py:641-644), two tiles spawned with the PREPARE draws below, the
     * ascending index list -- and then played, in ONE launch.  board_in / valid_in receive the post-reset board and mask
     * of those games, so every array equals what ml2048_prepare followed by ml2048_step leaves behind.
     * reset_rank / reset_chunk_base / reset_id_base come from ml2048_autoreset_scan (run on the same stream right before);
     * `id` must be writable then.  A game counts as over when its mask is all zero, which is what `terminated` records
     * (game_numba.py:734-735): the two must agree, as they do for every state the library itself produces.
     * The launch is a PROGRAMMATIC DEPENDENT of the kernel before it on `stream` (the scan releases its dependents early):
     * the step reads its boards while the scan still runs and waits before it touches what the scan reads or writes, so
     * board_in / valid_in / step must be complete before the scan is enqueued -- true for any in-order use of one stream. */
    const int32_t *reset_rank;       /* [ceil(num_games / 32)]: finished games in lower groups of the same 1024-group chunk */
    const int32_t *reset_chunk_base; /* [ceil(groups / 1024)]: finished games in lower chunks */
    const int64_t *reset_id_base;    /* device scalar: id of the first game this step resets */
    int64_t *reset_indices;          /* [num_games] out or null: ascending slots reset by this step (np.flatnonzero, :629) */
    const uint8_t *randperm;         /* replay mode: the permutation table itself (reset takes the first two entries, :648-655) */
    int64_t rand_base;               /* prepare's _rand_step + rand_offset (:651); sched entries carry their own */
    uint64_t prepare_philox_counter; /* Philox mode: the counter ml2048_prepare would have used */
} ml2048_step_args;

/* Arguments of the auto-reset.  Replaces the host loop of VecGame.prepare (game_numba.py:629-658):
 * every terminated slot, in ascending slot order, is cleared, gets the next id, two spawned tiles and
 * a mask.  Works in place on the CURRENT boards/masks. */
typedef struct {
    uint32_t struct_size;
    int32_t rng_mode;
    int32_t onehot_dtype;
    int32_t reserved0;
    int64_t num_games;
    int64_t slot_base;

    void *board;           /* [num_games][16] */
    void *valid;           /* [num_games][4] */
    int32_t *id;           /* [num_games] (game_numba.py:641-644) */
    int32_t *step;         /* {step, score} records, as in ml2048_step_args */
    float *score;
    float *reward;
    uint8_t *terminated;   /* [ceil16(num_games)] : padded to a multiple of 16 bytes, padding zero */
    uint8_t *invalid;
    uint8_t *merged;       /* or null */
    void *onehot;          /* or null: rows of reset games are rewritten */

    const uint8_t *randperm;
    int64_t rand_base;     /* _rand_step + rand_offset (:651) */
    uint32_t two_mask;
    uint32_t two_threshold;
    uint64_t philox_seed;
    uint64_t philox_counter;

    int64_t *game_count;   /* device scalar: next id; advanced by the number of resets (:641-642).
                              With id_offset != null (multi-GPU global ids) it is NOT advanced here. */
    const int64_t *id_offset; /* or null: device scalar added to ids of this shard (exclusive scan over ranks) */
    int64_t *reset_count;  /* device scalar out: number of slots reset by this call */
    int64_t *reset_indices;/* [num_games] out, ascending slots (np.flatnonzero, :629), or null */
    int32_t *scratch;      /* [ml2048_prepare_scratch_ints(num_games)] */

    /* device-resident schedule (or null), see ml2048_sched_entry; prepare never advances the cursor */
    const ml2048_sched_entry *sched;
    const int64_t *sched_cursor;
    int64_t table_stride;  /* bytes between consecutive slots of the table ring (randperm = slot 0) */
    int32_t *age;          /* [num_games] or null: cleared for every reset slot (see ml2048_step_args.age) */
} ml2048_prepare_args;

/* ---- entry points ---------------------------------------------------------------------------- */

ML2048_API int ml2048_abi_version(void);

/* ints of scratch ml2048_prepare needs for num_games */
ML2048_API int64_t ml2048_prepare_scratch_ints(int64_t num_games);

/* _vec_step + VecGame.step body: game_numba.py:660-738 */
ML2048_API int ml2048_step(const ml2048_step_args *args, void *stream);

/* VecGame.prepare reset loop: game_numba.py:629-658.  ml2048_prepare runs it in one launch: a single-block kernel up to
 * 8192 games, above that one cooperative launch (a grid of co-resident blocks with one grid-wide barrier between counting
 * and resetting; needs cudaDevAttrCooperativeLaunch, else -- or with ML2048_PREPARE=split in the environment, or for
 * shards too large for it -- count + apply below).  Semantically ml2048_prepare = count + apply.  The two halves
 * are exported so a multi-GPU caller can exchange per-rank reset counts between them (all_gather of
 * *reset_count -> id_offset) and keep ids globally slot-ordered like the single-process reference:
 *   count: np.flatnonzero(terminated) bookkeeping (:629) -> *reset_count, slot-ordered offsets in scratch
 *   apply: the per-slot reset body (:634-656) */
ML2048_API int ml2048_prepare(const ml2048_prepare_args *args, void *stream);
ML2048_API int ml2048_prepare_count(const ml2048_prepare_args *args, void *stream);
ML2048_API int ml2048_prepare_apply(const ml2048_prepare_args *args, void *stream);

/* VecGame.reset data part (game_numba.py:613-617): zero all per-game state, mark every game terminated */
ML2048_API int ml2048_reset_state(void *board_a, void *board_b, void *valid_a, void *valid_b, int32_t *id, int32_t *step, float *score,
                       float *reward, uint8_t *terminated, uint8_t *invalid, uint8_t *merged, int64_t num_games, void *stream);

/* CNNEncoder.forward input encoding as a stand-alone op: policy/_network.py:86-95 */
ML2048_API int ml2048_encode_onehot(const void *board, void *out, int32_t onehot_dtype, int64_t num_games, void *stream);

/* _compute_valid_actions over a batch: game_numba.py:259-289 */
ML2048_API int ml2048_valid_actions(const void *board, void *valid_out, int64_t num_games, void *stream);

/* the four moves of every board without spawning (game_numba.py:93-134, :408-504 at :728): after [n][4][16],
 * reward [n][4] f32 (reward_kind; 0 for a direction that does not change the board), valid [n][4] u8,
 * merged [n][4][16] or null */
ML2048_API int ml2048_afterstates(const void *board, void *after_out, float *reward_out, uint8_t *valid_out,
                                  uint8_t *merged_out, int32_t reward_kind, int64_t num_games, void *stream);

/* n-tuple network (no reference counterpart): K = num_tuples (1..16) tuples of len[t] (1..6) distinct cells (cell = row*4+col,
 * 0..15) given as HOST arrays cells [K][6] (entries past len[t] ignored) and len [K].  weights: num_weights = sum_t 16^len[t]
 * float32 entries, tuple t's table from offset sum_{u<t} 16^len[u].  V(s) = sum over t = 0..K-1 (outer), g = 0..7 (inner) of
 * weights[offset_t + idx_t,g(s)] as float32 adds from 0.0f, where image g maps cell (r,c) to (r,c) (r,3-c) (3-r,c) (3-r,3-c)
 * (c,r) (c,3-r) (3-c,r) (3-c,3-r) and idx = sum_j min(cell_j, 15) << 4j: any byte gives an in-bounds index, exponents >= 16
 * share the entries of 15.  value [n] f32. */
ML2048_API int ml2048_ntuple_value(const void *board, const float *weights, int64_t num_weights, const uint8_t *cells, const uint8_t *len,
                                   int32_t num_tuples, float *value_out, int64_t num_games, void *stream);

/* greedy afterstate move: q_a = reward_a + V(afterstate_a) over the directions that change the board (reward_a and
 * afterstate_a as ml2048_afterstates gives them); the largest q wins, NaN ranks as -inf, ties go to the smallest direction.
 * Writes the action (u8 or i64: exactly one non-null), the chosen afterstate [n][16], its reward and its value.  A board with
 * no valid direction: action 0, afterstate = board, reward 0, value 0. */
ML2048_API int ml2048_ntuple_greedy(const void *board, const float *weights, int64_t num_weights, const uint8_t *cells, const uint8_t *len,
                                    int32_t num_tuples, int32_t reward_kind, uint8_t *action_u8, int64_t *action_i64, void *after_out,
                                    float *reward_out, float *value_out, int64_t num_games, void *stream);

/* one synchronous TD(0) batch: delta[i] = alpha * (target[i] - V(after[i])) with the weights as they were before the call
 * (0 where mask[i] == 0; mask may be null = all games), then weights[entry] += delta[i] for every masked-in game and each of
 * its 8 * K entries.  The adds are float atomics: their order within one entry is unspecified, so the weights are
 * reproducible up to the fp32 rounding of that order (delta is deterministic). */
ML2048_API int ml2048_ntuple_td_update(const void *after, const float *target, const uint8_t *mask, float alpha, float *weights,
                                       int64_t num_weights, const uint8_t *cells, const uint8_t *len, int32_t num_tuples,
                                       float *delta_out, int64_t num_games, void *stream);

/* _update_count (runner.py:120-136): hist[max exponent] += 1 for every game with terminated != 0;
 * with terminated == null: VecGame.summary's histogram over all live boards (game_numba.py:593-596).
 * hist20 is [20] unsigned long long, accumulated (not cleared). */
ML2048_API int ml2048_max_tile_hist(const void *board, const uint8_t *terminated, int64_t num_games, unsigned long long *hist20, void *stream);

/* The result flags of a step for a HOST caller, one byte per game: bits 0..3 = valid_actions (left, right, up, down;
 * game_numba.py:540), bit 4 = terminated (:546), bit 5 = invalid (:547).  `terminated` / `invalid` may be null (bits 0).
 * VecGame.step(host actions, fetch=...) ships this byte over PCIe instead of the six bytes of the three arrays and rebuilds
 * them with ml2048_unpack_flags (host code; `threads` worker threads, any of the three outputs may be null). */
ML2048_API int ml2048_pack_flags(const void *valid, const uint8_t *terminated, const uint8_t *invalid, uint8_t *packed, int64_t num_games,
                                 void *stream);
ML2048_API void ml2048_unpack_flags(const uint8_t *host_packed, int64_t num_games, uint8_t *host_valid4, uint8_t *host_terminated,
                                    uint8_t *host_invalid, int32_t threads);
/* ... for a result that arrives in slices [slice_lo[k], slice_hi[k]): events[k] is the cudaEvent_t recorded after slice k's packed
 * bytes were copied (null = already there).  The worker threads wait for the events themselves; returns 0 or a cudaError_t. */
ML2048_API int ml2048_unpack_flags_sliced(const uint8_t *host_packed, int32_t num_slices, const int64_t *slice_lo, const int64_t *slice_hi,
                                          void *const *events, uint8_t *host_valid4, uint8_t *host_terminated, uint8_t *host_invalid,
                                          int32_t threads);

/* uniform-over-valid action sampler (policy/random.py:17-27) as a stand-alone op: draws the policy-stream word of
 * (philox_seed, slot_base + i, philox_counter), i.e. the action ML2048_ACTIONS_RANDOM_VALID picks inside ml2048_step */
ML2048_API int ml2048_sample_random_valid(const void *valid, uint8_t *actions_out, int64_t num_games, int64_t slot_base,
                               uint64_t philox_seed, uint64_t philox_counter, void *stream);

/* _sample_action (policy/actor_critic.py:56-76) as a stand-alone op: masked categorical sample + log-probability.
 * valid: [num_games][4] bool/u8; actions_u8 / actions_i64: either may be null; log_prob: [num_games] or null */
ML2048_API int ml2048_sample_masked_categorical(const float *logits, const void *valid, uint8_t *actions_u8, int64_t *actions_i64,
                                                float *log_prob, int64_t num_games, int64_t slot_base, uint64_t philox_seed,
                                                uint64_t philox_counter, void *stream);

/* compute_gae's recurrence (gae.py:50, :65-68) over (use, step, game) f32 tensors, one thread per (use, game):
 *   delta = gamma * v1 * (1 - terminated) + reward - v0;  tmp = delta[t] + (tmp * gamma*lambda) * (1 - terminated[t]), t descending
 * rounded exactly like the reference's torch fp32 ops (no fused multiply-add). */
ML2048_API int ml2048_gae(const float *v0, const float *v1, const float *reward, const uint8_t *terminated, float *adv,
                          int64_t use_count, int64_t step_count, int64_t game_count, float gamma, float coef, void *stream);

/* ---- fused auto-reset: the scan that ranks the finished games -----------------------------------------------------
 * One launch over the `terminated` flags ([ceil16(num_games)], padded like ml2048_prepare's): per group of 32 slots the
 * number of finished games, reset_rank[w] = exclusive prefix of those counts inside the group's chunk of 1024 groups,
 * reset_chunk_base[c] = exclusive prefix over chunks, *reset_id_base = *game_count (+ *id_offset), *game_count += total
 * (unless id_offset is set: sharded ids, the caller adds the global total), *reset_count = total.
 * scratch: [ml2048_autoreset_scratch_ints(num_games)] int32, zero before the first call. */
ML2048_API int ml2048_autoreset_scan(const uint8_t *terminated, int32_t *reset_rank, int32_t *reset_chunk_base, int64_t num_games,
                                     int64_t *game_count, const int64_t *id_offset, int64_t *reset_id_base, int64_t *reset_count,
                                     int32_t *scratch, void *stream);
ML2048_API int64_t ml2048_autoreset_scratch_ints(int64_t num_games);

/* host helpers (no GPU work) */
ML2048_API uint32_t ml2048_two_mask(const float *host_randfloat16, double two_prob);   /* game_numba.py:207 (f32 -> f64 compare) */
ML2048_API uint32_t ml2048_two_threshold(double two_prob);
/* cudaMemcpyAsync (kind inferred from the pointers; pinned host memory for a truly asynchronous copy) and cudaStreamSynchronize
 * for host callers without a CUDA binding of their own: 0 or a cudaError_t. */
ML2048_API int ml2048_copy_async(void *dst, const void *src, int64_t bytes, void *stream);
ML2048_API int ml2048_stream_wait(void *stream);

/* ---- compressible device memory (the only entry points that allocate) ------------------------------------------------
 * A mostly-zero output written in full every step (the one-hot observation) costs fewer HBM bytes in memory the L2 may
 * store compressed.  ml2048_alloc_compressible reserves a virtual range of `bytes` rounded up to the allocation granularity
 * on `device`, backs it with cuMemCreate(allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC) allocations, maps
 * them and grants read/write access to that device only.  If one allocation is not granted compression, the range is
 * built again from 8, then 64 equal allocations, each checked on its own; `granted` counts the bytes the driver granted
 * compression (read back, possibly 0).  The contents are undefined.  Returns 0, ML2048_E_NULL / ML2048_E_SIZE,
 * ML2048_E_UNSUPPORTED (no driver, no such device, or no generic compression on it; *out is then all zero), or a
 * positive CUresult of the driver call that failed (nothing stays allocated).
 * ml2048_free_compressible synchronises the device (work queued on any stream may still write the range), unmaps,
 * releases and unreserves it, and zeroes *c; a zeroed *c is a no-op. */
#define ML2048_COMPRESSIBLE_MAX_CHUNKS 64
typedef struct {
    uint64_t ptr;      /* device address of the range, 0 when nothing is mapped */
    uint64_t size;     /* mapped bytes: the request rounded up to the granularity (per allocation) */
    uint64_t granted;  /* bytes of the range whose allocation the driver granted generic compression */
    int32_t device;
    int32_t chunks;    /* equal allocations behind the range */
    uint64_t handles[ML2048_COMPRESSIBLE_MAX_CHUNKS];
} ml2048_compressible;

ML2048_API int ml2048_alloc_compressible(int32_t device, int64_t bytes, ml2048_compressible *out);
ML2048_API int ml2048_free_compressible(ml2048_compressible *c);

/* Philox mode, the host half of one prepare(): the reference refreshes its spawn tables when `random() >= 0.9`
 * (game_numba.py:622-624) and the 2-vs-4 choice then stays tied to the CELL until the next refresh (:207).  The same two
 * draws from the counter-based stream, keyed by (seed, prepare counter) so that every shard computes identical values:
 * *coin_u32 = a uniform 32-bit word (refresh iff >= 0.9 * 2^32), *mask16 = sixteen Bernoulli(two_prob) bits, bit c for cell c. */
ML2048_API void ml2048_philox_epoch_draws(uint64_t philox_seed, uint64_t prepare_counter, double two_prob, uint32_t *coin_u32,
                                          uint32_t *mask16);
/* Philox4x32-10 and Philox2x32-10 on the host (known-answer tests; the kernels use the same rounds) */
ML2048_API void ml2048_philox4x32_10(const uint32_t counter[4], const uint32_t key[2], uint32_t out[4]);
ML2048_API void ml2048_philox2x32_10(const uint32_t counter[2], uint32_t key, uint32_t out[2]);
/* randperm (u8 [rows][16], each row a permutation of 0..15, game_numba.py:578,610) -> inverse-form keys used by
 * ml2048_step: the kernel picks the empty cell of smallest rank = the first empty cell of the table walk (:198-204) */
ML2048_API int ml2048_pack_randperm_keys(const uint8_t *host_randperm, uint8_t *host_keys, int64_t rows);

/* ---- host random schedule (no GPU work) -------------------------------------------------------------------------
 * State of numpy's PCG64 bit generator (`Generator.bit_generator.state`), and the four draws the reference makes from
 * it per prepare()/step(): random() (game_numba.py:622), integers(0, 1024) (:626, :670), permuted(axis=1) and
 * random(float32) (:590-591).  Same bit stream as numpy; verified against the installed numpy at start-up. */
typedef struct {
    uint64_t state_hi, state_lo; /* 128-bit LCG state */
    uint64_t inc_hi, inc_lo;     /* 128-bit increment */
    int32_t has_uint32;          /* a buffered 32-bit half is pending */
    uint32_t uinteger;           /* the buffered half */
} ml2048_pcg64;

ML2048_API double ml2048_pcg64_random(ml2048_pcg64 *g);
ML2048_API int64_t ml2048_pcg64_integers(ml2048_pcg64 *g, int64_t high);
ML2048_API void ml2048_pcg64_random_f32(ml2048_pcg64 *g, float *out, int64_t n);
ML2048_API void ml2048_pcg64_permuted_rows_u8(ml2048_pcg64 *g, uint8_t *x, int64_t rows, int64_t cols);

#ifdef __cplusplus
}
#endif
#endif /* ML2048_B200_H */
