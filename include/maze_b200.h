/*
 * maze_b200.h -- C ABI of the B200-native batched maze environment (libmaze_b200.so).
 *
 * The reference (Fabri000/Maze-Solving-Agent-Gymnasium) is pure Python and has no FFI; this
 * header therefore *defines* the boundary a maintainer would bind (ctypes stub in
 * INTEGRATION.md).  Each entry point names the reference code it replaces.
 *
 * Conventions
 *   - every data pointer is a DEVICE pointer owned by the caller (PyTorch tensors' data_ptr());
 *     the library allocates nothing across the boundary except the opaque maze_ctx, which owns
 *     two small device-side reward look-up tables and a scratch counter block
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*); the caller
 *     serialises calls on one ctx
 *   - return value: 0 ok, <0 argument error (MAZE_E_*), >0 a cudaError_t; never throws, never
 *     exits; maze_last_error(ctx) gives the text of the last failure
 *   - sm_100a only: there is no CPU fallback and no other architecture in the fatbin
 *
 * Block-grid vocabulary (reference lib/maze_generation.py:16-19,33): a maze is an H x W grid of
 * blocks, 0 wall / 1 floor / 2 goal, H = W = 2N+1 for N x N logical cells.  A maze lives in a
 * "slot" of `slot` bytes (>= H*W, row-major with pitch W).
 */
#ifndef MAZE_B200_H
#define MAZE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MAZE_ABI_VERSION 14

/* argument errors */
#define MAZE_E_NULL   (-1) /* required pointer is NULL                        */
#define MAZE_E_RANGE  (-2) /* size / shape / id out of range                  */
#define MAZE_E_SHAPE  (-3) /* even or too small / too large block shape       */
#define MAZE_E_ALGO   (-4) /* unknown generator id                            */
#define MAZE_E_ALIGN  (-5) /* pointer not aligned as documented               */

/* limits */
#define MAZE_MAX_DIM      255  /* H, W <= 255 (positions are stored in one byte each)        */
#define MAZE_GEN_MAX_DIM  131  /* generator / fields kernels stage one maze in shared memory */
#define MAZE_GEN_MAX_CELLS 64  /* generators hold one 64-bit word per lattice row: bordered shapes up to
                                  129 x 129 (64 x 64 cells), toroidal shapes up to 127 x 127 (generated at
                                  shape + 2 = 129); a slot asking for more is left untouched and gets
                                  MAZE_META_SOL_LEN = -1                                              */
#define MAZE_WINDOW       15   /* simple_maze_env.py:130 WINDOW_DIM                          */

/* generator ids: lib/maze_generation.py:24-30 */
#define MAZE_ALGO_RPRIM     0  /* "r-prim"    random_prim_visit   :59-99   */
#define MAZE_ALGO_DFS       1  /* "dfs"       deept_first_visit   :101-128 */
#define MAZE_ALGO_PRIMKILL  2  /* "prim&kill" prim_and_kill_visit :130-185 */

/* per-maze metadata record: int32[MAZE_META_WORDS], 32 bytes, 32-byte aligned */
#define MAZE_META_WORDS 8
#define MAZE_META_H          0
#define MAZE_META_W          1
#define MAZE_META_START      2  /* start_r | start_c << 16                                   */
#define MAZE_META_GOAL       3  /* goal_r  | goal_c  << 16                                   */
#define MAZE_META_MAX_STEPS  4  /* simple_maze_env.py:52-58 (written by maze_fields)         */
#define MAZE_META_FLAGS      5  /* bit0 toroidal; bits 8-15 generator id                     */
#define MAZE_META_SOL_LEN    6  /* len(path(start->goal)) in blocks (written by maze_fields) */
#define MAZE_META_SPARE      7
#define MAZE_FLAG_TOROIDAL 1

/* step-table byte (one per block, written by maze_fields): everything the step needs */
#define MAZE_TAB_OPEN      0x01 /* block is not a wall                                       */
#define MAZE_TAB_CODE_SHIFT 1   /* bits 1-3: best-next action 0..3, 4 = none (best dir 0,0)  */
#define MAZE_TAB_D4_SHIFT   4   /* bits 4-5: D_goal mod 4 (reward needs D[prev]-D[cur] only) */

/* per-env packed state: one uint64, little-endian bytes
 *   0 row | 1 col | 2 consecutive-invalid (saturating) | 3 flags | 4-5 steps_taken (u16)
 *   6 visit epoch (1..255) | 7 step-table byte of the current block                         */
#define MAZE_ST_NEEDS_RESET 0x01 /* episode ended on the previous step (autoreset pending)   */
#define MAZE_ST_WON         0x02 /* ... and it ended by reaching the goal                    */
#define MAZE_ST_MOVE_SHIFT  2    /* bits 2-3: last successful move                           */
#define MAZE_ST_NMOVES_SHIFT 4   /* bits 4-5: successful moves this episode, saturating at 2 */

/* maze_step mode bits */
#define MAZE_STEP_AUTORESET   0x01 /* gymnasium next-step autoreset                          */
#define MAZE_STEP_WIN_NEXT    0x02 /* on autoreset after a win move to maze (m + stride) % M */
#define MAZE_STEP_WIN_QUEUE   0x04 /* on a win append the env's maze slot to the regen queue */
#define MAZE_STEP_PACKED      0x08 /* also write one packed uint32 record per env to batch.packed   */
#define MAZE_STEP_NO_WIDE     0x10 /* with MAZE_STEP_PACKED: skip agent / best_dir / reward / terminated /
                                      truncated (the record holds the same information in 4 bytes
                                      instead of 26; `target` is still written when it changes)  */

/* Packed step record (MAZE_STEP_PACKED): everything base_maze_env.py:116-122,210 returns for one env except
 * `target` (which changes only with the maze), bit-exactly recoverable on the host:
 *   bits 0-7 row | 8-15 col | 16-18 best-next code (0..3 = action towards the best neighbour, 4 = none;
 *   best dir = agent - wrapped neighbour) | 19 terminated | 20 truncated | 21-22 reward kind | 23-30 reward index
 * reward = maze_reward_lut(kind)[index] for kind 0 (revisit), 1 (invalid move), 2 (shaping: index 0 farther,
 * 1 same, 2 closer); kind 3: index 0 -> 0.0 (reset step), 1 -> 1.0 (goal), 2 -> -1.0 (truncation).
 * maze_step_decode_host turns records back into the wide arrays. */
#define MAZE_REC_CODE_SHIFT   16
#define MAZE_REC_TERM_SHIFT   19
#define MAZE_REC_TRUNC_SHIFT  20
#define MAZE_REC_KIND_SHIFT   21
#define MAZE_REC_INDEX_SHIFT  23
#define MAZE_REC_KIND_REVISIT 0
#define MAZE_REC_KIND_INVALID 1
#define MAZE_REC_KIND_SHAPING 2
#define MAZE_REC_KIND_CONST   3
#define MAZE_REC_CONST_ZERO      0
#define MAZE_REC_CONST_ONE       1
#define MAZE_REC_CONST_MINUS_ONE 2
#define MAZE_REC_REWARD(kind, index) (((uint32_t)(kind) << MAZE_REC_KIND_SHIFT) | ((uint32_t)(index) << MAZE_REC_INDEX_SHIFT))

typedef struct maze_ctx maze_ctx;

/* Batch of environments, structure of arrays.  All device pointers. */
typedef struct maze_env_batch {
    int32_t   num_envs;    /* B                                                              */
    int32_t   num_mazes;   /* M maze slots                                                   */
    int32_t   slot;        /* bytes per maze slot in `table`; cells per env in `visits`      */
    int32_t   pool_stride; /* MAZE_STEP_WIN_NEXT increment                                   */
    const int32_t* meta;   /* [M, 8]                                                         */
    const uint8_t* table;  /* [M, slot] step-table bytes                                     */
    int32_t*  env_maze;    /* [B] maze slot of each env                                      */
    uint64_t* state;       /* [B] packed state                                               */
    uint16_t* visits;      /* epoch << 8 | saturating visit count of (block idx, env e) at
                              idx * visit_cell_stride + e * visit_env_stride: cell-major
                              [slot, B] (strides B, 1) for the -v0 step; env-major [B, slot]
                              (strides 1, slot), best with visit_tiled = 1, when the 15x15
                              window is read every step or several steps fuse into a launch   */
    /* outputs of step / reset (reference obs dict of base_maze_env.py:116-122) */
    int32_t*  agent;       /* [B, 2] int32                                                   */
    int32_t*  target;      /* [B, 2]                                                         */
    int32_t*  best_dir;    /* [B, 2]  agent - best_next                                      */
    double*   reward;      /* [B]                                                            */
    uint8_t*  terminated;  /* [B]                                                            */
    uint8_t*  truncated;   /* [B]                                                            */
    /* optional episode statistics (may be NULL) */
    double*   ep_return;   /* [B] running return of the current episode                      */
    int64_t*  stats;       /* [4] episodes, wins, truncations, steps (atomic counters)       */
    double*   stats_return;/* [1] sum of finished episodes' returns                          */
    /* optional regeneration queue (MAZE_STEP_WIN_QUEUE) */
    int32_t*  queue;       /* [B] maze slots whose env won                                   */
    int32_t*  queue_count; /* [1]                                                            */
    int64_t   visit_cell_stride;
    int64_t   visit_env_stride;
    int32_t   visit_tiled; /* 0: block idx = r * W + c.  1: 4 x 4 block tiles, one 32-byte sector each:
                              idx = ((r >> 2) * ((W + 3) >> 2) + (c >> 2)) * 16 + (r & 3) * 4 + (c & 3),
                              so an agent walking a corridor keeps hitting the same sector      */
    int32_t   visit_slot;  /* visit entries per env (>= slot; tiled: >= 16 * ceil(H/4) * ceil(W/4)) */
    int32_t*  target_dirty;/* optional [1] (may be NULL): set to 1 by every launch that writes `target`.  An env's
                              target only changes when its maze does -- maze_reset, or the restart after a win --
                              so maze_step rewrites `target` only then, and a host mirror of the outputs can skip
                              the device-to-host copy of `target` on all other steps                       */
    uint32_t* packed;      /* optional [B] (may be NULL): packed step records, written under MAZE_STEP_PACKED        */
    uint32_t* visit_bits;  /* optional (may be NULL): one bit per block, "visited in the current episode", bit (r, c) of
                              env e = bit c & 31 of word e * visit_bits_stride + r * visit_bits_pitch + (c >> 5).  Kept
                              beside the counters by every stepping kernel (set on a legal move, cleared when an episode
                              starts); the -v1 window and the replay encode read their non_visited channel from it: a
                              15 x 15 window is 15 consecutive bitmap rows (180 contiguous bytes at 81 x 81) instead of
                              up to 25 scattered 32-byte sectors of counters                                          */
    int32_t   visit_bits_pitch;   /* words per bitmap row: ceil(max W / 32)                                          */
    int32_t   visit_bits_stride;  /* words per env: max H * pitch rounded up to a multiple of 4                       */
    int32_t   flags;       /* MAZE_BATCH_BORDERED: the caller promises that no maze of `meta` is toroidal.  With visit_bits,
                              maze_window and maze_dqn_push then run their bordered kernels (two envs per half-warp in
                              flight, no generic gather compiled in); without the flag nothing is assumed              */
    int32_t   reserved;
} maze_env_batch;
#define MAZE_BATCH_BORDERED 1

/* sizeof of the ABI structs as this library was compiled (a binding checks its own layout against it):
 * which = 0 maze_env_batch, 1 maze_q_agent, 2 maze_replay, 3 maze_step_trace, 4 maze_dqn_net; -1 for anything else. */
int  maze_sizeof(int which);

int  maze_abi_version(void);
int  maze_ctx_create(maze_ctx** out, int device);
void maze_ctx_destroy(maze_ctx* ctx);
const char* maze_last_error(maze_ctx* ctx);

/* Host-side copy of the float64 reward look-up tables the kernels use.
 * kind 0: revisit penalty  0.0 - (1 - exp(-0.2  * count))   base_maze_env.py:194
 * kind 1: invalid penalty  0.0 - (1 - exp(-0.15 * k))       base_maze_env.py:200
 * kind 2: shaping reward   delta * 0.5 - 0.05, delta = -1,0,+1 in out[0..2]  :192
 * `out` is a HOST pointer to 256 doubles. */
int maze_reward_lut(maze_ctx* ctx, int kind, double* out);

/* Per-maze fields: BFS from the goal over the block graph, then the step table and the step
 * budget.  Replaces the per-step A* of base_maze_env.py:189-190,224-262 (lib/a_star_algos/*)
 * and set_max_steps (simple_maze_env.py:52-58, metrics_calculator.py:16,22-26).
 *   grids [M, slot] uint8 block grids (0/1/2); meta [M, 8] with H, W, START, GOAL, FLAGS set;
 *   writes table [M, slot] and meta MAX_STEPS / SOL_LEN.
 *   ids: optional [n] list of maze slots to process (NULL = slots 0..n-1). */
int maze_fields(maze_ctx* ctx, const uint8_t* grids, int32_t* meta, uint8_t* table,
                const int32_t* ids, int n, int slot, void* stream);

/* One transition for every env: BaseMazeEnv.step (base_maze_env.py:163-210) with the move rule
 * of lib/maze_view.py:167-180 / :184-197, plus the observation of :116-122.
 * actions [B] uint8 in 0..3. */
int maze_step(maze_ctx* ctx, const maze_env_batch* b, const uint8_t* actions, uint32_t mode, void* stream);

/* HOST-side decode of n packed step records (plain C loop, no GPU): fills the wide arrays maze_step writes --
 * agent [n, 2] int32, best_dir [n, 2] int32, reward [n] float64, terminated / truncated [n] uint8 (any may be NULL).
 * shape [n, 2] int32 holds each env's (H, W) and toroidal [n] uint8 its topology; both may be NULL for bordered
 * (euclidean) mazes, where best dir never wraps.  Bit-identical to the wide outputs of the same step. */
int maze_step_decode_host(const uint32_t* records, int64_t n, const int32_t* shape, const uint8_t* toroidal, int32_t* agent,
                          int32_t* best_dir, double* reward, uint8_t* terminated, uint8_t* truncated);

/* Measurement aid, not part of the env path (tools/perf_scatter_rmw.py, DESIGN.md section 4.1): one launch that
 * streams maze_step's coalesced words for every env of `b` (streams != 0) and lets rmw_per_1024 of every 1024 envs do
 * one 2-byte read-modify-write in arr (uint16 [n_elems]) -- pattern 0: uniform random element; 1: cell-major
 * cell * B + env with a random cell per env; 2: as 1 with one cell per warp.  Pattern 1 sends retouch_per_1024 of
 * every 1024 envs that did an RMW in launch - 1 back to that launch's cell.  order 1 runs the CTAs in reverse on odd
 * launches, as maze_step does; hints 0..3 pick the L2 policies (csrc/maze_bench.cu).  Overwrites b's outputs and state. */
int maze_bench_scatter_rmw(maze_ctx* ctx, const maze_env_batch* b, const uint8_t* actions, uint16_t* arr, int64_t n_elems, int pattern,
                           int rmw_per_1024, uint32_t launch, int streams, int order, int retouch_per_1024, int hints, void* stream);

/* k_steps consecutive transitions per env in one call, for action sequences known in advance
 * (scripted / random exploration, replaying tapes): exactly the result of k_steps maze_step calls
 * with actions[k] = actions + k * B, but with the env state in registers for the whole burst, so that
 * the visit counters a walking agent keeps coming back to are served by L1 / L2 (best with the tiled
 * visit layout: 2.1x the throughput of per-step launches at K = 64 with every per-step output written).
 *   actions   [k_steps, B] uint8
 *   trace     optional per-step outputs (NULL = only the last step's, in the batch arrays):
 *             agent / best_dir [k_steps, B, 2] int32, reward [k_steps, B] float64,
 *             terminated / truncated [k_steps, B] uint8 (any member may be NULL)
 *   chunk_envs  0 = one launch over all envs; > 0 = process the envs in chunks of this size
 * MAZE_STEP_WIN_QUEUE is not available here (regeneration needs a launch between steps). */
typedef struct maze_step_trace {
    int32_t* agent;
    int32_t* best_dir;
    double*  reward;
    uint8_t* terminated;
    uint8_t* truncated;
} maze_step_trace;
int maze_step_many(maze_ctx* ctx, const maze_env_batch* b, const uint8_t* actions, int k_steps, uint32_t mode,
                   const maze_step_trace* trace, int chunk_envs, void* stream);

/* BaseMazeEnv.reset (base_maze_env.py:136-161) for envs with mask[e] != 0 (mask NULL = all).
 * Writes agent/target/best_dir; reward 0, flags 0. */
int maze_reset(maze_ctx* ctx, const maze_env_batch* b, const uint8_t* mask, void* stream);

/* Batched generation on the device: gen_maze (lib/maze_generation.py:6-35) and, for slots whose
 * meta FLAGS has MAZE_FLAG_TOROIDAL, gen_maze_no_border (:37-56; generated at shape+2, goal
 * chosen on the bordered maze, outer ring stripped).  Per slot the caller sets meta H, W (final
 * block shape, odd) and FLAGS (toroidal bit, generator id in bits 8-15); the kernel writes the
 * block grid (0/1/2; `grids` may be NULL), START, GOAL, SOL_LEN, MAX_STEPS, the step table, and
 * increments SPARE (generation count of the slot, part of the RNG key).
 *   ids       optional [n] slot list (NULL = slots 0..n-1)
 *   count_dev optional device int32: number of valid entries of ids (then n = capacity); lets a
 *             regeneration queue filled by maze_step be drained without a host round trip
 *   max_h/w   largest final shape among the slots (sizes shared memory)
 *   candidates 1 = the raw generator; k > 1 = BaseMazeEnv.generate_maze (base_maze_env.py:78-97,
 *             toroidal_maze_env.py:40-54): draw k mazes, keep the one with the lowest McClendon
 *             difficulty (strict <, the first wins ties); difficulty is taken on the bordered maze
 *   difficulty optional [n] out: difficulty of the maze kept for ids[k] (NULL with candidates 1
 *             skips the evaluation)
 *   RNG       Philox4x32-10, key = seed, counter = (slot_id_base + slot, generation count,
 *             candidate): results do not depend on how slots are sharded over GPUs. *
 * Bulk best-of-k (candidates > 1, count_dev NULL, n >= 16) runs as two kernels and keeps the candidates'
 * wall planes in a ctx-owned scratch buffer (<= 8 192 x candidates x 1 KB, allocated on first use, freed by
 * maze_ctx_destroy); the result is identical to the single-kernel path used for regeneration queues. */
int maze_generate(maze_ctx* ctx, uint8_t* grids, int32_t* meta, uint8_t* table, const int32_t* ids,
                  const int32_t* count_dev, int n, int slot, int max_h, int max_w,
                  uint64_t seed, int64_t slot_id_base, int candidates, double* difficulty, void* stream);

/* Curriculum step for the slots whose env just won (drain of the maze_step regeneration queue, run
 * before maze_generate):  wins[slot] += 1; variable-size envs grow the slot's shape by `grow` blocks
 * per axis while it stays <= (max_h, max_w) (simple_variable_maze_env.py:93-112: +(4, 4) per win);
 * the generator id becomes algo_a once wins >= wins_a and algo_b once wins >= wins_b
 * (off_policy_trainer.py:302-310: prim&kill after 5 wins, dfs after 10; pass -1 to keep the id).
 *   ids / count_dev / n as for maze_generate; wins [M] int32. */
int maze_curriculum(maze_ctx* ctx, int32_t* meta, int32_t* wins, const int32_t* ids, const int32_t* count_dev,
                    int n, int grow, int max_h, int max_w, int wins_a, int algo_a, int wins_b, int algo_b, void* stream);

/* Regeneration ahead of time (the update_maze() of off_policy_trainer.py:60-71 / :190-214 without its latency).  A
 * shadow ring (shadow_grids / shadow_table [depth, M, slot], shadow_meta [depth, M, 8]: ring entry j of slot m at index
 * j * M + m, same layouts as the live pool) holds for every slot the mazes its next `depth` regenerations would draw:
 * maze_generate keys its random stream by (seed, slot id, generation count), so M(m, g) can be drawn early; it lives in
 * entry g % depth.  ready_gen [depth, M] int32: g + 1 once the entry holds M(m, g) completely, 0 while it is being redrawn.
 *   maze_regen_swap     (stepping stream) for the `*queue_count` winners in `queue`: copy the entry of the live generation
 *                       count over the live slot if it is ready, else append the slot to slow_queue (the caller then
 *                       runs maze_generate on slow_queue / slow_count in place, as without a ring); every winner is
 *                       appended to refill_queue once per `batch` (queued_tag [M], initialised to -1).  stats [2]
 *                       (optional) counts fast / slow slots; wins [M] (optional) is the curriculum's win count, incremented
 *                       for the slots installed from the ring (maze_curriculum does it for the slow ones).  slow_count
 *                       must be zero on entry.
 *   maze_regen_prepare  (side stream) for the slots of refill_queue: ring entries that already hold the maze they should
 *                       are left alone, the others are un-published (ready_gen = 0), get their generation count and the
 *                       shape / generator the curriculum gives that count -- maze_curriculum's rule (grow, max shape, generator
 *                       thresholds; grow = 0 and algo = -1: none) applied in closed form to a snapshot of the slot records
 *                       and win counts taken when the ring was built (base_meta [M, 8], base_wins [M] or NULL) -- and are
 *                       appended to work_queue [depth, M] / work_count [depth] of their ring index.  Then, per ring index j: maze_generate(entry-j slices of the ring,
 *                       ids = work_queue[j], count_dev = work_count + j), and
 *   maze_regen_publish  (side stream) ready_gen = the entry's generation count for everything in the work queues.
 * Every path installs the same maze, so results do not depend on how far the side stream is behind. */
int maze_regen_swap(maze_ctx* ctx, uint8_t* grids, uint8_t* table, int32_t* meta, const uint8_t* shadow_grids, const uint8_t* shadow_table,
                    const int32_t* shadow_meta, const int32_t* ready_gen, int depth, const int32_t* queue, const int32_t* queue_count, int n,
                    int slot, int32_t* refill_queue, int32_t* refill_count, int32_t* queued_tag, int batch, int32_t* slow_queue,
                    int32_t* slow_count, int32_t* stats, int32_t* wins, void* stream);
int maze_regen_prepare(maze_ctx* ctx, const int32_t* meta, const int32_t* base_meta, const int32_t* base_wins, int grow, int max_h, int max_w,
                       int wins_a, int algo_a, int wins_b, int algo_b, int32_t* shadow_meta, int32_t* ready_gen, int depth,
                       const int32_t* refill_queue, const int32_t* refill_count, int n, int32_t* work_queue, int32_t* work_count, void* stream);
int maze_regen_publish(maze_ctx* ctx, const int32_t* shadow_meta, int32_t* ready_gen, int depth, const int32_t* work_queue,
                       const int32_t* work_count, int n, void* stream);

/* Enriched (-v1) observation: SimpleEnrichMazeEnv._get_obs (simple_maze_env.py:151-158) and the
 * toroidal / variable-size variants (toroidal_maze_env.py:164-172, simple_variable_maze_env.py:
 * 170-179, toroidal_variable_maze_env.py:186-194) for the current position of every env:
 *   window      [B, 3, 15, 15] float32 = [maze == 0, maze == 1 (goal excluded), non_visited] of the
 *               15 x 15 crop around the agent: lib/maze_handler.py:4-54 (euclid: clamped into the
 *               grid, so not centred near the border), :56-80 (torus: centred, wraps), :82-99
 *   agent_norm  [B, 2] float64 = agent / maze_shape, target_norm likewise (either may be NULL)
 * Needs H, W >= 15.  Reads the step table, so the goal block must be the pool's goal (value 2).
 * `window` must be 16-byte aligned (it is written with 16-byte stores). */
int maze_window(maze_ctx* ctx, const maze_env_batch* b, float* window, double* agent_norm, double* target_norm,
                void* stream);

/* get_mask_direction (simple_maze_env.py:41-50, toroidal_maze_env.py:57-70; lib/maze_handler.py:
 * 122-162): mask [B, 4] float32 in action order (down, up, right, left), 1 where the neighbour
 * block is open.  probs != 0: once an episode has made two successful moves the entry pointing
 * back to the previous block is overwritten with 0.25 (the toroidal env builds that direction
 * column-first, so the 0.25 lands on a rotated index -- reproduced). */
int maze_direction_mask(maze_ctx* ctx, const maze_env_batch* b, int probs, float* mask, void* stream);

/* ---- tabular Q-learning / double Q-learning on the device -------------------------------------
 * agents/q_agent.py:8-79 (QAgent) and agents/dq_agent.py:5-73 (DQAgent).  The reference keys its
 * tables by str(obs) of {'agent', 'target', 'best dir'}; the device table is an open-addressing hash
 * table keyed by the same triple (packed: agent row/col, target row/col, best-dir code, agent id),
 * rows of 4 float64 that start at zero like the reference's defaultdict.  `envs_per_agent`
 * consecutive envs share one agent (1 = independent replicas, the faithful reading of the
 * reference; num_envs = one learner fed by every env: concurrent updates of one entry race and one
 * wins, and gamma moves by eta / envs_per_agent per finished episode).
 * Every env keeps its own `steps_done` for the epsilon schedule. */
#define MAZE_Q_EMPTY     0xffffffffffffffffull
#define MAZE_Q_NO_SLOT   0xffffffffu
typedef struct maze_q_agent {
    int64_t   capacity;        /* rows; power of two, <= 2^31                                   */
    uint64_t* keys;            /* [capacity] packed observation keys, MAZE_Q_EMPTY when free    */
    double*   q_a;             /* [capacity, 4]  q_values (QAgent) / q_a_values (DQAgent)       */
    double*   q_b;             /* [capacity, 4]  q_b_values; NULL selects plain Q-learning      */
    int32_t*  overflow;        /* [1] set when a key found no free row (grow the table)         */
    int32_t   envs_per_agent;
    int32_t   eps_len;
    const double* eps_lut;     /* [eps_len] epsilon by steps_done (maze_q_epsilon_lut), the last
                                  entry is used beyond the end                                  */
    double*   gamma;           /* [ceil(B / envs_per_agent)] discount factor of each agent      */
    double    lr;              /* learning rate                                                 */
    double    eta;             /* update_hyperparameter step: gamma += eta if return > 0 else -= */
    /* per-env learner state */
    uint32_t* slot;            /* [B] row of the env's current observation, MAZE_Q_NO_SLOT = unknown */
    uint32_t* steps_done;      /* [B] get_action calls made for this env                        */
    uint8_t*  last_action;     /* [B] action chosen by maze_q_act (consumed by maze_q_update)   */
    double*   ep_return;       /* [B] cumulative reward of the running episode                  */
    /* randomness: Philox4x32-10 keyed by (seed, env_id_base + env, steps_done) ... */
    uint64_t  seed;
    int64_t   env_id_base;
    /* ... unless replay tapes are given (tests: the reference's recorded numpy draws) */
    const double*  u_tape;     /* [u_len, B] values np.random.random() returned, in call order  */
    const uint8_t* a_tape;     /* [a_len, B] values action_space.sample() returned              */
    uint32_t* tape_pos;        /* [2, B] cursors into u_tape / a_tape                           */
    int32_t   u_len, a_len;
} maze_q_agent;

/* Host helper: out[i] = final + (initial - final) * exp(-1. * i / decay)  (q_agent.py:49), computed
 * with libm exp on the host like the reference.  `out` is a HOST pointer to n doubles. */
int maze_q_epsilon_lut(double initial_epsilon, double final_epsilon, double decay, double* out, int n);

/* QAgent.get_action / DQAgent.get_action for every env (q_agent.py:44-54, dq_agent.py:36-47):
 * epsilon-greedy on q_a at the env's current observation; writes actions[B] (uint8) and remembers
 * them in agent->last_action.  Envs waiting for an autoreset make no decision (action 0). */
int maze_q_act(maze_ctx* ctx, const maze_env_batch* b, const maze_q_agent* agent, uint8_t* actions, void* stream);

/* QAgent.update / DQAgent.update (q_agent.py:56-72, dq_agent.py:49-66) for the transition maze_step
 * just made with agent->last_action: obs = the row remembered in agent->slot, next_obs = the env's
 * new state, reward / terminated from the batch outputs.  Envs whose step was an autoreset only
 * re-anchor their row.  On episode end applies update_hyperparameter (gamma +- eta,
 * off_policy_trainer.py:76-78: increment iff the episode return is > 0). */
int maze_q_update(maze_ctx* ctx, const maze_env_batch* b, const maze_q_agent* agent, void* stream);

/* Fused rollout: k_steps iterations of { get_action ; BaseMazeEnv.step ; update } per env in ONE
 * launch (the loop of off_policy_trainer.py:38-51), state kept in registers, with next-step
 * autoreset.  Leaves the batch outputs (obs, reward, terminated, truncated) of the last step. */
int maze_q_rollout(maze_ctx* ctx, const maze_env_batch* b, const maze_q_agent* agent, int k_steps, uint32_t mode,
                   void* stream);

/* ---- DQN / DDQN data path (the steps either side of the env in the neural trainers) ------------
 * lib/replay_memory.py:8-24 (ReplayMemory: deque + uniform sample), agents/ddqn_agent.py:95-108
 * (epsilon-greedy whose exploration draws from get_mask_direction(probs=True)), and the state the
 * trainer builds from the -v1 observation (lib/trainers/off_policy_trainer.py:153-171):
 * state = (float32[6] = agent / shape, target / shape, best dir ; float32[3, 15, 15] window).
 * The ring keeps windows BIT-PACKED (3 channels x 8 words = 96 B instead of 2 700 B; word k of a
 * channel holds window rows 2 k in bits 0-14 and 2 k + 1 in bits 16-30) and unpacks them when a
 * batch is sampled. */
#define MAZE_WINDOW_WORDS 24   /* 3 channels x 8 uint32 (225 of 256 bits used per channel)        */
typedef struct maze_replay {
    int64_t   capacity;     /* transitions in the ring                                            */
    unsigned long long* pushed; /* [1] device counter: transitions pushed so far                  */
    float*    vec;          /* [capacity, 6]  state vector                                        */
    float*    next_vec;     /* [capacity, 6]                                                      */
    uint32_t* win;          /* [capacity, MAZE_WINDOW_WORDS] packed window of the state           */
    uint32_t* next_win;     /* [capacity, MAZE_WINDOW_WORDS]                                      */
    uint8_t*  action;       /* [capacity]                                                         */
    float*    reward;       /* [capacity]                                                         */
    /* per-env staging: the observation the env's next transition starts from */
    float*    stage_vec;    /* [B, 6]                                                             */
    uint32_t* stage_win;    /* [B, MAZE_WINDOW_WORDS]                                             */
    int32_t   without_replacement; /* 1: a batch holds n DISTINCT transitions (random.sample, lib/replay_memory.py:20-21;
                               falls back to independent draws while fewer than n are stored); 0: independent
                               uniform draws                                                        */
    int32_t   reserved;
} maze_replay;

/* Encode the current observation of every env into the staging area (after maze_reset). */
int maze_dqn_observe(maze_ctx* ctx, const maze_env_batch* b, const maze_replay* r, void* stream);

/* agent.memorize(state, action, reward, next_state) for the transition maze_step just made with
 * `actions` (off_policy_trainer.py:171; next_state is never None there, terminal states included):
 * appends (staged observation, action, reward, new observation) to the ring and re-stages the new
 * observation.  Envs whose step was an autoreset only re-stage. */
int maze_dqn_push(maze_ctx* ctx, const maze_env_batch* b, const maze_replay* r, const uint8_t* actions, void* stream);

/* memory.sample(n): n transitions drawn uniformly from the filled part of the ring (distinct ones when
 * replay.without_replacement is set -- random.sample, lib/replay_memory.py:20-21 -- by taking the first n images of a
 * keyed pseudo-random permutation of the filled slots; Philox keyed by seed / draw either way), unpacked into dense
 * tensors: vec / next_vec [n, 6] float32,
 * win / next_win [n, 3, 15, 15] float32, action [n] int64, reward [n] float32. */
int maze_dqn_sample(maze_ctx* ctx, const maze_replay* r, int n, uint64_t seed, uint64_t draw, float* vec, float* win,
                    float* next_vec, float* next_win, int64_t* action, float* reward, void* stream);

/* DDQNAgent.get_action for every env (ddqn_agent.py:98-108): with probability eps_lut[steps_done[e]]
 * a random action drawn from get_mask_direction(probs=True) / sum, otherwise argmax of q_values[e]
 * ([B, 4] float32, the policy network's output).  steps_done [B] uint32 is advanced for every env
 * that makes a decision (not for envs waiting for an autoreset). */
int maze_dqn_select(maze_ctx* ctx, const maze_env_batch* b, const float* q_values, const double* eps_lut, int eps_len,
                    uint32_t* steps_done, uint64_t seed, int64_t env_id_base, uint8_t* actions, void* stream);

/* ---- DQN / DDQN network on the tensor cores (north star item 4; BASELINE.json configs[4]) ------------
 * The net of agents/ddqn_agent.py:18-52 (dqn_agent.py:19-57 is the same without Dropout):
 *   Conv2d(3, 32, 3, padding 1) + LeakyReLU + Dropout(p) + MaxPool2d(2, 2) on the 3 x 15 x 15 window -> 32 x 7 x 7 = 1568
 *   cat(conv features, 6 state floats) -> Linear(1574, 1024) + LeakyReLU -> Linear(1024, 512) + ReLU -> Linear(512, 4)
 * and its update: update = 0 (ddqn_agent.py:113-152): q(s, a) of the source net, a* = argmax q_source(s', .),
 * y = r + gamma * q_target(s', a*); update = 1 (the plain DQN target): y = r + gamma * max_a q_target(s', a), no source
 * forward on s'.  Then MSE loss (mean), elementwise gradient clamp to +-1, AdamW.  Neither target masks terminal states.
 *
 * Dropout: p = maze_dqn_net.dropout (0 = none, the default; the reference's DDQN uses 0.2 and, never calling eval(), drops
 * in every forward).  It applies in training mode (eval = 0) to every forward of maze_dqn_backward (each draws its own
 * mask) and to maze_dqn_forward / maze_dqn_features; eval = 1 turns it off everywhere, like nn.Module.eval().
 *   pooled = first maximum over the 2 x 2 candidates of  keep ? fp32(LeakyReLU(conv + bias) * s) : +0,  then bf16,
 *   s = fp32(1 / (1 - p)) (1.25 at p = 0.2).  A dropped element is +0 (torch's x * 0 is -0 for a negative x; the two
 *   compare equal, so only the sign of a pooled zero differs).
 * The keep bit of an element is a pure function of (dropout_seed, draw, forward id, sample, element):
 *   Philox4x32-10, key (dropout_seed lo, hi), counter (e / 8, sample index, draw lo 32 bits, forward id),
 *   e = ((py * 7 + px) * 32 + channel) * 4 + 2 dy + dx over the 14 x 14 conv positions (2 py + dy, 2 px + dx) the pool
 *   reads; the block's 16-bit draw k = e % 8 is bits 16 (k & 1) .. +15 of output word k / 2;
 *   keep iff draw < round(65536 (1 - p))  (P(keep) = 0.800003 at p = 0.2).
 *   Forward ids: 0 source net on s, 1 source net on s', 2 target net on s', 3 maze_dqn_forward / maze_dqn_features.
 * A caller bumps `draw` between calls (the Python DQNNet does on every forward, features and backward call) so that
 * each call draws fresh masks; equal seeds and equal call sequences give bit-identical results.
 *
 * Parameters live in ONE flat fp32 buffer per net (source `params`, target `target`), laid out as
 *   conv weight [32, 3, 3, 3] | conv bias [32] | fc1 weight [1024, 1600] | fc1 bias [1024] |
 *   fc2 weight [512, 1024] | fc2 bias [512] | fc3 weight [4, 512] | fc3 bias [4]
 * where fc1's 1600 input columns are the 1568 conv features (channel * 49 + row * 7 + col, as
 * fw.view(batch, -1) orders them), the 6 state floats, and 26 zero columns (K padded to a multiple of 64 for the
 * tensor-core tiles; their weights and gradients stay zero).  Gradients and the AdamW moments use the same
 * layout.  The bf16 copies are the tensor-core operands: w1 / w2 as stored ([out, in], the forward pass) and
 * transposed ([in, out], the backward-data pass); maze_dqn_net_refresh rebuilds them from the fp32 masters. */
#define MAZE_NET_IN       1600   /* 1568 + 6, padded                                             */
#define MAZE_NET_IN_USED  1574
#define MAZE_NET_H1       1024
#define MAZE_NET_H2       512
#define MAZE_NET_OFF_CONV_W 0
#define MAZE_NET_OFF_CONV_B 864
#define MAZE_NET_OFF_W1     896
#define MAZE_NET_OFF_B1     (MAZE_NET_OFF_W1 + MAZE_NET_H1 * MAZE_NET_IN)
#define MAZE_NET_OFF_W2     (MAZE_NET_OFF_B1 + MAZE_NET_H1)
#define MAZE_NET_OFF_B2     (MAZE_NET_OFF_W2 + MAZE_NET_H2 * MAZE_NET_H1)
#define MAZE_NET_OFF_W3     (MAZE_NET_OFF_B2 + MAZE_NET_H2)
#define MAZE_NET_OFF_B3     (MAZE_NET_OFF_W3 + 4 * MAZE_NET_H2)
#define MAZE_NET_PARAMS     (MAZE_NET_OFF_B3 + 4)   /* 2 167 172 floats                         */
typedef struct maze_dqn_net {
    float*    params;     /* [MAZE_NET_PARAMS] source net, fp32 master                              */
    float*    target;     /* [MAZE_NET_PARAMS] target net                                           */
    float*    grads;      /* [MAZE_NET_PARAMS] gradient accumulators; zero between steps (training) */
    float*    adam_m;     /* [MAZE_NET_PARAMS] AdamW first moment                      (training)   */
    float*    adam_v;     /* [MAZE_NET_PARAMS] AdamW second moment                     (training)   */
    uint16_t* w1_bf16;    /* [1024, 1600] bf16 source fc1 weight                                    */
    uint16_t* w2_bf16;    /* [512, 1024]                                                            */
    uint16_t* w1t_bf16;   /* [1600, 1024] transposed                                   (training)   */
    uint16_t* w2t_bf16;   /* [1024, 512]                                               (training)   */
    uint16_t* tw1_bf16;   /* target net operands                                                    */
    uint16_t* tw2_bf16;
    void*     workspace;  /* maze_dqn_net_workspace_bytes(max_batch) bytes, 256-byte aligned        */
    float*    loss;       /* [1] loss of the last maze_dqn_backward                     (training)   */
    int32_t   max_batch;  /* samples per call the workspace was sized for                           */
    int32_t   reserved;
    float     dropout;    /* Dropout p in [0, 1); 0 = no dropout                                    */
    int32_t   update;     /* 0 double-Q target (DDQN), 1 max target (DQN)                           */
    int32_t   eval;       /* 0 training mode (dropout active, as in the reference), 1 evaluation    */
    int32_t   reserved2;
    uint64_t  dropout_seed;  /* Philox key of the dropout masks                                     */
    uint64_t  draw;          /* call counter: its low 32 bits are a word of the mask counter        */
} maze_dqn_net;              /* all-zero new fields: no dropout, double-Q (the behaviour of ABI 13) */

int64_t maze_dqn_net_workspace_bytes(int max_batch);

/* Rebuild the bf16 operand copies of one net (which = 0 source, 1 target) from its fp32 parameters: after
 * initialisation, load_state_dict, or update_target (ddqn_agent.py:161-162: copy params -> target, then refresh 1). */
int maze_dqn_net_refresh(maze_ctx* ctx, const maze_dqn_net* net, int which, void* stream);

/* net(state) for n samples (ddqn_agent.py:44-49, :106): vec [n, 6] float32, win [n, MAZE_WINDOW_WORDS] packed windows
 * (the replay ring's format: DeviceReplay.stage_vec / stage_win are valid inputs), q_out [n, 4] float32. */
int maze_dqn_forward(maze_ctx* ctx, const maze_dqn_net* net, int which, const float* vec, const uint32_t* win, int n,
                     float* q_out, void* stream);

/* The conv stage alone: X [n, MAZE_NET_IN] bf16 feature rows; pool_idx (optional, [n, 1568] uint8: bits 0-1 the
 * max-pool choice dy * 2 + dx, bit 2 the winner's pre-activation > 0, bit 3 the winner was dropped -- always 0 without
 * dropout).  Dropout as for forward id 3.  Exposed for the parity tests. */
int maze_dqn_features(maze_ctx* ctx, const maze_dqn_net* net, int which, const float* vec, const uint32_t* win, int n,
                      uint16_t* X, uint8_t* pool_idx, void* stream);

/* optimize_model up to loss.backward() (ddqn_agent.py:113-144) on a batch of n transitions (n a multiple of 8):
 * adds d loss / d params into net->grads (so that ranks can be summed before the optimiser runs), writes the loss
 * to net->loss and, if qsa_out is not NULL, q(s, a) [n].  action [n] uint8, reward [n] float32.
 * fc_ready_event (optional cudaEvent_t): recorded on `stream` once every gradient except the conv layer's -- the flat
 * buffer from MAZE_NET_OFF_W1 on, 99.96 % of it -- is complete, so that a gradient all-reduce can overlap the rest of
 * the backward pass (the backward-data GEMM into the conv features and the conv weight gradient). */
int maze_dqn_backward(maze_ctx* ctx, const maze_dqn_net* net, const float* vec, const uint32_t* win, const float* next_vec,
                      const uint32_t* next_win, const uint8_t* action, const float* reward, int n, float gamma,
                      float* qsa_out, void* fc_ready_event, void* stream);

/* param.grad.clamp_(-clamp, clamp) (ddqn_agent.py:146-147; clamp <= 0 disables) on grads * grad_scale, then one
 * torch.optim.AdamW step (`step` counts from 1), then zeroes the gradient accumulators and refreshes the source
 * net's bf16 operands.  grad_scale = 1 / world_size after an all-reduce(sum) of net->grads reproduces DDP's mean. */
int maze_dqn_adamw(maze_ctx* ctx, const maze_dqn_net* net, float lr, float beta1, float beta2, float eps, float weight_decay,
                   int64_t step, float grad_scale, float clamp, void* stream);

/* In-situ launch times of maze_dqn_backward: while enabled, every launch of a backward call is followed by a CUDA event
 * on the caller's stream; _read waits for the last call's events and returns the `count` per-launch durations (ms) in
 * launch order with their labels (label_bytes per entry, NUL-terminated; labels may be NULL).  This is how bench.py
 * measures the dominant kernel's duration inside the step (ncu's replays are serialised and cold-cache). */
int maze_dqn_net_profile(maze_ctx* ctx, int enable);
int maze_dqn_net_profile_read(maze_ctx* ctx, float* ms, char* labels, int label_bytes, int cap, int* count);

/* memory.sample(n) that keeps the windows packed: the same draw as maze_dqn_sample (same seed / draw -> same
 * transitions), 212 bytes per transition instead of 5.5 KB.  action [n] uint8. */
int maze_dqn_sample_packed(maze_ctx* ctx, const maze_replay* r, int n, uint64_t seed, uint64_t draw, float* vec, uint32_t* win,
                           float* next_vec, uint32_t* next_win, uint8_t* action, float* reward, void* stream);

/* The tensor-core GEMM underneath: C[M, N] = A[M, K] . B[N, K]^T with bf16 row-major operands (row pitches lda, ldb
 * in elements, multiples of 8; 16-byte aligned bases), N a multiple of 8.  epilogue 0: C bf16 = act(acc + bias)
 * (act 0 none, 1 LeakyReLU(0.01), 2 ReLU; bias may be NULL); 1: C bf16 = acc * act'(aux) with aux [M, ldaux] bf16 the
 * stored activation; 2: C fp32 += acc (atomic, `splits` CTAs along K); 3: as 2 with TRANSPOSED operands, A [K, M] and
 * B [K, N] row-major, i.e. C += A^T . B (the weight gradients, straight from [batch, features] activations; M a multiple
 * of 8).  tile_n 128 or 256 (one CTA per 128 x tile_n tile), or 512: CTA pairs (tcgen05 cta_group::2) on 256 x 256 tiles,
 * epilogues 0 and 1 only. */
int maze_dqn_gemm_bf16(maze_ctx* ctx, const uint16_t* A, int lda, const uint16_t* B, int ldb, void* C, int ldc, int M, int N, int K,
                       int epilogue, int act, const float* bias, const uint16_t* aux, int ldaux, int tile_n, int splits, void* stream);

/* Difficulty metrics of pool mazes, one record of MAZE_METRIC_WORDS doubles per processed slot
 * (out[k] belongs to ids[k], or to slot k when ids is NULL):
 *   McClendon difficulty / complexity  lib/maze_difficulty_evaluation/maze_complexity_evaluation.py:310-329
 *     (graph construction :57-91, hallways :186-221, branches :223-259, honouring the `break` of :209-214)
 *   Kim-Crawfis L / DE / D              lib/maze_difficulty_evaluation/metrics_calculator.py:22-26,87-127,71-85
 * These are the six columns of the README table (generation_algos_metrics_evaluations.py:31-43).
 * Mazes must be perfect (spanning trees); toroidal slots are scored on the zero-padded grid, i.e.
 * the bordered maze gen_maze_no_border scored (lib/maze_generation.py:48-56).  A slot whose goal
 * cannot be reached from its start gets NaNs.  Floating-point sums run in a different order than
 * networkx iteration: parity is to 1e-9 relative, L / DE / D are exact. */
#define MAZE_METRIC_WORDS 8
#define MAZE_METRIC_DIFFICULTY 0
#define MAZE_METRIC_COMPLEXITY 1
#define MAZE_METRIC_L          2
#define MAZE_METRIC_DE         3
#define MAZE_METRIC_D          4
#define MAZE_METRIC_SOL_LEN    5  /* len(path(start->goal)) in blocks                          */
#define MAZE_METRIC_DE_COUNT   6  /* dead ends counted by calculate_DE                         */
int maze_difficulty(maze_ctx* ctx, const uint8_t* grids, const int32_t* meta, const int32_t* ids,
                    int n, int slot, int max_h, int max_w, double* out, void* stream);

/* maze_difficulty plus the Kim-Crawfis metrics MetricsCalculator defines but nothing in the
 * reference calls (lib/maze_difficulty_evaluation/metrics_calculator.py): one extra record of
 * MAZE_METRIC_EXT_WORDS doubles per processed slot in ext_out.  All are bit-identical to the
 * reference (same divisions; the dead-end sums run in its row-major dead-end order).
 *   density :18-20; T :28-37, J :39-53, CR :55-69 of the solution path;
 *   AC, FDE, BDE = the three terms of DE (calculate_DE_sub :100-127);
 *   L_DE :224-241; T_DE / D_sharp / L_sharp :175-222 for dead-end types AC, FDE, BDE (3 words each).
 * find_decision (:243-255) iterates an empty range and always returns None; L_DE and L_sharp are
 * therefore plain sums of len(de_path) / CE, which is what is computed here. */
#define MAZE_METRIC_EXT_WORDS   20
#define MAZE_METRIC_EXT_DENSITY 0
#define MAZE_METRIC_EXT_T       1
#define MAZE_METRIC_EXT_J       2
#define MAZE_METRIC_EXT_CR      3
#define MAZE_METRIC_EXT_AC      4
#define MAZE_METRIC_EXT_FDE     5
#define MAZE_METRIC_EXT_BDE     6
#define MAZE_METRIC_EXT_L_DE    7
#define MAZE_METRIC_EXT_T_DE    8   /* [3]: AC, FDE, BDE */
#define MAZE_METRIC_EXT_D_SHARP 11  /* [3] */
#define MAZE_METRIC_EXT_L_SHARP 14  /* [3] */
int maze_difficulty_ext(maze_ctx* ctx, const uint8_t* grids, const int32_t* meta, const int32_t* ids,
                        int n, int slot, int max_h, int max_w, double* out, double* ext_out, void* stream);

/* The frame MazeViewTemplate draws (lib/maze_view.py:12-14,88-104,148-152; render_mode "rgb_array",
 * base_maze_env.py:15,212-222) for n envs (env_ids NULL = envs 0..n-1): out uint8 [n, out_h, out_w, 3],
 * out_h / out_w = 16 x the pool's maximum shape; 16 x 16 tiles in CELL_COLORS with a one-pixel
 * outline, orange on blocks the agent has left in the current episode, the agent as an 8 x 8 square;
 * pixels beyond a (smaller) maze and the window's last row / column are black.  The reference never
 * repaints outlines on reset, so its trails accumulate over episodes on one maze; here a frame shows
 * the current episode only (state lives in the visit counters, not in a surface). */
#define MAZE_RENDER_TILE 16
int maze_render(maze_ctx* ctx, const maze_env_batch* b, const int32_t* env_ids, int n, uint8_t* out,
                int out_h, int out_w, void* stream);

/* ---- packed maze sets (SURVEY.md section 8(f) rank 3: wire / on-disk interchange) -------------------
 * Record k of `packed` (packed_stride bytes) belongs to slot ids[k] (slot k when ids is NULL); H, W,
 * goal and flags of a slot come from its meta record, which the caller fills before maze_unpack
 * (then maze_fields rebuilds the step table).  The reference has no such format (its mazes are Python
 * lists of lists, lib/maze_generation.py:17); the file layout built on it is documented in
 * maze_b200/mazeset.py.
 *   MAZE_PACK_BITMAP  1 bit per block (open != 0), row-major, LSB first, (H*W + 7) / 8 bytes:
 *                     lossless for every grid, both topologies
 *   MAZE_PACK_WALLS   4 wall bits per logical cell (N 1, E 2, S 4, W 8; set = wall), two cells per
 *                     byte, low nibble first, (cells + 1) / 2 bytes: bordered (euclidean) mazes whose
 *                     logical cells are all open, i.e. every generator output (800 B for 40 x 40) */
#define MAZE_PACK_BITMAP 0
#define MAZE_PACK_WALLS  1
int maze_pack(maze_ctx* ctx, const uint8_t* grids, const int32_t* meta, const int32_t* ids, int n, int slot,
              int format, uint8_t* packed, int packed_stride, void* stream);
int maze_unpack(maze_ctx* ctx, const uint8_t* packed, int packed_stride, int format, uint8_t* grids,
                const int32_t* meta, const int32_t* ids, int n, int slot, void* stream);

/* generate_collection_of_mazes' tensor encode (lib/maze_generation.py:236-242): out int32 [n, 3, h, w]
 * = [wall (== 0), tile (== 1, the goal is neither), non_visited (!= 0, start cleared)] of n slots of
 * one shape. */
int maze_collection_encode(maze_ctx* ctx, const uint8_t* grids, const int32_t* meta, const int32_t* ids, int n,
                           int slot, int h, int w, int32_t* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MAZE_B200_H */
