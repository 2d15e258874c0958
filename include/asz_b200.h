/*
 * asz_b200.h -- C ABI of the B200-native AlphaSnake-Zero self-play engine (libasz_b200.so).
 *
 * The reference (Fool-Yang/AlphaSnake-Zero) is pure Python and has no FFI of its own; the seams this library sits
 * behind are the duck-typed Python classes of code/utils/ (SURVEY.md section 8(b)).  Every entry point below names
 * the reference interface it replaces (file:line under /root/reference/code/utils/).  The Python mirror of those
 * classes lives in alphasnake_zero_b200/utils/ and binds this header with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - plain C types only; every function returns 0 on success or a negative asz_status, asz_last_error() explains;
 *   - pointers named d_* are DEVICE pointers (e.g. torch tensor .data_ptr()), h_* are HOST pointers;
 *   - `stream` is a cudaStream_t passed as void* (NULL = the legacy default stream); calls only enqueue work on
 *     that stream unless documented as synchronous (the *_host / readback calls);
 *   - one engine per GPU (the device current at asz_engine_create), calls on one engine are not thread-safe
 *     (the reference is single-threaded);
 *   - snakes are indexed by id (0..S-1), slot = game*8 + snake in per-snake arrays (8 = ASZ_MAX_SNAKES);
 *   - relative moves are 0 = left, 1 = straight, 2 = right (game.py:92).
 */
#ifndef ASZ_B200_H
#define ASZ_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ASZ_MAX_SNAKES 8
#define ASZ_VERSION 2

typedef enum {
  ASZ_OK = 0,
  ASZ_ERR_ARG = -1,      /* bad argument / unsupported configuration */
  ASZ_ERR_CUDA = -2,     /* a CUDA runtime call failed */
  ASZ_ERR_STATE = -3,    /* call not valid in the engine's current state */
  ASZ_ERR_CAPACITY = -4  /* an output or table capacity was exceeded */
} asz_status;

/* Engine configuration.  Mirrors the constructor arguments of Game / MPGameRunner (game.py:13, mp_game_runner.py:7)
 * and Agent (agent.py:9-10). */
typedef struct {
  int32_t side;            /* board height == width: 7, 11 or 19 (the standard boards of game.py:22-28) */
  int32_t snakes;          /* S, 1..8 (game.py:25-29 samples S of 8 start cells) */
  int32_t health_dec;      /* game.py:13 health_dec */
  float food_chance;       /* game.py:13 food_spawn_chance (0.15 in the reference's runners) */
  int32_t games;           /* G, number of root games held by this engine (mp_game_runner.py:13) */
  uint64_t seed;           /* key of the engine's counter-based RNG (Philox4x32-10) */
  /* search (0 disables the search subsystem and its allocations) */
  int32_t max_depth;       /* agent.py:10 max_MCTS_depth */
  int32_t max_breadth;     /* agent.py:10 max_MCTS_breadth */
  float softmax_base;      /* agent.py:9 softmax_base */
  int32_t training;        /* agent.py:9 training */
  int32_t table_log2;      /* log2 of the Q-table capacity in slots (0 = choose from G, breadth, depth) */
  int32_t numpy1_mask;     /* 0: obstacle threshold compared in float32 (NumPy >= 2), 1: in float64 (NumPy 1.18),
                              alpha_nnet.py:75-76, SURVEY.md D-11 */
} asz_config;

typedef struct asz_engine asz_engine;

const char* asz_last_error(void);
int asz_version(void);

/* ---- lifecycle ------------------------------------------------------------------------------------------------ */
/* MPGameRunner.__init__ (mp_game_runner.py:7-20): allocates G games on the current device; games are NOT initialised
 * until asz_reset / asz_set_state. */
int asz_engine_create(asz_engine** out, const asz_config* cfg);
int asz_engine_destroy(asz_engine* e);
/* Game.__init__ for every game (game.py:13-61) with the engine's RNG; episode counters restart at 0. */
int asz_reset(asz_engine* e, void* stream);

/* ---- state interchange (debug / replay / tests); synchronous; all HOST int32 arrays --------------------------
 * canonical dump of one game:
 *   snake[S*6]   = alive, health, length, last_move, head_cell (-1 none), reward (0 none, 1, -1)
 *   owner[side^2] (-1 none), dist[side^2] (distance from tail of the topmost segment, 0 none), food[side^2] (0/1)
 *   counters[8]  = wall, body, head, starve, food_eaten, game_length, episode, done
 * Replaces direct attribute access on Game objects (game.snakes, game.food, game.rewards, counters; game.py:20-61). */
int asz_get_state(asz_engine* e, int32_t game, int32_t* h_snake, int32_t* h_owner, int32_t* h_dist, int32_t* h_food,
                  int32_t* h_counters);
int asz_set_state(asz_engine* e, int32_t game, const int32_t* h_snake, const int32_t* h_owner, const int32_t* h_dist,
                  const int32_t* h_food, const int32_t* h_counters);

/* ---- lockstep tic + fused plane encode (Game.tic game.py:87-205, Game.get_states game.py:68-69, 215-257) ------
 * flags */
#define ASZ_STEP_TIC 1u          /* advance every live game by one tic */
#define ASZ_STEP_ENCODE 2u       /* write the plane of every live snake (after the tic) into d_planes */
#define ASZ_STEP_AUTO_RESET 4u   /* a game that ends is re-initialised in the same launch (its final rewards and
                                    counters are reported first); config-2 workload of BASELINE.json */
#define ASZ_STEP_RANDOM_ACT 8u   /* ignore d_actions, draw uniform relative moves from the engine RNG */
#define ASZ_STEP_KEYS 16u        /* also write the 128-bit plane key of every row into d_keys */
/* spawn modes */
#define ASZ_SPAWN_NONE 0         /* never spawn (Game.subgame, game.py:268) */
#define ASZ_SPAWN_REPLAY 1       /* d_spawn_cells[g] = cell index of the food spawned this tic, or -1 (trace replay) */
#define ASZ_SPAWN_NATIVE 2       /* engine RNG: coin `random() <= chance` or board without food, uniform empty cell */

typedef struct {
  uint32_t flags;
  int32_t spawn_mode;
  const uint8_t* d_actions;      /* [G*8] relative move per (game, snake id); read where the snake is alive */
  const int32_t* d_spawn_cells;  /* [G] for ASZ_SPAWN_REPLAY */
  float* d_planes;               /* [max_rows][2*side-1][2*side-1][3] float32 NHWC, rows compacted; 32-byte aligned; rows are
                                    plane_pitch floats apart (room for max_rows * plane_pitch floats) */
  int32_t* d_row_ids;            /* [max_rows] game*8 + snake of every row written */
  uint64_t* d_keys;              /* [max_rows*2] when ASZ_STEP_KEYS */
  int32_t max_rows;
  int32_t* d_row_count;          /* [1] number of rows written by this call (the call zeroes it first) */
  uint8_t* d_ended;              /* [G] 1 when the game ended in this tic (may be NULL) */
  int8_t* d_rewards;             /* [G*8] rewards after this tic per (game, snake id): 1 winner, -1 dead, 0 alive or no such snake
                                    (game.py:162-203); final where d_ended[g] = 1; all 0 for a game that was finished before
                                    this tic and was not stepped (may be NULL) */
  int32_t row_base;              /* rows are written at [row_base, row_base + n) of d_planes / d_row_ids / d_keys; max_rows
                                    stays the absolute capacity (rows past it are dropped, *d_row_count still counts them) */
  int32_t plane_pitch;           /* floats between consecutive rows of d_planes; must equal asz_plane_pitch() with ASZ_STEP_ENCODE
                                    (ASZ_ERR_ARG otherwise): the plane size rounded up to 8 floats, so that every row starts on a
                                    32-byte sector, the layout of the engine's own buffers (the pad floats after each plane are
                                    written but carry no meaning) */
} asz_step_args;

/* Enqueues one fused launch.  Row order inside d_planes is unspecified across games (rows of one game are
 * contiguous and in ascending snake id, the reference's live-list order, game.py:69); d_row_ids identifies them. */
int asz_env_step(asz_engine* e, const asz_step_args* args, void* stream);

/* Host-buffer convenience wrapper used for end-to-end timing: copies h_actions (pinned, [G*8]) to the device, runs
 * asz_env_step into the engine's internal plane buffer, copies the per-game results back and synchronises.
 * h_ended [G], h_rewards [G*8], h_row_count [1]; h_planes may be NULL (planes stay device resident for the network)
 * or a pinned buffer that receives rows*plane floats. */
int asz_env_step_host(asz_engine* e, uint32_t flags, int32_t spawn_mode, const uint8_t* h_actions,
                      const int32_t* h_spawn_cells, uint8_t* h_ended, int8_t* h_rewards, int32_t* h_row_count,
                      float* h_planes, int32_t* h_row_ids, void* stream);

/* The same step as two calls, so that a caller can keep two steps in flight: asz_env_submit_host enqueues the copy of the
 * step's inputs (on a copy stream of the engine: it runs under the previous step's kernel), the launch and the result
 * transfers, and returns a ticket (0 or 1) without waiting; asz_env_wait_host blocks until that step's h_ended / h_rewards
 * are complete in host memory and returns its row count.  At most two tickets are outstanding (a third submit is an
 * error); steps execute in submission order on `stream`, and the planes of a step stay in the engine's buffer until the next
 * step's launch, in stream order, overwrites them (enqueue their consumer on `stream` between the two submits).  The host
 * buffers of a step must stay untouched until its wait returns (two steps in flight need two sets of result buffers).
 * This is Game.tic for a batch of games whose next moves do not depend on this step's result at the time of the call:
 * uniform-random play (BASELINE.json configs[1]), replayed traces, or two populations stepped alternately. */
int asz_env_submit_host(asz_engine* e, uint32_t flags, int32_t spawn_mode, const uint8_t* h_actions,
                        const int32_t* h_spawn_cells, uint8_t* h_ended, int8_t* h_rewards, void* stream, int32_t* ticket);
int asz_env_wait_host(asz_engine* e, int32_t ticket, int32_t* h_row_count);

/* Running totals over games that ended since the last asz_reset (mp_game_runner.py:56-61, 71-76 divides by G):
 * h_totals[16] = wall, body, head, starve, food_eaten, game_length, episodes_finished, tics_executed, planes_written,
 * then 7 reserved slots (0).  Synchronous. */
int asz_get_totals(asz_engine* e, uint64_t* h_totals);

/* device pointers of the packed root-game records, read-only for callers: d_ptrs[0] = cells (u16 [G][padded cells]),
 * d_ptrs[1] = snakes (u64 [G][8]: head:16 | len:16 | health low byte:8 | last_move:2 | alive:1 | reward:2 | pad:3 |
 * health high byte:8; health is a signed 16-bit value, it can be <= 0 for a head-on winner, game.py:156-165), d_ptrs[2] = meta
 * (u32 [G][8]: game_length, episode, wall, body, head, starve, food_eaten, flags bit0 = finished).  Replaces
 * iterating `games` for liveness (mp_game_runner.py:40-42). */
/* measurement builds only (nvcc -DASZ_ENV_PROFILE, tools/env_profile.py): per-phase cycle sums of env_step_kernel since
 * the last call, h_cycles[8] = record wait, tic, write-back, work-counter wait + prefetch, cell view + row wait, encode,
 * two unused slots; all zero in the product build.  Synchronous. */
int asz_internal_profile(asz_engine* e, uint64_t* h_cycles);
int asz_internal_state(asz_engine* e, void** d_ptrs);
/* device pointer of the engine's internal plane buffer (capacity G*S rows, asz_plane_pitch() floats apart) and row-id buffer */
float* asz_internal_planes(asz_engine* e);
int32_t* asz_internal_row_ids(asz_engine* e);
size_t asz_plane_floats(const asz_engine* e);
/* row pitch (floats) of the engine's internal plane buffers: asz_plane_floats rounded up to a multiple of 8 */
size_t asz_plane_pitch(const asz_engine* e);

/* ---- search: Agent.make_moves (agent.py:25-111) = epochs x (MCTSMPGameRunner.run, mp_game_runner.py:85-115, over
 * MCTSAgent.make_moves, agent.py:161-223) ------------------------------------------------------------------------
 * Call sequence for one root turn (what Agent.make_moves does for `games`, the engine's current root games):
 *
 *   asz_search_begin                                   ages the table (agent.py:30-31)
 *   repeat max_breadth / min(8, max_breadth) times:    agent.py:37
 *     asz_search_epoch_begin                           8 sub-games per live root game (agent.py:39-50)
 *     for step = 1 .. max_depth + 1:
 *       asz_search_step_probe  -> n_miss               tic of the previous step's moves, leave check and terminal
 *                                                      backup (agent.py:60-72), keys, table probe, planes of the
 *                                                      misses in asz_search_eval_planes() (agent.py:170-186)
 *       <value network on n_miss planes, AlphaNNet.v contract, into asz_search_eval_values() or d_values>
 *       asz_search_step_sample                         priors, softermax, sample, estimated reward (agent.py:193-214);
 *                                                      skipped after the closing probe (step == max_depth + 1)
 *   asz_search_finish                                  root Q and root moves (agent.py:74-99), eviction (agent.py:101-110)
 *
 * Trace buffers (device, uint8): tree moves [epochs][max_depth][games*P][S] indexed by absolute sub-game id
 * game*P + sibling; trace_mode 0 = sample with the engine RNG, 1 = replay (read), 2 = sample and record (write).
 * Root trace [games*8] by slot (replay of the root moves when training). */
int asz_search_begin(asz_engine* e, void* stream);
int asz_search_epoch_begin(asz_engine* e, void* stream);
/* h_n_miss != NULL: synchronises the stream and returns the number of planes queued for the network */
int asz_search_step_probe(asz_engine* e, int32_t* h_n_miss, void* stream);
/* d_values: [n_miss][3] float32 network outputs WITH the obstacle mask applied, or NULL = asz_search_eval_values() */
int asz_search_step_sample(asz_engine* e, const float* d_values, uint8_t* d_trace, int32_t trace_mode, void* stream);
/* d_root_q [games*8*3], d_root_moves [games*8] (255 = no row) or NULL to keep them in the engine's buffers.
 * Returns ASZ_ERR_CAPACITY (after writing the outputs and closing the turn) when the Q table overflowed during the turn:
 * the dropped rows make the result differ from the reference's, so it is never silent. */
int asz_search_finish(asz_engine* e, const uint8_t* d_root_trace, float* d_root_q, uint8_t* d_root_moves, void* stream);
/* deterministic stub value function (value from the plane key + obstacle mask) on the queued planes; device side count */
int asz_search_stub_values(asz_engine* e, void* stream);
/* the whole sequence above with the stub value function and no host synchronisation in the loops */
int asz_search_run_stub(asz_engine* e, uint8_t* d_trace, int32_t trace_mode, const uint8_t* d_root_trace, void* stream);
/* the whole sequence above with the value network of asz_net_create (declared below) as AlphaNNet.v: Agent.make_moves
 * (agent.py:25-111) for one root turn in one call; the host only waits for each step's miss count */
struct asz_net;
int asz_search_run_net(asz_engine* e, struct asz_net* net, uint8_t* d_trace, int32_t trace_mode, const uint8_t* d_root_trace,
                       void* stream);
/* AlphaNNet.v's obstacle mask (alpha_nnet.py:63-76) applied in place to d_values [n][3] for d_planes [n][plane] */
int asz_obstacle_mask(asz_engine* e, const float* d_planes, int32_t n, float* d_values, void* stream);
/* test hook: Agent.softermax (agent.py:114-122), numpy.random.choice([0,1,2], p) for a given uniform draw u (float64),
 * and Agent.argmaxs (agent.py:124-137) on n rows of 3 values; all DEVICE pointers */
int asz_debug_policy(const float* d_z, const double* d_u, int32_t n, float base, float* d_pmf, int32_t* d_choice,
                     int32_t* d_argmax, void* stream);
/* Agent.clear (agent.py:140-147): drops the table */
int asz_search_clear(asz_engine* e, void* stream);
/* h_info[8] = P (sub-games per root game), epochs, max steps, sub-games, max eval rows, table log2 capacity, root turn, epoch */
int asz_search_info(asz_engine* e, int32_t* h_info);
float* asz_search_eval_planes(asz_engine* e);   /* device [max eval rows][plane] float32 */
float* asz_search_eval_values(asz_engine* e);   /* device [max eval rows][3] float32 */
float* asz_search_root_q(asz_engine* e);        /* device [games*8][3] */
uint8_t* asz_search_root_moves(asz_engine* e);  /* device [games*8] */
/* h_stats[16] = evals, node visits, hits(unused), sub-games, sub-game tics, tag collisions, inserts, re-created,
 * occupied slots, overflow (probes that found no free slot; asz_search_finish fails with ASZ_ERR_CAPACITY when this grew
 * during the turn), table compactions, of which between two epochs of one turn, ... ; synchronous */
int asz_search_stats(asz_engine* e, uint64_t* h_stats);
/* live (not evicted) table entries: keys [cap*2], W [cap*3], N [cap*3], age [cap]; *h_count = live entries. Synchronous.
 * Replaces inspection of Agent.cached_values / total_rewards / visit_cnts / cache_hit (agent.py:16-19); Q = W / N. */
int asz_search_table_dump(asz_engine* e, int32_t cap, uint64_t* h_keys, float* h_w, float* h_n, int32_t* h_age,
                          int32_t* h_count);

/* ---- training records: Agent.records / Agent.values (agent.py:21-23, 93-97) kept in HBM, and the trainer's sample +
 * mirror augmentation (alpha_snake_zero_trainer.py:62-77, 93-100) as one gather kernel ------------------------------
 * The reference appends one (root state, root Q) pair per live snake per root turn to two host lists; here the root
 * planes are encoded straight into an engine-owned store and only the moves go to the host each turn. */
/* allocates room for capacity_rows records (plane + 3 values + id + turn each); an earlier store is dropped.  The store
 * doubles when an append might not fit (device pointers from the accessors below change then). */
int asz_records_enable(asz_engine* e, int64_t capacity_rows);
/* agent.py:93-97 after asz_search_finish: state of every live snake of every live root game + its root Q row
 * (d_root_q [games*8][3], NULL = the engine's root Q buffer).  Records of one call are contiguous, rows of a game
 * contiguous in ascending snake id, game order unspecified (asz_records_ids tells).  Synchronises the stream;
 * *h_count = records held afterwards; ASZ_ERR_CAPACITY when the store cannot grow (nothing is dropped silently). */
int asz_records_append(asz_engine* e, const float* d_root_q, int64_t* h_count, void* stream);
int asz_records_count(asz_engine* e, int64_t* h_count);
/* Agent.clear (agent.py:140-147) for the records */
int asz_records_clear(asz_engine* e);
/* alpha_snake_zero_trainer.py:70-77: X = records[idx], V = values[idx]; with mirror != 0 the flipped copies
 * (states flipped along the width axis, values reversed: :93-100) follow the n originals.  d_idx [n] int64 DEVICE
 * indices (the reference draws them with random.sample on the host); d_X [(mirror ? 2 : 1) * n][plane], d_V [..][3]. */
int asz_records_gather(asz_engine* e, const int64_t* d_idx, int32_t n, int32_t mirror, float* d_X, float* d_V, void* stream);
float* asz_records_planes(asz_engine* e);     /* device [capacity][asz_plane_pitch()] */
float* asz_records_values(asz_engine* e);     /* device [capacity][3] */
int32_t* asz_records_ids(asz_engine* e);      /* device [capacity] game*8 + snake */
int32_t* asz_records_turns(asz_engine* e);    /* device [capacity] index of the append call */

/* ---- value network: AlphaNNet.v_net.predict (alpha_nnet.py:19-56, 62), inference only --------------------------
 * Weights are passed as DEVICE pointers in the layouts the kernels consume (alphasnake_zero_b200/net.py builds them
 * from the Keras-layout arrays: conv kernels HWIO, dense (in, out), BN gamma/beta/moving mean/variance, eps 1e-3):
 *   w_conv[0]     bf16 [1][4][128][8]   first convolution as a K=32 GEMM over im2col rows, k = (dy*3+dx)*3 + c
 *   w_conv[1..8]  bf16 [9][16][128][8]  [tap = dy*3+dx][cin / 8][cout][cin % 8]
 *   scale/bias    fp32 [128]            BatchNorm folded: y = conv * scale + bias
 *   head_w        fp32 [128]            1x1 head convolution; head_scale/head_bias = its folded BatchNorm
 *   dense1_w      fp32 [(2*side-1)^2][128], dense1_b [128], dense2_w [128][3], dense2_b [3] */
typedef struct {
  int32_t side;
  const void* w_conv[9];
  const float* scale[9];
  const float* bias[9];
  const float* head_w;
  float head_scale;
  float head_bias;
  const float* dense1_w;
  const float* dense1_b;
  const float* dense2_w;
  const float* dense2_b;
} asz_net_weights;

typedef struct asz_net asz_net;
/* chunk_images: images processed per pass (sizes the activation workspace: ~31 KB... 124 KB per image and buffer) */
int asz_net_create(asz_net** out, const asz_net_weights* w, int32_t chunk_images);
int asz_net_destroy(asz_net* net);
/* the per-generation weight push (alpha_snake_zero_trainer.py:52-57, 79-83): *w replaces the network's weight pointers
 * (same side; arrays stay owned by the caller) and the operands derived from them are rebuilt on `stream` */
int asz_net_update_weights(asz_net* net, const asz_net_weights* w, void* stream);
/* d_planes [count][2*side-1][2*side-1][3] float32 NHWC -> d_values [count][3] float32 tanh outputs (no obstacle mask;
 * asz_obstacle_mask applies AlphaNNet.v's mask).  bf16 operands, fp32 accumulation. */
int asz_net_forward(asz_net* net, const float* d_planes, int32_t count, float* d_values, void* stream);
/* the same for rows that are plane_pitch floats apart (asz_plane_pitch(): the engine's own plane buffers) */
int asz_net_forward_pitched(asz_net* net, const float* d_planes, int32_t plane_pitch, int32_t count, float* d_values, void* stream);
/* test hook: runs the tower up to convolution `layer` (0 = first conv, 1..8 = residual convs in order) and exports
 * that layer's output as float32 [count][2*side-1][2*side-1][128] ([..][1] for layer 8: the fused 1x1 head conv) */
int asz_net_debug_layer(asz_net* net, const float* d_planes, int32_t count, int32_t layer, float* d_act, void* stream);

/* fp8 networks (opt-in; outside the bf16 network's accuracy, DESIGN.md 4.3): activations stored as e4m3, residual
 * convolutions 1..8 with e4m3 operands and fp32 accumulation; the first convolution, the head and the dense layers as above.
 * Fields of w that differ from asz_net_weights':
 *   w_conv[1..8]  e4m3 [9][8][128][16]  [tap][cin / 16][cout][cin % 16], the weights divided by a per-output-channel scale
 *   scale[i]      fp32 [128]            folded BatchNorm scale times that weight scale times act_scale[i-1] (i >= 1)
 *   act_scale[i]  the power of two by which layer i's outputs are divided before they are stored as e4m3 (saturating at
 *                 +-448); ASZ_ERR_ARG unless every entry is one in [2^-125, 2^126] (act_scale[8] is not used: layer 8
 *                 is the fused head)
 * Every other entry point taking an asz_net* works on an fp8 network unchanged (asz_net_debug_layer exports the stored values
 * times act_scale: exact in fp32).  asz_net_update_weights refuses an fp8 network and asz_net_update_weights_fp8 a bf16 one. */
typedef struct {
  asz_net_weights w;
  float act_scale[9];
} asz_net_weights_fp8;
int asz_net_create_fp8(asz_net** out, const asz_net_weights_fp8* w, int32_t chunk_images);
int asz_net_update_weights_fp8(asz_net* net, const asz_net_weights_fp8* w, void* stream);

/* ---- pit: pit_mp_game_runner.MPGameRunner.run(Alice, Bob, Alice_snake_cnt) (pit_mp_game_runner.py:14-63) with
 * pit_agent.Agent (pit_agent.py:10-28) on both sides, played on the engine's root games without planes through the host (either
 * side may play the search Agent instead: asz_pit_set_search below) --------------------------------------------------------
 * Snakes with id < alice_snakes are Alice's, the others Bob's.  One turn: the rows of the running games are gathered into one
 * team buffer (Alice's, then Bob's, each in (game, snake) order), each side's network values its segment (one forward when
 * both sides share a network), AlphaNNet.v's obstacle mask and Agent.argmaxs pick the moves (every other slot plays 1, as in
 * the loop's np.ones((G, 8))), every unfinished game is stepped (a game decided early keeps being stepped with move 1 for its
 * live snakes, exactly like the loop), and the referee decides: a game that ended in this tic is won by the lowest snake id
 * with reward +1 (none = draw); otherwise, when one team has no live snake left, by the lowest live id.  The host waits once
 * per turn, for (rows of Alice, rows of Bob, games running).
 * Results: winners[g] = snake id or -1 (draw, or still running), decided_turn[g] = number of tics played when game g was
 * decided, -1 while it is running.  A game that was already finished when the match begins is decided at turn 0 with winner
 * -1 (the reference's loop fails on such a game). */
typedef struct {
  asz_net* net;          /* the side's value network (same board side and device as the engine), or NULL = stand-in player */
  int32_t stub_word;     /* net == NULL: value of move a = 16 bits (16a..16a+15) of word stub_word (0 or 1) of the plane key,
                            mapped to [-1, 1) (asz_search_stub_values uses word 1, a searched stand-in side this word),
                            then the obstacle mask */
} asz_pit_player;
/* starts a match on the current root games (encodes their planes; ASZ_STEP_KEYS when a stand-in plays) and synchronises;
 * *h_running (may be NULL) = games running.  ASZ_ERR_ARG: a network of another board side or device, alice_snakes outside
 * 0..S, stub_word not 0/1.  A new begin abandons a match in progress. */
int asz_pit_begin(asz_engine* e, const asz_pit_player* alice, const asz_pit_player* bob, int32_t alice_snakes, int32_t* h_running,
                  void* stream);
/* one turn; spawn_mode ASZ_SPAWN_NATIVE / ASZ_SPAWN_REPLAY (d_spawn_cells [G], entries below -1 read as -1) / ASZ_SPAWN_NONE;
 * d_moves [G*8] (may be NULL) receives the moves played this turn, 255 = no move; *h_running = games still running.  A turn
 * when no game is running does nothing.  ASZ_ERR_STATE without a begin. */
int asz_pit_turn(asz_engine* e, int32_t spawn_mode, const int32_t* d_spawn_cells, uint8_t* d_moves, int32_t* h_running,
                 void* stream);
/* ends the match: d_winners [G], d_decided_turn [G] (DEVICE, either may be NULL), *h_turns = turns played.  Synchronous.
 * Returns ASZ_ERR_STATE, after writing the results, when games are still running. */
int asz_pit_finish(asz_engine* e, int32_t* d_winners, int32_t* d_decided_turn, int32_t* h_turns, void* stream);
/* the whole match: begin, native spawn until every game is decided (max_turns 0) or max_turns turns are played, finish
 * (ASZ_ERR_STATE, only ever with the results so far written, when max_turns ends it with games running).  It abandons a
 * match in progress, and its own match is closed when it returns, whatever the outcome. */
int asz_pit_run(asz_engine* e, const asz_pit_player* alice, const asz_pit_player* bob, int32_t alice_snakes, int32_t max_turns,
                int32_t* d_winners, int32_t* d_decided_turn, int32_t* h_turns, void* stream);
/* counters of the current or last match: h_stats[4] = turns, rows valued by a network, rows valued by a stand-in player,
 * milliseconds of the network forwards (CUDA events around each turn's forwards) */
int asz_pit_stats(asz_engine* e, double* h_stats);

/* ---- pit with search agents: either side plays utils/agent.Agent (agent.py:25-111) with training=False --------------------
 * A searched side's turn: the match's running games are copied into the side's searcher engine (the others arrive finished,
 * so the search leaves them alone), one root-turn search runs on it with the side's network (asz_search_run_net) or, for a
 * stand-in side, the stub value function reading key word stub_word, and the side's snakes play the argmaxs of their root Q
 * (the searcher's root moves).  Every snake inside that search is modelled with the side's network; the other side's moves
 * from it are discarded.  The rest of the turn is the pit above.  asz_pit_begin clears both searchers' tables; across the
 * turns of a match a table ages and evicts as agent.py:30-31, 101-110.  A side without a searcher plays argmax as before.
 * A searcher's Q table overflow is ASZ_ERR_CAPACITY from asz_pit_turn after the turn is played (a row the search dropped
 * moves straight) and from asz_pit_run after the results so far are written. */
/* copies the packed root records (cells, snakes, meta) of src into dst on their device; a game with d_skip[g] != 0
 * (DEVICE [G], may be NULL) arrives with its finished flag set.  ASZ_ERR_ARG: board side, snake count, game count or
 * device differ, or dst == src. */
int asz_copy_root_games(asz_engine* dst, const asz_engine* src, const uint8_t* d_skip, void* stream);
/* attaches (searcher != NULL) or detaches the searcher of side 0 (Alice) or 1 (Bob) for e's next asz_pit_begin / asz_pit_run.
 * A searcher is an engine with search configured (max_depth / max_breadth / softmax_base of the side's Agent), training = 0, and
 * the board side, snake count, game count, device, health_dec and numpy1_mask of e; it must stay alive while attached.
 * asz_pit_begin refuses (ASZ_ERR_ARG) a searcher that does not match, e itself, and one searcher on both sides. */
int asz_pit_set_search(asz_engine* e, int32_t side, asz_engine* searcher);
/* counters of the current or last match: h_stats[2] = rows moved by a search, milliseconds of the searched sides' copies
 * and searches (host clock; each search ends in a host synchronisation) */
int asz_pit_search_stats(asz_engine* e, double* h_stats);

#ifdef __cplusplus
}
#endif
#endif /* ASZ_B200_H */
