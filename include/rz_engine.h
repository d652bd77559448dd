/*
 * rz_engine.h -- C ABI of librz_engine.so: the B200-native self-play hot path of reversi-alpha-zero.
 *
 * The reference (mokemokechicken/reversi-alpha-zero) has no FFI seam: its self-play path is Python
 * calling Python (SURVEY.md section 8(b)).  Each entry point below therefore names the reference
 * *Python* interface it replaces (path:line under /root/reference/src/reversi_zero/); the ctypes
 * binding a maintainer would add on the reference side is shown in INTEGRATION.md and is what
 * reversi-alpha-zero_b200/reversi_zero_b200/_cabi.py contains.
 *
 * Conventions
 *   - every function returns int: 0 (RZ_OK) or a negative RZ_E* code; rz_last_error() gives the
 *     thread-local message.  CUDA errors are captured and reported, never abort()ed.
 *   - plain pointers and sizes only; the caller owns every buffer it passes in.  `*_dev` functions
 *     take DEVICE pointers and a cudaStream_t (as void*, 0 = default stream) and are asynchronous;
 *     functions without the suffix take HOST pointers, stage through the library's own device
 *     buffers and return after the result is in the host buffer.
 *   - board encoding (lib/bitboard.py:11-17): uint64 bitboard, bit i = square y*8+x, bit 0 top-left.
 *   - Player: 1 = black, 2 = white (env/reversi_env.py:9); Winner: 0 = none, 1 = black, 2 = white,
 *     3 = draw (env/reversi_env.py:11).
 *   - handles are not thread-safe; one engine per GPU driven by one host thread (exception: rz_engine_poll, see there).
 */
#ifndef RZ_ENGINE_H
#define RZ_ENGINE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RZ_OK 0
#define RZ_EINVAL (-1)   /* bad argument */
#define RZ_ECUDA (-2)    /* CUDA runtime / launch error (message has the CUDA string) */
#define RZ_ENOMEM (-3)   /* host or device allocation failed */
#define RZ_ESTATE (-4)   /* call not valid in this state (e.g. weights not loaded) */
#define RZ_ECAPACITY (-5) /* an engine arena overflowed (nodes / edges / records) */
#define RZ_EIO (-6)      /* file I/O failed */

#define RZ_ABI_VERSION 3

int rz_abi_version(void);
const char* rz_last_error(void);
/* number of CUDA devices visible; RZ_ECUDA if the runtime cannot initialise. */
int rz_device_count(int* count);

/* ------------------------------------------------------------------------------------------------
 * K1 -- stateless batched bitboard operators (lib/bitboard.py, env/reversi_env.py).
 * ---------------------------------------------------------------------------------------------- */

/* legal-move mask per position.  Replaces lib/bitboard.py:53-67 find_correct_moves (+ :95-116). */
int rz_find_correct_moves_dev(const uint64_t* own, const uint64_t* enemy, uint64_t* out, size_t n, void* stream);
int rz_find_correct_moves(const uint64_t* own, const uint64_t* enemy, uint64_t* out, size_t n);

/* flipped-disc mask for a move at pos[i] (0..63); like the reference it does NOT check that pos is
 * empty or legal (returns 0 when nothing is outflanked).  Replaces lib/bitboard.py:70-92 calc_flip. */
int rz_calc_flip_dev(const uint8_t* pos, const uint64_t* own, const uint64_t* enemy, uint64_t* out, size_t n, void* stream);
int rz_calc_flip(const uint8_t* pos, const uint64_t* own, const uint64_t* enemy, uint64_t* out, size_t n);

/* one ReversiEnv.step per environment, structure-of-arrays, in place.  action[i] in 0..63, or -1 for
 * None (= resign).  Semantics of env/reversi_env.py:42-85: illegal move => mover loses; opponent
 * without a move => auto-pass; neither side can move => game over, winner by disc count.
 * legal_out (nullable) receives the legal-move mask of the side to move after the step (0 if done). */
int rz_step_dev(uint64_t* black, uint64_t* white, uint8_t* next_player, uint8_t* turn, uint8_t* done,
                uint8_t* winner, const int8_t* action, uint64_t* legal_out, size_t n, void* stream);
int rz_step(uint64_t* black, uint64_t* white, uint8_t* next_player, uint8_t* turn, uint8_t* done,
            uint8_t* winner, const int8_t* action, uint64_t* legal_out, size_t n);

/* board dihedral transform t in 0..7: flip_vertical if (t & 4), then (t & 3) x rotate90 -- the order
 * of agent/player.py:166-179 and :300-305.  Replaces lib/bitboard.py:119-159. */
int rz_dihedral_dev(const uint64_t* x, const uint8_t* t, uint64_t* out, size_t n, void* stream);

/* endgame solver (lib/alt/reversi_solver_cython.pyx:40-127 ReversiSolver.solve, the variant agent/player.py:15
 * imports), batched: for each position of the side to move, move[i] = best square and score[i] = its value in the
 * mover's frame.  exactly[i] != 0: exact final disc difference, first best move in ascending order; exactly[i] == 0:
 * win/loss/draw mode with the reference's early stop (only the sign of the score and the move are meaningful).
 * move[i] = -1 (score 0): no legal move, or more than 12 empty squares (the analogue of the reference's timeout,
 * after which ReversiPlayer falls back to the search). */
int rz_solve_dev(const uint64_t* own, const uint64_t* enemy, const uint8_t* exactly, int8_t* move, int8_t* score, size_t n,
                 void* stream);
int rz_solve(const uint64_t* own, const uint64_t* enemy, const uint8_t* exactly, int8_t* move, int8_t* score, size_t n);

/* Scalar host twins for the single-environment Python objects (ReversiEnv / Board used by the
 * reference's evaluate.py, nboard.py, game_model.py): same header-only code as the device kernels
 * (csrc/rz_bitboard.cuh), compiled for the host.  Not a fallback for the batched path. */
typedef struct rz_env_state {
    uint64_t black, white;
    uint8_t next_player, turn, done, winner;
} rz_env_state;
uint64_t rz_find_correct_moves_host(uint64_t own, uint64_t enemy);
uint64_t rz_calc_flip_host(int pos, uint64_t own, uint64_t enemy);
uint64_t rz_dihedral_host(uint64_t x, int t);
/* Host twin of the BIT-SLICED formulation the batched GPU operators use (csrc/rz_bitsliced.cuh: 32 positions per thread,
 * one register per square): pos == NULL: out[i] = find_correct_moves(own[i], enemy[i]); else out[i] = calc_flip(pos[i], ..).
 * Same header compiled for the host; exists so that the formulation can be held against the oracle without a GPU. */
int rz_bitsliced_host(const uint8_t* pos, const uint64_t* own, const uint64_t* enemy, uint64_t* out, size_t n);
void rz_env_reset_host(rz_env_state* s);                                              /* reversi_env.py:26-32 */
void rz_env_update_host(rz_env_state* s, uint64_t black, uint64_t white, int next_player); /* :34-40 */
void rz_env_step_host(rz_env_state* s, int action /* -1 = None */);                   /* :42-74 */

/* ------------------------------------------------------------------------------------------------
 * NN -- policy/value residual CNN inference (agent/model.py:28-72 forward, agent/api.py:30-45).
 * ---------------------------------------------------------------------------------------------- */
typedef struct rz_net rz_net;

typedef struct rz_net_cfg {
    int32_t filters;     /* ModelConfig.cnn_filter_num   (config.py:189) */
    int32_t res_blocks;  /* ModelConfig.res_layer_num    (config.py:191) */
    int32_t value_fc;    /* ModelConfig.value_fc_size    (config.py:193) */
    int32_t kernel_size; /* ModelConfig.cnn_filter_size  (config.py:190); only 3 is supported */
} rz_net_cfg;

#define RZ_NET_IMPL_AUTO 0    /* tcgen05 tower when filters == 256, else the generic kernel */
#define RZ_NET_IMPL_GENERIC 1 /* CUDA-core fp32 kernel, any configuration */
#define RZ_NET_IMPL_TCGEN05 2 /* fused persistent tcgen05 tower (filters must be 256) */

int rz_net_create(const rz_net_cfg* cfg, int device, rz_net** out);
int rz_net_destroy(rz_net* net);
/* number of float32 values in the weight blob for this configuration.  Blob layout (Keras tensor
 * layouts, in this order): for conv0, then res{i}.conv1, res{i}.conv2 (i = 0..res_blocks-1):
 *   kernel[kh][kw][Cin][Cout], bias[Cout], bn_gamma, bn_beta, bn_mean, bn_var [Cout];
 * policy_conv (1x1, Cout = 2) same six tensors; policy_fc kernel[128][64], bias[64];
 * value_conv (1x1, Cout = 1) same six; value_fc1 kernel[64][V], bias[V]; value_fc2 kernel[V][1], bias[1].
 * BatchNormalization epsilon = 1e-3 (Keras default), inference statistics. */
int rz_net_blob_size(const rz_net* net, size_t* n_floats);
int rz_net_load_weights(rz_net* net, const float* blob_host, size_t n_floats);
/* same, blob already in device memory (e.g. after an NCCL broadcast from rank 0). */
int rz_net_load_weights_dev(rz_net* net, const float* blob_dev, size_t n_floats, void* stream);

/* batched forward from bitboards: plane 0 = own (side to move), plane 1 = enemy.
 * policy[n][64] softmax probabilities, value[n] tanh.  Device pointers. */
int rz_net_predict_dev(rz_net* net, const uint64_t* own, const uint64_t* enemy, float* policy, float* value,
                       size_t n, int impl, void* stream);
/* diagnostic variant of the tcgen05 path: additionally writes the fp32 residual-tower output
 * tower[n][64 pixels][256 channels] (pixel = y*8+x) so tests can localise a numerical difference. */
int rz_net_debug_tower_dev(rz_net* net, const uint64_t* own, const uint64_t* enemy, float* policy, float* value,
                           float* tower, size_t n, void* stream);
/* same, plus the head outputs BEFORE softmax / tanh -- policy_logits[n][64] (the input of the policy_out softmax,
 * agent/model.py:47) and value_logit[n] (the input of the value_out tanh, :55) -- so that the north-star tolerance
 * ("policy/value logits within 1e-3") can be asserted on the logits themselves; tower may be NULL. */
int rz_net_debug_heads_dev(rz_net* net, const uint64_t* own, const uint64_t* enemy, float* policy, float* value,
                           float* tower, float* policy_logits, float* value_logit, size_t n, void* stream);
/* ReversiModelAPI.predict (agent/api.py:30-45): planes uint8 [n][2][8][8] with values {0,1}, host
 * buffers in, policy[n][64] / value[n] host buffers out. */
int rz_net_predict(rz_net* net, const uint8_t* planes, float* policy, float* value, size_t n, int impl);

/* ------------------------------------------------------------------------------------------------
 * Engine -- on-device MCTS self-play (agent/player.py ReversiPlayer, worker/self_play.py).
 * ---------------------------------------------------------------------------------------------- */
typedef struct rz_engine rz_engine;

#define RZ_EVAL_NET 0  /* leaves evaluated by the rz_net */
#define RZ_EVAL_FAKE 1 /* deterministic test evaluator: policy 1/64, value (#own - #enemy)/64 */

typedef struct rz_engine_cfg {
    int32_t games;                  /* concurrent game slots on this GPU */
    int32_t simulation_num_per_move; /* PlayConfig.simulation_num_per_move (config.py:129) */
    int32_t parallel_search_num;    /* :141, <= 16 */
    int32_t virtual_loss;           /* :139 */
    int32_t change_tau_turn;        /* :138 */
    int32_t thinking_loop;          /* :132 */
    int32_t required_visit_to_decide_action; /* :133 */
    int32_t start_rethinking_turn;  /* :134 */
    int32_t allowed_resign_turn;    /* :145 */
    int32_t use_resign_threshold;   /* 0 => resign_threshold is None (:144) */
    int32_t share_mtcs_info;        /* share_mtcs_info_in_self_play (:130) */
    int32_t eval_mode;              /* RZ_EVAL_* */
    int32_t net_impl;               /* RZ_NET_IMPL_* */
    int32_t max_plies;              /* per-game ply log capacity, 0 => 64 */
    int32_t warm_start;             /* 1: the FIRST game of every slot begins after a random number (0..57) of
                                       random legal plies, so a fresh engine is in steady state (game phases
                                       spread uniformly) instead of all slots marching in lock step; those
                                       pre-played plies are not searched and not recorded */
    int32_t overlap_groups;         /* 0 = auto (2 when games >= 256), 1, or 2: slot groups whose MCTS tick overlaps
                                       the other group's network launch on a second stream */
    int32_t max_sims_per_wave;      /* simulations one game may START in one wave (0 = 2 x parallel_search_num).  Bounds
                                       the work of a wave for games whose simulations end in terminal positions without
                                       needing the network (endgame), so no slot delays the whole batch. */
    int32_t use_solver_turn;        /* PlayConfig.use_solver_turn (config.py:154): from this turn on the move is the exact
                                       endgame solution (agent/player.py:100-103,150-161) and the ply is not training data;
                                       0 = off.  Positions the device solver refuses (> 12 empties) are searched instead. */
    int32_t use_solver_turn_in_simulation; /* :155, agent/player.py:237-251: WLD-solved nodes inside the search; 0 = off.
                                       Solves are resumable: each wave advances the unfinished ones for at most
                                       RZ_SOLVER_BUDGET_US microseconds (environment, read by rz_engine_create; default
                                       2000) and a game waits until its solves are done -- results do not depend on it. */
    int32_t reset_mtcs_info_per_game; /* PlayConfig.reset_mtcs_info_per_game (config.py:131; worker/self_play.py:111-134): a
                                       slot keeps its statistics for this many consecutive games (0 / 1: every game starts
                                       empty, ch5.yml; mini.yml uses 3).  Arenas grow by the same factor. */
    int32_t max_searches_per_game;  /* sizes the per-game node arena: nodes = this x simulation_num_per_move;
                                       0 = 60 x min(thinking_loop, 2).  Rethinking (thinking_loop > 1) is skipped
                                       when the arena could no longer hold one search per remaining ply. */
    int32_t arena_simulation_num;   /* the largest simulation count rz_engine_set_simulation_num will be asked for during this
                                       engine's life (the maximum over schedule_of_simulation_num_per_move and .force-sim,
                                       worker/self_play.py:262-272); the arenas are sized for it.  0 = simulation_num_per_move. */
    float c_puct;                   /* :135 */
    float noise_eps;                /* :136 */
    float dirichlet_alpha;          /* :137 */
    float resign_threshold;         /* :144 */
    float disable_resignation_rate; /* :146 */
    uint64_t seed;                  /* Philox key */
    uint64_t first_game_id;         /* ids handed to slots: first_game_id + k * game_id_stride */
    uint64_t game_id_stride;        /* (rank-strided sharding across GPUs, SURVEY 8(e)) */
    uint64_t max_games;             /* stop starting new games after this many (0 = unlimited) */
} rz_engine_cfg;

/* one decided ply of a finished game (compact form of what ReversiPlayer.moves holds,
 * agent/player.py:166-179; the 8 symmetries are expanded by rz_write_play_data). */
typedef struct rz_ply {
    uint64_t own, enemy;  /* position in the mover's frame */
    int32_t n_visit[64];  /* root visit counts N(s,a) at decision time */
    int16_t action;       /* 0..63, -1 = resigned */
    uint8_t player;       /* 1 black / 2 white */
    uint8_t loops;        /* thinking loops used */
    uint8_t recorded;     /* 1 if this ply is training data (0 for a resignation) */
    uint8_t pad;
    uint16_t waves;       /* engine waves this slot spent deciding the ply (saturating; measurement only, no reference twin) */
    float n;              /* ActionWithEvaluation.n */
    float q;              /* ActionWithEvaluation.q */
} rz_ply;

typedef struct rz_game {
    uint64_t game_id;
    uint64_t black, white;  /* final position */
    int32_t first_ply;      /* index into the ply array returned by the same poll */
    int32_t n_plies;
    int32_t expansions;     /* NN evaluations spent on this game */
    int32_t simulations;
    uint8_t winner;         /* Winner enum */
    int8_t black_z;         /* +1 / -1 / 0 */
    uint8_t resign_enabled;
    uint8_t resigned_mask;  /* bit0 black wanted to resign, bit1 white */
    uint8_t turn;           /* ReversiEnv.turn at the end */
    uint8_t black_net;      /* evaluation matches: 0 = black was played by the first network, 1 = by the second */
    uint8_t pad[2];
    int32_t table_nodes;    /* positions in the slot's statistics table at the end of the game (half of the reference's
                               len(mtcs_info.var_p), which also holds every colour-swapped mirror key, worker/self_play.py:127) */
    int32_t pad2;
} rz_game;

typedef struct rz_stats {
    uint64_t games_started, games_finished;
    uint64_t expansions;    /* leaves evaluated == "node expansions" */
    uint64_t simulations;
    uint64_t waves;
    uint64_t plies;
    uint64_t nn_launches, mcts_launches; /* kernels launched by the engine */
    uint64_t max_nodes_used, max_edges_used;
    double nn_ms, mcts_ms; /* device time (CUDA events on the engine's stream) spent in the two kernel families */
    double run_ms;         /* device time from the first to the last wave of each rz_engine_run call, accumulated */
} rz_stats;

int rz_engine_create(const rz_engine_cfg* cfg, rz_net* net /* may be NULL for RZ_EVAL_FAKE */, int device,
                     rz_engine** out);
int rz_engine_destroy(rz_engine* e);
/* run waves until at least `finished_target` games (cumulative) have finished or `max_waves` waves
 * were executed (0 = no limit).  Finished games accumulate in a host-side queue until polled.
 * rz_engine_poll (and only it) may be called from a second host thread while rz_engine_run is in progress: the queue is
 * a mutex-protected single-producer / single-consumer hand-off, which is how the worker's writer thread overlaps
 * harvesting and play_data output with the waves (the reference overlaps through processes, worker/self_play.py:36-41). */
int rz_engine_run(rz_engine* e, uint64_t finished_target, uint64_t max_waves);
/* pop up to game_cap finished games (and their plies, up to ply_cap) from the queue. */
int rz_engine_poll(rz_engine* e, rz_game* games, size_t game_cap, size_t* n_games, rz_ply* plies, size_t ply_cap,
                   size_t* n_plies);
int rz_engine_stats(rz_engine* e, rz_stats* out);
/* no slot starts a game whose local index (slot + games already started by the slot x games) is >= max_games; 0 = no
 * limit, 1 = let the resident games finish and start nothing (rz_engine_run then returns when every slot is idle). */
int rz_engine_set_max_games(rz_engine* e, uint64_t max_games);
/* warm_start only: weight[t] (t = 0 .. n-1, n <= 60) is proportional to the time a game spends at turn t; the first
 * game of every slot then begins at turn t with probability weight[t] / sum and its first search runs a uniformly drawn
 * fraction of simulation_num_per_move (of the waves the profile gives the turn, where that is less), i.e. the slots start in the stationary state of an engine that has been running
 * for a long time (used by bench.py, which measures finished games per second over a window shorter than a game).
 * Without this call the turns 0..57 are equally likely.  Call before the first rz_engine_run. */
int rz_engine_set_warm_start_profile(rz_engine* e, const float* weight, int n);
/* change the per-move simulation count for games started from now on
 * (SelfPlayWorker.decide_simulation_num_per_move, worker/self_play.py:262-272). */
int rz_engine_set_simulation_num(rz_engine* e, int32_t sims);
/* evaluation matches (worker/evaluate.py:44-96: best model vs challenger): with a second network set, the game with
 * local index i is played by the first network as black when i is even and by the second when i is odd (the
 * reference draws the colours at random, :70), and every search is evaluated by the mover's own network.  Use
 * share_mtcs_info = 0 (the reference gives each evaluation player its own statistics).  RZ_EVAL_FAKE: the "second
 * network" is the deterministic evaluator with the value negated.  NULL switches back to one network.  Call before
 * the first rz_engine_run. */
int rz_engine_set_second_net(rz_engine* e, rz_net* net_b, int enable);
/* update the resignation rule for decisions taken from now on (SelfPlayWorker's threshold auto-tuner,
 * worker/self_play.py:250-260). */
int rz_engine_set_resign_threshold(rz_engine* e, int use_resign_threshold, float resign_threshold);
/* single-position search (ReversiPlayer.action outside the self-play loop: evaluate.py, nboard.py, GUI; also the
 * parity-test hook): every slot searches (own, enemy) with `player` to move for simulation_num_per_move
 * simulations; returns the root statistics of slot `slot`: n_visit[64], w_sum[64] (mover's frame).
 * keep_tree != 0 keeps the slot's transposition table from earlier calls (the reference's MCTSInfo that
 * persists across the moves of a game, agent/player.py:44-47); 0 starts from an empty table. */
int rz_engine_search_root(rz_engine* e, uint64_t own, uint64_t enemy, int player, int slot, int keep_tree,
                          int32_t* n_visit, float* w_sum);

/* ------------------------------------------------------------------------------------------------
 * play_data writer -- the reference's output contract (worker/self_play.py:180-194,
 * lib/data_helper.py:23-25): one JSON array of [[own, enemy], [p0..p63], z] records, all of black's
 * records of a game then all of white's, each recorded ply expanded to its 8 symmetries in the order
 * of agent/player.py:166-179.  Written to path + ".tmp" and renamed.  save_policy_of_tau_1 /
 * change_tau_turn select the stored policy exactly as agent/player.py:132,366-385.
 * ---------------------------------------------------------------------------------------------- */
int rz_write_play_data(const char* path, const rz_game* games, size_t n_games, const rz_ply* plies,
                       int save_policy_of_tau_1, int change_tau_turn, size_t* n_records);

/* ------------------------------------------------------------------------------------------------
 * Trainer-side ingest (SURVEY 8(f).4) -- replaces the pure-Python per-record loop of
 * OptimizeWorker.convert_to_training_data (worker/optimize.py:215-231) applied to
 * read_game_data_from_file (lib/data_helper.py:28-30).
 *
 * A "play row" is one recorded ply before the 8-symmetry expansion: 280 bytes instead of ~5 KB of JSON text.
 * rz_write_play_rows writes the rows of the same games, in the same order, as rz_write_play_data writes records
 * (file: 32-byte header {"RZROWS\0\1", int32 save_policy_of_tau_1, int32 change_tau_turn, uint64 n_rows, 8 bytes 0}
 * + n_rows rows).  rz_ingest[_dev] expands rows into the arrays the reference trainer builds from the JSON file:
 *   planes [8*n_rows][2][8][8] uint8   == np.array(state_list)   (bit_to_array, lib/bitboard.py:136-138)
 *   policy [8*n_rows][64]      float32 == np.array(policy_list) rounded to the float32 Keras feeds the model
 *   z      [8*n_rows]          float32 == np.array(z_list)
 * row r, symmetry t (t = flip*4 + rot, agent/player.py:166-179) -> output record 8*r + t.
 * ---------------------------------------------------------------------------------------------- */
typedef struct rz_play_row {
    uint64_t own, enemy;  /* position in the mover's frame */
    int32_t n_visit[64];  /* root visit counts at decision time */
    int32_t z;            /* game result from the mover's point of view: +1 / 0 / -1 */
    int32_t pad;
} rz_play_row;

int rz_write_play_rows(const char* path, const rz_game* games, size_t n_games, const rz_ply* plies,
                       int save_policy_of_tau_1, int change_tau_turn, size_t* n_rows);
/* rows == NULL: only report n_rows and the two policy settings stored in the header */
int rz_read_play_rows(const char* path, rz_play_row* rows, size_t capacity, size_t* n_rows,
                      int* save_policy_of_tau_1, int* change_tau_turn);
int rz_ingest_dev(const rz_play_row* rows, size_t n_rows, int save_policy_of_tau_1, int change_tau_turn,
                  uint8_t* planes, float* policy, float* z, void* stream);   /* device pointers */
int rz_ingest(const rz_play_row* rows, size_t n_rows, int save_policy_of_tau_1, int change_tau_turn,
              uint8_t* planes, float* policy, float* z);                       /* host pointers */

#ifdef __cplusplus
}
#endif
#endif /* RZ_ENGINE_H */
