/* caro_b200.h -- C ABI of the B200-native MCTS self-play engine (libcaro_b200.so).
 *
 * Drop-in boundary for the hot path of nh273/caro-ai (SURVEY.md section 8).  The reference has no
 * FFI layer of its own -- its seam is the Python API of lib/mcts.py, lib/game/ and lib/model.py --
 * so every entry point below names the reference function(s) whose work it replaces
 * (paths relative to the reference tree) and INTEGRATION.md shows the ctypes stub a maintainer of
 * the reference would add at each of those call sites.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only; no torch / C++ types cross this boundary.
 *   - `d_` parameters are DEVICE pointers (sm_100a, same device as the engine's workspace);
 *     `h_` parameters are HOST pointers.  `stream` is a cudaStream_t passed as void* (NULL =
 *     default stream).  All launches are asynchronous on `stream` unless stated otherwise.
 *   - every function returns 0 on success, a negative CARO_E_* code otherwise;
 *     caro_last_error() gives the message for the calling thread.  There is NO CPU fallback:
 *     without a CUDA device the compute entry points fail with CARO_E_CUDA.
 *   - an engine handle is not thread-safe; distinct handles are independent.
 *
 * Board encodings (device side; the reference's state integers are converted on the host by
 * caro_ai_b200.game, see DESIGN.md section 4):
 *   Connect4 : caro_c4_board  {mask, black}, bit = 7*col + row (row 0 = bottom, bit 6 of each
 *              column is an always-empty sentinel).
 *   m,n,k    : caro_mnk_board {w[4], b[4]}, bit = row*n + col (= the action index), n <= 15.
 *   Caro     : the m,n,k board, (n, k) bounds, actions, planes and draw rule; only the win test
 *              differs.  A move wins iff in at least one of the four directions the maximal run
 *              of the mover's stones through the new cell is >= k (overlines count) AND that run
 *              is not blocked at both ends, an end being blocked when the cell just past it is on
 *              the board and holds an opponent stone.  The board edge never blocks.  A blocked run
 *              stays on the board and the game goes on.
 */
#ifndef CARO_B200_H_
#define CARO_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CARO_ABI_VERSION 2

enum { CARO_OK = 0, CARO_E_ARG = -1, CARO_E_CUDA = -2, CARO_E_STATE = -3, CARO_E_CAPACITY = -4 };

enum { CARO_GAME_CONNECT4 = 0, CARO_GAME_MNK = 1, CARO_GAME_CARO = 2 };

typedef struct { uint64_t mask, black; } caro_c4_board;
typedef struct { uint64_t w[4], b[4]; } caro_mnk_board;

int caro_abi_version(void);
const char* caro_last_error(void);
/* Number of CUDA devices visible to the library (0 when there is none; never throws). */
int caro_device_count(void);

/* ------------------------------------------------------------------------------------------
 * Stand-alone board kernels -- rows a11..a16 of SURVEY.md section 8.
 * `d_boards` is an array of `count` caro_c4_board (game = CONNECT4) or caro_mnk_board (MNK, CARO).
 * ------------------------------------------------------------------------------------------ */

/* game.move for a batch: lib/game/connect_four/connect_four.py:241-265 (+ _check_won :206-239),
 * lib/game/tictactoe/tictactoe.py:210-235 (+ tictactoe_helpers.check_win :7-56).
 * d_won[i] = 1 if the move wins, d_draw[i] = 1 if it does not win and leaves no legal move
 * (lib/utils.py:92-96, lib/mcts.py:145-146).  In-place is allowed (d_out == d_boards). */
int caro_boards_apply(int game, int n, int k, const void* d_boards, const int32_t* d_actions,
                      const uint8_t* d_players, int64_t count, void* d_out, uint8_t* d_won,
                      uint8_t* d_draw, void* stream);

/* game.possible_moves / invalid_moves as a bitmask per board (bit a set = action a legal):
 * connect_four.py:157-173, tictactoe.py:137-162.  d_mask is [count][mask_words] uint32,
 * mask_words = (A + 31) / 32. */
int caro_boards_legal_mask(int game, int n, int k, const void* d_boards, int64_t count,
                           uint32_t* d_mask, void* stream);

/* game.states_to_training_batch: connect_four.py:175-204, tictactoe.py:164-208.
 * d_planes is float32 [count][2][H][W], plane 0 = tokens of d_who[i], row 0 = top. */
int caro_boards_encode_planes(int game, int n, int k, const void* d_boards, const uint8_t* d_who,
                              int64_t count, float* d_planes, void* stream);

/* MCTS._backup (lib/mcts.py:225-246) along one path on caller-owned flat arrays: for i = depth-1 .. 0,
 * N[e_i] += 1; W[e_i] += v; Q[e_i] = W/N; v = -v, starting from v = -value (float32 arithmetic).
 * d_edge_index[i] = flat index of (state_i, action_i).  Used by the dict-view facade (lib/test_mcts.py:15-38). */
int caro_backup_path(int32_t* d_n, float* d_w, float* d_q, const int64_t* d_edge_index, int depth,
                     float value, void* stream);

/* ------------------------------------------------------------------------------------------
 * Policy/value network -- row a17 (lib/model.py:10-94) + the softmax of lib/mcts.py:216.
 * Weights are handed over ALREADY FOLDED (eval-mode BatchNorm merged into the convolutions,
 * done on the host by caro_ai_b200.model.fold_state_dict) as one float32 blob:
 *   conv_in  w[F][2][3][3] b[F] | blocks x ( w[F][F][3][3] b[F] ) |      (blocks = 5, F = 64 in the reference)
 *   conv_val w[F] b[1] | value.0 w[20][HW] b[20] | value.2 w[20] b[1] |
 *   conv_policy w[2][F] b[2] | policy.0 w[A][2*HW] b[A]
 * F (the filters of every convolution) is 64 or 128.
 * ------------------------------------------------------------------------------------------ */
typedef struct caro_net caro_net;

size_t caro_net_blob_floats(int rows, int cols, int actions);
/* The same for a tower of `blocks` residual blocks (1..20; the reference has 5, lib/model.py:21-45): the blob then holds
 * `blocks` x ( w[64][64][3][3] b[64] ) groups, and caro_net_create reads the depth off the blob's length.  The width is
 * 64 filters.  Returns 0 for an unsupported depth. */
size_t caro_net_blob_floats_deep(int rows, int cols, int actions, int blocks);
/* The same for any supported shape: `blocks` 1..20 residual blocks of `filters` = 64 or 128 filters.  Returns 0 for an
 * unsupported depth or width; with filters = 64 it equals caro_net_blob_floats_deep. */
size_t caro_net_blob_floats_shape(int rows, int cols, int actions, int blocks, int filters);
/* Copies and re-packs the blob into device memory owned by the handle (bf16 UMMA operand images
 * for the tensor-core tower + fp32 copies for the heads).  Synchronous.  The width is 64 filters. */
int caro_net_create(int rows, int cols, int actions, const float* h_blob, size_t n_floats,
                    caro_net** out);
/* caro_net_create for a stated shape (`blocks` 1..20, `filters` 64 or 128).  Every argument, the blob's size included, is
 * checked before the device is looked for: a bad shape returns CARO_E_ARG on any machine.  A 128-filter handle runs
 * impl 7 (wide tower, fp16 operands), 0 / 3 (wide tower, bf16 operands), 8 (wide tower, bf16 hi + lo split precision)
 * and 1 (SIMT); see caro_net_forward. */
int caro_net_create_shape(int rows, int cols, int actions, int blocks, int filters, const float* h_blob, size_t n_floats,
                          caro_net** out);
int caro_net_update(caro_net* net, const float* h_blob, size_t n_floats);
void caro_net_destroy(caro_net* net);
/* Debug only: d_trace = device buffer of >= 8001 int64 (zeroed) that CTA 0 of the tensor-core kernels (net_tc.cu, net_wide.cu) fills with
 * (tag, clock64) pairs -- the pipeline timeline used to tune the kernel; NULL switches tracing off. */
int caro_net_set_trace(caro_net* net, void* d_trace);

/* The tensor-core tower is a persistent kernel with one CTA per SM that owns the SM's whole shared memory.
 * Limiting it to `ctas` SMs (0 = all) leaves the remaining SMs to the tree kernels of the other half-batch, which
 * the self-play pipeline runs on side streams underneath the network pass (caro_engine_play_multi). */
int caro_net_set_grid_limit(caro_net* net, int ctas);

/* Forward pass over a compact batch of leaf positions given as boards + side to move.
 *   d_count : device int32 holding the number of valid leaves (<= max_count); read on device, so
 *             no host synchronisation is needed between search steps.  May be NULL, then
 *             max_count leaves are evaluated.
 *   d_probs : float32 [max_count][A] softmax priors (over ALL actions, like the reference).
 *   d_values: float32 [max_count]    tanh value head.
 *   impl    : 0 = tcgen05 bf16 tensor-core tower (product path: one bf16 pass, fp32 accumulate); boards up to
 *                 6 x 7 run the row-tiled kernel (net_rt.cu), larger ones the tap-per-MMA kernel (net_tc.cu),
 *             3 = tcgen05 bf16 tower, tap-per-MMA kernel for every board size (A/B comparisons),
 *             2 = split-precision tcgen05 tower (hi / lo pairs of activations and weights, 3 MMAs per product:
 *                 fp32-class accuracy for trained checkpoints with large logits).  Boards up to 6 x 7 run the
 *                 row-tiled fp16 hi + lo kernel (net_rx.cu, ~2.3x the one-pass time), larger ones the
 *                 tap-per-MMA bf16 hi + lo kernel (net_tc.cu, ~3.5x),
 *             4 = the tap-per-MMA split-precision kernel for every board size (A/B comparisons),
 *             5 = the row-tiled bf16 tower as CTA pairs (tcgen05 cta_group::2: clusters of two CTAs, each fetching half of
 *                 every B operand; bit-identical to impl 0, boards up to 6 x 7 only; measured slower than impl 0, kept for
 *                 A/B runs -- CARO_RT_PAIR=1 in the environment makes impl 0 use it),
 *             7 = one-pass FP16 row-tiled tower (boards up to 6 x 7): activations and weights fp16, fp32 accumulate -- the same
 *                 tcgen05 kind::f16 rate as bf16 with 11 instead of 8 mantissa bits on both operands, and the fp16 activations ARE
 *                 the residual stream (no e5m2 tail): 3.7e-5 / 8.1e-5 off fp32 on random-init Connect4 networks (impl 0: 1.1e-4 /
 *                 5.0e-4) and 8 % faster.  fp16's range is the caller's to check: the host mirror's precision="auto" measures
 *                 impl 7, then impl 0 against impl 1 on the device after every weight upload and falls back to impl 2,
 *             6 = the tap-per-MMA bf16 tower as CTA pairs (each CTA stores 32 of the 64 output channels of every tap; bit-identical
 *                 to impl 3; no faster stand-alone -- an M = 128, K = 16 MMA takes 48 cycles whatever N <= 64 is --, +1.5 % inside the
 *                 Caro self-play step; CARO_TC_PAIR=1 makes impl 0 / 3 use it),
 *             1 = fp32 SIMT tower (numerics reference kernel used by the tests).
 *           128-filter handles (caro_net_create_shape): 7 = the wide tap-per-MMA tower (net_wide.cu: M = 128, N = 128, K = 16
 *           MMAs, weights streamed tap by tap) with fp16 operands, 0 and 3 = the same tower with bf16 operands, 8 = the same
 *           tower in split precision (bf16 hi + lo activations and weights, hi*hi + lo*hi + hi*lo per product, fp32
 *           residual stream: fp32-class accuracy for trained wide networks), 1 = the SIMT tower; 2, 4, 5 and 6 return
 *           CARO_E_ARG.  Impl 8 runs on 128-filter handles only: a 64-filter handle returns CARO_E_ARG (its split tower is 2). */
int caro_net_forward(caro_net* net, int game, int n, int k, const void* d_boards,
                     const uint8_t* d_who, const int32_t* d_count, int64_t max_count,
                     float* d_probs, float* d_values, int impl, void* stream);

/* ------------------------------------------------------------------------------------------
 * Self-play / search engine -- rows a1..a10, a18, a19.
 * G games advance in lock-step; every game owns `trees_per_game` private arenas
 * (1 = one tree shared by both sides, train.py:185; 2 = one tree per side, lib/utils.py:58-59).
 * ------------------------------------------------------------------------------------------ */
typedef struct caro_engine caro_engine;

typedef struct {
  int32_t game;            /* CARO_GAME_* */
  int32_t n, k;            /* m,n,k and Caro only */
  int32_t games;           /* G */
  int32_t trees_per_game;  /* 1 or 2 */
  int32_t max_batch;       /* largest batch_size (descents per minibatch) that will be used, 1..32 */
  int32_t node_capacity;   /* nodes per tree arena */
  int32_t replay_capacity; /* entries in the device replay ring (0 = no replay recording) */
  double c_puct;           /* config.py:26 */
  double alpha;            /* config.py:27 */
  double explore;          /* config.py:28 */
  uint64_t seed;           /* Philox key */
  uint32_t flags;          /* CARO_FLAG_*: throughput-mode extensions that are NOT in the reference (SURVEY.md section 8f-4);
                              0 = reference behaviour (bit-exact trees) */
  uint32_t reserved;
} caro_engine_config;

/* Extensions, all off by default.  With any of them set the search is no longer the reference's (lib/mcts.py:248-287);
 * virtual loss, masked priors and the fresh and recycled trees are checked bit for bit against their restatement in the test
 * oracle (tests/test_gpu_search_matrix.py, tests/test_gpu_flag_matrix.py), and their effect on play statistically
 * (tests/test_gpu_round2.py).
 *   VIRTUAL_LOSS   the batch_size descents of a minibatch are made one after the other per game, and every edge an
 *                  earlier descent of the same minibatch went through counts as one extra visit that lost
 *                  (N + 1, W - 1 in the PUCT score; the tree itself is not modified, so the back-up is unchanged): the
 *                  descents spread out instead of piling onto the same leaf (lib/mcts.py:273-278 drops ~70 % of them).
 *   MASK_PRIORS    the network's priors are zeroed on illegal moves and renormalised when a node is created
 *                  (the reference keeps the raw softmax and masks only the PUCT score, lib/mcts.py:86-95).
 *   FRESH_TREE     a game's tree is cleared after each of its moves instead of being kept for the whole game
 *                  (lib/utils.py:58-59 keeps it): arena demand is bounded by the searches of ONE move, which is what
 *                  long 15 x 15 games at 1,600 descents per move need.
 *   RECYCLE_TREE   the tree is kept from move to move until it fills more than half of its arena and is cleared then: no
 *                  overflow while one move's searches fit half an arena, and most moves still reuse the previous subtree
 *                  (a cruder stand-in for COMPACT_TREE).
 *   COMPACT_TREE   after every move the nodes whose position can no longer occur (it does not contain the new root position:
 *                  tokens are only ever added) are dropped and the survivors moved to the front of the arena.  NOT a change of
 *                  the search: a dropped state can never be looked up again, so every N / W / Q / P that can still be reached,
 *                  and with it every later search, policy and move, is bit-identical to the reference's keep-everything tree
 *                  (lib/mcts.py:29-46).  The arena then holds the last few moves' searches instead of the whole game's: what
 *                  whole 15 x 15 games at 1,600 descents per move need.  node_capacity must fit a shared-memory index map
 *                  (<= ~45,000 nodes). */
enum { CARO_FLAG_VIRTUAL_LOSS = 1, CARO_FLAG_MASK_PRIORS = 2, CARO_FLAG_FRESH_TREE = 4, CARO_FLAG_RECYCLE_TREE = 8,
       CARO_FLAG_COMPACT_TREE = 16 };

/* Resignation (extension, off by default; the reference plays every game to its end).  Not a flag: it is switched and
 * tuned at run time by caro_engine_set_resign, whose parameters live in device memory (region "resign_params"), so a
 * ply graph captured by caro_engine_play_multi reads the current values on every replay.
 *   The rule, decided in caro_engine_advance from the root row of the mover's tree: with total = sum N[a] > 0,
 *     v_root = (sum over a, in action order, of (double)W[a]) / total          (double adds, one double division)
 *     v_best = (double)f32(W[best] / N[best]), best = the most visited action (lowest index on ties)
 *     stat   = max(v_root, v_best)                                              (mover's point of view)
 *   A game that is not a playthrough game resigns when stat < threshold: its history entry for the ply is written, the
 *   ply is counted, no move is played (d_action_out = -1) and the game ends lost for the mover (result, win counters and
 *   replay z as for any finished game; auto_restart re-seats the slot).  total == 0: no statistic, no resignation.
 *   A game is a playthrough game when, at its start (caro_engine_reset, or an auto-restart), resignation is enabled and
 *   u01d(Philox(uid, 0, 0; seed ^ 'RESG')) < playthrough.  It never resigns; it keeps each player's smallest stat
 *   (+inf until that player has one) and, when it ends, appends one record to the log ring.
 *   threshold = -1.0 never fires (stat >= -1 exactly): "log only".
 *   A false positive at threshold t is a logged game in which some player with min_stat < t did not lose (won or drew).
 * Regions: "resign_params" {int32 enabled, int32 pad, double threshold, double playthrough},
 *          "resign_playthrough" uint8 [G] (1 = the current game is a playthrough game),
 *          "resign_min" double [G][2] (the current playthrough game's minima per player),
 *          "resign_log" [G] records of 24 bytes {double min_stat[2]; int32 result (player 0's view); int32 plies},
 *                       record k in slot k % G,
 *          "resign_counters" uint64 [2]: [0] games resigned, [1] playthrough games logged (= the log cursor).
 * They follow every other region, so no other offset depends on them. */

/* Bytes of device workspace the engine needs; the caller allocates it (e.g. a torch uint8 CUDA
 * tensor) and keeps it alive for the life of the handle. */
size_t caro_engine_workspace_bytes(const caro_engine_config* cfg);
int caro_engine_create(const caro_engine_config* cfg, void* d_workspace, size_t bytes,
                       caro_engine** out, void* stream);
void caro_engine_destroy(caro_engine* e);

/* Offset/size of a named region of the workspace (for zero-copy views from the host language):
 * "nodes" (int32 [nodes][4][Apad]: one record per node with rows N | W | P | cached child link; bits 0-28 of an N word =
 * the visit count, bits 29-30 = the solver's proof of the edge, bit 31 = "W has absorbed a float32 network value"; Q =
 * f32(W / N) is not stored), "node_board","node_count","root_board",
 * "root_player","status","ply",
 * "result","leaf_board","leaf_player","leaf_count",
 * "desc" (one record per descent of the current minibatch, [G][max_batch]: bytes 0 kind, 1 side to move at the leaf,
 * 2-3 path length, 4-7 compact leaf slot (-1 = none), 8-11 terminal value (float), 16-31 transposition key, 32.. the leaf
 * board; 64 bytes for Connect4, 96 for m,n,k), "desc_path" (uint32 [G][max_batch][max plies]: (node << 8) | action from
 * the root down), "queue_len", "queue" (8-byte back-up queue entries {descent u8, kind u8, path length u16, leaf slot or
 * float bits of a terminal value i32} in the order of lib/mcts.py:269-278), "counters","replay_board","replay_player",
 * "replay_pi","replay_z","replay_cursor".
 * elem_bytes receives the element size, dims[0..3] the logical shape (unused dims = 0). */
int caro_engine_region(const caro_engine* e, const char* name, size_t* offset, size_t* bytes,
                       int32_t* elem_bytes, int64_t dims[4]);

/* MCTS.clear (lib/mcts.py:39-43) for the trees of the games selected by h_game_mask (NULL = all),
 * and re-seating of the games at the initial position.  first_player: 0/1 fixed, -1 = random per
 * game (lib/utils.py:66). */
int caro_engine_reset(caro_engine* e, const uint8_t* h_game_mask, int first_player, void* stream);
/* Sets root positions explicitly (host buffers; one H2D copy): the `state_int, player` arguments
 * of MCTS.search_batch (lib/mcts.py:162-163).  Trees are kept. */
int caro_engine_set_roots(caro_engine* e, const void* h_boards, const uint8_t* h_players,
                          void* stream);

/* One minibatch of descents, split so that a caller can supply the network outputs itself:
 *   select : lib/mcts.py:97-148 find_leaf x batch_size on the frozen tree, incl. _add_noise
 *            (:48-62), _calculate_upper_bound (:64-84), _mask_invalid_actions (:86-95).
 *            d_noise = NULL -> Philox Dirichlet; else float64 [G][batch][A] injected noise.
 *            d_noise_out (optional) receives the noise actually used, same shape.
 *   plan   : lib/mcts.py:265-278 terminal / expand split + duplicate-leaf drop, and the gather of
 *            the unique leaves into the compact batch (region "leaf_board"/"leaf_player"/"leaf_count").
 *   expand_backup : lib/mcts.py:178-190,219-223 _create_node and :225-246 _backup in queue order.
 *            d_probs float32 [leaf_count][A], d_values float32 [leaf_count]. */
int caro_engine_select(caro_engine* e, int batch, int minibatch_index, const double* d_noise,
                       double* d_noise_out, void* stream);
int caro_engine_plan(caro_engine* e, int batch, void* stream);
int caro_engine_expand_backup(caro_engine* e, int batch, const float* d_probs,
                              const float* d_values, void* stream);

/* MCTS.search_batch (lib/mcts.py:162-176) with the built-in network: `count` x
 * (select, plan, net forward, expand_backup), no host synchronisation inside.  The minibatches are
 * numbered first_minibatch .. first_minibatch + count - 1 for the Philox noise address (the reference draws
 * fresh Dirichlet noise for every descent, lib/mcts.py:131-132: a caller that searches the same game, ply and
 * side repeatedly passes a running index so that no noise vector is replayed). */
int caro_engine_search(caro_engine* e, caro_net* net, int count, int batch, int first_minibatch,
                       int net_impl, void* stream);

/* MCTS.get_policy_value (lib/mcts.py:289-313) for every game's root:
 * d_pi float64 [G][A], d_q float32 [G][A], d_n int32 [G][A].  tau_mode: 0 -> tau = 0, 1 -> tau = 1,
 * 2 -> per game, tau = 1 while ply < tau_plies else 0 (lib/utils.py:68,97-99). */
int caro_engine_root_policy(caro_engine* e, int tau_mode, int tau_plies, double* d_pi, float* d_q,
                            int32_t* d_n, void* stream);

/* One ply of lib/utils.py:76-99 play_game for every active game: policy(tau) -> np.random.choice
 * (d_uniform float64 [G] injected, or NULL -> Philox) -> game.move -> win / draw bookkeeping ->
 * history; finished games are written to the replay ring with alternating z (:101-106) and, if
 * auto_restart != 0, re-seated with a cleared tree (first player random, or fixed if >= 0).
 * d_action_out (optional) int32 [G] receives the sampled actions (-1 for inactive games). */
int caro_engine_advance(caro_engine* e, int tau_plies, const double* d_uniform, int auto_restart,
                        int first_player, int32_t* d_action_out, void* stream);

/* Convenience: `moves` x (search, advance) enqueued back to back. */
int caro_engine_play(caro_engine* e, caro_net* net_p0, caro_net* net_p1, int moves, int count,
                     int batch, int tau_plies, int auto_restart, int first_player, int net_impl,
                     void* stream);

/* The same plies for n = 1..8 engines (parts of the game batch) as a software pipeline: every part's kernels run
 * on a private side stream, chained by CUDA events -- one part's tree kernels (noise / select / plan, expand+backup,
 * advance) execute underneath the other parts' network passes.  Self-play only (one network).  `stream` is joined
 * with the side streams before returning. General form: n = 1..8 parts in round robin.  With three parts the tree kernels of one part have two network
 * passes to hide under (they run 3-5x slower next to the persistent network kernel than alone).  While profiling
 * is off, one ply (n x count x 5 kernels + n) is captured into a CUDA graph once and replayed per ply. */
int caro_engine_play_multi(caro_engine** engines, int n, caro_net* net, int moves, int count, int batch,
                           int tau_plies, int auto_restart, int first_player, int net_impl, void* stream);

/* train.py:85-94 (`random.sample(replay_buffer, BATCH_SIZE)` -> states_to_training_batch / probs / values tensors) on the
 * device: `d_entries` int64 [count] are absolute entry numbers of the replay ring (entry k lives in slot k % replay_capacity;
 * valid numbers are [cursor - min(cursor, capacity), cursor), "replay_cursor" region); the rows are written as
 * d_planes float32 [count][2][H][W] (from the stored side to move's point of view), d_pi float32 [count][A] and
 * d_z float32 [count] (lib/utils.py:101-106) without a host round trip.
 * d_symmetry (extension, NULL = off; the reference has no augmentation): int32 [count], sample i is written through the
 * board symmetry d_symmetry[i] -- bit 0 mirrors the columns (Connect4: 0..1), bit 1 the rows, bit 2 transposes (square
 * m,n,k boards: 0..7); planes and policy target are transformed together. */
int caro_engine_replay_gather(caro_engine* e, const int64_t* d_entries, const int32_t* d_symmetry, int64_t count,
                              float* d_planes, float* d_pi, float* d_z, void* stream);

/* Optional per-phase timing of caro_engine_search with CUDA events on the launching stream.
 * profile_read synchronises `stream` and returns the summed milliseconds of
 * [0] select, [1] plan, [2] network forward, [3] expand+backup, [4] Dirichlet-noise kernels since the last read,
 * plus the number of engine kernels launched by search/play in that window. */
/* enable: 0 = off, 1 = network kernel only (2 events per minibatch), 2 = all four phases. */
int caro_engine_profile(caro_engine* e, int enable);
int caro_engine_profile_read(caro_engine* e, double h_ms[5], uint64_t* h_launches, void* stream);

/* Resignation parameters (the rule beside CARO_FLAG_*), enqueued on `stream` and read by every later
 * advance; the playthrough share applies to games that start after the call.  enable = 0 switches resignation off.
 * Returns CARO_E_ARG (before touching the device) for a null handle, a threshold that is NaN or outside [-1, 1], or a
 * playthrough share that is NaN or outside [0, 1]. */
int caro_engine_set_resign(caro_engine* e, int enable, double threshold, double playthrough, void* stream);

/* MCTS solver (extension, off by default; the reference's search never knows that a position is decided).  Switched at
 * run time by caro_engine_set_solver; the mask lives in device memory (region "solver_params"), and the engine re-captures
 * a ply graph of caro_engine_play_multi when the solver goes from off to on or back.
 *   Edge status, for the side to move at the edge's node, in bits 29-30 of the edge's N word ("nodes" region; the visit
 *   count is bits 0-28): 0 UNKNOWN, 1 WIN, 2 LOSS, 3 DRAW.  A node is WIN if a legal edge is WIN, LOSS if every legal
 *   edge is LOSS, DRAW if every legal edge is proven, none WIN and one DRAW, else UNKNOWN.
 *   Select (solver on for the root player): a descent that reaches a proven node below the root stops there as a terminal
 *   with value +1 / -1 / 0 for the node's mover (no network evaluation); a proven root makes no descent; LOSS edges are left
 *   out of the argmax (a node with a WIN edge, or with LOSS edges only, is proven and never scored).
 *   Back-up: values as without the solver; then, in back-up queue order, each terminal entry proves its last edge (leaf
 *   value -1: WIN, 0: DRAW, +1: LOSS) and walks up its own path while the node above is proven, setting the next edge to
 *   the negated node status.
 *   Root policy and advance: a proven-WIN root gives pi one-hot on its lowest WIN edge whatever tau is; otherwise LOSS
 *   edges are zeroed in the visit counts pi and the move are drawn from (tau = 0: argmax over the rest), unless that
 *   leaves no visit.  The pi the move was drawn from is the one written to the history and the replay ring; the Philox
 *   choice stream is unchanged.
 * Regions: "solver_params" {int32 players, int32 pad}, "solver_counters" uint64 [2]: [0] descents stopped at a proven node,
 *          [1] edges proven.  They follow every other region. */
/* players: bit p = searches whose root player is p use the solver (with two trees per game: tree p).  Returns CARO_E_ARG
 * (before touching the device) for a null handle, a mask outside 0..3, a mask of 1 or 2 on an engine with one tree per
 * game (its tree serves both players), and a non-zero mask on a virtual-loss engine.  Enqueued on `stream`. */
int caro_engine_set_solver(caro_engine* e, int players, void* stream);

/* Gumbel root search (extension, off by default; Danihelka et al., "Policy improvement by planning with Gumbel", ICLR
 * 2022).  Switched at run time by caro_engine_set_gumbel; the parameters live in device memory (region "gumbel_params"),
 * and the engine re-captures a ply graph of caro_engine_play_multi when Gumbel goes from off to on or back.  Only the ROOT
 * of a Gumbel player's searches changes: below it descents keep PUCT, and plan, expansion and back-up are unchanged.
 * A search is one caro_engine_search / play / play_multi call: C minibatches i = 0 .. C-1 of b descents.
 *   1. Draws.  At minibatch 0, for every action a: g(a) = -log(-log(u)) in double, u = k * 2^-53 with k the top 53 bits
 *      of Philox stream kStreamGumbel addressed by (uid, search_index, ply, a) (k = 0 is replaced by 1/2: u lies in the
 *      open interval (0, 1)).  search_index is 0 for play / play_multi and first_minibatch for caro_engine_search.  The
 *      draws are stored unscaled in "gumbel_g" (double [G][A]); illegal actions' draws are never read.
 *   2. Scores, all in double, with P the stored prior and N masked with the count mask:
 *        q(a)     = Q of a visited edge as the root branch of select computes it (f32(W/N), or the float64 quotient of
 *                   an edge whose W has absorbed no float32 value); for an unvisited edge, the prior-weighted mean
 *                   sum_b P(b) q(b) / sum_b P(b) over the visited legal edges b (sums in action order), or 0 when no
 *                   legal edge is visited.  (mctx's completed Q also mixes in the network value of the root, which the
 *                   node record does not keep; it is left out.)
 *        sigma(a) = ((c_visit + max_b N(b)) * c_scale) * ((q(a) + 1) * 0.5)
 *        base(a)  = gumbel_scale * g(a) + log P(a)          (P = 0 gives -inf)
 *        score(a) = base(a) + sigma(a);   logit(a) = log P(a) + sigma(a)
 *      Every comparison breaks ties towards the lowest action index.
 *   3. Schedule.  m = min(m_param, legal moves); H = ceil(log2 m) phases; phase p keeps r_p = min(m, max(2, ceil(m/2^p)))
 *      survivors.  i0 = the first minibatch at which the root is in the tree; before it descents are not forced (the
 *      first one expands the root as without Gumbel).  Local minibatch k = i - i0 of C' = C - i0 is in phase
 *      floor(k H / C') (0 when H = 0).  At k = 0 (phase 0) the survivors are the top m legal actions by base; whenever the
 *      phase changes (phases are skipped when C' < H) they become the top r_p of the current survivors by score, on the
 *      tree as it stands after the previous minibatch's back-up.  Survivors are kept in score order (best first); descent j
 *      of minibatch k takes survivor number ((k - k_phase_start) * b + j) mod r_p at the root.
 *   4. Policy target pi'(a) = softmax over the legal actions of logit, on the final tree: exp(logit - max) summed over the
 *      legal actions in action order, each quotient stored as float32; uniform over the legal moves when every legal
 *      logit is -inf.  pi' replaces the visit distribution in the history and the replay ring (z is unchanged), and
 *      caro_engine_root_policy returns it for tau_mode 1 and 2 (the tau schedule does not apply).
 *   5. Move = argmax of score over the current survivors on the final tree (over every legal action when no phase ran).
 *      caro_engine_root_policy with tau_mode 0 returns a one-hot on it.  The Philox choice stream is not consumed
 *      differently, so a non-Gumbel player's moves do not shift.
 * Regions: "gumbel_params" {int32 players, int32 m, double c_visit, double c_scale, double gumbel_scale};
 *          "gumbel_g" double [G][A]; "gumbel_state" [G] records of 80 bytes {int32 i0 (-1: root not yet in the tree),
 *          int32 phase (-1: none ran), int32 k_phase_start, int16 m, int16 r, int16 survivors[32]}; "gumbel_root"
 *          int16 [G][max_batch]: the forced root action of each descent of the coming minibatch, or -1.  They follow every
 *          other region; zero means off. */
/* players: bit p = searches whose root player is p use the Gumbel root search.  Returns CARO_E_ARG (before touching the
 * device) for a null handle, a mask outside 0..3, a mask of 1 or 2 with one tree per game, a non-zero mask on a
 * virtual-loss engine or while the solver mask is non-zero, m outside 1..32, and a negative, NaN or infinite c_visit,
 * c_scale or gumbel_scale.  (caro_engine_set_solver in turn refuses a non-zero mask while Gumbel is on.)  Enqueued on
 * `stream`.  Defaults of the paper and mctx: m 16, c_visit 50, c_scale 0.1, gumbel_scale 1. */
int caro_engine_set_gumbel(caro_engine* e, int players, int m, double c_visit, double c_scale, double gumbel_scale,
                           void* stream);
/* The split-API step that callers supplying their own network outputs enqueue before caro_engine_select of minibatch
 * `minibatch` (0 .. count-1) of a search of `count` minibatches (caro_engine_search, play and play_multi enqueue it
 * themselves): the draws at minibatch 0, the phase and survivors, and "gumbel_root".  Returns CARO_E_ARG for a null
 * handle, search_index < 0, count < 1, minibatch outside 0..count-1 or a batch outside 1..max_batch; does nothing while
 * Gumbel is off. */
int caro_engine_gumbel_plan(caro_engine* e, int search_index, int minibatch, int count, int batch, void* stream);

/* Host copies of the 64-bit counters (synchronises `stream`): [0] leaf evaluations, [1] finished
 * games, [2] plies played, [3] wins of player 0, [4] wins of player 1, [5] draws, [6] descents,
 * [7] error flags (bit 0 arena full, bit 1 replay overrun, bit 2 illegal action sampled). */
int caro_engine_counters(caro_engine* e, uint64_t h_out[8], void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CARO_B200_H_ */
