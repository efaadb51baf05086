// Device-side data layout of the self-play engine: node records with per-game arenas (structure of arrays inside
// a node: [N | W | P | child link] rows, one 128-byte line per Connect4 node), a per-arena open-addressing
// transposition table, per-descent records and the compact leaf batch.
//
// Replaces the four `state_int -> list[A]` dicts of lib/mcts.py:29-36 and the Python queues of
// lib/mcts.py:259-287.  See DESIGN.md section 4 for the byte budget.
#pragma once
#include <stdint.h>
#include "rules.cuh"

namespace caro {

enum : uint8_t { KIND_SKIP = 0, KIND_TERMINAL = 1, KIND_EXPAND = 2 };
enum : uint8_t { ST_ACTIVE = 0, ST_FINISHED = 1 };
enum { CTR_LEAVES = 0, CTR_GAMES, CTR_PLIES, CTR_WIN0, CTR_WIN1, CTR_DRAW, CTR_DESCENTS, CTR_ERRORS, CTR_COUNT };
constexpr int kNetBit = (int)0x80000000u;   // flag bit inside an N word
constexpr int kCountMask = 0x1fffffff;      // visit count: bits 0..28 (counts stay far below 2^29)
// Solver (extension): bits 29-30 of an N word hold the edge's proof for the side to move at the node
constexpr int kProofShift = 29;
constexpr int kProofMask = 3 << kProofShift;
enum : int { PROOF_UNKNOWN = 0, PROOF_WIN = 1, PROOF_LOSS = 2, PROOF_DRAW = 3 };
enum : unsigned long long { ERR_ARENA_FULL = 1ull, ERR_REPLAY_OVERRUN = 2ull, ERR_ILLEGAL_ACTION = 4ull };

struct alignas(16) HashSlot {
  uint64_t key;   // Key128::lo
  int32_t node;   // arena-local node index
  uint32_t gen;   // slot is live iff gen == tree_gen[tree] (clear() == ++gen, no memset)
};

// One descent of the current minibatch (lib/mcts.py:97-148 returns value, leaf state, leaf player, states[], actions[]).
// ONE record per descent -- 64 bytes for Connect4 (two sectors of one line), 96 for m,n,k -- instead of eight parallel
// arrays: select writes it with four 16-byte stores, plan and expand+backup read what they need with one or two loads
// (the parallel arrays cost ~10 sectors per descent for <= 40 useful bytes: 4.8x the algorithmic DRAM traffic).
struct alignas(16) DescHead {
  uint8_t kind;      // KIND_*
  uint8_t player;    // side to move at the leaf
  uint16_t len;      // path length (edges from the root to the leaf)
  int32_t slot;      // compact leaf slot of an expand entry (plan), -1 otherwise
  float value;       // terminal value (-1 / 0), lib/mcts.py:140-146
  uint32_t pad_;
  uint64_t key_lo, key_hi;  // transposition key of the leaf
};
template <class Board>
struct alignas(32) DescRec {
  DescHead h;
  Board board;       // leaf position
};

// One entry of a game's back-up queue in back-up order (lib/mcts.py:269-278): everything expand+backup needs to start
// its loads at once (no order -> kind -> slot -> value chain).  `slot` holds the float bits of the value for a terminal.
struct alignas(8) QEntry {
  uint8_t j;         // descent index within the minibatch
  uint8_t kind;
  uint16_t len;
  int32_t slot;
};

struct Dims {
  int G;          // games
  int tpg;        // trees per game
  int B;          // max descents per minibatch (stride of per-descent arrays)
  int A;          // actions
  int Apad;       // entries per row of a node record (A rounded up to 8)
  int RS;         // 32-bit words per node record = 4 * Apad: [N | W | P | C] rows of Apad entries each
  int node_cap;   // nodes per arena
  int hash_cap;   // slots per arena (power of two, 2x node_cap)
  int max_depth;  // path stride = max plies of the game
  int max_plies;  // history stride
  int replay_cap;
  unsigned flags;  // CARO_FLAG_* (include/caro_b200.h): throughput-mode extensions, 0 = the reference's search
};
enum : unsigned { FLAG_VIRTUAL_LOSS = 1u, FLAG_MASK_PRIORS = 2u, FLAG_FRESH_TREE = 4u, FLAG_RECYCLE_TREE = 8u, FLAG_COMPACT_TREE = 16u };

// Resignation (extension, off by default; include/caro_b200.h caro_engine_set_resign).  The parameters live in device memory
// and are read by advance_kernel / reset_kernel at run time, so a captured ply graph never holds stale values.
struct alignas(8) ResignParams {
  int32_t enabled;     // 0 = off: no statistic, no resignation, no log
  int32_t pad_;
  double threshold;    // the side to move resigns when its root statistic is < threshold
  double playthrough;  // share of games (drawn per game at its start) that never resign and are logged instead
};
// One finished playthrough game: the smallest root statistic each player saw, the result from player 0's point of view
struct alignas(8) ResignRecord {
  double min_stat[2];
  int32_t result;
  int32_t plies;
};
static_assert(sizeof(ResignRecord) == 24, "resign log records are 24 bytes");
enum { RCTR_RESIGNED = 0, RCTR_LOGGED, RCTR_COUNT };

// MCTS solver (extension, off by default; include/caro_b200.h caro_engine_set_solver).  Read by the select, expand +
// back-up, root policy and advance kernels at run time, like the resignation parameters.
struct alignas(8) SolverParams {
  int32_t players;  // bit p: searches whose root player is p use the solver
  int32_t pad_;
};
enum { SCTR_STOPPED = 0, SCTR_PROVEN, SCTR_COUNT };

// Gumbel root search (extension, off by default; include/caro_b200.h caro_engine_set_gumbel).  Read by
// gumbel_plan_kernel and the GUMBEL instances of root_policy_kernel / advance_kernel at run time.
struct alignas(8) GumbelParams {
  int32_t players;      // bit p: searches whose root player is p search their root by Gumbel sequential halving
  int32_t m;            // root actions sampled per search (1..32)
  double c_visit, c_scale;  // sigma(q) = (c_visit + max_b N(b)) * c_scale * q
  double gumbel_scale;  // scale of the Gumbel draws in the survivor score and the move
};
constexpr int kGumbelMaxM = 32;
// Per game: where the current search stands (action indices only, so compaction and tree clears leave it valid)
struct alignas(8) GumbelState {
  int32_t i0;      // first minibatch of the search at which the root was in the tree (-1: not yet)
  int32_t phase;   // current halving phase (-1: none ran)
  int32_t kstart;  // local minibatch (k = i - i0) at which the current phase began
  int16_t m;       // min(m, legal moves) of this search
  int16_t r;       // current survivors
  int16_t surv[kGumbelMaxM];  // survivors [0, r) in score order (best first)
};
static_assert(sizeof(GumbelState) == 80, "gumbel_state records are 80 bytes");

struct SearchParams {
  double c_puct, alpha, explore;
  uint32_t seed_lo, seed_hi;
};

template <class Board>
struct View {
  // ---- tree arenas (index = tree * node_cap + node) --------------------------------------
  // One record of RS = 4 * Apad words per node, rows [N | W | P | C]; the four pointers below address row 0 / 1 / 2 / 3
  // of record 0, so X[(nb + node) * RS + a] is entry a of row X.  A Connect4 record is one aligned 128-byte line: a
  // descent step reads exactly that line, a back-up touches its first 64 bytes, an expansion writes it whole.
  int32_t* N;          // visit counts (lib/mcts.py:30) in bits 0..28; bits 29-30: solver proof; bit 31 (kNetBit): W(s,a) has absorbed a float32
                       // network value (numpy promotion state of the reference's python-float / np.float32 sums)
  float* W;            // total value (lib/mcts.py:32).  The mean value Q (lib/mcts.py:34) is not stored: it always
                       // equals f32(W / N) (0 while N == 0) and is recomputed where it is read
  float* P;            // priors (lib/mcts.py:36)
  int32_t* C;          // cached child node per edge (-1 = not linked yet): a pure cache of the
                       // transposition lookup, so an interior step of a descent is ONE dependent access
  uint64_t* key_hi;    // [..]  upper 64 fingerprint bits (m,n,k only)
  Board* node_board;   // [..]  position of the node (export / dict views)
  uint8_t* node_player;  // [..] side to move when the node was created
  HashSlot* ht;        // [trees][hash_cap]
  int32_t* node_count; // [trees]
  uint32_t* tree_gen;  // [trees]
  // ---- games -------------------------------------------------------------------------------
  Board* root_board;   // [G]
  uint8_t* root_player;  // [G]
  uint8_t* status;     // [G]
  int32_t* ply;        // [G] completed non-terminal plies (== `step` of lib/utils.py:69)
  int32_t* result;     // [G] last finished game: +1 player0 won, -1 player1 won, 0 draw
  uint64_t* uid;       // [G] RNG sub-stream id of the current game
  uint32_t* played;    // [G] games finished in this slot
  Board* hist_board;   // [G][max_plies]
  uint8_t* hist_player;  // [G][max_plies]
  float* hist_pi;      // [G][max_plies][A]
  // ---- per descent (index = g*B + j) -------------------------------------------------------
  DescRec<Board>* desc;    // [G*B]
  uint32_t* d_path;        // [G*B][max_depth]  (arena-local node index << 8) | action, root first
  // ---- minibatch plan ----------------------------------------------------------------------
  int32_t* q_len;      // [G]
  QEntry* q_entry;     // [G][B] back-up queue
  // ---- compact leaf batch ------------------------------------------------------------------
  Board* leaf_board;   // [G*B]
  uint8_t* leaf_player;  // [G*B]
  int32_t* leaf_count; // [1]
  double* noise;       // [G][B][A] Dirichlet noise of the coming minibatch (Philox path)
  float* probs;        // [G*B][A]  network outputs (built-in net path)
  float* values;       // [G*B]
  // ---- replay ring -------------------------------------------------------------------------
  Board* rp_board;
  uint8_t* rp_player;
  float* rp_pi;        // [replay_cap][A]
  float* rp_z;
  unsigned long long* rp_cursor;  // [1] total entries ever written
  // ---- counters ------------------------------------------------------------------------------
  unsigned long long* ctr;  // [CTR_COUNT]
  // ---- resignation (extension) -----------------------------------------------------------------
  ResignParams* resign_params;   // [1]
  uint8_t* resign_playthrough;   // [G] the current game is a playthrough game
  double* resign_min;            // [G][2] smallest statistic per player of the current playthrough game
  ResignRecord* resign_log;      // [G] ring of finished playthrough games (slot = cursor % G)
  unsigned long long* resign_ctr;  // [RCTR_COUNT] games resigned, playthrough games logged (= log cursor)
  // ---- MCTS solver (extension) ------------------------------------------------------------------
  SolverParams* solver_params;     // [1]
  unsigned long long* solver_ctr;  // [SCTR_COUNT] descents stopped at a proven node, edges proven
  // ---- Gumbel root search (extension) -----------------------------------------------------------
  GumbelParams* gumbel_params;     // [1]
  double* gumbel_g;                // [G][A] unscaled Gumbel draws of the current search
  GumbelState* gumbel_state;       // [G]
  int16_t* gumbel_root;            // [G][B] forced root action of each descent of the coming minibatch (-1: PUCT)
};

}  // namespace caro
