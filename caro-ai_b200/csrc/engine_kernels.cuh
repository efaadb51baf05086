// Search kernels: PUCT select (one lane-group per descent), minibatch plan (dedup + leaf gather),
// expand + ordered back-up (one warp per game), root policy and the per-ply game step.
//
// Arithmetic contract (SURVEY.md A.4 = the reference under numpy >= 2): interior scores float32
// with no FMA contraction, root (noisy) scores float64, W/Q float32, ties -> lowest action.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include "engine.cuh"
#include "rng.cuh"

namespace caro {

// ------------------------------------------------------------------------------ small helpers
template <int GW>
__device__ __forceinline__ unsigned group_mask() {
  if (GW == 32) return 0xffffffffu;
  const unsigned lane = threadIdx.x & 31u;
  return ((1u << GW) - 1u) << (lane & ~(unsigned)(GW - 1));
}

__device__ __forceinline__ HashSlot load_slot(const HashSlot* p) {
  const uint4 v = *reinterpret_cast<const uint4*>(p);
  HashSlot s;
  s.key = ((uint64_t)v.y << 32) | v.x;
  s.node = (int32_t)v.z;
  s.gen = v.w;
  return s;
}

__device__ __forceinline__ uint32_t slot_home(uint64_t key_lo, int cap) {
  return (uint32_t)mix64(key_lo) & (uint32_t)(cap - 1);
}

// Transposition lookup, GW slots probed per round by the GW lanes of a descent group
// (is_leaf, lib/mcts.py:150-160).  Returns the arena-local node index or -1.
template <int GW>
__device__ __forceinline__ int ht_lookup(const HashSlot* __restrict__ ht, int cap, uint32_t gen, Key128 key,
                                         const uint64_t* __restrict__ key_hi /* arena base or nullptr */,
                                         int gl, unsigned gmask) {
  const uint32_t home = slot_home(key.lo, cap);
  const int gbase = (threadIdx.x & 31) & ~(GW - 1);
  for (int it = 0; it < cap; it += GW) {
    const uint32_t idx = (home + (uint32_t)(it + gl)) & (uint32_t)(cap - 1);
    const HashSlot sl = load_slot(ht + idx);
    const bool empty = sl.gen != gen;
    bool match = !empty && sl.key == key.lo;
    if (match && key_hi != nullptr) match = key_hi[sl.node] == key.hi;
    const unsigned bm = __ballot_sync(gmask, match) >> gbase;
    const unsigned be = __ballot_sync(gmask, empty) >> gbase;
    const int fm = bm ? (__ffs(bm) - 1) : 64;
    const int fe = be ? (__ffs(be) - 1) : 64;
    if (fm < fe) return __shfl_sync(gmask, sl.node, gbase + fm);
    if (fe < 64) return -1;
  }
  return -1;
}

// single-thread variant (expand / policy kernels)
__device__ __forceinline__ int ht_lookup1(const HashSlot* __restrict__ ht, int cap, uint32_t gen, Key128 key,
                                          const uint64_t* __restrict__ key_hi) {
  uint32_t idx = slot_home(key.lo, cap);
  for (int it = 0; it < cap; ++it) {
    const HashSlot sl = load_slot(ht + idx);
    if (sl.gen != gen) return -1;
    if (sl.key == key.lo && (key_hi == nullptr || key_hi[sl.node] == key.hi)) return sl.node;
    idx = (idx + 1u) & (uint32_t)(cap - 1);
  }
  return -1;
}

// The descent's record (engine.cuh): head = two 16-byte stores, board = 16-byte stores.
template <class Board>
__device__ __forceinline__ void store_desc(DescRec<Board>* __restrict__ rec, int kind, int player, int len, float value, Key128 key,
                                           const Board& board) {
  DescHead h;
  h.kind = (uint8_t)kind;
  h.player = (uint8_t)player;
  h.len = (uint16_t)len;
  h.slot = -1;
  h.value = value;
  h.pad_ = 0u;
  h.key_lo = key.lo;
  h.key_hi = key.hi;
  rec->h = h;
  rec->board = board;
}
template <class Board>
__device__ __forceinline__ void store_desc_skip(DescRec<Board>* __restrict__ rec) {
  DescHead h;
  h.kind = KIND_SKIP;
  h.player = 0;
  h.len = 0;
  h.slot = -1;
  h.value = 0.0f;
  h.pad_ = 0u;
  h.key_lo = 0ull;
  h.key_hi = 0ull;
  rec->h = h;
}

template <class R>
struct RulesTraits {
  static constexpr bool kHasKeyHi = true;
};
template <>
struct RulesTraits<C4Rules> {
  static constexpr bool kHasKeyHi = false;
};

// ---------------------------------------------------------------------------------- MCTS solver (extension)
// A node's status from its legal edges' proofs: WIN if one is WIN, LOSS if all are LOSS, DRAW if all are proven, none is
// WIN and one is DRAW.  A node always has a legal edge (terminal positions never become nodes).
__device__ __forceinline__ int proof_status(bool any_win, bool all_loss, bool all_proven, bool any_draw) {
  return any_win ? PROOF_WIN : (all_loss ? PROOF_LOSS : ((all_proven && any_draw) ? PROOF_DRAW : PROOF_UNKNOWN));
}
// value of a proven node for its mover, and the proof of the edge into a node of status `st` for the mover above
__device__ __forceinline__ float proof_value(int st) { return st == PROOF_WIN ? 1.0f : (st == PROOF_LOSS ? -1.0f : 0.0f); }
__device__ __forceinline__ int proof_negate(int st) { return st == PROOF_WIN ? PROOF_LOSS : (st == PROOF_LOSS ? PROOF_WIN : st); }
// is the solver on for searches of game g (root player `who`)?
template <class Board>
__device__ __forceinline__ bool solver_on(const View<Board>& e, int who) { return (e.solver_params->players >> who) & 1; }

// ------------------------------------------------------------------------------- Dirichlet noise
// np.random.dirichlet([alpha] * A) for every descent of the coming minibatch (lib/mcts.py:56), Philox-addressed by
// (seed, game uid, ply, side to move, minibatch, descent, action).  Kept out of select_kernel: the sampler's
// registers and code would otherwise halve that kernel's occupancy.  Layout float64 [G][batch][A].
template <int GW, int APL>
__global__ void __launch_bounds__(256)
noise_kernel(const uint64_t* __restrict__ uid_g, const int32_t* __restrict__ ply_g, const uint8_t* __restrict__ player_g,
             Dims dm, SearchParams sp, int batch, int mb_index, double* __restrict__ noise) {
  const long long gthread = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long grp = gthread / GW;
  if (grp >= (long long)dm.G * batch) return;
  const int gl = threadIdx.x & (GW - 1);
  const unsigned gmask = group_mask<GW>();
  const int g = (int)(grp / batch), j = (int)(grp % batch);
  const int A = dm.A;
  const uint64_t uid = uid_g[g];
  const uint32_t ply = (uint32_t)ply_g[g];
  const uint32_t who = player_g[g];
  float z[APL];
  float zs = 0.0f;
#pragma unroll
  for (int i = 0; i < APL; ++i) {
    const int a = gl + i * GW;
    z[i] = 0.0f;
    if (a < A)
      z[i] = gamma_small((float)sp.alpha, sp.seed_lo ^ kStreamDirichlet, sp.seed_hi, (uint32_t)uid,
                         (uint32_t)(uid >> 32) ^ (ply << 16) ^ who, ((uint32_t)(mb_index * batch + j) << 8) | (uint32_t)a);
    zs += z[i];
  }
  double zd = (double)zs;
#pragma unroll
  for (int off = GW / 2; off > 0; off >>= 1) zd += __shfl_xor_sync(gmask, zd, off);
#pragma unroll
  for (int i = 0; i < APL; ++i) {
    const int a = gl + i * GW;
    if (a < A) noise[((size_t)g * batch + j) * A + a] = __ddiv_rn((double)z[i], zd);
  }
}

// ---------------------------------------------------------------------------------- select
// One group of GW lanes per descent, APL actions per lane (action = lane + i*GW).
// SOLVER (extension): the body reads the proofs of the N words when the solver is on for the game's root player.  A
// descent that reaches a proven node below the root stops there as a terminal (value +1 / -1 / 0 for the node's mover),
// a proven root makes no descent at all, and LOSS edges are left out of the argmax.  (The lowest WIN edge of a node with
// a WIN edge, and the argmax over LOSS edges when all legal edges are LOSS, are never taken here: such a node is proven.)
// GUMBEL (extension): a descent whose gumbel_root entry (written by gumbel_plan_kernel) is an action takes it at the root
// without scoring the root; every other step, and every descent whose entry is -1, is the reference's.
template <class R, int GW, int APL, bool SOLVER, bool GUMBEL>
__device__ __forceinline__ void select_group_body(const View<typename R::Board>& e, const R& rules, const Dims& dm,
                                                  const SearchParams& sp, int batch, const double* __restrict__ noise_in,
                                                  long long gthread) {
  using Board = typename R::Board;
  const long long grp = gthread / GW;
  if (grp >= (long long)dm.G * batch) return;
  const int gl = threadIdx.x & (GW - 1);
  const unsigned gmask = group_mask<GW>();
  const int g = (int)(grp / batch), j = (int)(grp % batch);
  const size_t di = (size_t)g * dm.B + j;
  if (e.status[g] != ST_ACTIVE) {
    if (gl == 0) store_desc_skip(e.desc + di);
    return;
  }
  const int A = dm.A;
  Board s = e.root_board[g];
  int who = e.root_player[g];
  const bool sol = SOLVER && solver_on(e, who);
  const int forced = GUMBEL ? (int)e.gumbel_root[di] : -1;  // Gumbel root search: the planned root action, or -1
  const int tree = g * dm.tpg + (dm.tpg == 2 ? who : 0);
  const uint32_t gen = e.tree_gen[tree];
  const HashSlot* ht = e.ht + (size_t)tree * dm.hash_cap;
  const size_t nb = (size_t)tree * dm.node_cap;
  const uint64_t* khi = RulesTraits<R>::kHasKeyHi ? (e.key_hi + nb) : nullptr;

  const float c_f = (float)sp.c_puct;                 // python float * np.float32 -> float32 (NEP 50)
  const float keep_f = (float)(1.0 - sp.explore);     // (1 - EXPLORE) * prob, lib/mcts.py:59
  Key128 key = rules.key(s);
  int node = ht_lookup<GW>(ht, dm.hash_cap, gen, key, khi, gl, gmask);
  int depth = 0;
  int kind = KIND_EXPAND;
  float term_value = 0.0f;
  uint32_t* path = e.d_path + di * dm.max_depth;

  while (node >= 0) {
    const size_t row = (nb + (size_t)node) * dm.RS;
    int n_loc[APL], c_loc[APL];
    float w_loc[APL], p_loc[APL];
    bool net_loc[APL];
    int sum_n = 0;
#pragma unroll
    for (int i = 0; i < APL; ++i) {
      const int a = gl + i * GW;
      if (a < A) {
        const int raw = e.N[row + a];
        n_loc[i] = raw & kCountMask;
        net_loc[i] = raw < 0;
        w_loc[i] = e.W[row + a];
        p_loc[i] = e.P[row + a];
        c_loc[i] = e.C[row + a];
      } else {
        n_loc[i] = 0;
        net_loc[i] = false;
        w_loc[i] = 0.0f;
        p_loc[i] = 0.0f;
        c_loc[i] = -1;
      }
      sum_n += n_loc[i];
    }
#pragma unroll
    for (int off = GW / 2; off > 0; off >>= 1) sum_n += __shfl_xor_sync(gmask, sum_n, off);
    unsigned loss_m = 0u;  // bit i: my action gl + i * GW is a LOSS edge (solver)
    if (sol) {
      bool win = false, all_loss = true, all_proven = true, draw = false;
#pragma unroll
      for (int i = 0; i < APL; ++i) {
        const int a = gl + i * GW;
        if (a < A && rules.legal(s, a)) {
          const int pf = (e.N[row + a] >> kProofShift) & 3;
          win = win || pf == PROOF_WIN;
          draw = draw || pf == PROOF_DRAW;
          all_loss = all_loss && pf == PROOF_LOSS;
          all_proven = all_proven && pf != PROOF_UNKNOWN;
          loss_m |= (pf == PROOF_LOSS ? 1u : 0u) << i;
        }
      }
      const int st = proof_status(__any_sync(gmask, win), __all_sync(gmask, all_loss), __all_sync(gmask, all_proven),
                                  __any_sync(gmask, draw));
      if (st != PROOF_UNKNOWN) {
        if (depth == 0) {  // proven root: no descent
          if (gl == 0) store_desc_skip(e.desc + di);
          return;
        }
        kind = KIND_TERMINAL;
        term_value = proof_value(st);
        if (gl == 0) atomicAdd(e.solver_ctr + SCTR_STOPPED, 1ull);
        break;
      }
    }

    double best = -INFINITY;
    int best_a = 0x7fffffff;
    if (GUMBEL && depth == 0 && forced >= 0) {
      best = 0.0;  // every lane agrees: the group argmax below keeps the forced action
      best_a = forced;
    } else if (depth == 0) {
      // ---- root: Dirichlet noise + float64 scores (lib/mcts.py:48-62,131-132) -------------
      double z[APL];
#pragma unroll
      for (int i = 0; i < APL; ++i) {
        const int a = gl + i * GW;
        z[i] = (a < A) ? noise_in[((size_t)g * batch + j) * A + a] : 0.0;
      }
      const double sq = sqrt((double)sum_n);
#pragma unroll
      for (int i = 0; i < APL; ++i) {
        const int a = gl + i * GW;
        if (a < A && rules.legal(s, a) && !((loss_m >> i) & 1u)) {
          const double pn = __dadd_rn((double)__fmul_rn(keep_f, p_loc[i]), __dmul_rn(sp.explore, z[i]));
          const double u = __ddiv_rn(__dmul_rn(__dmul_rn(sp.c_puct, pn), sq), (double)(1 + n_loc[i]));
          // Q keeps python-float (float64) precision until a float32 value touched W(s,a)
          double q64 = 0.0;  // value_avg (lib/mcts.py:244) is not stored: f32(W/N), or the float64 quotient of a python-float edge
          if (n_loc[i] > 0)
            q64 = net_loc[i] ? (double)__fdiv_rn(w_loc[i], (float)n_loc[i]) : __ddiv_rn((double)w_loc[i], (double)n_loc[i]);
          const double sc = __dadd_rn(q64, u);
          if (sc > best) {
            best = sc;
            best_a = a;
          }
        }
      }
    } else {
      // ---- interior: float32 scores (lib/mcts.py:64-84 under NEP 50) ----------------------
      // float32(math.sqrt(sum N)): for integers below 2^24 the float64 root rounded to float32 equals the correctly
      // rounded float32 root (no double-rounding case exists), so the cheap instruction is bit-identical
      const float sq = __fsqrt_rn((float)sum_n);
#pragma unroll
      for (int i = 0; i < APL; ++i) {
        const int a = gl + i * GW;
        if (a < A && rules.legal(s, a) && !((loss_m >> i) & 1u)) {
          const float t = __fdiv_rn(__fmul_rn(__fmul_rn(c_f, p_loc[i]), sq), (float)(1 + n_loc[i]));
          const float q = n_loc[i] > 0 ? __fdiv_rn(w_loc[i], (float)n_loc[i]) : 0.0f;  // value_avg, lib/mcts.py:244
          const double sc = (double)__fadd_rn(q, t);
          if (sc > best) {
            best = sc;
            best_a = a;
          }
        }
      }
    }
    // first maximum over the group (np.argmax, lib/mcts.py:136)
#pragma unroll
    for (int off = GW / 2; off > 0; off >>= 1) {
      const double ob = __shfl_xor_sync(gmask, best, off);
      const int oa = __shfl_xor_sync(gmask, best_a, off);
      if (ob > best || (ob == best && oa < best_a)) {
        best = ob;
        best_a = oa;
      }
    }
    const int a = best_a;
    if (gl == 0) path[depth] = ((uint32_t)node << 8) | (uint32_t)a;
    ++depth;
    const bool won = rules.apply(s, a, who);  // lib/mcts.py:138-139
    who ^= 1;
    if (won) {
      kind = KIND_TERMINAL;
      term_value = -1.0f;  // lib/mcts.py:140-142
      break;
    }
    if (!rules.any_legal(s)) {
      kind = KIND_TERMINAL;
      term_value = 0.0f;   // lib/mcts.py:145-146
      break;
    }
    key = rules.key(s);
    // child link cached on the edge?  (set the first time the lookup succeeds; nodes are never removed)
    int mine = -1;
#pragma unroll
    for (int i = 0; i < APL; ++i)
      if (i == a / GW) mine = c_loc[i];
    const int linked = __shfl_sync(gmask, mine, ((threadIdx.x & 31) & ~(GW - 1)) + (a % GW));
    if (linked >= 0) {
      node = linked;
    } else {
      node = ht_lookup<GW>(ht, dm.hash_cap, gen, key, khi, gl, gmask);
      if (node >= 0 && gl == 0) e.C[row + a] = node;
    }
  }
  if (gl == 0) store_desc(e.desc + di, kind, who, depth, term_value, key, s);
}

// SOLVER = false is the reference's search.  The host launches the SOLVER instance while the engine's solver mask is
// non-zero (a run-time branch on the mask would cost the plain instances registers); it then checks the mask per game.
// GUMBEL instances likewise run only while the engine's Gumbel mask is non-zero (the two masks are never both non-zero).
template <class R, int GW, int APL, bool SOLVER, bool GUMBEL>
__global__ void __launch_bounds__(256, (APL == 1 && sizeof(typename R::Board) <= 16) ? 7 : (APL == 8 ? 2 : 1))
select_kernel(View<typename R::Board> e, R rules, Dims dm, SearchParams sp, int batch,
              const double* __restrict__ noise_in) {
  const long long gthread = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gthread == 0) {
    *e.leaf_count = 0;  // plan_kernel (next launch on the stream) accumulates into it
  }
  select_group_body<R, GW, APL, SOLVER, GUMBEL>(e, rules, dm, sp, batch, noise_in, gthread);
}

// Thread-per-descent variant for small action spaces (A <= 16: Connect4, 3x3 / 4x4 boards).  The board update,
// key and transposition probe are scalar work; with one lane-group per descent they are replicated on every
// lane and the kernel becomes issue-bound (ncu: 12.7 M warp instructions per launch).  Here each lane owns a whole
// descent and loops over the <= 16 actions; the arithmetic and its order are identical to select_kernel.
template <class R, int ROWV, bool SOLVER, bool GUMBEL>  // ROWV = Apad / 4 = number of 16-byte vectors per row; SOLVER, GUMBEL: as select_group_body
__device__ __forceinline__ void select_thread_body(const View<typename R::Board>& e, const R& rules, const Dims& dm,
                                                   const SearchParams& sp, int batch, const double* __restrict__ noise_in,
                                                   long long grp) {
  using Board = typename R::Board;
  if (grp >= (long long)dm.G * batch) return;
  const int g = (int)(grp / batch), j = (int)(grp % batch);
  const size_t di = (size_t)g * dm.B + j;
  if (e.status[g] != ST_ACTIVE) {
    store_desc_skip(e.desc + di);
    return;
  }
  const int A = dm.A;
  Board s = e.root_board[g];
  int who = e.root_player[g];
  const bool sol = SOLVER && solver_on(e, who);
  const int forced = GUMBEL ? (int)e.gumbel_root[di] : -1;  // Gumbel root search: the planned root action, or -1
  const int tree = g * dm.tpg + (dm.tpg == 2 ? who : 0);
  const uint32_t gen = e.tree_gen[tree];
  const HashSlot* ht = e.ht + (size_t)tree * dm.hash_cap;
  const size_t nb = (size_t)tree * dm.node_cap;
  const uint64_t* khi = RulesTraits<R>::kHasKeyHi ? (e.key_hi + nb) : nullptr;
  const float c_f = (float)sp.c_puct;
  const float keep_f = (float)(1.0 - sp.explore);
  Key128 key = rules.key(s);
  int node = ht_lookup1(ht, dm.hash_cap, gen, key, khi);
  int depth = 0, kind = KIND_EXPAND;
  float term_value = 0.0f;
  uint32_t* path = e.d_path + di * dm.max_depth;
  while (node >= 0) {
    const size_t row = (nb + (size_t)node) * dm.RS;  // the record [N | W | P | C]: 16 * ROWV consecutive words
    int n_loc[ROWV * 4], c_loc[ROWV * 4];
    float w_loc[ROWV * 4], p_loc[ROWV * 4];
#pragma unroll
    for (int v = 0; v < ROWV; ++v) {
      const int4 nv = reinterpret_cast<const int4*>(e.N + row)[v];
      const float4 wv = reinterpret_cast<const float4*>(e.W + row)[v];
      const float4 pv = reinterpret_cast<const float4*>(e.P + row)[v];
      const int4 cv = reinterpret_cast<const int4*>(e.C + row)[v];
      n_loc[4 * v] = nv.x; n_loc[4 * v + 1] = nv.y; n_loc[4 * v + 2] = nv.z; n_loc[4 * v + 3] = nv.w;
      w_loc[4 * v] = wv.x; w_loc[4 * v + 1] = wv.y; w_loc[4 * v + 2] = wv.z; w_loc[4 * v + 3] = wv.w;
      p_loc[4 * v] = pv.x; p_loc[4 * v + 1] = pv.y; p_loc[4 * v + 2] = pv.z; p_loc[4 * v + 3] = pv.w;
      c_loc[4 * v] = cv.x; c_loc[4 * v + 1] = cv.y; c_loc[4 * v + 2] = cv.z; c_loc[4 * v + 3] = cv.w;
    }
    unsigned net_bits = 0u;  // bit a: W(s,a) has absorbed a float32 value (bit 31 of the N word)
    unsigned loss_m = 0u;    // bit a: a LOSS edge (solver)
    int sum_n = 0;
    if (sol) {
      bool win = false, all_loss = true, all_proven = true, draw = false;
#pragma unroll
      for (int a = 0; a < ROWV * 4; ++a) {
        if (a < A && rules.legal(s, a)) {
          const int pf = (n_loc[a] >> kProofShift) & 3;
          win = win || pf == PROOF_WIN;
          draw = draw || pf == PROOF_DRAW;
          all_loss = all_loss && pf == PROOF_LOSS;
          all_proven = all_proven && pf != PROOF_UNKNOWN;
          loss_m |= (pf == PROOF_LOSS ? 1u : 0u) << a;
        }
      }
      const int st = proof_status(win, all_loss, all_proven, draw);
      if (st != PROOF_UNKNOWN) {
        if (depth == 0) {  // proven root: no descent
          store_desc_skip(e.desc + di);
          return;
        }
        kind = KIND_TERMINAL;
        term_value = proof_value(st);
        atomicAdd(e.solver_ctr + SCTR_STOPPED, 1ull);
        break;
      }
    }
#pragma unroll
    for (int a = 0; a < ROWV * 4; ++a) {
      net_bits |= (n_loc[a] < 0 ? 1u : 0u) << a;
      n_loc[a] &= kCountMask;
      sum_n += (a < A) ? n_loc[a] : 0;
    }
    double best = -INFINITY;
    int best_a = 0, best_c = -1;
    if (GUMBEL && depth == 0 && forced >= 0) {
      best_a = forced;
#pragma unroll
      for (int a = 0; a < ROWV * 4; ++a)
        if (a == forced) best_c = c_loc[a];
    } else if (depth == 0) {  // root: Dirichlet noise + float64 scores (lib/mcts.py:48-62,131-132)
      const double sq = sqrt((double)sum_n);
      const double* z = noise_in + ((size_t)g * batch + j) * A;
#pragma unroll
      for (int a = 0; a < ROWV * 4; ++a) {
        if (a < A && rules.legal(s, a) && !((loss_m >> a) & 1u)) {
          const double pn = __dadd_rn((double)__fmul_rn(keep_f, p_loc[a]), __dmul_rn(sp.explore, z[a]));
          const double u = __ddiv_rn(__dmul_rn(__dmul_rn(sp.c_puct, pn), sq), (double)(1 + n_loc[a]));
          // Q keeps python-float (float64) precision until a float32 value touched W(s,a)
          double q64 = 0.0;
          if (n_loc[a] > 0)
            q64 = ((net_bits >> a) & 1u) ? (double)__fdiv_rn(w_loc[a], (float)n_loc[a])
                                         : __ddiv_rn((double)w_loc[a], (double)n_loc[a]);
          const double sc = __dadd_rn(q64, u);
          if (sc > best) {
            best = sc;
            best_a = a;
            best_c = c_loc[a];
          }
        }
      }
    } else {  // interior: float32 scores (lib/mcts.py:64-84 under NEP 50)
      const float sq = __fsqrt_rn((float)sum_n);
      float bestf = -INFINITY;
#pragma unroll
      for (int a = 0; a < ROWV * 4; ++a) {
        if (a < A && rules.legal(s, a) && !((loss_m >> a) & 1u)) {
          const float t = __fdiv_rn(__fmul_rn(__fmul_rn(c_f, p_loc[a]), sq), (float)(1 + n_loc[a]));
          const float q = n_loc[a] > 0 ? __fdiv_rn(w_loc[a], (float)n_loc[a]) : 0.0f;  // value_avg, lib/mcts.py:244
          const float sc = __fadd_rn(q, t);
          if (sc > bestf) {
            bestf = sc;
            best_a = a;
            best_c = c_loc[a];
          }
        }
      }
    }
    const int a = best_a;
    path[depth] = ((uint32_t)node << 8) | (uint32_t)a;
    ++depth;
    const bool won = rules.apply(s, a, who);
    who ^= 1;
    if (won) {
      kind = KIND_TERMINAL;
      term_value = -1.0f;
      break;
    }
    if (!rules.any_legal(s)) {
      kind = KIND_TERMINAL;
      term_value = 0.0f;
      break;
    }
    key = rules.key(s);
    if (best_c >= 0) {
      node = best_c;
    } else {
      node = ht_lookup1(ht, dm.hash_cap, gen, key, khi);
      if (node >= 0) e.C[row + a] = node;
    }
  }
  store_desc(e.desc + di, kind, who, depth, term_value, key, s);
}

template <class R, int ROWV, bool SOLVER, bool GUMBEL>
__global__ void __launch_bounds__(128)
select_thread_kernel(View<typename R::Board> e, R rules, Dims dm, SearchParams sp, int batch,
                     const double* __restrict__ noise_in) {
  const long long grp = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (grp == 0) *e.leaf_count = 0;  // plan_kernel (next launch on the stream) accumulates into it
  select_thread_body<R, ROWV, SOLVER, GUMBEL>(e, rules, dm, sp, batch, noise_in, grp);
}

// The same descent with at most 64 registers (8 blocks per SM instead of 5): for launches of more descents than fit the
// GPU at once, where the number of resident warps, not the latency of one descent, sets the kernel's duration.
template <class R, int ROWV, int BPS, bool SOLVER, bool GUMBEL>
__global__ void __launch_bounds__(128, BPS)
select_thread_dense_kernel(View<typename R::Board> e, R rules, Dims dm, SearchParams sp, int batch,
                           const double* __restrict__ noise_in) {
  const long long grp = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (grp == 0) *e.leaf_count = 0;
  select_thread_body<R, ROWV, SOLVER, GUMBEL>(e, rules, dm, sp, batch, noise_in, grp);
}

// ------------------------------------------------------------- select with virtual loss (extension)
// CARO_FLAG_VIRTUAL_LOSS (not in the reference; SURVEY.md section 8f-4).  The reference's `batch` descents of a minibatch
// all see the same frozen tree and differ only through the root noise, so ~70 % of them end on a leaf another descent of
// the same minibatch has already planned and are dropped (lib/mcts.py:273-278).  Here the descents of a game are made ONE
// AFTER THE OTHER by one thread, and an edge (s, a) that k earlier descents of this minibatch went through is scored as if
// it had k more visits that all lost: N + k, W - k, sum N + k in the PUCT formula.  The virtual visits are a pure function
// of the earlier paths (re-read from the path records of this minibatch), the tree itself is not touched, so plan and
// expand+backup run unchanged and nothing has to be undone.  Same arithmetic as select_thread_body otherwise (float64 at
// the noisy root, float32 below); works for any action count (the rows are read action by action).
template <class R>
__global__ void __launch_bounds__(64)
select_vl_kernel(View<typename R::Board> e, R rules, Dims dm, SearchParams sp, int batch, const double* __restrict__ noise_in) {
  using Board = typename R::Board;
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g == 0) *e.leaf_count = 0;
  if (g >= dm.G) return;
  const size_t d0 = (size_t)g * dm.B;
  if (e.status[g] != ST_ACTIVE) {
    for (int j = 0; j < batch; ++j) store_desc_skip(e.desc + d0 + j);
    return;
  }
  const int A = dm.A;
  const Board root = e.root_board[g];
  const int root_who = e.root_player[g];
  const int tree = g * dm.tpg + (dm.tpg == 2 ? root_who : 0);
  const uint32_t gen = e.tree_gen[tree];
  const HashSlot* ht = e.ht + (size_t)tree * dm.hash_cap;
  const size_t nb = (size_t)tree * dm.node_cap;
  const uint64_t* khi = RulesTraits<R>::kHasKeyHi ? (e.key_hi + nb) : nullptr;
  const float c_f = (float)sp.c_puct;
  const float keep_f = (float)(1.0 - sp.explore);
  const int root_node = ht_lookup1(ht, dm.hash_cap, gen, rules.key(root), khi);
  int lens[32];  // path lengths of this minibatch's earlier descents (batch <= 32)
  for (int j = 0; j < batch; ++j) {
    Board s = root;
    int who = root_who;
    Key128 key = rules.key(s);
    int node = root_node, depth = 0, kind = KIND_EXPAND;
    float term_value = 0.0f;
    uint32_t* path = e.d_path + (d0 + j) * dm.max_depth;
    while (node >= 0) {
      // virtual visits at this node: the edges earlier descents took from it (a position sits at one depth only)
      int va[32], nv = 0;
      for (int i = 0; i < j; ++i)
        if (lens[i] > depth) {
          const uint32_t pe = e.d_path[(d0 + i) * dm.max_depth + depth];
          if ((int)(pe >> 8) == node) va[nv++] = (int)(pe & 0xffu);
        }
      const size_t row = (nb + (size_t)node) * dm.RS;
      int sum_n = nv;
      for (int a = 0; a < A; ++a) sum_n += e.N[row + a] & kCountMask;
      double best = -INFINITY;
      int best_a = 0;
      const double sq64 = sqrt((double)sum_n);
      const float sq32 = __fsqrt_rn((float)sum_n);
      const double* z = noise_in + ((size_t)g * batch + j) * A;
      for (int a = 0; a < A; ++a) {
        if (!rules.legal(s, a)) continue;
        int k = 0;
        for (int i = 0; i < nv; ++i) k += va[i] == a ? 1 : 0;
        const int n = (e.N[row + a] & kCountMask) + k;
        const float w = e.W[row + a] - (float)k;
        const float p = e.P[row + a];
        double sc;
        if (depth == 0) {
          const double pn = __dadd_rn((double)__fmul_rn(keep_f, p), __dmul_rn(sp.explore, z[a]));
          const double u = __ddiv_rn(__dmul_rn(__dmul_rn(sp.c_puct, pn), sq64), (double)(1 + n));
          sc = __dadd_rn(n > 0 ? (double)__fdiv_rn(w, (float)n) : 0.0, u);
        } else {
          const float t = __fdiv_rn(__fmul_rn(__fmul_rn(c_f, p), sq32), (float)(1 + n));
          sc = (double)__fadd_rn(n > 0 ? __fdiv_rn(w, (float)n) : 0.0f, t);
        }
        if (sc > best) {
          best = sc;
          best_a = a;
        }
      }
      const int a = best_a;
      path[depth] = ((uint32_t)node << 8) | (uint32_t)a;
      ++depth;
      const bool won = rules.apply(s, a, who);
      who ^= 1;
      if (won) {
        kind = KIND_TERMINAL;
        term_value = -1.0f;
        break;
      }
      if (!rules.any_legal(s)) {
        kind = KIND_TERMINAL;
        term_value = 0.0f;
        break;
      }
      key = rules.key(s);
      const int linked = e.C[row + a];
      if (linked >= 0) {
        node = linked;
      } else {
        node = ht_lookup1(ht, dm.hash_cap, gen, key, khi);
        if (node >= 0) e.C[row + a] = node;
      }
    }
    lens[j] = depth;
    store_desc(e.desc + d0 + j, kind, who, depth, term_value, key, s);
  }
}

// The same search with eight lanes per game (A <= 8: Connect4), lane = action: the descents of a game are still made one after
// the other (that is what virtual loss means), but every level of a descent is one coalesced 128-byte record load and a
// three-step shuffle argmax instead of a serial loop over the actions, and eight times as many warps are in flight -- the
// one-thread-per-game kernel left 64 warps per 8,192 games, and IT, not the tower, set the pace of the extension mode.
// Identical choices to select_vl_kernel (same arithmetic per action, first maximum = lowest action).
template <class R>
__global__ void __launch_bounds__(256)
select_vl_group_kernel(View<typename R::Board> e, R rules, Dims dm, SearchParams sp, int batch, const double* __restrict__ noise_in) {
  using Board = typename R::Board;
  constexpr int GW = 8;
  const int gthread = blockIdx.x * blockDim.x + threadIdx.x;
  if (gthread == 0) *e.leaf_count = 0;
  const int g = gthread / GW;
  if (g >= dm.G) return;  // whole groups leave together (blockDim is a multiple of GW)
  const int gl = threadIdx.x & (GW - 1);
  const unsigned gmask = group_mask<GW>();
  const int gbase = (threadIdx.x & 31) & ~(GW - 1);
  const size_t d0 = (size_t)g * dm.B;
  if (e.status[g] != ST_ACTIVE) {
    for (int j = gl; j < batch; j += GW) store_desc_skip(e.desc + d0 + j);
    return;
  }
  const int A = dm.A;
  const Board root = e.root_board[g];
  const int root_who = e.root_player[g];
  const int tree = g * dm.tpg + (dm.tpg == 2 ? root_who : 0);
  const uint32_t gen = e.tree_gen[tree];
  const HashSlot* ht = e.ht + (size_t)tree * dm.hash_cap;
  const size_t nb = (size_t)tree * dm.node_cap;
  const uint64_t* khi = RulesTraits<R>::kHasKeyHi ? (e.key_hi + nb) : nullptr;
  const float c_f = (float)sp.c_puct;
  const float keep_f = (float)(1.0 - sp.explore);
  const int root_node = ht_lookup<GW>(ht, dm.hash_cap, gen, rules.key(root), khi, gl, gmask);
  const bool mine = gl < A;
  int len_reg = 0;  // lane i keeps the path length of descent i (batch <= 8) -- descents 8.. are looked up in the records
  for (int j = 0; j < batch; ++j) {
    Board s = root;
    int who = root_who;
    Key128 key = rules.key(s);
    int node = root_node, depth = 0, kind = KIND_EXPAND;
    float term_value = 0.0f;
    uint32_t* path = e.d_path + (d0 + j) * dm.max_depth;
    while (node >= 0) {
      const size_t row = (nb + (size_t)node) * dm.RS;
      // virtual visits of MY edge: earlier descents of this minibatch that went through (node, action = lane)
      int k = 0;
      for (int i = 0; i < j; ++i) {
        const int len_i = i < GW ? __shfl_sync(gmask, len_reg, gbase + i) : (int)e.desc[d0 + i].h.len;
        if (len_i > depth) {
          const uint32_t pe = e.d_path[(d0 + i) * dm.max_depth + depth];
          if ((int)(pe >> 8) == node) k += ((int)(pe & 0xffu) == gl) ? 1 : 0;
        }
      }
      int n = 0, c_link = -1;
      float w = 0.0f, p = 0.0f;
      if (mine) {
        n = (e.N[row + gl] & kCountMask) + k;
        w = e.W[row + gl] - (float)k;
        p = e.P[row + gl];
        c_link = e.C[row + gl];
      }
      int sum_n = mine ? n : 0;
#pragma unroll
      for (int off = GW / 2; off > 0; off >>= 1) sum_n += __shfl_xor_sync(gmask, sum_n, off);
      double sc = -INFINITY;
      if (mine && rules.legal(s, gl)) {
        if (depth == 0) {
          const double z = noise_in[((size_t)g * batch + j) * A + gl];
          const double pn = __dadd_rn((double)__fmul_rn(keep_f, p), __dmul_rn(sp.explore, z));
          const double u = __ddiv_rn(__dmul_rn(__dmul_rn(sp.c_puct, pn), sqrt((double)sum_n)), (double)(1 + n));
          sc = __dadd_rn(n > 0 ? (double)__fdiv_rn(w, (float)n) : 0.0, u);
        } else {
          const float t = __fdiv_rn(__fmul_rn(__fmul_rn(c_f, p), __fsqrt_rn((float)sum_n)), (float)(1 + n));
          sc = (double)__fadd_rn(n > 0 ? __fdiv_rn(w, (float)n) : 0.0f, t);
        }
      }
      int best_a = gl;
#pragma unroll
      for (int off = GW / 2; off > 0; off >>= 1) {
        const double ob = __shfl_xor_sync(gmask, sc, off);
        const int oa = __shfl_xor_sync(gmask, best_a, off);
        if (ob > sc || (ob == sc && oa < best_a)) {
          sc = ob;
          best_a = oa;
        }
      }
      const int a = best_a;
      if (gl == 0) path[depth] = ((uint32_t)node << 8) | (uint32_t)a;
      ++depth;
      const bool won = rules.apply(s, a, who);
      who ^= 1;
      if (won) {
        kind = KIND_TERMINAL;
        term_value = -1.0f;
        break;
      }
      if (!rules.any_legal(s)) {
        kind = KIND_TERMINAL;
        term_value = 0.0f;
        break;
      }
      key = rules.key(s);
      const int linked = __shfl_sync(gmask, c_link, gbase + a);
      if (linked >= 0) {
        node = linked;
      } else {
        node = ht_lookup<GW>(ht, dm.hash_cap, gen, key, khi, gl, gmask);
        if (node >= 0 && gl == 0) e.C[row + a] = node;
      }
    }
    if (gl == (j & (GW - 1)) && j < GW) len_reg = depth;
    if (gl == 0) store_desc(e.desc + d0 + j, kind, who, depth, term_value, key, s);
    __syncwarp(gmask);  // the path and the record of this descent are read by the whole group from the next descent on
  }
}

// ------------------------------------------------------------------------------------ plan
// Back-up queue = terminal descents in descent order, then the first occurrence of every distinct new leaf
// (lib/mcts.py:265-278); unique leaves are appended to the compact batch (order across games is arbitrary; results do
// not depend on it).  GP lanes per game (batch <= GP <= 32), lane j owns descent j, so every load of the per-descent
// records is issued at once instead of as a dependent chain.
template <class Board, int GP>
__device__ __forceinline__ void plan_body(const View<Board>& e, const Dims& dm, int batch, int gthread) {
  const int g = gthread / GP;
  const int j = threadIdx.x & (GP - 1);
  const int lane = threadIdx.x & 31;
  const int gbase = lane & ~(GP - 1);
  const unsigned gmask = group_mask<GP>();
  const bool in_range = g < dm.G;
  const bool live = in_range && e.status[g] == ST_ACTIVE;
  const size_t d0 = (size_t)(in_range ? g : 0) * dm.B;
  int kind = KIND_SKIP, len = 0;
  uint64_t lo = 0, hi = 0;
  float tval = 0.0f;
  if (live && j < batch) {
    const DescHead h = e.desc[d0 + j].h;  // one 32-byte sector
    kind = h.kind;
    len = h.len;
    tval = h.value;
    lo = h.key_lo;
    hi = h.key_hi;
  }
  const unsigned below = (1u << j) - 1u;
  const unsigned term_m = (__ballot_sync(gmask, kind == KIND_TERMINAL) >> gbase) & ((GP == 32) ? 0xffffffffu : ((1u << GP) - 1u));
  bool dup = false;
#pragma unroll
  for (int i = 0; i < GP; ++i) {
    const uint64_t olo = __shfl_sync(gmask, lo, gbase + i);
    const uint64_t ohi = __shfl_sync(gmask, hi, gbase + i);
    const int okind = __shfl_sync(gmask, kind, gbase + i);
    dup = dup || (i < j && okind == KIND_EXPAND && olo == lo && ohi == hi);
  }
  const bool uniq = kind == KIND_EXPAND && !dup;
  const unsigned uniq_m = (__ballot_sync(gmask, uniq) >> gbase) & ((GP == 32) ? 0xffffffffu : ((1u << GP) - 1u));
  const int n_term = __popc(term_m), n_new = __popc(uniq_m);
  // reservation in the compact leaf batch: ONE global atomic per block of 256 threads (warp prefix sums, the warps' totals meet in
  // shared memory).  One atomic per warp plus two counter updates per game on the same three addresses were what the
  // kernel's time consisted of at 64 k games (~150 k same-address atomics at ~0.45 ns each = 66 us for 25 MB of traffic).
  __shared__ int s_warp_total[8], s_block_base;
  __shared__ unsigned long long s_leaves, s_descents;
  const int warp_in_block = threadIdx.x >> 5;
  if (threadIdx.x == 0) {
    s_leaves = 0ull;
    s_descents = 0ull;
  }
  int base = 0;
  const int mine = (j == 0) ? n_new : 0;
  int incl = mine;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, off);
    if (lane >= off) incl += v;
  }
  if (lane == 31) s_warp_total[warp_in_block] = incl;
  __syncthreads();
  if (threadIdx.x == 0) {
    int total = 0;
    for (int w = 0; w < 8; ++w) {
      const int t = s_warp_total[w];
      s_warp_total[w] = total;  // exclusive prefix over the block's warps
      total += t;
    }
    s_block_base = total > 0 ? atomicAdd(e.leaf_count, total) : 0;
  }
  __syncthreads();
  base = __shfl_sync(0xffffffffu, s_block_base + s_warp_total[warp_in_block] + incl - mine, gbase);  // exclusive prefix at the group leader
  if (in_range && j == 0) {
    e.q_len[g] = live ? n_term + n_new : 0;
    if (live) {
      if (n_new) atomicAdd(&s_leaves, (unsigned long long)n_new);
      atomicAdd(&s_descents, (unsigned long long)batch);
    }
  }
  if (live) {
    if (kind == KIND_TERMINAL) {
      e.q_entry[d0 + __popc(term_m & below)] = QEntry{(uint8_t)j, (uint8_t)KIND_TERMINAL, (uint16_t)len, __float_as_int(tval)};
    } else if (uniq) {
      const int r = __popc(uniq_m & below);
      const int slot = base + r;
      e.q_entry[d0 + n_term + r] = QEntry{(uint8_t)j, (uint8_t)KIND_EXPAND, (uint16_t)len, slot};
      e.desc[d0 + j].h.slot = slot;
      e.leaf_board[slot] = e.desc[d0 + j].board;
      e.leaf_player[slot] = e.desc[d0 + j].h.player;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (s_leaves) atomicAdd(e.ctr + CTR_LEAVES, s_leaves);
    if (s_descents) atomicAdd(e.ctr + CTR_DESCENTS, s_descents);
  }
}

template <class Board, int GP>
__global__ void __launch_bounds__(256)
plan_kernel(View<Board> e, Dims dm, int batch) {
  plan_body<Board, GP>(e, dm, batch, blockIdx.x * blockDim.x + threadIdx.x);
}

// --------------------------------------------------------------------------- expand + backup
// Claim a hash slot for `key_lo` with a CAS on the generation word, so that the (<= batch) insertions of one
// minibatch can proceed concurrently from different lanes.  Keys of one minibatch are distinct (plan dedup).
__device__ __forceinline__ void ht_insert_cas(HashSlot* __restrict__ ht, int cap, uint32_t gen, uint64_t key_lo, int node) {
  uint32_t idx = slot_home(key_lo, cap);
  for (int it = 0; it < cap; ++it) {
    uint32_t* gword = reinterpret_cast<uint32_t*>(ht + idx) + 3;
    const uint32_t seen = *gword;
    if (seen != gen && atomicCAS(gword, seen, gen) == seen) {
      ht[idx].key = key_lo;
      ht[idx].node = node;
      return;
    }
    idx = (idx + 1u) & (uint32_t)(cap - 1);
  }
}

// Batched variant (batch <= BK <= 32).  One warp per game.
//   phase 1: lane q owns queue entry q: its metadata chain (order -> kind/slot/value/path length) is loaded by all
//            lanes at once; new nodes get their arena index by a warp prefix sum and their hash slot by CAS;
//   phase 2: lane i owns path depth i (an edge always sits at the same depth, hence on the same lane): it loads
//            N/W of its edge in EVERY queued path up front, then replays the queue IN ORDER in registers
//            (float32 W sums are order dependent), forwarding values between entries that hit the same edge,
//            and stores each distinct edge once.
//   solver (SOLVER and the solver on for the root player): after phase 2, in queue order, every terminal entry proves its
//            last edge (leaf value -1: WIN, 0: DRAW, +1: LOSS, for the edge's mover) and walks up its own path while the
//            node above is proven, setting the next edge to the negated status.  The order decides which parent of a
//            transposition learns first.
template <class R, int BK, int GW = 32, bool SOLVER = false>  // GW lanes per game (BK <= GW): 32 = one warp per game, 8 = four games per warp
__device__ __forceinline__ void expand_backup_body(const View<typename R::Board>& e, const Dims& dm, int batch,
                                                   const float* __restrict__ probs, const float* __restrict__ values, int g,
                                                   int lane32) {
  static_assert(BK <= GW, "one lane per queue entry");
  const int lane = lane32 & (GW - 1);           // lane within the game's group
  const int gbase = lane32 & ~(GW - 1);         // first warp lane of the group
  const unsigned gmask = group_mask<GW>();
  if (g >= dm.G || e.status[g] != ST_ACTIVE) return;
  const int who0 = e.root_player[g];
  const int tree = g * dm.tpg + (dm.tpg == 2 ? who0 : 0);
  const uint32_t gen = e.tree_gen[tree];
  HashSlot* ht = e.ht + (size_t)tree * dm.hash_cap;
  const size_t nb = (size_t)tree * dm.node_cap;
  const size_t d0 = (size_t)g * dm.B;
  const int qn = e.q_len[g];
  const int count0 = e.node_count[tree];
  // ---- phase 1 -------------------------------------------------------------------------------------
  int my_di = 0, my_kind = KIND_SKIP, my_slot = -1, my_len = 0;
  float my_val = 0.0f;
  if (lane < qn) {  // the queue entry carries everything: no order -> kind -> slot chain of dependent loads
    const QEntry q = e.q_entry[d0 + lane];
    my_di = q.j;
    my_kind = q.kind;
    my_len = q.len;
    if (my_kind == KIND_EXPAND) {
      my_slot = q.slot;
      my_val = values[my_slot];
    } else {
      my_val = __int_as_float(q.slot);
    }
  }
  const unsigned exp_m = (__ballot_sync(gmask, my_kind == KIND_EXPAND) >> gbase) & (GW == 32 ? 0xffffffffu : ((1u << GW) - 1u));
  const int n_new = __popc(exp_m);
  int my_node = count0 + __popc(exp_m & ((1u << lane) - 1u));
  const bool creates = my_kind == KIND_EXPAND && my_node < dm.node_cap;
  if (my_kind == KIND_EXPAND && !creates) atomicOr(e.ctr + CTR_ERRORS, ERR_ARENA_FULL);
  if (creates) {  // _create_node, lib/mcts.py:178-190 (scalars + hash slot by the owning lane)
    const DescRec<typename R::Board>* rec = e.desc + d0 + my_di;
    const DescHead h = rec->h;
    e.node_board[nb + my_node] = rec->board;
    e.node_player[nb + my_node] = h.player;
    if (RulesTraits<R>::kHasKeyHi) e.key_hi[nb + my_node] = h.key_hi;
    ht_insert_cas(ht, dm.hash_cap, gen, h.key_lo, my_node);
  }
  // rows of the new nodes, all lanes cooperating
  for (int q = 0; q < qn; ++q) {
    const bool cr = __shfl_sync(gmask, (int)creates, gbase + q) != 0;
    if (!cr) continue;
    const int node = __shfl_sync(gmask, my_node, gbase + q);
    const int slot = __shfl_sync(gmask, my_slot, gbase + q);
    const size_t row = (nb + (size_t)node) * dm.RS;
    float denom = 1.0f;
    const bool mask = (dm.flags & FLAG_MASK_PRIORS) != 0u;
    typename R::Board nboard;
    if (mask) {  // extension: priors of illegal moves zeroed, the rest renormalised (the reference keeps the raw softmax)
      const int di = __shfl_sync(gmask, my_di, gbase + q);
      nboard = e.desc[d0 + di].board;
      const R legality{};
      float part = 0.0f;
      for (int a = lane; a < dm.A; a += GW)
        if (legality.legal(nboard, a)) part += probs[(size_t)slot * dm.A + a];
#pragma unroll
      for (int off = GW / 2; off > 0; off >>= 1) part += __shfl_xor_sync(gmask, part, off);
      denom = part > 0.0f ? part : 1.0f;  // no legal mass: the legal priors are all 0 and stay 0
    }
    for (int a = lane; a < dm.Apad; a += GW) {
      e.N[row + a] = 0;
      e.W[row + a] = 0.0f;
      float p = (a < dm.A) ? probs[(size_t)slot * dm.A + a] : 0.0f;
      // a division, not p * (1 / part): correctly rounded, and a lone legal move gets exactly 1
      if (mask && a < dm.A) p = R{}.legal(nboard, a) ? __fdiv_rn(p, denom) : 0.0f;
      e.P[row + a] = p;
      e.C[row + a] = -1;
    }
  }
  if (lane == 0) e.node_count[tree] = min(count0 + n_new, dm.node_cap);
  // ---- phase 2: _backup, lib/mcts.py:225-246 ---------------------------------------------------------
  int max_len = my_len;
#pragma unroll
  for (int off = GW / 2; off > 0; off >>= 1) max_len = max(max_len, __shfl_xor_sync(gmask, max_len, off));
  for (int i0 = 0; i0 < max_len; i0 += GW) {
    const int i = i0 + lane;
    long long idx[BK];
    int n_v[BK], net[BK];
    float w_v[BK], cur[BK];
#pragma unroll
    for (int q = 0; q < BK; ++q) {
      const int di = __shfl_sync(gmask, my_di, gbase + q);
      const int len = __shfl_sync(gmask, my_len, gbase + q);
      const float v = __shfl_sync(gmask, my_val, gbase + q);
      const int kind = __shfl_sync(gmask, my_kind, gbase + q);
      idx[q] = -1;
      n_v[q] = 0;
      net[q] = 0;
      w_v[q] = 0.0f;
      cur[q] = 0.0f;
      if (q < qn && i < len) {
        const uint32_t pe = e.d_path[(d0 + di) * dm.max_depth + i];
        const int node = (int)(pe >> 8);
        const int a = (int)(pe & 0xffu);
        idx[q] = (long long)((nb + (size_t)node) * dm.RS + a);
        n_v[q] = e.N[idx[q]];
        w_v[q] = e.W[idx[q]];
        cur[q] = ((len - 1 - i) & 1) ? v : -v;
        net[q] = kind == KIND_EXPAND ? kNetBit : 0;
      }
    }
#pragma unroll
    for (int q = 0; q < BK; ++q) {
      if (idx[q] < 0) continue;
#pragma unroll
      for (int p = 0; p < q; ++p)
        if (idx[p] == idx[q]) {  // latest earlier entry on the same edge wins (p ascending)
          n_v[q] = n_v[p];
          w_v[q] = w_v[p];
        }
      n_v[q] = (n_v[q] + 1) | net[q];  // the count lives in bits 0..30, so the +1 never reaches the flag bit
      w_v[q] = __fadd_rn(w_v[q], cur[q]);
    }
#pragma unroll
    for (int q = 0; q < BK; ++q) {
      if (idx[q] < 0) continue;
      bool last = true;
#pragma unroll
      for (int p = q + 1; p < BK; ++p) last = last && (idx[p] != idx[q]);
      if (last) {
        e.N[idx[q]] = n_v[q];
        e.W[idx[q]] = w_v[q];
      }
    }
  }
  if (SOLVER && solver_on(e, who0)) {
    __syncwarp(gmask);  // phase 2's N words are visible to the whole group
    unsigned long long proven = 0ull;
    for (int q = 0; q < qn; ++q) {
      if (__shfl_sync(gmask, my_kind, gbase + q) != KIND_TERMINAL) continue;
      const int di = __shfl_sync(gmask, my_di, gbase + q);
      const int len = __shfl_sync(gmask, my_len, gbase + q);
      const float v = __shfl_sync(gmask, my_val, gbase + q);
      int st = v < 0.0f ? PROOF_WIN : (v > 0.0f ? PROOF_LOSS : PROOF_DRAW);
      for (int i = len - 1; i >= 0; --i) {
        const uint32_t pe = e.d_path[(d0 + di) * dm.max_depth + i];
        const size_t row = (nb + (size_t)(pe >> 8)) * dm.RS;
        if (lane == 0) {
          const int old = e.N[row + (pe & 0xffu)];
          proven += (old & kProofMask) ? 0ull : 1ull;
          e.N[row + (pe & 0xffu)] = (old & ~kProofMask) | (st << kProofShift);
        }
        __syncwarp(gmask);
        const typename R::Board b = e.node_board[nb + (pe >> 8)];
        bool win = false, all_loss = true, all_proven = true, draw = false;
        for (int a = lane; a < dm.A; a += GW) {
          if (R{}.legal(b, a)) {
            const int pf = (e.N[row + a] >> kProofShift) & 3;
            win = win || pf == PROOF_WIN;
            draw = draw || pf == PROOF_DRAW;
            all_loss = all_loss && pf == PROOF_LOSS;
            all_proven = all_proven && pf != PROOF_UNKNOWN;
          }
        }
        const int ns = proof_status(__any_sync(gmask, win), __all_sync(gmask, all_loss), __all_sync(gmask, all_proven),
                                    __any_sync(gmask, draw));
        if (ns == PROOF_UNKNOWN) break;
        st = proof_negate(ns);
      }
    }
    if (lane == 0 && proven) atomicAdd(e.solver_ctr + SCTR_PROVEN, proven);
  }
}

template <class R, int BK, bool SOLVER>
__global__ void __launch_bounds__(128)
expand_backup_kernel(View<typename R::Board> e, Dims dm, int batch, const float* __restrict__ probs,
                     const float* __restrict__ values) {
  expand_backup_body<R, BK, 32, SOLVER>(e, dm, batch, probs, values, (blockIdx.x * blockDim.x + threadIdx.x) >> 5, threadIdx.x & 31);
}

// Eight lanes per game (action rows of <= 8 entries, batch <= 8: Connect4): four games per warp, a quarter of the warps of
// the warp-per-game kernel for the same work.  The tree kernels of the self-play pipeline run in the few warp slots
// a tower CTA leaves free (+ 16 SMs of their own), where the number of warps, not the work, sets their time.
template <class R, bool SOLVER>
__global__ void __launch_bounds__(128)
expand_backup_group8_kernel(View<typename R::Board> e, Dims dm, int batch, const float* __restrict__ probs,
                            const float* __restrict__ values) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  expand_backup_body<R, 8, 8, SOLVER>(e, dm, batch, probs, values, t >> 3, threadIdx.x & 31);
}

// ------------------------------------------------------------------------------ root policy
// MCTS.get_policy_value (lib/mcts.py:289-313).  One thread per game.
template <class R>
__device__ __forceinline__ int root_node_of(const View<typename R::Board>& e, const R& rules, const Dims& dm, int g,
                                            size_t* nb_out) {
  const int who = e.root_player[g];
  const int tree = g * dm.tpg + (dm.tpg == 2 ? who : 0);
  const size_t nb = (size_t)tree * dm.node_cap;
  *nb_out = nb;
  const Key128 key = rules.key(e.root_board[g]);
  return ht_lookup1(e.ht + (size_t)tree * dm.hash_cap, dm.hash_cap, e.tree_gen[tree], key,
                    RulesTraits<R>::kHasKeyHi ? (e.key_hi + nb) : nullptr);
}

// Solver at the root (extension): the lowest WIN edge of a proven-WIN root (-1 = none), and whether LOSS edges are left
// out of pi and the move (they are, unless that leaves no visit).  Without the solver for the root player: (-1, false).
struct RootProof {
  int win_a;
  bool drop_loss;
};
template <class R>
__device__ __forceinline__ RootProof root_proof(const View<typename R::Board>& e, const R& rules, const Dims& dm, int g,
                                                size_t row) {
  RootProof rp{-1, false};
  if (!solver_on(e, e.root_player[g])) return rp;
  const typename R::Board s = e.root_board[g];
  long long kept = 0;
  for (int a = dm.A - 1; a >= 0; --a) {
    const int raw = e.N[row + a];
    const int pf = (raw >> kProofShift) & 3;
    if (pf == PROOF_WIN && rules.legal(s, a)) rp.win_a = a;
    if (pf != PROOF_LOSS) kept += raw & kCountMask;
  }
  rp.drop_loss = kept > 0;
  return rp;
}
// visit count of edge a as pi and the move see it
__device__ __forceinline__ int pi_count(int raw, const RootProof& rp) {
  return (rp.drop_loss && ((raw >> kProofShift) & 3) == PROOF_LOSS) ? 0 : (raw & kCountMask);
}

// ---------------------------------------------------------------------------------- Gumbel root search (extension)
// The rule is stated in include/caro_b200.h (caro_engine_set_gumbel) and restated by tests/gumbel_reference.py.  All
// arithmetic is float64, every sum runs in action order, ties go to the lowest action.
template <class Board>
__device__ __forceinline__ bool gumbel_on(const View<Board>& e, int who) { return (e.gumbel_params->players >> who) & 1; }

// Q of a visited root edge as the root branch of select computes it: f32(W / N) once W has absorbed a float32 value,
// else the float64 quotient of the python-float sum
__device__ __forceinline__ double root_edge_q(int raw, float w) {
  const int n = raw & kCountMask;
  return raw < 0 ? (double)__fdiv_rn(w, (float)n) : __ddiv_rn((double)w, (double)n);
}

struct GumbelRoot {
  double scale;  // (c_visit + max_b N(b)) * c_scale
  double qbar;   // completed Q of an unvisited edge: prior-weighted mean Q of the visited legal edges (0: none visited)
};
template <class R>
__device__ GumbelRoot gumbel_root_stats(const View<typename R::Board>& e, const R& rules, const typename R::Board& s, int A,
                                        size_t row, const GumbelParams& gp) {
  int max_n = 0;
  double sp = 0.0, spq = 0.0;
  for (int a = 0; a < A; ++a) {
    if (!rules.legal(s, a)) continue;
    const int raw = e.N[row + a];
    const int n = raw & kCountMask;
    max_n = n > max_n ? n : max_n;
    if (n > 0) {
      const double p = (double)e.P[row + a];
      sp = __dadd_rn(sp, p);
      spq = __dadd_rn(spq, __dmul_rn(p, root_edge_q(raw, e.W[row + a])));
    }
  }
  GumbelRoot gr;
  gr.scale = __dmul_rn(__dadd_rn(gp.c_visit, (double)max_n), gp.c_scale);
  gr.qbar = sp > 0.0 ? __ddiv_rn(spq, sp) : 0.0;
  return gr;
}
// sigma(q^(a)) with q^ = (q + 1) / 2
template <class Board>
__device__ __forceinline__ double gumbel_sigma(const View<Board>& e, size_t row, int a, const GumbelRoot& gr) {
  const int raw = e.N[row + a];
  const double q = (raw & kCountMask) > 0 ? root_edge_q(raw, e.W[row + a]) : gr.qbar;
  return __dmul_rn(gr.scale, __dmul_rn(__dadd_rn(q, 1.0), 0.5));
}
// gumbel_scale * g + log P: the phase-0 score; score = that + sigma; the policy logit = log P + sigma
__device__ __forceinline__ double gumbel_base(double gs, double g, float p) { return __dadd_rn(__dmul_rn(gs, g), log((double)p)); }

// survivors kept by phase p of a search that samples m actions
__device__ __forceinline__ int gumbel_survivors(int m, int p) {
  const int c = (m + (1 << p) - 1) >> p;
  const int r = c > 2 ? c : 2;
  return r < m ? r : m;
}
__device__ __forceinline__ int gumbel_phases(int m) {  // H = ceil(log2 m)
  int h = 0;
  while ((1 << h) < m) ++h;
  return h;
}

// pi' and the move of a Gumbel root, one thread (root_policy_kernel and advance_kernel)
struct GumbelPolicy {
  GumbelRoot gr;
  double lmax, sum;  // largest legal logit; sum over legal actions of exp(logit - lmax), in action order
  int nlegal, move;
};
template <class R>
__device__ GumbelPolicy gumbel_policy(const View<typename R::Board>& e, const R& rules, const Dims& dm, int g, size_t row) {
  const typename R::Board s = e.root_board[g];
  const GumbelParams gp = *e.gumbel_params;
  const int A = dm.A;
  GumbelPolicy out;
  out.gr = gumbel_root_stats<R>(e, rules, s, A, row, gp);
  out.lmax = -INFINITY;
  out.nlegal = 0;
  for (int a = 0; a < A; ++a) {
    if (!rules.legal(s, a)) continue;
    ++out.nlegal;
    const double l = __dadd_rn(log((double)e.P[row + a]), gumbel_sigma(e, row, a, out.gr));
    out.lmax = l > out.lmax ? l : out.lmax;
  }
  out.sum = 0.0;
  if (out.lmax > -INFINITY)
    for (int a = 0; a < A; ++a)
      if (rules.legal(s, a))
        out.sum = __dadd_rn(out.sum, exp(__dsub_rn(__dadd_rn(log((double)e.P[row + a]), gumbel_sigma(e, row, a, out.gr)), out.lmax)));
  // the move: argmax of the score over the current survivors, over every legal action when no phase ran
  const GumbelState* st = e.gumbel_state + g;
  const double* gg = e.gumbel_g + (size_t)g * A;
  const int r = st->phase >= 0 ? st->r : 0;
  double best = 0.0;
  int best_a = -1;
  for (int i = 0; i < (r > 0 ? r : A); ++i) {
    const int a = r > 0 ? st->surv[i] : i;
    if (r == 0 && !rules.legal(s, a)) continue;
    const double sc = __dadd_rn(gumbel_base(gp.gumbel_scale, gg[a], e.P[row + a]), gumbel_sigma(e, row, a, out.gr));
    if (best_a < 0 || sc > best || (sc == best && a < best_a)) {
      best = sc;
      best_a = a;
    }
  }
  out.move = best_a;
  return out;
}
// pi'(a) as stored (float32): softmax over the legal actions of log P + sigma, uniform when every legal logit is -inf
template <class R>
__device__ __forceinline__ float gumbel_pi(const GumbelPolicy& gpol, const View<typename R::Board>& e, const R& rules,
                                           const typename R::Board& s, size_t row, int a) {
  if (!rules.legal(s, a)) return 0.0f;
  if (!(gpol.lmax > -INFINITY)) return (float)__ddiv_rn(1.0, (double)gpol.nlegal);
  const double l = __dadd_rn(log((double)e.P[row + a]), gumbel_sigma(e, row, a, gpol.gr));
  return (float)__ddiv_rn(exp(__dsub_rn(l, gpol.lmax)), gpol.sum);
}

// Before select, one warp per game: at minibatch 0 of a search the draws g and a fresh state; from the first minibatch i0
// at which the root is in the tree, the survivors of the current phase and every descent's forced root action
// (gumbel_root, -1 = PUCT as the reference).  Arguments by value, so a captured ply graph replays it correctly.
template <class R>
__global__ void __launch_bounds__(128)
gumbel_plan_kernel(View<typename R::Board> e, R rules, Dims dm, SearchParams sp, int search_index, int mb, int count,
                   int batch) {
  constexpr int kMaxApl = 8;  // A <= 256
  const int g = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  if (g >= dm.G) return;  // whole warps leave together
  const int A = dm.A;
  int16_t* out = e.gumbel_root + (size_t)g * dm.B;
  GumbelState* st = e.gumbel_state + g;
  const GumbelParams gp = *e.gumbel_params;
  const bool on = e.status[g] == ST_ACTIVE && ((gp.players >> e.root_player[g]) & 1);
  int i0 = -1, phase = -1, kstart = 0, m = 0, r = 0;
  if (mb > 0) {
    i0 = st->i0;
    phase = st->phase;
    kstart = st->kstart;
    m = st->m;
    r = st->r;
  }
  if (on && mb == 0) {
    const uint64_t uid = e.uid[g];
    for (int a = lane; a < A; a += 32)
      e.gumbel_g[(size_t)g * A + a] = gumbel_draw(sp.seed_lo, sp.seed_hi, uid, (uint32_t)search_index, (uint32_t)e.ply[g], (uint32_t)a);
  }
  size_t nb = 0;
  const int node = on ? root_node_of<R>(e, rules, dm, g, &nb) : -1;
  if (node >= 0) {
    const size_t row = (nb + (size_t)node) * dm.RS;
    const typename R::Board s = e.root_board[g];
    const double* gg = e.gumbel_g + (size_t)g * A;
    if (i0 < 0) i0 = mb;
    const int k = mb - i0, cp = count - i0;
    if (phase < 0) {  // phase 0: the top m legal actions by gumbel_scale * g + log P
      double bs[kMaxApl];
      bool lg[kMaxApl];
      int nl = 0, rank[kMaxApl];
#pragma unroll
      for (int i = 0; i < kMaxApl; ++i) {
        const int a = lane + 32 * i;
        lg[i] = a < A && rules.legal(s, a);
        bs[i] = lg[i] ? gumbel_base(gp.gumbel_scale, gg[a], e.P[row + a]) : 0.0;
        nl += lg[i] ? 1 : 0;
        rank[i] = 0;
      }
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) nl += __shfl_xor_sync(0xffffffffu, nl, off);
      m = gp.m < nl ? gp.m : nl;
#pragma unroll
      for (int i2 = 0; i2 < kMaxApl; ++i2) {
        if (32 * i2 >= A) break;
        for (int l = 0; l < 32; ++l) {
          const double ob = __shfl_sync(0xffffffffu, bs[i2], l);
          const int ol = __shfl_sync(0xffffffffu, lg[i2] ? 1 : 0, l);
          const int b = l + 32 * i2;
#pragma unroll
          for (int i = 0; i < kMaxApl; ++i) {
            const int a = lane + 32 * i;
            rank[i] += (ol && (ob > bs[i] || (ob == bs[i] && b < a))) ? 1 : 0;
          }
        }
      }
#pragma unroll
      for (int i = 0; i < kMaxApl; ++i)
        if (lg[i] && rank[i] < m) st->surv[rank[i]] = (int16_t)(lane + 32 * i);
      phase = 0;
      kstart = 0;
      r = m;
      __syncwarp();
    }
    const int H = gumbel_phases(m);
    const int p = (int)(((long long)k * H) / cp);
    if (p != phase) {  // the top r_p of the current survivors by score on the tree as it stands
      const GumbelRoot gr = gumbel_root_stats<R>(e, rules, s, A, row, gp);
      const int rp = gumbel_survivors(m, p);
      const int a = lane < r ? (int)st->surv[lane] : -1;
      const double sc = lane < r ? __dadd_rn(gumbel_base(gp.gumbel_scale, gg[a], e.P[row + a]), gumbel_sigma(e, row, a, gr)) : 0.0;
      int rank = 0;
      for (int l = 0; l < r; ++l) {
        const double ob = __shfl_sync(0xffffffffu, sc, l);
        const int oa = __shfl_sync(0xffffffffu, a, l);
        rank += (ob > sc || (ob == sc && oa < a)) ? 1 : 0;
      }
      __syncwarp();
      if (lane < r && rank < rp) st->surv[rank] = (int16_t)a;
      r = rp;
      phase = p;
      kstart = k;
      __syncwarp();
    }
    for (int j = lane; j < batch; j += 32) out[j] = st->surv[((k - kstart) * batch + j) % r];
  } else {
    for (int j = lane; j < batch; j += 32) out[j] = -1;
  }
  if (lane == 0) {
    st->i0 = i0;
    st->phase = phase;
    st->kstart = kstart;
    st->m = (int16_t)m;
    st->r = (int16_t)r;
  }
}

// GUMBEL (extension): the instance the host launches while the engine's Gumbel mask is non-zero; a Gumbel root gives pi'
// (tau_mode 1 or 2: the tau schedule does not apply) or a one-hot on the Gumbel move (tau_mode 0).
template <class R, bool GUMBEL>
__global__ void root_policy_kernel(View<typename R::Board> e, R rules, Dims dm, int tau_mode, int tau_plies,
                                   double* __restrict__ pi, float* __restrict__ qout, int32_t* __restrict__ nout) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= dm.G) return;
  const int A = dm.A;
  size_t nb;
  const int node = root_node_of<R>(e, rules, dm, g, &nb);
  if (node < 0) {
    for (int a = 0; a < A; ++a) {
      if (pi) pi[(size_t)g * A + a] = 0.0;
      if (qout) qout[(size_t)g * A + a] = 0.0f;
      if (nout) nout[(size_t)g * A + a] = 0;
    }
    return;
  }
  const size_t row = (nb + (size_t)node) * dm.RS;
  if (GUMBEL && gumbel_on(e, e.root_player[g])) {
    const GumbelPolicy gpol = gumbel_policy<R>(e, rules, dm, g, row);
    const typename R::Board s = e.root_board[g];
    for (int a = 0; a < A; ++a) {
      const int n = e.N[row + a] & kCountMask;
      if (pi) pi[(size_t)g * A + a] = tau_mode == 0 ? (a == gpol.move ? 1.0 : 0.0) : (double)gumbel_pi<R>(gpol, e, rules, s, row, a);
      if (qout) qout[(size_t)g * A + a] = n > 0 ? __fdiv_rn(e.W[row + a], (float)n) : 0.0f;
      if (nout) nout[(size_t)g * A + a] = n;
    }
    return;
  }
  const int tau = tau_mode == 2 ? (e.ply[g] < tau_plies ? 1 : 0) : tau_mode;
  const RootProof rp = root_proof<R>(e, rules, dm, g, row);
  long long total = 0;
  int best_n = -1, best_a = 0;
  for (int a = 0; a < A; ++a) {
    const int n = pi_count(e.N[row + a], rp);
    total += n;
    if (n > best_n) {
      best_n = n;
      best_a = a;
    }
  }
  const bool one_hot = tau == 0 || rp.win_a >= 0;
  if (rp.win_a >= 0) best_a = rp.win_a;
  for (int a = 0; a < A; ++a) {
    const int n = e.N[row + a] & kCountMask;
    if (pi) pi[(size_t)g * A + a] = one_hot ? (a == best_a ? 1.0 : 0.0) : __ddiv_rn((double)pi_count(e.N[row + a], rp), (double)total);
    if (qout) qout[(size_t)g * A + a] = n > 0 ? __fdiv_rn(e.W[row + a], (float)n) : 0.0f;  // value_avg, lib/mcts.py:244
    if (nout) nout[(size_t)g * A + a] = n;
  }
}

// ----------------------------------------------------------------------------------- tree compaction
// CARO_FLAG_COMPACT_TREE: after a move, every node whose position can no longer occur (tokens are only added: it does not
// contain the new root position) is dropped and the survivors are moved to the front of the arena.  The reference never
// frees anything (its dicts keep every state of the game, lib/mcts.py:29-46), but a dropped state can never be looked up
// again, so N / W / Q / P of every state that can still be reached -- and with them every later search -- are unchanged:
// the arena then only has to hold the searches of the last few moves, whatever the length of the game.
// One block per tree: (1) reachability flags + an exclusive scan -> old -> new index map in shared memory, (2) records,
// boards, players and key tails moved in index order, a chunk at a time through shared memory (new index <= old index: a
// chunk's destinations lie in chunks that have been read), child links rewritten through the map, (3) the hash table is
// dropped (generation bump) and re-inserted from the surviving boards.
template <class R>
__global__ void __launch_bounds__(256)
compact_kernel(View<typename R::Board> e, R rules, Dims dm, int chunk_nodes) {
  using Board = typename R::Board;
  extern __shared__ __align__(16) uint32_t cs[];
  int32_t* map = reinterpret_cast<int32_t*>(cs);            // [node_cap]
  uint32_t* stage = cs + ((dm.node_cap + 3) & ~3);           // [chunk_nodes][RS], 16-byte aligned
  __shared__ int s_scan[256 / 32];
  __shared__ int s_base;
  const int tree = blockIdx.x;
  const int g = tree / dm.tpg;
  if (e.status[g] != ST_ACTIVE) return;
  const int count = e.node_count[tree];
  if (count <= 0) return;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t nb = (size_t)tree * dm.node_cap;
  const Board root = e.root_board[g];
  // ---- (1) map ----
  if (tid == 0) s_base = 0;
  __syncthreads();
  for (int i0 = 0; i0 < count; i0 += 256) {
    const int i = i0 + tid;
    const int keep = (i < count && R::reachable(root, e.node_board[nb + i])) ? 1 : 0;
    int x = keep;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, x, off);
      if (lane >= off) x += y;
    }
    if (lane == 31) s_scan[warp] = x;
    __syncthreads();
    int before = s_base;
    for (int w = 0; w < warp; ++w) before += s_scan[w];
    if (i < count) map[i] = keep ? before + x - 1 : -1;
    __syncthreads();
    if (tid == 255) s_base = before + x;
    __syncthreads();
  }
  const int kept = s_base;
  if (kept == count) return;  // nothing to drop (uniform for the block)
  // ---- (2) move ----
  uint4* rec = reinterpret_cast<uint4*>(e.N);  // records are 16 * Apad bytes, Apad a multiple of 8: 16-byte units throughout
  uint4* stage4 = reinterpret_cast<uint4*>(stage);
  const int RS = dm.RS / 4, c_row = 3 * dm.Apad / 4;
  for (int i0 = 0; i0 < count; i0 += chunk_nodes) {
    const int n_here = min(chunk_nodes, count - i0);
    for (int k = tid; k < n_here * RS; k += 256) {
      const int node = i0 + k / RS;
      if (map[node] >= 0 && map[node] != node) stage4[k] = rec[(nb + (size_t)node) * RS + (k % RS)];
    }
    // the small per-node fields travel in registers (one node per thread and pass)
    for (int n0 = 0; n0 < n_here; n0 += 256) {
      const int node = i0 + n0 + tid;
      const bool mine = n0 + tid < n_here && map[node] >= 0 && map[node] != node;
      Board b;
      uint8_t pl = 0;
      uint64_t kh = 0;
      if (mine) {
        b = e.node_board[nb + node];
        pl = e.node_player[nb + node];
        if (RulesTraits<R>::kHasKeyHi) kh = e.key_hi[nb + node];
      }
      __syncthreads();
      if (mine) {
        const int to = map[node];
        e.node_board[nb + to] = b;
        e.node_player[nb + to] = pl;
        if (RulesTraits<R>::kHasKeyHi) e.key_hi[nb + to] = kh;
      }
      __syncthreads();
    }
    __syncthreads();
    for (int k = tid; k < n_here * RS; k += 256) {
      const int node = i0 + k / RS, w = k % RS;
      const int to = map[node];
      if (to < 0) continue;
      const bool links = w >= c_row;  // child links go through the map (a surviving node's children survive with it)
      if (to == node && !links) continue;  // in place already
      uint4 v = to == node ? rec[(nb + (size_t)node) * RS + w] : stage4[k];
      if (links) {
        v.x = (uint32_t)((int32_t)v.x >= 0 ? map[(int32_t)v.x] : -1);
        v.y = (uint32_t)((int32_t)v.y >= 0 ? map[(int32_t)v.y] : -1);
        v.z = (uint32_t)((int32_t)v.z >= 0 ? map[(int32_t)v.z] : -1);
        v.w = (uint32_t)((int32_t)v.w >= 0 ? map[(int32_t)v.w] : -1);
      }
      rec[(nb + (size_t)to) * RS + w] = v;
    }
    __syncthreads();
  }
  // ---- (3) hash table ----
  const uint32_t gen = e.tree_gen[tree] + 1u;
  __syncthreads();
  if (tid == 0) {
    e.tree_gen[tree] = gen;
    e.node_count[tree] = kept;
  }
  HashSlot* ht = e.ht + (size_t)tree * dm.hash_cap;
  for (int i = tid; i < kept; i += 256) ht_insert_cas(ht, dm.hash_cap, gen, rules.key(e.node_board[nb + i]).lo, i);
}

// ----------------------------------------------------------------------------------- resignation
// Extension (caro_engine_set_resign, off by default).  A game that starts while resignation is on is a playthrough game
// with probability `playthrough` (a Philox draw of its uid): it never resigns and logs its per-player minima instead.
template <class Board>
__device__ __forceinline__ void resign_game_start(const View<Board>& e, const SearchParams& sp, int g, uint64_t uid) {
  const ResignParams rp = *e.resign_params;
  uint8_t play = 0;
  if (rp.enabled) {
    const Philox4 r = philox4x32_10((uint32_t)uid, (uint32_t)(uid >> 32), 0u, 0u, sp.seed_lo ^ kStreamResign, sp.seed_hi);
    play = u01d(r.v[0], r.v[1]) < rp.playthrough ? 1 : 0;
    e.resign_min[2 * g] = INFINITY;
    e.resign_min[2 * g + 1] = INFINITY;
  }
  e.resign_playthrough[g] = play;
}

// ----------------------------------------------------------------------------------- advance
// One ply of lib/utils.py:76-106 for every active game.  One thread per game.
// GUMBEL (extension): as root_policy_kernel; a Gumbel root plays the Gumbel move and records pi' whatever the ply.
template <class R, bool GUMBEL>
__global__ void advance_kernel(View<typename R::Board> e, R rules, Dims dm, SearchParams sp, int tau_plies,
                               const double* __restrict__ uniform_in, int auto_restart, int first_player,
                               int32_t* __restrict__ action_out) {
  using Board = typename R::Board;
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= dm.G) return;
  if (action_out) action_out[g] = -1;
  if (e.status[g] != ST_ACTIVE) return;
  const int A = dm.A;
  size_t nb;
  const int node = root_node_of<R>(e, rules, dm, g, &nb);
  Board s = e.root_board[g];
  const int who = e.root_player[g];
  const int ply = e.ply[g];
  const int tau = ply < tau_plies ? 1 : 0;  // lib/utils.py:68,97-99
  const ResignParams rp = *e.resign_params;
  // visit counts -> pi
  long long total = 0;
  int best_n = -1, best_a = 0;
  double sum_w = 0.0;  // resignation statistic: sum of W over the root's edges, in action order
  const size_t row = (nb + (size_t)(node < 0 ? 0 : node)) * dm.RS;
  if (node >= 0) {
    for (int a = 0; a < A; ++a) {
      const int n = e.N[row + a] & kCountMask;
      total += n;
      if (rp.enabled) sum_w = __dadd_rn(sum_w, (double)e.W[row + a]);
      if (n > best_n) {
        best_n = n;
        best_a = a;
      }
    }
  }
  // stat = max(mean root value, Q of the most visited edge), from the mover's point of view
  bool resign = false;
  if (rp.enabled && total > 0) {
    const double v_root = __ddiv_rn(sum_w, (double)total);
    const double v_best = (double)__fdiv_rn(e.W[row + best_a], (float)best_n);
    const double stat = v_root > v_best ? v_root : v_best;
    if (e.resign_playthrough[g]) {
      double* m = e.resign_min + 2 * g + who;
      if (stat < *m) *m = stat;
    } else {
      resign = stat < rp.threshold;
    }
  }
  // np.random.choice(A, p=pi): cdf = cumsum(p) / cumsum(p)[-1]; first index with cdf > u
  double u;
  if (uniform_in != nullptr) {
    u = uniform_in[g];
  } else {
    const uint64_t uid = e.uid[g];
    const Philox4 r = philox4x32_10((uint32_t)uid, (uint32_t)(uid >> 32), (uint32_t)ply, 0u,
                                    sp.seed_lo ^ kStreamChoice, sp.seed_hi);
    u = u01d(r.v[0], r.v[1]);
  }
  // solver (extension): a proven-WIN root plays its lowest WIN edge, otherwise LOSS edges leave pi and the move
  const RootProof pf = node >= 0 ? root_proof<R>(e, rules, dm, g, row) : RootProof{-1, false};
  if (pf.drop_loss) {
    total = 0;
    best_n = -1;
    for (int a = 0; a < A; ++a) {
      const int n = pi_count(e.N[row + a], pf);
      total += n;
      if (n > best_n) {
        best_n = n;
        best_a = a;
      }
    }
  }
  const bool one_hot = tau == 0 || total <= 0 || pf.win_a >= 0;
  if (pf.win_a >= 0) best_a = pf.win_a;
  int action = best_a;
  const bool gum = GUMBEL && node >= 0 && gumbel_on(e, who);
  GumbelPolicy gpol;
  if (gum) {
    gpol = gumbel_policy<R>(e, rules, dm, g, row);
    action = gpol.move;
  } else if (!one_hot) {
    double last = 0.0;
    for (int a = 0; a < A; ++a) last = __dadd_rn(last, __ddiv_rn((double)pi_count(e.N[row + a], pf), (double)total));
    double c = 0.0;
    action = A - 1;
    for (int a = 0; a < A; ++a) {
      c = __dadd_rn(c, __ddiv_rn((double)pi_count(e.N[row + a], pf), (double)total));
      if (__ddiv_rn(c, last) > u) {
        action = a;
        break;
      }
    }
  }
  if (action_out) action_out[g] = resign ? -1 : action;
  // history (lib/utils.py:81)
  const int hidx = ply < dm.max_plies ? ply : dm.max_plies - 1;
  const size_t h = (size_t)g * dm.max_plies + hidx;
  e.hist_board[h] = s;
  e.hist_player[h] = (uint8_t)who;
  for (int a = 0; a < A; ++a) {
    float p;
    if (gum) p = gumbel_pi<R>(gpol, e, rules, e.root_board[g], row, a);
    else if (one_hot) p = (a == best_a) ? 1.0f : 0.0f;
    else p = (float)__ddiv_rn((double)pi_count(e.N[row + a], pf), (double)total);
    e.hist_pi[h * A + a] = p;
  }
  bool won = false;
  if (!resign) {
    if (!rules.legal(s, action)) atomicOr(e.ctr + CTR_ERRORS, ERR_ILLEGAL_ACTION);  // "Impossible action selected"
    won = rules.apply(s, action, who);
  }
  atomicAdd(e.ctr + CTR_PLIES, 1ull);
  int finished = 0, res = 0;  // res from the last mover's point of view (lib/utils.py:88,94)
  if (resign) {
    finished = 1;
    res = -1;
  } else if (won) {
    finished = 1;
    res = 1;
  } else if (!rules.any_legal(s)) {
    finished = 1;
    res = 0;
  }
  if (!finished) {
    e.root_board[g] = s;
    e.root_player[g] = (uint8_t)(who ^ 1);
    e.ply[g] = ply + 1;
    // extensions: FRESH_TREE = no tree reuse between moves (arena demand bounded by one move's searches); RECYCLE_TREE = the tree
    // is kept from move to move, like the reference's, until it fills more than half of its arena, then cleared (never overflows
    // while one move's searches fit half an arena; most moves still start from the previous move's subtree)
    for (int t = 0; t < dm.tpg; ++t) {
      const bool clear = (dm.flags & FLAG_FRESH_TREE) ||
                         ((dm.flags & FLAG_RECYCLE_TREE) && e.node_count[g * dm.tpg + t] > dm.node_cap / 2);
      if (clear) {
        e.node_count[g * dm.tpg + t] = 0;
        e.tree_gen[g * dm.tpg + t] += 1u;
      }
    }
    return;
  }
  // ---- game over -------------------------------------------------------------------------
  const int n_hist = hidx + 1;
  const int result = who == 0 ? res : -res;  // net1 == player 0 (lib/utils.py:89)
  e.result[g] = result;
  atomicAdd(e.ctr + CTR_GAMES, 1ull);
  atomicAdd(e.ctr + (result == 0 ? CTR_DRAW : (result > 0 ? CTR_WIN0 : CTR_WIN1)), 1ull);
  if (resign) atomicAdd(e.resign_ctr + RCTR_RESIGNED, 1ull);
  if (rp.enabled && e.resign_playthrough[g]) {
    const unsigned long long k = atomicAdd(e.resign_ctr + RCTR_LOGGED, 1ull);
    ResignRecord rec;
    rec.min_stat[0] = e.resign_min[2 * g];
    rec.min_stat[1] = e.resign_min[2 * g + 1];
    rec.result = result;
    rec.plies = ply + 1;
    e.resign_log[k % (unsigned long long)dm.G] = rec;
  }
  if (dm.replay_cap > 0) {
    // lib/utils.py:101-106: z = result for the last entry, sign flips walking back
    const unsigned long long base = atomicAdd(e.rp_cursor, (unsigned long long)n_hist);
    if (n_hist > dm.replay_cap) atomicOr(e.ctr + CTR_ERRORS, ERR_REPLAY_OVERRUN);
    for (int t = 0; t < n_hist; ++t) {
      const size_t src = (size_t)g * dm.max_plies + t;
      const size_t dst = (size_t)((base + (unsigned long long)t) % (unsigned long long)dm.replay_cap);
      e.rp_board[dst] = e.hist_board[src];
      e.rp_player[dst] = e.hist_player[src];
      for (int a = 0; a < A; ++a) e.rp_pi[dst * A + a] = e.hist_pi[src * A + a];
      const int back = n_hist - 1 - t;
      e.rp_z[dst] = (float)((back & 1) ? -res : res);
    }
  }
  e.root_board[g] = s;  // terminal position stays visible until the slot is re-seated
  e.root_player[g] = (uint8_t)(who ^ 1);
  e.status[g] = ST_FINISHED;
  if (auto_restart) {
    const uint32_t played = e.played[g] + 1u;
    e.played[g] = played;
    const uint64_t uid = (uint64_t)g + (uint64_t)dm.G * (uint64_t)played;
    e.uid[g] = uid;
    int fp = first_player;
    if (fp < 0) {
      const Philox4 r = philox4x32_10((uint32_t)uid, (uint32_t)(uid >> 32), 0u, 0u, sp.seed_lo ^ kStreamFirst, sp.seed_hi);
      fp = (int)(r.v[0] & 1u);
    }
    e.root_board[g] = R::empty();
    e.root_player[g] = (uint8_t)fp;
    e.ply[g] = 0;
    e.status[g] = ST_ACTIVE;
    resign_game_start(e, sp, g, uid);
    for (int t = 0; t < dm.tpg; ++t) {  // MCTS.clear(): bump the generation, no memset
      e.node_count[g * dm.tpg + t] = 0;
      e.tree_gen[g * dm.tpg + t] += 1u;
    }
  }
}

// ----------------------------------------------------------------------------- replay -> SGD batch
// train.py:85-94 on the device: the sampled replay rows become the training tensors without leaving HBM -- network
// planes (game.states_to_training_batch of the stored position, from the side to move's point of view), the MCTS
// policy target and the outcome z.  `entry[i]` = absolute number of the sampled ring entry (slot = entry % capacity;
// the host draws the numbers with random.sample, like the reference).  One block per sample.
// `sym` (extension, nullptr = off; not in the reference): symmetry augmentation -- sample i is written through the board
// symmetry sym[i]: bit 0 mirrors the columns (the only symmetry of Connect4), bit 1 mirrors the rows, bit 2 transposes
// (square boards: the eight dihedral symmetries); planes and policy target are transformed together, z is invariant.
template <class R>
__global__ void __launch_bounds__(64)
replay_gather_kernel(View<typename R::Board> e, R rules, Dims dm, const long long* __restrict__ entry, const int32_t* __restrict__ sym,
                     long long count, float* __restrict__ planes, float* __restrict__ pi, float* __restrict__ z) {
  const long long i = blockIdx.x;
  if (i >= count) return;
  const size_t slot = (size_t)(entry[i] % (long long)dm.replay_cap);
  const typename R::Board s = e.rp_board[slot];
  const int who = e.rp_player[slot];
  const int H = rules.rows(), W = rules.cols(), HW = H * W;
  const int t = sym ? sym[i] : 0;
  auto source_cell = [&](int r, int c, int* sr, int* sc) {  // output cell (r, c) shows source cell (sr, sc)
    if (t & 4) { const int x = r; r = c; c = x; }
    *sr = (t & 2) ? H - 1 - r : r;
    *sc = (t & 1) ? W - 1 - c : c;
  };
  for (int o = threadIdx.x; o < 2 * HW; o += blockDim.x) {
    const int plane = o / HW, cell = o - plane * HW;
    int sr, sc;
    source_cell(cell / W, cell % W, &sr, &sc);
    planes[(size_t)i * 2 * HW + o] = (float)rules.plane_value(s, who, plane, sr, sc);
  }
  for (int a = threadIdx.x; a < dm.A; a += blockDim.x) {
    int src = a;
    if (dm.A == W) {  // column actions (Connect4)
      src = (t & 1) ? W - 1 - a : a;
    } else {          // cell actions, row-major (m,n,k)
      int sr, sc;
      source_cell(a / W, a % W, &sr, &sc);
      src = sr * W + sc;
    }
    pi[(size_t)i * dm.A + a] = e.rp_pi[slot * dm.A + src];
  }
  if (threadIdx.x == 0) z[i] = e.rp_z[slot];
}

// ----------------------------------------------------------------------------- resignation parameters
// One thread: the parameters arrive by value and are stored on the stream, behind every earlier ply.
__global__ void set_resign_kernel(ResignParams* __restrict__ dst, ResignParams p) { *dst = p; }
__global__ void set_solver_kernel(SolverParams* __restrict__ dst, SolverParams p) { *dst = p; }
__global__ void set_gumbel_kernel(GumbelParams* __restrict__ dst, GumbelParams p) { *dst = p; }

// ------------------------------------------------------------------------------------- reset
template <class R>
__global__ void reset_kernel(View<typename R::Board> e, Dims dm, SearchParams sp, const uint8_t* __restrict__ mask,
                             int first_player, int bump_uid) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= dm.G) return;
  if (mask != nullptr && mask[g] == 0) return;
  uint32_t played = e.played[g];
  if (bump_uid) {
    played += 1u;
    e.played[g] = played;
  }
  const uint64_t uid = (uint64_t)g + (uint64_t)dm.G * (uint64_t)played;
  e.uid[g] = uid;
  int fp = first_player;
  if (fp < 0) {
    const Philox4 r = philox4x32_10((uint32_t)uid, (uint32_t)(uid >> 32), 0u, 0u, sp.seed_lo ^ kStreamFirst, sp.seed_hi);
    fp = (int)(r.v[0] & 1u);
  }
  e.root_board[g] = R::empty();
  e.root_player[g] = (uint8_t)fp;
  e.ply[g] = 0;
  e.status[g] = ST_ACTIVE;
  e.result[g] = 0;
  resign_game_start(e, sp, g, uid);
  for (int t = 0; t < dm.tpg; ++t) {
    e.node_count[g * dm.tpg + t] = 0;
    e.tree_gen[g * dm.tpg + t] += 1u;
  }
}

}  // namespace caro
