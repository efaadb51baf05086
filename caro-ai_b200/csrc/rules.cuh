// Packed-bitboard game rules for the MCTS hot path (Connect4 6x7 and the m,n,k family).
//
// Replaces the reference's per-call big-int decode (lib/game/connect_four/connect_four.py:129-265,
// lib/game/tictactoe/tictactoe.py:116-235, lib/game/tictactoe/tictactoe_helpers.py:7-179) with
// integer shift/AND arithmetic.  Everything here is __host__ __device__ so the same code is
// exercised by the host-side self-check library (tests/native) without a GPU.
//
// Connect4 layout  : 7 bits per column (6 cells + 1 always-empty sentinel), bit = 7*col + row,
//                    row 0 = bottom.  `mask` = occupied cells, `black` = player-1 tokens.
// m,n,k layout     : bit = row*n + col (== the reference's action index), 256 bits per colour
//                    (n <= 15; 16 would also fit), `w` = player 0, `b` = player 1.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define CARO_HD __host__ __device__ __forceinline__
#else
#define CARO_HD inline
#endif

namespace caro {

struct Key128 {
  uint64_t lo, hi;
};

CARO_HD uint64_t mix64(uint64_t x) {  // splitmix64 finaliser
  x ^= x >> 30;
  x *= 0xbf58476d1ce4e5b9ULL;
  x ^= x >> 27;
  x *= 0x94d049bb133111ebULL;
  x ^= x >> 31;
  return x;
}

// ------------------------------------------------------------------------------------ Connect4
struct C4Board {
  uint64_t mask;   // occupied
  uint64_t black;  // player 1 (subset of mask)
};

struct C4Rules {
  using Board = C4Board;
  static constexpr int kActions = 7;
  static constexpr int kRows = 6;
  static constexpr int kCols = 7;
  static constexpr int kMaxPlies = 42;
  static constexpr uint64_t kBottom = 0x0040810204081ULL;           // bit 0 of every column
  static constexpr uint64_t kFull = kBottom * 0x3FULL;              // 42 playable cells
  static constexpr uint64_t kTop = kBottom << 5;                    // row 5 of every column

  CARO_HD int actions() const { return kActions; }
  CARO_HD int rows() const { return kRows; }
  CARO_HD int cols() const { return kCols; }

  CARO_HD static Board empty() { return Board{0ULL, 0ULL}; }
  // can position q still occur in a game that has reached position r?  (tokens are only ever added)
  CARO_HD static bool reachable(const Board& r, const Board& q) { return (r.mask & ~q.mask) == 0ULL && (q.black & r.mask) == r.black; }

  // connect_four.py:157-165 -- a column is playable while its top cell is empty
  CARO_HD bool legal(const Board& s, int col) const { return ((s.mask >> (7 * col + 5)) & 1ULL) == 0ULL; }
  CARO_HD bool any_legal(const Board& s) const { return (s.mask & kTop) != kTop; }

  // connect_four.py:241-265.  Drops `player`'s token into `col`; returns whether that token
  // completes a vertical / horizontal / diagonal run of >= 4 THROUGH the new cell -- exactly the
  // reference's rule (it only inspects lines through the new token, :206-239,258-263).
  CARO_HD bool apply(Board& s, int col, int player) const {
    const uint64_t colmask = 0x3FULL << (7 * col);                    // playable cells of the column
    const uint64_t bit = (s.mask + (1ULL << (7 * col))) & colmask;    // lowest empty cell (0 if full)
    s.mask |= bit;
    if (player) s.black |= bit;
    const uint64_t mine = player ? s.black : (s.mask ^ s.black);
    bool won = false;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int d = 0; d < 4; ++d) {
      const int sh = (d == 0) ? 1 : (d == 1) ? 7 : (d == 2) ? 8 : 6;  // vertical, horizontal, rising, falling
      uint64_t m = mine & (mine >> sh);
      m = m & (m >> (2 * sh));                                        // start cells of 4-runs
      const uint64_t cover = m | (m << sh) | (m << (2 * sh)) | (m << (3 * sh));
      won = won || ((cover & bit) != 0ULL);
    }
    return won;
  }

  // Injective 49-bit key: per column a guard bit above the stack, colours below it.
  CARO_HD Key128 key(const Board& s) const { return Key128{(s.mask + kBottom) | s.black, 0ULL}; }

  // Net input (connect_four.py:175-204): plane 0 = tokens of the player to move, plane 1 = all
  // other tokens; plane row 0 is the TOP of the board.
  CARO_HD int plane_value(const Board& s, int who, int plane, int prow, int pcol) const {
    const uint64_t bit = 1ULL << (7 * pcol + (kRows - 1 - prow));
    const uint64_t mine = who ? s.black : (s.mask ^ s.black);
    const uint64_t sel = plane == 0 ? mine : (s.mask ^ mine);
    return (sel & bit) ? 1 : 0;
  }
};

// ------------------------------------------------------------------------------------ m,n,k
struct MnkBoard {
  uint64_t w[4];  // player 0 tokens
  uint64_t b[4];  // player 1 tokens
};

struct MnkRules {
  using Board = MnkBoard;
  int n;  // board side (<= 15)
  int k;  // run length to win
  // 0: freestyle (any run >= k wins).  1: Caro -- a run >= k with an opponent stone just past BOTH of its ends does
  // not win (the board edge never blocks).  Read only once a direction already reaches k.
  int blocked_ends;

  CARO_HD int actions() const { return n * n; }
  CARO_HD int rows() const { return n; }
  CARO_HD int cols() const { return n; }

  CARO_HD static Board empty() {
    Board s;
    for (int i = 0; i < 4; ++i) s.w[i] = s.b[i] = 0ULL;
    return s;
  }
  // can position q still occur in a game that has reached position r?  (tokens are only ever added)
  CARO_HD static bool reachable(const Board& r, const Board& q) {
    bool ok = true;
    for (int i = 0; i < 4; ++i) ok = ok && (r.w[i] & ~q.w[i]) == 0ULL && (r.b[i] & ~q.b[i]) == 0ULL;
    return ok;
  }
  CARO_HD static bool test(const uint64_t* v, int idx) { return (v[idx >> 6] >> (idx & 63)) & 1ULL; }

  // tictactoe.py:137-162 -- empty cells are the legal moves
  CARO_HD bool legal(const Board& s, int a) const { return !test(s.w, a) && !test(s.b, a); }
  CARO_HD int occupied(const Board& s) const {
    int c = 0;
    for (int i = 0; i < 4; ++i) {
#if defined(__CUDA_ARCH__)
      c += __popcll(s.w[i] | s.b[i]);
#else
      c += __builtin_popcountll(s.w[i] | s.b[i]);
#endif
    }
    return c;
  }
  CARO_HD bool any_legal(const Board& s) const { return occupied(s) < n * n; }

  CARO_HD int ray(const uint64_t* mine, int r, int c, int dr, int dc) const {
    int cnt = 0;
    for (int i = 1; i < k; ++i) {
      const int rr = r + i * dr, cc = c + i * dc;
      if (rr < 0 || rr >= n || cc < 0 || cc >= n) break;
      if (!test(mine, rr * n + cc)) break;
      ++cnt;
    }
    return cnt;
  }

  // Caro: is the cell just past the END of the maximal run of `mine` from (r, c) along (dr, dc) an opponent stone?
  // The walk runs to the real end of the run (up to n - 1 cells), not ray's k - 1: overlines and dense boards have
  // runs longer than k.  Off the board is not a block.
  CARO_HD bool flank_blocked(const uint64_t* mine, const uint64_t* other, int r, int c, int dr, int dc) const {
    int rr = r + dr, cc = c + dc;
    while (rr >= 0 && rr < n && cc >= 0 && cc < n && test(mine, rr * n + cc)) {
      rr += dr;
      cc += dc;
    }
    return rr >= 0 && rr < n && cc >= 0 && cc < n && test(other, rr * n + cc);
  }

  // The line through (r, c) along +-(dr, dc) wins: a run >= k and, under Caro, not blocked at both ends.
  CARO_HD bool line_wins(const uint64_t* mine, const uint64_t* other, int r, int c, int dr, int dc) const {
    if (1 + ray(mine, r, c, dr, dc) + ray(mine, r, c, -dr, -dc) < k) return false;
    return !blocked_ends || !(flank_blocked(mine, other, r, c, dr, dc) && flank_blocked(mine, other, r, c, -dr, -dc));
  }

  // tictactoe.py:210-235 + tictactoe_helpers.py:7-56.  The reference scans the whole row /
  // column / diagonal / anti-diagonal through the move for ANY run >= k; in every position
  // reachable by legal play (the game stops at the first win) that equals "the run through the
  // new cell is >= k", which is what is evaluated here.  Like the reference the target cell is
  // overwritten without an emptiness check.  With blocked_ends set (Caro) a direction whose run
  // has an opponent stone past both ends does not win; another direction still may.
  CARO_HD bool apply(Board& s, int a, int player) const {
    const uint64_t bit = 1ULL << (a & 63);
    uint64_t* mine = player ? s.b : s.w;
    uint64_t* other = player ? s.w : s.b;
    mine[a >> 6] |= bit;
    other[a >> 6] &= ~bit;
    const int r = a / n, c = a - r * n;
    bool won = false;
    won = won || line_wins(mine, other, r, c, 0, 1);
    won = won || line_wins(mine, other, r, c, 1, 0);
    won = won || line_wins(mine, other, r, c, 1, 1);
    won = won || line_wins(mine, other, r, c, -1, 1);
    return won;
  }

  // 128-bit fingerprint of the 512-bit position (two independent mixing chains).  A transposition
  // is recognised only when all 128 bits agree (64 in the hash slot, 64 in the node).
  CARO_HD Key128 key(const Board& s) const {
    uint64_t a = 0x9E3779B97F4A7C15ULL, b = 0xD1B54A32D192ED03ULL;
    for (int i = 0; i < 4; ++i) {
      a = mix64(a ^ s.w[i]) + 0x632BE59BD9B4E019ULL * (uint64_t)(2 * i + 1);
      a = mix64(a ^ (s.b[i] * 0xFF51AFD7ED558CCDULL));
      b = mix64(b + s.b[i]) ^ (0xC2B2AE3D27D4EB4FULL * (uint64_t)(2 * i + 3));
      b = mix64(b + (s.w[i] ^ 0xA0761D6478BD642FULL));
    }
    return Key128{a | 1ULL, b};
  }

  // tictactoe.py:164-208: plane 0 = mover's cells, plane 1 = opponent's cells, row 0 = top.
  CARO_HD int plane_value(const Board& s, int who, int plane, int prow, int pcol) const {
    const int idx = prow * n + pcol;
    const uint64_t* mine = who ? s.b : s.w;
    const uint64_t* other = who ? s.w : s.b;
    return test(plane == 0 ? mine : other, idx) ? 1 : 0;
  }
};

}  // namespace caro
