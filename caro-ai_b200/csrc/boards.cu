// Stand-alone batched board kernels (SURVEY.md section 8 rows a11-a16): move + win/draw, legal-move masks
// and the network input planes, one thread per board (per output element for the planes).
#include <cuda_runtime.h>

#include "../../include/caro_b200.h"
#include "common_host.h"
#include "rules.cuh"

namespace caro {

template <class R>
__global__ void apply_kernel(R rules, const typename R::Board* __restrict__ in, const int32_t* __restrict__ actions,
                             const uint8_t* __restrict__ players, long long count, typename R::Board* __restrict__ out,
                             uint8_t* __restrict__ won, uint8_t* __restrict__ draw) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  typename R::Board s = in[i];
  const bool w = rules.apply(s, actions[i], players[i]);
  out[i] = s;
  if (won) won[i] = w ? 1 : 0;
  if (draw) draw[i] = (!w && !rules.any_legal(s)) ? 1 : 0;
}

template <class R>
__global__ void legal_kernel(R rules, const typename R::Board* __restrict__ in, long long count, int words,
                             uint32_t* __restrict__ mask) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const typename R::Board s = in[i];
  const int A = rules.actions();
  for (int w = 0; w < words; ++w) {
    uint32_t m = 0u;
    for (int b = 0; b < 32; ++b) {
      const int a = w * 32 + b;
      if (a < A && rules.legal(s, a)) m |= 1u << b;
    }
    mask[i * words + w] = m;
  }
}

template <class R>
__global__ void planes_kernel(R rules, const typename R::Board* __restrict__ in, const uint8_t* __restrict__ who,
                              long long count, float* __restrict__ planes) {
  const int H = rules.rows(), W = rules.cols();
  const long long per = 2LL * H * W;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= count * per) return;
  const long long i = t / per;
  const int r = (int)(t % per);
  const int plane = r / (H * W), row = (r / W) % H, col = r % W;
  planes[t] = (float)rules.plane_value(in[i], who[i], plane, row, col);
}

// Vectorised variant: every thread produces V (2 or 4) consecutive floats of one position's planes with one 8- or
// 16-byte store (2 H W is always even; the scalar kernel above reached 21 % of the HBM roofline on 4 M Connect4
// positions, this one is store-bandwidth-bound).
template <class R, int V>
__global__ void planes_vec_kernel(R rules, const typename R::Board* __restrict__ in, const uint8_t* __restrict__ who,
                                  long long count, float* __restrict__ planes) {
  const int H = rules.rows(), W = rules.cols();
  const int per = 2 * H * W, vec_per = per / V;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= count * vec_per) return;
  const long long i = t / vec_per;
  const int r0 = (int)(t - i * vec_per) * V;
  const typename R::Board s = in[i];
  const int wm = who[i];
  float v[V];
#pragma unroll
  for (int e = 0; e < V; ++e) {
    const int r = r0 + e;
    const int plane = r / (H * W), cell = r - plane * H * W;
    const int row = cell / W, col = cell - row * W;
    v[e] = (float)rules.plane_value(s, wm, plane, row, col);
  }
  float* dst = planes + i * per + r0;
  if (V == 4) *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[V - 1]);
  else *reinterpret_cast<float2*>(dst) = make_float2(v[0], v[1]);
}

// MCTS._backup (lib/mcts.py:225-246) on caller-provided flat N/W/Q arrays: the dict-view facade of
// caro_ai_b200.mcts.MCTS uses it when statistics were assigned from the host (lib/test_mcts.py:15-38).
__global__ void backup_path_kernel(int32_t* __restrict__ N, float* __restrict__ W, float* __restrict__ Q,
                                   const int64_t* __restrict__ edge, int depth, float value) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  float cur = -value;
  for (int i = depth - 1; i >= 0; --i) {
    const int64_t idx = edge[i];
    const int n = N[idx] + 1;
    const float w = __fadd_rn(W[idx], cur);
    N[idx] = n;
    W[idx] = w;
    Q[idx] = __fdiv_rn(w, (float)n);
    cur = -cur;
  }
}

}  // namespace caro

using namespace caro;

static inline cudaStream_t S(void* s) { return reinterpret_cast<cudaStream_t>(s); }

static int check_game(int game, int n, int k) {
  if (game == CARO_GAME_CONNECT4) return CARO_OK;
  if ((game == CARO_GAME_MNK || game == CARO_GAME_CARO) && n >= 2 && n <= 15 && k >= 2 && k <= n) return CARO_OK;
  return caro_fail(CARO_E_ARG, "unknown game or bad (n,k)");
}

// freestyle m,n,k or Caro (the same board; a run blocked at both ends does not win)
static MnkRules mnk_rules(int game, int n, int k) { return MnkRules{n, k, game == CARO_GAME_CARO ? 1 : 0}; }

extern "C" {

int caro_boards_apply(int game, int n, int k, const void* d_boards, const int32_t* d_actions, const uint8_t* d_players,
                      int64_t count, void* d_out, uint8_t* d_won, uint8_t* d_draw, void* stream) {
  if (check_game(game, n, k) != CARO_OK) return CARO_E_ARG;
  if (!d_boards || !d_actions || !d_players || !d_out || count < 0) return caro_fail(CARO_E_ARG, "null argument");
  if (caro_device_count() <= 0) return caro_fail(CARO_E_CUDA, "no CUDA device: the board kernels have no CPU fallback");
  if (count == 0) return CARO_OK;
  const unsigned grid = (unsigned)((count + 255) / 256);
  if (game == CARO_GAME_CONNECT4)
    apply_kernel<C4Rules><<<grid, 256, 0, S(stream)>>>(C4Rules(), (const C4Board*)d_boards, d_actions, d_players, count,
                                                       (C4Board*)d_out, d_won, d_draw);
  else
    apply_kernel<MnkRules><<<grid, 256, 0, S(stream)>>>(mnk_rules(game, n, k), (const MnkBoard*)d_boards, d_actions, d_players, count,
                                                        (MnkBoard*)d_out, d_won, d_draw);
  return caro_check_launch("apply_kernel");
}

int caro_boards_legal_mask(int game, int n, int k, const void* d_boards, int64_t count, uint32_t* d_mask, void* stream) {
  if (check_game(game, n, k) != CARO_OK) return CARO_E_ARG;
  if (!d_boards || !d_mask || count < 0) return caro_fail(CARO_E_ARG, "null argument");
  if (caro_device_count() <= 0) return caro_fail(CARO_E_CUDA, "no CUDA device: the board kernels have no CPU fallback");
  if (count == 0) return CARO_OK;
  const unsigned grid = (unsigned)((count + 255) / 256);
  if (game == CARO_GAME_CONNECT4)
    legal_kernel<C4Rules><<<grid, 256, 0, S(stream)>>>(C4Rules(), (const C4Board*)d_boards, count, 1, d_mask);
  else
    legal_kernel<MnkRules><<<grid, 256, 0, S(stream)>>>(mnk_rules(game, n, k), (const MnkBoard*)d_boards, count, (n * n + 31) / 32, d_mask);
  return caro_check_launch("legal_kernel");
}

int caro_backup_path(int32_t* d_n, float* d_w, float* d_q, const int64_t* d_edge_index, int depth, float value, void* stream) {
  if (!d_n || !d_w || !d_q || (!d_edge_index && depth > 0) || depth < 0) return caro_fail(CARO_E_ARG, "null argument");
  if (caro_device_count() <= 0) return caro_fail(CARO_E_CUDA, "no CUDA device: no CPU fallback");
  if (depth == 0) return CARO_OK;
  backup_path_kernel<<<1, 32, 0, S(stream)>>>(d_n, d_w, d_q, d_edge_index, depth, value);
  return caro_check_launch("backup_path_kernel");
}

int caro_boards_encode_planes(int game, int n, int k, const void* d_boards, const uint8_t* d_who, int64_t count,
                              float* d_planes, void* stream) {
  if (check_game(game, n, k) != CARO_OK) return CARO_E_ARG;
  if (!d_boards || !d_who || !d_planes || count < 0) return caro_fail(CARO_E_ARG, "null argument");
  if (caro_device_count() <= 0) return caro_fail(CARO_E_CUDA, "no CUDA device: the board kernels have no CPU fallback");
  if (count == 0) return CARO_OK;
  const long long per = game == CARO_GAME_CONNECT4 ? 84 : 2LL * n * n;
  const bool aligned = (reinterpret_cast<uintptr_t>(d_planes) & 15u) == 0;
  if (game == CARO_GAME_CONNECT4 && aligned) {
    const unsigned grid = (unsigned)((count * (per / 4) + 255) / 256);
    planes_vec_kernel<C4Rules, 4><<<grid, 256, 0, S(stream)>>>(C4Rules(), (const C4Board*)d_boards, d_who, count, d_planes);
  } else if (game != CARO_GAME_CONNECT4 && aligned && per % 4 == 0) {
    const unsigned grid = (unsigned)((count * (per / 4) + 255) / 256);
    planes_vec_kernel<MnkRules, 4><<<grid, 256, 0, S(stream)>>>(mnk_rules(game, n, k), (const MnkBoard*)d_boards, d_who, count, d_planes);
  } else if (game != CARO_GAME_CONNECT4 && aligned) {
    const unsigned grid = (unsigned)((count * (per / 2) + 255) / 256);
    planes_vec_kernel<MnkRules, 2><<<grid, 256, 0, S(stream)>>>(mnk_rules(game, n, k), (const MnkBoard*)d_boards, d_who, count, d_planes);
  } else {
    const unsigned grid = (unsigned)((count * per + 255) / 256);
    if (game == CARO_GAME_CONNECT4)
      planes_kernel<C4Rules><<<grid, 256, 0, S(stream)>>>(C4Rules(), (const C4Board*)d_boards, d_who, count, d_planes);
    else
      planes_kernel<MnkRules><<<grid, 256, 0, S(stream)>>>(mnk_rules(game, n, k), (const MnkBoard*)d_boards, d_who, count, d_planes);
  }
  return caro_check_launch("planes_kernel");
}

}  // extern "C"
