// Fused policy/value tower on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a only.
//
// lib/model.py:82-94 (eval-mode BatchNorm folded on the host) as ONE persistent kernel:
//   * one CTA per SM; a CTA takes a "group" of whole boards laid out as 512 padded positions
//     (row pitch W+1, one zero row after every board) = 4 UMMA M-tiles of 128 rows;
//   * every 3x3 convolution is an implicit GEMM: for each of the 9 taps, D[128 x 64] +=
//     A_tap[128 x 64] * W_tap[64 x 64]^T, where A_tap is the SAME shared-memory activation buffer
//     addressed with a row offset of (dy*pitch + dx) -- the activations are kept in the no-swizzle
//     K-major core-matrix layout (8 rows x 16 B contiguous), in which a row shift is just a
//     16-byte-granular change of the descriptor start address, so no im2col copy is ever made;
//   * bf16 operands, fp32 accumulation in TMEM (4 tiles x 64 columns); the fp32 residual stream
//     v <- v + lrelu(conv(v)) also lives in TMEM (4 x 64 columns), only the bf16 copy that feeds
//     the next layer's MMAs goes back to shared memory -- nothing but the boards (16 B / 64 B per
//     leaf) and the priors/value (A+1 floats) touches HBM per leaf;
//   * per-layer weight images (72 KB, pre-packed on the host in UMMA B-operand layout) stream from
//     L2 with cp.async.bulk + mbarrier while the previous layer's epilogue runs;
//   * heads (1x1 convs, FCs, tanh, softmax) run on the CUDA cores out of the last epilogue.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "../../include/caro_b200.h"
#include "common_host.h"
#include "net.h"
#include "rules.cuh"

#include "tc_common.cuh"
#include "rt_common.cuh"

namespace caro {

constexpr int kTileRows = 128;
constexpr int kHalo = 20;                                // zero positions before / after (>= pitch + 1)
constexpr int kTapBytes = 8 * 64 * 16;                   // 8,192: one tap of a 64->64 layer
constexpr int kTapBytesIn = 2 * 64 * 16;                 // 2,048: one tap of conv_in (K padded to 16)
constexpr int kLayerBytes = 9 * kTapBytes;               // 73,728
constexpr int kLayerBytesIn = 9 * kTapBytesIn;           // 18,432
constexpr int kHeadfeatSlots = 8;                         // scratch slots for exported head features (launches in flight)
constexpr int kHeadsInTowerMaxHW = 64;                    // larger boards run their FC heads in heads_tc_kernel (net_heads.cu)
constexpr int kSmemBiasLayers = 1 + kBlocks;             // biases of the first six layers sit in shared memory (the budget has 384 bytes to
                                                         // spare); deeper towers (BlobLayout::blocks > 5) read the others from global memory
constexpr int kEpiWarps = 8;                             // warps 0-7: epilogue; TMEM lane quarter = warp & 3, column half = warp >> 2
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr int kMmaWarp = kEpiWarps;                      // warp 8: TMEM owner + MMA issue for tiles 0,2
constexpr int kMmaWarps = 2;                             // warp 9: MMA issue for tiles 1,3 + weight streaming
constexpr int kHeadWarp = kMmaWarp + kMmaWarps;          // warps 10-11: FC heads + softmax, off the critical path
constexpr int kHeadWarps = 2;
constexpr int kHeadThreads = 32 * kHeadWarps;
constexpr int kThreads = kEpiThreads + 32 * kMmaWarps + kHeadThreads;


// Kernel configuration.
//   TILES = UMMA M-tiles (128 padded positions each) a CTA processes per pass,
//   SPLIT = "bf16x3" precision mode: activations and weights are kept as bf16 hi + lo pairs and every product is
//           evaluated as hi*hi + lo*hi + hi*lo (fp32 accumulate), ~16 mantissa bits instead of 8.  Needed for
//           trained checkpoints whose policy logits span +-100 (DESIGN.md section 2); 3x the tensor work and twice
//           the shared memory per row, hence 2 tiles per pass and a single (hi+lo) weight buffer.
//   PAIR  = two CTAs of a cluster run ONE cta_group::2 MMA stream of M = 256 (each CTA its own boards, accumulators, epilogue
//           and heads); each CTA stores and fetches only its 32 of the 64 output channels of every tap, 4 + 1 KB per MMA instead
//           of 4 + 2 -- this kernel IS bound by the shared-memory pipe (operand fetch 48 cycles per 32-cycle MMA).
template <int TILES, bool SPLIT, bool PAIR_ = false>
struct TcCfg {
  static constexpr int kTiles = TILES;
  static constexpr bool kSplit = SPLIT;
  static constexpr bool kPair = PAIR_;
  static_assert(!(SPLIT && PAIR_), "the pair form exists for the one-pass mode only");
  static constexpr int kBRows = PAIR_ ? 32 : 64;                    // B rows (output channels) a CTA stores per tap
  static constexpr int kTapB = 8 * kBRows * 16;                     // bytes of one tap of a 64 -> 64 layer
  static constexpr int kTapBIn = 2 * kBRows * 16;                   // conv_in (K padded to 16)
  static constexpr int kLayerB = 9 * kTapB;
  static constexpr int kGroupRows = TILES * kTileRows;
  static constexpr int kActRows = kGroupRows + 2 * kHalo;
  static constexpr int kChunkBytes = kActRows * 16;      // one 8-channel chunk of all positions
  static constexpr int kActBytes = 8 * kChunkBytes;      // one bf16 activation image (hi or lo)
  static constexpr int kActBufs = SPLIT ? 2 : 1;
  static constexpr int kWStages = SPLIT ? 1 : 2;         // weight buffers in flight
  static constexpr int kWParts = SPLIT ? 2 : 1;          // hi (+ lo) images per layer
  static constexpr int kWStageBytes = kWParts * kLayerB;
  static constexpr uint32_t kTmemCols = 2 * TILES * 64;  // accumulators + fp32 residual stream
  // dynamic shared memory carve-up (byte offsets from a 128-aligned base)
  static constexpr int kAct = 0;
  static constexpr int kWgt = kAct + kActBufs * kActBytes;
  static constexpr int kBias = kWgt + kWStages * kWStageBytes;     // float [6][64]
  static constexpr int kHeadW = kBias + kSmemBiasLayers * 64 * 4;  // float [3][64] + [3] biases (+pad)
  static constexpr int kHeadF = kHeadW + 4 * 64 * 4;               // float [rows][3] head features
  static constexpr int kFc = kHeadF + kGroupRows * 3 * 4;          // float hidden[nb][20] + logits[nb][A]
  static constexpr int kFcFloats = TILES * 256;
  static constexpr int kCellTab = kFc + kFcFloats * 4;             // uint16 [rows]: (board << 9) | (cell + 1), 0 = padding
  static constexpr int kBars = kCellTab + kGroupRows * 2;          // mbarriers + tmem base
  static constexpr int kTotal = kBars + 128;
  static_assert(kTotal <= 232448, "exceeds the 227 KB shared memory of an sm_100 CTA");
};
using TcFast = TcCfg<4, false>;
using TcExact = TcCfg<2, true>;
using TcPair = TcCfg<4, false, true>;


// ------------------------------------------------------------------------------------- kernel
// Roles: warps 0-7 = epilogue (warp w owns TMEM lanes [32(w&3), +32) = rows of every tile, channels 32(w>>2)..+32),
//        warp 8    = TMEM allocation, elected-lane MMA issue for tiles 0 and 2,
//        warp 9    = elected-lane MMA issue for tiles 1 and 3, weight streaming (cp.async.bulk).
//        Two issuing warps so that one tile's barrier waits overlap the other tile's MMAs (the tensor pipe's
//        queue is shallow: with one issuer the waits showed up as ~25 % idle gaps in the timeline).
// Pipeline per layer L (tiles t = 0..3, in-place activation buffer):
//   MMA(L,t)  needs act_ready[t-1..t+1] of the previous stage (their bf16 rows + tile t's accumulator drained)
//   EPI(L,t)  needs acc_full[min(t+1,3)]  (tile t+1 reads the last rows of tile t as its halo)
// so the epilogue of tile t runs underneath the MMAs of tile t+2 / the next layer's tile t-1.
template <class R, class K>
__global__ void __launch_bounds__(kThreads, 1)
net_tc_kernel(R rules, TcGeom gm, const typename R::Board* __restrict__ boards, const uint8_t* __restrict__ who,
              const int32_t* __restrict__ d_count, long long max_count, const uint8_t* __restrict__ wimg,
              const float* __restrict__ bias_g, const float* __restrict__ blob, BlobLayout L,
              const float* __restrict__ pol_fc_t, const float* __restrict__ val_fc1_t, float* __restrict__ probs,
              float* __restrict__ values, uint8_t* __restrict__ headfeat_out, size_t headfeat_lo_off, int headfeat_kc8,
              long long* __restrict__ trace) {
  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t* act = smem + K::kAct;
  uint8_t* wgt = smem + K::kWgt;
  float* bias_s = reinterpret_cast<float*>(smem + K::kBias);
  float* headw_s = reinterpret_cast<float*>(smem + K::kHeadW);
  float* headf_s = reinterpret_cast<float*>(smem + K::kHeadF);
  float* fc_s = reinterpret_cast<float*>(smem + K::kFc);
  uint64_t* bar_w = reinterpret_cast<uint64_t*>(smem + K::kBars);  // [2] weights buffer filled
  uint64_t* bar_acc = bar_w + 2;                                        // [4] accumulator tile complete
  uint64_t* bar_act = bar_w + 6;                                        // [4] activation tile rewritten / accumulator drained
  uint64_t* bar_feat = bar_w + 10;                                      // [0] head features complete, [1] consumed + re-zeroed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_w + 12);
  uint64_t* bar_wp = bar_w + 13;                                        // [2] PAIR, leader: the peer's weights buffer filled
  uint16_t* cell_tab = reinterpret_cast<uint16_t*>(smem + K::kCellTab);
  constexpr bool PAIR = K::kPair;

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const long long count = d_count ? min((long long)*d_count, max_count) : max_count;
  const int nb = gm.boards_per_group;
  const long long n_groups = (count + nb - 1) / nb;
  // PAIR: the unit of work is a PAIR of groups, the CTA of rank r takes the r-th; an odd tail leaves the peer an empty group
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;
  const long long unit = PAIR ? (long long)(blockIdx.x >> 1) : (long long)blockIdx.x;
  const long long n_units = PAIR ? (long long)(gridDim.x >> 1) : (long long)gridDim.x;
  const long long work = PAIR ? (n_groups + 1) / 2 : n_groups;
  if (unit >= work) return;  // uniform per CTA (pair), before any barrier / TMEM use
  const int my_groups = (int)((work - unit + n_units - 1) / n_units);
  auto group_leaf0 = [&](int gi) { return ((unit + (long long)gi * n_units) * (PAIR ? 2 : 1) + rank) * nb; };
  auto group_valid = [&](long long leaf0) { return (int)max(0ll, min((long long)nb, count - leaf0)); };

  // ---- one-time setup ---------------------------------------------------------------------
  for (int i = tid; i < K::kActBufs * K::kActBytes / 16; i += kThreads) reinterpret_cast<uint4*>(act)[i] = make_uint4(0, 0, 0, 0);
  const int n_layers = 1 + L.blocks;
  for (int i = tid; i < min(n_layers, kSmemBiasLayers) * 64; i += kThreads) bias_s[i] = bias_g[i];
  for (int p = tid; p < K::kGroupRows; p += kThreads) {  // padded position -> (board, cell) once, no divisions in the hot loop
    const int b = p / gm.block, within = p - b * gm.block;
    const int r = within / gm.pitch, c = within - r * gm.pitch;
    cell_tab[p] = (b < nb && r < gm.H && c < gm.W) ? (uint16_t)((b << 9) | (r * gm.W + c + 1)) : (uint16_t)0;
  }
  for (int i = tid; i < K::kGroupRows * 3; i += kThreads) headf_s[i] = 0.0f;
  for (int i = tid; i < 64; i += kThreads) {
    headw_s[i] = blob[L.val_conv_w + i];
    headw_s[64 + i] = blob[L.pol_conv_w + i];
    headw_s[128 + i] = blob[L.pol_conv_w + 64 + i];
  }
  if (tid == 0) {
    headw_s[192] = blob[L.val_conv_b];
    headw_s[193] = blob[L.pol_conv_b];
    headw_s[194] = blob[L.pol_conv_b + 1];
    mbar_init(bar_w + 0, 1);
    mbar_init(bar_w + 1, 1);
    mbar_init(bar_wp + 0, 1);
    mbar_init(bar_wp + 1, 1);
    for (int t = 0; t < 4; ++t) {
      mbar_init(bar_acc + t, 1);
      mbar_init(bar_act + t, PAIR ? 2 * kEpiWarps : kEpiThreads);  // PAIR: one arrival per epilogue warp of either CTA
    }
    mbar_init(bar_feat + 0, kEpiThreads);
    mbar_init(bar_feat + 1, kHeadThreads);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kMmaWarp) {
    __syncwarp();
    if (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(K::kTmemCols)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(K::kTmemCols)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();  // the peer's barriers are initialised and its TMEM allocated before anything reaches across
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp >= kHeadWarp) {
    // ===================== head warps: FC heads of group g while the pipeline already runs group g+1.  The last
    // group of a CTA is left to the epilogue warps (4x the threads, and they are idle by then) ==================
    const int htid = tid - kHeadWarp * 32;
    for (int gi = 0; gi + 1 < my_groups; ++gi) {
      const long long leaf0 = group_leaf0(gi);
      const int nvalid = group_valid(leaf0);
      mbar_wait(bar_feat + 0, (uint32_t)gi & 1u);
      if (headfeat_out != nullptr) export_heads<kHeadThreads, 2>(gm, nvalid, leaf0, htid, headf_s, headw_s + 192, headfeat_out, headfeat_lo_off, headfeat_kc8);
      else run_heads<kHeadThreads, 2>(gm, nb, nvalid, leaf0, htid, headf_s, fc_s, headw_s + 192, blob, L, pol_fc_t, val_fc1_t, probs, values);
      mbar_arrive(bar_feat + 1);  // features consumed, slots re-zeroed, scratch free
      if (htid == 0) TC_TRACE(5, gi);  // heads done
    }
  } else if (warp >= kMmaWarp) {
    // ===================== MMA issuers: the whole warp runs the loop (so that the descriptor arithmetic
    // stays warp-uniform -> uniform registers), one elected lane issues TMA / MMA / commit ====================
    const int mw = warp - kMmaWarp;  // 0: tiles 0,2   1: tiles 1,3 + weights
    uint32_t elected;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(elected));
    const uint32_t act_addr = smem_u32(act);
    const uint32_t wgt_addr = smem_u32(wgt);
    const int total_layers = my_groups * n_layers;
    auto load_layer = [&](int gl) {  // global layer index -> weight stage gl % kWStages (hi image, then lo)
      const int l = gl % n_layers;
      uint8_t* dst = wgt + (gl % K::kWStages) * K::kWStageBytes;
      uint64_t* bar = bar_w + (gl % K::kWStages);
      const int tap_bytes = l == 0 ? K::kTapBIn : K::kTapB;
      const int layer_bytes = 9 * tap_bytes;
      // global image: conv_in {hi, lo}, then per block {hi, lo}; PAIR: one compact image per rank, hi only, half the rows per tap
      const uint8_t* src = PAIR ? wimg + (size_t)rank * (9 * K::kTapBIn + (size_t)(n_layers - 1) * K::kLayerB) +
                                      (l == 0 ? 0 : 9 * K::kTapBIn + (size_t)(l - 1) * K::kLayerB)
                                : (l == 0 ? wimg : wimg + 2 * kLayerBytesIn + (size_t)(l - 1) * 2 * kLayerBytes);
      mbar_expect_tx(bar, (uint32_t)(K::kWParts * layer_bytes));
      for (int part = 0; part < K::kWParts; ++part)
        for (int tap = 0; tap < 9; ++tap)
          bulk_g2s(dst + part * K::kLayerB + tap * tap_bytes, src + (size_t)part * layer_bytes + tap * tap_bytes, tap_bytes, bar);
    };
    if (mw == 1 && elected) {
      load_layer(0);
      if (K::kWStages > 1 && total_layers > 1) load_layer(1);
    }
    if (PAIR && rank != 0) {
      // PAIR, peer CTA: the leader issues the MMAs of both.  Warp 9 keeps streaming this CTA's half of the weights -- layer gl+1
      // as soon as every tile of layer gl-1 has committed (the multicast commits arrive here too): its buffer is free then --,
      // warp 8 reports "weights landed" to the leader (a local wait, then one remote arrive per layer).
      if (mw == 1 && elected) {
        for (int gl = 1; gl + 1 < total_layers; ++gl) {
          for (int t = 0; t < K::kTiles; ++t) mbar_wait(bar_acc + t, (uint32_t)(gl - 1) & 1u);
          load_layer(gl + 1);
        }
      }
      if (mw == 0 && elected) {
        const uint32_t wp_leader = mapa_a(smem_u32(bar_wp), 0u);
        for (int gl = 0; gl < total_layers; ++gl) {
          mbar_wait(bar_w + (gl % K::kWStages), (uint32_t)(gl / K::kWStages) & 1u);
          mbar_arrive_cluster_a(wp_leader + 8u * (uint32_t)(gl % K::kWStages));
        }
      }
      __syncwarp();
    } else {
    // descriptor templates: only the 14-bit start-address field (units of 16 B) changes per MMA
    const uint64_t a_desc0 = make_desc(act_addr + (uint32_t)kHalo * 16u, K::kChunkBytes, 128u);
    const uint64_t b_desc0 = make_desc(wgt_addr, (uint32_t)K::kBRows * 16u, 128u);
    constexpr uint64_t kALo = (uint64_t)(K::kActBytes / 16);   // lo activation image
    constexpr uint64_t kBLo = (uint64_t)(K::kLayerB / 16);     // lo weight image
    // one MMA of this kernel: cta_group::1 (M = 128) or, PAIR, cta_group::2 (M = 256 over both CTAs, half of B from each)
    auto mma = [&](uint32_t d, uint64_t ad, uint64_t bd, uint32_t acc) {
      if (PAIR) umma_bf16_pair(d, ad, bd, rt_idesc_pair(64), acc);
      else umma_bf16(d, ad, bd, kIdesc, acc);
    };
    const int pitch = gm.pitch;
    for (int gl = 0; gl < total_layers; ++gl) {
      const bool first = (gl % n_layers) == 0;
      const uint64_t b_layer = b_desc0 + (uint64_t)((uint32_t)(gl % K::kWStages) * (K::kWStageBytes / 16));
      mbar_wait(bar_w + (gl % K::kWStages), (uint32_t)(gl / K::kWStages) & 1u);
      if (PAIR) mbar_wait(bar_wp + (gl % K::kWStages), (uint32_t)(gl / K::kWStages) & 1u);
      if (elected) TC_TRACE(6, gl * 2 + mw);  // weights present
      const uint32_t act_par = (uint32_t)gl & 1u;  // stage gl of bar_act = "input / epilogue of layer gl-1"
#pragma unroll 1
      for (int t = mw; t < K::kTiles; t += 2) {
        // MMA(gl,t) reads the rows of tiles t-1..t+1 as rewritten by the previous stage
        if (t > 0) mbar_wait(bar_act + t - 1, act_par);
        mbar_wait(bar_act + t, act_par);
        if (t + 1 < K::kTiles) mbar_wait(bar_act + t + 1, act_par);
        tc_fence_after();
        if (elected) TC_TRACE(0, gl * 4 + t);  // MMA issue start
        const uint32_t d_tmem = tmem_base + (uint32_t)(t * 64);
        const uint64_t a_tile = a_desc0 + (uint64_t)(uint32_t)(t * kTileRows);
        if (elected) {
          if (first) {  // conv_in: the 0/1 input planes are exact in bf16, so there is no lo activation term
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) {
              const int sh = (tap / 3 - 1) * pitch + (tap % 3 - 1);
              const uint64_t ad = a_tile + (uint64_t)(int64_t)sh;
              const uint64_t bd = b_layer + (uint64_t)(tap * (K::kTapBIn / 16));
              mma(d_tmem, ad, bd, tap > 0 ? 1u : 0u);
              if (K::kSplit) mma(d_tmem, ad, bd + kBLo, 1u);
            }
          } else {
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) {
              const int sh = (tap / 3 - 1) * pitch + (tap % 3 - 1);
#pragma unroll
              for (int kk = 0; kk < 4; ++kk) {
                const uint64_t ad = a_tile + (uint64_t)(int64_t)(sh + kk * 2 * K::kActRows);
                const uint64_t bd = b_layer + (uint64_t)(tap * (K::kTapB / 16) + kk * (2 * K::kBRows));
                mma(d_tmem, ad, bd, (tap | kk) ? 1u : 0u);
                if (K::kSplit) {
                  mma(d_tmem, ad + kALo, bd, 1u);   // lo(a) * hi(w)
                  mma(d_tmem, ad, bd + kBLo, 1u);   // hi(a) * lo(w)
                }
              }
            }
          }
          if (PAIR) umma_commit_pair_a(smem_u32(bar_acc + t));
          else umma_commit(bar_acc + t);
          TC_TRACE(1, gl * 4 + t);  // MMA issued + committed
        }
        __syncwarp();
        if (t == 1 && gl + 1 < total_layers) {
          if (K::kWStages > 1) {
            // tile 1 waited on the rewritten rows of tiles 0..2, whose epilogues waited on every commit of layer
            // gl-1: all MMAs of layer gl-1 are complete, its weight buffer is free for layer gl+1
            if (gl >= 1 && elected) load_layer(gl + 1);
          } else {
            // single weight buffer: layer gl+1 can only stream in once every MMA of layer gl has completed
            for (int tt = 0; tt < K::kTiles; ++tt) mbar_wait(bar_acc + tt, (uint32_t)gl & 1u);
            if (elected) load_layer(gl + 1);
            __syncwarp();
          }
        }
      }
    }
    }  // leader / single-CTA form
  } else {
    // ========================================= epilogue warps =========================================
    // Code size matters here (the v1 kernel was 127 KB of SASS and lived in instruction-cache misses):
    // tiles are a real loop, only the 32-channel body is unrolled.
    const int quarter = warp & 3, half = warp >> 2;
    const int row = quarter * 32 + (tid & 31);               // row of the tile = TMEM lane
    const uint32_t lane_base = (uint32_t)(quarter * 32) << 16;
    const int HW = gm.H * gm.W;
    float* featc = headf_s;  // dense head features [board][3][HW], accumulated by the two column halves
    // "tile t rewritten, accumulator drained".  PAIR: the barrier lives in the leader CTA and counts WARPS of both CTAs
    const uint32_t act_leader = PAIR ? mapa_a(smem_u32(bar_act), 0u) : 0u;
    auto act_arrive = [&](int t) {
      if (PAIR) {
        __syncwarp();
        if ((tid & 31) == 0) mbar_arrive_cluster_a(act_leader + 8u * (uint32_t)t);
      } else {
        mbar_arrive(bar_act + t);
      }
    };

    auto write_inputs = [&](long long leaf0) {
#pragma unroll 1
      for (int t = 0; t < K::kTiles; ++t) {
        const int p = t * kTileRows + row;
        uint32_t lo = 0u;
        if (half == 0) {
          const uint32_t tab = cell_tab[p];
          const long long leaf = leaf0 + (tab >> 9);
          if (tab != 0u && leaf < count) {
            const int cell = (int)(tab & 511u) - 1;
            const typename R::Board s = boards[leaf];
            const int wm = who[leaf];
            const int r = cell / gm.W, c = cell - r * gm.W;
            const uint32_t mine = rules.plane_value(s, wm, 0, r, c) ? 0x3F80u : 0u;  // bf16(1.0)
            const uint32_t other = rules.plane_value(s, wm, 1, r, c) ? 0x3F80u : 0u;
            lo = mine | (other << 16);
          }
        }
        *reinterpret_cast<uint4*>(act + (size_t)(half * K::kActRows + kHalo + p) * 16) = make_uint4(lo, 0u, 0u, 0u);
        fence_async_smem();
        act_arrive(t);
      }
    };

    write_inputs(group_leaf0(0));
    for (int gi = 0; gi < my_groups; ++gi) {
      const long long leaf0 = group_leaf0(gi);
#pragma unroll 1
      for (int layer = 0; layer < n_layers; ++layer) {
        const int gl = gi * n_layers + layer;
        const uint32_t acc_par = (uint32_t)gl & 1u;
        const bool last = layer == n_layers - 1;
        const bool has_res = layer > 0;
        const bool bias_in_smem = layer < kSmemBiasLayers;
        const float4* bl4 = reinterpret_cast<const float4*>(bias_s + (bias_in_smem ? layer : 0) * 64 + half * 32);
        const float4* bg4 = reinterpret_cast<const float4*>(bias_g + layer * 64 + half * 32);
#pragma unroll 1
        for (int t = 0; t < K::kTiles; ++t) {
          // tile t's own accumulator AND tile t+1's (it reads the tail rows of tile t as its halo); the two
          // tiles are issued by different warps, so neither commit implies the other
          mbar_wait(bar_acc + t, acc_par);
          if (t + 1 < K::kTiles) mbar_wait(bar_acc + t + 1, acc_par);
          __syncwarp();
          tc_fence_after();
          if (tid == 0) TC_TRACE(2, gl * 4 + t);  // epilogue start (warp 0)
          const int p = t * kTileRows + row;
          const uint32_t tab = cell_tab[p];
          const bool real = tab != 0u;
          const uint32_t a_acc = tmem_base + lane_base + (uint32_t)(t * 64 + half * 32);
          const uint32_t a_res = a_acc + (uint32_t)(K::kTiles * 64);
          uint32_t ra[32], rr[32];
          TMEM_LD16(a_acc, ra);
          TMEM_LD16(a_acc + 16u, (ra + 16));
          if (has_res) {
            TMEM_LD16(a_res, rr);
            TMEM_LD16(a_res + 16u, (rr + 16));
          }
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const float4 bq = bias_in_smem ? bl4[q] : __ldg(bg4 + q);
            const float bb[4] = {bq.x, bq.y, bq.z, bq.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int j = q * 4 + e;
              float v = lrelu_tc(__uint_as_float(ra[j]) + bb[e]);
              if (has_res) v += __uint_as_float(rr[j]);
              rr[j] = __float_as_uint(v);
            }
          }
          if (!last) {
            TMEM_ST16(a_res, rr);
            TMEM_ST16(a_res + 16u, (rr + 16));
#pragma unroll
            for (int c8 = 0; c8 < 4; ++c8) {
              uint32_t packed[4], packed_lo[4];
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float v0 = __uint_as_float(rr[c8 * 8 + 2 * j]), v1 = __uint_as_float(rr[c8 * 8 + 2 * j + 1]);
                const __nv_bfloat162 h = __floats2bfloat162_rn(v0, v1);
                packed[j] = real ? *reinterpret_cast<const uint32_t*>(&h) : 0u;
                if (K::kSplit) {  // lo = bf16(v - hi): the second 8 mantissa bits
                  const __nv_bfloat162 l2 = __floats2bfloat162_rn(v0 - __low2float(h), v1 - __high2float(h));
                  packed_lo[j] = real ? *reinterpret_cast<const uint32_t*>(&l2) : 0u;
                }
              }
              uint8_t* dst = act + (size_t)((half * 4 + c8) * K::kActRows + kHalo + p) * 16;
              *reinterpret_cast<uint4*>(dst) = make_uint4(packed[0], packed[1], packed[2], packed[3]);
              if (K::kSplit)
                *reinterpret_cast<uint4*>(dst + K::kActBytes) = make_uint4(packed_lo[0], packed_lo[1], packed_lo[2], packed_lo[3]);
            }
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            fence_async_smem();
            tc_fence_before();
            act_arrive(t);
            if (tid == 0) TC_TRACE(3, gl * 4 + t);  // epilogue done (warp 0)
          } else {
            // 1x1 head convolutions: this thread holds 32 of the 64 channels, the partner warp the rest
            const float4* hw4 = reinterpret_cast<const float4*>(headw_s + half * 32);
            float av = 0.0f, ap0 = 0.0f, ap1 = 0.0f;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              const float4 w0 = hw4[q], w1 = hw4[16 + q], w2 = hw4[32 + q];
              const float v0 = __uint_as_float(rr[q * 4]), v1 = __uint_as_float(rr[q * 4 + 1]);
              const float v2 = __uint_as_float(rr[q * 4 + 2]), v3 = __uint_as_float(rr[q * 4 + 3]);
              av = fmaf(v0, w0.x, fmaf(v1, w0.y, fmaf(v2, w0.z, fmaf(v3, w0.w, av))));
              ap0 = fmaf(v0, w1.x, fmaf(v1, w1.y, fmaf(v2, w1.z, fmaf(v3, w1.w, ap0))));
              ap1 = fmaf(v0, w2.x, fmaf(v1, w2.y, fmaf(v2, w2.z, fmaf(v3, w2.w, ap1))));
            }
            if (gi > 0 && t == 0) mbar_wait(bar_feat + 1, (uint32_t)(gi - 1) & 1u);  // slots re-zeroed by the head warps
            if (real) {  // two commutative contributions onto a zeroed slot: order-independent result
              const int b = (int)(tab >> 9), cell = (int)(tab & 511u) - 1;
              atomicAdd(&featc[(b * 3 + 0) * HW + cell], av);
              atomicAdd(&featc[(b * 3 + 1) * HW + cell], ap0);
              atomicAdd(&featc[(b * 3 + 2) * HW + cell], ap1);
            }
          }
        }
      }
      tc_fence_before();  // the last layer's accumulators have been read (wait::ld above)
      if (gi + 1 < my_groups) {
        mbar_arrive(bar_feat + 0);  // this thread's head features are in place (release) -> head warps
        write_inputs(group_leaf0(gi + 1));
        if (tid == 0) TC_TRACE(4, gi);  // last-layer epilogue + next inputs done
      } else {
        // last group of this CTA: nothing left to overlap with, so all eight epilogue warps do the heads
        asm volatile("bar.sync 1, 256;" ::: "memory");
        const int nvalid = group_valid(leaf0);
        if (headfeat_out != nullptr) export_heads<kEpiThreads, 1>(gm, nvalid, leaf0, tid, headf_s, headw_s + 192, headfeat_out, headfeat_lo_off, headfeat_kc8);
        else run_heads<kEpiThreads, 1>(gm, nb, nvalid, leaf0, tid, headf_s, fc_s, headw_s + 192, blob, L, pol_fc_t, val_fc1_t, probs, values);
        if (tid == 0) TC_TRACE(5, gi);
      }
    }
  }

  // ---- teardown ---------------------------------------------------------------------------------
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();  // no CTA of a pair leaves (or frees TMEM) while the other may still be signalled or read
  if (warp == kMmaWarp) {
    __syncwarp();
    if (PAIR) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(K::kTmemCols) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(K::kTmemCols) : "memory");
  }
}

// ------------------------------------------------------------------------------ host: packing
static uint16_t f32_to_bf16(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40u);  // NaN
  const uint32_t lsb = (u >> 16) & 1u;
  u += 0x7fffu + lsb;  // round to nearest even
  return (uint16_t)(u >> 16);
}

}  // namespace caro

using namespace caro;

int caro_net_tc_pack(caro_net* net, const float* h) {
  const BlobLayout& L = net->layout;
  // global image: conv_in {hi, lo}, then per residual block {hi, lo}; each part is a stack of 9 tap images in the
  // UMMA B-operand layout [8-channel chunk][n = 64 out channels][8 in channels] (no-swizzle K-major core matrices)
  const int blocks = L.blocks;
  const size_t img_bytes = 2 * ((size_t)kLayerBytesIn + (size_t)blocks * kLayerBytes);
  std::vector<uint16_t> img(img_bytes / 2, 0);
  auto put = [&](size_t part_base, size_t tap_bytes, int tap, int co, int ci, float w) {
    const uint16_t hi = f32_to_bf16(w);
    uint32_t hb = (uint32_t)hi << 16;
    float hf;
    memcpy(&hf, &hb, 4);
    const uint16_t lo = f32_to_bf16(w - hf);
    const size_t off = ((size_t)tap * tap_bytes + (size_t)((ci / 8) * 64 + co) * 16) / 2 + (ci % 8);
    img[part_base / 2 + off] = hi;
    img[(part_base + 9 * tap_bytes) / 2 + off] = lo;
  };
  for (int tap = 0; tap < 9; ++tap)
    for (int co = 0; co < 64; ++co)
      for (int ci = 0; ci < 2; ++ci) put(0, kTapBytesIn, tap, co, ci, h[L.conv_in_w + ((size_t)(co * 2 + ci) * 9 + tap)]);
  for (int l = 0; l < blocks; ++l) {
    const size_t base = 2 * (size_t)kLayerBytesIn + (size_t)l * 2 * kLayerBytes;
    for (int tap = 0; tap < 9; ++tap)
      for (int co = 0; co < 64; ++co)
        for (int ci = 0; ci < 64; ++ci) put(base, kTapBytes, tap, co, ci, h[L.conv_w[l] + ((size_t)(co * 64 + ci) * 9 + tap)]);
  }
  std::vector<float> bias((size_t)(1 + blocks) * 64);
  for (int co = 0; co < 64; ++co) bias[co] = h[L.conv_in_b + co];
  for (int l = 0; l < blocks; ++l)
    for (int co = 0; co < 64; ++co) bias[(size_t)(l + 1) * 64 + co] = h[L.conv_b[l] + co];
  const int HW = net->H * net->W, A = net->A;
  // transposed FC weights, policy [2*HW][A] followed by value-FC1 [HW][20]: a warp's outputs read contiguous floats
  std::vector<float> polt((size_t)2 * HW * A + (size_t)HW * 20);
  for (int a = 0; a < A; ++a)
    for (int i = 0; i < 2 * HW; ++i) polt[(size_t)i * A + a] = h[L.pol_fc_w + (size_t)a * 2 * HW + i];
  for (int i = 0; i < 20; ++i)
    for (int c = 0; c < HW; ++c) polt[(size_t)2 * HW * A + (size_t)c * 20 + i] = h[L.val_fc1_w + (size_t)i * HW + c];
  cudaError_t ce = cudaSuccess;
  if (HW > kHeadsInTowerMaxHW && caro_net_heads_supported(net)) {  // large boards: FC heads on the tensor cores from exported features
    if (!net->d_headfeat) {
      net->headfeat_leaves = 32768;  // per slot; larger launches fall back to the FC heads inside the tower
      // one slot = hi + lo image of [leaves / 128][K / 8][128][8] bf16 (738 MB in all for 15x15)
      const size_t image = (size_t)net->headfeat_leaves * caro_net_heads_kc64(net) * 64 * 2;
      ce = cudaMalloc(&net->d_headfeat, (size_t)kHeadfeatSlots * 2 * image);
      if (ce != cudaSuccess) return caro_fail(CARO_E_CUDA, cudaGetErrorString(ce));
    }
    const int hrc = caro_net_heads_pack(net, h);
    if (hrc != CARO_OK) return hrc;
  }
  // CTA-pair form: one compact image per cluster rank (hi part only): per tap [8-channel chunk][32 of the 64 out channels][8]
  const size_t pair_bytes = 9 * (size_t)TcPair::kTapBIn + (size_t)blocks * TcPair::kLayerB;
  std::vector<uint16_t> pimg(2 * pair_bytes / 2, 0);
  for (int r = 0; r < 2; ++r) {
    auto copy_taps = [&](size_t src_base, size_t src_tap_bytes, size_t dst_base, size_t dst_tap_bytes, int chunks) {
      for (int tap = 0; tap < 9; ++tap)
        for (int ch = 0; ch < chunks; ++ch)
          for (int row = 0; row < 32; ++row)
            for (int e = 0; e < 8; ++e)
              pimg[((size_t)r * pair_bytes + dst_base + tap * dst_tap_bytes + (size_t)(ch * 32 + row) * 16) / 2 + e] =
                  img[(src_base + tap * src_tap_bytes + (size_t)(ch * 64 + 32 * r + row) * 16) / 2 + e];
    };
    copy_taps(0, kTapBytesIn, 0, TcPair::kTapBIn, 2);
    for (int l = 0; l < blocks; ++l)
      copy_taps(2 * (size_t)kLayerBytesIn + (size_t)l * 2 * kLayerBytes, kTapBytes, 9 * (size_t)TcPair::kTapBIn + (size_t)l * TcPair::kLayerB,
                TcPair::kTapB, 8);
  }
  if (!net->d_tc_pair_weights) ce = cudaMalloc(&net->d_tc_pair_weights, 2 * pair_bytes);
  if (ce == cudaSuccess) ce = cudaMemcpy(net->d_tc_pair_weights, pimg.data(), 2 * pair_bytes, cudaMemcpyHostToDevice);
  if (ce == cudaSuccess && !net->d_tc_weights) ce = cudaMalloc(&net->d_tc_weights, img_bytes);
  if (ce == cudaSuccess && !net->d_tc_bias) ce = cudaMalloc(&net->d_tc_bias, bias.size() * sizeof(float));
  if (ce == cudaSuccess && !net->d_pol_fc_t) ce = cudaMalloc(&net->d_pol_fc_t, polt.size() * sizeof(float));
  if (ce == cudaSuccess) ce = cudaMemcpy(net->d_tc_weights, img.data(), img_bytes, cudaMemcpyHostToDevice);
  if (ce == cudaSuccess) ce = cudaMemcpy(net->d_tc_bias, bias.data(), bias.size() * sizeof(float), cudaMemcpyHostToDevice);
  if (ce == cudaSuccess) ce = cudaMemcpy(net->d_pol_fc_t, polt.data(), polt.size() * sizeof(float), cudaMemcpyHostToDevice);
  if (ce != cudaSuccess) return caro_fail(CARO_E_CUDA, cudaGetErrorString(ce));
  return CARO_OK;
}

void caro_net_tc_free(caro_net* net) {
  if (net->d_tc_weights) cudaFree(net->d_tc_weights);
  if (net->d_tc_pair_weights) cudaFree(net->d_tc_pair_weights);
  net->d_tc_pair_weights = nullptr;
  if (net->d_tc_bias) cudaFree(net->d_tc_bias);
  if (net->d_pol_fc_t) cudaFree(net->d_pol_fc_t);
  if (net->d_headfeat) cudaFree(net->d_headfeat);
  net->d_headfeat = nullptr;
  net->d_tc_weights = nullptr;
  net->d_tc_bias = nullptr;
  net->d_pol_fc_t = nullptr;
}

template <class R, class K>
static int launch_tc(const R& rules, caro_net* net, const void* boards, const uint8_t* who, const int32_t* d_count,
                     int64_t max_count, float* probs, float* values, cudaStream_t st) {
  TcGeom gm;
  gm.H = net->H;
  gm.W = net->W;
  gm.A = net->A;
  gm.pitch = net->W + 1;
  gm.block = (net->H + 1) * gm.pitch;
  // as many boards as the group's rows hold, capped by the 32-board limit and the FC scratch (only 2 x 2 boards reach the
  // caps: the rows past the last board are padding)
  gm.boards_per_group = std::min(std::min(K::kGroupRows / gm.block, 32), K::kFcFloats / (20 + gm.A));
  if (gm.boards_per_group < 1 || gm.pitch + 1 > kHalo)
    return caro_fail(CARO_E_ARG, "board does not fit the tensor-core tile geometry");
  const int lim = net->grid_limit > 0 ? net->grid_limit : net->pipeline_limit;
  const int sm_count = lim > 0 && lim < net->sm_count ? lim : net->sm_count;
  auto kern = net_tc_kernel<R, K>;
  const long long max_groups = (max_count + gm.boards_per_group - 1) / gm.boards_per_group;
  const unsigned grid = (unsigned)(max_groups < sm_count ? max_groups : sm_count);
  const int HW = net->H * net->W;
  // the exported head features go to one of kHeadfeatSlots scratch slots, round robin per launch: launches of different
  // parts of the self-play pipeline can be in flight at the same time on different streams (and the slot is baked
  // into a captured graph node), so they must not share a buffer
  uint8_t* headfeat = nullptr;
  const int kc64 = caro_net_heads_kc64(net);
  const size_t image = (size_t)net->headfeat_leaves * kc64 * 64 * 2;  // bytes of one (hi or lo) image of a slot
  if (net->d_headfeat != nullptr && max_count <= net->headfeat_leaves)
    headfeat = (uint8_t*)net->d_headfeat + (size_t)(net->headfeat_seq++ % kHeadfeatSlots) * 2 * image;
  if (K::kPair) {  // clusters of two CTAs (one TPC each)
    const long long max_units = (max_groups + 1) / 2;
    const long long max_pairs = sm_count / 2 > 0 ? sm_count / 2 : 1;
    const unsigned pairs = (unsigned)(max_units < max_pairs ? max_units : max_pairs);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * pairs);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = K::kTotal;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const cudaError_t ce = cudaLaunchKernelEx(&cfg, kern, rules, gm, (const typename R::Board*)boards, who, d_count, (long long)max_count,
                                              (const uint8_t*)net->d_tc_pair_weights, (const float*)net->d_tc_bias, (const float*)net->d_blob,
                                              net->layout, (const float*)net->d_pol_fc_t,
                                              (const float*)(net->d_pol_fc_t + (size_t)2 * HW * net->A), probs, values, headfeat, image,
                                              kc64 * 8, (long long*)net->d_trace);
    if (ce != cudaSuccess) return caro_fail(CARO_E_CUDA, cudaGetErrorString(ce));
  } else {
    kern<<<grid, kThreads, K::kTotal, st>>>(rules, gm, (const typename R::Board*)boards, who, d_count, (long long)max_count,
                                            (const uint8_t*)net->d_tc_weights, net->d_tc_bias, net->d_blob, net->layout,
                                            net->d_pol_fc_t, net->d_pol_fc_t + (size_t)2 * HW * net->A, probs, values, headfeat, image,
                                            kc64 * 8, (long long*)net->d_trace);
  }
  int rc = caro_check_launch("net_tc_kernel");
  if (rc == CARO_OK && headfeat != nullptr) rc = caro_net_heads_forward(net, headfeat, image, d_count, max_count, probs, values, st);
  return rc;
}

// Sets the dynamic shared memory attribute of every instantiation up front (caro_net_create), so that no
// attribute call can fall inside a CUDA-graph capture of the search loop.
int caro_net_tc_prepare() {
  cudaError_t ce = cudaFuncSetAttribute(net_tc_kernel<C4Rules, TcFast>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcFast::kTotal);
  if (ce == cudaSuccess) ce = cudaFuncSetAttribute(net_tc_kernel<C4Rules, TcExact>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcExact::kTotal);
  if (ce == cudaSuccess) ce = cudaFuncSetAttribute(net_tc_kernel<MnkRules, TcFast>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcFast::kTotal);
  if (ce == cudaSuccess) ce = cudaFuncSetAttribute(net_tc_kernel<MnkRules, TcExact>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcExact::kTotal);
  if (ce == cudaSuccess) ce = cudaFuncSetAttribute(net_tc_kernel<C4Rules, TcPair>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcPair::kTotal);
  if (ce == cudaSuccess) ce = cudaFuncSetAttribute(net_tc_kernel<MnkRules, TcPair>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcPair::kTotal);
  if (ce != cudaSuccess) return caro_fail(CARO_E_CUDA, cudaGetErrorString(ce));
  return CARO_OK;
}

int caro_net_tc_forward(caro_net* net, int game, int n, int k, const void* d_boards, const uint8_t* d_who,
                        const int32_t* d_count, int64_t max_count, float* d_probs, float* d_values, int exact, cudaStream_t st) {
  // exact: 0 = one pass, 1 = split precision, 2 = one pass as CTA pairs (cta_group::2); CARO_TC_PAIR=1 turns 0 into 2
  static const bool pair_env = getenv("CARO_TC_PAIR") ? atoi(getenv("CARO_TC_PAIR")) != 0 : false;
  if (exact == 0 && pair_env) exact = 2;
  if (game == CARO_GAME_CONNECT4) {
    if (exact == 1) return launch_tc<C4Rules, TcExact>(C4Rules(), net, d_boards, d_who, d_count, max_count, d_probs, d_values, st);
    if (exact == 2) return launch_tc<C4Rules, TcPair>(C4Rules(), net, d_boards, d_who, d_count, max_count, d_probs, d_values, st);
    return launch_tc<C4Rules, TcFast>(C4Rules(), net, d_boards, d_who, d_count, max_count, d_probs, d_values, st);
  }
  if (exact == 1) return launch_tc<MnkRules, TcExact>(MnkRules{n, k}, net, d_boards, d_who, d_count, max_count, d_probs, d_values, st);
  if (exact == 2) return launch_tc<MnkRules, TcPair>(MnkRules{n, k}, net, d_boards, d_who, d_count, max_count, d_probs, d_values, st);
  return launch_tc<MnkRules, TcFast>(MnkRules{n, k}, net, d_boards, d_who, d_count, max_count, d_probs, d_values, st);
}
