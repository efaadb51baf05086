// Fused policy/value tower of 128-filter networks on the tcgen05 tensor cores, sm_100a only.
//
// The tap-per-MMA implicit GEMM of net_tc.cu (no im2col: activations in the no-swizzle K-major core-matrix layout,
// every 3x3 tap is a shift of the A descriptor's start address), re-planned for 128 channels:
//   * one MMA is M = 128 rows x N = 128 output channels x K = 16; a residual layer is 9 taps x 8 k-steps = 72 MMAs per
//     tile.  With N = 128 one MMA fetches 4 KB of A and 4 KB of B, which at 128 B/clk matches its 64-cycle tensor floor
//     (at 64 filters the operand path was 1.5x the floor, DESIGN.md section 4);
//   * TMEM: two tiles of 128 fp32 accumulator columns + two tiles of 128 fp32 residual-stream columns = all 512
//     columns, so a CTA takes a group of 2 tiles = 256 padded positions (row pitch W+1, one zero row after every board);
//   * shared memory: one fp16 / bf16 activation image (296 rows x 128 channels, 75,776 B) rewritten in place, and a ring
//     of 4 weight slots of one tap each (128 x 128 x 2 B = 32 KB; a layer is 288 KB and cannot be resident).  A producer
//     warp streams taps into the ring with cp.async.bulk (full / empty mbarriers); the MMA warp issues each tap for both
//     tiles before releasing its slot, so every weight byte is read from L2 once per group and layer;
//   * per layer the MMAs of both tiles run, then the epilogue (bias, LeakyReLU, residual add in fp32 TMEM, the fp16 /
//     bf16 copy back to shared memory) -- the next layer's taps need the rows of both tiles, so the two phases do not
//     overlap within a CTA;
//   * heads: the 1x1 head convolutions reduce over 128 channels in the last epilogue; boards with HW <= 64 run the FC
//     heads and the softmax in the kernel (run_heads), larger boards export the activated head features for
//     heads_tc_kernel (net_heads.cu), whose K = 3 HW does not depend on the width.
// The operand mode is a compile-time switch (WideOps): fp16, bf16, or bf16 hi + lo pairs (lo = bf16(x - bf16(x))) with
// every product evaluated as hi*hi + lo*hi + hi*lo, the arithmetic of net_tc.cu's SPLIT form, for trained networks whose
// logits one 8-bit-mantissa pass cannot hold to 1e-3.  The split mode keeps a hi and a lo activation image (151,552 B)
// and streams each tap's hi and lo weight images through a ring of two 32 KB slots.  The residual stream is fp32 in every
// mode.  Every sum has a fixed order, so a leaf's outputs do not depend on the batch, the grid or d_count.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math.h>

#include <algorithm>
#include <vector>

#include "../../include/caro_b200.h"
#include "common_host.h"
#include "net.h"
#include "rules.cuh"

#include "tc_common.cuh"
#include "rt_common.cuh"

namespace caro {
namespace wide {

constexpr int F = kWideFilters;
constexpr int kTiles = 2;
constexpr int kTileRows = 128;
constexpr int kHalo = 20;                             // zero positions before / after the group (>= pitch + 1)
constexpr int kGroupRows = kTiles * kTileRows;        // 256
constexpr int kActRows = kGroupRows + 2 * kHalo;      // 296
constexpr int kChunkBytes = kActRows * 16;            // one 8-channel chunk of all positions
constexpr int kActBytes = (F / 8) * kChunkBytes;      // 75,776
constexpr int kTapBytes = (F / 8) * F * 16;           // 32,768: one tap of a 128 -> 128 layer, [ci / 8][co][ci % 8]
constexpr int kTapBytesIn = 2 * F * 16;               // 4,096: one tap of conv_in (K padded to 16)
constexpr int kLayerBytesIn = 9 * kTapBytesIn;
constexpr int kLayerBytes = 9 * kTapBytes;
constexpr int kHeadfeatSlots = 8;                     // scratch slots for exported head features (launches in flight)
constexpr int kHeadsInTowerMaxHW = 64;                // larger boards run their FC heads in heads_tc_kernel
constexpr int kFcFloats = 512;                        // FC scratch: hidden[nb][20] + logits[nb][A]
constexpr uint32_t kTmemCols = 2 * kTiles * F;        // 512

constexpr int kEpiWarps = 8;   // warps 0-7: epilogue; TMEM lane quarter = warp & 3, channel half = warp >> 2
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr int kMmaWarp = kEpiWarps;       // warp 8: TMEM owner, MMA issue
constexpr int kLoadWarp = kEpiWarps + 1;  // warp 9: weight streaming
constexpr int kThreads = kEpiThreads + 64;

enum WideOps { kOpsF16 = 0, kOpsBf16 = 1, kOpsBf16x3 = 2 };

// Per operand mode: the weight ring and the dynamic shared memory carve-up (byte offsets).
template <int OPS>
struct WideCfg {
  static constexpr bool kF16 = OPS == kOpsF16;
  static constexpr bool kSplit = OPS == kOpsBf16x3;
  static constexpr int kParts = kSplit ? 2 : 1;  // images of the activations and of every weight tap: hi (+ lo)
  // weight ring of 32 KB slots, one tap image each: one-pass 4 taps in flight, split 2 (on a B200, 2 x 32 KB slots ran the
  // split tower 3-5 % faster than 4 x 16 KB half images: profiles/r4_wide_split_ring.jsonl)
  static constexpr int kSlots = kSplit ? 2 : 4;
  static constexpr int kAct = 0;
  static constexpr int kWgt = kAct + kParts * kActBytes;
  static constexpr int kHeadW = kWgt + kSlots * kTapBytes;         // float [3][128] head conv weights + [3] biases
  static constexpr int kHeadF = kHeadW + 400 * 4;                  // float [rows][3] head features
  static constexpr int kFc = kHeadF + kGroupRows * 3 * 4;
  static constexpr int kCellTab = kFc + kFcFloats * 4;             // uint16 [rows]: (board << 9) | (cell + 1), 0 = padding
  static constexpr int kBars = kCellTab + kGroupRows * 2;
  static constexpr int kTotal = kBars + 128;
  static_assert(kTotal <= 232448, "exceeds the 227 KB shared memory of an sm_100 CTA");
  static_assert(kWgt % 128 == 0 && kBars % 8 == 0, "alignment");
};
static_assert(WideCfg<kOpsBf16x3>::kTotal == 224448, "split mode: 2 x 75,776 B activations + 2 x 32 KB ring + 7,360 B");

template <bool F16>
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  if (F16) {
    const __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&h);
  }
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}

// The lo halves of a bf16 hi pair (a in the low 16 bits): bf16(a - hi(a)), bf16(b - hi(b)); the differences are exact.
__device__ __forceinline__ uint32_t pack2_lo(uint32_t hi, float a, float b) {
  return pack2<false>(a - __uint_as_float(hi << 16), b - __uint_as_float(hi & 0xffff0000u));
}

// Roles: warps 0-7 = epilogue (warp w: TMEM lanes [32(w&3), +32) = rows of both tiles, channels 64(w>>2)..+64, read in
//        32-column chunks), warp 8 = TMEM allocation + elected-lane MMA issue, warp 9 = elected-lane weight streaming.
// Barriers: full[s] / empty[s] = weight slot s landed / read by its MMAs; acc = every MMA of a layer complete;
//           act = the layer's input rows written and the accumulators drained (kEpiThreads arrivals).
// Weight stream: per tap its image (one-pass) or its hi, then its lo image (split), one ring slot each.  Per image and
// tile the MMAs run K-step by K-step: the hi image issues a_hi*w_hi then a_lo*w_hi, the lo image a_hi*w_lo (conv_in: its
// 0/1 input planes have no lo part, so only a_hi*w_hi and a_hi*w_lo).
// Timeline (caro_net_set_trace, CTA 0, slot = kind * 1000 + global layer): 0 = layer input ready (MMA warp), 1 = last
// commit of the layer issued, 2 = accumulators complete (epilogue warp 0), 3 = epilogue done, 4 = cycles the MMA warp
// waited for weight slots during the layer (a count, not a clock).
template <class R, int OPS>
__global__ void __launch_bounds__(kThreads, 1)
net_wide_kernel(R rules, TcGeom gm, const typename R::Board* __restrict__ boards, const uint8_t* __restrict__ who,
                const int32_t* __restrict__ d_count, long long max_count, const uint8_t* __restrict__ wimg, size_t wimg_lo_off,
                const float* __restrict__ bias_g, const float* __restrict__ blob, BlobLayout L,
                const float* __restrict__ pol_fc_t, const float* __restrict__ val_fc1_t, float* __restrict__ probs,
                float* __restrict__ values, uint8_t* __restrict__ headfeat_out, size_t headfeat_lo_off, int headfeat_kc8,
                long long* __restrict__ trace) {
  using K = WideCfg<OPS>;
  constexpr bool F16 = K::kF16;
  constexpr int kSlots = K::kSlots;
  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t* act = smem + K::kAct;
  uint8_t* wgt = smem + K::kWgt;
  float* headw_s = reinterpret_cast<float*>(smem + K::kHeadW);
  float* headf_s = reinterpret_cast<float*>(smem + K::kHeadF);
  float* fc_s = reinterpret_cast<float*>(smem + K::kFc);
  uint16_t* cell_tab = reinterpret_cast<uint16_t*>(smem + K::kCellTab);
  uint64_t* bar_full = reinterpret_cast<uint64_t*>(smem + K::kBars);
  uint64_t* bar_empty = bar_full + kSlots;
  uint64_t* bar_acc = bar_empty + kSlots;
  uint64_t* bar_act = bar_acc + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_act + 1);

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const long long count = d_count ? min((long long)*d_count, max_count) : max_count;
  const int nb = gm.boards_per_group;
  const long long n_groups = (count + nb - 1) / nb;
  if ((long long)blockIdx.x >= n_groups) return;  // uniform per CTA, before any barrier / TMEM use
  const int my_groups = (int)((n_groups - blockIdx.x + gridDim.x - 1) / gridDim.x);
  auto group_leaf0 = [&](int gi) { return ((long long)blockIdx.x + (long long)gi * gridDim.x) * nb; };
  const int n_layers = 1 + L.blocks;

  // ---- one-time setup ---------------------------------------------------------------------
  for (int i = tid; i < K::kParts * kActBytes / 16; i += kThreads) reinterpret_cast<uint4*>(act)[i] = make_uint4(0, 0, 0, 0);
  for (int p = tid; p < kGroupRows; p += kThreads) {
    const int b = p / gm.block, within = p - b * gm.block;
    const int r = within / gm.pitch, c = within - r * gm.pitch;
    cell_tab[p] = (b < nb && r < gm.H && c < gm.W) ? (uint16_t)((b << 9) | (r * gm.W + c + 1)) : (uint16_t)0;
  }
  for (int i = tid; i < kGroupRows * 3; i += kThreads) headf_s[i] = 0.0f;
  for (int i = tid; i < F; i += kThreads) {
    headw_s[i] = blob[L.val_conv_w + i];
    headw_s[F + i] = blob[L.pol_conv_w + i];
    headw_s[2 * F + i] = blob[L.pol_conv_w + F + i];
  }
  if (tid == 0) {
    headw_s[3 * F] = blob[L.val_conv_b];
    headw_s[3 * F + 1] = blob[L.pol_conv_b];
    headw_s[3 * F + 2] = blob[L.pol_conv_b + 1];
    for (int s = 0; s < kSlots; ++s) {
      mbar_init(bar_full + s, 1);
      mbar_init(bar_empty + s, 1);
    }
    mbar_init(bar_acc, 1);
    mbar_init(bar_act, kEpiThreads);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kMmaWarp) {
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int total_layers = my_groups * n_layers;

  if (warp == kLoadWarp) {
    // ===================== weight producer: tap images in issue order, kSlots ahead of the MMAs =====================
    if ((tid & 31) == 0) {
      int g = 0;
      for (int gl = 0; gl < total_layers; ++gl) {
        const int l = gl % n_layers;
        const int tap_bytes = l == 0 ? kTapBytesIn : kTapBytes;
        const uint8_t* src = l == 0 ? wimg : wimg + kLayerBytesIn + (size_t)(l - 1) * kLayerBytes;
        for (int tap = 0; tap < 9; ++tap) {
          for (int part = 0; part < K::kParts; ++part, ++g) {
            const int s = g % kSlots;
            if (g >= kSlots) mbar_wait(bar_empty + s, (uint32_t)(g / kSlots - 1) & 1u);
            mbar_expect_tx(bar_full + s, (uint32_t)tap_bytes);
            bulk_g2s(wgt + s * kTapBytes, src + part * wimg_lo_off + (size_t)tap * tap_bytes, (uint32_t)tap_bytes, bar_full + s);
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == kMmaWarp) {
    // ===================== MMA issue: tap-major, both tiles per tap image ==========================================
    uint32_t elected;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(elected));
    const uint64_t a_desc0 = make_desc(smem_u32(act) + (uint32_t)kHalo * 16u, kChunkBytes, 128u);
    const uint64_t b_desc0 = make_desc(smem_u32(wgt), (uint32_t)F * 16u, 128u);
    constexpr uint64_t kALo = (uint64_t)(kActBytes / 16);  // lo activation image
    constexpr uint32_t idesc = rt_idesc_fmt<F16>((uint32_t)F);
    const int pitch = gm.pitch;
    int g = 0;
    for (int gl = 0; gl < total_layers; ++gl) {
      const bool first = (gl % n_layers) == 0;
      mbar_wait(bar_act, (uint32_t)gl & 1u);
      tc_fence_after();
      if (elected) TC_TRACE(0, gl);
      long long wait_cycles = 0;
#pragma unroll 1
      for (int tap = 0; tap < 9; ++tap) {
        const int sh = (tap / 3 - 1) * pitch + (tap % 3 - 1);
#pragma unroll 1
        for (int part = 0; part < K::kParts; ++part, ++g) {
          const int s = g % kSlots;
          if (trace != nullptr) {
            const long long t0 = clock64();
            mbar_wait(bar_full + s, (uint32_t)(g / kSlots) & 1u);
            wait_cycles += clock64() - t0;
          } else {
            mbar_wait(bar_full + s, (uint32_t)(g / kSlots) & 1u);
          }
          tc_fence_after();
          const bool w_lo = part == 1;
          const uint64_t bd = b_desc0 + (uint64_t)(uint32_t)(s * (kTapBytes / 16));
          if (elected) {
#pragma unroll
            for (int t = 0; t < kTiles; ++t) {
              const uint32_t d = tmem_base + (uint32_t)(t * F);
              const uint64_t ad = a_desc0 + (uint64_t)(int64_t)(t * kTileRows + sh);
              if (first) {  // conv_in: K = 2 input planes padded to 16 (split: a_hi * w_hi, then a_hi * w_lo)
                umma_bf16(d, ad, bd, idesc, (tap > 0 || w_lo) ? 1u : 0u);
              } else {
#pragma unroll
                for (int kk = 0; kk < F / 16; ++kk) {
                  const uint64_t a = ad + (uint64_t)(kk * 2 * kActRows);
                  const uint64_t b = bd + (uint64_t)(kk * 2 * F);
                  if (w_lo) {
                    umma_bf16(d, a, b, idesc, 1u);  // hi(a) * lo(w)
                  } else {
                    umma_bf16(d, a, b, idesc, (tap | kk) ? 1u : 0u);
                    if (K::kSplit) umma_bf16(d, a + kALo, b, idesc, 1u);  // lo(a) * hi(w)
                  }
                }
              }
            }
            umma_commit(bar_empty + s);  // the slot is free once these MMAs have read it
            if (tap == 8 && part == K::kParts - 1) umma_commit(bar_acc);
          }
          __syncwarp();
        }
      }
      if (elected) {
        TC_TRACE(1, gl);
        if (trace != nullptr && blockIdx.x == 0 && gl < 1000) trace[4000 + gl] = wait_cycles;
      }
    }
  } else {
    // ========================================= epilogue warps =========================================
    const int quarter = warp & 3, half = warp >> 2;
    const int row = quarter * 32 + (tid & 31);
    const uint32_t lane_base = (uint32_t)(quarter * 32) << 16;
    const int HW = gm.H * gm.W;
    const float* head_b = headw_s + 3 * F;  // the three head biases

    auto write_inputs = [&](long long leaf0) {
#pragma unroll 1
      for (int t = 0; t < kTiles; ++t) {
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
            const uint32_t one = F16 ? 0x3C00u : 0x3F80u;
            const uint32_t mine = rules.plane_value(s, wm, 0, r, c) ? one : 0u;
            const uint32_t other = rules.plane_value(s, wm, 1, r, c) ? one : 0u;
            lo = mine | (other << 16);
          }
        }
        // half 0 writes input channels 0..7 (the two planes), half 1 zeroes channels 8..15: conv_in reads K = 16
        *reinterpret_cast<uint4*>(act + (size_t)(half * kActRows + kHalo + p) * 16) = make_uint4(lo, 0u, 0u, 0u);
      }
      fence_async_smem();
      mbar_arrive(bar_act);
    };

    write_inputs(group_leaf0(0));
    for (int gi = 0; gi < my_groups; ++gi) {
      const long long leaf0 = group_leaf0(gi);
      const int nvalid = (int)max(0ll, min((long long)nb, count - leaf0));
#pragma unroll 1
      for (int layer = 0; layer < n_layers; ++layer) {
        const int gl = gi * n_layers + layer;
        const bool last = layer == n_layers - 1;
        const bool has_res = layer > 0;
        mbar_wait(bar_acc, (uint32_t)gl & 1u);
        __syncwarp();
        tc_fence_after();
        if (tid == 0) TC_TRACE(2, gl);
#pragma unroll 1
        for (int t = 0; t < kTiles; ++t) {
          const int p = t * kTileRows + row;
          const uint32_t tab = cell_tab[p];
          const bool real = tab != 0u;
          float av = 0.0f, ap0 = 0.0f, ap1 = 0.0f;
#pragma unroll 1
          for (int c = 0; c < 2; ++c) {
            const int ch0 = half * 64 + c * 32;  // first of this chunk's 32 channels
            const uint32_t a_acc = tmem_base + lane_base + (uint32_t)(t * F + ch0);
            const uint32_t a_res = a_acc + (uint32_t)(kTiles * F);
            uint32_t ra[32], rr[32];
            TMEM_LD16(a_acc, ra);
            TMEM_LD16(a_acc + 16u, (ra + 16));
            if (has_res) {
              TMEM_LD16(a_res, rr);
              TMEM_LD16(a_res + 16u, (rr + 16));
            }
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            const float4* bg4 = reinterpret_cast<const float4*>(bias_g + (size_t)layer * F + ch0);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              const float4 bq = __ldg(bg4 + q);
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
                  packed[j] = real ? pack2<F16>(v0, v1) : 0u;
                  if (K::kSplit) packed_lo[j] = real ? pack2_lo(packed[j], v0, v1) : 0u;
                }
                uint8_t* dst = act + (size_t)((ch0 / 8 + c8) * kActRows + kHalo + p) * 16;
                *reinterpret_cast<uint4*>(dst) = make_uint4(packed[0], packed[1], packed[2], packed[3]);
                if (K::kSplit) *reinterpret_cast<uint4*>(dst + kActBytes) = make_uint4(packed_lo[0], packed_lo[1], packed_lo[2], packed_lo[3]);
              }
            } else {  // 1x1 head convolutions over this chunk's 32 channels, in channel order
              const float4* hw4 = reinterpret_cast<const float4*>(headw_s + ch0);
#pragma unroll
              for (int q = 0; q < 8; ++q) {
                const float4 w0 = hw4[q], w1 = hw4[F / 4 + q], w2 = hw4[F / 2 + q];
                const float v0 = __uint_as_float(rr[q * 4]), v1 = __uint_as_float(rr[q * 4 + 1]);
                const float v2 = __uint_as_float(rr[q * 4 + 2]), v3 = __uint_as_float(rr[q * 4 + 3]);
                av = fmaf(v3, w0.w, fmaf(v2, w0.z, fmaf(v1, w0.y, fmaf(v0, w0.x, av))));
                ap0 = fmaf(v3, w1.w, fmaf(v2, w1.z, fmaf(v1, w1.y, fmaf(v0, w1.x, ap0))));
                ap1 = fmaf(v3, w2.w, fmaf(v2, w2.z, fmaf(v1, w2.y, fmaf(v0, w2.x, ap1))));
              }
            }
          }
          if (last && real) {  // two commutative contributions (the channel halves) onto a zeroed slot: order-independent
            const int b = (int)(tab >> 9), cell = (int)(tab & 511u) - 1;
            atomicAdd(&headf_s[(b * 3 + 0) * HW + cell], av);
            atomicAdd(&headf_s[(b * 3 + 1) * HW + cell], ap0);
            atomicAdd(&headf_s[(b * 3 + 2) * HW + cell], ap1);
          }
        }
        if (!last) {
          asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
          fence_async_smem();
          tc_fence_before();
          mbar_arrive(bar_act);
        }
        if (tid == 0) TC_TRACE(3, gl);
      }
      tc_fence_before();  // the last layer's accumulators have been read (wait::ld above)
      if (gi + 1 < my_groups) write_inputs(group_leaf0(gi + 1));  // the next group's conv_in runs under these heads
      asm volatile("bar.sync 1, 256;" ::: "memory");              // every head feature of the group is in place
      if (headfeat_out != nullptr)
        export_heads<kEpiThreads, 1>(gm, nvalid, leaf0, tid, headf_s, head_b, headfeat_out, headfeat_lo_off, headfeat_kc8);
      else
        run_heads<kEpiThreads, 1>(gm, nb, nvalid, leaf0, tid, headf_s, fc_s, head_b, blob, L, pol_fc_t, val_fc1_t, probs, values);
    }
  }

  // ---- teardown ---------------------------------------------------------------------------------
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    __syncwarp();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

template <class R, int OPS>
static int launch_wide(const R& rules, caro_net* net, const void* boards, const uint8_t* who, const int32_t* d_count,
                       int64_t max_count, float* probs, float* values, cudaStream_t st) {
  TcGeom gm;
  gm.H = net->H;
  gm.W = net->W;
  gm.A = net->A;
  gm.pitch = net->W + 1;
  gm.block = (net->H + 1) * gm.pitch;
  // as many boards as the group's rows hold, capped by the 32-board limit and the FC scratch (only 2 x 2 boards reach the
  // caps: the rows past the last board are padding)
  gm.boards_per_group = std::min(std::min(kGroupRows / gm.block, 32), kFcFloats / (20 + gm.A));
  if (gm.boards_per_group < 1 || gm.pitch + 1 > kHalo)
    return caro_fail(CARO_E_ARG, "board does not fit the wide tensor-core tile geometry");
  const int lim = net->grid_limit > 0 ? net->grid_limit : net->pipeline_limit;
  const int sm_count = lim > 0 && lim < net->sm_count ? lim : net->sm_count;
  const long long max_groups = (max_count + gm.boards_per_group - 1) / gm.boards_per_group;
  const unsigned grid = (unsigned)(max_groups < sm_count ? max_groups : sm_count);
  const int HW = net->H * net->W;
  // exported head features: one of kHeadfeatSlots slots, round robin per launch (parts of the self-play pipeline can be in
  // flight on different streams, and the slot is baked into a captured graph node)
  uint8_t* headfeat = nullptr;
  const int kc64 = caro_net_heads_kc64(net);
  const size_t image = (size_t)net->headfeat_leaves * kc64 * 64 * 2;
  if (net->d_headfeat != nullptr && max_count <= net->headfeat_leaves)
    headfeat = (uint8_t*)net->d_headfeat + (size_t)(net->headfeat_seq++ % kHeadfeatSlots) * 2 * image;
  const size_t img_bytes = (size_t)kLayerBytesIn + (size_t)net->layout.blocks * kLayerBytes;
  const uint8_t* wimg = (const uint8_t*)net->d_wide_weights + (OPS == kOpsF16 ? 0 : img_bytes);  // bf16 (hi), then lo
  net_wide_kernel<R, OPS><<<grid, kThreads, WideCfg<OPS>::kTotal, st>>>(
      rules, gm, (const typename R::Board*)boards, who, d_count, (long long)max_count, wimg, img_bytes, net->d_tc_bias, net->d_blob,
      net->layout, net->d_pol_fc_t, net->d_pol_fc_t + (size_t)2 * HW * net->A, probs, values, headfeat, image, kc64 * 8,
      (long long*)net->d_trace);
  int rc = caro_check_launch("net_wide_kernel");
  if (rc == CARO_OK && headfeat != nullptr) rc = caro_net_heads_forward(net, headfeat, image, d_count, max_count, probs, values, st);
  return rc;
}

}  // namespace wide
}  // namespace caro

using namespace caro;
using namespace caro::wide;

// Weight images: fp16, bf16 (= the hi image of the split mode), then the split mode's lo image bf16(w - bf16(w)); each is
// conv_in (9 taps of kTapBytesIn) followed by 9 taps of kTapBytes per residual block, every tap in the UMMA B-operand
// layout [8-channel chunk of ci][co = 0..127][ci % 8] (no-swizzle K-major).
// Also the conv biases [1 + blocks][128], the transposed FC weights of the in-kernel heads and, for boards with
// HW > 64, the head-feature slots + B image of heads_tc_kernel -- the same buffers the 64-wide towers use.
int caro_net_wide_pack(caro_net* net, const float* h) {
  const BlobLayout& L = net->layout;
  const int blocks = L.blocks;
  const size_t img_bytes = (size_t)kLayerBytesIn + (size_t)blocks * kLayerBytes;
  std::vector<uint16_t> img(3 * img_bytes / 2, 0);  // three images of img_bytes / 2 halves each
  auto put = [&](size_t tap_base, int co, int ci, float w) {
    const size_t off = (tap_base + (size_t)((ci / 8) * F + co) * 16) / 2 + (ci % 8);
    const __half_raw hr = __float2half_rn(w);
    const __nv_bfloat16 hi = __float2bfloat16_rn(w);
    const __nv_bfloat16_raw br = hi;
    const __nv_bfloat16_raw lr = __float2bfloat16_rn(w - __bfloat162float(hi));
    img[off] = hr.x;
    img[img_bytes / 2 + off] = br.x;
    img[img_bytes + off] = lr.x;
  };
  for (int tap = 0; tap < 9; ++tap)
    for (int co = 0; co < F; ++co)
      for (int ci = 0; ci < 2; ++ci) put((size_t)tap * kTapBytesIn, co, ci, h[L.conv_in_w + ((size_t)(co * 2 + ci) * 9 + tap)]);
  for (int l = 0; l < blocks; ++l)
    for (int tap = 0; tap < 9; ++tap) {
      const size_t base = (size_t)kLayerBytesIn + (size_t)l * kLayerBytes + (size_t)tap * kTapBytes;
      for (int co = 0; co < F; ++co)
        for (int ci = 0; ci < F; ++ci) put(base, co, ci, h[L.conv_w[l] + ((size_t)(co * F + ci) * 9 + tap)]);
    }
  std::vector<float> bias((size_t)(1 + blocks) * F);
  for (int co = 0; co < F; ++co) bias[co] = h[L.conv_in_b + co];
  for (int l = 0; l < blocks; ++l)
    for (int co = 0; co < F; ++co) bias[(size_t)(l + 1) * F + co] = h[L.conv_b[l] + co];
  const int HW = net->H * net->W, A = net->A;
  std::vector<float> polt((size_t)2 * HW * A + (size_t)HW * 20);
  for (int a = 0; a < A; ++a)
    for (int i = 0; i < 2 * HW; ++i) polt[(size_t)i * A + a] = h[L.pol_fc_w + (size_t)a * 2 * HW + i];
  for (int i = 0; i < 20; ++i)
    for (int c = 0; c < HW; ++c) polt[(size_t)2 * HW * A + (size_t)c * 20 + i] = h[L.val_fc1_w + (size_t)i * HW + c];
  cudaError_t ce = cudaSuccess;
  if (HW > kHeadsInTowerMaxHW && caro_net_heads_supported(net)) {
    if (!net->d_headfeat) {
      net->headfeat_leaves = 32768;  // per slot; larger launches run the FC heads inside the tower
      const size_t image = (size_t)net->headfeat_leaves * caro_net_heads_kc64(net) * 64 * 2;
      ce = cudaMalloc(&net->d_headfeat, (size_t)kHeadfeatSlots * 2 * image);
      if (ce != cudaSuccess) return caro_fail(CARO_E_CUDA, cudaGetErrorString(ce));
    }
    const int hrc = caro_net_heads_pack(net, h);
    if (hrc != CARO_OK) return hrc;
  }
  if (!net->d_wide_weights) ce = cudaMalloc(&net->d_wide_weights, 3 * img_bytes);
  if (ce == cudaSuccess && !net->d_tc_bias) ce = cudaMalloc(&net->d_tc_bias, bias.size() * sizeof(float));
  if (ce == cudaSuccess && !net->d_pol_fc_t) ce = cudaMalloc(&net->d_pol_fc_t, polt.size() * sizeof(float));
  if (ce == cudaSuccess) ce = cudaMemcpy(net->d_wide_weights, img.data(), 3 * img_bytes, cudaMemcpyHostToDevice);
  if (ce == cudaSuccess) ce = cudaMemcpy(net->d_tc_bias, bias.data(), bias.size() * sizeof(float), cudaMemcpyHostToDevice);
  if (ce == cudaSuccess) ce = cudaMemcpy(net->d_pol_fc_t, polt.data(), polt.size() * sizeof(float), cudaMemcpyHostToDevice);
  if (ce != cudaSuccess) return caro_fail(CARO_E_CUDA, cudaGetErrorString(ce));
  return CARO_OK;
}

// d_tc_bias, d_pol_fc_t and d_headfeat are released by caro_net_tc_free.
void caro_net_wide_free(caro_net* net) {
  if (net->d_wide_weights) cudaFree(net->d_wide_weights);
  net->d_wide_weights = nullptr;
}

// Sets the dynamic shared memory attribute of every instantiation up front (caro_net_create), so that no attribute call
// can fall inside a CUDA-graph capture of the search loop.
template <class R>
static cudaError_t prepare_ops() {
  cudaError_t ce = cudaFuncSetAttribute(net_wide_kernel<R, kOpsF16>, cudaFuncAttributeMaxDynamicSharedMemorySize, WideCfg<kOpsF16>::kTotal);
  if (ce == cudaSuccess) ce = cudaFuncSetAttribute(net_wide_kernel<R, kOpsBf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, WideCfg<kOpsBf16>::kTotal);
  if (ce == cudaSuccess) ce = cudaFuncSetAttribute(net_wide_kernel<R, kOpsBf16x3>, cudaFuncAttributeMaxDynamicSharedMemorySize, WideCfg<kOpsBf16x3>::kTotal);
  return ce;
}

int caro_net_wide_prepare() {
  cudaError_t ce = prepare_ops<C4Rules>();
  if (ce == cudaSuccess) ce = prepare_ops<MnkRules>();
  if (ce != cudaSuccess) return caro_fail(CARO_E_CUDA, cudaGetErrorString(ce));
  return CARO_OK;
}

template <class R>
static int forward_ops(const R& rules, caro_net* net, const void* d_boards, const uint8_t* d_who, const int32_t* d_count, int64_t max_count,
                       float* d_probs, float* d_values, int ops, cudaStream_t st) {
  if (ops == kOpsF16) return launch_wide<R, kOpsF16>(rules, net, d_boards, d_who, d_count, max_count, d_probs, d_values, st);
  if (ops == kOpsBf16x3) return launch_wide<R, kOpsBf16x3>(rules, net, d_boards, d_who, d_count, max_count, d_probs, d_values, st);
  return launch_wide<R, kOpsBf16>(rules, net, d_boards, d_who, d_count, max_count, d_probs, d_values, st);
}

int caro_net_wide_forward(caro_net* net, int game, int n, int k, const void* d_boards, const uint8_t* d_who,
                          const int32_t* d_count, int64_t max_count, float* d_probs, float* d_values, int ops, cudaStream_t st) {
  if (game == CARO_GAME_CONNECT4) return forward_ops(C4Rules(), net, d_boards, d_who, d_count, max_count, d_probs, d_values, ops, st);
  return forward_ops(MnkRules{n, k}, net, d_boards, d_who, d_count, max_count, d_probs, d_values, ops, st);
}
