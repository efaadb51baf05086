// Shared device helpers of the tcgen05 towers (net_tc.cu, net_rt.cu, net_wide.cu): PTX wrappers, descriptors, TMEM
// load/store macros, the debug timeline macro, the head-feature export and the fully connected heads.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "net.h"

namespace caro {

struct TcGeom {
  int H, W, A, pitch, block, boards_per_group;
};

// ---------------------------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must surface as a launch error, never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) __trap();
  }
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// Wait for something that is far away (the head warps for the end of a pass, the weight producer for a region):
// sleep between the polls instead of spinning -- under sustained load the tower runs into the 1,000 W power cap
// (SM clock 1,965 -> ~1,770 MHz), and a fifth of its instruction stream used to be barrier polling.
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    __nanosleep(200);
    if (clock64() - t0 > 4000000000LL) __trap();
  }
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

#define TMEM_LD16(addr, r)                                                                                              \
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];" \
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),        \
                 "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])   \
               : "r"(addr))
#define TMEM_ST16(addr, r)                                                                                              \
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" \
               ::"r"(addr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),     \
               "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])             \
               : "memory")

// Shared-memory matrix descriptor, no-swizzle K-major canonical layout (cute::UMMA::SmemDescriptor):
//   [0,14) start >> 4 | [16,30) LBO >> 4 (stride between the two 8-element K chunks)
//   | [32,46) SBO >> 4 (stride between 8-row groups) | [46,48) version = 1 | [61,64) layout = 0
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((smem_addr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}
// Instruction descriptor (cute::UMMA::InstrDescriptor): D=f32, A=B=bf16, both K-major, N=64, M=128
constexpr uint32_t kIdesc = (1u << 4) | (1u << 7) | (1u << 10) | ((64u >> 3) << 17) | ((128u >> 4) << 24);

__device__ __forceinline__ float lrelu_tc(float x) { return fmaxf(x, kLeaky * x); }

// Optional timeline (debug): CTA 0 stores clock64() into a fixed slot per event (fire-and-forget store,
// no atomics, so the pipeline is not perturbed): slot = kind * 1000 + gl * 4 + t.
#define TC_TRACE(kind, idx)                                                                      \
  do {                                                                                           \
    if (trace != nullptr && blockIdx.x == 0 && (idx) < 1000) trace[(kind) * 1000 + (idx)] = clock64(); \
  } while (0)

// Large boards (Caro 15x15: 225 actions, 450 x 225 policy FC) do not run their FC heads inside the tower: two head warps
// re-reading 405 KB of FC weights for every 2-board group made the heads, not the convolutions, the bottleneck (1.9 ms
// per 4,096 leaves, of which ~0.3 ms tower).  The tower only exports, per leaf, the ACTIVATED outputs of the 1x1 head
// convolutions (bias + LeakyReLU applied here; `head_b` = the three head biases) as bf16 hi + lo pairs, already in the UMMA A-operand layout of the heads
// GEMM (net_heads.cu): images [tile of 128 leaves][K / 8][128 rows][8], K = 3 HW padded to 64, one 16-byte store per
// (leaf, 8 features) and image; heads_tc_kernel then evaluates both FC layers on the tensor cores.
template <int TEAM, int BAR>
__device__ __noinline__ void export_heads(const TcGeom& gm, int nvalid, long long leaf0, int ttid, float* headf_s, const float* head_b,
                                          uint8_t* __restrict__ out_hi, size_t lo_off, int kc8) {
  const int HW = gm.H * gm.W, K = 3 * HW;
  const float hb0 = head_b[0], hb1 = head_b[1], hb2 = head_b[2];
#pragma unroll 1
  for (int item = ttid; item < nvalid * kc8; item += TEAM) {
    const int b = item / kc8, c8 = item - b * kc8;
    const long long leaf = leaf0 + b;
    const float* f = headf_s + (size_t)b * K;
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float v[2];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int k = c8 * 8 + 2 * e + u;
        v[u] = k < K ? lrelu_tc(f[k] + (k < HW ? hb0 : (k < 2 * HW ? hb1 : hb2))) : 0.0f;
      }
      const __nv_bfloat162 h2 = __floats2bfloat162_rn(v[0], v[1]);
      const __nv_bfloat162 l2 = __floats2bfloat162_rn(v[0] - __low2float(h2), v[1] - __high2float(h2));
      hi[e] = *reinterpret_cast<const uint32_t*>(&h2);
      lo[e] = *reinterpret_cast<const uint32_t*>(&l2);
    }
    uint8_t* dst = out_hi + (((size_t)(leaf >> 7) * kc8 + c8) * 128 + (size_t)(leaf & 127)) * 16;
    *reinterpret_cast<uint4*>(dst) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(dst + lo_off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
  asm volatile("bar.sync %0, %1;" ::"n"(BAR), "n"(TEAM) : "memory");
#pragma unroll 1
  for (int i = ttid; i < nvalid * K; i += TEAM) headf_s[i] = 0.0f;  // re-arm the accumulation slots
  asm volatile("bar.sync %0, %1;" ::"n"(BAR), "n"(TEAM) : "memory");
}

// Fully connected heads of one group: value FC1 (HW -> 20) + FC2 + tanh, policy FC (2 HW -> A) + softmax over all
// A actions (lib/model.py:56-72,90-93, lib/mcts.py:216), for all (board, output) pairs in parallel with coalesced
// transposed weights; bias + LeakyReLU of the 1x1 head convolutions are applied on the fly.  Executed by a "team"
// of TEAM threads (the two head warps, or -- for a CTA's last group -- the eight epilogue warps, which have
// nothing else left to do), synchronised with the named barrier BAR.
// NF > 1: the head features arrive as NF partial arrays (stride fstride floats) that are summed here in a fixed
// order, so that the result does not depend on the order in which the epilogue warps finished.
template <int TEAM, int BAR, int NF = 1>
__device__ __noinline__ void run_heads(const TcGeom& gm, int nb, int nvalid, long long leaf0, int ttid, float* headf_s,
                                          float* fc_s, const float* head_b, const float* __restrict__ blob, const BlobLayout& L,
                                          const float* __restrict__ pol_fc_t, const float* __restrict__ val_fc1_t,
                                          float* __restrict__ probs, float* __restrict__ values, int fstride = 0) {
  const int HW = gm.H * gm.W;
  if (NF > 1) {  // fold the partial arrays into the first one (fixed order), then proceed as usual
#pragma unroll 1
    for (int i = ttid; i < nvalid * 3 * HW; i += TEAM) {
      float v = headf_s[i];
#pragma unroll
      for (int k = 1; k < NF; ++k) {
        v += headf_s[i + k * fstride];
        headf_s[i + k * fstride] = 0.0f;  // re-arm
      }
      headf_s[i] = v;
    }
    asm volatile("bar.sync %0, %1;" ::"n"(BAR), "n"(TEAM) : "memory");
  }
  const float* featc = headf_s;
  const int per_board = 20 + gm.A;
  float* hid = fc_s;  // [nb][20] value hidden units, logits behind them
  float* logit = fc_s + nb * 20;
  const float hb0 = head_b[0], hb1 = head_b[1], hb2 = head_b[2];
#pragma unroll 1
  for (int o = ttid; o < nvalid * per_board; o += TEAM) {
    const int b = o / per_board, i = o - b * per_board;
    const float* feat = featc + (size_t)b * 3 * HW;
    float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
    if (i < 20) {
      const float* wt = val_fc1_t + i;
      int cell = 0;
      for (; cell + 3 < HW; cell += 4) {
        a0 = fmaf(__ldg(wt + (size_t)cell * 20), lrelu_tc(feat[cell] + hb0), a0);
        a1 = fmaf(__ldg(wt + (size_t)(cell + 1) * 20), lrelu_tc(feat[cell + 1] + hb0), a1);
        a2 = fmaf(__ldg(wt + (size_t)(cell + 2) * 20), lrelu_tc(feat[cell + 2] + hb0), a2);
        a3 = fmaf(__ldg(wt + (size_t)(cell + 3) * 20), lrelu_tc(feat[cell + 3] + hb0), a3);
      }
      for (; cell < HW; ++cell) a0 = fmaf(__ldg(wt + (size_t)cell * 20), lrelu_tc(feat[cell] + hb0), a0);
      hid[b * 20 + i] = lrelu_tc(blob[L.val_fc1_b + i] + (a0 + a1) + (a2 + a3));
    } else {
      const int a = i - 20;
      const float* wt = pol_fc_t + a;
      const float* f2 = feat + HW;
      for (int chn = 0; chn < 2; ++chn) {
        const float hb = chn ? hb2 : hb1;
        const float* w2 = wt + (size_t)chn * HW * gm.A;
        const float* fc = f2 + chn * HW;
        int cell = 0;
        for (; cell + 3 < HW; cell += 4) {
          a0 = fmaf(__ldg(w2 + (size_t)cell * gm.A), lrelu_tc(fc[cell] + hb), a0);
          a1 = fmaf(__ldg(w2 + (size_t)(cell + 1) * gm.A), lrelu_tc(fc[cell + 1] + hb), a1);
          a2 = fmaf(__ldg(w2 + (size_t)(cell + 2) * gm.A), lrelu_tc(fc[cell + 2] + hb), a2);
          a3 = fmaf(__ldg(w2 + (size_t)(cell + 3) * gm.A), lrelu_tc(fc[cell + 3] + hb), a3);
        }
        for (; cell < HW; ++cell) a0 = fmaf(__ldg(w2 + (size_t)cell * gm.A), lrelu_tc(fc[cell] + hb), a0);
      }
      logit[b * gm.A + a] = blob[L.pol_fc_b + a] + (a0 + a1) + (a2 + a3);
    }
  }
  asm volatile("bar.sync %0, %1;" ::"n"(BAR), "n"(TEAM) : "memory");
#pragma unroll 1
  for (int i = ttid; i < nvalid * 3 * HW; i += TEAM) headf_s[i] = 0.0f;  // re-arm the accumulation slots
#pragma unroll 1
  for (int b = ttid >> 5; b < nvalid; b += TEAM / 32) {
    const int lane = ttid & 31;
    if (lane == 0) {
      float acc = blob[L.val_fc2_b];
      for (int i = 0; i < 20; ++i) acc = fmaf(blob[L.val_fc2_w + i], hid[b * 20 + i], acc);
      values[leaf0 + b] = tanhf(acc);
    }
    const float* lrow = logit + b * gm.A;
    float* prow = probs + (size_t)(leaf0 + b) * gm.A;
    float mx = -INFINITY;
#pragma unroll 1
    for (int a = lane; a < gm.A; a += 32) mx = fmaxf(mx, lrow[a]);
    for (int off = 16; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
    float sum = 0.0f;
#pragma unroll 1
    for (int a = lane; a < gm.A; a += 32) sum += expf(lrow[a] - mx);
    for (int off = 16; off > 0; off >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
#pragma unroll 1
    for (int a = lane; a < gm.A; a += 32) prow[a] = expf(lrow[a] - mx) / sum;
  }
  asm volatile("bar.sync %0, %1;" ::"n"(BAR), "n"(TEAM) : "memory");  // hid / logit / slots are reused by the next group
}

}  // namespace caro
