// Network handle + the fp32 SIMT tower (numerics reference kernel; the product path is net_tc.cu).
//
// lib/model.py:82-94 with eval-mode BatchNorm folded into the convolutions on the host:
//   v = lrelu(conv_in(x)); 5 x { v = v + lrelu(conv_i(v)) };
//   value = tanh(fc2(lrelu(fc1(lrelu(conv_val(v))))));  policy = softmax(fc(lrelu(conv_policy(v))))
#include <cuda_runtime.h>
#include <math.h>

#include <atomic>

#include "../../include/caro_b200.h"
#include "common_host.h"
#include "net.h"
#include "rules.cuh"

namespace caro {

__device__ __forceinline__ float lrelu(float x) { return x > 0.0f ? x : kLeaky * x; }

// One block per leaf, F filters.  Dynamic smem: 2 x [F][HW] activations + head scratch.  For F = 128 the two activation
// buffers alone take 230,400 B at 15 x 15, so the head scratch reuses the buffer the last layer read from: everything
// stays in the block's own shared memory, and launches that overlap on other streams share nothing.
template <class R, int F>
__global__ void __launch_bounds__(256)
net_simt_kernel(R rules, const typename R::Board* __restrict__ boards, const uint8_t* __restrict__ who,
                const int32_t* __restrict__ d_count, long long max_count, const float* __restrict__ blob, BlobLayout L,
                int A, float* __restrict__ probs, float* __restrict__ values) {
  extern __shared__ float sm[];
  const int H = rules.rows(), W = rules.cols(), HW = H * W;
  const long long count = d_count ? min((long long)*d_count, max_count) : max_count;
  float* buf0 = sm;
  float* buf1 = sm + F * HW;
  for (long long leaf = blockIdx.x; leaf < count; leaf += gridDim.x) {
    const typename R::Board s = boards[leaf];
    const int wm = who[leaf];
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * HW; i += blockDim.x)
      buf1[i] = (float)rules.plane_value(s, wm, i / HW, (i % HW) / W, i % W);
    __syncthreads();
    // conv_in: 2 -> F
    for (int o = threadIdx.x; o < F * HW; o += blockDim.x) {
      const int co = o / HW, pos = o % HW, r = pos / W, c = pos % W;
      float acc = blob[L.conv_in_b + co];
      for (int ci = 0; ci < 2; ++ci)
        for (int ky = 0; ky < 3; ++ky) {
          const int rr = r + ky - 1;
          if (rr < 0 || rr >= H) continue;
          for (int kx = 0; kx < 3; ++kx) {
            const int cc = c + kx - 1;
            if (cc < 0 || cc >= W) continue;
            acc += blob[L.conv_in_w + ((co * 2 + ci) * 3 + ky) * 3 + kx] * buf1[ci * HW + rr * W + cc];
          }
        }
      buf0[o] = lrelu(acc);
    }
    __syncthreads();
    float* cur = buf0;
    float* nxt = buf1;
    for (int layer = 0; layer < L.blocks; ++layer) {
      const float* wgt = blob + L.conv_w[layer];
      const float* bias = blob + L.conv_b[layer];
      for (int o = threadIdx.x; o < F * HW; o += blockDim.x) {
        const int co = o / HW, pos = o % HW, r = pos / W, c = pos % W;
        float acc = bias[co];
        for (int ci = 0; ci < F; ++ci) {
          const float* wk = wgt + (size_t)(co * F + ci) * 9;
          const float* in = cur + ci * HW;
          for (int ky = 0; ky < 3; ++ky) {
            const int rr = r + ky - 1;
            if (rr < 0 || rr >= H) continue;
            for (int kx = 0; kx < 3; ++kx) {
              const int cc = c + kx - 1;
              if (cc < 0 || cc >= W) continue;
              acc += wk[ky * 3 + kx] * in[rr * W + cc];
            }
          }
        }
        nxt[o] = cur[o] + lrelu(acc);
      }
      __syncthreads();
      float* t = cur;
      cur = nxt;
      nxt = t;
    }
    float* head = F == kFilters ? buf1 + F * HW : nxt;  // [3*HW + 32 + A]
    // heads: 1x1 convs (value: 1 channel, policy: 2 channels)
    for (int i = threadIdx.x; i < 3 * HW; i += blockDim.x) {
      const int ch = i / HW, pos = i % HW;
      const float* wv = ch == 0 ? blob + L.val_conv_w : blob + L.pol_conv_w + (ch - 1) * F;
      float acc = ch == 0 ? blob[L.val_conv_b] : blob[L.pol_conv_b + ch - 1];
      for (int ci = 0; ci < F; ++ci) acc += wv[ci] * cur[ci * HW + pos];
      head[i] = lrelu(acc);  // [0,HW) value plane, [HW,3HW) policy planes (channel-major, lib/model.py:93)
    }
    __syncthreads();
    float* hid = head + 3 * HW;       // [20]
    float* logit = hid + 32;          // [A]
    for (int i = threadIdx.x; i < 20 + A; i += blockDim.x) {
      if (i < 20) {
        float acc = blob[L.val_fc1_b + i];
        for (int p = 0; p < HW; ++p) acc += blob[L.val_fc1_w + (size_t)i * HW + p] * head[p];
        hid[i] = lrelu(acc);
      } else {
        const int a = i - 20;
        float acc = blob[L.pol_fc_b + a];
        for (int p = 0; p < 2 * HW; ++p) acc += blob[L.pol_fc_w + (size_t)a * 2 * HW + p] * head[HW + p];
        logit[a] = acc;
      }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      float acc = blob[L.val_fc2_b];
      for (int i = 0; i < 20; ++i) acc += blob[L.val_fc2_w + i] * hid[i];
      values[leaf] = tanhf(acc);
    }
    if (threadIdx.x < 32) {  // softmax over all A actions (lib/mcts.py:216), one warp
      float mx = -INFINITY;
      for (int a = threadIdx.x; a < A; a += 32) mx = fmaxf(mx, logit[a]);
      for (int off = 16; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
      float sum = 0.0f;
      for (int a = threadIdx.x; a < A; a += 32) sum += expf(logit[a] - mx);
      for (int off = 16; off > 0; off >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
      for (int a = threadIdx.x; a < A; a += 32) probs[leaf * A + a] = expf(logit[a] - mx) / sum;
    }
  }
}

template <class R>
int launch_simt(const R& rules, const caro_net* net, const void* boards, const uint8_t* who, const int32_t* d_count,
                int64_t max_count, float* probs, float* values, cudaStream_t st) {
  const int HW = net->H * net->W;
  const unsigned grid = (unsigned)(max_count < 148 * 8 ? (max_count > 0 ? max_count : 1) : 148 * 8);
  if (net->layout.filters == kWideFilters) {  // the head scratch lives in the spare activation buffer
    const size_t smem = sizeof(float) * ((size_t)2 * kWideFilters * HW + 8);
    auto kern = net_simt_kernel<R, kWideFilters>;
    cudaError_t ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (ce != cudaSuccess) return caro_fail(CARO_E_CUDA, cudaGetErrorString(ce));
    kern<<<grid, 256, smem, st>>>(rules, (const typename R::Board*)boards, who, d_count, (long long)max_count, net->d_blob,
                                  net->layout, net->A, probs, values);
    return caro_check_launch("net_simt_kernel");
  }
  const size_t smem = sizeof(float) * ((size_t)2 * kFilters * HW + 3 * HW + 32 + net->A + 8);
  auto kern = net_simt_kernel<R, kFilters>;
  cudaError_t ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (ce != cudaSuccess) return caro_fail(CARO_E_CUDA, cudaGetErrorString(ce));
  kern<<<grid, 256, smem, st>>>(rules, (const typename R::Board*)boards, who, d_count, (long long)max_count, net->d_blob,
                                net->layout, net->A, probs, values);
  return caro_check_launch("net_simt_kernel");
}

}  // namespace caro

using namespace caro;

extern "C" {

size_t caro_net_blob_floats(int rows, int cols, int actions) { return blob_layout(rows, cols, actions).total; }

size_t caro_net_blob_floats_deep(int rows, int cols, int actions, int blocks) {
  if (blocks < 1 || blocks > kMaxBlocks) return 0;
  return blob_layout(rows, cols, actions, blocks).total;
}

size_t caro_net_blob_floats_shape(int rows, int cols, int actions, int blocks, int filters) {
  if (blocks < 1 || blocks > kMaxBlocks || (filters != kFilters && filters != kWideFilters)) return 0;
  return blob_layout(rows, cols, actions, blocks, filters).total;
}

int caro_net_update(caro_net* net, const float* h_blob, size_t n_floats) {
  if (!net || !h_blob) return caro_fail(CARO_E_ARG, "null argument");
  if (n_floats != net->layout.total) return caro_fail(CARO_E_ARG, "weight blob has the wrong size");
  caro_pipeline_forget(0, net->serial);  // a captured ply holds the previous constants by value
  net->version += 1;
  // the weight images are rewritten in place: searches that are still running on the pipeline's non-blocking streams must
  // have finished with the old ones (an update is rare: NetWrapper.sync after a promotion)
  if (cudaDeviceSynchronize() != cudaSuccess) return caro_fail(CARO_E_CUDA, "device error before the weight update");
  cudaError_t ce = cudaMemcpy(net->d_blob, h_blob, n_floats * sizeof(float), cudaMemcpyHostToDevice);
  if (ce != cudaSuccess) return caro_fail(CARO_E_CUDA, cudaGetErrorString(ce));
  if (net->layout.filters == kWideFilters) return caro_net_wide_pack(net, h_blob);
  const int rc = caro_net_tc_pack(net, h_blob);
  if (rc != CARO_OK) return rc;
  if (!caro_net_rt_supports(net)) return CARO_OK;
  const int rc2 = caro_net_rt_pack(net, h_blob);
  return rc2 != CARO_OK ? rc2 : caro_net_rx_pack(net, h_blob);
}

// Allocates and fills a handle once the caller has validated the shape and found a device.
static int net_create(int rows, int cols, int actions, const BlobLayout& layout, const float* h_blob, size_t n_floats, caro_net** out) {
  static std::atomic<unsigned long long> next_serial{0};
  caro_net* net = new caro_net();
  net->serial = ++next_serial;
  net->version = 0;
  net->H = rows;
  net->W = cols;
  net->A = actions;
  net->layout = layout;
  net->d_blob = nullptr;
  net->d_tc_weights = nullptr;
  net->d_rt_weights = nullptr;
  net->d_rt_pair_weights = nullptr;
  net->d_rt_f16_weights = nullptr;
  net->d_tc_pair_weights = nullptr;
  net->d_rt_scratch = nullptr;
  net->rt_scratch_seq = 0;
  net->d_rx_weights = nullptr;
  net->d_wide_weights = nullptr;
  net->d_tc_bias = nullptr;
  net->d_pol_fc_t = nullptr;
  net->d_trace = nullptr;
  net->d_headfeat = nullptr;
  net->d_heads_b = nullptr;
  net->headfeat_leaves = 0;
  net->headfeat_seq = 0;
  net->grid_limit = 0;
  net->pipeline_limit = 0;
  {
    int dev = 0;
    cudaGetDevice(&dev);
    net->sm_count = 148;
    cudaDeviceGetAttribute(&net->sm_count, cudaDevAttrMultiProcessorCount, dev);
    int prc = caro_net_tc_prepare();
    if (prc == CARO_OK) prc = caro_net_rt_prepare();
    if (prc == CARO_OK) prc = caro_net_rx_prepare();
    if (prc == CARO_OK) prc = caro_net_heads_prepare();
    if (prc == CARO_OK) prc = caro_net_wide_prepare();
    if (prc != CARO_OK) {
      delete net;
      return prc;
    }
  }
  if (n_floats != net->layout.total) {
    delete net;
    return caro_fail(CARO_E_ARG, "weight blob has the wrong size");
  }
  cudaError_t ce = cudaMalloc(&net->d_blob, n_floats * sizeof(float));
  if (ce != cudaSuccess) {
    caro_net_destroy(net);
    return caro_fail(CARO_E_CUDA, cudaGetErrorString(ce));
  }
  const int rc = caro_net_update(net, h_blob, n_floats);
  if (rc != CARO_OK) {
    caro_net_destroy(net);
    return rc;
  }
  *out = net;
  return CARO_OK;
}

static bool bad_net_shape(int rows, int cols, int actions) {
  return rows < 2 || cols < 2 || rows > 15 || cols > 15 || actions < 1 || actions > 255;
}

int caro_net_create(int rows, int cols, int actions, const float* h_blob, size_t n_floats, caro_net** out) {
  if (!out || !h_blob) return caro_fail(CARO_E_ARG, "null argument");
  if (bad_net_shape(rows, cols, actions)) return caro_fail(CARO_E_ARG, "bad net shape");
  if (caro_device_count() <= 0) return caro_fail(CARO_E_CUDA, "no CUDA device: the network has no CPU fallback");
  // the depth of the tower is read off the blob's length: base + blocks x (64 x 64 x 9 + 64) floats
  const size_t per_block = (size_t)kFilters * kFilters * 9 + kFilters;
  const size_t base = blob_layout(rows, cols, actions, 1).total - per_block;
  const size_t blocks = n_floats > base ? (n_floats - base) / per_block : 0;
  if (blocks < 1 || blocks > (size_t)kMaxBlocks || base + blocks * per_block != n_floats)
    return caro_fail(CARO_E_ARG, "weight blob has the wrong size");
  return net_create(rows, cols, actions, blob_layout(rows, cols, actions, (int)blocks), h_blob, n_floats, out);
}

int caro_net_create_shape(int rows, int cols, int actions, int blocks, int filters, const float* h_blob, size_t n_floats,
                          caro_net** out) {
  if (!out || !h_blob) return caro_fail(CARO_E_ARG, "null argument");
  if (bad_net_shape(rows, cols, actions)) return caro_fail(CARO_E_ARG, "bad net shape");
  if (blocks < 1 || blocks > kMaxBlocks) return caro_fail(CARO_E_ARG, "bad tower depth: 1 .. 20 residual blocks are supported");
  if (filters != kFilters && filters != kWideFilters) return caro_fail(CARO_E_ARG, "bad tower width: 64 or 128 filters are supported");
  const BlobLayout layout = blob_layout(rows, cols, actions, blocks, filters);
  if (n_floats != layout.total) return caro_fail(CARO_E_ARG, "weight blob has the wrong size for the stated shape");
  if (caro_device_count() <= 0) return caro_fail(CARO_E_CUDA, "no CUDA device: the network has no CPU fallback");
  return net_create(rows, cols, actions, layout, h_blob, n_floats, out);
}

int caro_net_set_grid_limit(caro_net* net, int ctas) {
  if (!net || ctas < 0) return caro_fail(CARO_E_ARG, "bad grid limit");
  net->grid_limit = ctas;
  return CARO_OK;
}

int caro_net_set_trace(caro_net* net, void* d_trace) {
  if (!net) return caro_fail(CARO_E_ARG, "null net");
  net->d_trace = d_trace;
  return CARO_OK;
}

void caro_net_destroy(caro_net* net) {
  if (!net) return;
  caro_pipeline_forget(0, net->serial);
  caro_net_tc_free(net);
  caro_net_rt_free(net);
  caro_net_rx_free(net);
  caro_net_heads_free(net);
  caro_net_wide_free(net);
  if (net->d_blob) cudaFree(net->d_blob);
  delete net;
}

int caro_net_forward(caro_net* net, int game, int n, int k, const void* d_boards, const uint8_t* d_who,
                     const int32_t* d_count, int64_t max_count, float* d_probs, float* d_values, int impl, void* stream) {
  if (!net || !d_boards || !d_who || !d_probs || !d_values) return caro_fail(CARO_E_ARG, "null argument");
  if (max_count <= 0) return CARO_OK;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (game == CARO_GAME_CONNECT4) {
    if (net->H != 6 || net->W != 7 || net->A != 7) return caro_fail(CARO_E_ARG, "net shape does not match Connect4");
  } else if (game == CARO_GAME_MNK || game == CARO_GAME_CARO) {  // the network does not depend on the win rule
    if (net->H != n || net->W != n || net->A != n * n) return caro_fail(CARO_E_ARG, "net shape does not match the m,n,k board");
  } else {
    return caro_fail(CARO_E_ARG, "unknown game");
  }
  if (net->layout.filters == kWideFilters && impl != 1) {
    // 128 filters: impl 7 = the wide tower with fp16 operands, 0 / 3 = the same with bf16 operands, 8 = bf16 hi + lo
    if (impl != 0 && impl != 3 && impl != 7 && impl != 8)
      return caro_fail(CARO_E_ARG, "a 128-filter network runs impl 0, 1, 3, 7 or 8 only (no CTA-pair or row-tiled tower; "
                                   "its split-precision tower is impl 8)");
    return caro_net_wide_forward(net, game, n, k, d_boards, d_who, d_count, max_count, d_probs, d_values,
                                 impl == 7 ? 0 : impl == 8 ? 2 : 1, st);
  }
  if (impl == 8)
    return caro_fail(CARO_E_ARG, "impl 8 is the split-precision tower of 128 filters; a 64-filter network runs impl 2 for split precision");
  if (impl == 1) {
    if (game == CARO_GAME_CONNECT4) return launch_simt<C4Rules>(C4Rules(), net, d_boards, d_who, d_count, max_count, d_probs, d_values, st);
    return launch_simt<MnkRules>(MnkRules{n, k}, net, d_boards, d_who, d_count, max_count, d_probs, d_values, st);
  }
  if ((impl == 0 || impl == 5 || impl == 7) && caro_net_rt_supports(net))
    return caro_net_rt_forward(net, game, n, k, d_boards, d_who, d_count, max_count, d_probs, d_values, impl == 5 ? 1 : impl == 7 ? 2 : 0, st);
  if (impl == 2 && caro_net_rt_supports(net))
    return caro_net_rx_forward(net, game, n, k, d_boards, d_who, d_count, max_count, d_probs, d_values, st);
  if (impl == 0 || impl == 2 || impl == 3 || impl == 4 || impl == 6)
    return caro_net_tc_forward(net, game, n, k, d_boards, d_who, d_count, max_count, d_probs, d_values,
                               (impl == 2 || impl == 4) ? 1 : impl == 6 ? 2 : 0, st);
  return caro_fail(CARO_E_ARG, "unknown net impl");
}

}  // extern "C"
