// Internal definition of the network handle shared by net.cu (handle, SIMT tower) and
// net_tc.cu (tcgen05 tower).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace caro {

constexpr int kFilters = 64;      // lib/model.py:7
constexpr int kWideFilters = 128; // the only other width: net_wide.cu's tower and the SIMT tower's wide instance
constexpr int kBlocks = 5;        // conv_1 .. conv_5: the reference's depth (lib/model.py:21-45)
constexpr int kMaxBlocks = 20;    // deepest tower the kernels accept ("deep residual net" of BASELINE configs[3]): the number of
                                  // residual blocks is a run-time property of the weight blob
constexpr float kLeaky = 0.01f;   // nn.LeakyReLU default slope

// Offsets (in floats) of the folded-weight blob described in include/caro_b200.h
struct BlobLayout {
  size_t conv_in_w, conv_in_b;
  size_t conv_w[kMaxBlocks], conv_b[kMaxBlocks];
  int blocks;
  int filters;  // kFilters or kWideFilters
  size_t val_conv_w, val_conv_b, val_fc1_w, val_fc1_b, val_fc2_w, val_fc2_b;
  size_t pol_conv_w, pol_conv_b, pol_fc_w, pol_fc_b;
  size_t total;
};

inline BlobLayout blob_layout(int H, int W, int A, int blocks = kBlocks, int filters = kFilters) {
  BlobLayout L;
  L.blocks = blocks;
  L.filters = filters;
  const size_t F = (size_t)filters;
  for (int i = 0; i < kMaxBlocks; ++i) L.conv_w[i] = L.conv_b[i] = 0;
  size_t o = 0;
  const size_t hw = (size_t)H * W;
  auto take = [&](size_t n) { size_t r = o; o += n; return r; };
  L.conv_in_w = take(F * 2 * 9);
  L.conv_in_b = take(F);
  for (int i = 0; i < blocks; ++i) {
    L.conv_w[i] = take(F * F * 9);
    L.conv_b[i] = take(F);
  }
  L.val_conv_w = take(F);
  L.val_conv_b = take(1);
  L.val_fc1_w = take(20 * hw);
  L.val_fc1_b = take(20);
  L.val_fc2_w = take(20);
  L.val_fc2_b = take(1);
  L.pol_conv_w = take(2 * F);
  L.pol_conv_b = take(2);
  L.pol_fc_w = take((size_t)A * 2 * hw);
  L.pol_fc_b = take(A);
  L.total = o;
  return L;
}

}  // namespace caro

struct caro_net {
  int H, W, A;
  caro::BlobLayout layout;
  float* d_blob;        // fp32 folded weights (SIMT tower + heads of both towers)
  void* d_tc_weights;   // bf16 UMMA B-operand images, one per (layer, tap) -- see net_tc.cu
  void* d_rt_weights;   // bf16 UMMA B-operand blocks of the row-tiled tower -- see net_rt.cu
  void* d_tc_pair_weights;  // tap-per-MMA tower as CTA pairs: one compact bf16 image per cluster rank
  void* d_rt_f16_weights;   // the row-tiled tower's blocks in fp16 (F16 mode)
  void* d_rt_pair_weights;  // the same for the CTA-pair form: one image per cluster rank, 7 KB blocks
  void* d_rt_scratch;       // CTA-pair form: head features + FC scratch of every CTA, kRtScratchSlots launches in flight
  unsigned rt_scratch_seq;  // next slot (round robin per launch)
  void* d_rx_weights;   // fp16 hi / lo UMMA B-operand blocks of the split-precision row-tiled tower -- see net_rx.cu
  void* d_wide_weights; // 128-wide handles: fp16, bf16 (hi) and bf16 lo UMMA B-operand images of every (layer, tap) -- see net_wide.cu
  alignas(16) float h_rt_consts[(caro::kMaxBlocks + 1) * 64 + 3 * 64 + 4 + 1536 + 4];  // host copy of the row-tiled tower's by-value constants (RtConsts)
  float* d_tc_bias;     // [1 + blocks][filters] folded conv biases
  float* d_pol_fc_t;    // policy FC transposed to [2*HW][A] (+ value FC1 [HW][20]) for coalesced reads in the TC epilogue
  void* d_headfeat;     // large boards: exported activated head features, bf16 hi + lo images in the A-operand layout of net_heads.cu
  void* d_heads_b;      // large boards: bf16 hi + lo B-operand image of the FC heads GEMM (net_heads.cu)
  long long headfeat_leaves;  // capacity of ONE slot of d_headfeat in leaves
  unsigned headfeat_seq;      // next slot (round robin per launch)
  void* d_trace;        // optional debug timeline buffer (caro_net_set_trace), normally null
  int sm_count;         // multiprocessors of the device the handle was created on
  int grid_limit;       // > 0: CTAs (= SMs) the persistent tower may occupy (caro_net_set_grid_limit), 0 = all
  unsigned long long serial;   // unique per created handle (keys the cached ply graph of the parts pipeline)
  unsigned long long version;  // bumped by every caro_net_update: the tower's constants travel BY VALUE in its kernel parameters
  int pipeline_limit;   // > 0 while the parts pipeline issues / captures a ply and the user has set no limit: sm_count - sm_count / 9
};

// engine.cu: drop cached ply graphs that refer to an engine / a network (0 = none)
void caro_pipeline_forget(unsigned long long engine_serial, unsigned long long net_serial);

// net_tc.cu
int caro_net_tc_pack(caro_net* net, const float* h_blob);
int caro_net_tc_prepare();
void caro_net_tc_free(caro_net* net);
int caro_net_tc_forward(caro_net* net, int game, int n, int k, const void* d_boards, const uint8_t* d_who,
                        const int32_t* d_count, int64_t max_count, float* d_probs, float* d_values, int exact, cudaStream_t st);

// net_rt.cu (row-tiled tower for boards up to 6 x 7)
int caro_net_rt_pack(caro_net* net, const float* h_blob);
int caro_net_rt_prepare();
void caro_net_rt_free(caro_net* net);
bool caro_net_rt_supports(const caro_net* net);
int caro_net_rt_forward(caro_net* net, int game, int n, int k, const void* d_boards, const uint8_t* d_who,
                        const int32_t* d_count, int64_t max_count, float* d_probs, float* d_values, int mode, cudaStream_t st);

// net_wide.cu (tap-per-MMA tower of 128-filter networks, N = 128 per MMA, weights streamed tap by tap)
// ops: 0 = fp16 operands, 1 = bf16 operands, 2 = bf16 hi + lo operands (3 MMAs per product)
int caro_net_wide_pack(caro_net* net, const float* h_blob);
int caro_net_wide_prepare();
void caro_net_wide_free(caro_net* net);
int caro_net_wide_forward(caro_net* net, int game, int n, int k, const void* d_boards, const uint8_t* d_who,
                          const int32_t* d_count, int64_t max_count, float* d_probs, float* d_values, int ops, cudaStream_t st);

// net_rx.cu (split-precision row-tiled tower, fp16 hi + lo, boards up to 6 x 7)
int caro_net_rx_pack(caro_net* net, const float* h_blob);
int caro_net_rx_prepare();
void caro_net_rx_free(caro_net* net);
int caro_net_rx_forward(caro_net* net, int game, int n, int k, const void* d_boards, const uint8_t* d_who,
                        const int32_t* d_count, int64_t max_count, float* d_probs, float* d_values, cudaStream_t st);

// net_heads.cu (FC heads of large boards as one split-precision tcgen05 GEMM per 128 leaves)
int caro_net_heads_kc64(const caro_net* net);
bool caro_net_heads_supported(const caro_net* net);
int caro_net_heads_pack(caro_net* net, const float* h_blob);
int caro_net_heads_prepare();
void caro_net_heads_free(caro_net* net);
int caro_net_heads_forward(caro_net* net, const void* a_img, size_t a_lo_off, const int32_t* d_count, int64_t max_count,
                           float* d_probs, float* d_values, cudaStream_t st);
