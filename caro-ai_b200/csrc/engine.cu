// Host side of the engine: workspace carving, kernel dispatch per game family, C ABI.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/caro_b200.h"
#include "common_host.h"
#include "engine_kernels.cuh"
#include "net.h"

namespace caro {

struct Region {
  std::string name;
  size_t offset, bytes;
  int elem;
  int64_t dims[4];
};

struct Carver {
  size_t cur = 0;
  std::vector<Region> regions;
  size_t add(const char* name, size_t elem, int64_t d0, int64_t d1 = 0, int64_t d2 = 0, int64_t d3 = 0) {
    size_t count = (size_t)d0 * (size_t)(d1 ? d1 : 1) * (size_t)(d2 ? d2 : 1) * (size_t)(d3 ? d3 : 1);
    cur = (cur + 255) & ~(size_t)255;
    Region r{name, cur, count * elem, (int)elem, {d0, d1, d2, d3}};
    regions.push_back(r);
    cur += count * elem;
    return r.offset;
  }
};

// compact_kernel's dynamic shared memory: an index map of node_cap words + a staging buffer of `chunk` node records
static size_t compact_smem_bytes(const Dims& dm, int chunk) { return ((size_t)((dm.node_cap + 3) & ~3) + (size_t)chunk * dm.RS) * 4; }
static int compact_chunk_nodes(const Dims& dm) {
  const long long budget = 220 * 1024 - (long long)((dm.node_cap + 3) & ~3) * 4;
  long long chunk = budget / ((long long)dm.RS * 4);
  if (chunk > 256) chunk = 256;
  return chunk < 1 ? 0 : (int)chunk;
}

static int round_pow2(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

}  // namespace caro

using namespace caro;

struct caro_engine {
  caro_engine_config cfg;
  Dims dm;
  SearchParams sp;
  int max_plies;
  size_t board_bytes;
  char* ws;
  size_t ws_bytes;
  Carver carve;
  View<C4Board> v_c4;
  View<MnkBoard> v_mnk;
  MnkRules mnk;
  // optional per-phase CUDA-event timing of the search loop (bench / roofline accounting)
  int profiling = 0;  // 0 off, 1 network spans only (cheap: 2 events per minibatch), 2 all four phases
  std::vector<cudaEvent_t> events;
  size_t events_used = 0;
  std::vector<std::pair<size_t, size_t>> spans[5];  // (start, end) event indices per phase (4 = Dirichlet noise kernel)
  size_t open_span[5] = {0, 0, 0, 0, 0};
  unsigned long long launches = 0;
  cudaEvent_t sync_a = nullptr, sync_b = nullptr;  // cross-stream hand-offs (pair pipeline)
  bool lean_tree = false;  // set while the parts pipeline issues launches: prefer tree kernels with few warps
  unsigned long long serial = 0;  // unique per created engine (keys the cached ply graph; heap addresses are reused)
  int solver_players = 0;  // the mask last enqueued by caro_engine_set_solver: picks the select / back-up instances
  int gumbel_players = 0;  // the mask last enqueued by caro_engine_set_gumbel: picks the select / root policy / advance
                           // instances and whether searches launch gumbel_plan_kernel
  size_t next_event() {
    if (events_used == events.size()) {
      cudaEvent_t ev;
      cudaEventCreate(&ev);
      events.push_back(ev);
    }
    return events_used++;
  }
  void span_begin(int ph, cudaStream_t st) {
    if (profiling == 0 || (profiling == 1 && ph != 2)) return;
    open_span[ph] = next_event();
    cudaEventRecord(events[open_span[ph]], st);
  }
  void span_end(int ph, cudaStream_t st) {
    if (profiling == 0 || (profiling == 1 && ph != 2)) return;
    const size_t ev = next_event();
    cudaEventRecord(events[ev], st);
    spans[ph].push_back({open_span[ph], ev});
  }
};

namespace {

template <class Board>
void build_view(Carver& c, const Dims& dm, char* base, View<Board>* v) {
  const int64_t trees = (int64_t)dm.G * dm.tpg;
  const int64_t nodes = trees * dm.node_cap;
  const int64_t GB = (int64_t)dm.G * dm.B;
  auto P = [&](size_t off) { return base ? base + off : (char*)nullptr; };
#define CARVE(field, name, type, ...) v->field = reinterpret_cast<type*>(P(c.add(name, sizeof(type), __VA_ARGS__)))
  CARVE(N, "nodes", int32_t, nodes, 4, dm.Apad);  // node records: rows [N | W | P | C] (engine.cuh)
  v->W = reinterpret_cast<float*>(v->N) + dm.Apad;
  v->P = reinterpret_cast<float*>(v->N) + 2 * dm.Apad;
  v->C = v->N + 3 * dm.Apad;
  CARVE(key_hi, "key_hi", uint64_t, nodes);
  CARVE(node_board, "node_board", Board, nodes);
  CARVE(node_player, "node_player", uint8_t, nodes);
  CARVE(ht, "hash", HashSlot, trees, dm.hash_cap);
  CARVE(node_count, "node_count", int32_t, trees);
  CARVE(tree_gen, "tree_gen", uint32_t, trees);
  CARVE(root_board, "root_board", Board, dm.G);
  CARVE(root_player, "root_player", uint8_t, dm.G);
  CARVE(status, "status", uint8_t, dm.G);
  CARVE(ply, "ply", int32_t, dm.G);
  CARVE(result, "result", int32_t, dm.G);
  CARVE(uid, "uid", uint64_t, dm.G);
  CARVE(played, "played", uint32_t, dm.G);
  CARVE(hist_board, "hist_board", Board, dm.G, dm.max_plies);
  CARVE(hist_player, "hist_player", uint8_t, dm.G, dm.max_plies);
  CARVE(hist_pi, "hist_pi", float, dm.G, dm.max_plies, dm.A);
  CARVE(desc, "desc", DescRec<Board>, dm.G, dm.B);
  CARVE(d_path, "desc_path", uint32_t, dm.G, dm.B, dm.max_depth);
  CARVE(q_len, "queue_len", int32_t, dm.G);
  CARVE(q_entry, "queue", QEntry, dm.G, dm.B);
  CARVE(leaf_board, "leaf_board", Board, GB);
  CARVE(leaf_player, "leaf_player", uint8_t, GB);
  CARVE(leaf_count, "leaf_count", int32_t, 2);
  CARVE(noise, "noise", double, dm.G, dm.B, dm.A);
  CARVE(probs, "probs", float, GB, dm.A);
  CARVE(values, "values", float, GB);
  const int64_t rc = dm.replay_cap > 0 ? dm.replay_cap : 1;
  CARVE(rp_board, "replay_board", Board, rc);
  CARVE(rp_player, "replay_player", uint8_t, rc);
  CARVE(rp_pi, "replay_pi", float, rc, dm.A);
  CARVE(rp_z, "replay_z", float, rc);
  CARVE(rp_cursor, "replay_cursor", unsigned long long, 1);
  CARVE(ctr, "counters", unsigned long long, CTR_COUNT);
  // resignation (extension): carved after every other region so that no earlier offset moves; zero (= off) at create
  CARVE(resign_params, "resign_params", ResignParams, 1);
  CARVE(resign_playthrough, "resign_playthrough", uint8_t, dm.G);
  CARVE(resign_min, "resign_min", double, dm.G, 2);
  CARVE(resign_log, "resign_log", ResignRecord, dm.G);
  CARVE(resign_ctr, "resign_counters", unsigned long long, RCTR_COUNT);
  // MCTS solver (extension): after the resignation regions, for the same reason
  CARVE(solver_params, "solver_params", SolverParams, 1);
  CARVE(solver_ctr, "solver_counters", unsigned long long, SCTR_COUNT);
  // Gumbel root search (extension): after the solver regions, for the same reason
  CARVE(gumbel_params, "gumbel_params", GumbelParams, 1);
  CARVE(gumbel_g, "gumbel_g", double, dm.G, dm.A);
  CARVE(gumbel_state, "gumbel_state", GumbelState, dm.G);
  CARVE(gumbel_root, "gumbel_root", int16_t, dm.G, dm.B);
#undef CARVE
}

int fill_dims(const caro_engine_config* cfg, Dims* dm, int* max_plies) {
  if (!cfg) return caro_fail(CARO_E_ARG, "null config");
  if (cfg->games <= 0 || cfg->node_capacity <= 0) return caro_fail(CARO_E_ARG, "games and node_capacity must be positive");
  if (cfg->trees_per_game != 1 && cfg->trees_per_game != 2) return caro_fail(CARO_E_ARG, "trees_per_game must be 1 or 2");
  if (cfg->max_batch <= 0 || cfg->max_batch > 32) return caro_fail(CARO_E_ARG, "max_batch must be in 1..32");
  int A, plies;
  if (cfg->game == CARO_GAME_CONNECT4) {
    A = 7;
    plies = 42;
  } else if (cfg->game == CARO_GAME_MNK || cfg->game == CARO_GAME_CARO) {
    if (cfg->n < 2 || cfg->n > 15 || cfg->k < 2 || cfg->k > cfg->n) return caro_fail(CARO_E_ARG, "m,n,k needs 2 <= k <= n <= 15");
    A = cfg->n * cfg->n;
    plies = A;
  } else {
    return caro_fail(CARO_E_ARG, "unknown game");
  }
  dm->G = cfg->games;
  dm->tpg = cfg->trees_per_game;
  dm->B = cfg->max_batch;
  dm->A = A;
  dm->Apad = (A + 7) & ~7;
  dm->RS = 4 * dm->Apad;
  dm->node_cap = cfg->node_capacity;
  dm->hash_cap = round_pow2(2 * cfg->node_capacity);
  dm->max_depth = plies;
  dm->max_plies = plies;
  dm->replay_cap = cfg->replay_capacity;
  dm->flags = cfg->flags;
  if (cfg->flags & ~31u) return caro_fail(CARO_E_ARG, "unknown engine flags");
  if ((cfg->flags & FLAG_COMPACT_TREE) && compact_chunk_nodes(*dm) < 1)
    return caro_fail(CARO_E_ARG, "CARO_FLAG_COMPACT_TREE: node_capacity does not fit the shared-memory index map");
  *max_plies = plies;
  return CARO_OK;
}

inline cudaStream_t S(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// the select instance for the action count and the number of descents
template <class R, bool SOLVER, bool GUMBEL, class Board>
void launch_select_kernel(const View<Board>& v, const R& rules, const Dims& dm, const SearchParams& sp, int batch,
                          const double* src, cudaStream_t st) {
  const long long groups = (long long)dm.G * batch;
  auto grid = [&](int gw) { return (unsigned)((groups * gw + 255) / 256); };
  const int A = dm.A;
#define SELECT(GW, APL) select_kernel<R, GW, APL, SOLVER, GUMBEL><<<grid(GW), 256, 0, st>>>(v, rules, dm, sp, batch, src)
  // more descents than the GPU holds at once (5 blocks of 90-register threads per SM): the 72-register build keeps 7 blocks
  // per SM resident (-20 % at 16 k games, -12 % at 64 k; a few spilled words; CARO_SELECT_DENSE=0 switches it off)
  static const bool dense = !(getenv("CARO_SELECT_DENSE") && atoi(getenv("CARO_SELECT_DENSE")) == 0);
  if (A <= 8 && dense && groups > 128ll * 5 * 148) select_thread_dense_kernel<R, 2, 7, SOLVER, GUMBEL><<<(unsigned)((groups + 127) / 128), 128, 0, st>>>(v, rules, dm, sp, batch, src);
  else if (A <= 8) select_thread_kernel<R, 2, SOLVER, GUMBEL><<<(unsigned)((groups + 127) / 128), 128, 0, st>>>(v, rules, dm, sp, batch, src);
  else if constexpr (!std::is_same<R, C4Rules>::value) {  // lane-group kernels: m,n,k boards only (Connect4 has 7 actions)
    if (A <= 16) select_thread_kernel<R, 4, SOLVER, GUMBEL><<<(unsigned)((groups + 127) / 128), 128, 0, st>>>(v, rules, dm, sp, batch, src);
    else if (A <= 32) SELECT(32, 1);
    else if (A <= 64) SELECT(32, 2);
    else if (A <= 128) SELECT(32, 4);
    else SELECT(32, 8);
  }
#undef SELECT
}

// group width / actions per lane for the select and noise kernels
template <class R, class Board>
int launch_select(const View<Board>& v, const R& rules, const Dims& dm, const SearchParams& sp, int batch, int mb,
                  const double* noise, double* noise_out, cudaStream_t st, int phase, bool solver, bool gumbel) {
  // phase 0: noise (unless injected) + select; 1: only generate the Philox noise of minibatch `mb` into v.noise;
  // 2: only select, reading v.noise as generated by an earlier phase-1 call (the self-play pipeline issues the
  // noise of minibatch i+1 underneath the network pass of minibatch i: it depends on (uid, ply, i) alone)
  const long long groups = (long long)dm.G * batch;
  auto grid = [&](int gw) { return (unsigned)((groups * gw + 255) / 256); };
  const int A = dm.A;
  const double* src = phase == 2 ? v.noise : noise;
  if (src == nullptr) {  // Philox path: generate this minibatch's Dirichlet vectors first
    double* dst = noise_out ? noise_out : v.noise;
#define NOISE(GW, APL) noise_kernel<GW, APL><<<grid(GW), 256, 0, st>>>(v.uid, v.ply, v.root_player, dm, sp, batch, mb, dst)
    if (A <= 8) NOISE(8, 1);
    else if (A <= 16) NOISE(16, 1);
    else if (A <= 32) NOISE(32, 1);
    else if (A <= 64) NOISE(32, 2);
    else if (A <= 128) NOISE(32, 4);
    else NOISE(32, 8);
#undef NOISE
    src = dst;
    if (phase == 1) return caro_check_launch("noise_kernel");
  } else if (noise_out != nullptr && phase != 2) {
    cudaMemcpyAsync(noise_out, noise, sizeof(double) * (size_t)groups * A, cudaMemcpyDeviceToDevice, st);
  }
  if (dm.flags & FLAG_VIRTUAL_LOSS) {  // extension: sequential descents per game with virtual loss (one thread per game)
    static const bool vl_group = !(getenv("CARO_VL_GROUP") && atoi(getenv("CARO_VL_GROUP")) == 0);
    if (A <= 8 && vl_group) select_vl_group_kernel<R><<<(unsigned)(((long long)dm.G * 8 + 255) / 256), 256, 0, st>>>(v, rules, dm, sp, batch, src);
    else select_vl_kernel<R><<<(unsigned)((dm.G + 63) / 64), 64, 0, st>>>(v, rules, dm, sp, batch, src);
    return caro_check_launch("select_vl_kernel");
  }
  if (solver) launch_select_kernel<R, true, false>(v, rules, dm, sp, batch, src, st);
  else if (gumbel) launch_select_kernel<R, false, true>(v, rules, dm, sp, batch, src, st);
  else launch_select_kernel<R, false, false>(v, rules, dm, sp, batch, src, st);
  return caro_check_launch("select_kernel");
}

}  // namespace

static int do_reset(caro_engine* e, const uint8_t* h_game_mask, int first_player, int bump, void* stream);
void caro_pipeline_forget(unsigned long long engine_serial, unsigned long long net_serial);

extern "C" {

size_t caro_engine_workspace_bytes(const caro_engine_config* cfg) {
  Dims dm;
  int plies;
  if (fill_dims(cfg, &dm, &plies) != CARO_OK) return 0;
  Carver c;
  if (cfg->game == CARO_GAME_CONNECT4) {
    View<C4Board> v;
    build_view<C4Board>(c, dm, nullptr, &v);
  } else {
    View<MnkBoard> v;
    build_view<MnkBoard>(c, dm, nullptr, &v);
  }
  return (c.cur + 255) & ~(size_t)255;
}

int caro_engine_create(const caro_engine_config* cfg, void* d_workspace, size_t bytes, caro_engine** out, void* stream) {
  if (!out || !d_workspace) return caro_fail(CARO_E_ARG, "null argument");
  if (caro_device_count() <= 0) return caro_fail(CARO_E_CUDA, "no CUDA device: the engine has no CPU fallback");
  Dims dm;
  int plies;
  int rc = fill_dims(cfg, &dm, &plies);
  if (rc != CARO_OK) return rc;
  const size_t need = caro_engine_workspace_bytes(cfg);
  if (bytes < need) return caro_fail(CARO_E_ARG, "workspace too small");
  static std::atomic<unsigned long long> next_serial{0};
  caro_engine* e = new caro_engine();
  e->serial = ++next_serial;
  e->cfg = *cfg;
  e->dm = dm;
  e->max_plies = plies;
  e->sp.c_puct = cfg->c_puct;
  e->sp.alpha = cfg->alpha;
  e->sp.explore = cfg->explore;
  e->sp.seed_lo = (uint32_t)cfg->seed;
  e->sp.seed_hi = (uint32_t)(cfg->seed >> 32);
  e->ws = (char*)d_workspace;
  e->ws_bytes = need;
  e->mnk.n = cfg->n;
  e->mnk.k = cfg->k;
  e->mnk.blocked_ends = cfg->game == CARO_GAME_CARO ? 1 : 0;
  if (cfg->game == CARO_GAME_CONNECT4) {
    build_view<C4Board>(e->carve, dm, e->ws, &e->v_c4);
    e->board_bytes = sizeof(C4Board);
  } else {
    build_view<MnkBoard>(e->carve, dm, e->ws, &e->v_mnk);
    e->board_bytes = sizeof(MnkBoard);
  }
  cudaError_t ce = cudaMemsetAsync(e->ws, 0, need, S(stream));
  if (ce == cudaSuccess && (dm.flags & FLAG_COMPACT_TREE)) {  // here, not at launch: launches may sit inside a graph capture
    // the attribute belongs to the kernel, not to the engine: keep it at the largest request of any engine created so far
    static std::atomic<int> most[2] = {{0}, {0}};
    const int which = cfg->game == CARO_GAME_CONNECT4 ? 0 : 1;
    int smem = (int)compact_smem_bytes(dm, compact_chunk_nodes(dm));
    int seen = most[which].load();
    while (smem > seen && !most[which].compare_exchange_weak(seen, smem)) {}
    smem = smem > seen ? smem : seen;
    if (which == 0) ce = cudaFuncSetAttribute(compact_kernel<C4Rules>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    else ce = cudaFuncSetAttribute(compact_kernel<MnkRules>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  }
  if (ce != cudaSuccess) {
    delete e;
    return caro_fail(CARO_E_CUDA, cudaGetErrorString(ce));
  }
  *out = e;
  return do_reset(e, nullptr, -1, 0, stream);
}

void caro_engine_destroy(caro_engine* e) {
  if (!e) return;
  caro_pipeline_forget(e->serial, 0);
  for (cudaEvent_t ev : e->events) cudaEventDestroy(ev);
  if (e->sync_a) cudaEventDestroy(e->sync_a);
  if (e->sync_b) cudaEventDestroy(e->sync_b);
  delete e;
}

int caro_engine_profile(caro_engine* e, int enable) {
  if (!e) return caro_fail(CARO_E_ARG, "null engine");
  e->profiling = enable < 0 ? 0 : (enable > 2 ? 2 : enable);
  e->events_used = 0;
  e->launches = 0;
  for (auto& v : e->spans) v.clear();
  return CARO_OK;
}

int caro_engine_profile_read(caro_engine* e, double h_ms[5], uint64_t* h_launches, void* stream) {
  if (!e || !h_ms) return caro_fail(CARO_E_ARG, "null argument");
  cudaError_t ce = cudaStreamSynchronize(S(stream));
  if (ce != cudaSuccess) return caro_fail(CARO_E_CUDA, cudaGetErrorString(ce));
  for (int ph = 0; ph < 5; ++ph) {
    h_ms[ph] = 0.0;
    for (const auto& sp : e->spans[ph]) {
      float ms = 0.0f;
      cudaEventElapsedTime(&ms, e->events[sp.first], e->events[sp.second]);
      h_ms[ph] += (double)ms;
    }
    e->spans[ph].clear();
  }
  if (h_launches) *h_launches = e->launches;
  e->events_used = 0;
  e->launches = 0;
  return CARO_OK;
}

int caro_engine_region(const caro_engine* e, const char* name, size_t* offset, size_t* bytes, int32_t* elem_bytes,
                       int64_t dims[4]) {
  if (!e || !name) return caro_fail(CARO_E_ARG, "null argument");
  for (const Region& r : e->carve.regions) {
    if (r.name == name) {
      if (offset) *offset = r.offset;
      if (bytes) *bytes = r.bytes;
      if (elem_bytes) *elem_bytes = r.elem;
      if (dims) memcpy(dims, r.dims, sizeof(r.dims));
      return CARO_OK;
    }
  }
  return caro_fail(CARO_E_ARG, "unknown region");
}

int caro_engine_reset(caro_engine* e, const uint8_t* h_game_mask, int first_player, void* stream) {
  return do_reset(e, h_game_mask, first_player, 1, stream);
}

}  // extern "C"

static int do_reset(caro_engine* e, const uint8_t* h_game_mask, int first_player, int bump, void* stream) {
  if (!e) return caro_fail(CARO_E_ARG, "null engine");
  uint8_t* d_mask = nullptr;
  if (h_game_mask) {
    // staged through the (currently unused) leaf_player region: G <= G*B bytes
    d_mask = e->cfg.game == CARO_GAME_CONNECT4 ? e->v_c4.leaf_player : e->v_mnk.leaf_player;
    cudaError_t ce = cudaMemcpyAsync(d_mask, h_game_mask, (size_t)e->dm.G, cudaMemcpyHostToDevice, S(stream));
    if (ce != cudaSuccess) return caro_fail(CARO_E_CUDA, cudaGetErrorString(ce));
  }
  const unsigned grid = (unsigned)((e->dm.G + 127) / 128);
  if (e->cfg.game == CARO_GAME_CONNECT4)
    reset_kernel<C4Rules><<<grid, 128, 0, S(stream)>>>(e->v_c4, e->dm, e->sp, d_mask, first_player, bump);
  else
    reset_kernel<MnkRules><<<grid, 128, 0, S(stream)>>>(e->v_mnk, e->dm, e->sp, d_mask, first_player, bump);
  return caro_check_launch("reset_kernel");
}

extern "C" {

int caro_engine_set_roots(caro_engine* e, const void* h_boards, const uint8_t* h_players, void* stream) {
  if (!e || !h_boards || !h_players) return caro_fail(CARO_E_ARG, "null argument");
  void* d_b = e->cfg.game == CARO_GAME_CONNECT4 ? (void*)e->v_c4.root_board : (void*)e->v_mnk.root_board;
  uint8_t* d_p = e->cfg.game == CARO_GAME_CONNECT4 ? e->v_c4.root_player : e->v_mnk.root_player;
  uint8_t* d_s = e->cfg.game == CARO_GAME_CONNECT4 ? e->v_c4.status : e->v_mnk.status;
  cudaError_t ce = cudaMemcpyAsync(d_b, h_boards, e->board_bytes * (size_t)e->dm.G, cudaMemcpyHostToDevice, S(stream));
  if (ce == cudaSuccess) ce = cudaMemcpyAsync(d_p, h_players, (size_t)e->dm.G, cudaMemcpyHostToDevice, S(stream));
  if (ce == cudaSuccess) ce = cudaMemsetAsync(d_s, ST_ACTIVE, (size_t)e->dm.G, S(stream));
  if (ce != cudaSuccess) return caro_fail(CARO_E_CUDA, cudaGetErrorString(ce));
  return CARO_OK;
}

int caro_engine_select(caro_engine* e, int batch, int minibatch_index, const double* d_noise, double* d_noise_out,
                       void* stream) {
  if (!e) return caro_fail(CARO_E_ARG, "null engine");
  if (batch <= 0 || batch > e->dm.B) return caro_fail(CARO_E_ARG, "batch exceeds max_batch");
  if (e->cfg.game == CARO_GAME_CONNECT4)
    return launch_select<C4Rules>(e->v_c4, C4Rules(), e->dm, e->sp, batch, minibatch_index, d_noise, d_noise_out, S(stream), 0,
                                  e->solver_players != 0, e->gumbel_players != 0);
  return launch_select<MnkRules>(e->v_mnk, e->mnk, e->dm, e->sp, batch, minibatch_index, d_noise, d_noise_out, S(stream), 0,
                                 e->solver_players != 0, e->gumbel_players != 0);
}

int caro_engine_plan(caro_engine* e, int batch, void* stream) {
  if (!e) return caro_fail(CARO_E_ARG, "null engine");
  if (batch <= 0 || batch > e->dm.B) return caro_fail(CARO_E_ARG, "batch exceeds max_batch");
  const bool c4 = e->cfg.game == CARO_GAME_CONNECT4;
  const int G = e->dm.G;
#define LAUNCH_PLAN(GP)                                                                                     \
  do {                                                                                                      \
    const unsigned grid = (unsigned)(((long long)G * GP + 255) / 256);                                      \
    if (c4) plan_kernel<C4Board, GP><<<grid, 256, 0, S(stream)>>>(e->v_c4, e->dm, batch);                   \
    else plan_kernel<MnkBoard, GP><<<grid, 256, 0, S(stream)>>>(e->v_mnk, e->dm, batch);                    \
  } while (0)
  if (batch <= 8) LAUNCH_PLAN(8);
  else if (batch <= 16) LAUNCH_PLAN(16);
  else LAUNCH_PLAN(32);
#undef LAUNCH_PLAN
  return caro_check_launch("plan_kernel");
}

int caro_engine_expand_backup(caro_engine* e, int batch, const float* d_probs, const float* d_values, void* stream) {
  if (!e || !d_probs || !d_values) return caro_fail(CARO_E_ARG, "null argument");
  const unsigned grid = (unsigned)(((long long)e->dm.G * 32 + 127) / 128);
  const bool c4 = e->cfg.game == CARO_GAME_CONNECT4;
  const bool sol = e->solver_players != 0;  // the proof pass lives in the SOLVER instances only
#define LAUNCH_EB(BK)                                                                                                       \
  do {                                                                                                                      \
    if (c4 && sol) expand_backup_kernel<C4Rules, BK, true><<<grid, 128, 0, S(stream)>>>(e->v_c4, e->dm, batch, d_probs, d_values); \
    else if (c4) expand_backup_kernel<C4Rules, BK, false><<<grid, 128, 0, S(stream)>>>(e->v_c4, e->dm, batch, d_probs, d_values); \
    else if (sol) expand_backup_kernel<MnkRules, BK, true><<<grid, 128, 0, S(stream)>>>(e->v_mnk, e->dm, batch, d_probs, d_values); \
    else expand_backup_kernel<MnkRules, BK, false><<<grid, 128, 0, S(stream)>>>(e->v_mnk, e->dm, batch, d_probs, d_values);  \
  } while (0)
  // eight lanes per game inside the parts pipeline (a quarter of the warps: +2.5 % there, where the tree kernels live in
  // the warp slots next to tower CTAs), one warp per game otherwise (20 us instead of 36 us stand-alone at 4,096 games)
  static const int group8 = getenv("CARO_EXPAND_GROUP8") ? atoi(getenv("CARO_EXPAND_GROUP8")) : 1;  // 0 never, 1 auto, 2 always
  // (and stand-alone from 32 k games per launch: 138 us instead of 194 us at 65,536 games -- a quarter of the warps, one wave less)
  if (batch <= 8 && e->dm.Apad <= 8 && c4 && group8 && (e->lean_tree || group8 == 2 || e->dm.G >= 32768)) {
    const unsigned g8 = (unsigned)(((long long)e->dm.G * 8 + 127) / 128);
    if (sol) expand_backup_group8_kernel<C4Rules, true><<<g8, 128, 0, S(stream)>>>(e->v_c4, e->dm, batch, d_probs, d_values);
    else expand_backup_group8_kernel<C4Rules, false><<<g8, 128, 0, S(stream)>>>(e->v_c4, e->dm, batch, d_probs, d_values);
  } else if (batch <= 8) LAUNCH_EB(8);
  else if (batch <= 16) LAUNCH_EB(16);
  else LAUNCH_EB(32);
#undef LAUNCH_EB
  return caro_check_launch("expand_backup_kernel");
}

}  // extern "C"

// One minibatch.  `s_tree` runs noise/select/plan and expand+backup, `s_net` the network; when they differ the
// hand-offs are CUDA events, so that another engine's tree kernels can run underneath this engine's network pass.
static int select_phase(caro_engine* e, int batch, int mb, int phase, cudaStream_t st) {
  if (e->cfg.game == CARO_GAME_CONNECT4)
    return launch_select<C4Rules>(e->v_c4, C4Rules(), e->dm, e->sp, batch, mb, nullptr, nullptr, st, phase, e->solver_players != 0,
                                  e->gumbel_players != 0);
  return launch_select<MnkRules>(e->v_mnk, e->mnk, e->dm, e->sp, batch, mb, nullptr, nullptr, st, phase, e->solver_players != 0,
                                 e->gumbel_players != 0);
}

// `prefetch`: 0 = noise + select as one step, 1 = minibatch i's noise was issued by the previous step, and this
// step issues minibatch i+1's (if `more`) right behind its plan kernel, i.e. underneath its own network pass.
// Minibatch `k` of `count` of the search numbered `search_index` draws the noise of minibatch i = search_index + k.
static int search_step(caro_engine* e, caro_net* net, int search_index, int k, int count, int batch, int net_impl,
                       cudaStream_t s_tree, cudaStream_t s_net, int prefetch = 0, bool more = false) {
  const int i = search_index + k;
  const bool c4 = e->cfg.game == CARO_GAME_CONNECT4;
  const void* lb = c4 ? (const void*)e->v_c4.leaf_board : (const void*)e->v_mnk.leaf_board;
  const uint8_t* lp = c4 ? e->v_c4.leaf_player : e->v_mnk.leaf_player;
  const int32_t* lc = c4 ? e->v_c4.leaf_count : e->v_mnk.leaf_count;
  float* pr = c4 ? e->v_c4.probs : e->v_mnk.probs;
  float* va = c4 ? e->v_c4.values : e->v_mnk.values;
  const bool cross = s_tree != s_net;
  if (cross && !e->sync_a) {
    cudaEventCreateWithFlags(&e->sync_a, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&e->sync_b, cudaEventDisableTiming);
  }
  int rc = CARO_OK;
  if (!(prefetch && i > 0)) {  // this minibatch's Dirichlet vectors (in the pipeline they were issued under the previous network pass)
    e->span_begin(4, s_tree);
    rc = select_phase(e, batch, i, 1, s_tree);
    e->span_end(4, s_tree);
  }
  if (rc == CARO_OK && e->gumbel_players != 0) rc = caro_engine_gumbel_plan(e, search_index, k, count, batch, s_tree);
  e->span_begin(0, s_tree);
  if (rc == CARO_OK) rc = select_phase(e, batch, i, 2, s_tree);
  e->span_end(0, s_tree);
  e->span_begin(1, s_tree);
  if (rc == CARO_OK) rc = caro_engine_plan(e, batch, s_tree);
  e->span_end(1, s_tree);
  if (cross) {
    cudaEventRecord(e->sync_a, s_tree);
    cudaStreamWaitEvent(s_net, e->sync_a, 0);
  }
  if (prefetch && more && rc == CARO_OK) rc = select_phase(e, batch, i + 1, 1, s_tree);
  e->span_begin(2, s_net);
  if (rc == CARO_OK)
    rc = caro_net_forward(net, e->cfg.game, e->cfg.n, e->cfg.k, lb, lp, lc, (int64_t)e->dm.G * batch, pr, va, net_impl, s_net);
  e->span_end(2, s_net);
  if (cross) {
    cudaEventRecord(e->sync_b, s_net);
    cudaStreamWaitEvent(s_tree, e->sync_b, 0);
  }
  e->span_begin(3, s_tree);
  if (rc == CARO_OK) rc = caro_engine_expand_backup(e, batch, pr, va, s_tree);
  e->span_end(3, s_tree);
  e->launches += e->gumbel_players != 0 ? 6 : 5;
  return rc;
}

// ------------------------------------------------------------------------------ parts pipeline
// Streams, events and the captured ply graph of the multi-part self-play pipeline, one context per CUDA device.  The
// graph bakes in workspace pointers, dimensions, network weight pointers, the tower's by-value constants and its grid,
// so it is keyed by the SERIAL NUMBERS of the engines and of the network (never reused, unlike heap addresses), the
// network's weight version and grid limit, and every scalar parameter; destroying an engine or a network drops any
// graph that refers to it (caro_pipeline_forget).
namespace {

constexpr int kMaxParts = 8;
constexpr int kMaxDevices = 64;

struct MultiGraph {  // one captured ply, replayed while its key stays the same
  cudaGraphExec_t exec = nullptr;
  unsigned long long engine_serial[kMaxParts] = {0};
  unsigned long long net_serial = 0, net_version = 0;
  int n = 0, count = 0, batch = 0, tau = 0, restart = 0, first = 0, impl = 0, grid_limit = 0;
  unsigned long long launches_per_ply = 0;
};

struct PipelineCtx {
  bool ready = false;
  cudaStream_t s_side[kMaxParts] = {nullptr};
  cudaStream_t s_cap = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join[kMaxParts] = {nullptr};
  MultiGraph mg;
};

PipelineCtx g_pipeline[kMaxDevices];

PipelineCtx* pipeline_ctx() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return nullptr;
  PipelineCtx* c = &g_pipeline[dev];
  if (!c->ready) {
    for (int h = 0; h < kMaxParts; ++h) {
      cudaStreamCreateWithFlags(&c->s_side[h], cudaStreamNonBlocking);
      cudaEventCreateWithFlags(&c->ev_join[h], cudaEventDisableTiming);
    }
    cudaStreamCreateWithFlags(&c->s_cap, cudaStreamNonBlocking);
    cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming);
    c->ready = true;
  }
  return c;
}

void drop_graph(MultiGraph* mg) {
  if (mg->exec) cudaGraphExecDestroy(mg->exec);
  *mg = MultiGraph();
}

}  // namespace

// Called by caro_engine_destroy / caro_net_destroy / caro_net_update: a cached ply graph that refers to the object
// must never be replayed again (its workspace / weight images may be freed or rewritten).
void caro_pipeline_forget(unsigned long long engine_serial, unsigned long long net_serial) {
  for (int d = 0; d < kMaxDevices; ++d) {
    MultiGraph* mg = &g_pipeline[d].mg;
    if (!mg->exec) continue;
    bool hit = net_serial != 0 && mg->net_serial == net_serial;
    for (int h = 0; h < mg->n; ++h) hit = hit || (engine_serial != 0 && mg->engine_serial[h] == engine_serial);
    if (hit) drop_graph(mg);
  }
}

extern "C" {

int caro_engine_search(caro_engine* e, caro_net* net, int count, int batch, int first_minibatch, int net_impl, void* stream) {
  if (!e || !net) return caro_fail(CARO_E_ARG, "null argument");
  if (first_minibatch < 0) return caro_fail(CARO_E_ARG, "first_minibatch must be >= 0");
  for (int i = 0; i < count; ++i) {
    const int rc = search_step(e, net, first_minibatch, i, count, batch, net_impl, S(stream), S(stream));
    if (rc != CARO_OK) return rc;
  }
  return CARO_OK;
}

// One ply of the multi-part pipeline: `count` minibatches of every part (round robin), then the advance kernels.
// Every part keeps its tree kernels AND its network passes on its own side stream: the parts are independent chains,
// and the tail of one part's network kernel (CTAs that ran out of groups) overlaps the head of the next part's.
static int multi_ply(caro_engine** es, int n, caro_net* net, int count, int batch, int tau_plies, int auto_restart,
                     int first_player, int net_impl, cudaStream_t* s_side) {
  int rc = CARO_OK;
  for (int h = 0; h < n; ++h) es[h]->lean_tree = n >= 2;
  struct LeanOff {
    caro_engine** es;
    int n;
    ~LeanOff() { for (int h = 0; h < n; ++h) es[h]->lean_tree = false; }
  } lean_off{es, n};
  for (int i = 0; i < count && rc == CARO_OK; ++i)
    for (int h = 0; h < n && rc == CARO_OK; ++h) rc = search_step(es[h], net, 0, i, count, batch, net_impl, s_side[h], s_side[h], 1, i + 1 < count);
  for (int h = 0; h < n && rc == CARO_OK; ++h) {
    rc = caro_engine_advance(es[h], tau_plies, nullptr, auto_restart, first_player, nullptr, s_side[h]);
    es[h]->launches += 1;
  }
  return rc;
}

int caro_engine_play_multi(caro_engine** engines, int n, caro_net* net, int moves, int count, int batch, int tau_plies,
                           int auto_restart, int first_player, int net_impl, void* stream) {
  if (!engines || !net || n < 1 || n > kMaxParts) return caro_fail(CARO_E_ARG, "need 1..8 engines and a network");
  for (int h = 0; h < n; ++h)
    if (!engines[h]) return caro_fail(CARO_E_ARG, "null engine");
  PipelineCtx* cx = pipeline_ctx();
  if (!cx) return caro_fail(CARO_E_CUDA, "no current CUDA device for the parts pipeline");
  // With profiling off the whole ply (n x count x 5 kernels + n) is captured once into a CUDA graph and replayed per
  // ply: the host issues one graph launch instead of ~500 n kernel launches and ~400 n event operations.
  bool profiling = false;
  for (int h = 0; h < n; ++h) profiling = profiling || engines[h]->profiling != 0;
  const bool use_graph = !profiling && !getenv("CARO_NO_GRAPH");
  auto fork_join = [&](cudaStream_t s_main, auto&& body) {
    cudaEventRecord(cx->ev_fork, s_main);
    for (int h = 0; h < n; ++h) cudaStreamWaitEvent(cx->s_side[h], cx->ev_fork, 0);
    const int rc = body();
    for (int h = 0; h < n; ++h) {
      cudaEventRecord(cx->ev_join[h], cx->s_side[h]);
      cudaStreamWaitEvent(s_main, cx->ev_join[h], 0);
    }
    return rc;
  };
  // with two or more parts the tower leaves a ninth of the SMs to the other parts' tree kernels (unless the caller
  // set its own limit); the value is baked into a captured ply graph, so it only has to hold while launches are issued
  struct PipelineGrid {
    caro_net* net;
    PipelineGrid(caro_net* n_, int parts) : net(n_) {
      if (parts >= 2 && !(getenv("CARO_PIPELINE_SMS") && atoi(getenv("CARO_PIPELINE_SMS")) == 0))
        net->pipeline_limit = getenv("CARO_PIPELINE_SMS") ? atoi(getenv("CARO_PIPELINE_SMS")) : net->sm_count - net->sm_count / 9;
    }
    ~PipelineGrid() { net->pipeline_limit = 0; }
  } pipeline_grid(net, n);
  if (use_graph) {
    MultiGraph& mg = cx->mg;
    bool same = mg.exec && mg.n == n && mg.net_serial == net->serial && mg.net_version == net->version &&
                mg.grid_limit == net->grid_limit && mg.count == count && mg.batch == batch && mg.tau == tau_plies &&
                mg.restart == auto_restart && mg.first == first_player && mg.impl == net_impl;
    for (int h = 0; h < n && same; ++h) same = mg.engine_serial[h] == engines[h]->serial;
    if (!same) {
      drop_graph(&mg);
      unsigned long long before = 0, after = 0, saved[kMaxParts];
      for (int h = 0; h < n; ++h) {
        saved[h] = engines[h]->launches;
        before += engines[h]->launches;
      }
      cudaGraph_t graph = nullptr;
      cudaGraphExec_t exec = nullptr;
      cudaError_t ce = cudaStreamBeginCapture(cx->s_cap, cudaStreamCaptureModeThreadLocal);
      int rc = CARO_OK;
      if (ce == cudaSuccess) {
        rc = fork_join(cx->s_cap, [&] {
          return multi_ply(engines, n, net, count, batch, tau_plies, auto_restart, first_player, net_impl, cx->s_side);
        });
        ce = cudaStreamEndCapture(cx->s_cap, &graph);
      }
      if (ce == cudaSuccess && rc == CARO_OK) ce = cudaGraphInstantiate(&exec, graph, 0);
      if (graph) cudaGraphDestroy(graph);
      for (int h = 0; h < n; ++h) {
        after += engines[h]->launches;
        engines[h]->launches = saved[h];  // capturing launches nothing
      }
      if (ce != cudaSuccess || rc != CARO_OK) {
        if (exec) cudaGraphExecDestroy(exec);
        cudaGetLastError();
        return caro_fail(CARO_E_CUDA, "CUDA graph capture of the self-play pipeline failed");
      }
      mg.exec = exec;
      mg.launches_per_ply = after - before;
      mg.n = n; mg.net_serial = net->serial; mg.net_version = net->version; mg.grid_limit = net->grid_limit;
      mg.count = count; mg.batch = batch; mg.tau = tau_plies;
      mg.restart = auto_restart; mg.first = first_player; mg.impl = net_impl;
      for (int h = 0; h < n; ++h) mg.engine_serial[h] = engines[h]->serial;
    }
    for (int m = 0; m < moves; ++m) {
      const cudaError_t ce = cudaGraphLaunch(mg.exec, S(stream));
      if (ce != cudaSuccess) return caro_fail(CARO_E_CUDA, cudaGetErrorString(ce));
      engines[0]->launches += mg.launches_per_ply;  // kernels executed by the replay (attributed to the first part)
    }
    return CARO_OK;
  }
  return fork_join(S(stream), [&] {
    int rc = CARO_OK;
    for (int m = 0; m < moves && rc == CARO_OK; ++m)
      rc = multi_ply(engines, n, net, count, batch, tau_plies, auto_restart, first_player, net_impl, cx->s_side);
    return rc;
  });
}

int caro_engine_root_policy(caro_engine* e, int tau_mode, int tau_plies, double* d_pi, float* d_q, int32_t* d_n, void* stream) {
  if (!e) return caro_fail(CARO_E_ARG, "null engine");
  const unsigned grid = (unsigned)((e->dm.G + 127) / 128);
  const bool gum = e->gumbel_players != 0;
  if (e->cfg.game == CARO_GAME_CONNECT4) {
    if (gum) root_policy_kernel<C4Rules, true><<<grid, 128, 0, S(stream)>>>(e->v_c4, C4Rules(), e->dm, tau_mode, tau_plies, d_pi, d_q, d_n);
    else root_policy_kernel<C4Rules, false><<<grid, 128, 0, S(stream)>>>(e->v_c4, C4Rules(), e->dm, tau_mode, tau_plies, d_pi, d_q, d_n);
  } else {
    if (gum) root_policy_kernel<MnkRules, true><<<grid, 128, 0, S(stream)>>>(e->v_mnk, e->mnk, e->dm, tau_mode, tau_plies, d_pi, d_q, d_n);
    else root_policy_kernel<MnkRules, false><<<grid, 128, 0, S(stream)>>>(e->v_mnk, e->mnk, e->dm, tau_mode, tau_plies, d_pi, d_q, d_n);
  }
  return caro_check_launch("root_policy_kernel");
}

int caro_engine_advance(caro_engine* e, int tau_plies, const double* d_uniform, int auto_restart, int first_player,
                        int32_t* d_action_out, void* stream) {
  if (!e) return caro_fail(CARO_E_ARG, "null engine");
  const unsigned grid = (unsigned)((e->dm.G + 127) / 128);
#define LAUNCH_ADVANCE(R, V, RULES, GUM) \
  advance_kernel<R, GUM><<<grid, 128, 0, S(stream)>>>(e->V, RULES, e->dm, e->sp, tau_plies, d_uniform, auto_restart, first_player, d_action_out)
  const bool gum = e->gumbel_players != 0;
  if (e->cfg.game == CARO_GAME_CONNECT4) {
    if (gum) LAUNCH_ADVANCE(C4Rules, v_c4, C4Rules(), true);
    else LAUNCH_ADVANCE(C4Rules, v_c4, C4Rules(), false);
  } else {
    if (gum) LAUNCH_ADVANCE(MnkRules, v_mnk, e->mnk, true);
    else LAUNCH_ADVANCE(MnkRules, v_mnk, e->mnk, false);
  }
#undef LAUNCH_ADVANCE
  int rc = caro_check_launch("advance_kernel");
  if (rc == CARO_OK && (e->dm.flags & FLAG_COMPACT_TREE)) {  // drop what the move made unreachable, pack the arenas
    const int chunk = compact_chunk_nodes(e->dm);
    const size_t smem = compact_smem_bytes(e->dm, chunk);
    const unsigned trees = (unsigned)(e->dm.G * e->dm.tpg);
    if (e->cfg.game == CARO_GAME_CONNECT4) compact_kernel<C4Rules><<<trees, 256, smem, S(stream)>>>(e->v_c4, C4Rules(), e->dm, chunk);
    else compact_kernel<MnkRules><<<trees, 256, smem, S(stream)>>>(e->v_mnk, e->mnk, e->dm, chunk);
    rc = caro_check_launch("compact_kernel");
  }
  return rc;
}

int caro_engine_play(caro_engine* e, caro_net* net_p0, caro_net* net_p1, int moves, int count, int batch, int tau_plies,
                     int auto_restart, int first_player, int net_impl, void* stream) {
  if (!e || !net_p0 || !net_p1) return caro_fail(CARO_E_ARG, "null argument");
  if (net_p0 != net_p1 && (first_player < 0 || auto_restart))
    return caro_fail(CARO_E_ARG, "two different nets need a fixed first player and no auto-restart (lock-step plies)");
  for (int m = 0; m < moves; ++m) {
    caro_net* net = net_p0;
    if (net_p0 != net_p1) net = ((first_player ^ (m & 1)) == 0) ? net_p0 : net_p1;
    int rc = caro_engine_search(e, net, count, batch, 0, net_impl, stream);
    if (rc == CARO_OK) rc = caro_engine_advance(e, tau_plies, nullptr, auto_restart, first_player, nullptr, stream);
    if (rc != CARO_OK) return rc;
    e->launches += 1;
  }
  return CARO_OK;
}

int caro_engine_replay_gather(caro_engine* e, const int64_t* d_entries, const int32_t* d_symmetry, int64_t count, float* d_planes,
                              float* d_pi, float* d_z, void* stream) {
  if (!e || !d_entries || !d_planes || !d_pi || !d_z) return caro_fail(CARO_E_ARG, "null argument");
  if (e->dm.replay_cap <= 0) return caro_fail(CARO_E_STATE, "the engine was created without a replay ring");
  if (count <= 0) return CARO_OK;
  const long long* ent = reinterpret_cast<const long long*>(d_entries);
  if (e->cfg.game == CARO_GAME_CONNECT4)
    replay_gather_kernel<C4Rules><<<(unsigned)count, 64, 0, S(stream)>>>(e->v_c4, C4Rules(), e->dm, ent, d_symmetry, (long long)count, d_planes, d_pi, d_z);
  else
    replay_gather_kernel<MnkRules><<<(unsigned)count, 64, 0, S(stream)>>>(e->v_mnk, e->mnk, e->dm, ent, d_symmetry, (long long)count, d_planes, d_pi, d_z);
  return caro_check_launch("replay_gather_kernel");
}

int caro_engine_set_resign(caro_engine* e, int enable, double threshold, double playthrough, void* stream) {
  if (!e) return caro_fail(CARO_E_ARG, "null engine");
  if (!(threshold >= -1.0 && threshold <= 1.0)) return caro_fail(CARO_E_ARG, "resign threshold must be in [-1, 1]");
  if (!(playthrough >= 0.0 && playthrough <= 1.0)) return caro_fail(CARO_E_ARG, "resign playthrough must be in [0, 1]");
  ResignParams p{};
  p.enabled = enable ? 1 : 0;
  p.threshold = threshold;
  p.playthrough = playthrough;
  ResignParams* dst = e->cfg.game == CARO_GAME_CONNECT4 ? e->v_c4.resign_params : e->v_mnk.resign_params;
  set_resign_kernel<<<1, 1, 0, S(stream)>>>(dst, p);
  return caro_check_launch("set_resign_kernel");
}

int caro_engine_set_solver(caro_engine* e, int players, void* stream) {
  if (!e) return caro_fail(CARO_E_ARG, "null engine");
  if (players < 0 || players > 3) return caro_fail(CARO_E_ARG, "solver players must be a mask in 0..3");
  if (players != 0 && (e->dm.flags & FLAG_VIRTUAL_LOSS))
    return caro_fail(CARO_E_ARG, "the solver does not run with virtual loss");
  if ((players == 1 || players == 2) && e->dm.tpg == 1)
    return caro_fail(CARO_E_ARG, "a per-player solver mask needs two trees per game (one tree serves both players)");
  if (players != 0 && e->gumbel_players != 0) return caro_fail(CARO_E_ARG, "the solver does not run with the Gumbel root search");
  SolverParams p{};
  p.players = players;
  SolverParams* dst = e->cfg.game == CARO_GAME_CONNECT4 ? e->v_c4.solver_params : e->v_mnk.solver_params;
  set_solver_kernel<<<1, 1, 0, S(stream)>>>(dst, p);
  const int rc = caro_check_launch("set_solver_kernel");
  if (rc == CARO_OK && (players != 0) != (e->solver_players != 0))
    caro_pipeline_forget(e->serial, 0);  // a captured ply graph holds the other select / back-up instances
  if (rc == CARO_OK) e->solver_players = players;
  return rc;
}

int caro_engine_set_gumbel(caro_engine* e, int players, int m, double c_visit, double c_scale, double gumbel_scale,
                           void* stream) {
  if (!e) return caro_fail(CARO_E_ARG, "null engine");
  if (players < 0 || players > 3) return caro_fail(CARO_E_ARG, "gumbel players must be a mask in 0..3");
  if ((players == 1 || players == 2) && e->dm.tpg == 1)
    return caro_fail(CARO_E_ARG, "a per-player gumbel mask needs two trees per game (one tree serves both players)");
  if (players != 0 && (e->dm.flags & FLAG_VIRTUAL_LOSS))
    return caro_fail(CARO_E_ARG, "the Gumbel root search does not run with virtual loss");
  if (players != 0 && e->solver_players != 0) return caro_fail(CARO_E_ARG, "the Gumbel root search does not run with the solver");
  if (m < 1 || m > kGumbelMaxM) return caro_fail(CARO_E_ARG, "gumbel m must be in 1..32");
  const double v[3] = {c_visit, c_scale, gumbel_scale};
  for (double x : v)
    if (!(x >= 0.0 && x <= 1.7976931348623157e308)) return caro_fail(CARO_E_ARG, "gumbel c_visit, c_scale and scale must be finite and >= 0");
  GumbelParams p{};
  p.players = players;
  p.m = m;
  p.c_visit = c_visit;
  p.c_scale = c_scale;
  p.gumbel_scale = gumbel_scale;
  GumbelParams* dst = e->cfg.game == CARO_GAME_CONNECT4 ? e->v_c4.gumbel_params : e->v_mnk.gumbel_params;
  set_gumbel_kernel<<<1, 1, 0, S(stream)>>>(dst, p);
  const int rc = caro_check_launch("set_gumbel_kernel");
  if (rc == CARO_OK && (players != 0) != (e->gumbel_players != 0))
    caro_pipeline_forget(e->serial, 0);  // a captured ply graph holds the other instances (and no gumbel_plan_kernel)
  if (rc == CARO_OK) e->gumbel_players = players;
  return rc;
}

int caro_engine_gumbel_plan(caro_engine* e, int search_index, int minibatch, int count, int batch, void* stream) {
  if (!e) return caro_fail(CARO_E_ARG, "null engine");
  if (search_index < 0 || count < 1 || minibatch < 0 || minibatch >= count)
    return caro_fail(CARO_E_ARG, "gumbel plan needs search_index >= 0 and 0 <= minibatch < count");
  if (batch <= 0 || batch > e->dm.B) return caro_fail(CARO_E_ARG, "batch exceeds max_batch");
  if (e->gumbel_players == 0) return CARO_OK;
  const unsigned grid = (unsigned)(((long long)e->dm.G * 32 + 127) / 128);
  if (e->cfg.game == CARO_GAME_CONNECT4)
    gumbel_plan_kernel<C4Rules><<<grid, 128, 0, S(stream)>>>(e->v_c4, C4Rules(), e->dm, e->sp, search_index, minibatch, count, batch);
  else
    gumbel_plan_kernel<MnkRules><<<grid, 128, 0, S(stream)>>>(e->v_mnk, e->mnk, e->dm, e->sp, search_index, minibatch, count, batch);
  return caro_check_launch("gumbel_plan_kernel");
}

int caro_engine_counters(caro_engine* e, uint64_t h_out[8], void* stream) {
  if (!e || !h_out) return caro_fail(CARO_E_ARG, "null argument");
  const unsigned long long* src = e->cfg.game == CARO_GAME_CONNECT4 ? e->v_c4.ctr : e->v_mnk.ctr;
  cudaError_t ce = cudaMemcpyAsync(h_out, src, 8 * sizeof(uint64_t), cudaMemcpyDeviceToHost, S(stream));
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(S(stream));
  if (ce != cudaSuccess) return caro_fail(CARO_E_CUDA, cudaGetErrorString(ce));
  return CARO_OK;
}

}  // extern "C"
