// azg_arena.cu -- K4: GPU-resident search arena (kernels + C ABI).
// Per-game logic lives in azg_arena_core.cuh (shared with the host check build); this file
// maps games onto lane groups and launches.  Grid sizing: 8 lanes per game, 128-thread CTAs
// (16 games each) -- the work per game is a short pointer chase through its own table
// (~150 B per visited node, SURVEY section 8d), so the kernels are latency-bound and want many
// resident warps rather than big CTAs.
#include "azg_arena_core.cuh"

#include <new>

struct azg_arena {
  AzgArenaView view;
  int game, n;
};

namespace {

constexpr int kLanes = 8;     // lanes per game
constexpr int kThreads = 128; // 16 games per CTA

__device__ __forceinline__ bool group_of(int G, int& g, int& lane, unsigned& mask) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  g = t / kLanes;
  lane = t % kLanes;
  mask = 0xFFu << ((threadIdx.x & 31) / kLanes * kLanes);
  return g < G;
}

// kNoise: root noise attached (azg_arena_set_root_noise); the launch picks the instance, so searches without noise run
// kernels that contain no mixing code
template <int kNoise>
__global__ void __launch_bounds__(kThreads) arena_select_kernel(AzgArenaView a, AzgState* leaf_states,
                                                                int32_t* leaf_mask) {
  int g, lane;
  unsigned mask;
  if (!group_of(a.G, g, lane, mask)) return;
  azg_select_game<kLanes, kNoise>(a, g, lane, mask, leaf_states, leaf_mask);
}

__global__ void __launch_bounds__(kThreads) arena_expand_backup_kernel(AzgArenaView a, const float* pi,
                                                                       const float* v) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g < a.G) azg_expand_backup_game(a, g, pi, v);
}

template <int kNoise>
__global__ void __launch_bounds__(kThreads) arena_select_compact_kernel(AzgArenaView a, AzgState* leaf_states,
                                                                        int32_t* leaf_mask, int32_t* leaf_game,
                                                                        int32_t* leaf_count) {
  int g, lane;
  unsigned mask;
  if (!group_of(a.G, g, lane, mask)) return;
  azg_select_game<kLanes, kNoise>(a, g, lane, mask, leaf_states, leaf_mask, leaf_game, leaf_count);
}

__global__ void __launch_bounds__(kThreads) arena_expand_backup_compact_kernel(AzgArenaView a, const float* pi,
                                                                               const float* v, const int32_t* leaf_game,
                                                                               const int32_t* leaf_count) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < *leaf_count) azg_expand_backup_game(a, leaf_game[i], pi, v, i);
}

__global__ void arena_reset_kernel(AzgArenaView a, const int32_t* ids, int count) {
  // one CTA per listed game: clear its hash slots and per-game scalars
  const int g = ids ? ids[blockIdx.x] : blockIdx.x;
  if (blockIdx.x >= count || g < 0 || g >= a.G) return;
  int32_t* hs = a.hslot + (size_t)g * a.hcap;
  for (int i = threadIdx.x; i < a.hcap; i += blockDim.x) hs[i] = 0;
  if (threadIdx.x == 0) {
    a.node_count[g] = 0;
    a.sims_left[g] = 0;
    a.pending[g] = -1;
    a.path_len[g] = 0;
    a.status[g] = 0;
  }
}

__global__ void arena_copy_kernel(AzgArenaView d, AzgArenaView s) {
  const int g = blockIdx.x;  // one CTA per game
  azg_copy_game_nodes(d, s, g, (int)threadIdx.x, (int)blockDim.x);
  __syncthreads();
  if (threadIdx.x == 0) azg_copy_game_finish(d, s, g);
}

__global__ void arena_set_roots_kernel(AzgArenaView a, const AzgState* s) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g < a.G) a.root[g] = s[g];
}

__global__ void arena_get_roots_kernel(AzgArenaView a, AzgState* s) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g < a.G) s[g] = a.root[g];
}

__global__ void arena_begin_kernel(AzgArenaView a, int n_sims) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g < a.G) a.sims_left[g] += n_sims;
}

__global__ void arena_root_noise_kernel(AzgArenaView a, uint64_t seed, const uint64_t* ids, double alpha, double* eta) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;  // one thread per game, actions in ascending order
  if (g < a.G) azg_root_noise_game(a, g, seed, ids[g], alpha, eta + (size_t)g * a.A);
}

__global__ void philox_kernel(uint64_t seed, const uint64_t* counters, int64_t n, uint64_t* words) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t c[4] = {counters[4 * i], counters[4 * i + 1], counters[4 * i + 2], counters[4 * i + 3]};
  azg_philox4x64_10(c, seed, 0);
  for (int j = 0; j < 4; ++j) words[4 * i + j] = c[j];
}

__global__ void arena_root_stats_kernel(AzgArenaView a, int32_t* N, double* Q, int8_t* qtag) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g < a.G) azg_root_stats_game(a, g, N, Q, qtag);
}

__global__ void arena_advance_kernel(AzgArenaView a, const int32_t* actions, double* ended, int8_t* ended_tag) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g < a.G) azg_advance_game(a, g, actions[g], ended, ended_tag);
}

__global__ void arena_status_kernel(AzgArenaView a, int32_t* status) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g < a.G) status[g] = a.status[g];
}

__global__ void rules_eval_kernel(AzgRules r, const AzgState* states, int64_t B, uint32_t* valids, double* ended,
                                  int8_t* ended_tag, AzgState* next) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  const AzgState s = states[i];
  const uint32_t m = azg_valids(r, s);
  const AzgVal e = azg_ended(r, s);
  valids[i] = m;
  ended[i] = e.d;
  ended_tag[i] = (int8_t)e.tag;
  for (int a = 0; a < r.A; ++a) {
    AzgState o;
    o.mine = 0;
    o.theirs = 0;
    if ((m >> a) & 1u) o = azg_next(r, s, a);
    next[i * r.A + a] = o;
  }
}

// Rollout leaf values: `tpr` threads per leaf (the power of two >= playouts, at most kRolloutThreads), one playout per
// thread and round, kRolloutThreads / tpr leaves per CTA.  Outcomes are summed as integers (warp shuffles, then one
// shared-memory atomic per warp and leaf), so v does not depend on the order of the reduction.
constexpr int kRolloutThreads = 256;

__global__ void __launch_bounds__(kRolloutThreads) rollout_eval_kernel(AzgRules r, const AzgState* states,
                                                                       const int32_t* games, int64_t rows,
                                                                       const int32_t* count, int playouts, int tpr,
                                                                       uint64_t seed, float* pi, float* v) {
  const int rpb = kRolloutThreads / tpr;
  const int64_t first = (int64_t)blockIdx.x * rpb;
  const int64_t live = count ? min((int64_t)*count, rows) : rows;
  if (first >= live) return;  // the whole CTA is past the leaf count
  __shared__ int sums[kRolloutThreads];
  const int slot = threadIdx.x / tpr, lane = threadIdx.x % tpr;
  const int64_t row = first + slot;
  const bool on = row < live;
  if (lane == 0) sums[slot] = 0;
  __syncthreads();
  AzgState s;
  s.mine = s.theirs = 0;
  int acc = 0;
  if (on) {
    s = states[row];
    const uint32_t g = games ? (uint32_t)games[row] : (uint32_t)row;
    for (int p = lane; p < playouts; p += tpr) acc += azg_rollout_outcome(r, s, seed, g, (uint32_t)p);
  }
  for (int off = min(tpr, 32) / 2; off > 0; off >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, off);
  if (on && (lane & 31) == 0) atomicAdd(&sums[slot], acc);
  __syncthreads();
  if (!on) return;
  if (lane == 0) v[row] = __fdiv_rn((float)sums[slot], (float)playouts);
  azg_rollout_policy(r, s, pi + row * r.A, lane, tpr);
}

inline int grid_for(int64_t n, int threads) { return (int)((n + threads - 1) / threads); }

}  // namespace

extern "C" {

size_t azg_arena_bytes(int game, int n, int n_games, int capacity_nodes, int max_depth) {
  AzgArenaView v;
  memset(&v, 0, sizeof(v));
  uint8_t blank_map[64];
  memset(blank_map, 'F', sizeof(blank_map));  // the map does not affect sizes
  if (azg_rules_init(&v.rules, game, n, blank_map)) return 0;
  if (n_games <= 0 || capacity_nodes <= 0 || max_depth <= 0) return 0;
  v.G = n_games;
  v.cap = capacity_nodes;
  v.hcap = azg_hash_capacity(capacity_nodes);
  v.max_depth = max_depth;
  v.A = v.rules.A;
  return azg_arena_carve(&v, nullptr);
}

int azg_arena_create(azg_arena** out, int game, int n, int n_games, int capacity_nodes, int max_depth,
                     double cpuct, void* device_mem, size_t device_bytes, const uint8_t* fl_map,
                     azg_stream stream) {
  AZG_REQUIRE(out != nullptr && device_mem != nullptr, "azg_arena_create: null pointer");
  AZG_REQUIRE(n_games > 0 && capacity_nodes > 0 && max_depth > 0 && max_depth <= 4096, "azg_arena_create: bad sizes");
  azg_arena* a = new (std::nothrow) azg_arena();
  AZG_REQUIRE(a != nullptr, "azg_arena_create: out of host memory");
  memset(a, 0, sizeof(*a));
  if (azg_rules_init(&a->view.rules, game, n, fl_map)) {
    delete a;
    azg_set_error("azg_arena_create: unsupported game %d / board size %d (Connect4, FrozenLake 2..8; TicTacToe 2..5: at most 32 actions)%s", game, n,
                  game == AZG_GAME_FROZENLAKE && !fl_map ? " / missing map" : "");
    return AZG_ERR_INVALID;
  }
  a->game = game;
  a->n = n;
  AzgArenaView& v = a->view;
  v.G = n_games;
  v.cap = capacity_nodes;
  v.hcap = azg_hash_capacity(capacity_nodes);
  v.max_depth = max_depth;
  v.A = v.rules.A;
  v.two_player = (game != AZG_GAME_FROZENLAKE);  // is_two_player, Connect4Game.py:121 / FrozenLakeGame.py:18
  v.cpuct = cpuct;
  v.p_f32 = (game == AZG_GAME_FROZENLAKE);
  const size_t need = azg_arena_carve(&v, (char*)device_mem);
  if (need > device_bytes) {
    delete a;
    azg_set_error("azg_arena_create: need %zu bytes of device memory, got %zu", need, device_bytes);
    return AZG_ERR_INVALID;
  }
  *out = a;
  // roots start as the all-zero state (empty board / FrozenLake start square) until azg_arena_set_roots; the caller's
  // memory may be recycled
  AZG_CUDA_CHECK(cudaMemsetAsync(v.root, 0, (size_t)n_games * sizeof(AzgState), (cudaStream_t)stream));
  return azg_arena_reset(a, nullptr, n_games, stream);
}

int azg_arena_destroy(azg_arena* a) {
  delete a;
  return AZG_OK;
}

int azg_arena_action_size(const azg_arena* a) { return a ? a->view.A : -1; }

int azg_arena_reset(azg_arena* a, const int32_t* game_ids, int count, azg_stream stream) {
  AZG_REQUIRE(a != nullptr, "azg_arena_reset: null arena");
  if (!game_ids) count = a->view.G;
  if (count <= 0) return AZG_OK;
  arena_reset_kernel<<<count, 256, 0, (cudaStream_t)stream>>>(a->view, game_ids, count);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

int azg_arena_copy_from(azg_arena* dst, const azg_arena* src, azg_stream stream) {
  AZG_REQUIRE(dst && src && dst != src, "azg_arena_copy_from: bad arenas");
  const AzgArenaView &d = dst->view, &s = src->view;
  AZG_REQUIRE(dst->game == src->game && dst->n == src->n && d.G == s.G && d.A == s.A && d.max_depth >= s.max_depth && d.cap >= s.cap,
              "azg_arena_copy_from: the destination must be the same game with at least the source's capacity (%d < %d?)", d.cap, s.cap);
  arena_copy_kernel<<<d.G, 256, 0, (cudaStream_t)stream>>>(d, s);
  AZG_LAUNCH_CHECK();
  dst->view.semantics = s.semantics;  // a grown table continues the search it holds
  dst->view.noise = s.noise;
  dst->view.noise_eps = s.noise_eps;
  return AZG_OK;
}

int azg_arena_set_semantics(azg_arena* a, int semantics) {
  AZG_REQUIRE(a != nullptr, "azg_arena_set_semantics: null arena");
  return azg_view_set_semantics(&a->view, semantics);
}

int azg_arena_set_root_noise(azg_arena* a, const double* eta, double eps) {
  AZG_REQUIRE(a != nullptr, "azg_arena_set_root_noise: null arena");
  return azg_view_set_root_noise(&a->view, eta, eps);
}

int azg_arena_draw_root_noise(azg_arena* a, uint64_t seed, const uint64_t* ids, double alpha, double* eta, azg_stream stream) {
  AZG_REQUIRE(a != nullptr, "azg_arena_draw_root_noise: null arena");
  AZG_REQUIRE(alpha > 0.0 && alpha < INFINITY, "azg_arena_draw_root_noise: alpha must be finite and > 0, got %g", alpha);
  AZG_REQUIRE(ids && eta, "azg_arena_draw_root_noise: null pointer");
  arena_root_noise_kernel<<<grid_for(a->view.G, 128), 128, 0, (cudaStream_t)stream>>>(a->view, seed, ids, alpha, eta);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

int azg_philox4x64(uint64_t seed, const uint64_t* counters, int64_t n, uint64_t* words, azg_stream stream) {
  AZG_REQUIRE(n >= 0 && (n == 0 || (counters && words)), "azg_philox4x64: bad argument");
  if (n == 0) return AZG_OK;
  philox_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(seed, counters, n, words);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

int azg_rollout_eval(int game, int n, const uint64_t* states, const int32_t* games, int64_t rows, const int32_t* count,
                     int playouts, uint64_t seed, float* pi, float* v, azg_stream stream) {
  AzgRules r;
  const int rc = azg_rollout_setup(&r, game, n, playouts);
  if (rc != AZG_OK) return rc;
  AZG_REQUIRE(rows >= 0 && rows <= 0x7FFFFFFF, "azg_rollout_eval: rows must lie in [0, 2^31), got %lld", (long long)rows);
  AZG_REQUIRE(rows == 0 || (states && pi && v), "azg_rollout_eval: null pointer");
  if (rows == 0) return AZG_OK;
  int tpr = 1;
  while (tpr < playouts && tpr < kRolloutThreads) tpr <<= 1;
  rollout_eval_kernel<<<grid_for(rows, kRolloutThreads / tpr), kRolloutThreads, 0, (cudaStream_t)stream>>>(
      r, (const AzgState*)states, games, rows, count, playouts, tpr, seed, pi, v);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

int azg_arena_set_roots(azg_arena* a, const uint64_t* states, azg_stream stream) {
  AZG_REQUIRE(a && states, "azg_arena_set_roots: null pointer");
  arena_set_roots_kernel<<<grid_for(a->view.G, 256), 256, 0, (cudaStream_t)stream>>>(a->view, (const AzgState*)states);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

int azg_arena_get_roots(azg_arena* a, uint64_t* states, azg_stream stream) {
  AZG_REQUIRE(a && states, "azg_arena_get_roots: null pointer");
  arena_get_roots_kernel<<<grid_for(a->view.G, 256), 256, 0, (cudaStream_t)stream>>>(a->view, (AzgState*)states);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

int azg_arena_begin(azg_arena* a, int n_sims, azg_stream stream) {
  AZG_REQUIRE(a && n_sims >= 0, "azg_arena_begin: bad argument");
  arena_begin_kernel<<<grid_for(a->view.G, 256), 256, 0, (cudaStream_t)stream>>>(a->view, n_sims);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

int azg_arena_select(azg_arena* a, uint64_t* leaf_states, int32_t* leaf_mask, azg_stream stream) {
  AZG_REQUIRE(a && leaf_states && leaf_mask, "azg_arena_select: null pointer");
  const int64_t threads = (int64_t)a->view.G * kLanes;
  auto kernel = a->view.noise ? arena_select_kernel<1> : arena_select_kernel<0>;
  kernel<<<grid_for(threads, kThreads), kThreads, 0, (cudaStream_t)stream>>>(a->view, (AzgState*)leaf_states, leaf_mask);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

int azg_arena_select_compact(azg_arena* a, uint64_t* leaf_states, int32_t* leaf_mask, int32_t* leaf_game,
                             int32_t* leaf_count, azg_stream stream) {
  AZG_REQUIRE(a && leaf_states && leaf_mask && leaf_game && leaf_count, "azg_arena_select_compact: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  AZG_CUDA_CHECK(cudaMemsetAsync(leaf_count, 0, sizeof(int32_t), st));
  const int64_t threads = (int64_t)a->view.G * kLanes;
  auto kernel = a->view.noise ? arena_select_compact_kernel<1> : arena_select_compact_kernel<0>;
  kernel<<<grid_for(threads, kThreads), kThreads, 0, st>>>(a->view, (AzgState*)leaf_states, leaf_mask, leaf_game, leaf_count);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

int azg_arena_expand_backup_compact(azg_arena* a, const float* pi, const float* v, const int32_t* leaf_game,
                                    const int32_t* leaf_count, azg_stream stream) {
  AZG_REQUIRE(a && pi && v && leaf_game && leaf_count, "azg_arena_expand_backup_compact: null pointer");
  arena_expand_backup_compact_kernel<<<grid_for(a->view.G, kThreads), kThreads, 0, (cudaStream_t)stream>>>(
      a->view, pi, v, leaf_game, leaf_count);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

int azg_arena_expand_backup(azg_arena* a, const float* pi, const float* v, azg_stream stream) {
  AZG_REQUIRE(a && pi && v, "azg_arena_expand_backup: null pointer");
  arena_expand_backup_kernel<<<grid_for(a->view.G, kThreads), kThreads, 0, (cudaStream_t)stream>>>(a->view, pi, v);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

int azg_arena_root_stats(azg_arena* a, int32_t* N, double* Q, int8_t* qtag, azg_stream stream) {
  AZG_REQUIRE(a && N && Q && qtag, "azg_arena_root_stats: null pointer");
  arena_root_stats_kernel<<<grid_for(a->view.G, 128), 128, 0, (cudaStream_t)stream>>>(a->view, N, Q, qtag);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

int azg_arena_advance(azg_arena* a, const int32_t* actions, double* ended, int8_t* ended_tag, azg_stream stream) {
  AZG_REQUIRE(a && actions && ended && ended_tag, "azg_arena_advance: null pointer");
  arena_advance_kernel<<<grid_for(a->view.G, 256), 256, 0, (cudaStream_t)stream>>>(a->view, actions, ended, ended_tag);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

int azg_arena_status(azg_arena* a, int32_t* status, azg_stream stream) {
  AZG_REQUIRE(a && status, "azg_arena_status: null pointer");
  arena_status_kernel<<<grid_for(a->view.G, 256), 256, 0, (cudaStream_t)stream>>>(a->view, status);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

int azg_arena_export(azg_arena* a, int g, int* n_nodes, uint64_t* keys, double* es, int8_t* es_tag, int32_t* ns,
                     uint32_t* valids, int8_t* ptag, double* P, double* Q, int8_t* qtag, int32_t* N, azg_stream stream) {
  AZG_REQUIRE(a && n_nodes, "azg_arena_export: null pointer");
  const AzgArenaView& v = a->view;
  AZG_REQUIRE(g >= 0 && g < v.G, "azg_arena_export: game index %d out of range", g);
  cudaStream_t st = (cudaStream_t)stream;
  int32_t count = 0;
  AZG_CUDA_CHECK(cudaMemcpyAsync(&count, v.node_count + g, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  AZG_CUDA_CHECK(cudaStreamSynchronize(st));
  *n_nodes = count;
  const size_t c = (size_t)count, node0 = (size_t)g * v.cap, A = v.A;
  if (c == 0) return AZG_OK;
#define AZG_COPY(dst, src, bytes) \
  if (dst) AZG_CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, st))
  AZG_COPY(keys, v.key + node0, c * sizeof(AzgState));
  AZG_COPY(es, v.es + node0, c * sizeof(double));
  AZG_COPY(es_tag, v.es_tag + node0, c);
  AZG_COPY(ns, v.ns + node0, c * sizeof(int32_t));
  AZG_COPY(valids, v.valids + node0, c * sizeof(uint32_t));
  AZG_COPY(ptag, v.ptag + node0, c);
  AZG_COPY(P, v.P + node0 * A, c * A * sizeof(double));
  AZG_COPY(Q, v.Q + node0 * A, c * A * sizeof(double));
  AZG_COPY(qtag, v.qtag + node0 * A, c * A);
  AZG_COPY(N, v.N + node0 * A, c * A * sizeof(int32_t));
#undef AZG_COPY
  return AZG_OK;
}

int azg_rules_eval(int game, int n, const uint8_t* fl_map_host, const uint64_t* states, int64_t B, uint32_t* valids,
                   double* ended, int8_t* ended_tag, uint64_t* next, azg_stream stream) {
  AzgRules r;
  AZG_REQUIRE(azg_rules_init(&r, game, n, fl_map_host) == 0, "azg_rules_eval: unsupported game %d / size %d", game, n);
  AZG_REQUIRE(states && valids && ended && ended_tag && next, "azg_rules_eval: null pointer");
  if (B <= 0) return AZG_OK;
  rules_eval_kernel<<<grid_for(B, 256), 256, 0, (cudaStream_t)stream>>>(r, (const AzgState*)states, B, valids, ended,
                                                                         ended_tag, (AzgState*)next);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

}  // extern "C"
