// azg_arena_core.cuh -- per-game search logic of the arena, host/device.
//
// One *group* of W lanes owns one game (W = 8 on the GPU: four games per warp; W = 1 in the
// host check build of tests/hostcheck, where the same source runs sequentially).  All lanes of
// a group hold identical scalar state, so control flow is uniform inside a group; lane 0 does
// the table writes, every lane scores its own actions for the PUCT arg-max.
//
// What is reproduced, bit for bit (SURVEY.md section 0):
//   MCTS.search      MCTS.py:151-240   descend / leaf / select / backup
//   value types      NEP 50: float64 priors and PUCT score, float32 running-mean Q once a
//                    network value has joined, Python int/float before that
//   tie-breaking     strict '>' in ascending action order -> lowest index wins (MCTS.py:206-216)
// No FMA contraction anywhere in this file: every rounding is spelled out.
#pragma once
#include "azg_rules.cuh"

// ---- exactly-rounded arithmetic ---------------------------------------------------------
#if defined(__CUDA_ARCH__)
AZG_HD double azg_dmul(double a, double b) { return __dmul_rn(a, b); }
AZG_HD double azg_dadd(double a, double b) { return __dadd_rn(a, b); }
AZG_HD double azg_ddiv(double a, double b) { return __ddiv_rn(a, b); }
AZG_HD double azg_dsqrt(double a) { return __dsqrt_rn(a); }
AZG_HD float azg_fmul(float a, float b) { return __fmul_rn(a, b); }
AZG_HD float azg_fadd(float a, float b) { return __fadd_rn(a, b); }
AZG_HD float azg_fdiv(float a, float b) { return __fdiv_rn(a, b); }
#else
#include <math.h>
// host check build: compiled with -ffp-contract=off -O1 (see tests/hostcheck/build.py)
static inline double azg_dmul(double a, double b) { volatile double r = a * b; return r; }
static inline double azg_dadd(double a, double b) { volatile double r = a + b; return r; }
static inline double azg_ddiv(double a, double b) { volatile double r = a / b; return r; }
static inline double azg_dsqrt(double a) { volatile double r = sqrt(a); return r; }
static inline float azg_fmul(float a, float b) { volatile float r = a * b; return r; }
static inline float azg_fadd(float a, float b) { volatile float r = a + b; return r; }
static inline float azg_fdiv(float a, float b) { volatile float r = a / b; return r; }
#endif

#define AZG_MAX_A 65  // TicTacToe 8x8 + pass

struct AzgArenaView {
  AzgRules rules;
  int G, cap, hcap, max_depth, A, two_player;
  int semantics;  // AZG_SEARCH_REFERENCE / AZG_SEARCH_ALPHAZERO, read by azg_backup only
  int p_f32;  // valid masks are int8 (FrozenLakeGame.py:125): Ps and the PUCT score stay float32 (NEP 50)
  double cpuct;
  // Dirichlet root noise (azg_arena_set_root_noise): [G, A] float64, caller-owned, NULL = off.  Mixed into the prior
  // of the depth-0 node only, as (1 - noise_eps) P + noise_eps eta; the stored P is never modified.
  const double* noise;
  double noise_eps;
  // per game
  AzgState* root;       // [G]
  int32_t* sims_left;   // [G]
  int32_t* node_count;  // [G]
  int32_t* pending;     // [G] node index awaiting a prediction, -1 = none
  int32_t* path_len;    // [G]
  int32_t* path_node;   // [G, max_depth]
  int8_t* path_act;     // [G, max_depth]
  int32_t* status;      // [G] sticky error code
  int32_t* hslot;       // [G, hcap] node index + 1, 0 = empty
  // per node [G, cap]
  AzgState* key;
  double* es;       // Es value (MCTS.py:154-157); es_tag == AZG_TAG_NONE: not ended
  int8_t* es_tag;
  int32_t* ns;      // Ns; -1 = not expanded yet (s not in Ps)
  uint32_t* valids; // Vs bit mask
  int8_t* ptag;     // dtype of Ps[s]: 0 = float64, 1 = float32 (stored widened)
  // per edge [G, cap, A]
  double* P;    // Ps, float64
  double* Q;    // Qsa (float32 values stored widened, exact)
  int8_t* qtag; // AZG_TAG_NONE = (s,a) not in Qsa
  int32_t* N;   // Nsa
};

// ---- group helpers ----------------------------------------------------------------------
template <int W>
AZG_HD void azg_group_sync(unsigned mask) {
#if defined(__CUDA_ARCH__)
  if (W > 1) __syncwarp(mask);
#else
  (void)mask;
#endif
}

AZG_HD uint64_t azg_hash(AzgState s) {
  uint64_t h = s.mine * 0x9E3779B97F4A7C15ull ^ (s.theirs + 0x7F4A7C15F39CC060ull) * 0xC2B2AE3D27D4EB4Full;
  h ^= h >> 29;
  h *= 0xBF58476D1CE4E5B9ull;
  h ^= h >> 32;
  return h;
}

// node index of state s in game g's table, or -1
AZG_HD int azg_lookup(const AzgArenaView& a, int g, AzgState s) {
  const int32_t* hs = a.hslot + (size_t)g * a.hcap;
  const AzgState* keys = a.key + (size_t)g * a.cap;
  uint32_t slot = (uint32_t)azg_hash(s) & (uint32_t)(a.hcap - 1);
  for (int probe = 0; probe < a.hcap; ++probe) {
    const int32_t v = hs[slot];
    if (v == 0) return -1;
    const AzgState k = keys[v - 1];
    if (k.mine == s.mine && k.theirs == s.theirs) return v - 1;
    slot = (slot + 1) & (uint32_t)(a.hcap - 1);
  }
  return -1;
}

// lane 0 only: claim a new node for s (caller checked capacity); returns its index
AZG_HD int azg_insert(const AzgArenaView& a, int g, AzgState s, int idx) {
  int32_t* hs = a.hslot + (size_t)g * a.hcap;
  uint32_t slot = (uint32_t)azg_hash(s) & (uint32_t)(a.hcap - 1);
  while (hs[slot] != 0) slot = (slot + 1) & (uint32_t)(a.hcap - 1);
  hs[slot] = idx + 1;
  const size_t node = (size_t)g * a.cap + idx;
  a.key[node] = s;
  a.ns[node] = -1;
  a.valids[node] = 0;
  a.es[node] = 0.0;
  a.es_tag[node] = AZG_TAG_NONE;
  a.ptag[node] = 0;
  const size_t e0 = node * a.A;
  for (int i = 0; i < a.A; ++i) {
    a.qtag[e0 + i] = AZG_TAG_NONE;
    a.N[e0 + i] = 0;
    a.Q[e0 + i] = 0.0;
    a.P[e0 + i] = 0.0;
  }
  return idx;
}

AZG_HD AzgVal azg_neg(AzgVal v) {
  // -v: Python int 0 stays +0 (there is no negative int zero); floats flip the sign bit
  v.d = (v.tag == AZG_TAG_PYINT) ? (0.0 - v.d) : -v.d;
  return v;
}

// Qsa <- (Nsa*Qsa + v)/(Nsa+1), MCTS.py:229, with NEP 50 promotion (SURVEY section 0.3)
AZG_HD AzgVal azg_q_update(int n, AzgVal q, AzgVal v) {
  AzgVal o;
  if (q.tag != AZG_TAG_F32 && v.tag != AZG_TAG_F32) {
    // all-Python arithmetic: int*int, int+int exact; true division -> float (binary64)
    const double nq = azg_dmul((double)n, q.d);
    const double s = azg_dadd(nq, v.d);
    o.d = azg_ddiv(s, (double)(n + 1));
    o.tag = AZG_TAG_PYFLOAT;
    return o;
  }
  float nq;
  if (q.tag == AZG_TAG_F32) nq = azg_fmul((float)n, (float)q.d);  // int * float32 -> float32
  else nq = (float)azg_dmul((double)n, q.d);                       // Python product, then weak-cast to float32
  const float vv = (float)v.d;                                     // float32 as is; Python scalar weak-cast
  const float s = azg_fadd(nq, vv);
  o.d = (double)azg_fdiv(s, (float)(n + 1));
  o.tag = AZG_TAG_F32;
  return o;
}

// numpy.sum of a contiguous float64 vector (pairwise_sum in loops_utils.h.src: <8 sequential,
// <=128: eight running lanes combined as a tree, then the tail)
AZG_HD double azg_np_sum(const double* x, int n) {
  if (n < 8) {
    double r = -0.0;
    for (int i = 0; i < n; ++i) r = azg_dadd(r, x[i]);
    return azg_dadd(0.0, r);
  }
  double r[8];
  for (int j = 0; j < 8; ++j) r[j] = x[j];
  int i = 8;
  for (; i < n - (n % 8); i += 8)
    for (int j = 0; j < 8; ++j) r[j] = azg_dadd(r[j], x[i + j]);
  double res = azg_dadd(azg_dadd(azg_dadd(r[0], r[1]), azg_dadd(r[2], r[3])),
                        azg_dadd(azg_dadd(r[4], r[5]), azg_dadd(r[6], r[7])));
  for (; i < n; ++i) res = azg_dadd(res, x[i]);
  return azg_dadd(0.0, res);
}

// numpy.sum of a contiguous float32 vector: same blocking, float32 accumulators
AZG_HD float azg_np_sum_f32(const float* x, int n) {
  if (n < 8) {
    float r = -0.0f;
    for (int i = 0; i < n; ++i) r = azg_fadd(r, x[i]);
    return azg_fadd(0.0f, r);
  }
  float r[8];
  for (int j = 0; j < 8; ++j) r[j] = x[j];
  int i = 8;
  for (; i < n - (n % 8); i += 8)
    for (int j = 0; j < 8; ++j) r[j] = azg_fadd(r[j], x[i + j]);
  float res = azg_fadd(azg_fadd(azg_fadd(r[0], r[1]), azg_fadd(r[2], r[3])),
                       azg_fadd(azg_fadd(r[4], r[5]), azg_fadd(r[6], r[7])));
  for (; i < n; ++i) res = azg_fadd(res, x[i]);
  return azg_fadd(0.0f, res);
}

// lane 0: walk the recorded path back up, MCTS.py:228-240.  Two-player games negate v once per level after the edge
// update.  In the AlphaZero semantics the negation comes before the update instead (Q from the point of view of the
// player who picks the edge), which stores the same sequence as this walk started from -v.  The mode is a uniform
// branch rather than a template parameter: it is the same for all games of a launch, costs one negation per backup,
// and keeps one set of arena kernels for both modes.
AZG_HD void azg_backup(const AzgArenaView& a, int g, int depth, AzgVal v) {
  const int32_t* pn = a.path_node + (size_t)g * a.max_depth;
  const int8_t* pa = a.path_act + (size_t)g * a.max_depth;
  if (a.two_player && a.semantics == AZG_SEARCH_ALPHAZERO) v = azg_neg(v);
  for (int i = depth - 1; i >= 0; --i) {
    const size_t node = (size_t)g * a.cap + pn[i];
    const size_t e = node * a.A + pa[i];
    if (a.qtag[e] != AZG_TAG_NONE) {
      AzgVal q;
      q.d = a.Q[e];
      q.tag = a.qtag[e];
      const AzgVal nq = azg_q_update(a.N[e], q, v);
      a.Q[e] = nq.d;
      a.qtag[e] = (int8_t)nq.tag;
      a.N[e] += 1;
    } else {
      a.Q[e] = v.d;
      a.qtag[e] = (int8_t)v.tag;
      a.N[e] = 1;
    }
    a.ns[node] += 1;
    if (a.two_player) v = azg_neg(v);
  }
}

// PUCT arg-max over the valid actions of an expanded node, MCTS.py:202-216.
// noise_g >= 0 (root of game noise_g, noise on): the prior in both formulas is (1 - eps) P + eps eta[noise_g, act],
// rounded step by step; the stored P is left as it is.
template <int W>
AZG_HD int azg_select_action(const AzgArenaView& a, size_t node, int lane, unsigned mask, int noise_g = -1) {
  const uint32_t valids = a.valids[node];
  const double ns = (double)a.ns[node];
  const double sq_visited = azg_dsqrt(ns);                      // math.sqrt(Ns)
  const double sq_fresh = azg_dsqrt(azg_dadd(ns, 1e-8));        // math.sqrt(Ns + EPS)
  double best_u = -INFINITY;
  int best_a = -1;
  const bool pf32 = a.ptag[node] != 0;
  for (int act = lane; act < a.A; act += W) {
    if ((valids >> act) & 1u) {
      const size_t e = node * a.A + act;
      double u;
      if (!pf32) {  // float64 prior: every factor promotes to float64
        double p = a.P[e];
        if (noise_g >= 0)
          p = azg_dadd(azg_dmul(azg_dadd(1.0, -a.noise_eps), p), azg_dmul(a.noise_eps, a.noise[(size_t)noise_g * a.A + act]));
        const double cp = azg_dmul(a.cpuct, p);
        if (a.qtag[e] != AZG_TAG_NONE)
          u = azg_dadd(a.Q[e], azg_ddiv(azg_dmul(cp, sq_visited), (double)(1 + a.N[e])));
        else
          u = azg_dmul(cp, sq_fresh);
      } else {  // float32 prior: Python scalars are weak, the whole score stays float32
        const float cp = azg_fmul((float)a.cpuct, (float)a.P[e]);
        if (a.qtag[e] != AZG_TAG_NONE) {
          const float ex = azg_fdiv(azg_fmul(cp, (float)sq_visited), (float)(1 + a.N[e]));
          u = (double)azg_fadd((float)a.Q[e], ex);
        } else {
          u = (double)azg_fmul(cp, (float)sq_fresh);
        }
      }
      if (u > best_u) {
        best_u = u;
        best_a = act;
      }
    }
  }
#if defined(__CUDA_ARCH__)
  if (W > 1) {  // warp arg-max: larger score wins, equal scores -> lower action index
#pragma unroll
    for (int off = W / 2; off > 0; off >>= 1) {
      const double ou = __shfl_xor_sync(mask, best_u, off, W);
      const int oa = __shfl_xor_sync(mask, best_a, off, W);
      if (oa >= 0 && (best_a < 0 || ou > best_u || (ou == best_u && oa < best_a))) {
        best_u = ou;
        best_a = oa;
      }
    }
  }
#else
  (void)mask;
#endif
  return best_a;
}

// MCTS.search descend phase for game g; runs searches until one needs a prediction or the
// simulation budget is spent.
// leaf_game/leaf_count (optional): compacted output -- games that wait for a prediction claim consecutive
// slots; leaf_states then holds their positions densely and leaf_game the owning game of each slot.
// kNoise: 0 / 1 = root noise off / on, fixed at compile time (the GPU launches pick the kernel, so noise-off kernels carry
// none of the mixing code); -1 = read a.noise at run time (the host check build).
template <int W, int kNoise = -1>
AZG_HD void azg_select_game(const AzgArenaView& a, int g, int lane, unsigned mask, AzgState* leaf_states,
                            int32_t* leaf_mask, int32_t* leaf_game = nullptr, int32_t* leaf_count = nullptr) {
  const bool noisy = kNoise < 0 ? a.noise != nullptr : kNoise == 1;
  int sims = a.sims_left[g];
  int count = a.node_count[g];
  const bool waiting = a.pending[g] >= 0;
  int emit = waiting ? 1 : 0;
  AzgState emit_state = a.root[g];
  if (waiting) emit_state = a.key[(size_t)g * a.cap + a.pending[g]];
  bool failed = a.status[g] != 0;
  while (!waiting && !failed && sims > 0) {
    AzgState s = a.root[g];
    int depth = 0;
    AzgVal v;
    v.d = 0.0;
    v.tag = AZG_TAG_PYINT;
    bool need_eval = false;
    while (true) {
      if (depth >= a.max_depth) break;  // cycle policy: return 0 (DESIGN.md)
      int idx = azg_lookup(a, g, s);
      bool fresh = false;
      if (idx < 0) {
        if (count >= a.cap) {
          failed = true;
          if (lane == 0) a.status[g] = AZG_ERR_CAPACITY;
          break;
        }
        idx = count++;
        fresh = true;
        const AzgVal e = azg_ended(a.rules, s);  // Es[s] = getGameEnded(board, 1), MCTS.py:154-155
        if (lane == 0) {
          azg_insert(a, g, s, idx);
          const size_t node = (size_t)g * a.cap + idx;
          a.es[node] = e.d;
          a.es_tag[node] = (int8_t)e.tag;
        }
        azg_group_sync<W>(mask);
      }
      const size_t node = (size_t)g * a.cap + idx;
      const int etag = a.es_tag[node];
      if (etag != AZG_TAG_NONE) {  // terminal: return Es[s], MCTS.py:156-157
        v.d = a.es[node];
        v.tag = etag;
        break;
      }
      if (fresh || a.ns[node] < 0) {  // s not in Ps: leaf, MCTS.py:162-193 continues in expand_backup
        if (lane == 0) {
          a.valids[node] = azg_valids(a.rules, s);
          a.pending[g] = idx;
          a.path_len[g] = depth;
        }
        emit_state = s;
        need_eval = true;
        break;
      }
      const int act = azg_select_action<W>(a, node, lane, mask, (noisy && depth == 0) ? g : -1);  // noise: root only
      if (act < 0) break;  // no action: return 0, MCTS.py:218-219
      if (lane == 0) {
        a.path_node[(size_t)g * a.max_depth + depth] = idx;
        a.path_act[(size_t)g * a.max_depth + depth] = (int8_t)act;
      }
      ++depth;
      s = azg_next(a.rules, s, act);  // MCTS.py:221-224
    }
    if (failed) break;
    if (need_eval) {
      emit = 1;
      break;
    }
    if (lane == 0) azg_backup(a, g, depth, v);
    --sims;
    azg_group_sync<W>(mask);
  }
  if (lane == 0) {
    a.sims_left[g] = sims;
    a.node_count[g] = count;
    leaf_mask[g] = emit;
    if (leaf_count) {
      if (emit) {
#if defined(__CUDA_ARCH__)
        const int slot = atomicAdd(leaf_count, 1);
#else
        const int slot = (*leaf_count)++;
#endif
        leaf_states[slot] = emit_state;
        leaf_game[slot] = g;
      }
    } else if (emit) {
      leaf_states[g] = emit_state;
    }
  }
}

// MCTS.search leaf phase + backup for a game whose prediction arrived (lane 0 only)
// `row` = row of pi / vpred that holds game g's prediction (g itself, or its compact slot)
AZG_HD void azg_expand_backup_game(const AzgArenaView& a, int g, const float* pi, const float* vpred, int64_t row = -1) {
  if (row < 0) row = g;
  const int idx = a.pending[g];
  if (idx < 0) return;
  const size_t node = (size_t)g * a.cap + idx;
  const uint32_t valids = a.valids[node];
  double ps[AZG_MAX_A];
  const int A = a.A;
  int ptag = 0;
  if (!a.p_f32) {
    for (int i = 0; i < A; ++i)  // Ps = pi * valids: float32 * int64 -> float64, MCTS.py:180
      ps[i] = azg_dmul((double)pi[(size_t)row * A + i], (double)((valids >> i) & 1u));
    const double tot = azg_np_sum(ps, A);
    if (tot > 0) {
      for (int i = 0; i < A; ++i) ps[i] = azg_ddiv(ps[i], tot);  // MCTS.py:182-183
    } else {
      const double k = (double)azg_popc64((uint64_t)valids);      // valids / np.sum(valids), :186
      for (int i = 0; i < A; ++i) ps[i] = azg_ddiv((double)((valids >> i) & 1u), k);
    }
  } else {
    float pf[AZG_MAX_A];
    for (int i = 0; i < A; ++i)  // float32 * int8 -> float32
      pf[i] = azg_fmul(pi[(size_t)row * A + i], (float)((valids >> i) & 1u));
    const float tot = azg_np_sum_f32(pf, A);
    if (tot > 0) {
      for (int i = 0; i < A; ++i) ps[i] = (double)azg_fdiv(pf[i], tot);
      ptag = 1;
    } else {  // int8 array / int64 sum -> float64
      const double k = (double)azg_popc64((uint64_t)valids);
      for (int i = 0; i < A; ++i) ps[i] = azg_ddiv((double)((valids >> i) & 1u), k);
    }
  }
  a.ptag[node] = (int8_t)ptag;
  for (int i = 0; i < A; ++i) a.P[node * A + i] = ps[i];
  a.ns[node] = 0;  // MCTS.py:188
  AzgVal v;
  v.d = (double)vpred[row];  // numpy.float32 from the net, MCTS.py:190-193
  v.tag = AZG_TAG_F32;
  azg_backup(a, g, a.path_len[g], v);
  a.pending[g] = -1;
  a.sims_left[g] -= 1;
}

AZG_HD void azg_root_stats_game(const AzgArenaView& a, int g, int32_t* N, double* Q, int8_t* qtag) {
  const int idx = azg_lookup(a, g, a.root[g]);
  for (int i = 0; i < a.A; ++i) {
    const size_t o = (size_t)g * a.A + i;
    if (idx < 0) {
      N[o] = 0; Q[o] = 0.0; qtag[o] = AZG_TAG_NONE;
    } else {
      const size_t e = ((size_t)g * a.cap + idx) * a.A + i;
      N[o] = a.N[e]; Q[o] = a.Q[e]; qtag[o] = a.qtag[e];
    }
  }
}

AZG_HD void azg_advance_game(const AzgArenaView& a, int g, int action, double* ended, int8_t* ended_tag) {
  if (action >= 0) a.root[g] = azg_next(a.rules, a.root[g], action);
  const AzgVal e = azg_ended(a.rules, a.root[g]);
  ended[g] = e.d;
  ended_tag[g] = (int8_t)e.tag;
}

// ---- search semantics: validated once, shared by the library and the host check build ---------------------------
static inline int azg_view_set_semantics(AzgArenaView* v, int semantics) {
  AZG_REQUIRE(semantics == AZG_SEARCH_REFERENCE || semantics == AZG_SEARCH_ALPHAZERO,
              "azg_arena_set_semantics: unknown search semantics %d (0 = reference, 1 = alphazero)", semantics);
  v->semantics = semantics;
  return AZG_OK;
}
// ---- Dirichlet root noise ----------------------------------------------------------------------------------------
// Attach (eta != NULL) or detach the [G, A] noise buffer.  eps must lie in [0, 1] (NaN is refused); single-player arenas
// (FrozenLake: float32 priors, searches that cycle back to the root) take no noise.
static inline int azg_view_set_root_noise(AzgArenaView* v, const double* eta, double eps) {
  AZG_REQUIRE(eps >= 0.0 && eps <= 1.0, "azg_arena_set_root_noise: eps must lie in [0, 1], got %g", eps);
  AZG_REQUIRE(eta == nullptr || (v->two_player && !v->p_f32),
              "azg_arena_set_root_noise: root noise needs a two-player game (Connect4, TicTacToe)");
  v->noise = eta;
  v->noise_eps = eta ? eps : 0.0;
  return AZG_OK;
}

// Counter-based generator: Philox4x64-10 (Salmon et al., SC'11), the generator of numpy.random.Philox.  One block of the
// counter c under the key (k0, k1) gives four 64-bit words.
AZG_HD uint64_t azg_mulhi64(uint64_t a, uint64_t b) {
#if defined(__CUDA_ARCH__)
  return __umul64hi(a, b);
#else
  return (uint64_t)(((unsigned __int128)a * b) >> 64);
#endif
}

AZG_HD void azg_philox4x64_10(uint64_t c[4], uint64_t k0, uint64_t k1) {
  for (int r = 0; r < 10; ++r) {
    if (r > 0) {
      k0 += 0x9E3779B97F4A7C15ull;
      k1 += 0xBB67AE8584CAA73Bull;
    }
    const uint64_t m0 = 0xD2E7470EE14C6C93ull, m1 = 0xCA5A826395121157ull;
    const uint64_t hi0 = azg_mulhi64(m0, c[0]), lo0 = m0 * c[0];
    const uint64_t hi1 = azg_mulhi64(m1, c[2]), lo1 = m1 * c[2];
    const uint64_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
    c[0] = n0;
    c[1] = lo1;
    c[2] = n2;
    c[3] = lo0;
  }
}

// word -> (0, 1]: ((w >> 11) + 0.5) 2^-53 (the top word of the range rounds to 1.0; 0 is never produced)
AZG_HD double azg_u01(uint64_t w) { return azg_dmul(azg_dadd((double)(w >> 11), 0.5), 1.1102230246251565e-16); }

#if defined(__CUDA_ARCH__)
AZG_HD double azg_log(double x) { return log(x); }
AZG_HD double azg_exp(double x) { return exp(x); }
AZG_HD double azg_cos(double x) { return cos(x); }
#else
static inline double azg_log(double x) { return log(x); }
static inline double azg_exp(double x) { return exp(x); }
static inline double azg_cos(double x) { return cos(x); }
#endif

#define AZG_NOISE_ATTEMPTS 32

// log Gamma(alpha) draw for one (seed, id, action): Marsaglia-Tsang at shape alpha + 1, boosted back to alpha in log
// space (log u4 / alpha), so small alpha neither underflows nor divides 0 by 0.  Attempt k reads the block at counter
// (id, action, k, 0).  Returns the accepted attempt, or -1 when none of the AZG_NOISE_ATTEMPTS was accepted.
AZG_HD int azg_log_gamma(uint64_t seed, uint64_t id, int action, double alpha, double* lg) {
  const double d = azg_dadd(azg_dadd(alpha, 1.0), -(1.0 / 3.0));
  const double c = azg_ddiv(1.0, azg_dsqrt(azg_dmul(9.0, d)));
  for (int k = 0; k < AZG_NOISE_ATTEMPTS; ++k) {
    uint64_t w[4] = {id, (uint64_t)action, (uint64_t)k, 0};
    azg_philox4x64_10(w, seed, 0);
    const double u1 = azg_u01(w[0]), u2 = azg_u01(w[1]), u3 = azg_u01(w[2]), u4 = azg_u01(w[3]);
    const double x = azg_dmul(azg_dsqrt(azg_dmul(-2.0, azg_log(u1))), azg_cos(azg_dmul(u2, 6.283185307179586)));
    const double t = azg_dadd(1.0, azg_dmul(c, x));
    const double v = azg_dmul(azg_dmul(t, t), t);
    if (!(v > 0.0)) continue;
    const double lv = azg_log(v);
    const double rhs = azg_dadd(azg_dadd(azg_dadd(azg_dmul(azg_dmul(x, x), 0.5), d), -azg_dmul(d, v)), azg_dmul(d, lv));
    if (azg_log(u3) < rhs) {
      *lg = azg_dadd(azg_dadd(azg_log(d), lv), azg_ddiv(azg_log(u4), alpha));
      return k;
    }
  }
  return -1;
}

// eta ~ Dir(alpha) over the legal moves of game g's root, written to eta_row [A] (also the scratch of the log-Gammas):
// eta_a = exp(lg_a - max) / sum_b exp(lg_b - max), summed in ascending action order; 0 on illegal actions, a zero row
// for a terminal root.  Running out of attempts sets the sticky status AZG_ERR_NOISE and leaves a zero row.
AZG_HD void azg_root_noise_game(const AzgArenaView& a, int g, uint64_t seed, uint64_t id, double alpha, double* eta_row) {
  const AzgState s = a.root[g];
  const uint32_t valids = azg_ended(a.rules, s).tag == AZG_TAG_NONE ? azg_valids(a.rules, s) : 0u;
  double mx = -INFINITY;
  bool ok = true;
  for (int i = 0; i < a.A; ++i) {
    double lg = 0.0;
    if ((valids >> i) & 1u) {
      if (azg_log_gamma(seed, id, i, alpha, &lg) < 0) {
        ok = false;
        break;
      }
      if (lg > mx) mx = lg;
    }
    eta_row[i] = lg;
  }
  if (!ok) {
    a.status[g] = AZG_ERR_NOISE;
    for (int i = 0; i < a.A; ++i) eta_row[i] = 0.0;
    return;
  }
  double sum = 0.0;
  for (int i = 0; i < a.A; ++i) {
    const double e = ((valids >> i) & 1u) ? azg_exp(azg_dadd(eta_row[i], -mx)) : 0.0;
    eta_row[i] = e;
    sum = azg_dadd(sum, e);
  }
  for (int i = 0; i < a.A; ++i) eta_row[i] = ((valids >> i) & 1u) ? azg_ddiv(eta_row[i], sum) : 0.0;
}

#if !defined(__CUDACC__)
// The host check build (tests/hostcheck) compiles this file with a host compiler and binds every azg_arena_* entry
// point of include/azgnn_b200.h under an `azgh_` name.  Its handle is a struct whose first and only member is the
// view, so the handle points at the view.
extern "C" int azgh_arena_set_semantics(AzgArenaView* a, int semantics) { return azg_view_set_semantics(a, semantics); }
extern "C" int azgh_arena_set_root_noise(AzgArenaView* a, const double* eta, double eps) {
  AZG_REQUIRE(a != nullptr, "azg_arena_set_root_noise: null arena");
  return azg_view_set_root_noise(a, eta, eps);
}
// the same sampler on the host (host libm: log / cos / exp may differ from the device's in the last bit)
extern "C" int azgh_arena_draw_root_noise(AzgArenaView* a, uint64_t seed, const uint64_t* ids, double alpha, double* eta,
                                          void*) {
  AZG_REQUIRE(a != nullptr, "azg_arena_draw_root_noise: null arena");
  AZG_REQUIRE(alpha > 0.0 && alpha < INFINITY, "azg_arena_draw_root_noise: alpha must be finite and > 0, got %g", alpha);
  AZG_REQUIRE(ids && eta, "azg_arena_draw_root_noise: null pointer");
  for (int g = 0; g < a->G; ++g) azg_root_noise_game(*a, g, seed, ids[g], alpha, eta + (size_t)g * a->A);
  return AZG_OK;
}
extern "C" int azgh_philox4x64(uint64_t seed, const uint64_t* counters, int64_t n, uint64_t* words, void*) {
  for (int64_t i = 0; i < n; ++i) {
    uint64_t c[4] = {counters[4 * i], counters[4 * i + 1], counters[4 * i + 2], counters[4 * i + 3]};
    azg_philox4x64_10(c, seed, 0);
    for (int j = 0; j < 4; ++j) words[4 * i + j] = c[j];
  }
  return AZG_OK;
}
#endif

// ---- rollout baseline: leaves valued by uniformly random playouts ------------------------------------------------
#define AZG_ROLLOUT_MAX_PLAYOUTS 4096

// Arguments of azg_rollout_eval, checked once for the library and the host check build; fills *r on success.
static inline int azg_rollout_setup(AzgRules* r, int game, int n, int playouts) {
  AZG_REQUIRE(game == AZG_GAME_CONNECT4 || game == AZG_GAME_TICTACTOE,
              "azg_rollout_eval: two-player games only (Connect4, TicTacToe), got game %d", game);
  AZG_REQUIRE(game == AZG_GAME_CONNECT4 ? (n >= 4 && n <= 8) : (n >= 3 && n <= 5),
              "azg_rollout_eval: unsupported board size %d (Connect4 4..8, TicTacToe 3..5)", n);
  AZG_REQUIRE(playouts >= 1 && playouts <= AZG_ROLLOUT_MAX_PLAYOUTS, "azg_rollout_eval: playouts must lie in [1, %d], got %d",
              AZG_ROLLOUT_MAX_PLAYOUTS, playouts);
  AZG_REQUIRE(azg_rules_init(r, game, n, nullptr) == 0, "azg_rollout_eval: unsupported game %d / size %d", game, n);
  return AZG_OK;
}

// One uniformly random playout from s: +1 / 0 / -1 for the player to move at s (draws, Connect4's 1e-4 included, are 0).
// Ply t reads word t % 4 of the Philox4x64-10 block at counter (s.mine, s.theirs, (game << 32) | playout, t / 4) under the
// key (seed, 1) -- root noise uses (seed, 0), so the streams share no block -- and plays the j-th legal action in
// ascending order, j = mulhi64(word, k) for k legal actions.  The game is checked with azg_ended at ply 0 only: a
// position that has not ended can only end by the mover's new stone, so later plies test the lines through it (TicTacToe)
// or the mover's stones (Connect4), and a full board.  That is azg_ended's answer by construction (the host spec test pins
// it); the outcome of the state reached after ply t is negated t + 1 times, because the canonical board flips every ply.
AZG_HD int azg_rollout_outcome(const AzgRules& r, AzgState s, uint64_t seed, uint32_t game, uint32_t playout) {
  const AzgVal e0 = azg_ended(r, s);
  if (e0.tag != AZG_TAG_NONE) return e0.d == 1.0 ? 1 : (e0.d == -1.0 ? -1 : 0);
  const bool c4 = r.game == AZG_GAME_CONNECT4;
  const int n = r.n;
  uint64_t full = r.board_mask;  // Connect4: no legal column once every top cell is taken
  if (c4) {
    full = 0;
    for (int x = 0; x < n; ++x) full |= 1ull << (x * n + n - 1);
  }
  const uint64_t c0 = s.mine, c1 = s.theirs, c2 = ((uint64_t)game << 32) | playout;
  uint64_t w[4] = {0, 0, 0, 0};
  for (int t = 0;; ++t) {
    if ((t & 3) == 0) {
      w[0] = c0;
      w[1] = c1;
      w[2] = c2;
      w[3] = (uint64_t)(t >> 2);
      azg_philox4x64_10(w, seed, 1);
    }
    const int q = t & 3;  // selects by value: an indexed w[] would live in local memory
    const uint64_t word = q == 0 ? w[0] : q == 1 ? w[1] : q == 2 ? w[2] : w[3];
    uint32_t m = azg_valids(r, s);
    int j = (int)azg_mulhi64(word, (uint64_t)azg_popc64(m));
    while (j-- > 0) m &= m - 1;
    const int a = azg_popc64((uint64_t)((m & (0u - m)) - 1u));  // index of the lowest remaining set bit
    const AzgState nx = azg_next(r, s, a);
    const uint64_t mover = nx.theirs;
    bool won;
    if (c4) {
      won = azg_c4_wins(r, mover);
    } else {  // lines through cell a = x * n + y: row y, column x, and the diagonals it lies on
      const int x = a / n, y = a % n;
      won = (mover & r.lines[y]) == r.lines[y] || (mover & r.lines[n + x]) == r.lines[n + x] ||
            (x == y && (mover & r.lines[2 * n]) == r.lines[2 * n]) ||
            (x + y == n - 1 && (mover & r.lines[2 * n + 1]) == r.lines[2 * n + 1]);
    }
    if (won) return (t & 1) ? -1 : 1;  // the mover of ply t is the player to move at s when t is even
    if (((nx.mine | nx.theirs) & full) == full) return 0;
    s = nx;
  }
}

// pi row for a leaf: 1/k (float32, rounded to nearest) on its k legal moves (azg_valids), 0 elsewhere
AZG_HD void azg_rollout_policy(const AzgRules& r, AzgState s, float* pi_row, int lane, int lanes) {
  const uint32_t m = azg_valids(r, s);
  const float p = azg_fdiv(1.0f, (float)azg_popc64(m));
  for (int a = lane; a < r.A; a += lanes) pi_row[a] = ((m >> a) & 1u) ? p : 0.0f;
}

#if !defined(__CUDACC__)
// host check build of azg_rollout_eval (host pointers, rows one after the other)
extern "C" int azgh_rollout_eval(int game, int n, const uint64_t* states, const int32_t* games, int64_t rows,
                                 const int32_t* count, int playouts, uint64_t seed, float* pi, float* v, void*) {
  AzgRules r;
  const int rc = azg_rollout_setup(&r, game, n, playouts);
  if (rc != AZG_OK) return rc;
  AZG_REQUIRE(rows >= 0 && rows <= 0x7FFFFFFF, "azg_rollout_eval: rows must lie in [0, 2^31), got %lld", (long long)rows);
  AZG_REQUIRE(rows == 0 || (states && pi && v), "azg_rollout_eval: null pointer");
  const int64_t live = count ? (*count < rows ? *count : rows) : rows;
  for (int64_t i = 0; i < live; ++i) {
    AzgState s;
    s.mine = states[2 * i];
    s.theirs = states[2 * i + 1];
    const uint32_t g = games ? (uint32_t)games[i] : (uint32_t)i;
    int sum = 0;
    for (int p = 0; p < playouts; ++p) sum += azg_rollout_outcome(r, s, seed, g, (uint32_t)p);
    v[i] = azg_fdiv((float)sum, (float)playouts);
    azg_rollout_policy(r, s, pi + i * r.A, 0, 1);
  }
  return AZG_OK;
}
#endif

// ---- table growth: copy game g from `s` into the larger `d` (same game, A, max_depth; d.cap >= s.cap) ------------
// part 1 (any number of lanes): clear d's hash slots and copy the node and edge arrays verbatim (node indices are kept)
AZG_HD void azg_copy_game_nodes(const AzgArenaView& d, const AzgArenaView& s, int g, int lane, int lanes) {
  int32_t* hs = d.hslot + (size_t)g * d.hcap;
  for (int i = lane; i < d.hcap; i += lanes) hs[i] = 0;
  const int count = s.node_count[g];
  const size_t sn = (size_t)g * s.cap, dn = (size_t)g * d.cap, A = (size_t)s.A;
  for (int i = lane; i < count; i += lanes) {
    d.key[dn + i] = s.key[sn + i];
    d.es[dn + i] = s.es[sn + i];
    d.es_tag[dn + i] = s.es_tag[sn + i];
    d.ns[dn + i] = s.ns[sn + i];
    d.valids[dn + i] = s.valids[sn + i];
    d.ptag[dn + i] = s.ptag[sn + i];
    for (size_t e = 0; e < A; ++e) {
      d.P[(dn + i) * A + e] = s.P[(sn + i) * A + e];
      d.Q[(dn + i) * A + e] = s.Q[(sn + i) * A + e];
      d.qtag[(dn + i) * A + e] = s.qtag[(sn + i) * A + e];
      d.N[(dn + i) * A + e] = s.N[(sn + i) * A + e];
    }
  }
}
// part 2 (one lane, after part 1 is complete): per-game scalars, the search path, and the hash rebuilt for d.hcap
AZG_HD void azg_copy_game_finish(const AzgArenaView& d, const AzgArenaView& s, int g) {
  d.root[g] = s.root[g];
  d.sims_left[g] = s.sims_left[g];
  d.node_count[g] = s.node_count[g];
  d.pending[g] = s.pending[g];
  d.path_len[g] = s.path_len[g];
  d.status[g] = s.status[g];
  for (int i = 0; i < s.path_len[g] && i < d.max_depth; ++i) {
    d.path_node[(size_t)g * d.max_depth + i] = s.path_node[(size_t)g * s.max_depth + i];
    d.path_act[(size_t)g * d.max_depth + i] = s.path_act[(size_t)g * s.max_depth + i];
  }
  int32_t* hs = d.hslot + (size_t)g * d.hcap;
  const AzgState* keys = d.key + (size_t)g * d.cap;
  for (int i = 0; i < s.node_count[g]; ++i) {
    uint32_t slot = (uint32_t)azg_hash(keys[i]) & (uint32_t)(d.hcap - 1);
    while (hs[slot] != 0) slot = (slot + 1) & (uint32_t)(d.hcap - 1);
    hs[slot] = i + 1;
  }
}

// ---- memory carve-up shared by device and host builds -------------------------------------
static inline size_t azg_align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

static inline int azg_hash_capacity(int cap) {
  int h = 16;
  while (h < 2 * cap) h <<= 1;
  return h;
}

// lays the arrays out inside `base` (may be NULL to measure); returns total bytes
static inline size_t azg_arena_carve(AzgArenaView* v, char* base) {
  size_t off = 0;
  const size_t G = v->G, cap = v->cap, A = v->A, D = v->max_depth, H = v->hcap;
#define AZG_CARVE(field, type, count)                       \
  do {                                                      \
    off = azg_align_up(off, 256);                           \
    v->field = base ? (type*)(base + off) : (type*)nullptr; \
    off += sizeof(type) * (count);                          \
  } while (0)
  AZG_CARVE(root, AzgState, G);
  AZG_CARVE(sims_left, int32_t, G);
  AZG_CARVE(node_count, int32_t, G);
  AZG_CARVE(pending, int32_t, G);
  AZG_CARVE(path_len, int32_t, G);
  AZG_CARVE(path_node, int32_t, G * D);
  AZG_CARVE(path_act, int8_t, G * D);
  AZG_CARVE(status, int32_t, G);
  AZG_CARVE(hslot, int32_t, G * H);
  AZG_CARVE(key, AzgState, G * cap);
  AZG_CARVE(es, double, G * cap);
  AZG_CARVE(es_tag, int8_t, G * cap);
  AZG_CARVE(ns, int32_t, G * cap);
  AZG_CARVE(valids, uint32_t, G * cap);
  AZG_CARVE(ptag, int8_t, G * cap);
  AZG_CARVE(P, double, G * cap * A);
  AZG_CARVE(Q, double, G * cap * A);
  AZG_CARVE(qtag, int8_t, G * cap * A);
  AZG_CARVE(N, int32_t, G * cap * A);
#undef AZG_CARVE
  return azg_align_up(off, 256);
}
