// azg_replay.cu -- the example pipeline between self-play and training, on the device (SURVEY section 8f.1):
//
//   Coach.executeEpisode tail (Coach.py:45-49, 68-79): every stored position of a finished episode becomes
//     S symmetric examples (Connect4Game.getSymmetries :189-215 -- mirror, with its axis quirk;
//     TicTacToeGame.getSymmetries :187-200 -- 4 rotations x {flipped, not}; FrozenLake: identity) whose value is
//     the result signed for the player who was to move:  v = r * (-1)^(player != cur)
//   minibatch assembly of *.train (Connect4GNN.py:141-148): boards[idx] -> float32 [B,n,n], pi[idx], v[idx]
//
// Positions are the packed 16-byte states of the arena; policies stay float64 (the reference keeps Python floats)
// so that exported examples round-trip the reference's pickle format exactly.  A symmetry is a cell permutation
// given as a table (built on the host by applying the reference's own numpy calls to an index array, so the
// kernels hold no game knowledge): out cell d takes in cell perm[s][d], out policy entry a takes pi[pi_perm[s][a]].
#include "azg_common.cuh"

namespace {

struct State2 {
  uint64_t mine, theirs;
};

inline int grid_for(int64_t n, int threads) { return (int)((n + threads - 1) / threads); }

// One thread per (history entry e, symmetry s): writes example e*S + s.
//   states/pi/player: [E] history entries;  game[e]: index into result/cur/out_base tables of finished games
//   v = result[g] * (player[e] != cur[g] ? -1 : 1);  vtag carries the result's Python type (int / float)
__global__ void emit_examples_kernel(const State2* __restrict__ states, const double* __restrict__ pi,
                                     const int32_t* __restrict__ player, const int32_t* __restrict__ game,
                                     const double* __restrict__ result, const int8_t* __restrict__ result_tag,
                                     const int32_t* __restrict__ cur, int64_t E, int ncells, int A, int S,
                                     const int32_t* __restrict__ board_perm, const int32_t* __restrict__ pi_perm,
                                     State2* __restrict__ out_states, double* __restrict__ out_pi, double* __restrict__ out_v,
                                     int8_t* __restrict__ out_vtag) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= E * S) return;
  const int64_t e = i / S;
  const int s = (int)(i - e * S);
  const State2 in = states[e];
  State2 o{0ull, 0ull};
  const int32_t* bp = board_perm + (size_t)s * ncells;
  for (int d = 0; d < ncells; ++d) {
    const int src = bp[d];
    o.mine |= ((in.mine >> src) & 1ull) << d;
    o.theirs |= ((in.theirs >> src) & 1ull) << d;
  }
  out_states[i] = o;
  const int32_t* pp = pi_perm + (size_t)s * A;
  for (int a = 0; a < A; ++a) out_pi[i * A + a] = pi[e * A + pp[a]];
  if (out_v) {
    const int g = game[e];
    out_v[i] = result[g] * (player[e] != cur[g] ? -1.0 : 1.0);
    out_vtag[i] = result_tag[g];
  }
}

// FrozenLake states keep the agent cell index in `mine` (FrozenLakeGame.py:197-202): no bit permutation
__global__ void emit_examples_fl_kernel(const State2* __restrict__ states, const double* __restrict__ pi,
                                        const int32_t* __restrict__ player, const int32_t* __restrict__ game,
                                        const double* __restrict__ result, const int8_t* __restrict__ result_tag,
                                        const int32_t* __restrict__ cur, int64_t E, int A, State2* __restrict__ out_states,
                                        double* __restrict__ out_pi, double* __restrict__ out_v, int8_t* __restrict__ out_vtag) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  out_states[e] = states[e];
  for (int a = 0; a < A; ++a) out_pi[e * A + a] = pi[e * A + a];
  if (out_v) {
    const int g = game[e];
    out_v[e] = result[g] * (player[e] != cur[g] ? -1.0 : 1.0);
    out_vtag[e] = result_tag[g];
  }
}

// minibatch gather: one thread per (row, cell) for the boards, per (row, action) for pi, per row for v
__global__ void gather_examples_kernel(const State2* __restrict__ states, const double* __restrict__ pi, const double* __restrict__ v,
                                       const int64_t* __restrict__ idx, int B, int ncells, int A, int frozenlake,
                                       float* __restrict__ boards, float* __restrict__ out_pi, float* __restrict__ out_v) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int per = ncells + A + 1;
  if (i >= (int64_t)B * per) return;
  const int b = (int)(i / per), k = (int)(i - (int64_t)b * per);
  const int64_t src = idx[b];
  if (k < ncells) {
    const State2 s = states[src];
    float cell;
    if (frozenlake) cell = (int64_t)s.mine == k ? 1.0f : 0.0f;
    else cell = (float)((int)((s.mine >> k) & 1ull) - (int)((s.theirs >> k) & 1ull));
    boards[(size_t)b * ncells + k] = cell;
  } else if (k < ncells + A) {
    out_pi[(size_t)b * A + (k - ncells)] = (float)pi[src * A + (k - ncells)];
  } else {
    out_v[b] = (float)v[src];
  }
}


// ---- the host tail of a self-play move, on the device --------------------------------------------------------------------
// Per game, one thread (Coach.py:36-63 and MCTS.py:36-58, 94-143 between the searches of a move and the move itself):
//   getActionProb's tail   counts -> policy: temp 1: [(x + 1e-8)] / float(sum(.)) with CPython's left-to-right Neumaier `sum`;
//                          temp 0: uniform choice among the arg-max counts from the supplied uniform, one-hot policy
//   np.random.choice       inverse CDF of the policy at the supplied uniform (sequential cumsum, cdf /= cdf[-1])
//   history                (root state, policy, player, temp-0 flag) -> slot [t, g] of the episode history in HBM
//   expand_tree record     initial / expanded visit policies and the expanded value sum_a Q N / sum_a N with the NEP-50
//                          promotion order of the reference's scalar loop (Python number until the first np.float32 term)
// Every rounding is spelled out (no FMA contraction): the results equal selfplay.probs_from_counts / sample_actions and
// mcts.expanded_values bit for bit, which tests/test_selfplay_move_gpu.py checks through the C ABI and
// tests/test_replay_gpu.py through whole self-play runs.
constexpr int MOVE_MAX_A = 65;  // TicTacToe 8x8 + pass (MOVE_MAX_A of the arena core)
__global__ void __launch_bounds__(128) selfplay_move_kernel(azg_move_params p) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= p.G) return;
  const int A = p.A;
  const int t = p.slot[g];
  if (t < 0) {
    p.actions[g] = -1;
    return;
  }
  if (t >= p.T && (p.h_states || (p.n1 && p.rec_ip))) {  // no history row to write into: an error, nothing is written
    atomicOr(p.flags, 2);
    p.actions[g] = -1;
    return;
  }
  const int32_t* n0 = p.n0 + (size_t)g * A;
  double probs[MOVE_MAX_A];
  int act = 0;
  if (p.greedy[g]) {
    int best = n0[0], nbest = 0;
    for (int a = 1; a < A; ++a) best = n0[a] > best ? n0[a] : best;
    for (int a = 0; a < A; ++a) nbest += n0[a] == best;
    const long long k = (long long)__dmul_rn(p.u_tie[g], (double)nbest);
    int seen = 0, pick = 0;
    bool found = false;
    for (int a = 0; a < A; ++a) {
      seen += n0[a] == best;
      if (!found && (long long)seen > k) { pick = a; found = true; }
    }
    for (int a = 0; a < A; ++a) probs[a] = a == pick ? 1.0 : 0.0;
  } else {
    double f = __dadd_rn((double)n0[0], 1e-8), c = 0.0;
    for (int a = 1; a < A; ++a) {
      const double v = __dadd_rn((double)n0[a], 1e-8);
      const double s = __dadd_rn(f, v);
      c = __dadd_rn(c, fabs(f) >= fabs(v) ? __dadd_rn(__dadd_rn(f, -s), v) : __dadd_rn(__dadd_rn(v, -s), f));
      f = s;
    }
    const double tot = (c != 0.0 && isfinite(c)) ? __dadd_rn(f, c) : f;
    for (int a = 0; a < A; ++a) probs[a] = __ddiv_rn(__dadd_rn((double)n0[a], 1e-8), tot);
  }
  {  // numpy.random.choice(len(p), p=p): cdf = cumsum(p); cdf /= cdf[-1]; searchsorted(cdf, u, side='right')
    double cdf[MOVE_MAX_A];
    double run = 0.0;
    for (int a = 0; a < A; ++a) {
      run = a == 0 ? probs[0] : __dadd_rn(run, probs[a]);
      cdf[a] = run;
    }
    const double last = cdf[A - 1], u = p.u_sample[g];
    int cnt = 0;
    for (int a = 0; a < A; ++a) cnt += __ddiv_rn(cdf[a], last) <= u;
    act = cnt < A - 1 ? cnt : A - 1;
  }
  p.actions[g] = act;
  const size_t slot = (size_t)t * p.G + g;
  if (p.h_states) {
    p.h_states[2 * slot] = p.roots[2 * g];
    p.h_states[2 * slot + 1] = p.roots[2 * g + 1];
    for (int a = 0; a < A; ++a) p.h_pi[slot * A + a] = probs[a];
    p.h_player[slot] = p.player[g];
    p.h_int[slot] = p.greedy[g];
  }
  if (p.n1 && p.rec_ip) {
    // initial / expanded visit policies (MCTS.py:95-103, 125-130): N / sum(N), small integers: exact in any order
    const int32_t* n1 = p.n1 + (size_t)g * A;
    long long tot0 = 0, tot1 = 0;
    for (int a = 0; a < A; ++a) {
      tot0 += n0[a] > 0 ? n0[a] : 0;
      tot1 += n1[a] > 0 ? n1[a] : 0;
    }
    if (tot0 <= 0) atomicOr(p.flags, 1);  // no root visits: the host path's valid-move fallback is not reproduced here
    for (int a = 0; a < A; ++a) {
      const double ip = tot0 > 0 ? __ddiv_rn((double)(n0[a] > 0 ? n0[a] : 0), (double)tot0) : 0.0;
      p.rec_ip[slot * A + a] = ip;
      p.rec_ep[slot * A + a] = tot1 > 0 ? __ddiv_rn((double)(n1[a] > 0 ? n1[a] : 0), (double)tot1) : ip;
    }
    // expanded value (MCTS.py:132-143), see mcts.expanded_values
    const double* q1 = p.q1 + (size_t)g * A;
    const int8_t* t1 = p.t1 + (size_t)g * A;
    double acc64 = 0.0;
    float acc32 = 0.0f;
    bool is32 = false;
    long long cntv = 0;
    for (int a = 0; a < A; ++a) {
      const long long n = n1[a];
      const bool valid = t1[a] != AZG_TAG_NONE && n > 0;
      if (!valid) continue;
      const bool f32 = t1[a] == AZG_TAG_F32;
      if (!f32) {
        const double term64 = __dmul_rn(q1[a], (double)n);
        if (!is32) acc64 = __dadd_rn(acc64, term64);
        else acc32 = __fadd_rn(acc32, (float)term64);
      } else {
        const float term32 = __fmul_rn((float)q1[a], (float)n);
        acc32 = is32 ? __fadd_rn(acc32, term32) : __fadd_rn((float)acc64, term32);
        is32 = true;
      }
      cntv += n;
    }
    double ev;
    int8_t evtag;
    if (cntv > 0) {
      ev = is32 ? (double)__fdiv_rn(acc32, (float)cntv) : __ddiv_rn(acc64, (double)cntv);
      evtag = is32 ? AZG_TAG_F32 : AZG_TAG_PYFLOAT;
    } else {
      ev = (double)p.v0[g];
      evtag = AZG_TAG_F32;
    }
    p.rec_iv[slot] = p.v0[g];
    p.rec_ev[slot] = ev;
    p.rec_evtag[slot] = evtag;
  }
}

}  // namespace

extern "C" {

int azg_selfplay_move(const azg_move_params* p, azg_stream stream) {
  AZG_REQUIRE(p && p->G > 0 && p->A >= 1 && p->A <= MOVE_MAX_A, "azg_selfplay_move: bad sizes");
  AZG_REQUIRE(p->n0 && p->greedy && p->u_tie && p->u_sample && p->slot && p->actions && p->flags, "azg_selfplay_move: null pointer");
  AZG_REQUIRE(!p->h_states || (p->roots && p->player && p->h_pi && p->h_player && p->h_int && p->T > 0), "azg_selfplay_move: history buffers missing");
  AZG_REQUIRE(!p->n1 || !p->rec_ip || (p->q1 && p->t1 && p->v0 && p->rec_iv && p->rec_ep && p->rec_ev && p->rec_evtag && p->T > 0),
              "azg_selfplay_move: record buffers missing");
  selfplay_move_kernel<<<grid_for(p->G, 128), 128, 0, (cudaStream_t)stream>>>(*p);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

int azg_emit_examples(int frozenlake, const uint64_t* states, const double* pi, const int32_t* player, const int32_t* game,
                      const double* result, const int8_t* result_tag, const int32_t* cur, int64_t E, int ncells, int A, int S,
                      const int32_t* board_perm, const int32_t* pi_perm, uint64_t* out_states, double* out_pi, double* out_v,
                      int8_t* out_vtag, azg_stream stream) {
  AZG_REQUIRE(states && pi && out_states && out_pi && A >= 1 && S >= 1, "azg_emit_examples: bad argument");
  AZG_REQUIRE(!out_v || (player && game && result && result_tag && cur && out_vtag), "azg_emit_examples: value inputs missing");
  AZG_REQUIRE(frozenlake || (board_perm && pi_perm && ncells >= 1 && ncells <= 64), "azg_emit_examples: permutation tables missing");
  if (E <= 0) return AZG_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (frozenlake) {
    AZG_REQUIRE(S == 1, "azg_emit_examples: FrozenLake has no symmetries");
    emit_examples_fl_kernel<<<grid_for(E, 256), 256, 0, st>>>((const State2*)states, pi, player, game, result, result_tag, cur, E, A,
                                                              (State2*)out_states, out_pi, out_v, out_vtag);
  } else {
    emit_examples_kernel<<<grid_for(E * S, 256), 256, 0, st>>>((const State2*)states, pi, player, game, result, result_tag, cur, E,
                                                               ncells, A, S, board_perm, pi_perm, (State2*)out_states, out_pi,
                                                               out_v, out_vtag);
  }
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

int azg_gather_examples(int frozenlake, const uint64_t* states, const double* pi, const double* v, const int64_t* idx, int B,
                        int ncells, int A, float* boards, float* out_pi, float* out_v, azg_stream stream) {
  AZG_REQUIRE(states && pi && v && idx && boards && out_pi && out_v && ncells >= 1 && ncells <= 64 && A >= 1,
              "azg_gather_examples: bad argument");
  if (B <= 0) return AZG_OK;
  gather_examples_kernel<<<grid_for((int64_t)B * (ncells + A + 1), 256), 256, 0, (cudaStream_t)stream>>>(
      (const State2*)states, pi, v, idx, B, ncells, A, frozenlake, boards, out_pi, out_v);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

}  // extern "C"
