/* azgnn_b200.h -- C ABI of libazgnn_b200.so (sm_100a only).
 *
 * The reference (andrpac/alphazero-gnn) is pure Python and has no FFI; its seam for this
 * hot path is the duck-typed NeuralNet / MCTS surface (SURVEY.md section 8b).  Every entry
 * point below names the reference call it replaces.  Conventions:
 *   - plain C: pointers + sizes, no C++/torch types; all data pointers are DEVICE pointers
 *     to caller-owned memory unless a parameter says "host";
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*);
 *   - return value 0 = AZG_OK; otherwise azg_last_error() describes the failure
 *     (the Python wrappers raise RuntimeError -- no silent fallbacks, cf. MCTS.py:195-200);
 *   - the library keeps no global mutable state except the thread-local error string;
 *     an arena handle is thread-compatible (one user at a time).
 *
 * Position format ("state"): two uint64 per position, {mine, theirs}, canonical form
 * (player to move = +1, Connect4Game.py:185-187).  Bit x*n + y is cell board[x][y] of the
 * reference's n x n int64 array (Connect4: x = column, y = row from the bottom,
 * Connect4Game.py:18-22; TicTacToe: action a = x*n + y, TicTacToeGame.py:153).
 * FrozenLake: mine = agent cell index r*n + c, theirs = 0 (FrozenLakeGame.py:197-202).
 */
#ifndef AZGNN_B200_H
#define AZGNN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AZG_ABI_VERSION 3

#define AZG_OK 0
#define AZG_ERR_INVALID 1   /* bad argument */
#define AZG_ERR_CUDA 2      /* CUDA runtime error (message in azg_last_error) */
#define AZG_ERR_DEVICE 3    /* not an sm_100 device / no device */
#define AZG_ERR_CAPACITY 4  /* arena node table full */
#define AZG_ERR_NOISE 5     /* root noise: no Gamma draw accepted in 32 attempts (probability below 1e-40) */

#define AZG_GAME_CONNECT4 0
#define AZG_GAME_TICTACTOE 1
#define AZG_GAME_FROZENLAKE 2

/* which predictions to produce (MCTS.py:169-178 evaluates both when use_gnn) */
#define AZG_EVAL_STD 1 /* NeuralNet.predict            */
#define AZG_EVAL_GNN 2 /* NeuralNet.predict_with_gnn   */
#define AZG_EVAL_FOLD 4 /* with AZG_EVAL_GNN on the tensor-core path: output_transform.2 folded into the policy/value heads
                         (no non-linearity between them, gnn_utils.py:99-103 -> Connect4GNN.py:48-57): same pi/v within the
                         fp32 contract, half the F x F contractions.  Opt-in; ignored by the fp32 path. */

/* arithmetic of the dense F x F contractions (output_transform, gnn_utils.py:99-103) */
#define AZG_PREC_FP32 0   /* fp32 FFMA on CUDA cores                                  */
#define AZG_PREC_BF16X3 1 /* tcgen05 kind::f16, 3-term bf16 split, fp32 accumulate    */
#define AZG_PREC_BF16 2   /* tcgen05 kind::f16, bf16 operands, fp32 accumulate        */
#define AZG_PREC_F16F8 3  /* tcgen05 kind::f16 on fp16(x) fp16(w) + one K-concatenated block-scaled FP8 (kind::mxf8f6f4)
                             correction product, same fp32 accumulator: the 1e-5 contract at 2/3 of the bf16x3 MMA time
                             (Connect4 path; tile widths 128..224)                                                    */
#define AZG_PREC_F16F8_KS 4 /* AZG_PREC_F16F8 operands (same packed images), each F x F contraction accumulated in four
                             launches over a quarter of K with round-to-nearest fp32 adds of the partial sums in between:
                             the tensor core's truncating accumulation error, linear in the number of k-steps (~1e-5 at
                             K = 3136 on trained weights), is divided by four.  Connect4 path (azg_c4_forward*)        */
#define AZG_PREC_BF16X3_KS 5 /* the same K-split on the AZG_PREC_BF16X3 operands (three bf16 terms: the finer operand
                             representation, 12 instead of 8 MMA times per k-block)                                     */

/* value type tags (NumPy>=2 / NEP 50 semantics of MCTS.py:228-233, SURVEY section 0.3) */
#define AZG_TAG_NONE (-1) /* edge not in Qsa            */
#define AZG_TAG_F32 0     /* numpy.float32              */
#define AZG_TAG_PYFLOAT 1 /* Python float (binary64)    */
#define AZG_TAG_PYINT 2   /* Python int                 */

typedef void* azg_stream; /* cudaStream_t */

const char* azg_last_error(void);
int azg_abi_version(void);
/* host out-params; fails with AZG_ERR_DEVICE when the current device is not compute 10.x */
int azg_device_info(int* cc_major, int* cc_minor, int* sm_count);

/* measurement hooks (bench.py): number of kernels this library has launched so far, and optional
 * CUDA-event timing of the phases of a forward call on the launching stream.  phase: 0 trunk
 * (encode + convolutions), 1 dense F x F contractions, 2 heads, 3 arena kernels. */
unsigned long long azg_launch_count(void);
int azg_timing_enable(int on); /* also clears the records */
int azg_timing_read(int phase, double* total_ms, int* records);

/* ---------------------------------------------------------------- K1: encode ------------ */
/* cells [B, n*n] with values {-1,0,1} -> states [B,2].  cell_dtype selects the element type of
 * `cells` (the reference keeps boards as int64, Connect4Game.py:129-132; FrozenLake as float64
 * one-hot, FrozenLakeGame.py:76-78, for which the state is the arg-max cell).  Replaces the
 * per-call numpy->tensor hop torch.FloatTensor(board.astype(np.float64)) (Connect4GNN.py:71-72). */
#define AZG_CELL_I8 0
#define AZG_CELL_I64 1
#define AZG_CELL_F32 2
#define AZG_CELL_F64 3
int azg_pack_boards(const void* cells, int cell_dtype, int n, int64_t B, uint64_t* states, azg_stream stream);
/* states [B,2] -> fp32 planes [B, n*n] in {-1,0,1}: the network input of
 * Connect4Net.forward (Connect4Net.py:42) / TicTacToeNet.forward (TicTacToeNet.py:30). */
int azg_encode_planes(const uint64_t* states, int n, int64_t B, float* planes, azg_stream stream);
/* FrozenLake graph build of FrozenLakeNet.predict (FrozenLakeNet.py:197-213): node 0 = the
 * state, nodes 1..k = successors of the valid actions; writes one-hot node features
 * [B,5,n*n] (unused nodes zero) and the node count [B] (3..5). */
int azg_fl_encode_graph(const uint64_t* states, int n, int64_t B, float* nodes, int32_t* counts,
                        azg_stream stream);

/* ---------------------------------------------------------------- K2: forward ----------- */
/* Connect4 (connect4/Connect4Net.py:18-60, connect4/Connect4GNN.py:31-120).  fp32 tensors in
 * the reference's own layouts (Conv2d [Cout,Cin,3,3], Linear [out,in]). */
typedef struct azg_c4_params {
  const float *conv1_w, *conv1_b;         /* [32,1,3,3], [32]   */
  const float *conv2_w, *conv2_b;         /* [64,32,3,3], [64]  */
  const float *fc_policy_w, *fc_policy_b; /* [n+1, 64 n^2], [n+1] */
  const float *fc_value_w, *fc_value_b;   /* [1, 64 n^2], [1]   */
  const float *ot0_w, *ot0_b;             /* gnn.output_transform.0: [F,F], [F] (may be NULL without AZG_EVAL_GNN) */
  const float *ot2_w, *ot2_b;             /* gnn.output_transform.2: [F,F], [F] */
  const void* ot_packed;                  /* azg_c4_pack output for the tcgen05 precisions, else NULL */
} azg_c4_params;

size_t azg_c4_workspace_bytes(int n, int64_t B, int eval_mask, int prec);
/* Batched Connect4GNNWrapper.predict (+ predict_with_gnn): every row has the reference's B=1
 * semantics (each GNNLayer is the identity at B=1, gnn_utils.py:35-36).  Outputs: pi [B,n+1]
 * (= exp(log_softmax)), v [B] (= tanh).  Output pointers for a prediction not in eval_mask
 * may be NULL. */
int azg_c4_forward(const azg_c4_params* p, int n, const uint64_t* states, int64_t B, int eval_mask,
                   int prec, float* pi_std, float* v_std, float* pi_gnn, float* v_gnn,
                   void* workspace, size_t workspace_bytes, azg_stream stream);
/* Same with the number of valid positions decided on the device: dyn_rows (device int32, may be NULL)
 * holds how many of the B rows are live (the arena's compacted leaf count); rows beyond it are neither
 * computed nor written on the tensor-core path (the fp32 path evaluates all B rows). */
int azg_c4_forward_dyn(const azg_c4_params* p, int n, const uint64_t* states, int64_t B, const int32_t* dyn_rows,
                       int eval_mask, int prec, float* pi_std, float* v_std, float* pi_gnn, float* v_gnn,
                       void* workspace, size_t workspace_bytes, azg_stream stream);
/* Build the tcgen05 operand images of the weights (conv2, output_transform, heads) for
 * AZG_PREC_BF16X3 / AZG_PREC_BF16 / AZG_PREC_F16F8 (AZG_PREC_F16F8_KS / AZG_PREC_BF16X3_KS read the AZG_PREC_F16F8 / AZG_PREC_BF16X3 images and may be passed
 * instead: same bytes); the result goes into azg_c4_params.ot_packed.  Call again after
 * every optimizer step / load_checkpoint.  packed: device memory, 16-byte aligned. */
size_t azg_c4_packed_bytes(int n, int prec);
int azg_c4_pack(const azg_c4_params* p, int n, int prec, void* packed, size_t packed_bytes, azg_stream stream);

/* One dense layer on the tcgen05 path, for parity tests of the GEMM in isolation:
 * C[M,F] = act(A[M,F] . W[F,F]^T + bias), fp32 in/out, prec = AZG_PREC_BF16X3 | AZG_PREC_BF16 | AZG_PREC_F16F8 |
 * AZG_PREC_F16F8_KS | AZG_PREC_BF16X3_KS.
 * scratch: >= 2*(ceil(M/256)*256 + F)*F*2 + 1024 bytes (x3) or half of that (bf16). */
int azg_tc_linear(const float* A, const float* W, const float* bias, float* C, int64_t M, int F, int prec,
                  int relu, void* scratch, size_t scratch_bytes, azg_stream stream);

/* TicTacToe (tictactoe/TicTacToeNet.py:16-48, tictactoe/TicTacToeGNN.py:25-87) */
typedef struct azg_ttt_params {
  const float *conv1_w, *conv1_b, *conv2_w, *conv2_b, *conv3_w, *conv3_b; /* 1->32->64->128 */
  const float *fc1_w, *fc1_b, *fc_policy_w, *fc_policy_b;                 /* F->512->n^2+1 */
  const float *fc2_w, *fc2_b, *fc_value_w, *fc_value_b;                   /* F->512->1     */
  const float *ot0_w, *ot0_b, *ot2_w, *ot2_b;                             /* F->F->F       */
} azg_ttt_params;
size_t azg_ttt_workspace_bytes(int n, int64_t B, int eval_mask);
int azg_ttt_forward(const azg_ttt_params* p, int n, const uint64_t* states, int64_t B, int eval_mask,
                    float* pi_std, float* v_std, float* pi_gnn, float* v_gnn, void* workspace,
                    size_t workspace_bytes, azg_stream stream);

/* The same forward with conv2 / conv3 (im2col GEMMs whose A operand is written directly as tile images), fc1 / fc2
 * and output_transform on tcgen05 (prec = AZG_PREC_BF16X3: pi, v within 1e-5 of the fp32 module; AZG_PREC_BF16:
 * stated tolerance 5e-3); conv1 and the two small heads stay fp32.  `packed` = weight images from azg_ttt_pack
 * (azg_ttt_packed_bytes bytes, 1 KB aligned), rebuilt after every weight update. */
size_t azg_ttt_packed_bytes(int n, int prec);
int azg_ttt_pack(const azg_ttt_params* p, int n, int prec, void* packed, size_t packed_bytes, azg_stream stream);
size_t azg_ttt_tc_workspace_bytes(int n, int64_t B, int eval_mask);
int azg_ttt_forward_tc(const azg_ttt_params* p, const void* packed, int n, int prec, const uint64_t* states, int64_t B,
                       int eval_mask, float* pi_std, float* v_std, float* pi_gnn, float* v_gnn, void* workspace,
                       size_t workspace_bytes, azg_stream stream);

/* FrozenLake (frozenlake/FrozenLakeNet.py:178-230 predict, :297-334 EnhancedNNet.forward) */
typedef struct azg_fl_params {
  const float *fe0_w, *fe0_b; /* feature_extractor.0: [128, n^2] */
  const float *fe2_w, *fe2_b; /* feature_extractor.2: [E, 128]   */
  const float* const* gnn_w;  /* host array of `layers` device pointers, each [E,E] */
  const float* const* gnn_b;  /* host array of `layers` device pointers, each [E]   */
  const float *policy_w, *policy_b; /* [4,E] */
  const float *value_w, *value_b;   /* [1,E] */
} azg_fl_params;
int azg_fl_forward(const azg_fl_params* p, int n, int embedding_dim, int layers, const uint64_t* states,
                   int64_t B, float* pi, float* v, azg_stream stream);

/* generic dense layer on device tensors: C[M,N] = act(A[M,K] . W[N,K]^T + bias), fp32 FFMA.
 * (torch.nn.functional.linear as used throughout the reference nets.) relu: 0/1. */
int azg_linear_f32(const float* A, const float* W, const float* bias, float* C, int64_t M, int N, int K,
                   int relu, azg_stream stream);

/* ---------------------------------------------------------------- K3: training pieces ---- */
/* fp32 building blocks of Connect4GNNWrapper.train / TicTacToeGNNWrapper.train
 * (connect4/Connect4GNN.py:122-197); torch.autograd.Function wrappers route tensors between them,
 * the optimizer step stays in torch. */
/* C[M,N] = op(A) . op(B) + beta*C, row-major with leading dimensions; transX = 1: stored transposed */
int azg_gemm_f32(int transA, int transB, int64_t M, int N, int K, const float* A, int64_t lda, const float* B,
                 int64_t ldb, float* C, int64_t ldc, float beta, azg_stream stream);
int azg_mul_f32(const float* a, const float* b, float* out, int64_t n, azg_stream stream); /* dropout mask */
/* backward of Y = act(X W^T + b): dX [M,K], dW [N,K], db [N] (each may be NULL); relu: Y and an
 * M*N-float scratch are required */
int azg_linear_backward(const float* dY, const float* X, const float* W, const float* Y, int64_t M, int N, int K,
                        int relu, float* dX, float* dW, float* db, float* scratch, azg_stream stream);
/* backward of out = relu(conv3x3(in, w) + b) (Connect4Net.py:45-46); din may be NULL */
int azg_conv3x3_relu_forward(const float* in, const float* w, const float* b, float* out, int64_t B, int Cin, int Cout,
                             int H, int W, int pad, azg_stream stream);
int azg_conv3x3_relu_backward(const float* in, const float* w, const float* out, const float* dout, float* din,
                              float* dw, float* db, int64_t B, int Cin, int Cout, int H, int W, int pad,
                              azg_stream stream);
/* loss = (-sum(target_pi*log_softmax(logits)) + sum((target_v - tanh(vraw))^2)) / norm and its gradients
 * (Connect4GNN.py:150-152, 187-193); norm = the global batch size.  All outputs on the device. */
int azg_policy_value_loss(const float* logits, const float* vraw, const float* target_pi, const float* target_v,
                          int B, int A, float norm, float* loss, float* logp, float* v, float* dlogits,
                          float* dvraw, azg_stream stream);
/* FrozenLake graph layer aggregation relu(bmm(adj, support)) with the all-ones, symmetrically normalised
 * adjacency of FrozenLakeNet.create_adjacency (FrozenLakeNet.py:8-33, 55-74) for a batch of graphs:
 * sup/out/dout/dsup [B,5,E] (unused nodes zero), counts [B] int32 nodes per graph (3..5). */
int azg_graph_mean_relu_forward(const float* sup, const int32_t* counts, int64_t B, int E, float* out,
                                azg_stream stream);
int azg_graph_mean_relu_backward(const float* dout, const float* out, const int32_t* counts, int64_t B, int E,
                                 float* dsup, azg_stream stream);
/* Grid-graph layer of the roofline sweep (BASELINE configs[4]; SURVEY section 8d.5): relu(bmm(adj, sup)) with
 * adj = D^-1/2 (A + I) D^-1/2 of the gh x gw 4-neighbour grid (operator: FrozenLakeNet.GNNLayer,
 * FrozenLakeNet.py:8-33; normalisation: create_adjacency :68-72).  sup/out [B, gh*gw, H] fp32, H % 4 == 0,
 * gh, gw >= 1, gh*gw <= 2^30.  backward: dsup = adj * (dout * (out > 0)). */
int azg_grid_aggregate_relu_forward(const float* sup, int64_t B, int gh, int gw, int H, float* out, azg_stream stream);
int azg_grid_aggregate_relu_backward(const float* dout, const float* out, int64_t B, int gh, int gw, int H,
                                     float* dsup, azg_stream stream);
/* The same layer as ONE fused tensor-core kernel (csrc/azg_grid_tc.cu): each CTA owns tiles of whole graphs,
 * X W^T runs on tcgen05 (bf16x3 = fp32-level accuracy, or bf16), the <= 5-neighbour aggregation, rowsum*bias and
 * ReLU happen in the epilogue, so the support matrix never reaches HBM.
 *   forward:         out = relu(adj * (x W^T + b))                    x, out [B, gh*gw, H] fp32
 *   backward_input:  dx  = adj * ((dout * (out > 0)) W)
 * Weights are passed as operand images made by azg_grid_pack_weights (transpose = 1 for backward_input);
 * azg_grid_tc_supported: gh, gw >= 1, gh*gw <= 256 and H in {64, 128, 256}; both layer entry points refuse any
 * other shape.  bias [H] is required.  prec: AZG_PREC_BF16X3 or AZG_PREC_BF16. */
size_t azg_grid_packed_bytes(int H);
int azg_grid_tc_supported(int gh, int gw, int H);
int azg_grid_pack_weights(const float* w, int H, int transpose, void* packed, azg_stream stream);
int azg_grid_layer_tc_forward(const float* x, const void* packed_w, const float* bias, int64_t B, int gh, int gw, int H,
                              int prec, float* out, azg_stream stream);
int azg_grid_layer_tc_backward_input(const float* dout, const float* act, const void* packed_wt, int64_t B, int gh, int gw,
                                     int H, int prec, float* dx, azg_stream stream);
/*   backward_weights: dW[o,i] = sum_r S[r,o] x[r,i], db[o] = sum_r S[r,o] over all rows r of two row-major [rows, H]
 *   matrices (S = adj * (dout * (out > 0)), from azg_grid_aggregate_relu_backward): split-K over persistent CTAs on
 *   tcgen05 with MN-major operands, fixed-order reduction of the per-CTA partials.  H in {64, 128, 256};
 *   scratch: azg_grid_dw_scratch_floats(H) floats. */
size_t azg_grid_dw_scratch_floats(int H);
int azg_grid_layer_tc_backward_weights(const float* s, const float* x, int64_t rows, int H, int prec, float* dw, float* db,
                                       float* scratch, azg_stream stream);
/* Example pipeline between self-play and training, on the device (csrc/azg_replay.cu; SURVEY section 8f.1).
 * azg_emit_examples: every stored position of finished episodes -> S symmetric training examples with signed values
 *   (Coach.py:45-49, 68-79; Connect4Game.getSymmetries :189-215, TicTacToeGame.getSymmetries :187-200).
 *   states [E] packed positions, pi [E,A] float64, player [E], game [E] -> row of result / result_tag / cur (finished
 *   games); board_perm [S,ncells] and pi_perm [S,A]: output cell d / action a takes input cell board_perm[s][d] /
 *   entry pi_perm[s][a] (tables built on the host from the reference's own numpy calls).  Outputs: example e*S+s.
 *   out_v may be NULL (positions without a value, e.g. GNN records).  frozenlake != 0: S = 1, states copied.
 * azg_gather_examples: minibatch assembly (Connect4GNN.py:141-148): boards float32 [B,n,n], pi, v float32. */
/* azg_selfplay_move: what Coach.executeEpisode does between the searches of a move and the move itself (Coach.py:36-63),
 * for every game of the arena at once: getActionProb's tail (MCTS.py:36-58: counts -> policy with CPython's compensated `sum`,
 * temp-0 tie-break from u_tie), np.random.choice (inverse CDF at u_sample), the history slot [t, g] (root state, policy, player,
 * temp-0 flag) and, with n1 / q1 / t1 / v0, expand_tree's record (MCTS.py:94-143: initial / expanded visit policies, expanded
 * value with the NEP-50 promotion order).  The uniforms come from the caller's NumPy stream, so the results equal the host
 * path's bit for bit.  slot[g] < 0 skips the game (actions[g] = -1).  flags bit 0: a game had no root visits.
 * flags bit 1: with history or record buffers, a game's slot[g] >= T; that game gets actions[g] = -1 and no row is written.
 * Record buffers need T > 0 as history buffers do. */
typedef struct azg_move_params {
  int G, A, T;              /* games, actions, history slots per game */
  const int32_t* n0;        /* [G,A] root visit counts after the numMCTSSims searches */
  const int8_t* greedy;     /* [G] temp == 0 */
  const double* u_tie;      /* [G] */
  const double* u_sample;   /* [G] */
  const uint64_t* roots;    /* [G,2] packed root states */
  const int32_t* player;    /* [G] */
  const int32_t* slot;      /* [G] history slot of this move */
  const int32_t* n1;        /* [G,A] root counts after expand_by more searches, or NULL */
  const double* q1;         /* [G,A] */
  const int8_t* t1;         /* [G,A] Q type tags */
  const float* v0;          /* [G] standard root value */
  int32_t* actions;         /* [G] out */
  uint64_t* h_states;       /* [T,G,2] out, or NULL: no history */
  double* h_pi;             /* [T,G,A] */
  int32_t* h_player;        /* [T,G] */
  int8_t* h_int;            /* [T,G] */
  double* rec_ip;           /* [T,G,A] out, or NULL: no GNN records */
  float* rec_iv;            /* [T,G] */
  double* rec_ep;           /* [T,G,A] */
  double* rec_ev;           /* [T,G] */
  int8_t* rec_evtag;        /* [T,G] */
  int32_t* flags;           /* [1] */
} azg_move_params;
int azg_selfplay_move(const azg_move_params* p, azg_stream stream);
int azg_emit_examples(int frozenlake, const uint64_t* states, const double* pi, const int32_t* player, const int32_t* game,
                      const double* result, const int8_t* result_tag, const int32_t* cur, int64_t E, int ncells, int A, int S,
                      const int32_t* board_perm, const int32_t* pi_perm, uint64_t* out_states, double* out_pi, double* out_v,
                      int8_t* out_vtag, azg_stream stream);
int azg_gather_examples(int frozenlake, const uint64_t* states, const double* pi, const double* v, const int64_t* idx, int B,
                        int ncells, int A, float* boards, float* out_pi, float* out_v, azg_stream stream);
/* GNNLayer.forward / backward at B = P + 1 > 1 (gnn_utils.py:34-74): row 0 (f0) is the target, rows
 * 1.. (path) are attended over; only the target row changes. */
typedef struct azg_gnn_layer_params {
  const float *att0_w, *att0_b, *att2_w, *att2_b; /* attention: Linear(2F,128), Linear(128,1)   */
  const float *upd0_w, *upd0_b, *upd2_w, *upd2_b; /* update_net: Linear(2F,F), Linear(F,F)      */
  const float *gate_w, *gate_b;                   /* gate: Linear(2F,F)                         */
} azg_gnn_layer_params;
typedef struct azg_gnn_layer_grads {
  float *att0_w, *att0_b, *att2_w, *att2_b, *upd0_w, *upd0_b, *upd2_w, *upd2_b, *gate_w, *gate_b;
} azg_gnn_layer_grads;
size_t azg_gnn_layer_saved_floats(int P, int F);
size_t azg_gnn_layer_scratch_floats(int P, int F);
int azg_gnn_layer_forward(const azg_gnn_layer_params* p, const float* f0, const float* path, int P, int F,
                          float* out0, float* saved, azg_stream stream);
int azg_gnn_layer_backward(const azg_gnn_layer_params* p, const float* f0, const float* path, int P, int F,
                           const float* saved, const float* d_out0, float* d_f0, const azg_gnn_layer_grads* g,
                           float* scratch, azg_stream stream);

/* ---------------------------------------------------------------- K4: search arena ------ */
/* A GPU-resident set of n_games independent transposition tables, one per game, holding what
 * MCTS.__init__ keeps in Qsa/Nsa/Ns/Ps/Es/Vs (MCTS.py:15-21).  Simulations within one game are
 * strictly sequential (bit-exact statistics); games advance in lock step. */
typedef struct azg_arena azg_arena;

/* bytes of device memory the caller must provide to azg_arena_create */
size_t azg_arena_bytes(int game, int n, int n_games, int capacity_nodes, int max_depth);
/* Every game starts with an empty table and the all-zero root state (empty board / FrozenLake start square) until
 * azg_arena_set_roots.
 * fl_map: host pointer to n*n map characters ('S','F','H','G') for AZG_GAME_FROZENLAKE, else NULL.
 * max_depth: a search call entered at depth >= max_depth returns Python-int 0 (cycle policy for
 * single-player games, DESIGN.md; never reached in two-player games when > n*n+1). */
int azg_arena_create(azg_arena** out, int game, int n, int n_games, int capacity_nodes, int max_depth,
                     double cpuct, void* device_mem, size_t device_bytes, const uint8_t* fl_map,
                     azg_stream stream);
int azg_arena_destroy(azg_arena* a);
/* Table growth: the reference's dicts are unbounded (MCTS.py:15-21) and Coach / Arena reuse one MCTS object across all
 * arenaCompare games (Coach.py:128-142), so a table can outgrow any fixed capacity.  Copies every game of `src` (nodes,
 * edges, per-game search state) into `dst`, an arena of the same game / n_games / max_depth created with a larger
 * capacity_nodes, and rebuilds the hash for the new size; node indices are preserved.  `dst` takes `src`'s search
 * semantics and root noise attachment. */
int azg_arena_copy_from(azg_arena* dst, const azg_arena* src, azg_stream stream);
/* Backup semantics of a two-player search (single-player games are unaffected).  AZG_SEARCH_REFERENCE (the default
 * of a new arena): Qsa(s,a) holds the child's value before it is negated (MCTS.py:228-240), i.e. from the point of
 * view of the player to move at the child.  AZG_SEARCH_ALPHAZERO: the value is negated first, so Qsa(s,a) is held
 * from the point of view of the player to move at s, the one who picks a.  Takes effect from the next launch;
 * any other value is refused with AZG_ERR_INVALID. */
#define AZG_SEARCH_REFERENCE 0
#define AZG_SEARCH_ALPHAZERO 1
int azg_arena_set_semantics(azg_arena* a, int semantics);
/* Dirichlet noise at the root (two-player games only; opt-in, off in a new arena).  Attaches the caller-owned device
 * buffer eta [n_games, A] float64 (NULL detaches): from the next launch on, the PUCT scores of each game's depth-0 node
 * use the prior (1 - eps) P(root, a) + eps eta[g, a], with every rounding spelled out.  The stored P is never modified,
 * so deeper visits, azg_arena_export and expand_tree read the clean prior.  Refused (AZG_ERR_INVALID): eps outside
 * [0, 1] or NaN, a buffer on a single-player arena.  `azg_arena_copy_from` carries the attachment into a grown table. */
int azg_arena_set_root_noise(azg_arena* a, const double* eta, double eps);
/* eta [n_games, A] ~ Dir(alpha) over the legal moves of each game's current root, one thread per game:
 * log Gamma(alpha) per legal action by Marsaglia-Tsang at shape alpha + 1 with the boost in log space, at most 32
 * attempts (running out sets the sticky status AZG_ERR_NOISE); uniforms from Philox4x64-10 under the key (seed, 0) at
 * counter (ids[g], action, attempt, 0), so a game's draw depends on (seed, ids[g]) alone, never on its slot.
 * eta_a = exp(lg_a - max) / sum_b exp(lg_b - max) in ascending action order; 0 on illegal actions; a terminal root gets
 * a zero row.  ids: device uint64 [n_games].  Refuses alpha <= 0 or non-finite. */
int azg_arena_draw_root_noise(azg_arena* a, uint64_t seed, const uint64_t* ids, double alpha, double* eta, azg_stream stream);
/* the generator above, exposed for parity tests against numpy.random.Philox: counters [n,4] -> words [n,4] */
int azg_philox4x64(uint64_t seed, const uint64_t* counters, int64_t n, uint64_t* words, azg_stream stream);
/* Rollout baseline: the leaf evaluation of an MCTS player that needs no network.  For every row i below the leaf count,
 * v[i] = (sum of `playouts` outcomes) / playouts (float32, one rounding; the sum is an exact integer) and pi [rows, A] =
 * 1/k (float32) on the k legal moves (getValidMoves) of states[i], 0 elsewhere.  An outcome is +1 / 0 / -1 for the player
 * to move at states[i] after uniformly random play to the end (a draw, Connect4's 1e-4 included, is 0; a terminal state
 * is its own outcome); ply t of playout p reads word t % 4 of the Philox4x64-10 block at counter
 * (mine, theirs, (games[i] << 32) | p, t / 4) under the key (seed, 1) and plays the j-th legal action in ascending order,
 * j = mulhi64(word, k).  games: device int32 [rows], the game each row belongs to, or NULL = the row index.  count: device
 * int32 [1], the compact leaf count (rows at or past it are not written), or NULL = all rows.  Connect4 n = 4..8 and
 * TicTacToe n = 3..5; playouts in [1, 4096]; anything else, and null pointers with rows > 0, is refused (AZG_ERR_INVALID). */
int azg_rollout_eval(int game, int n, const uint64_t* states, const int32_t* games, int64_t rows, const int32_t* count,
                     int playouts, uint64_t seed, float* pi, float* v, azg_stream stream);
int azg_arena_action_size(const azg_arena* a);
/* new MCTS object for the listed games (Coach.py:96): clear their tables.  game_ids: device
 * int32 [count], or NULL = all games. */
int azg_arena_reset(azg_arena* a, const int32_t* game_ids, int count, azg_stream stream);
/* canonical root positions of every game, states [n_games,2] */
int azg_arena_set_roots(azg_arena* a, const uint64_t* states, azg_stream stream);
int azg_arena_get_roots(azg_arena* a, uint64_t* states, azg_stream stream);
/* grant every game `n_sims` more MCTS.search calls from its root (MCTS.py:33-34) */
int azg_arena_begin(azg_arena* a, int n_sims, azg_stream stream);
/* MCTS.search descend phase (MCTS.py:151-226) for every game with simulations left: runs
 * searches until one reaches an unexpanded non-terminal leaf (searches that end on a terminal
 * state are backed up immediately, MCTS.py:154-157).  Writes leaf_states [n_games,2] and
 * leaf_mask [n_games] (1 = this game waits for a prediction of leaf_states[g]). */
int azg_arena_select(azg_arena* a, uint64_t* leaf_states, int32_t* leaf_mask, azg_stream stream);
/* MCTS.search leaf + backup phase (MCTS.py:162-193, 228-240) for games with leaf_mask set:
 * pi [n_games,A] fp32 and v [n_games] fp32 are the predictions for leaf_states. */
int azg_arena_expand_backup(azg_arena* a, const float* pi, const float* v, azg_stream stream);
/* Compacted variants (no host synchronisation): the leaves that wait for a prediction are written
 * densely -- leaf_states [count,2], leaf_game [count] = owning game, leaf_count [1] on the device --
 * so the networks only evaluate `count` positions (azg_c4_forward_dyn reads the count on the device).
 * expand_backup_compact consumes pi [count,A] / v [count] in that order. */
int azg_arena_select_compact(azg_arena* a, uint64_t* leaf_states, int32_t* leaf_mask, int32_t* leaf_game,
                             int32_t* leaf_count, azg_stream stream);
int azg_arena_expand_backup_compact(azg_arena* a, const float* pi, const float* v, const int32_t* leaf_game,
                                    const int32_t* leaf_count, azg_stream stream);
/* root edge statistics for getActionProb / expand_tree (MCTS.py:36-37, 79-81, 121-143):
 * N [n_games,A] int32, Q [n_games,A] float64, qtag [n_games,A] int8 (AZG_TAG_*). */
int azg_arena_root_stats(azg_arena* a, int32_t* N, double* Q, int8_t* qtag, azg_stream stream);
/* play actions[g] (Coach.py:63-66): root <- canonical(next(root, a)); ended [n_games] float64 =
 * getGameEnded of the new root for the player to move (0 = running); ended_tag as AZG_TAG_*.
 * actions[g] < 0 leaves game g untouched. */
int azg_arena_advance(azg_arena* a, const int32_t* actions, double* ended, int8_t* ended_tag,
                      azg_stream stream);
/* sticky per-game error flags (0 = fine, AZG_ERR_CAPACITY ...), int32 [n_games] */
int azg_arena_status(azg_arena* a, int32_t* status, azg_stream stream);
/* test read-back of one game's table (the reference's public dicts): returns the node count via
 * host pointer n_nodes (synchronises `stream`).  Arrays are sized for capacity_nodes rows:
 * keys [cap,2] u64, es [cap] f64 (0 = not ended), es_tag [cap] i8, ns [cap] i32 (-1 = not in Ns/Ps),
 * valids [cap] u32 bit mask (Vs), ptag [cap] i8 (dtype of Ps[s]: 0 float64, 1 float32), P [cap,A] f64, Q [cap,A] f64, qtag [cap,A] i8, N [cap,A] i32. */
int azg_arena_export(azg_arena* a, int game_index, int* n_nodes, uint64_t* keys, double* es, int8_t* es_tag,
                     int32_t* ns, uint32_t* valids, int8_t* ptag, double* P, double* Q, int8_t* qtag, int32_t* N,
                     azg_stream stream);

/* rules as the arena applies them, exposed for parity tests against
 * Connect4Game.py:143-187 / TicTacToeGame.py:145-183 / FrozenLakeGame.py:88-187.
 * valids [B] u32 masks, ended [B] f64 (+tags), next [B,A,2] canonical successor states. */
int azg_rules_eval(int game, int n, const uint8_t* fl_map_host, const uint64_t* states, int64_t B,
                   uint32_t* valids, double* ended, int8_t* ended_tag, uint64_t* next, azg_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* AZGNN_B200_H */
