// azg_train.cu -- K3: forward/backward pieces of the training step (fp32, CUDA cores).
//
//   Connect4GNNWrapper.train / TicTacToeGNNWrapper.train   connect4/Connect4GNN.py:122-197
//   GNNLayer.forward at B > 1 (row 0 = target, rows 1.. = path states)   gnn_utils.py:34-74
//   losses  -sum(pi*logp)/B + sum((v_t - v)^2)/B                          Connect4GNN.py:150-152
//
// The batch is 64 rows: every contraction here is either a skinny GEMM against a big weight
// matrix or a rank-1 update of one, i.e. bound by streaming the 39-79 MB weight / gradient
// tensors once (SURVEY section 8d "K3: HBM bound").  One generic tiled SGEMM with arbitrary
// transposes and leading dimensions serves all of them; the rest are small fused element-wise
// kernels.  torch.autograd.Function wrappers (training.py) only route tensors.
#include "azg_common.cuh"

namespace {

inline int grid_for(int64_t n, int threads) { return (int)((n + threads - 1) / threads); }

// ------------------------------------------------------------------------------ generic SGEMM
// C[M,N] = op(A)[M,K] . op(B)[K,N] + beta * C     (row-major, leading dimensions lda/ldb/ldc)
//   TA = 0: A is [M,K] (A[m*lda + k]);  TA = 1: A is [K,M] (A[k*lda + m])
//   TB = 0: B is [K,N] (B[k*ldb + n]);  TB = 1: B is [N,K] (B[n*ldb + k])
constexpr int GT = 64, GK = 16;

template <bool TA, bool TB>
__global__ void __launch_bounds__(256) gemm_generic_kernel(int64_t M, int N, int K, const float* __restrict__ A, int64_t lda,
                                                           const float* __restrict__ B, int64_t ldb, float* __restrict__ C,
                                                           int64_t ldc, float beta, int kper, int64_t zstride_c) {
  // split-K: blockIdx.z owns the contraction range [z*kper, min(K, (z+1)*kper)) and its own C slab
  __shared__ float As[GK][GT + 4];
  __shared__ float Bs[GK][GT + 4];
  const int tid = threadIdx.x;
  const int64_t m0 = (int64_t)blockIdx.x * GT;  // M on grid.x (2^31 limit), N on grid.y
  const int n0 = blockIdx.y * GT;
  const int tx = tid & 15, ty = tid >> 4;
  float acc[4][4] = {};
  const int kbeg = blockIdx.z * kper;
  if (K > kbeg + kper) K = kbeg + kper;
  C += (size_t)blockIdx.z * zstride_c;
  for (int k0 = kbeg; k0 < K; k0 += GK) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int m, k;
      if (TA) { m = tid & 63; k = (tid >> 6) + 4 * i; } else { k = tid & 15; m = (tid >> 4) + 16 * i; }
      const int64_t gm = m0 + m;
      const int gk = k0 + k;
      float v = 0.0f;
      if (gm < M && gk < K) v = TA ? A[(int64_t)gk * lda + gm] : A[gm * lda + gk];
      As[k][m] = v;
      int n, kb;
      if (TB) { kb = tid & 15; n = (tid >> 4) + 16 * i; } else { n = tid & 63; kb = (tid >> 6) + 4 * i; }
      const int gn = n0 + n, gkb = k0 + kb;
      float w = 0.0f;
      if (gn < N && gkb < K) w = TB ? B[(int64_t)gn * ldb + gkb] : B[(int64_t)gkb * ldb + gn];
      Bs[kb][n] = w;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < GK; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        a[i] = As[kk][ty * 4 + i];
        b[i] = Bs[kk][tx * 4 + i];
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= N) continue;
      float* c = C + m * ldc + n;
      *c = (beta == 0.0f) ? acc[i][j] : acc[i][j] + beta * (*c);
    }
  }
}

int gemm_split(bool ta, bool tb, int64_t M, int N, int K, const float* A, int64_t lda, const float* B, int64_t ldb, float* C,
               int64_t ldc, float beta, int splits, int64_t zstride_c, cudaStream_t st) {
  if (M <= 0 || N <= 0) return AZG_OK;
  const int kper = (int)(((int64_t)(K + splits - 1) / splits + GK - 1) / GK * GK);
  dim3 grid((unsigned)((M + GT - 1) / GT), (N + GT - 1) / GT, splits);
  AZG_REQUIRE(grid.y <= 65535 && splits <= 65535, "gemm: N too large");
  if (ta && tb) gemm_generic_kernel<true, true><<<grid, 256, 0, st>>>(M, N, K, A, lda, B, ldb, C, ldc, beta, kper, zstride_c);
  else if (ta) gemm_generic_kernel<true, false><<<grid, 256, 0, st>>>(M, N, K, A, lda, B, ldb, C, ldc, beta, kper, zstride_c);
  else if (tb) gemm_generic_kernel<false, true><<<grid, 256, 0, st>>>(M, N, K, A, lda, B, ldb, C, ldc, beta, kper, zstride_c);
  else gemm_generic_kernel<false, false><<<grid, 256, 0, st>>>(M, N, K, A, lda, B, ldb, C, ldc, beta, kper, zstride_c);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

// ------------------------------------------------------------------------------ tiled SGEMM, asynchronous copies
// Same contract as gemm_generic_kernel for operands whose rows are 16-byte aligned (leading dimensions and
// base pointers multiples of 4 floats): 64 x 128 x 32 tiles, 3-stage cp.async pipeline that lands the operands
// in shared memory in their HBM orientation (no register staging, no transposing stores), 8 x 4 outputs per
// thread.  A warp owns 8 rows (its A reads are broadcasts), lanes spread over the 128 columns.
//   AK: A[m*lda + k] (k contiguous), else A[k*lda + m];   BK: B[n*ldb + k], else B[k*ldb + n]
constexpr int TM = 64, TN = 128, TKC = 32, TST = 3;
template <bool AK, bool BK>
struct TileSmem {
  static constexpr int A_ROWS = AK ? TM : TKC, A_LD = (AK ? TKC : TM) + 4;
  static constexpr int B_ROWS = BK ? TN : TKC, B_LD = (BK ? TKC : TN) + 4;
  static constexpr int A_FLOATS = A_ROWS * A_LD, B_FLOATS = B_ROWS * B_LD;
  static constexpr int STAGE_FLOATS = A_FLOATS + B_FLOATS;
  static constexpr int BYTES = TST * STAGE_FLOATS * 4;
};

__device__ __forceinline__ void cp_async16(float* smem_dst, const float* gsrc, int src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc),
               "r"(src_bytes)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

template <bool AK, bool BK>
__global__ void __launch_bounds__(256) gemm_tile_kernel(int64_t M, int N, int K, const float* __restrict__ A, int64_t lda,
                                                        const float* __restrict__ B, int64_t ldb, float* __restrict__ C,
                                                        int64_t ldc, float beta, int kper, int64_t zstride_c) {
  using S = TileSmem<AK, BK>;
  extern __shared__ __align__(16) float tile_smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t m0 = (int64_t)blockIdx.x * TM;
  const int n0 = blockIdx.y * TN;
  const int kbeg = blockIdx.z * kper;
  const int kend = K < kbeg + kper ? K : kbeg + kper;
  C += (size_t)blockIdx.z * zstride_c;
  const int chunks = kend > kbeg ? (kend - kbeg + TKC - 1) / TKC : 0;

  auto issue = [&](int chunk, int stage) {
    float* As = tile_smem + stage * S::STAGE_FLOATS;
    float* Bs = As + S::A_FLOATS;
    const int k0 = kbeg + chunk * TKC;
    // A: 512 float4
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int f = tid + 256 * i;
      if (AK) {
        const int r = f >> 3, c = (f & 7) * 4;
        const int64_t m = m0 + r;
        const int k = k0 + c;
        int valid = (m < M) ? (kend - k) : 0;
        valid = valid < 0 ? 0 : (valid > 4 ? 4 : valid);
        cp_async16(As + r * S::A_LD + c, valid ? A + m * lda + k : A, valid * 4);
      } else {
        const int r = f >> 4, c = (f & 15) * 4;
        const int k = k0 + r;
        const int64_t m = m0 + c;
        int64_t valid = (k < kend) ? (M - m) : 0;
        valid = valid < 0 ? 0 : (valid > 4 ? 4 : valid);
        cp_async16(As + r * S::A_LD + c, valid ? A + (int64_t)k * lda + m : A, (int)valid * 4);
      }
    }
    // B: 1024 float4
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int f = tid + 256 * i;
      if (BK) {
        const int r = f >> 3, c = (f & 7) * 4;
        const int n = n0 + r;
        const int k = k0 + c;
        int valid = (n < N) ? (kend - k) : 0;
        valid = valid < 0 ? 0 : (valid > 4 ? 4 : valid);
        cp_async16(Bs + r * S::B_LD + c, valid ? B + (int64_t)n * ldb + k : B, valid * 4);
      } else {
        const int r = f >> 5, c = (f & 31) * 4;
        const int k = k0 + r;
        const int n = n0 + c;
        int valid = (k < kend) ? (N - n) : 0;
        valid = valid < 0 ? 0 : (valid > 4 ? 4 : valid);
        cp_async16(Bs + r * S::B_LD + c, valid ? B + (int64_t)k * ldb + n : B, valid * 4);
      }
    }
  };

  float acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;

#pragma unroll
  for (int s = 0; s < TST - 1; ++s) {
    if (s < chunks) issue(s, s);
    cp_async_commit();
  }
  for (int c = 0; c < chunks; ++c) {
    cp_async_wait<TST - 2>();
    __syncthreads();
    if (c + TST - 1 < chunks) issue(c + TST - 1, (c + TST - 1) % TST);
    cp_async_commit();
    const float* As = tile_smem + (c % TST) * S::STAGE_FLOATS;
    const float* Bs = As + S::A_FLOATS;
#pragma unroll
    for (int k4 = 0; k4 < TKC; k4 += 4) {
      float a[8][4], b[4][4];  // [row][kk], [col][kk]
      if (AK) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 v = *reinterpret_cast<const float4*>(As + (warp * 8 + i) * S::A_LD + k4);
          a[i][0] = v.x; a[i][1] = v.y; a[i][2] = v.z; a[i][3] = v.w;
        }
      } else {
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          const float4 v0 = *reinterpret_cast<const float4*>(As + (k4 + kk) * S::A_LD + warp * 8);
          const float4 v1 = *reinterpret_cast<const float4*>(As + (k4 + kk) * S::A_LD + warp * 8 + 4);
          a[0][kk] = v0.x; a[1][kk] = v0.y; a[2][kk] = v0.z; a[3][kk] = v0.w;
          a[4][kk] = v1.x; a[5][kk] = v1.y; a[6][kk] = v1.z; a[7][kk] = v1.w;
        }
      }
      if (BK) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 v = *reinterpret_cast<const float4*>(Bs + (lane + 32 * j) * S::B_LD + k4);
          b[j][0] = v.x; b[j][1] = v.y; b[j][2] = v.z; b[j][3] = v.w;
        }
      } else {
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          const float4 v = *reinterpret_cast<const float4*>(Bs + (k4 + kk) * S::B_LD + lane * 4);
          b[0][kk] = v.x; b[1][kk] = v.y; b[2][kk] = v.z; b[3][kk] = v.w;
        }
      }
#pragma unroll
      for (int kk = 0; kk < 4; ++kk)
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i][kk], b[j][kk], acc[i][j]);
    }
  }
  cp_async_wait<0>();
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int64_t m = m0 + warp * 8 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + (BK ? lane + 32 * j : lane * 4 + j);
      if (n >= N) continue;
      float* c = C + m * ldc + n;
      *c = (beta == 0.0f) ? acc[i][j] : acc[i][j] + beta * (*c);
    }
  }
}

inline bool tile_ok(const float* A, int64_t lda, const float* B, int64_t ldb) {
  return ((uintptr_t)A & 15u) == 0 && ((uintptr_t)B & 15u) == 0 && (lda & 3) == 0 && (ldb & 3) == 0;
}

template <bool AK, bool BK>
int launch_tile(dim3 grid, int64_t M, int N, int K, const float* A, int64_t lda, const float* B, int64_t ldb, float* C,
                int64_t ldc, float beta, int kper, int64_t zstride_c, cudaStream_t st) {
  static bool attr = false;
  if (!attr) {
    AZG_CUDA_CHECK(cudaFuncSetAttribute(gemm_tile_kernel<AK, BK>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        TileSmem<AK, BK>::BYTES));
    attr = true;
  }
  gemm_tile_kernel<AK, BK><<<grid, 256, TileSmem<AK, BK>::BYTES, st>>>(M, N, K, A, lda, B, ldb, C, ldc, beta, kper, zstride_c);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

// split-K launch of the tiled kernel (slab z of C = partial product over k range z); ta/tb as in gemm_split
int gemm_tile_split(bool ta, bool tb, int64_t M, int N, int K, const float* A, int64_t lda, const float* B, int64_t ldb, float* C,
                    int64_t ldc, float beta, int splits, int64_t zstride_c, cudaStream_t st) {
  if (M <= 0 || N <= 0) return AZG_OK;
  const int kper = (int)(((int64_t)(K + splits - 1) / splits + TKC - 1) / TKC * TKC);
  dim3 grid((unsigned)((M + TM - 1) / TM), (N + TN - 1) / TN, splits);
  AZG_REQUIRE(grid.y <= 65535 && splits <= 65535, "gemm: N too large");
  // AK = A is [M,K] row-major = !ta;  BK = B is [N,K] row-major = tb
  if (!ta && tb) return launch_tile<true, true>(grid, M, N, K, A, lda, B, ldb, C, ldc, beta, kper, zstride_c, st);
  if (!ta && !tb) return launch_tile<true, false>(grid, M, N, K, A, lda, B, ldb, C, ldc, beta, kper, zstride_c, st);
  if (ta && tb) return launch_tile<false, true>(grid, M, N, K, A, lda, B, ldb, C, ldc, beta, kper, zstride_c, st);
  return launch_tile<false, false>(grid, M, N, K, A, lda, B, ldb, C, ldc, beta, kper, zstride_c, st);
}

// ------------------------------------------------------------------------------ weight streaming, M = 1
// The GNNLayer works on ONE target row against 39-79 MB weight matrices (gnn_utils.py:66-71), so its
// contractions are matrix-vector products / rank-1 updates whose only cost is streaming the matrix once.
__device__ __forceinline__ float warp_sum_f(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float dot4(float4 a, float4 b, float acc) {
  acc = fmaf(a.x, b.x, acc);
  acc = fmaf(a.y, b.y, acc);
  acc = fmaf(a.z, b.z, acc);
  return fmaf(a.w, b.w, acc);
}

// y[n] = act(W[n, :K] . x + bias[n]): one warp per GR rows, 128-bit streaming loads (8 x GR in flight per lane);
// x (<= 25 KB) is re-read through L1 by every warp.  Fixed summation order per lane + shuffle tree: deterministic.
constexpr int GR = 2, GEMV_WARPS = 1;  // one-warp CTAs: 1568 CTAs over 148 SMs balance to within 4 % (four-warp CTAs: 13 %)
__global__ void __launch_bounds__(GEMV_WARPS * 32) gemv_rows_kernel(const float* __restrict__ W, int64_t ldw,
                                                                    const float* __restrict__ x, const float* __restrict__ bias,
                                                                    float* __restrict__ y, int N, int K, int relu) {
  const int K4 = K >> 2;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n0 = (blockIdx.x * GEMV_WARPS + warp) * GR;
  if (n0 >= N) return;
  const float4* x4 = reinterpret_cast<const float4*>(x);
  const float4* w[GR];
  float acc[GR];
#pragma unroll
  for (int r = 0; r < GR; ++r) {
    const int n = n0 + r < N ? n0 + r : N - 1;
    w[r] = reinterpret_cast<const float4*>(W + (int64_t)n * ldw);
    acc[r] = 0.0f;
  }
  int k = lane;
  for (; k + 7 * 32 < K4; k += 8 * 32) {
    float4 wv[GR][8];
#pragma unroll
    for (int u = 0; u < 8; ++u)
#pragma unroll
      for (int r = 0; r < GR; ++r) wv[r][u] = __ldcs(w[r] + k + 32 * u);
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const float4 xv = __ldg(x4 + k + 32 * u);
#pragma unroll
      for (int r = 0; r < GR; ++r) acc[r] = dot4(wv[r][u], xv, acc[r]);
    }
  }
  for (; k < K4; k += 32) {
    const float4 xv = __ldg(x4 + k);
#pragma unroll
    for (int r = 0; r < GR; ++r) acc[r] = dot4(__ldcs(w[r] + k), xv, acc[r]);
  }
#pragma unroll
  for (int r = 0; r < GR; ++r) {
    const float s = warp_sum_f(acc[r]);
    if (lane == 0 && n0 + r < N) {
      const float v = s + (bias ? bias[n0 + r] : 0.0f);
      y[n0 + r] = relu ? fmaxf(v, 0.0f) : v;
    }
  }
}

// One pass over a [N, K] weight matrix for the backward of y = W x with upstream gradient g [N]:
//   DW: dW[n, k] = g[n] * x[k]                       (written, never read)
//   DX: part[chunk, k] = sum_{n in chunk} g[n] W[n, k]  (reduced over chunks in fixed order afterwards)
// CTA = 256 threads x float4 = 1024 columns, R1_ROWS rows.
constexpr int R1_ROWS = 32;
template <bool DX, bool DW>
__global__ void __launch_bounds__(256) rank1_bwd_kernel(const float* __restrict__ W, int64_t ldw, const float* __restrict__ g,
                                                        const float* __restrict__ x, float* __restrict__ dW, int64_t lddw,
                                                        float* __restrict__ part, int N, int K) {
  __shared__ float gs[R1_ROWS];
  const int n0 = blockIdx.y * R1_ROWS;
  const int rows = N - n0 < R1_ROWS ? N - n0 : R1_ROWS;
  if (threadIdx.x < R1_ROWS) gs[threadIdx.x] = threadIdx.x < rows ? g[n0 + threadIdx.x] : 0.0f;
  __syncthreads();
  const int k = (blockIdx.x * 256 + threadIdx.x) * 4;
  if (k >= K) return;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  float4 xv = make_float4(0.f, 0.f, 0.f, 0.f);
  if (DW) xv = *reinterpret_cast<const float4*>(x + k);
  const float* wp = W + (int64_t)n0 * ldw + k;
  float* dp = dW + (int64_t)n0 * lddw + k;
#pragma unroll 8
  for (int r = 0; r < rows; ++r) {
    const float gn = gs[r];
    if (DX) {
      const float4 w = __ldcs(reinterpret_cast<const float4*>(wp + (int64_t)r * ldw));
      acc.x = fmaf(gn, w.x, acc.x);
      acc.y = fmaf(gn, w.y, acc.y);
      acc.z = fmaf(gn, w.z, acc.z);
      acc.w = fmaf(gn, w.w, acc.w);
    }
    if (DW) __stcs(reinterpret_cast<float4*>(dp + (int64_t)r * lddw), make_float4(gn * xv.x, gn * xv.y, gn * xv.z, gn * xv.w));
  }
  if (DX) *reinterpret_cast<float4*>(part + (size_t)blockIdx.y * K + k) = acc;
}

// out[m, n] = beta * out[m, n] + sum_z part[z][m, n]   (fixed order; out has leading dimension ldc)
__global__ void reduce_parts_kernel(const float* __restrict__ part, int splits, int64_t M, int N, float* __restrict__ out,
                                    int64_t ldc, float beta) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M * N) return;
  float s = 0.0f;
  for (int z = 0; z < splits; ++z) s += part[(size_t)z * M * N + i];
  float* o = out + (i / N) * ldc + (i % N);
  *o = beta == 0.0f ? s : s + beta * (*o);
}

inline bool aligned16(const void* p) { return ((uintptr_t)p & 15u) == 0; }

// stream-ordered scratch for split reductions
struct Scratch {
  float* p = nullptr;
  cudaStream_t st;
  explicit Scratch(cudaStream_t s) : st(s) {}
  int get(size_t floats) { return cudaMallocAsync((void**)&p, sizeof(float) * floats, st) == cudaSuccess ? 0 : 1; }
  ~Scratch() {
    if (p) cudaFreeAsync(p, st);
  }
};

// y[N] = act(W[N, K] x + bias)
int gemv_rows(const float* W, int64_t ldw, const float* x, const float* bias, float* y, int N, int K, int relu, cudaStream_t st) {
  gemv_rows_kernel<<<grid_for(N, GEMV_WARPS * GR), GEMV_WARPS * 32, 0, st>>>(W, ldw, x, bias, y, N, K, relu);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}
inline bool gemv_rows_ok(const float* W, int64_t ldw, const float* x, int K) {
  return (K & 3) == 0 && (ldw & 3) == 0 && aligned16(W) && aligned16(x);
}

// backward of y = W x (W [N, K]): dW = g x^T (optional), dx = beta * dx + W^T g (optional)
int rank1_bwd(const float* W, int64_t ldw, const float* g, const float* x, float* dW, int64_t lddw, float* dx, float beta, int N,
              int K, cudaStream_t st) {
  dim3 grid(grid_for(K, 1024), grid_for(N, R1_ROWS));
  Scratch sc(st);
  if (dx && sc.get((size_t)grid.y * K)) {
    azg_set_error("rank1_bwd: scratch allocation failed");
    return AZG_ERR_CUDA;
  }
  if (dx && dW) rank1_bwd_kernel<true, true><<<grid, 256, 0, st>>>(W, ldw, g, x, dW, lddw, sc.p, N, K);
  else if (dx) rank1_bwd_kernel<true, false><<<grid, 256, 0, st>>>(W, ldw, g, x, nullptr, 0, sc.p, N, K);
  else if (dW) rank1_bwd_kernel<false, true><<<grid, 256, 0, st>>>(nullptr, 0, g, x, dW, lddw, nullptr, N, K);
  else return AZG_OK;
  AZG_LAUNCH_CHECK();
  if (dx) {
    reduce_parts_kernel<<<grid_for(K, 256), 256, 0, st>>>(sc.p, (int)grid.y, 1, K, dx, K, beta);
    AZG_LAUNCH_CHECK();
  }
  return AZG_OK;
}
inline bool rank1_ok(const float* W, int64_t ldw, const float* x, const float* dW, int64_t lddw, int K) {
  return (K & 3) == 0 && (!W || ((ldw & 3) == 0 && aligned16(W))) && (!dW || ((lddw & 3) == 0 && aligned16(dW) && aligned16(x)));
}

// C = op(A) op(B) + beta C with shape-driven dispatch:
//   M = 1 against a [N, K] matrix        -> gemv_rows (one streaming pass)
//   M = 1 against a [K, N] matrix        -> rank1_bwd DX pass
//   K = 1 (outer product)                -> rank1_bwd DW pass
//   few output tiles but a long K        -> split-K over enough CTAs to fill the SMs, fixed-order reduction
int gemm(bool ta, bool tb, int64_t M, int N, int K, const float* A, int64_t lda, const float* B, int64_t ldb, float* C,
         int64_t ldc, float beta, cudaStream_t st) {
  if (M <= 0 || N <= 0) return AZG_OK;
  if (M == 1 && !ta && tb && beta == 0.0f && gemv_rows_ok(B, ldb, A, K)) return gemv_rows(B, ldb, A, nullptr, C, N, K, 0, st);
  if (M == 1 && !ta && !tb && (beta == 0.0f || beta == 1.0f) && K >= 64 && rank1_ok(B, ldb, nullptr, nullptr, 0, N) && aligned16(C))
    return rank1_bwd(B, ldb, A, nullptr, nullptr, 0, C, beta, K, N, st);  // C[n] = sum_k A[k] B[k, n]
  if (K == 1 && ta && !tb && beta == 0.0f && rank1_ok(nullptr, 0, B, C, ldc, N))
    return rank1_bwd(nullptr, 0, A, B, C, ldc, nullptr, 0.0f, (int)M, N, st);  // C[m, n] = A[m] B[n]
  const bool tiled = tile_ok(A, lda, B, ldb);
  const int64_t ctas = tiled ? ((M + TM - 1) / TM) * ((N + TN - 1) / TN) : ((M + GT - 1) / GT) * ((N + GT - 1) / GT);
  if (ctas < 148 && K >= 256) {
    int splits = (int)((296 + ctas - 1) / ctas);
    if (splits > K / 64) splits = K / 64;
    if (splits > 1) {
      Scratch sc(st);
      if (sc.get((size_t)splits * M * N)) {
        azg_set_error("gemm: scratch allocation failed");
        return AZG_ERR_CUDA;
      }
      int rc = tiled ? gemm_tile_split(ta, tb, M, N, K, A, lda, B, ldb, sc.p, N, 0.0f, splits, M * (int64_t)N, st)
                     : gemm_split(ta, tb, M, N, K, A, lda, B, ldb, sc.p, N, 0.0f, splits, M * (int64_t)N, st);
      if (rc) return rc;
      reduce_parts_kernel<<<grid_for(M * N, 256), 256, 0, st>>>(sc.p, splits, M, N, C, ldc, beta);
      AZG_LAUNCH_CHECK();
      return AZG_OK;
    }
  }
  if (tiled) return gemm_tile_split(ta, tb, M, N, K, A, lda, B, ldb, C, ldc, beta, 1, 0, st);
  return gemm_split(ta, tb, M, N, K, A, lda, B, ldb, C, ldc, beta, 1, 0, st);
}

// out[i] = sum_s part[s*n + i] in fixed order (deterministic split-K reduction)
__global__ void reduce_splits_kernel(const float* __restrict__ part, int splits, int64_t n, float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s = 0.0f;
  for (int z = 0; z < splits; ++z) s += part[(size_t)z * n + i];
  out[i] = s;
}

// partial column sums: blockIdx.y owns rows [y*rper, (y+1)*rper)
__global__ void col_sum_split_kernel(const float* __restrict__ x, int64_t rows, int cols, int64_t rper, float* __restrict__ part) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  const int64_t r0 = (int64_t)blockIdx.y * rper, r1 = r0 + rper < rows ? r0 + rper : rows;
  float s = 0.0f;
  for (int64_t r = r0; r < r1; ++r) s += x[r * cols + c];
  part[(size_t)blockIdx.y * cols + c] = s;
}

// ------------------------------------------------------------------------------ element-wise
__global__ void mul_kernel(const float* a, const float* b, float* o, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) o[i] = a[i] * b[i];
}
__global__ void relu_bwd_kernel(const float* dy, const float* y, float* dx, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dx[i] = y[i] > 0.0f ? dy[i] : 0.0f;
}
__global__ void add_bias_act_kernel(float* x, const float* bias, int64_t rows, int cols, int relu) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * cols) return;
  float v = x[i] + (bias ? bias[i % cols] : 0.0f);
  x[i] = relu ? fmaxf(v, 0.0f) : v;
}
// out[c] = sum over rows of x[r, c] (bias gradients); one thread per column, fixed order
__global__ void col_sum_kernel(const float* x, int64_t rows, int cols, int64_t ld, float* out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  float s = 0.0f;
  for (int64_t r = 0; r < rows; ++r) s += x[r * ld + c];
  out[c] = s;
}
__global__ void axpy_kernel(float* y, const float* x, int64_t n) {  // y += x
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) y[i] += x[i];
}

// ------------------------------------------------------------------------------ conv backward
// g = dout * (out > 0);  dw[co,ci,kx,ky] = sum_{b,ox,oy} g * in[b,ci,ox+kx-p,oy+ky-p];  db[co] = sum g
__global__ void conv_bwd_weight_kernel(const float* __restrict__ in, const float* __restrict__ out,
                                       const float* __restrict__ dout, float* __restrict__ dw, float* __restrict__ db,
                                       int64_t B, int Cin, int Cout, int H, int W, int pad) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int Ho = H + 2 * pad - 2, Wo = W + 2 * pad - 2;
  const int total = Cout * Cin * 9;
  if (idx < total) {
    const int co = idx / (Cin * 9), r = idx % (Cin * 9), ci = r / 9, kx = (r % 9) / 3, ky = r % 3;
    float s = 0.0f;
    for (int64_t b = 0; b < B; ++b)
      for (int ox = 0; ox < Ho; ++ox) {
        const int x = ox + kx - pad;
        if (x < 0 || x >= H) continue;
        for (int oy = 0; oy < Wo; ++oy) {
          const int y = oy + ky - pad;
          if (y < 0 || y >= W) continue;
          const int64_t o = ((b * Cout + co) * Ho + ox) * Wo + oy;
          if (out[o] > 0.0f) s = fmaf(dout[o], in[((b * Cin + ci) * H + x) * W + y], s);
        }
      }
    dw[idx] = s;
  } else if (idx < total + Cout) {
    const int co = idx - total;
    float s = 0.0f;
    for (int64_t b = 0; b < B; ++b)
      for (int p = 0; p < Ho * Wo; ++p) {
        const int64_t o = (b * Cout + co) * Ho * Wo + p;
        if (out[o] > 0.0f) s += dout[o];
      }
    db[co] = s;
  }
}

// din[b,ci,x,y] = sum_{co,kx,ky} g[b,co,x-kx+p,y-ky+p] * w[co,ci,kx,ky]
__global__ void conv_bwd_data_kernel(const float* __restrict__ w, const float* __restrict__ out,
                                     const float* __restrict__ dout, float* __restrict__ din, int64_t B, int Cin, int Cout,
                                     int H, int W, int pad) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * Cin * H * W) return;
  const int Ho = H + 2 * pad - 2, Wo = W + 2 * pad - 2;
  const int y = (int)(idx % W), x = (int)((idx / W) % H), ci = (int)((idx / ((int64_t)W * H)) % Cin);
  const int64_t b = idx / ((int64_t)W * H * Cin);
  float s = 0.0f;
  for (int co = 0; co < Cout; ++co)
    for (int kx = 0; kx < 3; ++kx) {
      const int ox = x - kx + pad;
      if (ox < 0 || ox >= Ho) continue;
      for (int ky = 0; ky < 3; ++ky) {
        const int oy = y - ky + pad;
        if (oy < 0 || oy >= Wo) continue;
        const int64_t o = ((b * Cout + co) * Ho + ox) * Wo + oy;
        if (out[o] > 0.0f) s = fmaf(dout[o], w[((size_t)co * Cin + ci) * 9 + kx * 3 + ky], s);
      }
    }
  din[idx] = s;
}

// conv backward as contractions over (board, output cell): one pass writes
//   gt [(b,p), Cout]   = dout * (out > 0)        (ReLU gate applied, transposed so that (b,p) is the row index)
//   col[(b,p), Cin*9]  = 3x3 patch of `in` around output cell p (zero outside the board)
// then dw = gt^T col (split-K GEMM), db = column sums of gt, dcol = gt w, din = col2im(dcol).
__global__ void conv_bwd_pack_kernel(const float* __restrict__ in, const float* __restrict__ out, const float* __restrict__ dout,
                                     float* __restrict__ gt, float* __restrict__ col, int64_t B, int Cin, int Cout, int H, int W,
                                     int pad) {
  const int Ho = H + 2 * pad - 2, Wo = W + 2 * pad - 2, P = Ho * Wo, C9 = Cin * 9;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n_g = B * P * Cout, n_c = B * P * C9;
  if (i < n_g) {
    const int co = (int)(i % Cout);
    const int64_t bp = i / Cout;
    const int64_t o = ((bp / P) * Cout + co) * P + bp % P;
    gt[i] = out[o] > 0.0f ? dout[o] : 0.0f;
  } else if (i < n_g + n_c) {
    const int64_t j = i - n_g;
    const int r = (int)(j % C9), ci = r / 9, kx = (r % 9) / 3, ky = r % 3;
    const int64_t bp = j / C9;
    const int p = (int)(bp % P), x = p / Wo + kx - pad, y = p % Wo + ky - pad;
    col[j] = (x >= 0 && x < H && y >= 0 && y < W) ? in[(((bp / P) * Cin + ci) * H + x) * W + y] : 0.0f;
  }
}

// din[b,ci,x,y] = sum_{kx,ky} dcol[(b, x-kx+pad, y-ky+pad), ci*9 + kx*3 + ky]
__global__ void conv_col2im_kernel(const float* __restrict__ dcol, float* __restrict__ din, int64_t B, int Cin, int H, int W,
                                   int pad) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * Cin * H * W) return;
  const int Ho = H + 2 * pad - 2, Wo = W + 2 * pad - 2, C9 = Cin * 9;
  const int y = (int)(idx % W), x = (int)((idx / W) % H), ci = (int)((idx / ((int64_t)W * H)) % Cin);
  const int64_t b = idx / ((int64_t)W * H * Cin);
  float s = 0.0f;
#pragma unroll
  for (int kx = 0; kx < 3; ++kx) {
    const int ox = x - kx + pad;
    if (ox < 0 || ox >= Ho) continue;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      const int oy = y - ky + pad;
      if (oy < 0 || oy >= Wo) continue;
      s += dcol[((b * Ho + ox) * Wo + oy) * C9 + ci * 9 + kx * 3 + ky];
    }
  }
  din[idx] = s;
}

// ------------------------------------------------------------------------------ loss
// one CTA; rows strided over threads; deterministic block reduction of the scalar loss
__global__ void __launch_bounds__(256) policy_value_loss_kernel(const float* __restrict__ logits, const float* __restrict__ vraw,
                                                                const float* __restrict__ tpi, const float* __restrict__ tv,
                                                                int B, int A, float inv_norm, float* __restrict__ loss,
                                                                float* __restrict__ logp, float* __restrict__ v,
                                                                float* __restrict__ dlogits, float* __restrict__ dvraw) {
  __shared__ float red[256];
  float part = 0.0f;
  for (int r = threadIdx.x; r < B; r += blockDim.x) {
    const float* lg = logits + (size_t)r * A;
    float m = -INFINITY;
    for (int a = 0; a < A; ++a) m = fmaxf(m, lg[a]);
    float s = 0.0f;
    for (int a = 0; a < A; ++a) s += expf(lg[a] - m);
    const float lse = logf(s);
    float tsum = 0.0f, lpi = 0.0f;
    for (int a = 0; a < A; ++a) {
      const float lp = (lg[a] - m) - lse;
      logp[(size_t)r * A + a] = lp;
      tsum += tpi[(size_t)r * A + a];
      lpi += tpi[(size_t)r * A + a] * lp;
    }
    for (int a = 0; a < A; ++a)  // d(-sum pi*logp / norm)/dlogit = (softmax * sum(pi) - pi) / norm
      dlogits[(size_t)r * A + a] = (expf(logp[(size_t)r * A + a]) * tsum - tpi[(size_t)r * A + a]) * inv_norm;
    const float vv = tanhf(vraw[r]);
    v[r] = vv;
    const float diff = tv[r] - vv;
    dvraw[r] = -2.0f * diff * (1.0f - vv * vv) * inv_norm;
    part += (-lpi + diff * diff) * inv_norm;
  }
  red[threadIdx.x] = part;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) loss[0] = red[0];
}

// ------------------------------------------------------------------------------ GNN layer pieces
__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// h[i,:] = relu(S[i,:] + t0 + b0);  s[i] = sigmoid(h[i,:] . w2 + b2)     (one warp per path row)
__global__ void att_scores_kernel(float* __restrict__ S, const float* __restrict__ t0, const float* __restrict__ b0,
                                  const float* __restrict__ w2, const float* __restrict__ b2, int P, float* __restrict__ s) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= P) return;
  float acc = 0.0f;
  for (int j = lane; j < 128; j += 32) {
    const float h = fmaxf(S[(size_t)row * 128 + j] + t0[j] + b0[j], 0.0f);
    S[(size_t)row * 128 + j] = h;
    acc = fmaf(h, w2[j], acc);
  }
  acc = warp_sum(acc);
  if (lane == 0) s[row] = sigmoidf_(acc + b2[0]);
}

// alpha = s / sum(s) when the sum is positive (gnn_utils.py:58-59); single thread, fixed order
__global__ void att_normalise_kernel(const float* s, int P, float* alpha, float* tot) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  float t = 0.0f;
  for (int i = 0; i < P; ++i) t += s[i];
  tot[0] = t;
  for (int i = 0; i < P; ++i) alpha[i] = t > 0.0f ? s[i] / t : s[i];
}

// gate = sigmoid(gpre) (in place);  out0 = f0 + gate * upd
__global__ void gate_out_kernel(float* gate, const float* upd, const float* f0, float* out0, int F) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= F) return;
  const float g = sigmoidf_(gate[i]);
  gate[i] = g;
  out0[i] = f0[i] + g * upd[i];
}

__global__ void gate_bwd_kernel(const float* dout0, const float* gate, const float* upd, float* dgpre, float* dupd, int F) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= F) return;
  const float g = gate[i];
  dgpre[i] = dout0[i] * upd[i] * g * (1.0f - g);
  dupd[i] = dout0[i] * g;
}

// d_alpha -> d_z (pre-sigmoid attention logits); single thread
__global__ void att_bwd_kernel(const float* dalpha, const float* s, const float* tot, int P, float* dz) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const float t = tot[0];
  float dot = 0.0f;
  for (int i = 0; i < P; ++i) dot += dalpha[i] * s[i];
  for (int i = 0; i < P; ++i) {
    const float ds = t > 0.0f ? dalpha[i] / t - dot / (t * t) : dalpha[i];
    dz[i] = ds * s[i] * (1.0f - s[i]);
  }
}

// dhpre[i,j] = dz[i] * w2[j] * (h[i,j] > 0)
__global__ void att_hidden_bwd_kernel(const float* dz, const float* w2, const float* h, int P, float* dhpre) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P * 128) return;
  dhpre[i] = h[i] > 0.0f ? dz[i / 128] * w2[i % 128] : 0.0f;
}

// FrozenLake graph layer (FrozenLakeNet.py:8-33, 55-74): all-ones adjacency normalised to c = d*d,
// d = k^-1/2, so every valid node of graph b receives relu(c * sum_j sup[b,j,:]).
// sup/out: [B, 5, E] (unused nodes hold zeros), counts: [B] nodes per graph.
__global__ void graph_mean_relu_fwd_kernel(const float* __restrict__ sup, const int32_t* __restrict__ counts, int64_t B,
                                           int E, float* __restrict__ out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * E) return;
  const int64_t b = idx / E;
  const int e = (int)(idx % E), k = counts[b];
  const float d = 1.0f / sqrtf((float)k), c = d * d;
  float agg = 0.0f;
  for (int j = 0; j < k; ++j) agg = fmaf(c, sup[(b * 5 + j) * E + e], agg);
  agg = fmaxf(agg, 0.0f);
  for (int j = 0; j < 5; ++j) out[(b * 5 + j) * E + e] = j < k ? agg : 0.0f;
}

__global__ void graph_mean_relu_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ out,
                                           const int32_t* __restrict__ counts, int64_t B, int E, float* __restrict__ dsup) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * E) return;
  const int64_t b = idx / E;
  const int e = (int)(idx % E), k = counts[b];
  const float d = 1.0f / sqrtf((float)k), c = d * d;
  float g = 0.0f;
  for (int j = 0; j < k; ++j) g += dout[(b * 5 + j) * E + e];
  g = out[(b * 5) * E + e] > 0.0f ? g * c : 0.0f;
  for (int j = 0; j < 5; ++j) dsup[(b * 5 + j) * E + e] = j < k ? g : 0.0f;
}

// ---- grid-graph layer of the roofline sweep (BASELINE configs[4], SURVEY section 8d.5) -----------------
// relu(bmm(adj, support)) of FrozenLakeNet.GNNLayer (FrozenLakeNet.py:8-33) with adj = D^-1/2 (A + I) D^-1/2
// of the gh x gw 4-neighbour grid (normalisation as create_adjacency, FrozenLakeNet.py:68-72).  The adjacency
// is never materialised: each node gathers its <= 5 neighbours with coefficients d_i * d_j.
// One thread per (graph, node, 4 channels): 128-bit loads, neighbours of a CTA's graphs hit L1/L2.
__device__ __forceinline__ float grid_deg_inv_sqrt(int x, int y, int gh, int gw) {
  const int deg = 1 + (x > 0) + (x < gh - 1) + (y > 0) + (y < gw - 1);
  return 1.0f / sqrtf((float)deg);
}

constexpr int GRID_AGG_CHUNK = 256;              // nodes per neighbour table (10 KB of shared memory)
constexpr int64_t GRID_AGG_MAX_NODES = 1 << 30;  // node indices, node chunks and gh * gw stay inside int

// The loads of a thread's <= 5 neighbours are all issued before the first FMA, and the backward is held to 4 CTAs per SM
// (<= 64 registers).  Measured on an NVIDIA B200 at its 1,000 W power limit, aggregation alone, against the kernel that
// had no node chunks (both builds alternating within one run; GB/s of the fp32 rows of bench_sweep.py or of 20 timed
// launches on working sets above L2):
//  - with the chunk loop but loads interleaved with the FMAs (the compiler's schedule of the plain loop), the forward
//    dropped from 4,405-4,413 to 4,068-4,091 GB/s at 7x7, H = 128, B = 16,384 and from 4,620 to 4,184-4,194 at 16x16;
//  - loads first without the CTA bound, the backward took 80 registers (3 CTAs per SM) and fell from 2,972-2,993 to
//    2,405-2,466 GB/s at 3x3, H = 64, B = 131,072 (one pass of the node loop per graph);
//  - as written: forward 4,636-4,645 (was 4,448-4,454) at 7x7 and 4,733-4,737 (4,589-4,594) at 16x16, H = 128;
//    backward 4,325-4,359 (3,852-3,877) at 16x16, H = 256, and 2,936-2,969 (2,947-2,952) at 3x3, H = 64.
template <bool BWD>
__global__ void __launch_bounds__(256, BWD ? 4 : 0) grid_aggregate_kernel(const float* __restrict__ in, const float* __restrict__ act,
                                                             int64_t B, int gh, int gw, int H, float* __restrict__ out) {
  // FWD: out = relu(adj * in).            BWD: out = adj^T * (in * (act > 0)) = adj * (...), adj symmetric
  // Thread layout: x = 4-channel group, y = node slot; a CTA walks whole graphs.  The <= 5 (neighbour,
  // coefficient) pairs of every node are tabulated per CTA in shared memory, so the streaming loop is
  // index-math free: per output float4 at most five 128-bit loads (neighbours of a graph hit L1) and one store.
  // The table holds GRID_AGG_CHUNK nodes: larger graphs are walked one node chunk at a time, each chunk over all of
  // the CTA's graphs (graphs of up to GRID_AGG_CHUNK nodes: one chunk, the table is filled once).
  __shared__ int32_t nb_idx[GRID_AGG_CHUNK * 5];
  __shared__ float nb_coef[GRID_AGG_CHUNK * 5];
  const int H4 = H >> 2, n = gh * gw;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  const float4* in4 = reinterpret_cast<const float4*>(in);
  const float4* act4 = reinterpret_cast<const float4*>(act);
  float4* out4 = reinterpret_cast<float4*>(out);
  for (int base = 0; base < n; base += GRID_AGG_CHUNK) {
    const int cn = min(n - base, GRID_AGG_CHUNK);
    if (base > 0) __syncthreads();  // every thread is done reading the previous chunk's table
    for (int i = tid; i < cn * 5; i += blockDim.x * blockDim.y) {
      const int node = base + i / 5, k = i % 5, x = node / gw, y = node % gw;
      const int dx = (k == 1) ? -1 : (k == 2) ? 1 : 0, dy = (k == 3) ? -1 : (k == 4) ? 1 : 0;
      const int nx = x + dx, ny = y + dy;
      const bool ok = nx >= 0 && nx < gh && ny >= 0 && ny < gw;
      nb_idx[i] = ok ? nx * gw + ny : -1;
      nb_coef[i] = ok ? grid_deg_inv_sqrt(x, y, gh, gw) * grid_deg_inv_sqrt(nx, ny, gh, gw) : 0.0f;
    }
    __syncthreads();
    for (int64_t b = blockIdx.x; b < B; b += gridDim.x) {
      const int64_t g0 = b * n;
      for (int node = threadIdx.y; node < cn; node += blockDim.y) {
        for (int c4 = threadIdx.x; c4 < H4; c4 += blockDim.x) {
          float4 v[5], a[5];
#pragma unroll
          for (int k = 0; k < 5; ++k) {
            const int j = nb_idx[node * 5 + k];
            if (j < 0) continue;
            const size_t off = (size_t)(g0 + j) * H4 + c4;
            v[k] = in4[off];
            if (BWD) a[k] = act4[off];
          }
          float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int k = 0; k < 5; ++k) {
            if (nb_idx[node * 5 + k] < 0) continue;
            if (BWD) {
              v[k].x = a[k].x > 0.f ? v[k].x : 0.f; v[k].y = a[k].y > 0.f ? v[k].y : 0.f;
              v[k].z = a[k].z > 0.f ? v[k].z : 0.f; v[k].w = a[k].w > 0.f ? v[k].w : 0.f;
            }
            const float coef = nb_coef[node * 5 + k];
            acc.x = fmaf(coef, v[k].x, acc.x); acc.y = fmaf(coef, v[k].y, acc.y);
            acc.z = fmaf(coef, v[k].z, acc.z); acc.w = fmaf(coef, v[k].w, acc.w);
          }
          if (!BWD) { acc.x = fmaxf(acc.x, 0.f); acc.y = fmaxf(acc.y, 0.f); acc.z = fmaxf(acc.z, 0.f); acc.w = fmaxf(acc.w, 0.f); }
          out4[(size_t)(g0 + base + node) * H4 + c4] = acc;
        }
      }
    }
  }
}

template <bool BWD>
int launch_grid_aggregate(const float* in, const float* act, int64_t B, int gh, int gw, int H, float* out, cudaStream_t st) {
  const int H4 = H / 4;
  const int bx = H4 < 64 ? (H4 < 16 ? 16 : H4) : 64;  // 16..64 channel groups per row of threads
  dim3 block(bx, 256 / bx);
  const int grid = (int)(B < 148 * 16 ? B : 148 * 16);
  grid_aggregate_kernel<BWD><<<grid, block, 0, st>>>(in, act, B, gh, gw, H, out);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

struct Bump {
  float* p;
  float* take(size_t n) {
    float* r = p;
    p += (n + 63) / 64 * 64;
    return r;
  }
};

// layout of the `saved` buffer of a layer forward (floats)
struct LayerSaved {
  float *t0, *h, *s, *alpha, *tot, *agg, *cat2, *gate, *u1, *upd;
  static size_t carve(LayerSaved* L, float* base, int P, int F) {
    Bump b{base};
    float* t0 = b.take(128); float* h = b.take((size_t)P * 128); float* s = b.take(P); float* al = b.take(P);
    float* tot = b.take(1); float* agg = b.take(F); float* cat2 = b.take(2 * (size_t)F); float* gate = b.take(F);
    float* u1 = b.take(F); float* upd = b.take(F);
    if (L) { L->t0 = t0; L->h = h; L->s = s; L->alpha = al; L->tot = tot; L->agg = agg; L->cat2 = cat2; L->gate = gate; L->u1 = u1; L->upd = upd; }
    return (size_t)(b.p - base);
  }
};

int linear_fwd(const float* X, const float* W, int64_t ldw, const float* bias, float* Y, int64_t M, int N, int K, int relu,
               cudaStream_t st) {
  if (M == 1 && gemv_rows_ok(W, ldw, X, K)) return gemv_rows(W, ldw, X, bias, Y, N, K, relu, st);
  int rc = gemm(false, true, M, N, K, X, K, W, ldw, Y, N, 0.0f, st);
  if (rc) return rc;
  add_bias_act_kernel<<<grid_for(M * N, 256), 256, 0, st>>>(Y, bias, M, N, relu);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

}  // namespace

// small-batch Linear forward (azg_nets.cu routes azg_linear_f32 here when M is too small to fill its 128 x 128 tiles)
int azg_train_linear_fwd(const float* X, const float* W, const float* bias, float* Y, int64_t M, int N, int K, int relu,
                         cudaStream_t st) {
  return linear_fwd(X, W, K, bias, Y, M, N, K, relu, st);
}

extern "C" {

int azg_gemm_f32(int transA, int transB, int64_t M, int N, int K, const float* A, int64_t lda, const float* B, int64_t ldb,
                 float* C, int64_t ldc, float beta, azg_stream stream) {
  AZG_REQUIRE(A && B && C && K > 0, "azg_gemm_f32: bad argument");
  return gemm(transA != 0, transB != 0, M, N, K, A, lda, B, ldb, C, ldc, beta, (cudaStream_t)stream);
}

int azg_mul_f32(const float* a, const float* b, float* out, int64_t n, azg_stream stream) {
  AZG_REQUIRE(a && b && out, "azg_mul_f32: null pointer");
  if (n <= 0) return AZG_OK;
  mul_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(a, b, out, n);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

// Y = act(X W^T + b) backward: dX = g W, dW = g^T X, db = column sums of g, g = dY * (Y > 0) if relu.
// Any of dX / dW / db may be NULL.  scratch: M*N floats when relu, else unused.
int azg_linear_backward(const float* dY, const float* X, const float* W, const float* Y, int64_t M, int N, int K, int relu,
                        float* dX, float* dW, float* db, float* scratch, azg_stream stream) {
  AZG_REQUIRE(dY && X && W, "azg_linear_backward: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const float* g = dY;
  if (relu) {
    AZG_REQUIRE(Y && scratch, "azg_linear_backward: relu needs Y and scratch");
    relu_bwd_kernel<<<grid_for(M * N, 256), 256, 0, st>>>(dY, Y, scratch, M * N);
    AZG_LAUNCH_CHECK();
    g = scratch;
  }
  int rc;
  if (dX && (rc = gemm(false, false, M, K, N, g, N, W, K, dX, K, 0.0f, st))) return rc;
  // weight / bias gradients contract over the M rows: with a large batch (the grid-graph sweep) a single pass
  // would leave the whole contraction to (N/64)*(K/64) CTAs, so it is split over row chunks and reduced in
  // fixed order (deterministic)
  const int splits = M >= 8192 ? (int)(M / 4096 < 512 ? M / 4096 : 512) : 1;
  if (splits == 1) {
    if (dW && (rc = gemm(true, false, N, K, (int)M, g, N, X, K, dW, K, 0.0f, st))) return rc;
    if (db) {
      col_sum_kernel<<<grid_for(N, 128), 128, 0, st>>>(g, M, N, N, db);
      AZG_LAUNCH_CHECK();
    }
    return AZG_OK;
  }
  float* part = nullptr;
  const size_t wn = (size_t)N * K;
  AZG_CUDA_CHECK(cudaMallocAsync((void**)&part, sizeof(float) * (size_t)splits * (wn + N), st));
  if (dW) {
    if ((rc = gemm_split(true, false, N, K, (int)M, g, N, X, K, part, K, 0.0f, splits, (int64_t)wn, st))) return rc;
    reduce_splits_kernel<<<grid_for((int64_t)wn, 256), 256, 0, st>>>(part, splits, (int64_t)wn, dW);
    AZG_LAUNCH_CHECK();
  }
  if (db) {
    float* bpart = part + (size_t)splits * wn;
    const int64_t rper = (M + splits - 1) / splits;
    col_sum_split_kernel<<<dim3(grid_for(N, 128), splits), 128, 0, st>>>(g, M, N, rper, bpart);
    AZG_LAUNCH_CHECK();
    reduce_splits_kernel<<<grid_for(N, 256), 256, 0, st>>>(bpart, splits, N, db);
    AZG_LAUNCH_CHECK();
  }
  AZG_CUDA_CHECK(cudaFreeAsync(part, st));
  return AZG_OK;
}

// conv3x3 + ReLU backward (Connect4Net.py:45-46 / TicTacToeNet.py:33-35).  din may be NULL (first layer).
int azg_conv3x3_relu_backward(const float* in, const float* w, const float* out, const float* dout, float* din, float* dw,
                              float* db, int64_t B, int Cin, int Cout, int H, int W, int pad, azg_stream stream) {
  AZG_REQUIRE(in && w && out && dout && dw && db, "azg_conv3x3_relu_backward: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int Ho = H + 2 * pad - 2, Wo = W + 2 * pad - 2, C9 = Cin * 9;
  const int64_t R = B * Ho * Wo;  // rows of the contraction: (board, output cell)
  const size_t n_g = (size_t)R * Cout, n_c = (size_t)R * C9;
  if (R >= 256 && n_g + 2 * n_c <= ((size_t)1 << 28)) {
    const int splits = (int)(R / 64 < 64 ? R / 64 : 64);
    Scratch sc(st);
    if (sc.get(n_g + 2 * n_c + (size_t)splits * Cout + 256)) {
      azg_set_error("azg_conv3x3_relu_backward: scratch allocation failed");
      return AZG_ERR_CUDA;
    }
    float* gt = sc.p;
    float* col = gt + (n_g + 63) / 64 * 64;
    float* dcol = col + (n_c + 63) / 64 * 64;
    float* bpart = dcol + (n_c + 63) / 64 * 64;
    conv_bwd_pack_kernel<<<grid_for((int64_t)(n_g + n_c), 256), 256, 0, st>>>(in, out, dout, gt, col, B, Cin, Cout, H, W, pad);
    AZG_LAUNCH_CHECK();
    int rc;
    if ((rc = gemm(true, false, Cout, C9, (int)R, gt, Cout, col, C9, dw, C9, 0.0f, st))) return rc;
    col_sum_split_kernel<<<dim3(grid_for(Cout, 128), splits), 128, 0, st>>>(gt, R, Cout, (R + splits - 1) / splits, bpart);
    AZG_LAUNCH_CHECK();
    reduce_splits_kernel<<<grid_for(Cout, 256), 256, 0, st>>>(bpart, splits, Cout, db);
    AZG_LAUNCH_CHECK();
    if (din) {
      if ((rc = gemm(false, false, R, C9, Cout, gt, Cout, w, C9, dcol, C9, 0.0f, st))) return rc;
      conv_col2im_kernel<<<grid_for(B * Cin * H * W, 256), 256, 0, st>>>(dcol, din, B, Cin, H, W, pad);
      AZG_LAUNCH_CHECK();
    }
    return AZG_OK;
  }
  conv_bwd_weight_kernel<<<grid_for(Cout * Cin * 9 + Cout, 128), 128, 0, st>>>(in, out, dout, dw, db, B, Cin, Cout, H, W, pad);
  AZG_LAUNCH_CHECK();
  if (din) {
    conv_bwd_data_kernel<<<grid_for(B * Cin * H * W, 128), 128, 0, st>>>(w, out, dout, din, B, Cin, Cout, H, W, pad);
    AZG_LAUNCH_CHECK();
  }
  return AZG_OK;
}

// loss = (-sum(target_pi * log_softmax(logits)) + sum((target_v - tanh(vraw))^2)) / norm, with its gradients.
// Outputs: loss[1], logp[B,A], v[B], dlogits[B,A], dvraw[B] (all device).  norm = the GLOBAL batch size
// (the reference divides by size()[0]; data-parallel ranks pass the global B, SURVEY section 8e).
int azg_policy_value_loss(const float* logits, const float* vraw, const float* target_pi, const float* target_v, int B,
                          int A, float norm, float* loss, float* logp, float* v, float* dlogits, float* dvraw,
                          azg_stream stream) {
  AZG_REQUIRE(logits && vraw && target_pi && target_v && loss && logp && v && dlogits && dvraw && norm > 0,
              "azg_policy_value_loss: bad argument");
  policy_value_loss_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(logits, vraw, target_pi, target_v, B, A, 1.0f / norm, loss,
                                                                logp, v, dlogits, dvraw);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

int azg_graph_mean_relu_forward(const float* sup, const int32_t* counts, int64_t B, int E, float* out, azg_stream stream) {
  AZG_REQUIRE(sup && counts && out, "azg_graph_mean_relu_forward: null pointer");
  if (B <= 0) return AZG_OK;
  graph_mean_relu_fwd_kernel<<<grid_for(B * E, 256), 256, 0, (cudaStream_t)stream>>>(sup, counts, B, E, out);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

int azg_graph_mean_relu_backward(const float* dout, const float* out, const int32_t* counts, int64_t B, int E, float* dsup,
                                 azg_stream stream) {
  AZG_REQUIRE(dout && out && counts && dsup, "azg_graph_mean_relu_backward: null pointer");
  if (B <= 0) return AZG_OK;
  graph_mean_relu_bwd_kernel<<<grid_for(B * E, 256), 256, 0, (cudaStream_t)stream>>>(dout, out, counts, B, E, dsup);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

int azg_grid_aggregate_relu_forward(const float* sup, int64_t B, int gh, int gw, int H, float* out, azg_stream stream) {
  AZG_REQUIRE(sup && out && gh >= 1 && gw >= 1 && (int64_t)gh * gw <= GRID_AGG_MAX_NODES && H % 4 == 0,
              "azg_grid_aggregate_relu_forward: bad argument");
  if (B <= 0) return AZG_OK;
  return launch_grid_aggregate<false>(sup, nullptr, B, gh, gw, H, out, (cudaStream_t)stream);
}

int azg_grid_aggregate_relu_backward(const float* dout, const float* out, int64_t B, int gh, int gw, int H, float* dsup,
                                     azg_stream stream) {
  AZG_REQUIRE(dout && out && dsup && gh >= 1 && gw >= 1 && (int64_t)gh * gw <= GRID_AGG_MAX_NODES && H % 4 == 0,
              "azg_grid_aggregate_relu_backward: bad argument");
  if (B <= 0) return AZG_OK;
  return launch_grid_aggregate<true>(dout, out, B, gh, gw, H, dsup, (cudaStream_t)stream);
}

// ---- GNNLayer (gnn_utils.py:5-74) at B = P + 1 > 1 -----------------------------------------------
size_t azg_gnn_layer_saved_floats(int P, int F) { return LayerSaved::carve(nullptr, nullptr, P, F); }
size_t azg_gnn_layer_scratch_floats(int P, int F) { return 8 * (size_t)F + 2 * (size_t)P * 128 + 4 * (size_t)P + 1024; }

// f0 [F] = target row, path [P,F] = rows 1..; writes out0 [F] (the updated target row) and `saved`.
int azg_gnn_layer_forward(const azg_gnn_layer_params* p, const float* f0, const float* path, int P, int F, float* out0,
                          float* saved, azg_stream stream) {
  AZG_REQUIRE(p && f0 && path && out0 && saved && P >= 1, "azg_gnn_layer_forward: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  LayerSaved L;
  LayerSaved::carve(&L, saved, P, F);
  int rc;
  const int64_t F2 = 2 * (int64_t)F;
  // attention logits: W[:, :F] f0 (once) + W[:, F:] f_i
  if ((rc = gemm(false, true, 1, 128, F, f0, F, p->att0_w, F2, L.t0, 128, 0.0f, st))) return rc;
  if ((rc = gemm(false, true, P, 128, F, path, F, p->att0_w + F, F2, L.h, 128, 0.0f, st))) return rc;
  att_scores_kernel<<<grid_for((int64_t)P * 32, 256), 256, 0, st>>>(L.h, L.t0, p->att0_b, p->att2_w, p->att2_b, P, L.s);
  AZG_LAUNCH_CHECK();
  att_normalise_kernel<<<1, 32, 0, st>>>(L.s, P, L.alpha, L.tot);
  AZG_LAUNCH_CHECK();
  if ((rc = gemm(false, false, 1, F, P, L.alpha, P, path, F, L.agg, F, 0.0f, st))) return rc;  // sum_i alpha_i f_i
  AZG_CUDA_CHECK(cudaMemcpyAsync(L.cat2, f0, sizeof(float) * F, cudaMemcpyDeviceToDevice, st));
  AZG_CUDA_CHECK(cudaMemcpyAsync(L.cat2 + F, L.agg, sizeof(float) * F, cudaMemcpyDeviceToDevice, st));
  if ((rc = linear_fwd(L.cat2, p->gate_w, F2, p->gate_b, L.gate, 1, F, (int)F2, 0, st))) return rc;
  if ((rc = linear_fwd(L.cat2, p->upd0_w, F2, p->upd0_b, L.u1, 1, F, (int)F2, 1, st))) return rc;
  if ((rc = linear_fwd(L.u1, p->upd2_w, F, p->upd2_b, L.upd, 1, F, F, 0, st))) return rc;
  gate_out_kernel<<<grid_for(F, 256), 256, 0, st>>>(L.gate, L.upd, f0, out0, F);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

// d_out0 [F] -> parameter gradients (overwritten) and d_f0 [F] (gradient w.r.t. the input target row).
// Gradients w.r.t. the path rows are not produced: nothing trainable lies upstream of them in the GNN
// step (Connect4GNN.py:195-197 steps only the GNN optimizer; SURVEY section 8e).
int azg_gnn_layer_backward(const azg_gnn_layer_params* p, const float* f0, const float* path, int P, int F,
                           const float* saved, const float* d_out0, float* d_f0, const azg_gnn_layer_grads* g,
                           float* scratch, azg_stream stream) {
  AZG_REQUIRE(p && f0 && path && saved && d_out0 && d_f0 && g && scratch, "azg_gnn_layer_backward: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  LayerSaved L;
  LayerSaved::carve(&L, const_cast<float*>(saved), P, F);
  Bump b{scratch};
  float* dgpre = b.take(F); float* dupd = b.take(F); float* du1 = b.take(F); float* dcat2 = b.take(2 * (size_t)F);
  float* dalpha = b.take(P); float* dz = b.take(P); float* dhpre = b.take((size_t)P * 128); float* dhsum = b.take(128);
  const int64_t F2 = 2 * (int64_t)F;
  int rc;
  gate_bwd_kernel<<<grid_for(F, 256), 256, 0, st>>>(d_out0, L.gate, L.upd, dgpre, dupd, F);
  AZG_LAUNCH_CHECK();
  // each weight matrix is streamed ONCE: its gradient (rank-1) is written and its input gradient accumulated in one pass
  const bool fused = rank1_ok(p->gate_w, F2, L.cat2, g->gate_w, F2, (int)F2) && rank1_ok(p->upd2_w, F, L.u1, g->upd2_w, F, F) &&
                     rank1_ok(p->upd0_w, F2, L.cat2, g->upd0_w, F2, (int)F2);
  // gate = sigmoid(Wg cat2 + bg)
  if (fused) {
    if ((rc = rank1_bwd(p->gate_w, F2, dgpre, L.cat2, g->gate_w, F2, dcat2, 0.0f, F, (int)F2, st))) return rc;
  } else {
    if ((rc = gemm(true, false, F, (int)F2, 1, dgpre, F, L.cat2, F2, g->gate_w, F2, 0.0f, st))) return rc;
    if ((rc = gemm(false, false, 1, (int)F2, F, dgpre, F, p->gate_w, F2, dcat2, F2, 0.0f, st))) return rc;
  }
  AZG_CUDA_CHECK(cudaMemcpyAsync(g->gate_b, dgpre, sizeof(float) * F, cudaMemcpyDeviceToDevice, st));
  // upd = W2 relu(W0 cat2 + b0) + b2
  if (fused) {
    if ((rc = rank1_bwd(p->upd2_w, F, dupd, L.u1, g->upd2_w, F, du1, 0.0f, F, F, st))) return rc;
  } else {
    if ((rc = gemm(true, false, F, F, 1, dupd, F, L.u1, F, g->upd2_w, F, 0.0f, st))) return rc;
    if ((rc = gemm(false, false, 1, F, F, dupd, F, p->upd2_w, F, du1, F, 0.0f, st))) return rc;
  }
  AZG_CUDA_CHECK(cudaMemcpyAsync(g->upd2_b, dupd, sizeof(float) * F, cudaMemcpyDeviceToDevice, st));
  relu_bwd_kernel<<<grid_for(F, 256), 256, 0, st>>>(du1, L.u1, du1, F);
  AZG_LAUNCH_CHECK();
  if (fused) {
    if ((rc = rank1_bwd(p->upd0_w, F2, du1, L.cat2, g->upd0_w, F2, dcat2, 1.0f, F, (int)F2, st))) return rc;
  } else {
    if ((rc = gemm(true, false, F, (int)F2, 1, du1, F, L.cat2, F2, g->upd0_w, F2, 0.0f, st))) return rc;
    if ((rc = gemm(false, false, 1, (int)F2, F, du1, F, p->upd0_w, F2, dcat2, F2, 1.0f, st))) return rc;
  }
  AZG_CUDA_CHECK(cudaMemcpyAsync(g->upd0_b, du1, sizeof(float) * F, cudaMemcpyDeviceToDevice, st));
  // cat2 = [f0, agg];  out0 = f0 + ...
  AZG_CUDA_CHECK(cudaMemcpyAsync(d_f0, d_out0, sizeof(float) * F, cudaMemcpyDeviceToDevice, st));
  axpy_kernel<<<grid_for(F, 256), 256, 0, st>>>(d_f0, dcat2, F);
  AZG_LAUNCH_CHECK();
  // agg = sum_i alpha_i f_i  ->  d_alpha_i = d_agg . f_i
  if ((rc = gemm(false, true, 1, P, F, dcat2 + F, F, path, F, dalpha, P, 0.0f, st))) return rc;
  att_bwd_kernel<<<1, 32, 0, st>>>(dalpha, L.s, L.tot, P, dz);
  AZG_LAUNCH_CHECK();
  // z_i = w2 . h_i + b2
  if ((rc = gemm(false, false, 1, 128, P, dz, P, L.h, 128, g->att2_w, 128, 0.0f, st))) return rc;
  col_sum_kernel<<<1, 32, 0, st>>>(dz, P, 1, 1, g->att2_b);
  AZG_LAUNCH_CHECK();
  att_hidden_bwd_kernel<<<grid_for((int64_t)P * 128, 256), 256, 0, st>>>(dz, p->att2_w, L.h, P, dhpre);
  AZG_LAUNCH_CHECK();
  // hpre_i = W[:, :F] f0 + W[:, F:] f_i + b
  col_sum_kernel<<<1, 128, 0, st>>>(dhpre, P, 128, 128, dhsum);
  AZG_LAUNCH_CHECK();
  AZG_CUDA_CHECK(cudaMemcpyAsync(g->att0_b, dhsum, sizeof(float) * 128, cudaMemcpyDeviceToDevice, st));
  if ((rc = gemm(true, false, 128, F, 1, dhsum, 128, f0, F, g->att0_w, F2, 0.0f, st))) return rc;
  if ((rc = gemm(true, false, 128, F, P, dhpre, 128, path, F, g->att0_w + F, F2, 0.0f, st))) return rc;
  return gemm(false, false, 1, F, 128, dhsum, 128, p->att0_w, F2, d_f0, F, 1.0f, st);
}

}  // extern "C"
