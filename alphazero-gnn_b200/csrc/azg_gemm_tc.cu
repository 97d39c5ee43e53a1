// azg_gemm_tc.cu -- K2 main loop on the 5th-gen tensor cores: the two F x F contractions of
// PolicyValueGNN.output_transform (gnn_utils.py:99-103, F = 64 n^2 = 3136 for 7x7) for a batch
// of leaf positions:   H = relu(X W0^T + b0),   E = H W2^T + b2.
//
// Design (sm_100a only):
//   * Operands live in HBM as *tile images*: every [rows x 64] bf16 block is stored exactly as
//     the tensor core wants to see it in shared memory (8-row groups of 128-byte rows, 16-byte
//     chunks XOR-swizzled by the row index = the SWIZZLE_128B K-major canonical layout), so a
//     pipeline stage is filled by two plain bulk-async copies (cp.async.bulk -> UBLKCP) that
//     complete on an mbarrier; no tensor maps, no in-kernel shuffling.  Weights are re-tiled
//     once per optimizer step (azg_c4_pack); activations are written as images by the
//     producer (the f32->image kernel for X, the GEMM epilogue for H).
//   * Persistent, warp-specialised kernel: warp 0 = bulk-copy producer, warp 1 = MMA issuer (a single thread
//     issues tcgen05.mma), warp 2 = TMEM allocator, warps 4-7 = epilogue (tcgen05.ld -> bias/ReLU -> store).
//     Accumulators live in TMEM, double-buffered (2 x BN fp32 columns) so the epilogue of tile i overlaps the
//     main loop of tile i+1.  One instantiation per tile width:
//       TWO = 0  (BN = 64) one CTA per SM, M=128 x N=BN x K=16 MMAs, smem ring of 4 stages x (16 KB A + BN*128 B W);
//       TWO = 1  (BN >= 128) CTA pairs (cluster of 2, cta_group::2): 256 x BN x 16 MMAs issued by the leader CTA, each
//                CTA holds 128 rows of A and of the accumulator and BN/2 rows of the weight tile; a stage carries two
//                operand pairs (bf16x3: hi and lo of one k-block -> all three products; bf16: two k-blocks).  This is
//                the kernel of the Connect4 F x F contractions; it can also carry a 32-column side tile per m-unit
//                (GemmArgs::side_*: the standard policy/value heads ride on GEMM-1).
//   * AZG_PREC_BF16X3 (the 1e-5 parity mode): x = hi + lo with hi = bf16(x), lo = bf16(x - hi);
//     X W^T ~= Xhi Whi^T + Xhi Wlo^T + Xlo Whi^T, fp32 accumulate.  Implemented as ONE GEMM with a
//     3x longer K: the producer walks the k-blocks of [Xhi|Xhi|Xlo] against [Whi|Wlo|Whi]; the
//     MMA and epilogue code is the same as for plain bf16.
#include "azg_common.cuh"

#include <cuda_bf16.h>
#include <stdlib.h>

#include "azg_tc.cuh"

namespace tc {

// ---- epilogue output modes -----------------------------------------------------------------
enum { OUT_F32 = 0, OUT_IMG = 1, OUT_IMG_HILO = 2, OUT_HEADS = 3 };
constexpr int HEAD_ROWS = 10;    // <= 9 policy logits + 1 value (Connect4 n <= 8)
constexpr int HEAD_STRIDE = 16;  // floats per (row, n-tile) record of partial head sums

// K-split boundaries (k-blocks): equal parts.  (Tried: 40 % of K in the first work item so that the previous tile's real
// epilogue, ~20k cycles, hides under it -- 3 % faster, but the GEMM's distance from its exact emulation grew from 3.2e-6 to
// 4.0e-6: not kept.)
__host__ __device__ inline int ksplit_begin(int KB, int q, int nq) {
  return q <= 0 ? 0 : q >= nq ? KB : (int)((int64_t)KB * q / nq);
}

struct GemmArgs {
  const uint8_t* a_hi;  // activation images, tiles [128 x 64], (mt * KB + kb) * 16384
  const uint8_t* a_lo;  // (x3 only)
  const uint8_t* w_hi;  // weight images, tiles [BN x 64], (nt * KB + kb) * BN * 128
  const uint8_t* w_lo;  // (x3 only)
  const float* bias;    // [N]
  float* out_f32;       // OUT_F32: row-major [M, N]
  uint8_t* out_hi;      // OUT_IMG*: image with tiles [128 x 64] over (mt, N/64)
  uint8_t* out_lo;
  int64_t M;            // valid rows
  int m_tiles, n_tiles, KB;  // KB = K / 64 (per operand, before the x3 expansion)
  int x3;               // 0: bf16, 1: 3-term split
  int relu;
  int out_mode;
  const float* head_w;  // OUT_HEADS: [head_rows, N] fp32 (policy rows then the value row), reference order
  float* head_part;     // OUT_HEADS: [M, n_tiles, HEAD_STRIDE] partial sums, reduced in fixed order by heads_finalize
  int head_rows;
  const int32_t* dyn_rows;  // optional device scalar: number of valid rows this launch (<= M), read by the kernel
  // optional side tile (CTA-pair kernel only): one more n-tile of SIDE_N columns per m-unit contracts the same A rows
  // with a second, narrow weight image and writes fp32 [M, SIDE_N] (no ReLU) -- the standard policy/value heads of
  // `predict` ride on GEMM-1 instead of re-reading the feature image in their own launch
  const uint8_t* side_hi;  // [SIDE_N x K] weight image, tiles [SIDE_N x 64] at kb * SIDE_N * 128
  const uint8_t* side_lo;  // (x3 only)
  const float* side_bias;  // [SIDE_N]
  float* side_out;         // row-major [M, SIDE_N]
  // AZG_PREC_F16F8 (x3 = 1 and f8 = 1, CTA-pair kernel only): the "hi" images are fp16, the "lo" images are the FP8
  // correction rows of azg_tc.cuh; w_exp / side_exp point at the weight images' power-of-two scales (device ints
  // written by the pack kernels); activations use the fixed scale F8_A_SCALE
  int f8;
  const int32_t* w_exp;
  const int32_t* side_exp;
  // K-split accumulation (AZG_PREC_F16F8_KS, CTA-pair kernel with fused hi/lo stages only): this launch contracts the
  // k-blocks [kb0, kb0 + kbn) (kbn = 0: all KB) and its epilogue first adds `acc_in` (row-major fp32 [M, N] partial sums
  // of the earlier launches, may alias out_f32: every element is read and written by the same thread); `no_bias` leaves
  // the bias to the last launch; `side_acc` makes the side tile add to side_out instead of writing rr + bias.
  // The tensor core's fp32 accumulation truncates once per MMA, an error that grows linearly with the number of k-steps
  // (DESIGN.md section 4, "the accumulation floor"): C launches of K/C steps, summed here with round-to-nearest adds,
  // bring it down C times.
  int kb0, kbn;
  const float* acc_in;
  int no_bias, side_acc;
  // The same K-split INSIDE one launch (the default of AZG_PREC_F16F8_KS): every tile is contracted as `ksplit` consecutive
  // work items over a quarter of K each, on alternating TMEM accumulators, and the epilogue warps keep the running fp32
  // sum of a tile in `kpart` -- a per-CTA [128 x BN] scratch tile (gridDim.x of them, 17 MB in all) that every thread reads
  // and writes only at its own elements and that therefore never leaves L2.  Same adds in the same order as the
  // launch-level split: bit-identical results, without its 4.9 GB of partial-sum traffic per contraction.
  int ksplit;
  float* kpart;
};
// TMEM columns of the constant UE8M0 scale-factor regions (f8 mode; accumulators use 2 x BN <= 448 columns)
constexpr uint32_t SF_A_COL = 448, SF_W_COL = 464, SF_SIDE_COL = 480;
constexpr int SIDE_N = 32;
constexpr int SIDE_STAGE_BYTES = (SIDE_N / 2) * BK * 2;  // one CTA's half of a side weight tile stage

// TWO = CTA pair: cta_group::2 MMAs of 256 x BN (each CTA holds 128 rows of A and of the accumulator and
// BN/2 rows of the weight tile), which halves the weight bytes each SM reads from shared memory per MMA.
template <int BN, bool TWO>
struct Smem {
  static constexpr int NSTAGES = TWO ? 6 : STAGES;
  static constexpr int W_STAGE_BYTES = (TWO ? BN / 2 : BN) * BK * 2;  // this CTA's share of a weight tile stage
  static constexpr int W_TILE_BYTES = BN * BK * 2;                    // a whole weight tile stage in HBM
  static constexpr int STAGE_BYTES = A_STAGE_BYTES + W_STAGE_BYTES;
  static constexpr int BAR_OFFSET = NSTAGES * STAGE_BYTES;
  static constexpr int TOTAL = BAR_OFFSET + 256 + 1024;  // + barriers + alignment slack
};

// Epilogue of one accumulator tile for the calling thread's row (TMEM lane): side tile (standard heads) or main tile in
// any output mode.  `taddr` = this warp's lane quarter at the accumulator's first column; `release()` hands the
// accumulator back to the MMA issuer as soon as its last TMEM read is done.
// `grp` of `ngrp` epilogue groups (four warps each) takes every ngrp-th 32-column chunk of the tile; the partial head sums
// of a group go to slot nt * ngrp + grp of the row (fixed-order reduction in heads_finalize).
template <int BN, bool TWO, class Release>
__device__ __forceinline__ void epilogue_tile(const GemmArgs& g, uint32_t taddr, int mt, int nt, int r_local, int grp, int ngrp,
                                              Release release, float4* part = nullptr, int q = 0, int nq = 1) {
      // part / q / nq: in-kernel K-split -- work item q of nq of this tile.  Items before the last only fold their accumulator
      // into the CTA's partial-sum tile, the last one adds it and runs the tile's real epilogue.  The partial tile is stored
      // by groups of four columns, rows innermost: `part` points at this thread's row in group 0, group c is part[c * BM] --
      // a warp's 16-byte accesses are 512 contiguous bytes (row-major rows cost 32 wavefronts per instruction and took 58 %
      // of the shared-memory / L1 data pipe the tensor core reads its operands through: 6.4 instead of 4.x ms).
      const int64_t row = (int64_t)mt * BM + r_local;
      const int NKB = (g.n_tiles * BN) / BK;  // k-blocks of the output image
      if (TWO && nt == g.n_tiles) {  // side tile: SIDE_N fp32 columns + bias, row-major (one chunk: group 0)
        if (grp != 0) {
          release();
          return;
        }
        uint32_t rr[32];
        tmem_ld32(taddr, rr);
        tmem_ld_wait();
        tc_fence_before();
        release();
        if (nq > 1) {  // same order of adds as the launch-level split: ((rr0 + bias) + rr1) + ...
          float4* pp = part;
          float4* dst = reinterpret_cast<float4*>(g.side_out + row * SIDE_N);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 b4 = q ? pp[j * BM] : __ldg(reinterpret_cast<const float4*>(g.side_bias) + j);
            const float4 o = make_float4(__uint_as_float(rr[4 * j]) + b4.x, __uint_as_float(rr[4 * j + 1]) + b4.y,
                                         __uint_as_float(rr[4 * j + 2]) + b4.z, __uint_as_float(rr[4 * j + 3]) + b4.w);
            if (q + 1 < nq) pp[j * BM] = o;
            else if (row < g.M) dst[j] = o;
          }
          return;
        }
        if (row < g.M) {
          float4* dst = reinterpret_cast<float4*>(g.side_out + row * SIDE_N);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 b4 = g.side_acc ? dst[j] : __ldg(reinterpret_cast<const float4*>(g.side_bias) + j);
            dst[j] = make_float4(__uint_as_float(rr[4 * j]) + b4.x, __uint_as_float(rr[4 * j + 1]) + b4.y,
                                 __uint_as_float(rr[4 * j + 2]) + b4.z, __uint_as_float(rr[4 * j + 3]) + b4.w);
          }
        }
        return;
      }
      if (nq > 1 && q + 1 < nq) {  // fold this quarter's accumulator into the partial sums (no bias, no ReLU)
#pragma unroll 1
        for (int c0 = grp * 32; c0 < BN; c0 += 32 * ngrp) {
          uint32_t rr[32];
          tmem_ld32(taddr + (uint32_t)c0, rr);
          float4* pp = part + (c0 >> 2) * BM;
          float4 p4[8];
          if (q) {
#pragma unroll
            for (int j = 0; j < 8; ++j) p4[j] = pp[j * BM];
          }
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            if (q)
              pp[j * BM] = make_float4(__fadd_rn(p4[j].x, __uint_as_float(rr[4 * j])), __fadd_rn(p4[j].y, __uint_as_float(rr[4 * j + 1])),
                                  __fadd_rn(p4[j].z, __uint_as_float(rr[4 * j + 2])), __fadd_rn(p4[j].w, __uint_as_float(rr[4 * j + 3])));
            else
              pp[j * BM] = make_float4(__uint_as_float(rr[4 * j]), __uint_as_float(rr[4 * j + 1]), __uint_as_float(rr[4 * j + 2]),
                                       __uint_as_float(rr[4 * j + 3]));
          }
        }
        tc_fence_before();
        release();
        return;
      }
      float hacc[HEAD_ROWS];
#pragma unroll
      for (int a = 0; a < HEAD_ROWS; ++a) hacc[a] = 0.0f;
#pragma unroll 1
      for (int c0 = grp * 32; c0 < BN; c0 += 32 * ngrp) {
        uint32_t rr[32];
        tmem_ld32(taddr + (uint32_t)c0, rr);
        const int n0 = nt * BN + c0;
        float4 b4[8];  // the chunk's bias (warp-uniform addresses): 8 vector loads in flight under the TMEM load
        if (!g.no_bias) {
#pragma unroll
          for (int j = 0; j < 8; ++j) b4[j] = __ldg(reinterpret_cast<const float4*>(g.bias + n0) + j);
        }
        float v[32];
        if (g.acc_in || nq > 1) {  // K-split: partial sums of the earlier launches / work items (plain loads)
          const float4* src = nq > 1 ? part + (c0 >> 2) * BM
                                     : reinterpret_cast<const float4*>(g.acc_in + row * (int64_t)(g.n_tiles * BN) + n0);
          const int sstep = nq > 1 ? BM : 1;
          float4 p4[8];
          if (nq > 1 || row < g.M) {
#pragma unroll
            for (int j = 0; j < 8; ++j) p4[j] = src[j * sstep];
          } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) p4[j] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
          }
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            v[4 * j] = __fadd_rn(p4[j].x, __uint_as_float(rr[4 * j]));
            v[4 * j + 1] = __fadd_rn(p4[j].y, __uint_as_float(rr[4 * j + 1]));
            v[4 * j + 2] = __fadd_rn(p4[j].z, __uint_as_float(rr[4 * j + 2]));
            v[4 * j + 3] = __fadd_rn(p4[j].w, __uint_as_float(rr[4 * j + 3]));
          }
        } else {
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(rr[j]);
        }
        if (!g.no_bias) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            v[4 * j] += b4[j].x;
            v[4 * j + 1] += b4[j].y;
            v[4 * j + 2] += b4[j].z;
            v[4 * j + 3] += b4[j].w;
          }
        }
        if (g.relu) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.0f);
        }
        if (g.out_mode == OUT_HEADS) {
          // policy/value heads fused into the epilogue (Connect4GNN.py:48-57): this tile's share of
          // logits[a] = sum_n E[row, n] * Wh[a, n]; the head weights are warp-uniform loads
          const int N = g.n_tiles * BN;
#pragma unroll
          for (int a = 0; a < HEAD_ROWS; ++a) {
            if (a < g.head_rows) {
              const float4* wr = reinterpret_cast<const float4*>(g.head_w + (size_t)a * N + n0);
              float s = hacc[a];
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const float4 w4 = __ldg(wr + j);
                s = fmaf(v[4 * j], w4.x, fmaf(v[4 * j + 1], w4.y, fmaf(v[4 * j + 2], w4.z, fmaf(v[4 * j + 3], w4.w, s))));
              }
              hacc[a] = s;
            }
          }
        } else if (g.out_mode == OUT_F32) {
          if (row < g.M) {
            float4* dst = reinterpret_cast<float4*>(g.out_f32 + row * (int64_t)(g.n_tiles * BN) + n0);
#pragma unroll
            for (int j = 0; j < 8; ++j) dst[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          }
        } else {
          // next GEMM's A operand: columns are its K index; 32 columns = 4 x 16-byte chunks of one image row
          const int kb = n0 / BK, koff = n0 % BK;
          const size_t tile = ((size_t)mt * NKB + kb) * A_STAGE_BYTES;
          if (TWO && g.f8) {  // fp16 image + FP8 correction rows [2^sa h | 2^(sa+11) h_lo], 16 elements per 16-byte chunk
            const float s_main = (float)(1 << F8_A_SCALE), s_lo = (float)(1 << (F8_A_SCALE + F8_LO_SHIFT));
#pragma unroll
            for (int c = 0; c < 2; ++c) {
              uint4 h0, h1;
              uint2 m0, m1, l0, l1;
              split8_f16f8(v + c * 16, s_main, s_lo, h0, m0, l0);
              split8_f16f8(v + c * 16 + 8, s_main, s_lo, h1, m1, l1);
              const int k0 = koff + c * 16;
              *reinterpret_cast<uint4*>(g.out_hi + tile + image_offset(r_local, k0)) = h0;
              *reinterpret_cast<uint4*>(g.out_hi + tile + image_offset(r_local, k0 + 8)) = h1;
              *reinterpret_cast<uint4*>(g.out_lo + tile + image_offset_bytes(r_local, k0)) = make_uint4(m0.x, m0.y, m1.x, m1.y);
              *reinterpret_cast<uint4*>(g.out_lo + tile + image_offset_bytes(r_local, 64 + k0)) = make_uint4(l0.x, l0.y, l1.x, l1.y);
            }
            continue;
          }
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            uint32_t hi[4], lo[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              split_pair(v[c * 8 + 2 * e], v[c * 8 + 2 * e + 1], hi[e], lo[e]);
            }
            const size_t off = tile + image_offset(r_local, koff + c * 8);
            *reinterpret_cast<uint4*>(g.out_hi + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            if (g.out_mode == OUT_IMG_HILO) *reinterpret_cast<uint4*>(g.out_lo + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
          }
        }
      }
      tc_fence_before();
      release();  // the accumulator is back with the MMA issuer (the partial head sums still go out below)
      if (g.out_mode == OUT_HEADS && row < g.M) {
        float* dst = g.head_part + ((size_t)row * (g.n_tiles * ngrp) + nt * ngrp + grp) * HEAD_STRIDE;
#pragma unroll
        for (int a = 0; a < HEAD_ROWS; ++a)
          if (a < g.head_rows) dst[a] = hacc[a];
      }
}

constexpr int KPART_MAX_CTAS = 256;                      // in-kernel K-split: per-CTA partial-sum tiles the scratch is sized for
constexpr int EPI_GROUPS = 2;                           // epilogue warps 4-7 and 8-11
constexpr int GEMM_THREADS = 128 + 128 * EPI_GROUPS;     // producer, MMA issuer, TMEM allocator, spare + the epilogue groups
template <int BN, bool TWO>
__global__ void __launch_bounds__(GEMM_THREADS, 1) gemm_bf16_tc_kernel(GemmArgs g) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // SWIZZLE_128B wants 1024-B alignment
  using S = Smem<BN, TWO>;
  constexpr int NS = S::NSTAGES;
  uint64_t* full = (uint64_t*)(smem + S::BAR_OFFSET);
  uint64_t* empty = full + NS;
  uint64_t* pfull = empty + NS;  // TWO: "the peer CTA's stage has landed", arrived remotely by the peer
  uint64_t* tfull = pfull + NS;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = (uint32_t*)(tempty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr uint32_t TMEM_COLS = 512;  // 2 accumulator stages of BN <= 256 fp32 columns
  const uint32_t rank = TWO ? cluster_ctarank() : 0u;
  if (g.dyn_rows) {  // row count decided on the device (compacted leaf batches): no host round trip
    const int64_t rows = *g.dyn_rows;
    if (rows < g.M) g.M = rows;
    g.m_tiles = (int)((g.M + BM - 1) / BM);
  }
  const int unit = TWO ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;      // scheduling unit: CTA or CTA pair
  const int n_units = TWO ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const int m_units = TWO ? (g.m_tiles + 1) / 2 : g.m_tiles;             // a pair owns two consecutive m-tiles

  if (warp == 1 && lane == 0) {
    for (int s = 0; s < NS; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
      mbar_init(&pfull[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull[a], 1);
      mbar_init(&tempty[a], (TWO ? 256 : 128) * EPI_GROUPS);
    }
    fence_barrier_init();
  }
  if (warp == 2) {
    if (TWO) tmem_alloc2(tmem_slot, TMEM_COLS);
    else tmem_alloc(tmem_slot, TMEM_COLS);
  }
  tc_fence_before();
  __syncthreads();
  if (TWO) cluster_sync_all();  // both CTAs' barriers exist before any remote arrive / multicast commit
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (TWO && g.f8) {
    // uniform block scales: every scale-factor byte the tensor core can read is the same power of two, so the
    // regions are written once (whatever the scale-factor layout) -- A: 2^-(sa+11), W: 2^-sw
    if (warp >= 4 && warp < 8) {
      const uint32_t lane_base = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
      tmem_st16_const(lane_base + SF_A_COL, ue8m0x4(-(F8_A_SCALE + F8_LO_SHIFT)));
      tmem_st16_const(lane_base + SF_W_COL, ue8m0x4(g.w_exp ? -(*g.w_exp) : 0));
      tmem_st16_const(lane_base + SF_SIDE_COL, ue8m0x4(g.side_exp ? -(*g.side_exp) : 0));
      tmem_st_wait();
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
  }

  const int nt_all = g.n_tiles + ((TWO && g.side_hi) ? 1 : 0);  // n-tile index g.n_tiles = the side tile
  const int total_tiles = m_units * nt_all;
  // CTA pair: a stage holds TWO operand pairs (60 KB per CTA, 3 stages) and feeds 8-12 MMAs per barrier
  // round trip.  bf16x3: hi and lo of both operands of one k-block -> all three products, so every operand
  // byte crosses L2 -> smem once instead of 1.5 times.  Plain bf16: two consecutive k-blocks.
  // Single CTA: one pair per stage; the bf16x3 split is walked as three K segments [Xhi|Xhi|Xlo] x [Whi|Wlo|Whi].
  const bool fused3 = TWO && g.x3;
  const bool dual = TWO && !g.x3;
  const int NSR = TWO ? 3 : NS;                                            // stages in use
  const uint32_t stage_bytes = TWO ? 2 * S::STAGE_BYTES : S::STAGE_BYTES;
  const int kb_total = fused3 ? (g.kbn ? g.kbn : g.KB) : dual ? (g.KB + 1) / 2 : (g.x3 ? 3 * g.KB : g.KB);
  const int kb_first = fused3 ? g.kb0 : 0;  // K-split launches (fused hi/lo stages only, checked by the launcher)
  const int nq = (fused3 && g.ksplit > 1) ? g.ksplit : 1;  // in-kernel K-split: work items per tile
  // f8 launches that issue only one of the two products (K-split: main quarters and the correction product go to
  // different accumulators; AZG_F8_TERMS diagnostics) fill only the half of the stage that product reads
  const bool need_hi = !(TWO && g.f8) || (g.f8 & 1), need_lo = !(TWO && g.f8) || (g.f8 & 2);

  if (warp == 0) {
    // ================= producer: bulk copies of operand tile images =================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int t = unit; t < total_tiles; t += n_units) {
        const int mt = (t / nt_all) * (TWO ? 2 : 1) + (int)rank, nt = t % nt_all;
        const bool side = TWO && nt == g.n_tiles;
        for (int kb = 0; kb < kb_total; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          uint8_t* sa = smem + stage * stage_bytes;
          if (side) {  // same stage layout, the weight part is this CTA's 16 rows of the [32 x 64] side tile
            const int k0 = dual ? 2 * kb : kb_first + kb, parts = (fused3 || k0 + 1 < g.KB) ? 2 : 1;
            mbar_expect_tx(&full[stage], (fused3 ? (int)need_hi + (int)need_lo : parts) * (A_STAGE_BYTES + SIDE_STAGE_BYTES));
            for (int pt = 0; pt < parts; ++pt) {
              if (fused3 && !(pt ? need_lo : need_hi)) continue;
              const int kk = fused3 ? k0 : k0 + pt;
              const size_t ao = ((size_t)mt * g.KB + kk) * A_STAGE_BYTES;
              const size_t wo = (size_t)kk * (2 * SIDE_STAGE_BYTES) + (size_t)rank * SIDE_STAGE_BYTES;
              const bool lo = fused3 && pt == 1;
              bulk_g2s(sa + pt * S::STAGE_BYTES, (lo ? g.a_lo : g.a_hi) + ao, A_STAGE_BYTES, &full[stage]);
              bulk_g2s(sa + pt * S::STAGE_BYTES + A_STAGE_BYTES, (lo ? g.side_lo : g.side_hi) + wo, SIDE_STAGE_BYTES, &full[stage]);
            }
            if (++stage == NSR) {
              stage = 0;
              phase ^= 1;
            }
            continue;
          }
          if (dual) {  // [A(k0) | W(k0) half | A(k0+1) | W(k0+1) half]; an odd K leaves the last second half unused
            const int k0 = 2 * kb, parts = (k0 + 1 < g.KB) ? 2 : 1;
            mbar_expect_tx(&full[stage], parts * S::STAGE_BYTES);
            for (int pt = 0; pt < parts; ++pt) {
              const size_t ao = ((size_t)mt * g.KB + k0 + pt) * A_STAGE_BYTES;
              const size_t wo = ((size_t)nt * g.KB + k0 + pt) * S::W_TILE_BYTES + (size_t)rank * S::W_STAGE_BYTES;
              bulk_g2s(sa + pt * S::STAGE_BYTES, g.a_hi + ao, A_STAGE_BYTES, &full[stage]);
              bulk_g2s(sa + pt * S::STAGE_BYTES + A_STAGE_BYTES, g.w_hi + wo, S::W_STAGE_BYTES, &full[stage]);
            }
            if (++stage == NSR) {
              stage = 0;
              phase ^= 1;
            }
            continue;
          }
          mbar_expect_tx(&full[stage], fused3 ? ((uint32_t)need_hi + (uint32_t)need_lo) * S::STAGE_BYTES : stage_bytes);
          if (fused3) {  // [A_hi | W_hi half | A_lo | W_lo half]
            const size_t ao = ((size_t)mt * g.KB + kb_first + kb) * A_STAGE_BYTES;
            const size_t wo = ((size_t)nt * g.KB + kb_first + kb) * S::W_TILE_BYTES + (size_t)rank * S::W_STAGE_BYTES;
            if (need_hi) {
              bulk_g2s(sa, g.a_hi + ao, A_STAGE_BYTES, &full[stage]);
              bulk_g2s(sa + A_STAGE_BYTES, g.w_hi + wo, S::W_STAGE_BYTES, &full[stage]);
            }
            if (need_lo) {
              bulk_g2s(sa + S::STAGE_BYTES, g.a_lo + ao, A_STAGE_BYTES, &full[stage]);
              bulk_g2s(sa + S::STAGE_BYTES + A_STAGE_BYTES, g.w_lo + wo, S::W_STAGE_BYTES, &full[stage]);
            }
          } else {
            // x3: [Xhi|Xhi|Xlo] against [Whi|Wlo|Whi]
            const int seg = g.x3 ? kb / g.KB : 0, kk = g.x3 ? kb % g.KB : kb;
            const uint8_t* a_src = (seg == 2 ? g.a_lo : g.a_hi) + ((size_t)mt * g.KB + kk) * A_STAGE_BYTES;
            const uint8_t* w_src = (seg == 1 ? g.w_lo : g.w_hi) + ((size_t)nt * g.KB + kk) * S::W_TILE_BYTES +
                                   (size_t)rank * S::W_STAGE_BYTES;  // pair: this CTA's half of the tile's rows
            bulk_g2s(sa, a_src, A_STAGE_BYTES, &full[stage]);
            bulk_g2s(sa + A_STAGE_BYTES, w_src, S::W_STAGE_BYTES, &full[stage]);
          }
          if (++stage == NSR) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer: one thread (of the leader CTA when paired) =================
    if (lane == 0 && rank == 0) {
      constexpr uint32_t idesc_main = make_idesc(TWO ? 2 * BM : BM, BN);
      constexpr uint32_t idesc_side = make_idesc(TWO ? 2 * BM : BM, SIDE_N);
      constexpr uint32_t idesc_main_h = make_idesc_f16(2 * BM, BN), idesc_side_h = make_idesc_f16(2 * BM, SIDE_N);
      constexpr uint32_t idesc_main_q = make_idesc_mxf8(2 * BM, BN), idesc_side_q = make_idesc_mxf8(2 * BM, SIDE_N);
      const bool f8 = TWO && g.f8;
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int t = unit; t < total_tiles; t += n_units)
      for (int kq = 0; kq < nq; ++kq) {  // in-kernel K-split: one accumulator per quarter of K
        const int kq_n = nq > 1 ? ksplit_begin(kb_total, kq + 1, nq) - ksplit_begin(kb_total, kq, nq) : kb_total;
        if (TWO) mbar_wait_cluster(&tempty[acc], acc_phase ^ 1);  // both CTAs' epilogues drained this accumulator
        else mbar_wait(&tempty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
        const bool side_tile = TWO && t % nt_all == g.n_tiles;
        const uint32_t idesc = side_tile ? (f8 ? idesc_side_h : idesc_side) : (f8 ? idesc_main_h : idesc_main);
        const uint32_t idesc_q = side_tile ? idesc_side_q : idesc_main_q;
        const uint32_t sfa = tmem_base + SF_A_COL, sfb = tmem_base + (side_tile ? SF_SIDE_COL : SF_W_COL);
        for (int kb = 0; kb < kq_n; ++kb) {
          mbar_wait(&full[stage], phase);  // operands have landed
          if (TWO) mbar_wait_cluster(&pfull[stage], phase);  // ... in the peer CTA as well
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * stage_bytes);
          const uint64_t adesc = make_smem_desc(sa);
          const uint64_t bdesc = make_smem_desc(sa + A_STAGE_BYTES);
          uint32_t accf = kb != 0;  // f8 mode with a term switched off (AZG_F8_TERMS, diagnostics): first MMA of the tile overwrites
          if (!f8 || (g.f8 & 1)) {
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) {  // advance 32 bytes (2 x 16-byte units) per K=16 step
              if (TWO) umma2_bf16(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kb | k) != 0);
              else umma_bf16(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kb | k) != 0);
            }
            accf = 1;
          }
          if (TWO && dual && 2 * kb + 1 < g.KB) {  // second k-block of the stage
            const uint64_t adesc1 = make_smem_desc(sa + S::STAGE_BYTES);
            const uint64_t bdesc1 = make_smem_desc(sa + S::STAGE_BYTES + A_STAGE_BYTES);
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) umma2_bf16(d_tmem, adesc1 + (uint64_t)(2 * k), bdesc1 + (uint64_t)(2 * k), idesc, 1);
          }
          if (TWO && fused3 && f8) {  // + the K-concatenated FP8 correction product (4 x K = 32) from the same stage
            if (g.f8 & 2) {
              const uint64_t adesc_lo = make_smem_desc(sa + S::STAGE_BYTES);
              const uint64_t bdesc_lo = make_smem_desc(sa + S::STAGE_BYTES + A_STAGE_BYTES);
#pragma unroll
              for (int k = 0; k < 4; ++k)
                umma2_mxf8(d_tmem, adesc_lo + (uint64_t)(2 * k), bdesc_lo + (uint64_t)(2 * k), idesc_q, sfa, sfb, accf | (uint32_t)k);
            }
          } else if (TWO && fused3) {  // + Xhi Wlo^T + Xlo Whi^T from the same stage
            const uint64_t adesc_lo = make_smem_desc(sa + S::STAGE_BYTES);
            const uint64_t bdesc_lo = make_smem_desc(sa + S::STAGE_BYTES + A_STAGE_BYTES);
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) umma2_bf16(d_tmem, adesc + (uint64_t)(2 * k), bdesc_lo + (uint64_t)(2 * k), idesc, 1);
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) umma2_bf16(d_tmem, adesc_lo + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, 1);
          }
          if (TWO) umma2_commit(&empty[stage]);  // frees the smem slot (in both CTAs) once these MMAs have read it
          else umma_commit(&empty[stage]);
          if (++stage == NSR) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (TWO) umma2_commit(&tfull[acc]);  // accumulator complete -> epilogue (of both CTAs)
        else umma_commit(&tfull[acc]);
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    } else if (TWO && lane == 0) {
      // peer CTA: relay "my stage has landed" to the leader (a bulk copy can only signal its own CTA)
      const uint32_t leader_pfull = map_to_cta(&pfull[0], 0);
      int stage = 0;
      uint32_t phase = 0;
      for (int t = unit; t < total_tiles; t += n_units) {
        for (int kb = 0; kb < kb_total; ++kb) {
          mbar_wait(&full[stage], phase);
          mbar_arrive_cluster(leader_pfull + (uint32_t)stage * 8u);
          if (++stage == NSR) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp >= 4) {
    // ================= epilogue: TMEM -> registers -> bias/ReLU -> HBM =================
    // The epilogue of a 128 x 224 tile takes ~40k cycles with four warps (global loads of bias / head weights and the
    // scattered image stores), as long as the 8-MMA main loop of the fp16+FP8 split (ncu source view, r02 v1: epilogue
    // warps busy 68 % of the time, tensor pipe 78 %): two groups of four warps split the tile's 32-column chunks.
    const int q = warp & 3;              // TMEM lane quarter this warp may read
    const int r_local = q * 32 + lane;   // row of the tile == TMEM lane
    const int grp = (warp - 4) >> 2;
    int acc = 0;
    uint32_t acc_phase = 0;
    const uint32_t leader_tempty = TWO ? map_to_cta(&tempty[0], 0) : 0u;
    float4* part = nq > 1 ? reinterpret_cast<float4*>(g.kpart) + (size_t)blockIdx.x * (BM * (BN / 4)) + r_local : nullptr;  // this thread's row of the CTA's partial tile
    for (int t = unit; t < total_tiles; t += n_units)
    for (int kq = 0; kq < nq; ++kq) {
      const int mt = (t / nt_all) * (TWO ? 2 : 1) + (int)rank, nt = t % nt_all;
      mbar_wait(&tfull[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BN);
      if (TWO) epilogue_tile<BN, TWO>(g, taddr, mt, nt, r_local, grp, EPI_GROUPS, [&] { mbar_arrive_cluster(leader_tempty + (uint32_t)acc * 8u); }, part, kq, nq);
      else epilogue_tile<BN, TWO>(g, taddr, mt, nt, r_local, grp, EPI_GROUPS, [&] { mbar_arrive(&tempty[acc]); });
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (TWO) cluster_sync_all();  // the leader's MMAs read the peer's shared memory: leave together
  if (warp == 2) {
    tc_fence_after();
    if (TWO) tmem_dealloc2(tmem_base, TMEM_COLS);
    else tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ---- image builders --------------------------------------------------------------------------
// fp32 row-major [rows, K] -> bf16 tile images (hi, optionally lo) with R-row tiles.
// One thread per 16-byte output chunk (8 elements): 32-byte coalesced reads, 16-byte writes.
// f8_mode 1 / 2: AZG_PREC_F16F8 activation / weight format (fp16 image + FP8 correction rows, scale 2^*f8_exp for weights)
__global__ void __launch_bounds__(256) f32_to_image_kernel(const float* __restrict__ src, int64_t rows, int64_t rows_padded,
                                                           int K, int R, uint8_t* __restrict__ hi, uint8_t* __restrict__ lo,
                                                           int f8_mode = 0, const int32_t* __restrict__ f8_exp = nullptr) {
  const int chunks_per_row = K / 8;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows_padded * chunks_per_row) return;
  const int64_t row = idx / chunks_per_row;
  const int c = (int)(idx % chunks_per_row);
  float x[8];
  if (row < rows) {
    const float4 a = *reinterpret_cast<const float4*>(src + row * K + c * 8);
    const float4 b = *reinterpret_cast<const float4*>(src + row * K + c * 8 + 4);
    x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j) x[j] = 0.0f;
  }
  const int KB = K / BK;
  const int64_t tile_row = row / R;
  const int r = (int)(row % R), kb = (c * 8) / BK, k = (c * 8) % BK;
  if (f8_mode) {
    const int e = f8_mode == 2 ? *f8_exp : F8_A_SCALE;
    split_store_f16f8(x, hi, lo, ((size_t)tile_row * KB + kb) * ((size_t)R * 128), r, k, ldexpf(1.0f, e), ldexpf(1.0f, e + F8_LO_SHIFT),
                      f8_mode == 2);
    return;
  }
  uint32_t h[4], l[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    split_pair(x[2 * e], x[2 * e + 1], h[e], l[e]);
  }
  const size_t off = ((size_t)tile_row * KB + kb) * ((size_t)R * 128) + image_offset(r, k);
  *reinterpret_cast<uint4*>(hi + off) = make_uint4(h[0], h[1], h[2], h[3]);
  if (lo) *reinterpret_cast<uint4*>(lo + off) = make_uint4(l[0], l[1], l[2], l[3]);
}

inline int pick_bn(int F) {
  if (F % 224 == 0) return 224;
  if (F % 256 == 0) return 256;
  if (F % 160 == 0) return 160;
  return 0;
}
// AZG_PREC_F16F8 keeps 64 TMEM columns for its scale factors: two accumulator stages of <= 224 columns
inline int pick_bn_f8(int F) {
  if (F % 224 == 0) return 224;
  if (F % 160 == 0) return 160;
  if (F % 128 == 0) return 128;
  return 0;
}

// max |w| over a tensor (bits of a non-negative float order like unsigned integers) -> *exp = the largest e with
// 2^e max|w| <= 448 (e4m3 range), so the scaled weights use the top binades of the format
__global__ void __launch_bounds__(256) absmax_kernel(const float* __restrict__ w, int64_t n, uint32_t* __restrict__ bits) {
  float m = 0.0f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) m = fmaxf(m, fabsf(w[i]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(bits, __float_as_uint(m));
}
__global__ void scale_exp_kernel(const uint32_t* __restrict__ bits, int32_t* __restrict__ exp_out) {
  const float m = __uint_as_float(*bits);
  int e = 0;
  if (m > 0.0f && m < INFINITY) {
    e = (int)floorf(log2f(448.0f / m));
    while (ldexpf(m, e) > 448.0f) --e;  // log2f rounding
    while (ldexpf(m, e + 1) <= 448.0f) ++e;
    e = e > 100 ? 100 : (e < -100 ? -100 : e);
  }
  *exp_out = e;
}
// writes the scale exponent of `w` to *exp_out (device); `bits` is a 4-byte device scratch word
int weight_scale_exp(const float* w, int64_t n, uint32_t* bits, int32_t* exp_out, cudaStream_t st) {
  AZG_CUDA_CHECK(cudaMemsetAsync(bits, 0, 4, st));
  const int grid = (int)((n + 255) / 256 < 1184 ? (n + 255) / 256 : 1184);
  absmax_kernel<<<grid, 256, 0, st>>>(w, n, bits);
  AZG_LAUNCH_CHECK();
  scale_exp_kernel<<<1, 1, 0, st>>>(bits, exp_out);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

static int f8_terms() {  // AZG_F8_TERMS=1 / 2: only the fp16 product / only the FP8 correction product (diagnostics)
  static int terms = -1;
  if (terms < 0) {
    const char* e = getenv("AZG_F8_TERMS");
    terms = e ? (atoi(e) & 3) : 3;
    if (terms == 0) terms = 3;
  }
  return terms;
}

template <int BN, bool TWO>
int launch_gemm_impl(const GemmArgs& g, cudaStream_t st) {
  static bool configured = false;
  int dev = 0, sms = 0;
  AZG_CUDA_CHECK(cudaGetDevice(&dev));
  AZG_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  using S = Smem<BN, TWO>;
  if (!configured) {
    AZG_CUDA_CHECK(cudaFuncSetAttribute(gemm_bf16_tc_kernel<BN, TWO>, cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL));
    configured = true;
  }
  const int units = (TWO ? (g.m_tiles + 1) / 2 : g.m_tiles) * (g.n_tiles + ((TWO && g.side_hi) ? 1 : 0));
  int grid = TWO ? 2 * (units < sms / 2 ? units : sms / 2) : (units < sms ? units : sms);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(GEMM_THREADS);
  cfg.dynamicSmemBytes = S::TOTAL;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = TWO ? 2 : 1;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  AZG_REQUIRE(g.ksplit <= 1 || grid <= KPART_MAX_CTAS, "tcgen05 GEMM: %d CTAs exceed the partial-sum scratch of the in-kernel K-split", grid);
  AZG_CUDA_CHECK(cudaLaunchKernelEx(&cfg, gemm_bf16_tc_kernel<BN, TWO>, g));
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}


// Tried and removed (round 2): a variant in which a CTA pair computes two n-tiles per activation stage (256 x 448 super-tile,
// 44 KB sub-stages, fills 49 instead of 67 B/clk per SM).  Its two 224-column accumulators fill TMEM, so they cannot be
// double-buffered and the epilogue (tens of thousands of cycles per tile, see the epilogue comment in gemm_bf16_tc_kernel)
// is exposed: 5.8 ms instead of 4.1 ms for the two contractions.

// Tile widths of 128 columns and more run on the CTA-pair kernel (BN/2 weight rows per CTA, a multiple of 8), 64 on the
// single-CTA kernel.  A pair owns two consecutive m-tiles, so the A image of a pair launch must cover an even number of
// m-tiles even when m_tiles is odd: every caller pads its activation images to a multiple of 2 * BM rows.
template <int BN>
int launch_gemm(const GemmArgs& g, cudaStream_t st) {
  const bool ksplit_launch = g.kbn || g.kb0 || g.acc_in || g.no_bias || g.side_acc;
  if constexpr (BN >= 128) {
    AZG_REQUIRE(!ksplit_launch || (g.x3 && g.kb0 >= 0 && g.kb0 + g.kbn <= g.KB),
                "tcgen05 GEMM: K-split launches run on the split precisions only");
    AZG_REQUIRE(g.ksplit <= 1 || (g.x3 && g.kpart && !g.kbn && !g.acc_in && g.KB >= g.ksplit),
                "tcgen05 GEMM: the in-kernel K-split runs on the split precisions only");
    AZG_REQUIRE(!g.f8 || (BN <= 224 && g.x3), "tcgen05 GEMM: the fp16+FP8 split needs a tile width of 128..224 columns");
    return launch_gemm_impl<BN, true>(g, st);
  } else {
    AZG_REQUIRE(!ksplit_launch && g.ksplit <= 1 && !g.f8 && !g.side_hi,
                "tcgen05 GEMM: the K-split, the fp16+FP8 split and the side tile run on the CTA-pair kernel (tile width >= 128)");
    return launch_gemm_impl<BN, false>(g, st);
  }
}

// partial head-sum slots per n-tile (one per epilogue group)
int head_slots_per_tile(const GemmArgs&) { return EPI_GROUPS; }

int run_gemm(int BN, const GemmArgs& g, cudaStream_t st) {
  switch (BN) {
    case 224: return launch_gemm<224>(g, st);
    case 256: return launch_gemm<256>(g, st);
    case 160: return launch_gemm<160>(g, st);
    case 128: return launch_gemm<128>(g, st);
    case 64: return launch_gemm<64>(g, st);
  }
  azg_set_error("tcgen05 GEMM: no tile width for this feature size");
  return AZG_ERR_INVALID;
}

int to_image(const float* src, int64_t rows, int64_t rows_padded, int K, int R, uint8_t* hi, uint8_t* lo, cudaStream_t st,
             int f8_mode = 0, const int32_t* f8_exp = nullptr) {
  const int64_t n = rows_padded * (K / 8);
  f32_to_image_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(src, rows, rows_padded, K, R, hi, lo, f8_mode, f8_exp);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}


// ---- Connect4 trunk on the tensor cores ------------------------------------------------------
// conv2 (32 -> 64 channels, 3x3, pad 1) as an implicit GEMM:  rows m = (board b, cell p),
// K = (tap, cin) = 9*32 = 288 (padded to 320 = 5 k-blocks), N = 64 output channels.
constexpr int C2_K = 320, C2_KB = C2_K / BK;

// conv2 weights [64,32,3,3] -> [64 x 320] image, k = tap*32 + cin (zero padded)
__global__ void conv2_weight_image_kernel(const float* __restrict__ w2, uint8_t* __restrict__ hi, uint8_t* __restrict__ lo) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 64 * (C2_K / 8)) return;
  const int co = idx / (C2_K / 8), c = idx % (C2_K / 8);
  float x8[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int k = c * 8 + e, tap = k >> 5, ci = k & 31;
    x8[e] = (k < 288) ? w2[(co * 32 + ci) * 9 + tap] : 0.0f;
  }
  const size_t off = (size_t)(c >> 3) * (64 * 128) + image_offset(co, (c & 7) * 8);
  split_store(x8, hi, lo, off);
}

// Linear weight [N, F] whose input index is the reference's flatten order k = co*nn + p
// (Connect4Net.py:49) -> image over the feature image's order k' = p*64 + co
__global__ void __launch_bounds__(256) permuted_weight_image_kernel(const float* __restrict__ w, int N, int F, int nn, int R,
                                                                    uint8_t* __restrict__ hi, uint8_t* __restrict__ lo,
                                                                    const int32_t* __restrict__ f8_exp = nullptr) {
  const int chunks = F / 8;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)N * chunks) return;
  const int row = (int)(idx / chunks), c = (int)(idx % chunks);
  float x8[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int kp = c * 8 + e, pc = kp >> 6, co = kp & 63;
    x8[e] = w[(size_t)row * F + co * nn + pc];
  }
  const int KB = F / BK;
  if (f8_exp) {  // AZG_PREC_F16F8 weight format
    const int e = *f8_exp;
    split_store_f16f8(x8, hi, lo, ((size_t)(row / R) * KB + (c >> 3)) * ((size_t)R * 128), row % R, (c & 7) * 8, ldexpf(1.0f, e),
                      ldexpf(1.0f, e + F8_LO_SHIFT), true);
    return;
  }
  const size_t off = ((size_t)(row / R) * KB + (c >> 3)) * ((size_t)R * 128) + image_offset(row % R, (c & 7) * 8);
  split_store(x8, hi, lo, off);
}

// logits = fixed-order sum of the per-tile partial head sums + bias; then exp(log_softmax) and tanh
// AZG_EVAL_FOLD: no non-linearity lies between output_transform.2 and the policy/value heads
// (gnn_utils.py:99-103 -> Connect4GNN.py:48-57), so   heads(W2 h + b2) = ([Wp; Wv] W2) h + ([Wp; Wv] b2 + [bp; bv]).
// fold_w[a, j] = sum_n hc[a, n] W2[n, j]  (fp64 accumulation, once per weight version, n split over FOLD_SPLITS blocks and
// reduced in fixed order); hc = concatenated heads [32, F].
constexpr int FOLD_SPLITS = 16;
// blockIdx.y owns the n range [y*per, (y+1)*per): part[y][a][j] = sum_n hc[a, n] W2[n, j] in fp64
__global__ void __launch_bounds__(128) fold_heads_partial_kernel(const float* __restrict__ hc, const float* __restrict__ w2, int rows,
                                                                 int F, int per, double* __restrict__ part) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= F) return;
  const int n0 = blockIdx.y * per, n1 = n0 + per < F ? n0 + per : F;
  double acc[HEAD_ROWS];
#pragma unroll
  for (int a = 0; a < HEAD_ROWS; ++a) acc[a] = 0.0;
  for (int n = n0; n < n1; ++n) {
    const double w = (double)w2[(size_t)n * F + j];
#pragma unroll
    for (int a = 0; a < HEAD_ROWS; ++a)
      if (a < rows) acc[a] += (double)__ldg(hc + (size_t)a * F + n) * w;
  }
#pragma unroll
  for (int a = 0; a < HEAD_ROWS; ++a)
    if (a < rows) part[((size_t)blockIdx.y * HEAD_ROWS + a) * F + j] = acc[a];
}

// fold_w = fixed-order sum of the partials; fold_b[a] = sum_n hc[a, n] b2[n] + bias32[a]
__global__ void __launch_bounds__(128) fold_heads_finish_kernel(const double* __restrict__ part, const float* __restrict__ hc,
                                                                const float* __restrict__ b2, const float* __restrict__ bias32,
                                                                int rows, int F, float* __restrict__ fold_w,
                                                                float* __restrict__ fold_b) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < F) {
    for (int a = 0; a < rows; ++a) {
      double s = 0.0;
      for (int y = 0; y < FOLD_SPLITS; ++y) s += part[((size_t)y * HEAD_ROWS + a) * F + j];
      fold_w[(size_t)a * F + j] = (float)s;
    }
  } else if (j - F < rows) {
    const int a = j - F;
    double acc = (double)bias32[a];
    for (int n = 0; n < F; ++n) acc += (double)hc[(size_t)a * F + n] * (double)b2[n];
    fold_b[a] = (float)acc;
  }
}

__global__ void heads_finalize_kernel(const float* __restrict__ part, int n_tiles, int A, const float* __restrict__ bp,
                                      const float* __restrict__ bv, int64_t B, const int32_t* __restrict__ dyn_rows,
                                      float* __restrict__ pi, float* __restrict__ v) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= B || (dyn_rows && row >= *dyn_rows)) return;
  float logit[HEAD_ROWS];
#pragma unroll
  for (int a = 0; a < HEAD_ROWS; ++a) logit[a] = 0.0f;
  const float* p = part + (size_t)row * n_tiles * HEAD_STRIDE;
  for (int t = 0; t < n_tiles; ++t)
#pragma unroll
    for (int a = 0; a < HEAD_ROWS; ++a)
      if (a <= A) logit[a] += p[t * HEAD_STRIDE + a];
  float m = -INFINITY;
#pragma unroll
  for (int a = 0; a < HEAD_ROWS; ++a)
    if (a < A) { logit[a] += __ldg(bp + a); m = fmaxf(m, logit[a]); }
  float sum = 0.0f;
#pragma unroll
  for (int a = 0; a < HEAD_ROWS; ++a)
    if (a < A) sum += expf(logit[a] - m);
  const float lse = logf(sum);
  float vraw = 0.0f;
#pragma unroll
  for (int a = 0; a < HEAD_ROWS; ++a) {
    if (a < A) pi[row * A + a] = expf((logit[a] - m) - lse);
    if (a == A) vraw = logit[a];
  }
  v[row] = tanhf(vraw + __ldg(bv));
}

// [policy rows ; value row ; zero rows up to 32] in the reference's input order, fp32 (fused-heads
// epilogue of GEMM-2 and source of the std-heads weight image)
__global__ void concat_heads_kernel(const float* __restrict__ wp, const float* __restrict__ wv, const float* __restrict__ bp,
                                    const float* __restrict__ bv, int A, int F, float* __restrict__ out,
                                    float* __restrict__ bias32) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < 32) bias32[idx] = idx < A ? bp[idx] : (idx == A ? bv[0] : 0.0f);
  if (idx >= (int64_t)32 * F) return;
  const int row = (int)(idx / F), k = (int)(idx % F);
  out[idx] = row < A ? wp[(size_t)row * F + k] : (row == A ? wv[k] : 0.0f);
}

// std heads from the [B,32] logits block produced by GEMM-1's side tile (bias already added)
__global__ void heads32_finalize_kernel(const float* __restrict__ lg, int A, int64_t B, const int32_t* __restrict__ dyn_rows,
                                        float* __restrict__ pi, float* __restrict__ v) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= B || (dyn_rows && row >= *dyn_rows)) return;
  const float* x = lg + row * 32;
  float m = -INFINITY;
  for (int a = 0; a < A; ++a) m = fmaxf(m, x[a]);
  float sum = 0.0f;
  for (int a = 0; a < A; ++a) sum += expf(x[a] - m);
  const float lse = logf(sum);
  for (int a = 0; a < A; ++a) pi[row * A + a] = expf((x[a] - m) - lse);
  v[row] = tanhf(x[A]);
}

// ---- fused trunk: encode + conv1 + conv2 in one kernel on the tensor cores ----------------------------------------------
// One persistent CTA per SM, 20 warps.  conv2 is an implicit GEMM over SHIFTED operand descriptors:
//   * relu(conv1) of a tile's boards is stored in a padded plane of 128-byte cells [32 ch hi (64 B) | 32 ch lo (64 B)],
//     SWIZZLE_128B by the cell index, raster pitch n+1: the right border of a board row IS the left border of the next row
//     and the bottom border row of a board IS the top border row of the next board, so board b's cell (x, y) sits at plane
//     cell b (n+1)^2 + (x+1)(n+1) + (y+1);
//   * GEMM row r = b (n+1)^2 + x (n+1) + y (the position of tap (0,0)); tap (kx, ky) of EVERY row is then plane cell
//     r + kx (n+1) + ky: the A operand of a tap is the same 128 rows at a different START ADDRESS (any multiple of 128 B:
//     the tensor core applies the 128-byte swizzle to absolute shared-memory address bits, so a plane written with
//     chunk ^ (cell & 7) reads back correctly from every start; measured on B200 -- with the descriptor's base-offset
//     field set to the start's phase the results are WRONG, with the field left 0 they equal an explicit im2col operand
//     bit for bit), K-advance inside the 128-byte cell selects hi / lo and the 16-channel half.
//     18 K = 16 steps (9 taps x 2) against the [64 x 320] conv2 weight image, no patch copies, no padded k-block.
//     (Copying the nine patches of every cell into operand stages instead cost 320 KB of shared-memory -> shared-memory
//     traffic per 128-row tile on top of the tensor core's own 280 KB of operand reads: 1.04-1.12 instead of 0.61-0.71 ms
//     per step of 65,536 positions, profiles/r01_trunk_fused_v8.txt and r02_trunk_fused2.txt.)
// Rows between boards compute garbage from border / neighbouring cells and are dropped by the epilogue (n = 7: 2 boards per
// tile, rows 0-54 and 64-118).
// conv1 runs on the tensor core too: the builder warps (two threads per tile row) encode the 3x3 neighbourhood of the row's
// cell straight from the packed position (bits -> bf16 {-1, 0, +1}), written three times along K into a conv1 operand stage,
// against [w_hi | w_mid | w_lo] (three bf16 terms = the full fp32 weight, the {-1,0,1} operand is exact, fp32 accumulation):
// 3 MMAs of 128 x 32 x 16 per tile; the builders read the result back from TMEM (+bias, ReLU, hi/lo split into the plane).
// (As FFMA with lanes = channels and broadcast LDS of the planes, conv1 took 42 % of the builders' time: 18 LDS per two
// cells queued behind the tensor core's own shared-memory reads; on the tensor core it is 3 MMAs and one tcgen05.ld per
// thread.)  Planes, conv1 operand stages and conv1 TMEM regions are double-buffered so that tile i+1's conv1 and plane
// write-back run under tile i's 36 conv2 MMAs.
constexpr int TR_W_BYTES = C2_KB * 64 * 128;  // conv2 weight image [64 x 320] bf16 = 40 KB
constexpr int TR_W1_BYTES = 32 * 128;         // conv1 weight image [32 x 64] bf16: cols 0-8 hi, 16-24 mid, 32-40 lo
struct TrunkArgs {
  const uint64_t* states;
  const float *w1, *b1, *b2;   // conv1 weights/bias, conv2 bias
  const uint8_t *w_hi, *w_lo;  // conv2 weight images
  uint8_t *f_hi, *f_lo;        // feature image out
  int64_t B;
  int n;
  const int32_t* dyn_rows;  // optional device scalar: number of positions this launch (<= B)
  int out_f8;               // feature image in the AZG_PREC_F16F8 activation format (the convolutions stay bf16x3)
};

constexpr int T2_PLANE_CELLS = 152;                       // 128 rows + 2 (n+1) + 2 tap reach, n <= 8
constexpr int T2_PLANE_BYTES = T2_PLANE_CELLS * 128;      // 19 KB, 1024-byte multiple

template <bool X3>
struct Trunk2Smem {
  static constexpr int W_OFF = 0;
  static constexpr int W1_OFF = (X3 ? 2 : 1) * TR_W_BYTES;
  static constexpr int PLANE_OFF = W1_OFF + TR_W1_BYTES;
  static constexpr int C1_OFF = PLANE_OFF + 2 * T2_PLANE_BYTES;
  static constexpr int STG_OFF = C1_OFF + 2 * A_STAGE_BYTES;  // epilogue staging: 128 rows x [128 B hi image row | 128 B lo image row]
  static constexpr int MISC_OFF = STG_OFF + 128 * 256;
  static constexpr int TOTAL = MISC_OFF + 1024 + 1024;
};

constexpr int T2_THREADS = 640;  // 8 builder warps, MMA, TMEM/barrier setup, 2 idle, 2 x 4 epilogue warps

// (A CTA-pair version -- every tcgen05.mma issued once for two CTAs' tiles, cta_group::2 -- was bit-identical and not faster,
// 0.655 vs 0.63-0.67 ms: the instruction count is not the bound, profiles/r02_trunk_fused2.txt.)
template <bool X3>
__global__ void __launch_bounds__(T2_THREADS, 1) c4_trunk2_tc_kernel(TrunkArgs t) {
  using S = Trunk2Smem<X3>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* w_s = smem + S::W_OFF;
  uint8_t* w1img = smem + S::W1_OFF;
  uint8_t* planes = smem + S::PLANE_OFF;
  uint8_t* c1st = smem + S::C1_OFF;
  uint64_t* c1_full = (uint64_t*)(smem + S::MISC_OFF);  // [2] conv1 operand written (256 builders)
  uint64_t* c1_free = c1_full + 2;                       // [2] conv1 MMAs have read the operand stage
  uint64_t* c1_done = c1_free + 2;                       // [2] conv1 result is in its TMEM region
  uint64_t* c1_tfree = c1_done + 2;                      // [2] builders have read the conv1 TMEM region (256)
  uint64_t* pl_full = c1_tfree + 2;                      // [2] plane written (256 builders)
  uint64_t* pl_free = pl_full + 2;                       // [2] conv2 MMAs have read the plane
  uint64_t* tfull = pl_free + 2;                         // [2] accumulator complete
  uint64_t* tempty = tfull + 2;                          // [2] accumulator drained (128 epilogue threads)
  uint64_t* wbar = tempty + 2;
  uint32_t* tmem_slot = (uint32_t*)(wbar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n = t.n, nn = n * n, rp = n + 1, bp = rp * rp;  // row pitch and board pitch of the shared-border raster
  const int G = (127 - (nn + n - 2)) / bp + 1;                // boards per 128-row tile
  if (t.dyn_rows && *t.dyn_rows < t.B) t.B = *t.dyn_rows;
  const int64_t tiles = (t.B + G - 1) / G;
  constexpr int BN = 64;
  constexpr int ACC_COLS = X3 ? 128 : 64;
  constexpr uint32_t TMEM_COLS = 512;
  constexpr uint32_t C1_COL = 2 * ACC_COLS;  // two conv1 regions of 32 columns

  for (int i = threadIdx.x; i < 2 * T2_PLANE_BYTES / 16; i += blockDim.x) reinterpret_cast<uint4*>(planes)[i] = make_uint4(0, 0, 0, 0);
  for (int i = threadIdx.x; i < 2 * A_STAGE_BYTES / 16; i += blockDim.x) reinterpret_cast<uint4*>(c1st)[i] = make_uint4(0, 0, 0, 0);
  for (int i = threadIdx.x; i < 32 * 64; i += blockDim.x) {  // conv1 weights as three bf16 terms along K (Connect4Net.py:32)
    const int ch = i >> 6, col = i & 63, term = col >> 4, k = col & 15;
    float v = 0.0f;
    if (term < 3 && k < 9) {
      const float w = t.w1[ch * 9 + k];
      const float hi = __bfloat162float(__float2bfloat16_rn(w));
      const float mid = __bfloat162float(__float2bfloat16_rn(w - hi));
      v = term == 0 ? hi : term == 1 ? mid : (w - hi) - mid;
    }
    *reinterpret_cast<__nv_bfloat16*>(w1img + image_offset(ch, col)) = __float2bfloat16_rn(v);
  }
  if (warp == 9 && lane == 0) {
    for (int k = 0; k < 2; ++k) {
      mbar_init(&c1_full[k], 256);
      mbar_init(&c1_free[k], 1);
      mbar_init(&c1_done[k], 1);
      mbar_init(&c1_tfree[k], 256);
      mbar_init(&pl_full[k], 256);
      mbar_init(&pl_free[k], 1);
      mbar_init(&tfull[k], 1);
      mbar_init(&tempty[k], 256);
    }
    mbar_init(wbar, 1);
    fence_barrier_init();
  }
  if (warp == 9) tmem_alloc(tmem_slot, TMEM_COLS);
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 9) {
    if (lane == 0) {  // conv2 weight images -> smem, once
      mbar_expect_tx(wbar, (X3 ? 2 : 1) * TR_W_BYTES);
      if (X3) {
        for (int kb = 0; kb < C2_KB; ++kb) {
          bulk_g2s(w_s + kb * 16384, t.w_hi + kb * 8192, 8192, wbar);
          bulk_g2s(w_s + kb * 16384 + 8192, t.w_lo + kb * 8192, 8192, wbar);
        }
      } else {
        bulk_g2s(w_s, t.w_hi, TR_W_BYTES, wbar);
      }
    }
  } else if (warp < 8) {
    // ============ builders: two threads per tile row (16 conv1 channels each) ============
    const int r = threadIdx.x & 127, half = threadIdx.x >> 7;
    const int bl = r / bp, p = r - bl * bp, x = p / rp, y = p - x * rp;
    const bool row_valid = bl < G && x < n && y < n;
    const int pc = x * n + y;  // bit of the cell in the packed position
    uint32_t tap_ok = 0;
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      const int xx = x + k / 3 - 1, yy = y + k % 3 - 1;
      if (row_valid && xx >= 0 && xx < n && yy >= 0 && yy < n) tap_ok |= 1u << k;
    }
    float bias16[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) bias16[j] = __ldg(t.b1 + half * 16 + j);
    const uint32_t cell = (uint32_t)(r + rp + 1);  // plane cell of this row's own position
    uint64_t nm = 0, nt = 0;
    auto fetch = [&](int64_t tile) {
      nm = nt = 0;
      const int64_t b = tile * G + bl;
      if (row_valid && tile < tiles && b < t.B) { nm = t.states[2 * b]; nt = t.states[2 * b + 1]; }
    };
    auto c1_operand = [&](int k, uint32_t it) {  // K1 encode + conv1 operand of the tile whose position is in (nm, nt)
      mbar_wait(&c1_free[k], ((it >> 1) & 1u) ^ 1u);
      uint8_t* sa = c1st + k * A_STAGE_BYTES;
      uint32_t pk[5];
#pragma unroll
      for (int q = 0; q < 9; ++q) {
        const int sh = (pc + (q / 3 - 1) * n + (q % 3 - 1)) & 63;
        const uint32_t ok = (tap_ok >> q) & 1u;
        const uint32_t m = (uint32_t)(nm >> sh) & ok, o = (uint32_t)(nt >> sh) & ok;
        const uint32_t v = (m ? 0x3F80u : 0u) | (o ? 0xBF80u : 0u);
        if (q & 1) pk[q >> 1] |= v << 16;
        else pk[q >> 1] = v;
      }
      const uint4 c_even = make_uint4(pk[0], pk[1], pk[2], pk[3]), c_odd = make_uint4(pk[4], 0, 0, 0);
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        const int c = half * 3 + j;
        *reinterpret_cast<uint4*>(sa + image_offset(r, c * 8)) = (c & 1) ? c_odd : c_even;
      }
      fence_async_smem();
      mbar_arrive(&c1_full[k]);
    };
    fetch(blockIdx.x);
    if ((int64_t)blockIdx.x < tiles) c1_operand(0, 0);
    fetch((int64_t)blockIdx.x + gridDim.x);
    uint32_t it = 0;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x, ++it) {
      const int k = (int)(it & 1u);
      const uint32_t ph = (it >> 1) & 1u;
      const bool has_next = tile + gridDim.x < tiles;
      if (has_next) {  // the next tile's conv1 operand depends on nothing the tensor core produces: build it first, so that
        c1_operand(k ^ 1, it + 1);  // conv1(it+1) is queued before conv2(it) and only the plane write-back below sits
        fetch(tile + 2 * (int64_t)gridDim.x);  // between a conv1 result and the conv2 MMAs that need it
      }
      mbar_wait(&c1_done[k], ph);
      tc_fence_after();
      uint32_t rr[16];
      tmem_ld16(tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + C1_COL + (uint32_t)(k * 32 + half * 16), rr);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(&c1_tfree[k]);
      mbar_wait(&pl_free[k], ph ^ 1u);  // the conv2 MMAs of tile it-2 have read this plane
      if (row_valid && tile * G + bl < t.B) {
        float v[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = fmaxf(__uint_as_float(rr[j]) + bias16[j], 0.0f);
        uint8_t* crow = planes + k * T2_PLANE_BYTES + cell * 128u;
        const uint32_t sw = cell & 7u;
#pragma unroll
        for (int c = 0; c < 2; ++c) {  // chunks 2 half + c (hi) and 4 + 2 half + c (lo) of the 128-byte cell
          uint32_t h[4], l[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) split_pair(v[c * 8 + 2 * e], v[c * 8 + 2 * e + 1], h[e], l[e]);
          const uint32_t q = (uint32_t)(half * 2 + c);
          *reinterpret_cast<uint4*>(crow + (((q ^ sw) & 7u) << 4)) = make_uint4(h[0], h[1], h[2], h[3]);
          if (X3) *reinterpret_cast<uint4*>(crow + ((((q + 4u) ^ sw) & 7u) << 4)) = make_uint4(l[0], l[1], l[2], l[3]);
        }
      }
      fence_async_smem();
      mbar_arrive(&pl_full[k]);
    }
  } else if (warp == 8) {
    // ======================= MMA issuer =======================
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc(BM, BN);
      constexpr uint32_t idesc_c1 = make_idesc(BM, 32);
      constexpr uint32_t idesc_cat = make_idesc(BM, 2 * BN);
      mbar_wait(wbar, 0);
      const uint32_t w_addr = smem_u32(w_s);
      const uint64_t b_c1 = make_smem_desc(smem_u32(w1img));
      auto conv1 = [&](int k, uint32_t it) {  // [A | A | A] x [w_hi | w_mid | w_lo]^T -> conv1 region k
        mbar_wait(&c1_full[k], (it >> 1) & 1u);
        mbar_wait(&c1_tfree[k], ((it >> 1) & 1u) ^ 1u);  // the builders have read the region's previous content
        tc_fence_after();
        const uint64_t a_c1 = make_smem_desc(smem_u32(c1st + k * A_STAGE_BYTES));
#pragma unroll
        for (int q = 0; q < 3; ++q) umma_bf16(tmem_base + C1_COL + (uint32_t)(k * 32), a_c1 + 2 * q, b_c1 + 2 * q, idesc_c1, q != 0);
        umma_commit(&c1_free[k]);
        umma_commit(&c1_done[k]);
      };
      if ((int64_t)blockIdx.x < tiles) conv1(0, 0);
      // descriptor increments of the nine taps in 16-byte units (the single issuing thread should spend its cycles on
      // tcgen05.mma, not on address arithmetic: everything but two additions per step is hoisted or a constant)
      uint32_t tap16[9];
#pragma unroll
      for (int q = 0; q < 9; ++q) tap16[q] = (uint32_t)((q / 3) * rp + (q % 3)) * 8u;
      const uint64_t b_base = make_smem_desc(w_addr);
      const uint64_t a_base[2] = {make_smem_desc(smem_u32(planes)), make_smem_desc(smem_u32(planes + T2_PLANE_BYTES))};
      uint32_t it = 0;
      for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x, ++it) {
        const int k = (int)(it & 1u);
        const uint32_t ph = (it >> 1) & 1u;
        if (tile + gridDim.x < tiles) conv1(k ^ 1, it + 1);  // before this tile's conv2: its write-back overlaps the 36 MMAs
        mbar_wait(&pl_full[k], ph);
        mbar_wait(&tempty[k], ph ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(k * ACC_COLS);
#pragma unroll
        for (int s = 0; s < 18; ++s) {
          // base-offset field of the shifted descriptor stays 0 (see the header comment)
          const uint64_t a_hi = a_base[k] + (uint64_t)(tap16[s >> 1] + (uint32_t)(s & 1) * 2u);
          const uint64_t b_w = b_base + (uint64_t)((s >> 2) * (X3 ? 2 : 1) * (64 * 128 / 16) + 2 * (s & 3));
          if (X3) {
            // Both correction products go to columns 64-127: the tensor core's fp32 accumulation truncates once per MMA
            // by up to an ulp OF THE ACCUMULATOR, so small terms added to the large hi x W_hi sum would double its
            // truncation bias (36 instead of 18 accumulations); among themselves they cost nothing measurable.
            umma_bf16(d_tmem, a_hi, b_w, idesc_cat, s != 0);     // hi x [W_hi ; W_lo]: columns 0-63 and 64-127
            umma_bf16(d_tmem + BN, a_hi + 4, b_w, idesc, 1);     // lo (64 bytes further in the cell) x W_hi: columns 64-127
          } else {
            umma_bf16(d_tmem, a_hi, b_w, idesc, s != 0);
          }
        }
        umma_commit(&pl_free[k]);
        umma_commit(&tfull[k]);
      }
    }
  } else if (warp >= 12) {
    // ======================= epilogue: two groups of four warps, alternate 16-column chunks =======================
    // A GEMM row is one (board, cell): its 64 channels are ONE 128-byte row of the feature image (tile = cell, row = board),
    // so the 32 rows of a warp go to 32 different image tiles.  Writing them straight from the accumulator registers costs
    // 32 partial cache lines per 16-byte store instruction (ncu: LSU wavefronts 41 % of the data pipe the tensor core
    // needs, r02_trunk2 capture); instead the converted rows are staged in shared memory (conflict-free XOR by the row)
    // and copied out with eight lanes per row: every store instruction writes four whole 128-byte lines.
    const int q = warp & 3, r = q * 32 + lane, grp = (warp - 12) >> 2, wl = warp - 12;
    uint8_t* stg = smem + S::STG_OFF;
    float4 bias4[2][4];  // conv2 bias of this group's two chunks
#pragma unroll
    for (int c = 0; c < 2; ++c)
#pragma unroll
      for (int j = 0; j < 4; ++j) bias4[c][j] = __ldg(reinterpret_cast<const float4*>(t.b2 + grp * 16 + c * 32) + j);
    // copy-out mapping: warp wl owns tile rows 16 wl .. 16 wl + 15; per pass i a lane moves chunk (lane & 7) of row
    // 16 wl + 4 i + (lane >> 3)
    int co_bl[4], co_pc[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int rr_ = 16 * wl + 4 * i + (lane >> 3);
      const int b_ = rr_ / bp, p_ = rr_ - b_ * bp, x_ = p_ / rp, y_ = p_ - x_ * rp;
      co_bl[i] = (b_ < G && x_ < n && y_ < n) ? b_ : -1;
      co_pc[i] = x_ * n + y_;
    }
    const bool f8 = X3 && t.out_f8;
    uint32_t it = 0;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x, ++it) {
      const int k = (int)(it & 1u);
      const int rb = (int)((tile * G + r / bp) & 127);  // image row (board & 127) of this thread's tile row
      mbar_wait(&tfull[k], (it >> 1) & 1u);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(k * ACC_COLS);
      named_bar(3, 256);  // the previous tile's copy-out has read the staging rows
      uint8_t* srow = stg + r * 256;
      const uint32_t sx = (uint32_t)((rb ^ r) & 7);  // image swizzle (board row) composed with the staging swizzle (tile row)
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        const int c0 = grp * 16 + c * 32;
        uint32_t rr[16], r2[16];
        tmem_ld16(taddr + (uint32_t)c0, rr);
        if (X3) tmem_ld16(taddr + (uint32_t)(BN + c0), r2);
        tmem_ld_wait();
        float x16[16];
        const float* bb = reinterpret_cast<const float*>(bias4[c]);
#pragma unroll
        for (int e = 0; e < 16; ++e) {
          float d = __uint_as_float(rr[e]);
          if (X3) d += __uint_as_float(r2[e]);
          x16[e] = fmaxf(d + bb[e], 0.0f);
        }
        const uint32_t kc = (uint32_t)(c0 >> 3);  // first of the two 16-byte chunks of these 16 channels in the hi row
        if (f8) {
          const float s_main = (float)(1 << F8_A_SCALE), s_lo = (float)(1 << (F8_A_SCALE + F8_LO_SHIFT));
          uint4 h0, h1;
          uint2 m0, m1, l0, l1;
          split8_f16f8(x16, s_main, s_lo, h0, m0, l0);
          split8_f16f8(x16 + 8, s_main, s_lo, h1, m1, l1);
          *reinterpret_cast<uint4*>(srow + (((kc) ^ sx) << 4)) = h0;
          *reinterpret_cast<uint4*>(srow + (((kc + 1) ^ sx) << 4)) = h1;
          const uint32_t qc = (uint32_t)(c0 >> 4);  // correction row: 16 e4m3 per chunk, main half then lo half
          *reinterpret_cast<uint4*>(srow + 128 + (((qc) ^ sx) << 4)) = make_uint4(m0.x, m0.y, m1.x, m1.y);
          *reinterpret_cast<uint4*>(srow + 128 + (((qc + 4) ^ sx) << 4)) = make_uint4(l0.x, l0.y, l1.x, l1.y);
        } else {
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            uint32_t hi[4], lo[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) split_pair(x16[h * 8 + 2 * e], x16[h * 8 + 2 * e + 1], hi[e], lo[e]);
            *reinterpret_cast<uint4*>(srow + (((kc + h) ^ sx) << 4)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            if (X3) *reinterpret_cast<uint4*>(srow + 128 + (((kc + h) ^ sx) << 4)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&tempty[k]);
      named_bar(4, 256);  // all rows of the tile are staged
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int64_t b = tile * G + co_bl[i];
        if (co_bl[i] >= 0 && b < t.B) {
          const int row = 16 * wl + 4 * i + (lane >> 3), j = lane & 7;
          const int rbi = (int)(b & 127);
          // staging chunk that holds final position j of the image row: final position = kc ^ (rbi & 7), staged at kc ^ ((rbi ^ row) & 7)
          const uint32_t sj = (uint32_t)(j ^ (row & 7));
          const size_t g0 = ((size_t)(b >> 7) * nn + co_pc[i]) * A_STAGE_BYTES + (size_t)(rbi >> 3) * 1024 + (size_t)(rbi & 7) * 128 + (size_t)j * 16;
          *reinterpret_cast<uint4*>(t.f_hi + g0) = *reinterpret_cast<const uint4*>(stg + row * 256 + (sj << 4));
          if (X3) *reinterpret_cast<uint4*>(t.f_lo + g0) = *reinterpret_cast<const uint4*>(stg + row * 256 + 128 + (sj << 4));
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 9) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

template <bool X3>
int launch_trunk2(const TrunkArgs& t, cudaStream_t st) {
  static bool configured = false;
  int dev = 0, sms = 0;
  AZG_CUDA_CHECK(cudaGetDevice(&dev));
  AZG_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  if (!configured) {
    AZG_CUDA_CHECK(cudaFuncSetAttribute(c4_trunk2_tc_kernel<X3>, cudaFuncAttributeMaxDynamicSharedMemorySize, Trunk2Smem<X3>::TOTAL));
    configured = true;
  }
  const int n = t.n, bp = (n + 1) * (n + 1);
  const int G = (127 - (n * n + n - 2)) / bp + 1;
  const int64_t tiles = (t.B + G - 1) / G;
  const int grid = (int)(tiles < sms ? tiles : sms);
  c4_trunk2_tc_kernel<X3><<<grid, T2_THREADS, Trunk2Smem<X3>::TOTAL, st>>>(t);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

int make_image(const float* src, int64_t rows, int64_t rows_padded, int K, int R, uint8_t* hi, uint8_t* lo, cudaStream_t st,
               int f8_mode = 0, const int32_t* f8_exp = nullptr) {
  return to_image(src, rows, rows_padded, K, R, hi, lo, st, f8_mode, f8_exp);
}

}  // namespace tc

// ---------------------------------------------------------------------------------------------
// Packed weight blob of the tensor-core Connect4 path (azg_c4_pack), sections 1024-B aligned:
//   W0 (output_transform.0, input order permuted to the feature image) hi [lo]
//   W2 (output_transform.2) hi [lo] | conv2 [64 x 320] hi [lo] | head weights (fp32, and as a weight image) | folded heads
namespace {
struct PackLayout {
  size_t w0_hi, w0_lo, w2_hi, w2_lo, c2_hi, c2_lo, heads_cat, hd_hi, hd_lo, bias32, fold_w, fold_b, scales, total;
  bool x3, gnn, f8;  // x3: hi + lo images (bf16x3 and the fp16+FP8 split); f8: the latter
};
// AZG_PREC_F16F8_KS runs on the operand images of AZG_PREC_F16F8 (same packed blob, same tile widths); it differs in how
// the F x F contractions are launched (KSPLIT launches over a quarter of K each, see GemmArgs::kb0)
constexpr int KSPLIT = 4;
inline bool ksplit_by_launches() {  // AZG_KSPLIT=launches: four launches per contraction instead of four work items per tile
  static int mode = -1;
  if (mode < 0) {
    const char* e = getenv("AZG_KSPLIT");
    mode = (e && strcmp(e, "launches") == 0) ? 1 : 0;
  }
  return mode == 1;
}
inline int prec_base(int prec) { return prec == AZG_PREC_F16F8_KS ? AZG_PREC_F16F8 : prec == AZG_PREC_BF16X3_KS ? AZG_PREC_BF16X3 : prec; }
inline bool prec_ksplit(int prec) { return prec == AZG_PREC_F16F8_KS || prec == AZG_PREC_BF16X3_KS; }
inline bool prec_is_tc(int prec) {
  prec = prec_base(prec);
  return prec == AZG_PREC_BF16X3 || prec == AZG_PREC_BF16 || prec == AZG_PREC_F16F8;
}
inline int prec_bn(int F, int prec) { return prec_base(prec) == AZG_PREC_F16F8 ? tc::pick_bn_f8(F) : tc::pick_bn(F); }

size_t up1k(size_t v) { return (v + 1023) / 1024 * 1024; }

PackLayout pack_layout(int n, int prec, bool gnn) {
  PackLayout L{};
  prec = prec_base(prec);
  const size_t F = 64 * (size_t)n * n, wimg = F * F * 2, cimg = 64 * (size_t)tc::C2_K * 2;
  L.x3 = prec == AZG_PREC_BF16X3 || prec == AZG_PREC_F16F8;
  L.f8 = prec == AZG_PREC_F16F8;
  L.gnn = gnn;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = up1k(off + bytes); return o; };
  if (gnn) {
    L.w0_hi = take(wimg);
    L.w0_lo = L.x3 ? take(wimg) : 0;
    L.w2_hi = take(wimg);
    L.w2_lo = L.x3 ? take(wimg) : 0;
  }
  L.c2_hi = take(cimg);
  L.c2_lo = L.x3 ? take(cimg) : 0;
  L.heads_cat = take((size_t)32 * F * 4);       // reference order, zero-padded to 32 rows (GEMM-2 epilogue)
  L.hd_hi = take((size_t)32 * F * 2);           // std heads as a [32 x F] weight image (feature-image order)
  L.hd_lo = L.x3 ? take((size_t)32 * F * 2) : 0;
  L.bias32 = take(32 * 4);
  L.fold_w = gnn ? take((size_t)tc::HEAD_ROWS * F * 4) : 0;  // [Wp; Wv] W2 (AZG_EVAL_FOLD)
  L.fold_b = gnn ? take(32 * 4) : 0;                         // [Wp; Wv] b2 + [bp; bv]
  L.scales = take(64);  // f8: int32 scale exponents of the W0, W2 and std-heads images [0..2], absmax scratch words [8..10]
  L.total = off;
  return L;
}

struct ScratchLayout {
  size_t f_hi, f_lo, h_hi, h_lo, part, lg32, acc, total;
};

ScratchLayout scratch_layout(int n, int64_t B, int prec, bool gnn) {
  ScratchLayout S{};
  const bool ksplit = prec_ksplit(prec);
  prec = prec_base(prec);
  const bool x3 = prec == AZG_PREC_BF16X3 || prec == AZG_PREC_F16F8;
  const size_t nn = (size_t)n * n, F = 64 * nn;
  const size_t Mp = (size_t)azg_ceil_div(B, 2 * tc::BM) * 2 * tc::BM;  // even number of m-tiles (CTA pairs)
  const size_t fimg = Mp * F * 2;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = up1k(off + bytes); return o; };
  S.f_hi = take(fimg);
  S.f_lo = x3 ? take(fimg) : 0;
  S.lg32 = take(Mp * 32 * sizeof(float));
  if (gnn) {
    S.h_hi = take(fimg);
    S.h_lo = x3 ? take(fimg) : 0;
    const int BNp = prec_bn((int)F, prec);
    S.part = take(Mp * (size_t)(BNp ? 2 * (F / BNp) : 32) * tc::HEAD_STRIDE * sizeof(float));  // two epilogue groups per n-tile
    // K-split partial sums: one [128 x 256] fp32 tile per CTA (in-kernel split), or the whole [Mp, F] matrix when the
    // split is made of launches (AZG_KSPLIT=launches, the bit-identical reference of the in-kernel form)
    if (ksplit) S.acc = take(ksplit_by_launches() ? Mp * F * sizeof(float) : (size_t)tc::KPART_MAX_CTAS * tc::BM * 256 * sizeof(float));
  }
  S.total = off + 1024;
  return S;
}
}  // namespace

size_t azg_tc_scratch_bytes(int n, int64_t B, int prec) { return scratch_layout(n, B, prec, true).total; }

// Whole Connect4 leaf evaluation on the tensor-core path: fused trunk (encode + conv1 + conv2) -> feature image ->
// [std heads] -> [output_transform GEMMs -> fused GNN heads].
int azg_tc_c4_forward(const void* packed, const azg_c4_params* p, int n, int prec, const uint64_t* states, int64_t B,
                      int eval_mask, float* pi_std, float* v_std, float* pi_gnn, float* v_gnn, void* scratch,
                      size_t scratch_bytes, const int32_t* dyn_rows, cudaStream_t st) {
  const int nn = n * n, F = 64 * nn, A = n + 1, BN = prec_bn(F, prec);
  AZG_REQUIRE(BN != 0, "tcgen05 path: unsupported board size %d", n);
  const int ks = prec_ksplit(prec) ? KSPLIT : 1;  // work items (or launches) per F x F contraction (K-split accumulation)
  const ScratchLayout S = scratch_layout(n, B, prec, true);
  prec = prec_base(prec);
  const bool f8 = prec == AZG_PREC_F16F8, x3 = prec == AZG_PREC_BF16X3 || f8, gnn = (eval_mask & AZG_EVAL_GNN) != 0;
  const PackLayout L = pack_layout(n, prec, true);
  AZG_REQUIRE(scratch && scratch_bytes >= S.total, "tcgen05 path: scratch %zu < %zu", scratch_bytes, S.total);
  uint8_t* sc = (uint8_t*)(((uintptr_t)scratch + 1023) & ~(uintptr_t)1023);
  const uint8_t* w = (const uint8_t*)packed;
  uint8_t *f_hi = sc + S.f_hi, *f_lo = x3 ? sc + S.f_lo : nullptr;
  uint8_t *h_hi = sc + S.h_hi, *h_lo = x3 ? sc + S.h_lo : nullptr;
  int rc;
  // One contraction = one launch, or (AZG_PREC_F16F8_KS) `ks` launches over consecutive quarters of K: all but the last
  // leave raw fp32 partial sums in S.acc (no bias, no ReLU), the last adds them to its accumulator and runs the normal
  // fused epilogue; the side tile (standard heads) accumulates in its own [M, 32] output.
  auto run_contraction = [&](const tc::GemmArgs& full) -> int {
    if (ks <= 1) return tc::run_gemm(BN, full, st);
    AZG_REQUIRE(full.KB >= ks && x3, "tcgen05 path: K-split needs one of the split precisions and KB >= %d", ks);
    float* acc = (float*)(sc + S.acc);
    if (!ksplit_by_launches()) {  // default: the split happens inside the kernel, partial sums stay in L2
      tc::GemmArgs q = full;
      q.ksplit = ks;
      q.kpart = acc;
      return tc::run_gemm(BN, q, st);
    }
    // (Tried: the FP8 correction product in a launch of its own over the whole K, so that the main accumulators see half as
    // many truncating accumulations -- the GEMM's distance from its exact emulation fell from 3.2e-6 to 1.7e-6, pi / v on a
    // trained checkpoint did not move (what is left there is the 16-17 bit operand representation of the trunk and the
    // splits), and the step grew from 7.0 to 8.8 ms: not kept.)
    for (int c = 0; c < ks; ++c) {
      tc::GemmArgs q = full;
      q.kb0 = tc::ksplit_begin(full.KB, c, ks);
      q.kbn = tc::ksplit_begin(full.KB, c + 1, ks) - q.kb0;
      q.side_acc = c > 0;
      q.acc_in = (c > 0 && full.n_tiles > 0) ? acc : nullptr;
      if (c + 1 < ks) {
        q.out_mode = tc::OUT_F32; q.out_f32 = acc; q.out_hi = q.out_lo = nullptr; q.no_bias = 1; q.relu = 0;
      }
      const int r = tc::run_gemm(BN, q, st);
      if (r) return r;
    }
    return AZG_OK;
  };
  azg_phase_begin(AZG_PHASE_TRUNK, st);
  tc::TrunkArgs t{};
  t.states = states; t.w1 = p->conv1_w; t.b1 = p->conv1_b; t.b2 = p->conv2_b;
  t.w_hi = w + L.c2_hi; t.w_lo = x3 ? w + L.c2_lo : nullptr; t.f_hi = f_hi; t.f_lo = f_lo; t.B = B; t.n = n;
  t.dyn_rows = dyn_rows;
  t.out_f8 = f8 ? 1 : 0;
  rc = x3 ? tc::launch_trunk2<true>(t, st) : tc::launch_trunk2<false>(t, st);
  if (rc) return rc;
  azg_phase_end(AZG_PHASE_TRUNK, st);
  // predict's heads ride on GEMM-1 as a side tile
  const int32_t* scales = (const int32_t*)(w + L.scales);
  const bool std_side = (eval_mask & AZG_EVAL_STD) != 0;
  if (std_side && !gnn) {  // std only: the same side-tile code with no main n-tiles (bit-identical to the combined call)
    AZG_REQUIRE(pi_std && v_std && A <= 9, "tcgen05 path: bad std outputs");
    azg_phase_begin(AZG_PHASE_HEADS, st);
    tc::GemmArgs h{};
    h.M = B; h.m_tiles = (int)azg_ceil_div(B, tc::BM); h.n_tiles = 0; h.KB = F / tc::BK; h.x3 = x3;
    h.a_hi = f_hi; h.a_lo = f_lo; h.dyn_rows = dyn_rows;
    h.side_hi = w + L.hd_hi; h.side_lo = x3 ? w + L.hd_lo : nullptr;
    h.side_bias = (const float*)(w + L.bias32); h.side_out = (float*)(sc + S.lg32);
    h.f8 = f8 ? tc::f8_terms() : 0; h.side_exp = scales + 2;
    if ((rc = run_contraction(h))) return rc;
    tc::heads32_finalize_kernel<<<(unsigned)((B + 127) / 128), 128, 0, st>>>((const float*)(sc + S.lg32), A, B, dyn_rows, pi_std, v_std);
    AZG_LAUNCH_CHECK();
    azg_phase_end(AZG_PHASE_HEADS, st);
    return AZG_OK;
  }
  if (!gnn) return AZG_OK;
  azg_phase_begin(AZG_PHASE_GEMM, st);
  tc::GemmArgs g{};
  g.M = B;
  g.m_tiles = (int)azg_ceil_div(B, tc::BM);
  g.n_tiles = F / BN;
  g.KB = F / tc::BK;
  g.x3 = x3;
  g.dyn_rows = dyn_rows;
  g.a_hi = f_hi; g.a_lo = f_lo; g.w_hi = w + L.w0_hi; g.w_lo = x3 ? w + L.w0_lo : nullptr; g.bias = p->ot0_b; g.relu = 1;
  g.f8 = f8 ? tc::f8_terms() : 0; g.w_exp = scales + 0; g.side_exp = scales + 2;
  AZG_REQUIRE(g.n_tiles <= 32 && A + 1 <= tc::HEAD_ROWS, "tcgen05 path: head fusion limits exceeded");
  if (std_side) {
    AZG_REQUIRE(pi_std && v_std && A <= 9, "tcgen05 path: bad std outputs");
    g.side_hi = w + L.hd_hi; g.side_lo = x3 ? w + L.hd_lo : nullptr;
    g.side_bias = (const float*)(w + L.bias32); g.side_out = (float*)(sc + S.lg32);
  }
  auto finish_std = [&]() -> int {  // log_softmax / tanh of the side tile's logits (inside the HEADS phase)
    if (!std_side) return AZG_OK;
    tc::heads32_finalize_kernel<<<(unsigned)((B + 127) / 128), 128, 0, st>>>((const float*)(sc + S.lg32), A, B, dyn_rows, pi_std, v_std);
    AZG_LAUNCH_CHECK();
    return AZG_OK;
  };
  if (eval_mask & AZG_EVAL_FOLD) {
    // output_transform.2 and the heads folded into one [A+1, F] matrix (see fold_heads_kernel): GEMM-1's epilogue
    // applies it to relu(H) tile by tile; H and E never exist in HBM and the second F x F contraction is gone
    g.out_mode = tc::OUT_HEADS; g.out_hi = g.out_lo = nullptr; g.out_f32 = nullptr;
    g.head_w = (const float*)(w + L.fold_w); g.head_rows = A + 1; g.head_part = (float*)(sc + S.part);
    if ((rc = run_contraction(g))) return rc;
    azg_phase_end(AZG_PHASE_GEMM, st);
    azg_phase_begin(AZG_PHASE_HEADS, st);
    const float* fb = (const float*)(w + L.fold_b);
    tc::heads_finalize_kernel<<<(unsigned)((B + 127) / 128), 128, 0, st>>>(g.head_part, g.n_tiles * tc::head_slots_per_tile(g), A, fb, fb + A, B, dyn_rows,
                                                                          pi_gnn, v_gnn);
    AZG_LAUNCH_CHECK();
    if ((rc = finish_std())) return rc;
    azg_phase_end(AZG_PHASE_HEADS, st);
    return AZG_OK;
  }
  g.out_mode = x3 ? tc::OUT_IMG_HILO : tc::OUT_IMG; g.out_hi = h_hi; g.out_lo = h_lo;
  if ((rc = run_contraction(g))) return rc;
  g.side_hi = g.side_lo = nullptr;  // GEMM-2 has no side tile
  g.a_hi = h_hi; g.a_lo = h_lo; g.w_hi = w + L.w2_hi; g.w_lo = x3 ? w + L.w2_lo : nullptr; g.bias = p->ot2_b; g.relu = 0;
  g.w_exp = scales + 1;
  g.out_mode = tc::OUT_HEADS; g.out_hi = g.out_lo = nullptr; g.out_f32 = nullptr;
  g.head_w = (const float*)(w + L.heads_cat); g.head_rows = A + 1; g.head_part = (float*)(sc + S.part);
  if ((rc = run_contraction(g))) return rc;
  azg_phase_end(AZG_PHASE_GEMM, st);
  azg_phase_begin(AZG_PHASE_HEADS, st);
  tc::heads_finalize_kernel<<<(unsigned)((B + 127) / 128), 128, 0, st>>>(g.head_part, g.n_tiles * tc::head_slots_per_tile(g), A, p->fc_policy_b,
                                                                        p->fc_value_b, B, dyn_rows, pi_gnn, v_gnn);
  AZG_LAUNCH_CHECK();
  if ((rc = finish_std())) return rc;
  azg_phase_end(AZG_PHASE_HEADS, st);
  return AZG_OK;
}

extern "C" {

size_t azg_c4_packed_bytes(int n, int prec) {
  const int F = 64 * n * n;
  if (n < 4 || n > 8 || !prec_is_tc(prec) || prec_bn(F, prec) == 0) return 0;
  return pack_layout(n, prec, true).total + 1024;
}

int azg_c4_pack(const azg_c4_params* p, int n, int prec, void* packed, size_t packed_bytes, azg_stream stream) {
  const int nn = n * n, F = 64 * nn, A = n + 1, BN = prec_is_tc(prec) ? prec_bn(F, prec) : 0;
  AZG_REQUIRE(p && packed && p->conv2_w && p->fc_policy_w && p->fc_value_w, "azg_c4_pack: null pointer");
  AZG_REQUIRE(n >= 4 && n <= 8 && BN != 0, "azg_c4_pack: unsupported n=%d prec=%d", n, prec);
  AZG_REQUIRE(packed_bytes >= azg_c4_packed_bytes(n, prec), "azg_c4_pack: buffer too small");
  AZG_REQUIRE(((uintptr_t)packed & 15) == 0, "azg_c4_pack: buffer must be 16-byte aligned (bulk-copy source)");
  const PackLayout L = pack_layout(n, prec, true);
  const bool x3 = L.x3, f8 = L.f8;
  uint8_t* w = (uint8_t*)packed;
  cudaStream_t st = (cudaStream_t)stream;
  int32_t* scales = (int32_t*)(w + L.scales);
  uint32_t* bits = (uint32_t*)(w + L.scales) + 8;
  int rc;
  if (p->ot0_w && p->ot2_w) {
    if (f8) {  // per-tensor power-of-two scales of the FP8 correction rows
      if ((rc = tc::weight_scale_exp(p->ot0_w, (int64_t)F * F, bits + 0, scales + 0, st))) return rc;
      if ((rc = tc::weight_scale_exp(p->ot2_w, (int64_t)F * F, bits + 1, scales + 1, st))) return rc;
    }
    const int64_t cnt = (int64_t)F * (F / 8);
    tc::permuted_weight_image_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, st>>>(p->ot0_w, F, F, nn, BN, w + L.w0_hi,
                                                                                   x3 ? w + L.w0_lo : nullptr, f8 ? scales + 0 : nullptr);
    AZG_LAUNCH_CHECK();
    rc = tc::make_image(p->ot2_w, F, F, F, BN, w + L.w2_hi, x3 ? w + L.w2_lo : nullptr, st, f8 ? 2 : 0, scales + 1);
    if (rc) return rc;
  }
  tc::conv2_weight_image_kernel<<<(64 * (tc::C2_K / 8) + 127) / 128, 128, 0, st>>>(p->conv2_w, w + L.c2_hi, x3 ? w + L.c2_lo : nullptr);
  AZG_LAUNCH_CHECK();
  tc::concat_heads_kernel<<<(unsigned)(((int64_t)32 * F + 255) / 256), 256, 0, st>>>(
      p->fc_policy_w, p->fc_value_w, p->fc_policy_b, p->fc_value_b, A, F, (float*)(w + L.heads_cat), (float*)(w + L.bias32));
  AZG_LAUNCH_CHECK();
  if (p->ot2_w && p->ot2_b) {
    double* part = nullptr;
    AZG_CUDA_CHECK(cudaMallocAsync((void**)&part, sizeof(double) * tc::FOLD_SPLITS * tc::HEAD_ROWS * (size_t)F, st));
    const int per = (F + tc::FOLD_SPLITS - 1) / tc::FOLD_SPLITS;
    tc::fold_heads_partial_kernel<<<dim3((F + 127) / 128, tc::FOLD_SPLITS), 128, 0, st>>>((const float*)(w + L.heads_cat), p->ot2_w,
                                                                                         A + 1, F, per, part);
    AZG_LAUNCH_CHECK();
    tc::fold_heads_finish_kernel<<<(F + 32 + 127) / 128, 128, 0, st>>>(part, (const float*)(w + L.heads_cat), p->ot2_b,
                                                                       (const float*)(w + L.bias32), A + 1, F,
                                                                       (float*)(w + L.fold_w), (float*)(w + L.fold_b));
    AZG_LAUNCH_CHECK();
    AZG_CUDA_CHECK(cudaFreeAsync(part, st));
  }
  {
    const int64_t cnt = (int64_t)32 * (F / 8);
    if (f8 && (rc = tc::weight_scale_exp((const float*)(w + L.heads_cat), (int64_t)32 * F, bits + 2, scales + 2, st))) return rc;
    tc::permuted_weight_image_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, st>>>((const float*)(w + L.heads_cat), 32, F, nn, 32,
                                                                                   w + L.hd_hi, x3 ? w + L.hd_lo : nullptr,
                                                                                   f8 ? scales + 2 : nullptr);
    AZG_LAUNCH_CHECK();
  }
  return AZG_OK;
}

}  // extern "C" (reopened below)

// ---- TicTacToe on the tensor cores (tictactoe/TicTacToeNet.py:28-48, TicTacToeGNN.py:25-87) ------------------------
// conv2 / conv3 as im2col GEMMs whose A operand is written straight as tile images (the fp32 patch matrix never
// exists), fc1 / fc2 / output_transform as GEMMs over image copies of their fp32 inputs; conv1 and the two small
// heads stay on the fp32 kernels.  Weight images: one blob per precision, rebuilt after weight updates.
namespace {

// patches of boards [b0, b0+nb) -> A operand images, rows (board, cell), K = (ci, kx, ky) zero-padded to Kp
__global__ void im2col3x3_image_kernel(const float* __restrict__ in, int in_nhwc, int64_t b0, int64_t nb, int Cin, int H, int W,
                                       int pad, int Kp, int64_t rows_padded, uint8_t* __restrict__ hi, uint8_t* __restrict__ lo) {
  const int Ho = H + 2 * pad - 2, Wo = W + 2 * pad - 2, P = Ho * Wo, K = Cin * 9, chunks = Kp / 8;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows_padded * chunks) return;
  const int64_t row = idx / chunks;
  const int c = (int)(idx % chunks);
  float x8[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) x8[e] = 0.0f;
  if (row < nb * P) {
    const int64_t b = b0 + row / P;
    const int p = (int)(row % P), ox = p / Wo, oy = p % Wo;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int k = c * 8 + e;
      if (k < K) {
        const int ci = k / 9, kx = (k % 9) / 3, ky = k % 3, x = ox + kx - pad, y = oy + ky - pad;
        if (x >= 0 && x < H && y >= 0 && y < W)
          x8[e] = in_nhwc ? in[((b * H + x) * W + y) * Cin + ci] : in[((b * Cin + ci) * H + x) * W + y];
      }
    }
  }
  const int KB = Kp / tc::BK;
  const size_t off = ((size_t)(row / 128) * KB + (c * 8) / tc::BK) * ((size_t)128 * 128) + tc::image_offset((int)(row % 128), (c * 8) % tc::BK);
  tc::split_store(x8, hi, lo, off);
}

// W [N, K] fp32 -> [N x Kp] weight images with BN-row tiles (columns K..Kp-1 zero)
__global__ void weight_image_padded_kernel(const float* __restrict__ w, int N, int K, int Kp, int BN, uint8_t* __restrict__ hi,
                                           uint8_t* __restrict__ lo) {
  const int chunks = Kp / 8;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= N * chunks) return;
  const int n = idx / chunks, c = idx % chunks;
  float x8[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) x8[e] = (c * 8 + e < K) ? w[(size_t)n * K + c * 8 + e] : 0.0f;
  const int KB = Kp / tc::BK;
  const size_t off = ((size_t)(n / BN) * KB + (c * 8) / tc::BK) * ((size_t)BN * 128) + tc::image_offset(n % BN, (c * 8) % tc::BK);
  tc::split_store(x8, hi, lo, off);
}

struct TttLayer {
  int N, K, Kp, BN;
  size_t hi, lo;
};
struct TttPack {
  TttLayer conv2, conv3, fc1, fc2, ot0, ot2;
  size_t total;
};

int ttt_bn(int N) { return N % 256 == 0 ? 256 : 64; }

TttPack ttt_pack_layout(int n, bool x3) {
  const int F = 128 * (n - 2) * (n - 2);
  TttPack L{};
  size_t off = 0;
  auto lay = [&](int N, int K) {
    TttLayer l{N, K, (K + 63) / 64 * 64, ttt_bn(N), 0, 0};
    const size_t img = (size_t)N * l.Kp * 2;
    l.hi = off; off = up1k(off + img);
    if (x3) { l.lo = off; off = up1k(off + img); }
    return l;
  };
  L.conv2 = lay(64, 288); L.conv3 = lay(128, 576); L.fc1 = lay(512, F); L.fc2 = lay(512, F); L.ot0 = lay(F, F); L.ot2 = lay(F, F);
  L.total = off;
  return L;
}

constexpr size_t TTT_IMG_BYTES = (size_t)128 << 20;  // per image (hi or lo) of an im2col chunk

struct TttScratch {
  size_t planes, c1, c2, f_nhwc, feat, hid, enh, h1, h2, a_hi, a_lo, total;
};
TttScratch ttt_scratch_layout(int n, int64_t B, bool gnn) {
  const size_t nn = (size_t)n * n, P = (size_t)(n - 2) * (n - 2), F = 128 * P;
  TttScratch S{};
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = up1k(off + bytes); return o; };
  S.planes = take(B * nn * 4); S.c1 = take(B * 32 * nn * 4); S.c2 = take(B * 64 * nn * 4); S.f_nhwc = take(B * F * 4);
  S.feat = take(B * F * 4); S.h1 = take(B * 512 * 4); S.h2 = take(B * 512 * 4);
  if (gnn) { S.hid = take(B * F * 4); S.enh = take(B * F * 4); }
  const size_t Mp = (size_t)azg_ceil_div(B, 256) * 256;
  const size_t fc_img = Mp * (F > 512 ? F : 512) * 2;
  const size_t img = fc_img > TTT_IMG_BYTES ? fc_img : TTT_IMG_BYTES;
  S.a_hi = take(img + 65536); S.a_lo = take(img + 65536);
  S.total = off;
  return S;
}

// C[M, N] = act(image(A) W^T + b): the A images are already in a_hi / a_lo
int ttt_gemm(const uint8_t* a_hi, const uint8_t* a_lo, int64_t M, const TttLayer& l, const uint8_t* w, const float* bias, int relu,
             bool x3, float* C, cudaStream_t st) {
  tc::GemmArgs g{};
  g.M = M; g.m_tiles = (int)azg_ceil_div(M, tc::BM); g.n_tiles = l.N / l.BN; g.KB = l.Kp / tc::BK; g.x3 = x3;
  g.a_hi = a_hi; g.a_lo = x3 ? a_lo : nullptr; g.w_hi = w + l.hi; g.w_lo = x3 ? w + l.lo : nullptr; g.bias = bias; g.relu = relu;
  g.out_mode = tc::OUT_F32; g.out_f32 = C;
  return tc::run_gemm(l.BN, g, st);
}

// relu(conv3x3) over all boards in chunks: im2col images -> GEMM -> (board, cell, channel) rows
int ttt_conv_tc(const float* in, int in_nhwc, const TttLayer& l, const uint8_t* w, const float* bias, float* out_nhwc, int64_t B,
                int Cin, int H, int W, int pad, bool x3, uint8_t* a_hi, uint8_t* a_lo, cudaStream_t st) {
  const int Ho = H + 2 * pad - 2, Wo = W + 2 * pad - 2, P = Ho * Wo;
  int64_t chunk = (int64_t)(TTT_IMG_BYTES / ((size_t)P * l.Kp * 2)) / 256 * 256;
  if (chunk < 256) chunk = 256;
  for (int64_t b0 = 0; b0 < B; b0 += chunk) {
    const int64_t nb = B - b0 < chunk ? B - b0 : chunk;
    const int64_t rows = nb * P, rows_p = azg_ceil_div(rows, 256) * 256;
    AZG_REQUIRE((size_t)rows_p * l.Kp * 2 <= TTT_IMG_BYTES + 65536, "ttt_conv_tc: image chunk overflow");
    const int64_t n = rows_p * (l.Kp / 8);
    im2col3x3_image_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(in, in_nhwc, b0, nb, Cin, H, W, pad, l.Kp, rows_p, a_hi,
                                                                       x3 ? a_lo : nullptr);
    AZG_LAUNCH_CHECK();
    int rc = ttt_gemm(a_hi, a_lo, rows, l, w, bias, 1, x3, out_nhwc + (size_t)b0 * P * l.N, st);
    if (rc) return rc;
  }
  return AZG_OK;
}

int ttt_linear_tc(const float* A, int64_t M, const TttLayer& l, const uint8_t* w, const float* bias, int relu, bool x3, float* C,
                  uint8_t* a_hi, uint8_t* a_lo, bool reuse_image, cudaStream_t st) {
  int rc;
  if (!reuse_image && (rc = tc::to_image(A, M, azg_ceil_div(M, 256) * 256, l.Kp, tc::BM, a_hi, x3 ? a_lo : nullptr, st))) return rc;
  return ttt_gemm(a_hi, a_lo, M, l, w, bias, relu, x3, C, st);
}

}  // namespace

// fp32 pieces of azg_nets.cu
int azg_ttt_fp32_front(const float* conv1_w, const float* conv1_b, int n, const uint64_t* states, int64_t B, float* planes, float* c1,
                       cudaStream_t st);
int azg_ttt_fp32_heads(const float* h1, const float* pw, const float* pb, int A, const float* h2, const float* vw, const float* vb,
                       int64_t B, float* pi, float* v, cudaStream_t st);
int azg_nhwc_to_nchw(const float* src, int64_t B, int P, int C, float* dst, cudaStream_t st);

extern "C" {

size_t azg_ttt_packed_bytes(int n, int prec) {
  if (n < 3 || n > 8 || prec == AZG_PREC_FP32) return 0;
  return ttt_pack_layout(n, prec == AZG_PREC_BF16X3).total + 1024;
}

int azg_ttt_pack(const azg_ttt_params* p, int n, int prec, void* packed, size_t packed_bytes, azg_stream stream) {
  AZG_REQUIRE(p && packed && n >= 3 && n <= 8 && (prec == AZG_PREC_BF16X3 || prec == AZG_PREC_BF16), "azg_ttt_pack: bad argument");
  AZG_REQUIRE(packed_bytes >= azg_ttt_packed_bytes(n, prec) && ((uintptr_t)packed & 1023) == 0, "azg_ttt_pack: buffer too small or not 1 KB aligned");
  const bool x3 = prec == AZG_PREC_BF16X3;
  const TttPack L = ttt_pack_layout(n, x3);
  uint8_t* w = (uint8_t*)packed;
  cudaStream_t st = (cudaStream_t)stream;
  struct { const TttLayer* l; const float* src; } items[] = {{&L.conv2, p->conv2_w}, {&L.conv3, p->conv3_w}, {&L.fc1, p->fc1_w},
                                                            {&L.fc2, p->fc2_w}, {&L.ot0, p->ot0_w}, {&L.ot2, p->ot2_w}};
  for (auto& it : items) {
    if (!it.src) continue;  // output_transform is absent without the GNN
    const int n_thr = it.l->N * (it.l->Kp / 8);
    weight_image_padded_kernel<<<(n_thr + 255) / 256, 256, 0, st>>>(it.src, it.l->N, it.l->K, it.l->Kp, it.l->BN, w + it.l->hi,
                                                                    x3 ? w + it.l->lo : nullptr);
    AZG_LAUNCH_CHECK();
  }
  return AZG_OK;
}

size_t azg_ttt_tc_workspace_bytes(int n, int64_t B, int eval_mask) {
  return ttt_scratch_layout(n, B, (eval_mask & AZG_EVAL_GNN) != 0).total + 1024;
}

int azg_ttt_forward_tc(const azg_ttt_params* p, const void* packed, int n, int prec, const uint64_t* states, int64_t B, int eval_mask,
                       float* pi_std, float* v_std, float* pi_gnn, float* v_gnn, void* workspace, size_t workspace_bytes,
                       azg_stream stream) {
  AZG_REQUIRE(p && packed && states && workspace, "azg_ttt_forward_tc: null pointer");
  AZG_REQUIRE(n >= 3 && n <= 8 && (eval_mask & ~3) == 0 && eval_mask != 0, "azg_ttt_forward_tc: bad n=%d or eval_mask=%d", n, eval_mask);
  AZG_REQUIRE(prec == AZG_PREC_BF16X3 || prec == AZG_PREC_BF16, "azg_ttt_forward_tc: precision must be bf16x3 or bf16");
  if (B <= 0) return AZG_OK;
  const bool x3 = prec == AZG_PREC_BF16X3, gnn = (eval_mask & AZG_EVAL_GNN) != 0;
  const TttPack L = ttt_pack_layout(n, x3);
  const TttScratch S = ttt_scratch_layout(n, B, gnn);
  AZG_REQUIRE(workspace_bytes >= S.total + 1024, "azg_ttt_forward_tc: workspace %zu < %zu", workspace_bytes, S.total + 1024);
  uint8_t* sc = (uint8_t*)(((uintptr_t)workspace + 1023) & ~(uintptr_t)1023);
  const uint8_t* w = (const uint8_t*)packed;
  cudaStream_t st = (cudaStream_t)stream;
  float *planes = (float*)(sc + S.planes), *c1 = (float*)(sc + S.c1), *c2 = (float*)(sc + S.c2), *f_nhwc = (float*)(sc + S.f_nhwc);
  float *feat = (float*)(sc + S.feat), *h1 = (float*)(sc + S.h1), *h2 = (float*)(sc + S.h2);
  float *hid = gnn ? (float*)(sc + S.hid) : nullptr, *enh = gnn ? (float*)(sc + S.enh) : nullptr;
  uint8_t *a_hi = sc + S.a_hi, *a_lo = sc + S.a_lo;
  const int P = (n - 2) * (n - 2), A = n * n + 1;
  int rc;
  if ((rc = azg_ttt_fp32_front(p->conv1_w, p->conv1_b, n, states, B, planes, c1, st))) return rc;
  if ((rc = ttt_conv_tc(c1, 0, L.conv2, w, p->conv2_b, c2, B, 32, n, n, 1, x3, a_hi, a_lo, st))) return rc;
  if ((rc = ttt_conv_tc(c2, 1, L.conv3, w, p->conv3_b, f_nhwc, B, 64, n, n, 0, x3, a_hi, a_lo, st))) return rc;
  if ((rc = azg_nhwc_to_nchw(f_nhwc, B, P, 128, feat, st))) return rc;
  for (int pass = 0; pass < 2; ++pass) {
    const int bit = pass == 0 ? AZG_EVAL_STD : AZG_EVAL_GNN;
    if (!(eval_mask & bit)) continue;
    const float* f = feat;
    float *pi = pi_std, *v = v_std;
    if (pass == 1) {
      AZG_REQUIRE(p->ot0_w && p->ot2_w, "azg_ttt_forward_tc: null output_transform weights");
      if ((rc = ttt_linear_tc(feat, B, L.ot0, w, p->ot0_b, 1, x3, hid, a_hi, a_lo, false, st))) return rc;
      if ((rc = ttt_linear_tc(hid, B, L.ot2, w, p->ot2_b, 0, x3, enh, a_hi, a_lo, false, st))) return rc;
      f = enh; pi = pi_gnn; v = v_gnn;
    }
    AZG_REQUIRE(pi && v, "azg_ttt_forward_tc: null outputs");
    if ((rc = ttt_linear_tc(f, B, L.fc1, w, p->fc1_b, 1, x3, h1, a_hi, a_lo, false, st))) return rc;
    if ((rc = ttt_linear_tc(f, B, L.fc2, w, p->fc2_b, 1, x3, h2, a_hi, a_lo, true, st))) return rc;  // same A image
    if ((rc = azg_ttt_fp32_heads(h1, p->fc_policy_w, p->fc_policy_b, A, h2, p->fc_value_w, p->fc_value_b, B, pi, v, st))) return rc;
  }
  return AZG_OK;
}

}  // extern "C"

extern "C" {

// Stand-alone dense layer on the tensor-core path, for parity tests of the GEMM itself:
// C[M,F] = act(A[M,F] . W[F,F]^T + bias), fp32 in/out, operands converted on the fly.
int azg_tc_linear(const float* A, const float* W, const float* bias, float* C, int64_t M, int F, int prec, int relu,
                  void* scratch, size_t scratch_bytes, azg_stream stream) {
  const int BN = prec_is_tc(prec) ? prec_bn(F, prec) : 0;
  AZG_REQUIRE(A && W && bias && C && scratch, "azg_tc_linear: null pointer");
  AZG_REQUIRE(BN != 0 && F % 64 == 0, "azg_tc_linear: unsupported F=%d prec=%d", F, prec);
  const int ks = prec_ksplit(prec) ? KSPLIT : 1;  // C doubles as the partial-sum buffer of the K-split launches
  prec = prec_base(prec);
  const bool f8 = prec == AZG_PREC_F16F8, x3 = prec == AZG_PREC_BF16X3 || f8;
  const int64_t m_tiles = azg_ceil_div(M, tc::BM), Mp = azg_ceil_div(M, 2 * tc::BM) * 2 * tc::BM;
  const size_t a_img = (size_t)Mp * F * 2, w_img = (size_t)F * F * 2;
  const size_t need = (x3 ? 2 : 1) * (a_img + w_img) + 2048;
  AZG_REQUIRE(scratch_bytes >= need, "azg_tc_linear: scratch %zu < %zu", scratch_bytes, need);
  uint8_t* base = (uint8_t*)(((uintptr_t)scratch + 1023) & ~(uintptr_t)1023);
  uint8_t *a_hi = base, *a_lo = x3 ? base + a_img : nullptr;
  uint8_t* wbase = base + (x3 ? 2 : 1) * a_img;
  uint8_t *w_hi = wbase, *w_lo = x3 ? wbase + w_img : nullptr;
  cudaStream_t st = (cudaStream_t)stream;
  int rc;
  int32_t* scales = (int32_t*)(wbase + (x3 ? 2 : 1) * w_img);  // [0] weight scale exponent, [1] absmax scratch
  if (f8 && (rc = tc::weight_scale_exp(W, (int64_t)F * F, (uint32_t*)scales + 1, scales, st))) return rc;
  if ((rc = tc::to_image(A, M, Mp, F, tc::BM, a_hi, a_lo, st, f8 ? 1 : 0, nullptr))) return rc;
  if ((rc = tc::to_image(W, F, F, F, BN, w_hi, w_lo, st, f8 ? 2 : 0, scales))) return rc;
  tc::GemmArgs g{};
  g.f8 = f8 ? tc::f8_terms() : 0; g.w_exp = scales;
  g.M = M; g.m_tiles = (int)m_tiles; g.n_tiles = F / BN; g.KB = F / tc::BK; g.x3 = x3;
  g.a_hi = a_hi; g.a_lo = a_lo; g.w_hi = w_hi; g.w_lo = w_lo; g.bias = bias; g.relu = relu;
  g.out_mode = tc::OUT_F32; g.out_f32 = C;
  if (ks > 1 && !ksplit_by_launches()) {
    AZG_REQUIRE(g.KB >= ks, "azg_tc_linear: K-split needs K >= %d", ks * tc::BK);
    float* part = nullptr;
    AZG_CUDA_CHECK(cudaMallocAsync((void**)&part, (size_t)tc::KPART_MAX_CTAS * tc::BM * 256 * sizeof(float), st));
    g.ksplit = ks;
    g.kpart = part;
    rc = tc::run_gemm(BN, g, st);
    AZG_CUDA_CHECK(cudaFreeAsync(part, st));
    return rc;
  }
  for (int c = 0; c < ks; ++c) {
    tc::GemmArgs q = g;
    if (ks > 1) {
      AZG_REQUIRE(g.KB >= ks, "azg_tc_linear: K-split needs K >= %d", ks * tc::BK);
      q.kb0 = tc::ksplit_begin(g.KB, c, ks);
      q.kbn = tc::ksplit_begin(g.KB, c + 1, ks) - q.kb0;
      q.acc_in = c > 0 ? C : nullptr;
      if (c + 1 < ks) { q.no_bias = 1; q.relu = 0; }
    }
    if ((rc = tc::run_gemm(BN, q, st))) return rc;
  }
  return AZG_OK;
}

}  // extern "C"
