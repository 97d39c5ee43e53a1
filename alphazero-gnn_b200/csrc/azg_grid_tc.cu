// azg_grid_tc.cu -- one fused kernel per grid-graph GNN layer on the 5th-gen tensor cores
// (BASELINE configs[4]; operator = FrozenLakeNet.GNNLayer, frozenlake/FrozenLakeNet.py:8-33, on gh x gw
// 4-neighbour grids normalised as create_adjacency, :68-72):
//
//     forward    out = relu( A^ (X W^T + b) )                    X, out: [B*n, H] fp32 row-major
//     backward   dX  = A^ ( (dOut * [out > 0]) W )               (A^ is symmetric, so A^ (G W) = (A^ G) W)
//
// Each CTA owns tiles of WHOLE graphs (G = 128 / n graphs = G*n <= 128 GEMM rows), one persistent CTA per SM:
//   warps 0-7    producers: 128-bit loads of the tile's fp32 rows (one k-block = 64 channels at a time, issued one
//                item ahead), split into bf16 hi/lo, stored as the SWIZZLE_128B operand image of the stage;
//                the weight images are resident in shared memory (one bulk copy per CTA) except for H = 256 in
//                bf16x3 (256 KB), where thread 0 streams the k-block's weight images into the stage from L2
//   warp 8       MMA issuer (one thread): M=128 x N=H x K=16 tcgen05.mma, 3 products per k-block in bf16x3
//   warp 9       TMEM allocation (2 accumulators of H fp32 columns), barrier init
//   warps 10-17  epilogue, two groups of four warps alternating 32-column chunks: TMEM -> registers -> fp32 staging
//                tile in shared memory (pre-scaled by d_row) -> every row sums its <= 5 neighbours -> * d_row
//                + rowsum*bias, ReLU -> whole 128-byte row segments to HBM
// so the support matrix X W^T never exists in HBM: algorithmic bytes per layer = 4H read + 4H written per node.
//
// MT = 2 (graphs of 129..256 nodes): a tile is 256 rows = two 128-row halves, each with its own TMEM accumulator; the
// pipeline items run (tile, half, k-block), so producers and MMA issuer only see "one more 128-row operand".  The
// staging tiles have 256 rows, so a node's neighbours are found across the half boundary: an epilogue thread stages
// tile rows r and 128 + r (same TMEM lane, the two accumulators) of its group's chunk.  Where only one staging tile
// fits (H = 256 in bf16x3) the eight warps form ONE group, thread = one of the 256 rows.
//
// PAIR (H = 256 in bf16x3, whose 256 KB of weight images do not fit one SM): a cluster of two CTAs, each with its own
// tiles, producers, accumulators and epilogue, shares ONE weight operand -- every tcgen05.mma is issued by the leader
// for both (cta_group::2, M = 256: 128 rows per CTA) and reads weight rows 0-127 from the leader's and 128-255 from
// the peer's shared memory, where they stay resident (128 KB each) instead of being re-streamed from L2 per tile.
#include "azg_tc.cuh"

namespace gridtc {
using namespace tc;

constexpr int GT_THREADS = 576;    // 8 producer warps, MMA, TMEM/barrier setup, 2 x 4 epilogue warps

template <int H, bool X3, int MT, bool PAIR>
struct GridSmem {
  static constexpr int ROWS = 128 * MT;                      // tile rows
  static constexpr int MISC_BYTES = MT == 1 ? 5120 : 8192;   // barriers (256 B), neighbour table [ROWS][5], row sums, d
  static constexpr int KB = H / BK;
  static constexpr int A_BYTES = (X3 ? 2 : 1) * A_STAGE_BYTES;
  static constexpr int W_HALF = H * 128;  // one k-block of one weight image
  static constexpr int W_BYTES = (X3 ? 2 : 1) * W_HALF;
  static constexpr int W_ROWS = PAIR ? H / 2 : H;  // weight rows (output features) this CTA holds
  static constexpr int W_HALF_RES = W_ROWS * 128;  // one k-block of one resident weight image
  static constexpr int W_TOTAL = KB * W_BYTES / (PAIR ? 2 : 1);  // the resident weight operand (hi and lo images)
  static constexpr int AVAIL = 232448 - 1024 - MISC_BYTES;
  static constexpr int ST32 = 2 * 128 * 36 * 4;  // two staging tiles of 32-column chunks
  static constexpr int ST_MIN = MT == 1 ? 2 * 128 * 16 * 4 : ROWS * 16 * 4;  // smallest staging: 16-column tiles (MT = 2: one tile)
  // WRES: the weight images stay resident in shared memory for the life of the CTA (one bulk copy at start) and a
  // pipeline stage holds only the A operand; otherwise (H = 256 in bf16x3: 256 KB of weights) every stage also
  // carries its k-block of the weights, re-streamed from L2 per tile.
  static constexpr bool WRES = (AVAIL - ST_MIN - W_TOTAL) / A_BYTES >= 2;
  static constexpr int STAGE_BYTES = A_BYTES + (WRES ? 0 : W_BYTES);
  static constexpr int W_RES_BYTES = WRES ? W_TOTAL : 0;
  // epilogue chunk = columns per tcgen05.ld; two staging tiles (one per epilogue group) of 128 rows.  32 columns (row
  // stride 144 B: a quarter-warp stores 8 rows x 16 B / gathers one row's 128 B without bank conflicts) unless that leaves
  // fewer than two stages; else 16 columns, rows of 64 B with the 16-byte unit XOR-swizzled by (row >> 1) & 3 (stg_unit):
  // a quarter-warp stores 8 rows -> 8 distinct units, gathers 2 rows (always of different parity) x 4 units -> 8 distinct.
  // MT = 2: two tiles of 32 columns, else two of 16, else (H = 256 in bf16x3) one of 16
  static constexpr int EC = (AVAIL - W_RES_BYTES - 2 * ROWS * 36 * 4) / STAGE_BYTES >= 2 ? 32 : 16;
  static constexpr int ST_LD = EC == 32 ? 36 : 16;
  static constexpr int ST_BYTES = ROWS * ST_LD * 4;
  static constexpr int NTILE = (AVAIL - W_RES_BYTES - 2 * ST_BYTES) / STAGE_BYTES >= 2 ? 2 : 1;
  static_assert(MT == 2 || NTILE == 2, "one staging tile per epilogue group");
  static constexpr int BUDGET = AVAIL - W_RES_BYTES - NTILE * ST_BYTES;
  static constexpr int NST = BUDGET / STAGE_BYTES < 6 ? BUDGET / STAGE_BYTES : 6;
  static constexpr int STAGE_OFF = W_RES_BYTES;
  static constexpr int ST_OFF = STAGE_OFF + NST * STAGE_BYTES;
  static constexpr int MISC_OFF = ST_OFF + NTILE * ST_BYTES;
  static constexpr int NACC = MT == 1 ? 2 : (4 * H <= 512 ? 4 : 2);  // TMEM accumulators of H columns (MT = 2: one per half)
  static constexpr int TOTAL = MISC_OFF + MISC_BYTES + 1024;
  static_assert(NST >= 2, "at least two pipeline stages");
  static_assert(!PAIR || WRES, "CTA pairs exist to keep the weights resident");
};

__device__ __forceinline__ void mbar_expect_tx_only(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}

// 4 fp32 -> 8 bytes of the hi (and lo) operand image
__device__ __forceinline__ void split_store4(float4 x, uint8_t* hi, uint8_t* lo, uint32_t off) {
  uint32_t h0, h1, l0, l1;
  split_pair(x.x, x.y, h0, l0);
  split_pair(x.z, x.w, h1, l1);
  *reinterpret_cast<uint2*>(hi + off) = make_uint2(h0, h1);
  if (lo) *reinterpret_cast<uint2*>(lo + off) = make_uint2(l0, l1);
}

// float4 index of 16-byte unit `c` of staging row `row`.  32-column chunks: rows of 144 B.  16-column chunks: rows of 64 B
// placed at slot = row with bits 0 and 2 exchanged, unit XOR-swizzled by (slot >> 1) & 3 -- a quarter-warp that stores 8
// consecutive rows (one unit each) or gathers rows x and x + 4 (four units each) touches 8 distinct 16-byte bank groups.
template <int EC, int ST_LD>
__device__ __forceinline__ int stg_unit(int row, int c) {
  if (EC == 32) return row * (ST_LD / 4) + c;
  const int slot = (row & ~5) | ((row & 1) << 2) | ((row >> 2) & 1);
  return slot * 4 + (c ^ ((slot >> 1) & 3));
}

__device__ __forceinline__ void add4(float4& s, const float4& t) {
  s.x += t.x; s.y += t.y; s.z += t.z; s.w += t.w;
}

// One thread's share of the neighbour gather: RUN = EC / 4 consecutive tile rows (run0 ...) x one 16-byte unit c4, i.e. a
// quarter-warp (EC = 32) covers whole 128-byte row segments in shared memory and in HBM.  Left / self / right neighbours
// are consecutive staged rows, so the run is walked with a three-row window: (RUN + 2) + 2 RUN shared loads per RUN
// outputs instead of 5 RUN (the gather's loads are what fills the shared-memory pipe: profiles/r02_grid_sweep.txt).
// out = d_row * (self + up + down + left + right, in this order) + rowsum * bias; masks = 5 valid bits per row of the run.
template <int EC, int ST_LD>
__device__ __forceinline__ void gather_run(const float4* src, int run0, uint64_t masks, int c4, int gw, const float* row_d,
                                           const float* row_sum, float4 b4, int relu, float* out_unit, int64_t row_base,
                                           int64_t total_rows, int H) {
  constexpr int RUN = EC / 4;
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  float4 prev = zero, cur = src[stg_unit<EC, ST_LD>(run0, c4)], next;
  if (masks & 8u) prev = src[stg_unit<EC, ST_LD>(run0 - 1, c4)];
#pragma unroll
  for (int k = 0; k < RUN; ++k) {
    const int row = run0 + k;
    const uint32_t m = (uint32_t)(masks >> (5 * k)) & 31u;
    next = zero;
    if (k + 1 < RUN || (m & 16u)) next = src[stg_unit<EC, ST_LD>(row + 1, c4)];
    float4 s = (m & 1u) ? cur : zero;
    if (m & 2u) add4(s, src[stg_unit<EC, ST_LD>(row - gw, c4)]);
    if (m & 4u) add4(s, src[stg_unit<EC, ST_LD>(row + gw, c4)]);
    if (m & 8u) add4(s, prev);
    if (m & 16u) add4(s, next);
    const float d = row_d[row], rs = row_sum[row];
    float4 v = make_float4(fmaf(d, s.x, rs * b4.x), fmaf(d, s.y, rs * b4.y), fmaf(d, s.z, rs * b4.z), fmaf(d, s.w, rs * b4.w));
    if (relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
    const int64_t grow = row_base + row;
    if (m != 0u && grow < total_rows) __stcs(reinterpret_cast<float4*>(out_unit + grow * H), v);
    prev = cur;
    cur = next;
  }
}

struct GridArgs {
  const float* x;      // FWD: layer input; BWD: upstream gradient dOut
  const float* act;    // BWD: the layer's output (ReLU gate), else null
  const uint8_t* w_hi; // weight image, k-block major: [KB][H rows x 64] (BWD: of W^T)
  const uint8_t* w_lo;
  const float* bias;   // FWD: [H]; BWD: null (no bias term)
  float* out;
  int64_t B;           // graphs
  int gh, gw;
  int relu;
};

template <int H, bool X3, bool BWD, int MT, bool PAIR>
__global__ void __launch_bounds__(GT_THREADS, 1) grid_layer_tc_kernel(GridArgs g) {  // 18 warps: 96 registers per thread
  using S = GridSmem<H, X3, MT, PAIR>;
  constexpr int KB = S::KB, NST = S::NST, EC = S::EC, ST_LD = S::ST_LD, ROWS = S::ROWS, NACC = S::NACC;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  float* staging = (float*)(smem + S::ST_OFF);
  uint64_t* full = (uint64_t*)(smem + S::MISC_OFF);
  uint64_t* empty = full + NST;
  uint64_t* tfull = empty + NST;
  uint64_t* tempty = tfull + NACC;
  uint64_t* wbar = tempty + NACC;
  uint64_t* peer_full = wbar + 1;             // PAIR, leader: the peer CTA's full[] and tempty[] events
  uint64_t* peer_tempty = peer_full + NST;
  uint32_t* tmem_slot = (uint32_t*)(peer_tempty + NACC);
  static_assert((2 * NST + 3 * NACC + 1) * 8 + 4 <= 256, "barrier block");
  float* nb_coef = (float*)(smem + S::MISC_OFF + 256);  // [ROWS][5]
  float* row_sum = nb_coef + ROWS * 5;                  // [ROWS]
  float* row_d = row_sum + ROWS;                        // [ROWS] deg^-1/2 (0 for unused tile rows)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n = g.gh * g.gw;
  const int G = ROWS / n;         // graphs per tile
  const int R = G * n;            // valid tile rows
  const int64_t tiles = (g.B + G - 1) / G;
  const int64_t total_rows = g.B * n;
  constexpr uint32_t TMEM_COLS = NACC * H < 32 ? 32 : NACC * H;
  // tiles of this CTA: j-th tile = tile_of(j).  A pair walks consecutive tiles (2 u + rank); at the tail the peer's tile
  // may not exist -- it then runs an all-zero tile through the same pipeline (no loads, no stores).
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;
  const int64_t unit = PAIR ? (int64_t)(blockIdx.x >> 1) : (int64_t)blockIdx.x;
  const int64_t n_units = PAIR ? (int64_t)(gridDim.x >> 1) : (int64_t)gridDim.x;
  const int64_t tile_units = PAIR ? (tiles + 1) / 2 : tiles;
  const int64_t my_tiles = (tile_units - unit + n_units - 1) / n_units;
  auto tile_of = [&](int64_t j) { const int64_t u = unit + j * n_units; return PAIR ? 2 * u + (int64_t)rank : u; };

  // neighbour table of a tile row: (tile row of the neighbour, d_i * d_j); identical for every tile
  for (int i = threadIdx.x; i < ROWS * 5; i += blockDim.x) {
    const int r = i / 5, k = i % 5;
    float coef = 0.0f;
    if (r < R) {
      const int slot = r / n, node = r - slot * n, x = node / g.gw, y = node - x * g.gw;
      const int dx = (k == 1) ? -1 : (k == 2) ? 1 : 0, dy = (k == 3) ? -1 : (k == 4) ? 1 : 0;
      const int nx = x + dx, ny = y + dy;
      if (nx >= 0 && nx < g.gh && ny >= 0 && ny < g.gw) {
        const int di = 1 + (x > 0) + (x < g.gh - 1) + (y > 0) + (y < g.gw - 1);
        const int dj = 1 + (nx > 0) + (nx < g.gh - 1) + (ny > 0) + (ny < g.gw - 1);
        coef = (1.0f / sqrtf((float)di)) * (1.0f / sqrtf((float)dj));
      }
    }
    nb_coef[i] = coef;
  }
  if (warp == 9 && lane == 0) {
    for (int s = 0; s < NST; ++s) {
      mbar_init(&full[s], 256);
      mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < NACC; ++a) {
      mbar_init(&tfull[a], 1);
      mbar_init(&tempty[a], S::NTILE == 2 ? 256 : 128);  // both epilogue groups drain an accumulator / one group: four warps
    }
    mbar_init(wbar, 1);
    for (int s = 0; s < NST; ++s) mbar_init(&peer_full[s], 1);
    for (int a = 0; a < NACC; ++a) mbar_init(&peer_tempty[a], 1);
    fence_barrier_init();
  }
  if (warp == 9) {
    if (PAIR) tmem_alloc2(tmem_slot, TMEM_COLS);
    else tmem_alloc(tmem_slot, TMEM_COLS);
  }
  __syncthreads();
  if (threadIdx.x < ROWS) {  // rowsum in the same order as the gather below
    float s = 0.0f;
#pragma unroll
    for (int k = 0; k < 5; ++k) s += nb_coef[threadIdx.x * 5 + k];
    row_sum[threadIdx.x] = s;
    row_d[threadIdx.x] = sqrtf(nb_coef[threadIdx.x * 5]);  // coefficient 0 of a row is d_r * d_r
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();  // both CTAs' barriers exist before any remote arrive / multicast commit
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (S::WRES && warp == 9 && lane == 0) {  // weight images -> shared memory, once per CTA (PAIR: this CTA's half of the rows)
    mbar_expect_tx(wbar, S::W_TOTAL);
    for (int kb = 0; kb < KB; ++kb) {
      const size_t src = (size_t)kb * S::W_HALF + (size_t)rank * S::W_HALF_RES;  // rows rank * W_ROWS ..: whole 8-row swizzle atoms
      bulk_g2s(smem + kb * S::W_HALF_RES, g.w_hi + src, S::W_HALF_RES, wbar);
      if (X3) bulk_g2s(smem + (KB + kb) * S::W_HALF_RES, g.w_lo + src, S::W_HALF_RES, wbar);
    }
  }
  if (warp < 8) {
    // =========================== producers ===========================
    // An item = one (tile, k-block): 128 rows x 64 channels = 8 row groups of 16 rows; a half-warp reads one row's
    // 256 B in one fully coalesced request.  Each thread keeps PF items (8 x PF float4) of loads in flight in a
    // register ring with static indices: a slot is refilled with the same row group of item + PF right after it has
    // been converted, so the global loads never wait for the pipeline.
    constexpr int PF = 1;  // 8 float4 (x2 in BWD) per thread = 32 KB (64 KB) of loads in flight per SM
    const int j4 = threadIdx.x & 15, r0 = threadIdx.x >> 4;  // rows r0 + 16 i, float4 j4 (4 channels) of the k-block
    constexpr int IPT = MT * KB;  // items per tile, ordered (half, k-block)
    const int64_t items = my_tiles * IPT;
    float4 v[PF][8];
    float4 a[PF][BWD ? 8 : 1];
    auto load = [&](int64_t it, int i, float4& vv, float4& aa) {
      const int64_t tile = tile_of(it / IPT);
      const int kb = (int)(it % KB);
      const int r = (int)((it % IPT) / KB) * 128 + r0 + 16 * i;  // tile row
      const int64_t row = tile * R + r;
      if (r < R && row < total_rows) {
        vv = __ldcs(reinterpret_cast<const float4*>(g.x + row * H + kb * BK) + j4);
        if (BWD) aa = __ldcs(reinterpret_cast<const float4*>(g.act + row * H + kb * BK) + j4);
      } else {
        vv = make_float4(0.f, 0.f, 0.f, 0.f);
        if (BWD) aa = make_float4(1.f, 1.f, 1.f, 1.f);
      }
    };
#pragma unroll
    for (int p = 0; p < PF; ++p)
      if (p < items) {
#pragma unroll
        for (int i = 0; i < 8; ++i) load(p, i, v[p][i], a[p][BWD ? i : 0]);
      }
    int stage = 0;
    uint32_t phase = 0;
    for (int64_t it0 = 0; it0 < items; it0 += PF) {
#pragma unroll
      for (int p = 0; p < PF; ++p) {
        const int64_t it = it0 + p;
        if (it >= items) break;
        const int kb = (int)(it % KB);
        const bool more = it + PF < items;
        uint8_t* sa = smem + S::STAGE_OFF + stage * S::STAGE_BYTES;
        mbar_wait(&empty[stage], phase ^ 1);
        if (!S::WRES && threadIdx.x == 0) {  // this k-block of the weight image(s): contiguous in HBM/L2, one bulk copy each
          mbar_expect_tx_only(&full[stage], S::W_BYTES);
          bulk_g2s(sa + S::A_BYTES, g.w_hi + (size_t)kb * S::W_HALF, S::W_HALF, &full[stage]);
          if (X3) bulk_g2s(sa + S::A_BYTES + S::W_HALF, g.w_lo + (size_t)kb * S::W_HALF, S::W_HALF, &full[stage]);
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          float4 x = v[p][i];
          if (BWD) {
            const float4 m = a[p][BWD ? i : 0];
            x.x = m.x > 0.0f ? x.x : 0.0f; x.y = m.y > 0.0f ? x.y : 0.0f; x.z = m.z > 0.0f ? x.z : 0.0f; x.w = m.w > 0.0f ? x.w : 0.0f;
          }
          split_store4(x, sa, X3 ? sa + A_STAGE_BYTES : nullptr, image_offset(r0 + 16 * i, j4 * 4));
          if (more) load(it + PF, i, v[p][i], a[p][BWD ? i : 0]);
        }
        fence_async_smem();
        mbar_arrive(&full[stage]);
        if (++stage == NST) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 8) {
    // =========================== MMA issuer ===========================
    if (lane == 0 && rank != 0) {
      // peer CTA of a pair: forward "accumulator drained" and "stage filled" to the leader, in the leader's wait order
      mbar_wait(wbar, 0);  // this CTA's weight rows are in place before the leader may issue anything
      const uint32_t l_full = map_to_cta(peer_full, 0), l_tempty = map_to_cta(peer_tempty, 0);
      int stage = 0, acc = 0;
      uint32_t phase = 0, acc_phase = 0;
      for (int64_t item = 0, n_items = my_tiles * MT; item < n_items; ++item) {
        mbar_wait(&tempty[acc], acc_phase ^ 1);
        mbar_arrive_cluster(l_tempty + (uint32_t)acc * 8u);
        for (int kb = 0; kb < KB; ++kb) {
          mbar_wait(&full[stage], phase);
          mbar_arrive_cluster(l_full + (uint32_t)stage * 8u);
          if (++stage == NST) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (++acc == NACC) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    } else if (lane == 0) {
      constexpr uint32_t idesc = make_idesc(PAIR ? 2 * BM : BM, H);
      auto mma = [&](uint32_t d, uint64_t a, uint64_t b, uint32_t acc_flag) {
        if (PAIR) umma2_bf16(d, a, b, idesc, acc_flag);
        else umma_bf16(d, a, b, idesc, acc_flag);
      };
      int stage = 0, acc = 0;
      uint32_t phase = 0, acc_phase = 0;
      if (S::WRES) mbar_wait(wbar, 0);
      const uint32_t w_res = smem_u32(smem);
      for (int64_t item = 0, n_items = my_tiles * MT; item < n_items; ++item) {  // (tile, half)
        mbar_wait(&tempty[acc], acc_phase ^ 1);
        if (PAIR) mbar_wait_cluster(&peer_tempty[acc], (uint32_t)((item / NACC) & 1));
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * H);
        for (int kb = 0; kb < KB; ++kb) {
          mbar_wait(&full[stage], phase);
          if (PAIR) mbar_wait_cluster(&peer_full[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + S::STAGE_OFF + stage * S::STAGE_BYTES);
          const uint64_t a_hi = make_smem_desc(sa), a_lo = make_smem_desc(sa + A_STAGE_BYTES);
          const uint64_t b_hi = make_smem_desc(S::WRES ? w_res + kb * S::W_HALF_RES : sa + S::A_BYTES);
          const uint64_t b_lo = make_smem_desc(S::WRES ? w_res + (KB + kb) * S::W_HALF_RES : sa + S::A_BYTES + S::W_HALF);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) mma(d_tmem, a_hi + 2 * k, b_hi + 2 * k, (kb | k) != 0);
          if (X3) {
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) mma(d_tmem, a_hi + 2 * k, b_lo + 2 * k, 1);
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) mma(d_tmem, a_lo + 2 * k, b_hi + 2 * k, 1);
          }
          if (PAIR) umma2_commit(&empty[stage]);
          else umma_commit(&empty[stage]);
          if (++stage == NST) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (PAIR) umma2_commit(&tfull[acc]);
        else umma_commit(&tfull[acc]);
        if (++acc == NACC) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
  } else if (warp >= 10 && S::NTILE == 1) {
    // =========================== epilogue, 256-row tiles, one staging tile: one group of eight warps ===========================
    // warps 10-13 drain the accumulator of rows 0-127, warps 14-17 the one of rows 128-255 (a warp reads the TMEM lane
    // quarter warp % 4); staging row = tile row, so the gather below crosses the half boundary like any other row.
    constexpr int LPR = EC / 4, RUN = EC / 4;  // lanes per row = rows per thread
    const int half = (warp - 10) >> 2;
    const int q = warp & 3, r = half * 128 + q * 32 + lane;
    const int c4 = lane % LPR, run0 = (r / LPR) * RUN;
    const float my_d = row_d[r];
    uint64_t run_mask = 0;  // 5 neighbour-valid bits per row of this thread's gather run
#pragma unroll
    for (int i = 0; i < RUN; ++i) {
#pragma unroll
      for (int k = 0; k < 5; ++k) run_mask |= (uint64_t)(nb_coef[(run0 + i) * 5 + k] != 0.0f ? 1u : 0u) << (5 * i + k);
    }
    const int gw = g.gw;
    int acc = half;
    uint32_t acc_phase = 0;
    for (int64_t j = 0; j < my_tiles; ++j) {
      const int64_t row_base = tile_of(j) * R;
      mbar_wait(&tfull[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * H);
#pragma unroll 1
      for (int c0 = 0; c0 < H; c0 += EC) {
        float* stg = staging;
        uint32_t rr[EC];
        if (EC == 32) tmem_ld32(taddr + (uint32_t)c0, rr);
        else tmem_ld16(taddr + (uint32_t)c0, rr);
        tmem_ld_wait();
        float4* dst = reinterpret_cast<float4*>(stg);
#pragma unroll
        for (int e = 0; e < EC / 4; ++e)
          dst[stg_unit<EC, ST_LD>(r, e)] = make_float4(my_d * __uint_as_float(rr[4 * e]), my_d * __uint_as_float(rr[4 * e + 1]),
                                                       my_d * __uint_as_float(rr[4 * e + 2]), my_d * __uint_as_float(rr[4 * e + 3]));
        float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (g.bias) b4 = __ldg(reinterpret_cast<const float4*>(g.bias + c0) + c4);
        named_bar(3, 256);  // the chunk of every tile row is staged
        gather_run<EC, ST_LD>(reinterpret_cast<const float4*>(stg), run0, run_mask, c4, gw, row_d, row_sum, b4, g.relu,
                              g.out + c0 + 4 * c4, row_base, total_rows, H);
        named_bar(4, 256);  // every row has gathered: the staging tile may be overwritten
      }
      tc_fence_before();
      mbar_arrive(&tempty[acc]);
      acc += 2;
      if (acc >= NACC) {
        acc = half;
        acc_phase ^= 1;
      }
    }
  } else if (warp >= 10) {
    // =========================== epilogue: two groups of four warps, alternating column chunks ===========================
    // Staging: thread = TMEM lane = tile row (MT = 2: rows r and 128 + r, one per accumulator) writes d_row * D[row, EC
    // columns] (d = deg^-1/2).  Gather: gather_run -- EC/4 lanes cover a row's chunk (contiguous in shared memory and in
    // HBM: whole lines), each walking EC/4 consecutive rows; out = d_row * (sum over {self, valid neighbours} of the staged
    // rows) + rowsum * bias.  Neighbours of row r: r -/+ gw (x -/+ 1), r -/+ 1 (y -/+ 1).
    constexpr int LPR = EC / 4, RUN = EC / 4;  // lanes per row = rows per thread in the gather
    const int grp = (warp - 10) >> 2;
    const int q = warp & 3, r = q * 32 + lane;
    const int c4 = lane % LPR, run0 = (r / LPR) * RUN;
    float* stg = staging + grp * (S::ST_BYTES / 4);
    float my_d[MT];
    uint64_t run_mask[MT];  // 5 neighbour-valid bits per row of this thread's gather run
#pragma unroll
    for (int h = 0; h < MT; ++h) {
      my_d[h] = row_d[h * 128 + r];
      run_mask[h] = 0;
#pragma unroll
      for (int i = 0; i < RUN; ++i) {
#pragma unroll
        for (int k = 0; k < 5; ++k) run_mask[h] |= (uint64_t)(nb_coef[(h * 128 + run0 + i) * 5 + k] != 0.0f ? 1u : 0u) << (5 * i + k);
      }
    }
    const int gw = g.gw;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int64_t j = 0; j < my_tiles; ++j) {
      const int64_t row_base = tile_of(j) * R;
#pragma unroll
      for (int h = 0; h < MT; ++h) mbar_wait(&tfull[acc + h], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * H);
#pragma unroll 1
      for (int c0 = grp * EC; c0 < H; c0 += 2 * EC) {
#pragma unroll
        for (int h = 0; h < MT; ++h) {
          uint32_t rr[EC];
          if (EC == 32) tmem_ld32(taddr + (uint32_t)(h * H + c0), rr);
          else tmem_ld16(taddr + (uint32_t)(h * H + c0), rr);
          tmem_ld_wait();
          float4* dst = reinterpret_cast<float4*>(stg);
#pragma unroll
          for (int e = 0; e < EC / 4; ++e)
            dst[stg_unit<EC, ST_LD>(h * 128 + r, e)] =
                make_float4(my_d[h] * __uint_as_float(rr[4 * e]), my_d[h] * __uint_as_float(rr[4 * e + 1]),
                            my_d[h] * __uint_as_float(rr[4 * e + 2]), my_d[h] * __uint_as_float(rr[4 * e + 3]));
        }
        float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (g.bias) b4 = __ldg(reinterpret_cast<const float4*>(g.bias + c0) + c4);
        named_bar(3 + 2 * grp, 128);  // the chunk of every row is staged
#pragma unroll
        for (int h = 0; h < MT; ++h)
          gather_run<EC, ST_LD>(reinterpret_cast<const float4*>(stg), h * 128 + run0, run_mask[h], c4, gw, row_d, row_sum, b4, g.relu,
                                g.out + c0 + 4 * c4, row_base, total_rows, H);
        named_bar(4 + 2 * grp, 128);  // every row has gathered: the staging tile may be overwritten
      }
      tc_fence_before();
#pragma unroll
      for (int h = 0; h < MT; ++h) mbar_arrive(&tempty[acc + h]);
      acc += MT;
      if (acc == NACC) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();  // the leader's MMAs read the peer's shared memory: leave together
  if (warp == 9) {
    tc_fence_after();
    if (PAIR) tmem_dealloc2(tmem_base, TMEM_COLS);
    else tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// W [H, H] fp32 row-major (nn.Linear weight: [out, in]) -> B-operand images, k-block major.
//   transpose = 0: B[nrow = out][k = in] = W[out][in]       (forward,  X W^T)
//   transpose = 1: B[nrow = in][k = out] = W[out][in]       (backward, G W)
__global__ void grid_weight_image_kernel(const float* __restrict__ w, int H, int transpose, uint8_t* __restrict__ hi,
                                         uint8_t* __restrict__ lo) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;  // one thread per (nrow, 8-wide k chunk)
  const int chunks = H / 8;
  if (idx >= H * chunks) return;
  const int nrow = idx / chunks, k0 = (idx % chunks) * 8;
  float x8[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) x8[e] = transpose ? w[(size_t)(k0 + e) * H + nrow] : w[(size_t)nrow * H + k0 + e];
  const size_t off = (size_t)(k0 / BK) * ((size_t)H * 128) + image_offset(nrow, k0 % BK);
  split_store(x8, hi, lo, off);
}

template <int H, bool X3, bool BWD, int MT, bool PAIR>
int launch(const GridArgs& g, cudaStream_t st) {
  static bool configured = false;
  using S = GridSmem<H, X3, MT, PAIR>;
  int dev = 0, sms = 0;
  AZG_CUDA_CHECK(cudaGetDevice(&dev));
  AZG_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  if (!configured) {
    AZG_CUDA_CHECK(cudaFuncSetAttribute(grid_layer_tc_kernel<H, X3, BWD, MT, PAIR>, cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL));
    configured = true;
  }
  const int G = S::ROWS / (g.gh * g.gw);
  const int64_t tiles = (g.B + G - 1) / G;
  const int64_t units = PAIR ? (tiles + 1) / 2 : tiles, max_units = PAIR ? sms / 2 : sms;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)((units < max_units ? units : max_units) * (PAIR ? 2 : 1)));
  cfg.blockDim = dim3(GT_THREADS);
  cfg.dynamicSmemBytes = S::TOTAL;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = PAIR ? 2 : 1;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  AZG_CUDA_CHECK(cudaLaunchKernelEx(&cfg, grid_layer_tc_kernel<H, X3, BWD, MT, PAIR>, g));
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

// ---- weight / bias gradient of the layer on the tensor cores ---------------------------------------------------
//   dW[o, i] = sum_r S[r, o] X[r, i],   db[o] = sum_r S[r, o]      S = A^ (dOut * [out > 0]),  r over all B*n rows
// The contraction index is the ROW of two row-major fp32 matrices, i.e. both operands are MN-major for the tensor
// core: a k-block of KR rows is stored as H/64 blocks of [KR k-rows x 64 elements] (128-byte rows, 8-row swizzle
// atoms) -- the same byte pattern the K-major images use, read through descriptors with the MN-major bits set
// (a_major = b_major = 1; LBO = block stride, SBO = 1024).  Split-K over persistent CTAs: each CTA accumulates its
// k-blocks in TMEM (M = 128 output features per accumulator, two accumulators for H = 256) and writes one partial
// [H, H]; a fixed-order reduction adds the partials (deterministic).
template <int H, bool X3>
struct DwSmem {
  static constexpr int KR = H == 256 ? 32 : 64;           // rows per k-block (16 float4 of loads in flight per thread)
  static constexpr int BLK = KR * 128;                    // one [KR x 64] block
  static constexpr int OPER = (H / 64) * BLK;             // one operand image (hi or lo)
  static constexpr int STAGE_BYTES = 2 * (X3 ? 2 : 1) * OPER;  // S and X
  static constexpr int NST = 3;
  static constexpr int ZERO_OFF = NST * STAGE_BYTES;      // H = 64: an all-zero block stands in for output features 64..127
  static constexpr int MISC_OFF = ZERO_OFF + (H < 128 ? BLK : 0);
  static constexpr int TOTAL = MISC_OFF + 4096 + 1024;
};

__device__ __forceinline__ uint64_t make_smem_desc_mn(uint32_t saddr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)(lbo_bytes >> 4) << 16;  // stride between 64-element blocks along M/N
  d |= (uint64_t)(1024 >> 4) << 32;       // stride between 8-row groups along K
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;                 // SWIZZLE_128B
  return d;
}

struct DwArgs {
  const float* s;   // [rows, H]
  const float* x;   // [rows, H]
  float* part_w;    // [grid, H, H]
  float* part_b;    // [grid, H]
  int64_t rows;
};

template <int H, bool X3>
__global__ void __launch_bounds__(512, 1) grid_dw_tc_kernel(DwArgs g) {
  using S = DwSmem<H, X3>;
  constexpr int KR = S::KR, NST = S::NST, MH = H < 128 ? 1 : H / 128;  // accumulators of 128 output features
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* full = (uint64_t*)(smem + S::MISC_OFF);
  uint64_t* empty = full + NST;
  uint64_t* tfull = empty + NST;
  uint32_t* tmem_slot = (uint32_t*)(tfull + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t kblocks = (g.rows + KR - 1) / KR;
  const int64_t items = kblocks > blockIdx.x ? (kblocks - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  constexpr uint32_t TMEM_COLS = MH * H < 32 ? 32 : MH * H;

  if (warp == 9 && lane == 0) {
    for (int s = 0; s < NST; ++s) {
      mbar_init(&full[s], 256);
      mbar_init(&empty[s], 1);
    }
    mbar_init(tfull, 1);
    fence_barrier_init();
  }
  if (warp == 9) tmem_alloc(tmem_slot, TMEM_COLS);
  if (H < 128) {
    for (int i = threadIdx.x; i < S::BLK / 16; i += blockDim.x) reinterpret_cast<uint4*>(smem + S::ZERO_OFF)[i] = make_uint4(0, 0, 0, 0);
    fence_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 8) {
    // producers: thread = (row group, float4 column); rows rg + RG*i of the k-block
    constexpr int C4 = H / 4, RG = 256 / C4, NI = KR / RG;
    const int c4 = threadIdx.x % C4, rg = threadIdx.x / C4;
    const int blk = (c4 * 4) / 64, col = (c4 * 4) % 64;
    float4 sv[NI], xv[NI];
    float4 dbacc = make_float4(0.f, 0.f, 0.f, 0.f);
    auto load = [&](int64_t it, int i, float4& a, float4& b) {
      const int64_t row = (blockIdx.x + it * (int64_t)gridDim.x) * KR + rg + RG * i;
      if (row < g.rows) {
        a = __ldcs(reinterpret_cast<const float4*>(g.s + row * H) + c4);
        b = __ldcs(reinterpret_cast<const float4*>(g.x + row * H) + c4);
      } else {
        a = b = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    if (items > 0) {
#pragma unroll
      for (int i = 0; i < NI; ++i) load(0, i, sv[i], xv[i]);
    }
    int stage = 0;
    uint32_t phase = 0;
    for (int64_t it = 0; it < items; ++it) {
      uint8_t* sa = smem + stage * S::STAGE_BYTES;  // [S hi][S lo][X hi][X lo]
      uint8_t* sx = sa + (X3 ? 2 : 1) * S::OPER;
      mbar_wait(&empty[stage], phase ^ 1);
      const bool more = it + 1 < items;
#pragma unroll
      for (int i = 0; i < NI; ++i) {
        const float4 a = sv[i], b = xv[i];
        dbacc.x += a.x; dbacc.y += a.y; dbacc.z += a.z; dbacc.w += a.w;
        const uint32_t off = (uint32_t)blk * S::BLK + image_offset(rg + RG * i, col);
        split_store4(a, sa, X3 ? sa + S::OPER : nullptr, off);
        split_store4(b, sx, X3 ? sx + S::OPER : nullptr, off);
        if (more) load(it + 1, i, sv[i], xv[i]);
      }
      fence_async_smem();
      mbar_arrive(&full[stage]);
      if (++stage == NST) {
        stage = 0;
        phase ^= 1;
      }
    }
    // db partial: sum the row groups' column sums in fixed order (rg = 0 .. RG-1)
    named_bar(1, 256);  // every producer is past its last stage write; reuse stage 0 as scratch once the MMAs are done
    mbar_wait(tfull, 0);
    float4* scratch = reinterpret_cast<float4*>(smem);
    scratch[rg * C4 + c4] = dbacc;
    named_bar(1, 256);
    if (rg == 0) {
      float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int r = 0; r < RG; ++r) {
        const float4 v = scratch[r * C4 + c4];
        t.x += v.x; t.y += v.y; t.z += v.z; t.w += v.w;
      }
      reinterpret_cast<float4*>(g.part_b + (size_t)blockIdx.x * H)[c4] = t;
    }
  } else if (warp == 8) {
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc(BM, H) | (1u << 15) | (1u << 16);  // A and B MN-major
      int stage = 0;
      uint32_t phase = 0;
      for (int64_t it = 0; it < items; ++it) {
        mbar_wait(&full[stage], phase);
        tc_fence_after();
        const uint32_t sa = smem_u32(smem + stage * S::STAGE_BYTES);
        const uint32_t sx = sa + (X3 ? 2 : 1) * S::OPER;
#pragma unroll
        for (int m = 0; m < MH; ++m) {
          const uint32_t d_tmem = tmem_base + (uint32_t)(m * H);
          const uint32_t a0 = sa + m * 2 * S::BLK;  // output features [128 m, 128 m + 128) = blocks 2m, 2m+1
          // H = 64: the operand has one block; the second block of the 128-row MMA is the zero block
          const uint32_t lbo_hi = H < 128 ? smem_u32(smem + S::ZERO_OFF) - a0 : (uint32_t)S::BLK;
          const uint32_t lbo_lo = H < 128 ? lbo_hi - S::OPER : (uint32_t)S::BLK;
#pragma unroll
          for (int k = 0; k < KR / 16; ++k) {
            const uint64_t a_hi = make_smem_desc_mn(a0 + k * 2048, lbo_hi), b_hi = make_smem_desc_mn(sx + k * 2048, S::BLK);
            umma_bf16(d_tmem, a_hi, b_hi, idesc, (it | k) != 0);
            if (X3) {
              const uint64_t a_lo = make_smem_desc_mn(a0 + S::OPER + k * 2048, lbo_lo);
              const uint64_t b_lo = make_smem_desc_mn(sx + S::OPER + k * 2048, S::BLK);
              umma_bf16(d_tmem, a_hi, b_lo, idesc, 1);
              umma_bf16(d_tmem, a_lo, b_hi, idesc, 1);
            }
          }
        }
        umma_commit(&empty[stage]);
        if (++stage == NST) {
          stage = 0;
          phase ^= 1;
        }
      }
      umma_commit(tfull);  // also arrives when nothing was issued
    }
  } else if (warp >= 12) {
    const int q = warp & 3, r = q * 32 + lane;
    mbar_wait(tfull, 0);
    tc_fence_after();
#pragma unroll 1
    for (int m = 0; m < MH; ++m) {
      float* dst = g.part_w + ((size_t)blockIdx.x * H + m * 128 + r) * H;
#pragma unroll 1
      for (int c0 = 0; c0 < H && m * 128 + r < H; c0 += 32) {
        uint32_t rr[32];
        if (items > 0) {
          tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(m * H + c0), rr);
          tmem_ld_wait();
        } else {
#pragma unroll
          for (int e = 0; e < 32; ++e) rr[e] = 0u;
        }
#pragma unroll
        for (int e = 0; e < 8; ++e)
          reinterpret_cast<float4*>(dst + c0)[e] = make_float4(__uint_as_float(rr[4 * e]), __uint_as_float(rr[4 * e + 1]),
                                                              __uint_as_float(rr[4 * e + 2]), __uint_as_float(rr[4 * e + 3]));
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

// out[i] = sum over CTAs of part[cta][i], fixed order
__global__ void reduce_cta_partials_kernel(const float* __restrict__ part, int ctas, int64_t n, float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s = 0.0f;
  for (int c = 0; c < ctas; ++c) s += part[(size_t)c * n + i];
  out[i] = s;
}

// most CTAs of one weight-gradient launch: azg_grid_dw_scratch_floats holds one [H, H] + [H] partial per CTA
constexpr int DW_MAX_CTAS = 160;

template <int H, bool X3>
int launch_dw(const float* s, const float* x, int64_t rows, float* dw, float* db, float* scratch, cudaStream_t st) {
  static bool configured = false;
  using S = DwSmem<H, X3>;
  int dev = 0, sms = 0;
  AZG_CUDA_CHECK(cudaGetDevice(&dev));
  AZG_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  if (!configured) {
    AZG_CUDA_CHECK(cudaFuncSetAttribute(grid_dw_tc_kernel<H, X3>, cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL));
    configured = true;
  }
  const int64_t kblocks = (rows + S::KR - 1) / S::KR;
  const int64_t ctas = sms < DW_MAX_CTAS ? sms : DW_MAX_CTAS;  // the kernel strides over the k-blocks by gridDim.x
  const int grid = (int)(kblocks < ctas ? kblocks : ctas);
  DwArgs g{s, x, scratch, scratch + (size_t)grid * H * H, rows};
  grid_dw_tc_kernel<H, X3><<<grid, 512, S::TOTAL, st>>>(g);
  AZG_LAUNCH_CHECK();
  reduce_cta_partials_kernel<<<(H * H + 255) / 256, 256, 0, st>>>(g.part_w, grid, (int64_t)H * H, dw);
  AZG_LAUNCH_CHECK();
  reduce_cta_partials_kernel<<<(H + 255) / 256, 256, 0, st>>>(g.part_b, grid, H, db);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

// 256-row tiles: needed above 128 nodes, and chosen below when they waste fewer tile rows (7x7: 245/256 instead of 98/128
// rows carry nodes, 9x9: 243/256 instead of 81/128 -- measured 9-15 % faster in bf16x3 for H <= 128; in bf16 mode only the
// 9x9-like cases gain).  AZG_GRID_TILE=256 / 128 forces the choice for graphs of up to 128 nodes (A/B runs, tests).
static int wide_tiles(int n, int H, bool x3) {
  static int forced = -1;
  if (forced < 0) {
    const char* e = getenv("AZG_GRID_TILE");
    forced = (e && strcmp(e, "256") == 0) ? 2 : (e && strcmp(e, "128") == 0) ? 1 : 0;
  }
  if (n > 128) return 1;
  if (forced) return forced == 2;
  if (H > 128) return 0;
  const float u1 = (float)((128 / n) * n) / 128.0f, u2 = (float)((256 / n) * n) / 256.0f;
  return u2 - u1 > (x3 ? 0.1f : 0.25f);
}

static int pair_h256() {  // AZG_GRID_PAIR=0: H = 256 in bf16x3 on single CTAs with streamed weights (A/B runs)
  static int on = -1;
  if (on < 0) {
    const char* e = getenv("AZG_GRID_PAIR");
    on = (e && strcmp(e, "0") == 0) ? 0 : 1;
  }
  return on;
}

template <bool BWD, int MT>
int dispatch_h(const GridArgs& g, int H, bool x3, cudaStream_t st) {
  switch (H) {
    case 64: return x3 ? launch<64, true, BWD, MT, false>(g, st) : launch<64, false, BWD, MT, false>(g, st);
    case 128: return x3 ? launch<128, true, BWD, MT, false>(g, st) : launch<128, false, BWD, MT, false>(g, st);
    case 256:
      if (!x3) return launch<256, false, BWD, MT, false>(g, st);
      // pairs keep the 256 KB of weight images resident (128 KB per CTA); with 256-row tiles there is no room left for the
      // second staging tile either way and the single CTA measured the same or better
      return (MT == 1 && pair_h256()) ? launch<256, true, BWD, 1, true>(g, st) : launch<256, true, BWD, MT, false>(g, st);
  }
  return -1;
}

template <bool BWD>
int dispatch(const GridArgs& g, int H, int prec, cudaStream_t st) {
  const bool x3 = prec == AZG_PREC_BF16X3;
  const int rc = wide_tiles(g.gh * g.gw, H, x3) ? dispatch_h<BWD, 2>(g, H, x3, st) : dispatch_h<BWD, 1>(g, H, x3, st);
  if (rc != -1) return rc;
  azg_set_error("grid layer: hidden size %d not in {64, 128, 256}", H);
  return AZG_ERR_INVALID;
}

}  // namespace gridtc

extern "C" {

size_t azg_grid_packed_bytes(int H) { return (size_t)H * H * 2 * 2; }  // hi image, lo image

int azg_grid_tc_supported(int gh, int gw, int H) {
  // each side is checked before the product, so gh * gw can neither be negative nor wrap into range
  return gh >= 1 && gw >= 1 && gh <= 256 && gw <= 256 && gh * gw <= 256 && (H == 64 || H == 128 || H == 256);
}

int azg_grid_pack_weights(const float* w, int H, int transpose, void* packed, azg_stream stream) {
  AZG_REQUIRE(w && packed && (H == 64 || H == 128 || H == 256), "azg_grid_pack_weights: bad argument");
  uint8_t* hi = (uint8_t*)packed;
  uint8_t* lo = hi + (size_t)H * H * 2;
  const int threads = H * (H / 8);
  gridtc::grid_weight_image_kernel<<<(threads + 255) / 256, 256, 0, (cudaStream_t)stream>>>(w, H, transpose, hi, lo);
  AZG_LAUNCH_CHECK();
  return AZG_OK;
}

int azg_grid_layer_tc_forward(const float* x, const void* packed_w, const float* bias, int64_t B, int gh, int gw, int H, int prec,
                              float* out, azg_stream stream) {
  AZG_REQUIRE(x && packed_w && bias && out, "azg_grid_layer_tc_forward: null pointer");
  AZG_REQUIRE(azg_grid_tc_supported(gh, gw, H), "azg_grid_layer_tc_forward: unsupported shape %dx%d, H=%d", gh, gw, H);
  AZG_REQUIRE(prec == AZG_PREC_BF16X3 || prec == AZG_PREC_BF16, "azg_grid_layer_tc_forward: precision must be bf16x3 or bf16");
  if (B <= 0) return AZG_OK;
  gridtc::GridArgs g{x, nullptr, (const uint8_t*)packed_w, (const uint8_t*)packed_w + (size_t)H * H * 2, bias, out, B, gh, gw, 1};
  return gridtc::dispatch<false>(g, H, prec, (cudaStream_t)stream);
}

int azg_grid_layer_tc_backward_input(const float* dout, const float* act, const void* packed_wt, int64_t B, int gh, int gw, int H,
                                     int prec, float* dx, azg_stream stream) {
  AZG_REQUIRE(dout && act && packed_wt && dx, "azg_grid_layer_tc_backward_input: null pointer");
  AZG_REQUIRE(azg_grid_tc_supported(gh, gw, H), "azg_grid_layer_tc_backward_input: unsupported shape %dx%d, H=%d", gh, gw, H);
  AZG_REQUIRE(prec == AZG_PREC_BF16X3 || prec == AZG_PREC_BF16, "azg_grid_layer_tc_backward_input: precision must be bf16x3 or bf16");
  if (B <= 0) return AZG_OK;
  gridtc::GridArgs g{dout, act, (const uint8_t*)packed_wt, (const uint8_t*)packed_wt + (size_t)H * H * 2, nullptr, dx, B, gh, gw, 0};
  return gridtc::dispatch<true>(g, H, prec, (cudaStream_t)stream);
}

size_t azg_grid_dw_scratch_floats(int H) { return (size_t)gridtc::DW_MAX_CTAS * ((size_t)H * H + H); }  // one partial per CTA

int azg_grid_layer_tc_backward_weights(const float* s, const float* x, int64_t rows, int H, int prec, float* dw, float* db,
                                       float* scratch, azg_stream stream) {
  AZG_REQUIRE(s && x && dw && db && scratch, "azg_grid_layer_tc_backward_weights: null pointer");
  AZG_REQUIRE(H == 64 || H == 128 || H == 256, "azg_grid_layer_tc_backward_weights: hidden size %d not in {64, 128, 256}", H);
  AZG_REQUIRE(prec == AZG_PREC_BF16X3 || prec == AZG_PREC_BF16, "azg_grid_layer_tc_backward_weights: precision must be bf16x3 or bf16");
  AZG_REQUIRE(rows > 0, "azg_grid_layer_tc_backward_weights: no rows");
  cudaStream_t st = (cudaStream_t)stream;
  const bool x3 = prec == AZG_PREC_BF16X3;
  if (H == 64) return x3 ? gridtc::launch_dw<64, true>(s, x, rows, dw, db, scratch, st) : gridtc::launch_dw<64, false>(s, x, rows, dw, db, scratch, st);
  if (H == 128) return x3 ? gridtc::launch_dw<128, true>(s, x, rows, dw, db, scratch, st) : gridtc::launch_dw<128, false>(s, x, rows, dw, db, scratch, st);
  return x3 ? gridtc::launch_dw<256, true>(s, x, rows, dw, db, scratch, st) : gridtc::launch_dw<256, false>(s, x, rows, dw, db, scratch, st);
}

}  // extern "C"
