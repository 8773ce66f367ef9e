// a6 backward on the 5th-generation tensor cores: gradient of the full-catalog softmax cross-entropy with the
// logits recomputed tile by tile (they never exist in HBM, in either direction).
//
//   g[m,j] = (exp(s[m,j] - lse[m]) - [j == target[m]]) * gscale,   s = h W^T + bias
//   d_h[m,:] = sum_j g[m,j] W[j,:]        d_W[j,:] += sum_m g[m,j] h[m,:]        d_bias[j] += sum_m g[m,j]
//
// Both products are the SAME kernel with the roles of the two matrices swapped:
//   X = 128 rows that stay resident (users for d_h, items for d_W), Y = 128-row tiles streamed past them;
//   S = X Y^T (tcgen05, bf16 hi/lo split, three MMAs, fp32 accumulation in TMEM)
//   G = exp2((S + rowb[r] + colb[c]) log2e) - [rowid[r] == colid[c]]   written back IN PLACE over S as packed bf16
//                                                                     hi/lo pairs (rows = TMEM lanes)
//   ACC += G Y   (A operand from TMEM; Y consumed a second time from the same shared-memory tile as an MN-major
//                 B operand, so neither a transpose nor a second copy exists)
// For d_h: rowb = -lse[m], rowid = target[m], colb = bias[j], colid = j.  For d_W the two sides swap and the row
// sums of G give d_bias.  A CTA owning an X tile needs no atomics; when there are fewer X tiles than SMs, or when the Y
// range is longer than MAX_RUN_TILES, the Y range is split and the partial results are added with red.global.
// Accumulation: every tcgen05.mma into ACC loses up to one fp32 ulp of the running partial (truncation-like when the
// partials have one sign), 24 MMAs per Y tile.  One run of 3,907 tiles (the d_h pass at 500k items) would lose ~3e-3 of
// |d_h| on coherent sums (an anisotropic catalog); runs of <= 256 tiles keep it near 2e-4 (tests/ce_cases.py).
// Operand format ("row images", one per 128 rows): [part hi|lo][16 slabs of 8 columns][128 rows][8 bf16] = 64 KB,
// built once per call by prepare_rows_kernel for h and for W (K is zero-padded to 128).
// Warps: 0-7 epilogue (TMEM lane quadrant = warp % 4, 64-column half = warp / 4), 8 producer (bulk copies + the
// per-column vectors of the Y tile), 9 MMA issuer.  S/G is double-buffered in TMEM so the G epilogue of tile t
// overlaps S of tile t+1 and the G.Y product of tile t-1.
//   replaces autograd of project + CrossEntropyLoss  model/influentialRS.py:214,303,307; model/evaluator.py:53-66.
#include "tc_common.cuh"

namespace irs {
namespace cet {

using namespace irs::tc;

constexpr int BM = 128, DP = 128, SLABS = DP / 8;
constexpr uint32_t LBO = BM * 16, SBO = 128;                 // K-major view: slab stride 2048, 8-row group stride 128
constexpr uint32_t PART = SLABS * LBO;                       // 32768
constexpr uint32_t TILE_BYTES = 2 * PART;                    // 65536
constexpr uint32_t OFF_X = 0, OFF_Y = TILE_BYTES;            // Y ring: 2 slots
constexpr uint32_t OFF_COL = OFF_Y + 2 * TILE_BYTES;         // per slot: float colterm[128], int colid[128]
constexpr uint32_t COL_BYTES = 128 * 8;
enum Bars { B_X = 0, B_YFULL = 1, B_YFREE = 3, B_SFULL = 5, B_GFULL = 7, B_ACC = 9, B_COUNT = 10 };
constexpr uint32_t OFF_BARS = OFF_COL + 2 * COL_BYTES;
constexpr uint32_t OFF_TMEM = OFF_BARS + B_COUNT * 8;
constexpr uint32_t SMEM_BYTES = OFF_TMEM + 16;
constexpr int THREADS = 10 * 32;
constexpr int WARP_PROD = 8, WARP_MMA = 9;
constexpr uint32_t T_ACC = 256;
constexpr int MAX_RUN_TILES = 256;                           // Y tiles one ACC accumulation may span

struct Params {
  const uint8_t* ximg; const uint8_t* yimg;      // row images
  const float* rowb; const int64_t* rowid64;     // per X row: additive term (or null = 0), id (or null = implicit index)
  const float* colb; const int64_t* colid64;     // per Y row
  int row_neg, col_neg;                          // 1: use -rowb / -colb (lse enters with a minus sign)
  int64_t RX, RY;                                // valid rows on each side
  int n_x_tiles, n_y_tiles, n_splits, tiles_per_split;
  float gscale;
  float* out; int64_t ld_out; int d;             // [RX, d] accumulated (+=) or null
  float* rowsum;                                 // [RX] accumulated (+=) or null
  int use_atomics;
  int* error_flag;
};

__device__ __forceinline__ float ex2f_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void tc_mma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile("{\n\t.reg .pred p;\n\t"
               "setp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
               :: "r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}

// src [R, d] fp32 (row stride ld) -> images [ceil(R/128)][hi|lo][16 slabs][128 rows][8 bf16], zero padded
__global__ void __launch_bounds__(256)
prepare_rows_kernel(const float* __restrict__ src, int64_t ld, int64_t R, int d, uint4* __restrict__ out) {
  const int64_t n_tiles = ceil_div(R, BM);
  const int64_t total = n_tiles * SLABS * BM;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(idx % BM);
    const int s = (int)((idx / BM) % SLABS);
    const int64_t t = idx / (BM * SLABS);
    const int64_t row = t * BM + r;
    float x[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) x[e] = (row < R && s * 8 + e < d) ? src[row * ld + s * 8 + e] : 0.f;
    uint4 hi, lo;
    split8(x, hi, lo);
    uint4* base = out + t * (TILE_BYTES / 16);
    base[s * BM + r] = hi;
    base[(PART / 16) + s * BM + r] = lo;
  }
}

__global__ void __launch_bounds__(THREADS, 1)
ce_bwd_tc_kernel(const Params p) {
  extern __shared__ __align__(128) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  auto bar = [&](int i) { return sbase + OFF_BARS + 8u * (uint32_t)i; };
  volatile uint32_t* tmem_holder = reinterpret_cast<volatile uint32_t*>(smem + OFF_TMEM);
  const int x_tile = blockIdx.x % p.n_x_tiles;
  const int split = blockIdx.x / p.n_x_tiles;
  const int y_begin = split * p.tiles_per_split;
  const int y_end = min(y_begin + p.tiles_per_split, p.n_y_tiles);
  const int T = y_end - y_begin;
  constexpr float l2e = 1.4426950408889634f;

  if (tid == 0) {
    mbar_init(bar(B_X), 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar(B_YFULL + i), 2); mbar_init(bar(B_YFREE + i), 1);
      mbar_init(bar(B_SFULL + i), 1); mbar_init(bar(B_GFULL + i), 256);
    }
    mbar_init(bar(B_ACC), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == WARP_MMA) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(sbase + OFF_TMEM), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (warp == WARP_PROD) {
    // ===== producer: the resident X tile once, then one 64 KB Y tile + its column vectors per step =====
    if (lane == 0) {
      mbar_arrive_expect_tx(bar(B_X), TILE_BYTES);
      bulk_g2s(sbase + OFF_X, p.ximg + (int64_t)x_tile * TILE_BYTES, TILE_BYTES, bar(B_X));
    }
    for (int t = 0; t < T; ++t) {
      const int slot = t & 1;
      mbar_wait(bar(B_YFREE + slot), (uint32_t)(((t >> 1) & 1) ^ 1), p.error_flag, 61);
      const int64_t yt = y_begin + t;
      if (lane == 0) {
        mbar_arrive_expect_tx(bar(B_YFULL + slot), TILE_BYTES);
        bulk_g2s(sbase + OFF_Y + slot * TILE_BYTES, p.yimg + yt * TILE_BYTES, TILE_BYTES, bar(B_YFULL + slot));
      }
      float* colterm = reinterpret_cast<float*>(smem + OFF_COL + slot * COL_BYTES);
      int* colid = reinterpret_cast<int*>(smem + OFF_COL + slot * COL_BYTES + 512);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c = lane + 32 * j;
        const int64_t yr = yt * BM + c;
        float term = -INFINITY;                      // padded Y rows contribute exp2(-inf) = 0
        int id = -2;
        if (yr < p.RY) {
          const float b = p.colb ? p.colb[yr] : 0.f;
          term = (p.col_neg ? -b : b) * l2e;
          id = p.colid64 ? (int)p.colid64[yr] : (int)yr;
          if (p.colid64 && p.colid64[yr] < 0) { term = -INFINITY; id = -2; }     // skipped row (target < 0)
        }
        colterm[c] = term;
        colid[c] = id;
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(bar(B_YFULL + slot));
    }
  } else if (warp == WARP_MMA) {
    if (lane == 0) {
      const uint32_t idesc_s = make_idesc_bf16(BM, 128);
      const uint32_t idesc_g = make_idesc_bf16(BM, 128) | (1u << 16);          // B operand (Y) MN-major
      auto issue_s = [&](int t) {
        const int b = t & 1;
        const uint32_t ys = sbase + OFF_Y + b * TILE_BYTES;
        const uint32_t dt = tmem_base + (uint32_t)b * 128u;
#pragma unroll
        for (int kk = 0; kk < DP / 16; ++kk) {
          const uint64_t x_hi = make_desc(sbase + OFF_X + (uint32_t)(2 * kk) * LBO, LBO, SBO);
          const uint64_t x_lo = make_desc(sbase + OFF_X + PART + (uint32_t)(2 * kk) * LBO, LBO, SBO);
          const uint64_t y_hi = make_desc(ys + (uint32_t)(2 * kk) * LBO, LBO, SBO);
          const uint64_t y_lo = make_desc(ys + PART + (uint32_t)(2 * kk) * LBO, LBO, SBO);
          tc_mma_bf16(dt, x_lo, y_hi, idesc_s, kk != 0 ? 1u : 0u);
          tc_mma_bf16(dt, x_hi, y_lo, idesc_s, 1u);
          tc_mma_bf16(dt, x_hi, y_hi, idesc_s, 1u);
        }
        tc_commit(bar(B_SFULL + b));
      };
      auto issue_gy = [&](int t) {
        const int b = t & 1;
        const uint32_t ys = sbase + OFF_Y + b * TILE_BYTES;
        const uint32_t gt = tmem_base + (uint32_t)b * 128u;
#pragma unroll
        for (int ks = 0; ks < BM / 16; ++ks) {                                   // 16 Y rows per step; blocks of 32 hold [hi 16 | lo 16] columns
          const uint32_t a_hi = gt + (uint32_t)((ks >> 1) * 32 + (ks & 1) * 8), a_lo = a_hi + 16u;
          // MN-major Y: rows (K) 16 B apart, 8-row groups 128 B apart (leading), 8-column slabs LBO apart (stride)
          const uint64_t y_hi = make_desc(ys + (uint32_t)(ks * 16) * 16u, 128u, LBO);
          const uint64_t y_lo = make_desc(ys + PART + (uint32_t)(ks * 16) * 16u, 128u, LBO);
          tc_mma_bf16_ts(tmem_base + T_ACC, a_lo, y_hi, idesc_g, (t | ks) != 0 ? 1u : 0u);
          tc_mma_bf16_ts(tmem_base + T_ACC, a_hi, y_lo, idesc_g, 1u);
          tc_mma_bf16_ts(tmem_base + T_ACC, a_hi, y_hi, idesc_g, 1u);
        }
        tc_commit(bar(B_YFREE + b));
      };
      mbar_wait(bar(B_X), 0u, p.error_flag, 62);
      for (int t = 0; t < T; ++t) {
        mbar_wait(bar(B_YFULL + (t & 1)), (uint32_t)((t >> 1) & 1), p.error_flag, 63);
        tc_fence_after();
        issue_s(t);
        if (t >= 1) {
          mbar_wait(bar(B_GFULL + ((t - 1) & 1)), (uint32_t)(((t - 1) >> 1) & 1), p.error_flag, 64);
          tc_fence_after();
          issue_gy(t - 1);
        }
      }
      if (T > 0) {
        mbar_wait(bar(B_GFULL + ((T - 1) & 1)), (uint32_t)(((T - 1) >> 1) & 1), p.error_flag, 65);
        tc_fence_after();
        issue_gy(T - 1);
      }
      tc_commit(bar(B_ACC));
    }
  } else if (warp < 8) {
    // ===== epilogue: thread <-> X row (TMEM lane), 64 columns (= Y rows) of every S tile =====
    const int quad = warp & 3, half = warp >> 2;
    const int row = quad * 32 + lane;
    const int64_t xr = (int64_t)x_tile * BM + row;
    const bool row_ok = xr < p.RX;
    float rowterm = -INFINITY;
    int rowid = -1;
    if (row_ok) {
      const float b = p.rowb ? p.rowb[xr] : 0.f;
      rowterm = (p.row_neg ? -b : b) * l2e;
      rowid = p.rowid64 ? (int)p.rowid64[xr] : (int)xr;
      if (p.rowid64 && p.rowid64[xr] < 0) { rowterm = -INFINITY; rowid = -1; }   // skipped row (target < 0)
    }
    const uint32_t tlane = tmem_base + (((uint32_t)(quad * 32)) << 16);
    float rs0 = 0.f, rs1 = 0.f, rs2 = 0.f, rs3 = 0.f;
    for (int t = 0; t < T; ++t) {
      const int b = t & 1;
      const float* colterm = reinterpret_cast<const float*>(smem + OFF_COL + b * COL_BYTES);
      const int* colid = reinterpret_cast<const int*>(smem + OFF_COL + b * COL_BYTES + 512);
      // the column vectors were published together with the Y tile
      mbar_wait(bar(B_YFULL + b), (uint32_t)((t >> 1) & 1), p.error_flag, 66);
      mbar_wait(bar(B_SFULL + b), (uint32_t)((t >> 1) & 1), p.error_flag, 67);
      tc_fence_after();
#pragma unroll
      for (int q2 = 0; q2 < 2; ++q2) {
        const int c0 = half * 64 + q2 * 32;
        uint32_t v[32];
        tc_ld32(tlane + (uint32_t)b * 128u + c0, v);
        tc_wait_ld();
        uint32_t pk[32];
#pragma unroll
        for (int s8 = 0; s8 < 4; ++s8) {
          float x[8];
          const float4 ct0 = *reinterpret_cast<const float4*>(colterm + c0 + s8 * 8), ct1 = *reinterpret_cast<const float4*>(colterm + c0 + s8 * 8 + 4);
          const int4 ci0 = *reinterpret_cast<const int4*>(colid + c0 + s8 * 8), ci1 = *reinterpret_cast<const int4*>(colid + c0 + s8 * 8 + 4);
          const float ct[8] = {ct0.x, ct0.y, ct0.z, ct0.w, ct1.x, ct1.y, ct1.z, ct1.w};
          const int ci[8] = {ci0.x, ci0.y, ci0.z, ci0.w, ci1.x, ci1.y, ci1.z, ci1.w};
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            float g = ex2f_approx(fmaf(__uint_as_float(v[s8 * 8 + e]), l2e, rowterm + ct[e]));
            if (ci[e] == rowid) g -= 1.0f;
            x[e] = g;
          }
          rs0 += x[0] + x[4]; rs1 += x[1] + x[5]; rs2 += x[2] + x[6]; rs3 += x[3] + x[7];
          uint4 hi, lo;
          split8(x, hi, lo);
          pk[s8 * 4 + 0] = hi.x; pk[s8 * 4 + 1] = hi.y; pk[s8 * 4 + 2] = hi.z; pk[s8 * 4 + 3] = hi.w;
          pk[16 + s8 * 4 + 0] = lo.x; pk[16 + s8 * 4 + 1] = lo.y; pk[16 + s8 * 4 + 2] = lo.z; pk[16 + s8 * 4 + 3] = lo.w;
        }
        tc_st32(tlane + (uint32_t)b * 128u + c0, pk);          // G over S, in place: [hi 16 columns | lo 16 columns]
      }
      tc_wait_st();
      tc_fence_before();
      mbar_arrive(bar(B_GFULL + b));
    }
    // ---- result: ACC * gscale added to out (this thread: 64 of the d columns), row sums to rowsum
    mbar_wait(bar(B_ACC), 0u, p.error_flag, 68);
    tc_fence_after();
    if (T > 0) {
#pragma unroll 1
      for (int q2 = 0; q2 < 2; ++q2) {
        const int c0 = half * 64 + q2 * 32;
        uint32_t v[32];
        tc_ld32(tlane + T_ACC + c0, v);
        tc_wait_ld();
        if (row_ok && p.out) {
          float* dst = p.out + xr * p.ld_out + c0;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            if (c0 + j < p.d) {
              const float val = __uint_as_float(v[j]) * p.gscale;
              if (p.use_atomics) atomicAdd(dst + j, val); else dst[j] += val;
            }
          }
        }
      }
      if (row_ok && p.rowsum) atomicAdd(p.rowsum + xr, ((rs0 + rs1) + (rs2 + rs3)) * p.gscale);
    }
    tc_fence_before();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == WARP_MMA) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(512u) : "memory");
  }
}

static void plan(int64_t RX, int64_t RY, int& n_x, int& n_y, int& n_splits, int& tps) {
  n_x = (int)ceil_div(RX, BM);
  n_y = (int)ceil_div(RY, BM);
  // at least ~2 waves of CTAs; a CTA amortises its X tile and pipeline fill over >= 16 Y tiles
  int64_t splits = 1;
  if (n_x < 2 * kNumSMs) splits = ceil_div((int64_t)2 * kNumSMs, n_x);
  const int64_t max_splits = ceil_div(n_y, 16) > 0 ? ceil_div(n_y, 16) : 1;
  if (splits > max_splits) splits = max_splits;
  tps = (int)ceil_div(n_y, splits);
  if (tps > MAX_RUN_TILES) tps = MAX_RUN_TILES;              // bound the fp32 error of one TMEM accumulation
  n_splits = (int)ceil_div(n_y, tps);
}

}  // namespace cet
}  // namespace irs

using namespace irs;

// workspace: the bf16 operand image of h, then that of W, then the error flag
struct CeBwdTcLayout { size_t wimg, flag, total; };
static CeBwdTcLayout ce_bwd_tc_layout(int M, int64_t N) {
  const size_t wimg = (size_t)ceil_div(M, cet::BM) * cet::TILE_BYTES;
  const size_t flag = wimg + (size_t)ceil_div(N, cet::BM) * cet::TILE_BYTES;
  return {wimg, flag, flag + 256};
}

extern "C" size_t irs_score_ce_bwd_tc_workspace_bytes(int M, int64_t N, int d) {
  if (M <= 0 || N <= 0 || d <= 0 || d > cet::DP) return 0;
  return ce_bwd_tc_layout(M, N).total;
}

extern "C" int irs_score_ce_bwd_tc(const float* h, int64_t ld_h, const float* W, const float* bias,
                                   const int64_t* target, const float* lse, float gscale,
                                   float* d_h, float* d_W, float* d_bias, int M, int64_t N, int d,
                                   void* workspace, size_t workspace_bytes, void* stream) {
  if (!h || !W || !target || !lse || !workspace) return IRS_E_BADARG;
  if (M <= 0 || N <= 0 || d <= 0) return IRS_E_BADARG;
  if (d > cet::DP || N > 0x7ffffffe) return IRS_E_SHAPE;
  if (workspace_bytes < irs_score_ce_bwd_tc_workspace_bytes(M, N, d)) return IRS_E_WORKSPACE;
  if ((uintptr_t)workspace & 15) return IRS_E_SHAPE;
  cudaStream_t s = (cudaStream_t)stream;
  const CeBwdTcLayout lay = ce_bwd_tc_layout(M, N);
  uint8_t* himg = (uint8_t*)workspace;
  uint8_t* wimg = himg + lay.wimg;
  int* error_flag = (int*)(himg + lay.flag);
  IRS_CUDA(cudaMemsetAsync(error_flag, 0, sizeof(int), s));
  cet::prepare_rows_kernel<<<kNumSMs * 8, 256, 0, s>>>(h, ld_h, M, d, (uint4*)himg);
  IRS_LAUNCHED();
  cet::prepare_rows_kernel<<<kNumSMs * 8, 256, 0, s>>>(W, d, N, d, (uint4*)wimg);
  IRS_LAUNCHED();
  IRS_CUDA(opt_in_smem(cet::ce_bwd_tc_kernel, cet::SMEM_BYTES));
  if (d_h != nullptr) {                                  // X = users, Y = items
    cet::Params p = {};
    p.ximg = himg; p.yimg = wimg; p.rowb = lse; p.row_neg = 1; p.rowid64 = target; p.colb = bias; p.col_neg = 0; p.colid64 = nullptr;
    p.RX = M; p.RY = N; p.gscale = gscale; p.out = d_h; p.ld_out = d; p.d = d; p.rowsum = nullptr; p.error_flag = error_flag;
    cet::plan(M, N, p.n_x_tiles, p.n_y_tiles, p.n_splits, p.tiles_per_split);
    p.use_atomics = p.n_splits > 1;
    IRS_CUDA(cudaMemsetAsync(d_h, 0, (size_t)M * d * sizeof(float), s));      // d_h is written, not accumulated
    cet::ce_bwd_tc_kernel<<<(unsigned)(p.n_x_tiles * p.n_splits), cet::THREADS, cet::SMEM_BYTES, s>>>(p);
    IRS_LAUNCHED();
  }
  if (d_W != nullptr || d_bias != nullptr) {             // X = items, Y = users (d_bias = the row sums of this pass)
    cet::Params p = {};
    p.ximg = wimg; p.yimg = himg; p.rowb = bias; p.row_neg = 0; p.rowid64 = nullptr; p.colb = lse; p.col_neg = 1; p.colid64 = target;
    p.RX = N; p.RY = M; p.gscale = gscale; p.out = d_W; p.ld_out = d; p.d = d; p.rowsum = d_bias; p.error_flag = error_flag;
    cet::plan(N, M, p.n_x_tiles, p.n_y_tiles, p.n_splits, p.tiles_per_split);
    p.use_atomics = p.n_splits > 1;
    cet::ce_bwd_tc_kernel<<<(unsigned)(p.n_x_tiles * p.n_splits), cet::THREADS, cet::SMEM_BYTES, s>>>(p);
    IRS_LAUNCHED();
  }
  return 0;
}
