// K5c on the 5th-generation tensor cores: full-catalog scoring  s = h W^T + bias  fused with the
// window mask and the arg-max, logits never leaving the SM.
//
// Precision.  The reference scores in fp32 and generated paths must agree with it, so a single
// bf16/tf32 MMA is not enough (SURVEY.md section 7: bf16 flips arg-maxes, error 9e-3).  Both
// operands are split  x = hi + lo  (two bf16) and three tcgen05.mma accumulate
//   lo_h*hi_W + hi_h*lo_W + hi_h*hi_W      (fp32 accumulation in TMEM, error ~1e-5 of |s|)
// The dropped lo*lo term is 2^-16 relative.  The decision is then re-scored exactly (fp32 FMA chain,
// same arithmetic as the CUDA-core engine) among the candidates within the error band of the
// leader, so the winner is the fp32 winner.
//
// Layout.  W is re-tiled ONCE per weight version (irs_scorer_prepare_weights) into the exact
// shared-memory image the MMA wants: for every 256-row catalog tile and every 32-wide K chunk, the
// hi and the lo halves as K-major / no-swizzle "core matrices" (8 rows x 16 bytes contiguous).  A
// pipeline stage is therefore ONE contiguous 32 KB cp.async.bulk (UBLKCP) with an mbarrier
// transaction count -- no tensor map, no swizzle, no per-row address generation.
//
// CTA = 128 users (UMMA M=128, one TMEM lane per user) x a contiguous range of catalog tiles.
// 10 warps: 0-7 epilogue (TMEM -> registers, bias, window mask, running chunk max; warp w owns TMEM
// lanes 32(w%4)..+31 and half w/4 of each tile's columns), 8 bulk-copy producer, 9 MMA issuer (single
// thread) + TMEM allocator.
// Two 256-column fp32 accumulators in TMEM (512 columns) double-buffer MMA against the epilogue.
//   reference: model/influentialRS.py:214 (project), :418-429 (softmax/topk/window filter/pick).
#include "scorer.cuh"
#include "tc_common.cuh"

namespace irs {
namespace tc {

constexpr int BM = 128;
constexpr int BN = 256;
constexpr int KC = 32;                 // K elements per stage
constexpr int STAGES = 4;                // ring slots of STAGE_BYTES (hi + lo images of one K chunk)
constexpr int MAX_STAGES = 8;            // barrier slots reserved in shared memory
constexpr int KMAX = 128;               // three-MMA schemes: hi and lo images of the A tile (2 x 32 KB)
constexpr int KMAX_SINGLE = 256;        // single-MMA schemes: only the hi image exists, it may span both A regions (64 KB)
constexpr int EPI_WARPS = 8;             // 2 per TMEM lane quadrant, each takes half of a tile's columns
constexpr int THREADS = (EPI_WARPS + 3) * 32;      // + producer, MMA issuer, second producer
constexpr uint32_t STAGE_BYTES = 2u * (KC / 8) * BN * 16;      // hi + lo : 32768
constexpr uint32_t STAGE_HALF = STAGE_BYTES / 2;               // 16384
constexpr uint32_t A_PART_BYTES = (KMAX / 8) * BM * 16;        // 32768 (hi), same for lo
constexpr uint32_t A_LBO = BM * 16;                            // K-direction core-matrix stride (bytes)
constexpr uint32_t B_LBO = BN * 16;
constexpr uint32_t SBO = 128;                                  // 8-row group stride (bytes)
constexpr uint32_t OFF_A_HI = 0;
constexpr uint32_t OFF_A_LO = A_PART_BYTES;
constexpr uint32_t OFF_B = 2 * A_PART_BYTES;
constexpr uint32_t OFF_BIAS = OFF_B + STAGES * STAGE_BYTES;    // float [8 epilogue warps][2 accumulators][128 columns]: warp private
constexpr uint32_t OFF_HN = OFF_BIAS + EPI_WARPS * 2 * 128 * 4; // float [BM]: |h_m|^2 of this CTA's rows
constexpr int SEG_TILES = 16;                                  // arg-max candidates are recorded per segment of 16 catalog tiles
constexpr int RCAP = 30;                                       // uncertain columns recorded per (row, split, half) in rank mode
constexpr int EXC = 16;                                        // excluded columns of a row cached per CTA (rest: global)
constexpr uint32_t OFF_EXC = OFF_HN + BM * 4;                  // int32 [BM][EXC]: the row's next excluded columns in this CTA's range
constexpr uint32_t OFF_BARS = OFF_EXC + BM * EXC * 4;          // uint64 [2*MAX_STAGES + 4]
constexpr uint32_t OFF_TMEM = OFF_BARS + (2 * MAX_STAGES + 4) * 8;
constexpr uint32_t SMEM_BYTES = OFF_TMEM + 16;
constexpr uint32_t TMEM_COLS = 512;

struct Params {
  const float* h; int64_t ld_h;
  const uint4* Wt;                  // prepared weights
  const float* bias;
  int M; int64_t N; int d; int n_chunks;
  const int32_t* excl_sorted; const int32_t* excl_count; int Lx;
  unsigned long long* slice_keys;   // [M, n_splits, n_segs, 2 halves, 3]: per (row, split, segment of SEG_TILES tiles, column half)
                                    // the three best 32-column chunks: key = (chunk max score, chunk first column | ambiguous flag)
  int n_segs;
  long long* timeline;              // debug: [3 roles][64 tiles][4 events] clock64 stamps of CTA 0 (null in production)
  float2* slice_ms;                 // LSE mode: [M, 2*n_splits] per (row, split, column half) running (max, sum exp(s - max))
  // MODE 2 (rank of a label): exact label score, per (row, split, column half) the count of columns surely ahead and the
  // list of columns whose tensor-core score is inside the error band of the label score (re-scored exactly afterwards)
  const float* label_score; int* rank_above; int* rank_unsure;
  float band_rel;
  int single;                       // 1: one bf16 MMA per K step (hi*hi) + a rigorous error band (arg-max only)
  const float* wmax2;               // max_j |W_j|^2 (written by irs_scorer_prepare_weights behind the images)
  float* chunk_max; int64_t ld_cm;  // MODE 3 (top-k): [M, ld_cm] best tensor-core score of every 32-column chunk (-inf: none alive)
  int m_tiles; int64_t n_tiles; int64_t tiles_per_split; int n_splits;
  int variant;                      // bit0: swap LBO/SBO (bring-up calibration only)
  int* error_flag;
};

constexpr uint32_t kIdesc = make_idesc_bf16(BM, BN);

// Error bands, relative to sum_k |h_k w_k| <= |h| |W_j| <= |h| max_j |W_j| (Cauchy-Schwarz).  bf16 keeps 8 significant bits:
// round to nearest has unit roundoff u = 2^-8 (1 + 2^-8 - 2^-20 rounds to 1).  tests/band_cases.py builds inputs that reach
// each bound, tests/test_scorer_bands_cpu.py checks them against these figures.
//
// Single MMA (hi*hi): a product is off by <= (2u + u^2) |h_k w_k|, so a score by <= (2u + u^2) |h| |W_j| = 2^-6.99 |h| |W_j|.
// Two scores may swap order only if they are within twice that, 2^-5.99; add for each score the fp32 accumulation of
// <= 256 products in the tensor core (256 * 2^-23, truncating) and the engine's FMA chain (256 * 2^-24):
// 2 (2u + u^2 + 256 * 2^-23 + 256 * 2^-24) = 0.015747, rounded up to 0.016 = 2^-5.97.
__device__ __forceinline__ float single_mma_band(float hnorm2, float wmax2) { return 0.016f * sqrtf(hnorm2 * wmax2); }

// Three MMAs (lo*hi + hi*lo + hi*hi): x = hi + lo + r with |lo| <= u |x| and |r| <= u^2 |x|; the dropped terms lo*lo, hi*r,
// r*hi (+ smaller) are <= 3u^2 (1 + 2u) = 4.61e-5 of |h_k w_k| (x = 1 + 2^-8 + 2^-17 loses 3.03e-5).  Bound on
// |s_tensor_core - s_fp32_engine| for d <= 128 (three-MMA schemes only exist there: KMAX): those terms + the fp32
// accumulation in the tensor core, budgeted as one truncation per tcgen05.mma of K = 16 (3 * 128 / 16 * 2^-23 = 2.9e-6;
// the accumulation probe in tests/test_gpu_scorer_bands.py measures 9.2e-7 on a B200 with worst-case inputs whose partial
// sums all have one sign) + the engine's 128-term FMA chain (128 * 2^-24 = 7.6e-6): 5.66e-5, rounded up.
// An arg-max compares two such scores.
static_assert(KMAX <= 128, "three_mma_band() is derived for d <= 128");
__device__ __forceinline__ float three_mma_band(float hnorm2, float wmax2) { return 5.7e-5f * sqrtf(hnorm2 * wmax2); }

__device__ __forceinline__ float ex2f_approx(float x) {     // MUFU.EX2 (ftz): exp2(-inf) = 0
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// ---- one-time weight preparation ----------------------------------------------------------------------
// out layout (uint4 = 8 bf16): [tile][chunk][part hi/lo][kslab 0..3][row 0..255]
__global__ void __launch_bounds__(256)
prepare_weights_kernel(const float* __restrict__ W, int64_t N, int d, int n_chunks, uint4* __restrict__ out) {
  const int64_t total = ceil_div(N, BN) * n_chunks * 4 * BN;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(idx % BN);
    const int s = (int)((idx / BN) % 4);
    const int c = (int)((idx / (BN * 4)) % n_chunks);
    const int64_t t = idx / ((int64_t)BN * 4 * n_chunks);
    const int64_t n = t * BN + r;
    const int k0 = c * KC + s * 8;
    float x[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) x[e] = (n < N && k0 + e < d) ? W[n * d + k0 + e] : 0.f;
    uint4 hi, lo;
    split8(x, hi, lo);
    const int64_t base = ((t * n_chunks + c) * 2) * 4 * BN;
    out[base + (int64_t)s * BN + r] = hi;
    out[base + (int64_t)(4 + s) * BN + r] = lo;
  }
}

// max_j |W_j|^2 -> *wmax2 (non-negative floats order like their bit patterns): the single-MMA arg-max needs a bound on
// the bf16 rounding error of a score, |h_m| |W_j| 2^-8
__global__ void __launch_bounds__(256)
weight_norm_kernel(const float* __restrict__ W, int64_t N, int d, float* __restrict__ wmax2) {
  float best = 0.f;
  for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (int64_t)gridDim.x * blockDim.x) {
    float acc = 0.f;
    for (int k = 0; k < d; ++k) { const float w = W[n * d + k]; acc = fmaf(w, w, acc); }
    best = fmaxf(best, acc);
  }
  best = warp_max(best);
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<unsigned int*>(wmax2), __float_as_uint(best));
}

// ---- the fused kernel ---------------------------------------------------------------------------------
// MODE 0: arg-max candidates (generation).  MODE 1: online log-sum-exp over the catalog (training / evaluator).
// MODE 2: rank of a label by counting.  MODE 3: maximum of every 32-column chunk -> top-k (k > 1), single-MMA only.
template <int MODE>
__global__ void __launch_bounds__(THREADS, 1)
score_tc_kernel(const Params p) {
  extern __shared__ __align__(128) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int m_tile = blockIdx.x % p.m_tiles;
  const int split = blockIdx.x / p.m_tiles;
  const int m0 = m_tile * BM;
  const int64_t tile_begin = (int64_t)split * p.tiles_per_split;
  const int64_t tile_end = min(tile_begin + p.tiles_per_split, p.n_tiles);
  const int n_chunks = p.n_chunks;

  auto bar_full = [&](int s) { return sbase + OFF_BARS + 8u * s; };
  auto bar_empty = [&](int s) { return sbase + OFF_BARS + 8u * (MAX_STAGES + s); };
  auto bar_tfull = [&](int a) { return sbase + OFF_BARS + 8u * (2 * MAX_STAGES + a); };
  auto bar_tempty = [&](int a) { return sbase + OFF_BARS + 8u * (2 * MAX_STAGES + 2 + a); };
  // Ring geometry.  Every wait on a slot and every tcgen05.commit that releases one costs the single MMA-issuing thread a
  // few hundred cycles (r2 timeline: 8 single MMAs issued in 2.3k cycles against an execution floor of 1.0k, 24 MMAs of the
  // three-MMA scheme in 3.9k; two producer warps or an 8-slot ring changed nothing).  Single-MMA modes copy only the hi
  // half of a K chunk (16 KB), so a 32 KB slot takes TWO chunks: half as many waits and commits per catalog tile.
  const bool hi_only = (MODE == 0 || MODE == 3) && p.single;
  const int cps = (hi_only && !(p.variant & 8)) ? 2 : 1;             // K chunks per ring slot
  volatile uint32_t* tmem_holder = reinterpret_cast<volatile uint32_t*>(smem + OFF_TMEM);

  if (tid == EPI_WARPS * 32) {
    for (int s = 0; s < MAX_STAGES; ++s) { mbar_init(bar_full(s), 1); mbar_init(bar_empty(s), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(bar_tfull(a), 1); mbar_init(bar_tempty(a), EPI_WARPS * 32); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == EPI_WARPS + 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 :: "r"(sbase + OFF_TMEM), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  // A operand: this CTA's 128 rows of h, split hi/lo, written in the canonical K-major image.
  float* hn2 = reinterpret_cast<float*>(smem + OFF_HN);
  for (int i = tid; i < BM; i += THREADS) hn2[i] = 0.f;
  __syncthreads();
  const bool vec_ok = ((reinterpret_cast<uintptr_t>(p.h) & 15) == 0) && (p.ld_h % 4 == 0) && (p.d % 8 == 0);
  if (vec_ok) {
    // thread <-> (row, half of the row's slabs): every lane walks its own row in 32-byte steps, so each 128-byte line it
    // touches is used by four consecutive loads (all issued before the first conversion)
    const int n_slabs = n_chunks * 4, per = (n_slabs + 1) / 2;
    const bool write_lo = n_chunks * KC <= KMAX;             // K > 128 (single-MMA only): the hi image spans both regions
    if (tid < 2 * BM) {
      const int r = tid % BM, s_lo = (tid / BM) * per, s1 = min(s_lo + per, n_slabs);
      const int m = m0 + r;
      const float4* src = reinterpret_cast<const float4*>(p.h + (int64_t)(m < p.M ? m : 0) * p.ld_h);
      float q = 0.f;
      for (int s0 = s_lo; s0 < s1; s0 += 8) {
        float4 v[16];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int slab = s0 + j;
          const bool ok = slab < s1 && m < p.M && slab * 8 < p.d;
          v[2 * j] = ok ? __ldg(src + slab * 2) : make_float4(0.f, 0.f, 0.f, 0.f);
          v[2 * j + 1] = ok ? __ldg(src + slab * 2 + 1) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int slab = s0 + j;
          if (slab < s1) {
            const float x[8] = {v[2 * j].x, v[2 * j].y, v[2 * j].z, v[2 * j].w, v[2 * j + 1].x, v[2 * j + 1].y, v[2 * j + 1].z, v[2 * j + 1].w};
#pragma unroll
            for (int e = 0; e < 8; ++e) q = fmaf(x[e], x[e], q);
            uint4 hi, lo;
            split8(x, hi, lo);
            *reinterpret_cast<uint4*>(smem + OFF_A_HI + slab * A_LBO + r * 16) = hi;
            if (write_lo) *reinterpret_cast<uint4*>(smem + OFF_A_LO + slab * A_LBO + r * 16) = lo;
          }
        }
      }
      if (MODE == 0 || MODE == 2) atomicAdd(hn2 + r, q);
    }
  } else {
  for (int idx = tid; idx < n_chunks * 4 * BM; idx += THREADS) {
    const int r = idx % BM, slab = idx / BM;
    const int m = m0 + r, k0 = slab * 8;
    float x[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) x[e] = (m < p.M && k0 + e < p.d) ? p.h[(int64_t)m * p.ld_h + k0 + e] : 0.f;
    if (MODE == 0 || MODE == 2) {
      float q = 0.f;
#pragma unroll
      for (int e = 0; e < 8; ++e) q = fmaf(x[e], x[e], q);
      atomicAdd(hn2 + r, q);
    }
    uint4 hi, lo;
    split8(x, hi, lo);
    *reinterpret_cast<uint4*>(smem + OFF_A_HI + slab * A_LBO + r * 16) = hi;
    if (n_chunks * KC <= KMAX) *reinterpret_cast<uint4*>(smem + OFF_A_LO + slab * A_LBO + r * 16) = lo;
  }
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");    // generic-proxy writes -> visible to the MMA
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (warp == EPI_WARPS || warp == EPI_WARPS + 2) {
    // ===== producers: one bulk copy per (tile, K chunk).  The copies ONE warp issues execute one after the other (~420
    // cycles each whatever their size up to 32 KB: profiles/micro/bulk_load_bench), copies of different warps overlap: with
    // two producer warps (even / odd copies, p.variant bit 2) the ring fills at twice the rate =====
    const int n_prod = (p.variant & 4) ? 2 : 1;
    const int me = (warp == EPI_WARPS) ? 0 : 1;
    if (lane == 0 && me < n_prod) {
      int stage = 0; uint32_t phase = 0; int turn = 0;                 // slot / phase of the running group, whose producer it is
      for (int64_t tile = tile_begin; tile < tile_end; ++tile) {
        for (int c0 = 0; c0 < n_chunks; c0 += cps) {
          if (turn == me) {
            const int nch = min(cps, n_chunks - c0);
            mbar_wait(bar_empty(stage), phase ^ 1u, p.error_flag, 1);
            const uint32_t nbytes = hi_only ? STAGE_HALF : STAGE_BYTES;                               // hi images come first
            mbar_arrive_expect_tx(bar_full(stage), nbytes * (uint32_t)nch);
            for (int j = 0; j < nch; ++j) {
              const uint4* src = p.Wt + ((tile * n_chunks + c0 + j) * (int64_t)(STAGE_BYTES / 16));
              bulk_g2s(sbase + OFF_B + stage * STAGE_BYTES + (uint32_t)j * STAGE_HALF, src, nbytes, bar_full(stage));
            }
          }
          if (++turn == n_prod) turn = 0;
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == EPI_WARPS + 1) {
    // ===== MMA issuer: a single thread drives the tensor core =====
    // Per-tile timeline (debug hook irs_scorer_debug_timeline, scripts/scorer_timeline.py), single-MMA mode: a tile's 8 MMAs
    // take ~2.0k cycles from the first wait for a stage to the last issue (their execution floor is 1k, and ncu shows the
    // tensor pipe 28 % active = at the floor when it runs), the epilogue of a tile ~2.4k, the tile period 2.9k.  Measured
    // and ruled out for the issue time: a second producer warp, a deeper ring (8 x 16 KB), spinning instead of the
    // suspending mbarrier wait (worse: 2.65k).  Shared-memory wavefronts (ncu) are at ~40 % of the pipe.  With three MMAs
    // per K step the issuer is MMA-bound (24 MMAs in 3.7k cycles).  Open for round 2 together with cta_group::2.
    if (lane == 0) {
      const bool swap = (p.variant & 1) != 0;
      const uint32_t a_lbo = swap ? SBO : A_LBO, a_sbo = swap ? A_LBO : SBO;
      const uint32_t b_lbo = swap ? SBO : B_LBO, b_sbo = swap ? B_LBO : SBO;
      int stage = 0; uint32_t phase = 0;
      int it = 0;
      for (int64_t tile = tile_begin; tile < tile_end; ++tile, ++it) {
        const int ab = it & 1;
        const uint32_t acc_phase = (uint32_t)(it >> 1) & 1u;
        if (p.timeline && blockIdx.x == 0 && it < 64) p.timeline[(0 * 64 + it) * 4 + 0] = clock64();
        mbar_wait(bar_tempty(ab), acc_phase ^ 1u, p.error_flag, 2);
        tc_fence_after();
        if (p.timeline && blockIdx.x == 0 && it < 64) p.timeline[(0 * 64 + it) * 4 + 1] = clock64();
        const uint32_t d_tmem = tmem_base + (uint32_t)(ab * BN);
        for (int c0 = 0; c0 < n_chunks; c0 += cps) {
          mbar_wait(bar_full(stage), phase, p.error_flag, 3);
          tc_fence_after();
          const int nch = min(cps, n_chunks - c0);
          for (int j = 0; j < nch; ++j) {
            const int c = c0 + j;
            const uint32_t bs = sbase + OFF_B + stage * STAGE_BYTES + (uint32_t)j * STAGE_HALF;
#pragma unroll
            for (int kk = 0; kk < KC / 16; ++kk) {
              const uint32_t a_off = (uint32_t)(c * 4 + kk * 2) * A_LBO;
              const uint32_t b_off = (uint32_t)(kk * 2) * B_LBO;
              const uint64_t a_hi = make_desc(sbase + OFF_A_HI + a_off, a_lbo, a_sbo);
              const uint64_t a_lo = make_desc(sbase + OFF_A_LO + a_off, a_lbo, a_sbo);
              const uint64_t b_hi = make_desc(bs + b_off, b_lbo, b_sbo);
              const uint64_t b_lo = make_desc(bs + STAGE_HALF + b_off, b_lbo, b_sbo);
              if (hi_only) {
                tc_mma_bf16(d_tmem, a_hi, b_hi, kIdesc, (c | kk) != 0 ? 1u : 0u);
              } else {
                tc_mma_bf16(d_tmem, a_lo, b_hi, kIdesc, (c | kk) != 0 ? 1u : 0u);   // small terms first
                tc_mma_bf16(d_tmem, a_hi, b_lo, kIdesc, 1u);
                tc_mma_bf16(d_tmem, a_hi, b_hi, kIdesc, 1u);
              }
            }
          }
          tc_commit(bar_empty(stage));          // slot reusable once these MMAs have read it
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
        tc_commit(bar_tfull(ab));               // accumulator complete -> epilogue
        if (p.timeline && blockIdx.x == 0 && it < 64) p.timeline[(0 * 64 + it) * 4 + 2] = clock64();
      }
    }
  } else {
    // ===== epilogue warps 0..7: thread <-> user row (TMEM lane = 32*(warp%4) + lane); warp/4 selects
    // which half of each tile's columns this warp scans.  Hot loop per element: one FADD (bias) and one
    // FMNMX.  Only the best 32-column CHUNK (and the runner-up chunk's score, for the ambiguity flag) is
    // tracked; the exact column is recovered by the fp32 re-scoring kernel.
    const int quad = warp & 3, half = warp >> 2;
    const int row = quad * 32 + lane;
    const int m = m0 + row;
    const bool row_ok = m < p.M;
    float best_v = -INFINITY, second_v = (MODE == 1) ? 0.f : -INFINITY, third_v = -INFINITY, fourth_v = -INFINITY;
    int best_c0 = -1, second_c0 = -1, third_c0 = -1;
    const int32_t* elist = nullptr;
    int ecnt = 0, eptr = 0;
    int64_t next_col = INT64_MAX;                               // next excluded column (register-cached)
    if (row_ok && p.excl_sorted != nullptr) {
      elist = p.excl_sorted + (int64_t)m * p.Lx;
      ecnt = p.excl_count[m];
      const int64_t first = tile_begin * BN;
      int lo = 0, hi = ecnt;
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (elist[mid] < first) lo = mid + 1; else hi = mid; }
      eptr = lo;
      if (eptr < ecnt) next_col = elist[eptr];
    }
    // the row's next EXC excluded columns go to shared memory once: the tile loop then advances through them with
    // shared-memory reads instead of one dependent global load per excluded column
    int32_t* exc_s = reinterpret_cast<int32_t*>(smem + OFF_EXC) + row * EXC;
    const int ebase = eptr;
    if (half == 0) {
#pragma unroll
      for (int e = 0; e < EXC; ++e) exc_s[e] = (elist != nullptr && ebase + e < ecnt) ? elist[ebase + e] : 0x7fffffff;
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
    auto fetch_excl = [&](int idx) -> int64_t {
      if (idx >= ecnt) return INT64_MAX;
      return (idx - ebase < EXC) ? (int64_t)exc_s[idx - ebase] : (int64_t)elist[idx];
    };
    // bias of this warp's 128 columns (its half of the tile), warp private: no CTA-wide barrier per tile.  The next
    // tile's values are fetched while the current tile is processed.
    float* bias_w = reinterpret_cast<float*>(smem + OFF_BIAS) + warp * 256;
    auto load_bias = [&](int64_t tile, float (&b4)[4]) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int64_t n = tile * BN + half * (BN / 2) + lane * 4 + e;
        b4[e] = (p.bias != nullptr && tile < tile_end && n < p.N) ? __ldg(p.bias + n) : 0.f;
      }
    };
    float bias_next[4];
    load_bias(tile_begin, bias_next);
    // rank mode: columns above label + E are surely ahead, below label - E surely behind, the rest is listed
    float thr_hi = INFINITY, thr_lo = INFINITY;
    int above = 0, n_uns = 0;
    int* uns_list = nullptr;
    if (MODE == 2 && row_ok) {
      const float lab = p.label_score[m];
      const float E = three_mma_band(hn2[row], *p.wmax2) + 1e-6f * fabsf(lab);
      thr_hi = lab + E; thr_lo = lab - E;                       // NaN label score (label out of range): nothing counts
      uns_list = p.rank_unsure + (((int64_t)m * p.n_splits + split) * 2 + half) * (1 + RCAP);
    }
    int it = 0;
    for (int64_t tile = tile_begin; tile < tile_end; ++tile, ++it) {
      const int ab = it & 1;
      const uint32_t acc_phase = (uint32_t)(it >> 1) & 1u;
      const int64_t n0 = tile * BN;
      *reinterpret_cast<float4*>(bias_w + ab * 128 + lane * 4) = make_float4(bias_next[0], bias_next[1], bias_next[2], bias_next[3]);
      load_bias(tile + 1, bias_next);
      __syncwarp();
      if (p.timeline && blockIdx.x == 0 && it < 64 && tid == 0) p.timeline[(1 * 64 + it) * 4 + 0] = clock64();
      mbar_wait(bar_tfull(ab), acc_phase, p.error_flag, 4);
      tc_fence_after();
      if (p.timeline && blockIdx.x == 0 && it < 64 && tid == 0) p.timeline[(1 * 64 + it) * 4 + 1] = clock64();
      const uint32_t tchunk0 = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(ab * BN + half * (BN / 2));
      float cm4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};     // MODE 3: this thread's four chunk maxima of the tile
      auto process = [&](const uint32_t (&v)[32], int cc) {
        const int ch = half * (BN / 64) + cc;
        const int64_t c0 = n0 + ch * 32;
        const float4* bs4 = reinterpret_cast<const float4*>(bias_w + ab * 128 + cc * 32);
        float sc[32];
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) {
          const float4 b = bs4[j4];
          sc[4 * j4 + 0] = __uint_as_float(v[4 * j4 + 0]) + b.x;
          sc[4 * j4 + 1] = __uint_as_float(v[4 * j4 + 1]) + b.y;
          sc[4 * j4 + 2] = __uint_as_float(v[4 * j4 + 2]) + b.z;
          sc[4 * j4 + 3] = __uint_as_float(v[4 * j4 + 3]) + b.w;
        }
        while (next_col < c0) { ++eptr; next_col = fetch_excl(eptr); }                          // other half's columns
        if (next_col < c0 + 32 || c0 + 32 > p.N) {              // rare: window items / catalog tail in this chunk
          uint32_t dead = 0u;
          while (next_col < c0 + 32) {
            dead |= 1u << (int)(next_col - c0);
            ++eptr; next_col = fetch_excl(eptr);
          }
          if (c0 + 32 > p.N) dead |= (c0 >= p.N) ? 0xffffffffu : (0xffffffffu << (int)(p.N - c0));
#pragma unroll
          for (int j = 0; j < 32; ++j) if ((dead >> j) & 1u) sc[j] = -INFINITY;
        }
        if (MODE == 2) {
          int a = 0, ge = 0;
#pragma unroll
          for (int j = 0; j < 32; ++j) { a += (sc[j] > thr_hi) ? 1 : 0; ge += (sc[j] >= thr_lo) ? 1 : 0; }
          above += a;
          if (ge != a) {                                        // rare: some column is inside the band
#pragma unroll
            for (int j = 0; j < 32; ++j) {                       // unrolled: sc[] must stay in registers
              if (sc[j] >= thr_lo && !(sc[j] > thr_hi)) {
                if (n_uns < RCAP) uns_list[1 + n_uns] = (int)(c0 + j);
                ++n_uns;
              }
            }
          }
          return;
        }
        float m0v = fmaxf(sc[0], sc[1]), m1v = fmaxf(sc[2], sc[3]), m2v = fmaxf(sc[4], sc[5]), m3v = fmaxf(sc[6], sc[7]);
#pragma unroll
        for (int j = 8; j < 32; j += 4) {
          m0v = fmaxf(m0v, sc[j]); m1v = fmaxf(m1v, sc[j + 1]); m2v = fmaxf(m2v, sc[j + 2]); m3v = fmaxf(m3v, sc[j + 3]);
        }
        const float cm = fmaxf(fmaxf(m0v, m1v), fmaxf(m2v, m3v));
        if (MODE == 3) { cm4[cc] = cm; return; }
        if (MODE == 0) {
          // branch-free insertion of (cm, c0) into the sorted (best, second, third | fourth) list: every thread has its
          // own list, so an if/else chain diverges in all 32 lanes (BSSY/BSYNC around each arm in the r1 SASS)
          const bool g1 = cm > best_v, g2 = cm > second_v, g3 = cm > third_v;
          const int ci = (int)c0;
          const float n4 = g3 ? third_v : fmaxf(fourth_v, cm);
          const float n3 = g2 ? second_v : (g3 ? cm : third_v);
          const int n3c = g2 ? second_c0 : (g3 ? ci : third_c0);
          const float n2 = g1 ? best_v : (g2 ? cm : second_v);
          const int n2c = g1 ? best_c0 : (g2 ? ci : second_c0);
          best_v = g1 ? cm : best_v; best_c0 = g1 ? ci : best_c0;
          second_v = n2; second_c0 = n2c; third_v = n3; third_c0 = n3c; fourth_v = n4;
        } else {
          // online log-sum-exp: best_v = running max, second_v = sum of exp(s - running max) (exp2 with log2(e) folded in)
          constexpr float l2e = 1.4426950408889634f;
          if (cm > best_v) {
            second_v *= ex2f_approx((best_v - cm) * l2e);         // first chunk: 0 * exp2(-inf) = 0
            best_v = cm;
          }
          if (best_v > -INFINITY) {
            const float nb = -best_v * l2e;
            float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              a0 += ex2f_approx(fmaf(sc[j], l2e, nb)); a1 += ex2f_approx(fmaf(sc[j + 1], l2e, nb));
              a2 += ex2f_approx(fmaf(sc[j + 2], l2e, nb)); a3 += ex2f_approx(fmaf(sc[j + 3], l2e, nb));
            }
            second_v += (a0 + a1) + (a2 + a3);
          }
        }
      };
      // four 32-column chunks per thread and tile, one TMEM load in flight behind the arithmetic
      {
        uint32_t va[32], vb[32];
        tc_ld32(tchunk0, va);
        tc_wait_ld();
        tc_ld32(tchunk0 + 32, vb);
        process(va, 0);
        tc_wait_ld();
        tc_ld32(tchunk0 + 64, va);
        process(vb, 1);
        tc_wait_ld();
        tc_ld32(tchunk0 + 96, vb);
        process(va, 2);
        tc_wait_ld();
        process(vb, 3);
      }
      tc_fence_before();
      mbar_arrive(bar_tempty(ab));
      if (MODE == 3 && row_ok)        // one 16-byte store per thread and tile; the two column halves fill a 32-byte sector
        *reinterpret_cast<float4*>(p.chunk_max + (int64_t)m * p.ld_cm + tile * (BN / 32) + half * 4) =
            make_float4(cm4[0], cm4[1], cm4[2], cm4[3]);
      if (p.timeline && blockIdx.x == 0 && it < 64 && tid == 0) p.timeline[(1 * 64 + it) * 4 + 2] = clock64();
      if (MODE == 0 && (((it + 1) % SEG_TILES) == 0 || tile + 1 == tile_end)) {
        // Candidates of this (row, split, segment, column half): its three best 32-column chunks.  If even the FOURTH
        // best chunk is inside the error band of the best one the fp32 winner could sit in a chunk that is not recorded:
        // flag the slice, the re-scoring kernel then scans the segment exactly.  Segments keep that rare (a few dozen
        // chunk maxima are well separated, hundreds are not) and bound what a flagged slice costs (4096 columns).
        if (row_ok) {
          unsigned long long k0 = 0ull, k1 = 0ull, k2 = 0ull;
          if (best_c0 >= 0 && best_v > -INFINITY) {
            const float band = p.band_rel * fmaxf(1.0f, fabsf(best_v)) +
                               (p.single ? single_mma_band(hn2[row], *p.wmax2) : 2.f * three_mma_band(hn2[row], *p.wmax2));
            const uint32_t flag = (best_v - fourth_v < band) ? 1u : 0u;
            k0 = pack_key(best_v, (uint32_t)best_c0 | flag);
            if (second_c0 >= 0 && second_v > -INFINITY) k1 = pack_key(second_v, (uint32_t)second_c0);
            if (third_c0 >= 0 && third_v > -INFINITY) k2 = pack_key(third_v, (uint32_t)third_c0);
          }
          unsigned long long* dst = p.slice_keys + ((((int64_t)m * p.n_splits + split) * p.n_segs + it / SEG_TILES) * 2 + half) * 3;
          dst[0] = k0; dst[1] = k1; dst[2] = k2;
        }
        best_v = -INFINITY; second_v = -INFINITY; third_v = -INFINITY; fourth_v = -INFINITY;
        best_c0 = -1; second_c0 = -1; third_c0 = -1;
      }
    }
    if (MODE == 0 && row_ok) {                        // segments this (shorter, last) split does not have
      for (int seg = (it + SEG_TILES - 1) / SEG_TILES; seg < p.n_segs; ++seg) {
        unsigned long long* dst = p.slice_keys + ((((int64_t)m * p.n_splits + split) * p.n_segs + seg) * 2 + half) * 3;
        dst[0] = 0ull; dst[1] = 0ull; dst[2] = 0ull;
      }
    }
    if (MODE == 2) {
      if (row_ok) {
        p.rank_above[((int64_t)m * p.n_splits + split) * 2 + half] = above;
        uns_list[0] = n_uns;
      }
    } else if (MODE == 1) {
      if (row_ok) p.slice_ms[((int64_t)m * p.n_splits + split) * 2 + half] = make_float2(best_v, second_v);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == EPI_WARPS + 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// ---- exact re-scoring of the near-leaders -----------------------------------------------------------------
// Candidates = for every (row, split, column half) the two 32-column chunks with the best tensor-core
// chunk maxima.  The leader's chunk is re-scored first; every candidate whose chunk maximum is within the error bound of
// one score below that exact score is then re-scored column by column with the fp32 FMA chain of the CUDA-core engine (excluded / out-of-range columns skipped); a flagged
// candidate (third-best chunk of its slice inside the band) triggers an exact scan of its whole split.
// The winner is the best exact (score desc, column asc) key.  One warp per row.
__device__ __forceinline__ bool is_excluded(const int32_t* lst, int cnt, int64_t col) {
  int lo = 0, hi = cnt;
  while (lo < hi) { const int mid = (lo + hi) >> 1; if (lst[mid] < col) lo = mid + 1; else hi = mid; }
  return lo < cnt && lst[lo] == col;
}

__global__ void __launch_bounds__(256)
rescore_finalize_kernel(const unsigned long long* __restrict__ slice_keys, int n_cand, const float* __restrict__ h,
                        int64_t ld_h, const float* __restrict__ W, const float* __restrict__ bias, int M, int64_t N, int d,
                        int64_t item_base, float band_rel, const float* __restrict__ wmax2, int single,
                        const int32_t* __restrict__ excl_sorted,
                        const int32_t* __restrict__ excl_count, int Lx, int64_t tiles_per_split, int n_segs,
                        const float* __restrict__ ext_lead, float* __restrict__ vals, int64_t* __restrict__ items) {
  const int lane = threadIdx.x & 31;
  const int m = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (m >= M) return;
  const unsigned long long* keys = slice_keys + (int64_t)m * n_cand;
  unsigned long long lead = 0ull;
  for (int c = lane; c < n_cand; c += 32) lead = keys[c] > lead ? keys[c] : lead;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long other = __shfl_xor_sync(0xffffffffu, lead, o);
    lead = other > lead ? other : lead;
  }
  if (lead == 0ull) {
    if (lane == 0) { vals[m] = -INFINITY; items[m] = -1; }
    return;
  }
  // catalog-sharded call (phase 2): the leader is the best tensor-core score over ALL shards, so a shard that cannot hold
  // the row's winner finds no candidate inside the band and returns (-inf, -1) without reading W
  const float lead_s = ext_lead ? fmaxf(key_score(lead), ext_lead[m]) : key_score(lead);
  // rounding-error band of this row: the single-MMA or the (doubled) three-MMA bound, on top of the band_rel floor
  float hn = 0.f;
  for (int kk = lane; kk < d; kk += 32) { const float x = h[(int64_t)m * ld_h + kk]; hn = fmaf(x, x, hn); }
  hn = warp_sum(hn);
  // E bounds |s_tensor_core - s_fp32| of one score (plus the band_rel floor for the bias addition)
  const float E = band_rel * fmaxf(1.0f, fabsf(lead_s)) + (single ? 0.5f * single_mma_band(hn, *wmax2) : three_mma_band(hn, *wmax2));
  const int32_t* lst = excl_sorted ? excl_sorted + (int64_t)m * Lx : nullptr;
  const int ecnt = excl_sorted ? excl_count[m] : 0;
  const float* hr = h + (int64_t)m * ld_h;
  unsigned long long best = 0ull;
  // (staging the 32 rows of W through shared memory for coalesced loads was measured: no gain -- the kernel is bound by
  // fetching 16 KB of W per candidate chunk from L2 / HBM, not by L1 wavefronts)
  const bool vec = ((d & 3) == 0) && ((reinterpret_cast<uintptr_t>(W) & 15) == 0) && ((reinterpret_cast<uintptr_t>(hr) & 15) == 0);
  auto exact = [&](int64_t col) {
    if (col >= N || (lst && is_excluded(lst, ecnt, col))) return;
    float acc = 0.f;
    if (vec) {                                          // 16-byte loads, the SAME sequential FMA chain over k
      const float4* wr = reinterpret_cast<const float4*>(W + col * d);
      const float4* h4 = reinterpret_cast<const float4*>(hr);
      for (int k4 = 0; k4 < d / 4; ++k4) {
        const float4 w = __ldg(wr + k4), x = h4[k4];
        acc = fmaf(x.x, w.x, acc); acc = fmaf(x.y, w.y, acc); acc = fmaf(x.z, w.z, acc); acc = fmaf(x.w, w.w, acc);
      }
    } else {
      for (int kk = 0; kk < d; ++kk) acc = fmaf(hr[kk], __ldg(W + col * d + kk), acc);
    }
    acc = acc + (bias ? __ldg(bias + col) : 0.f);
    const unsigned long long ek = pack_key(acc, (uint32_t)col);
    best = ek > best ? ek : best;
  };
  auto rescore = [&](unsigned long long key, int c) {   // whole warp: one candidate chunk, or its flagged segment
    const uint32_t cf = key_col(key);
    if (cf & 1u) {                                      // ambiguous slice: exact scan of its segment (both column halves)
      const int split = (c / 6) / n_segs, seg = (c / 6) % n_segs;
      const int64_t t0 = (int64_t)split * tiles_per_split + (int64_t)seg * SEG_TILES;
      const int64_t t1 = min(t0 + SEG_TILES, (int64_t)(split + 1) * tiles_per_split);
      const int64_t lo = t0 * BN, hi = min(t1 * BN, N);
      for (int64_t col = lo + lane; col < hi; col += 32) exact(col);
    } else {
      exact((int64_t)(cf & ~31u) + lane);
    }
  };
  auto warp_best = [&]() {
    unsigned long long b = best;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long other = __shfl_xor_sync(0xffffffffu, b, o);
      b = other > b ? other : b;
    }
    return b;
  };
  // The fp32 winner w scores >= any exact score L of a live column, and its chunk maximum is >= s_w - E >= L - E.  Whole
  // catalog (phase 0): re-score the leader's chunk first, L = its best exact score (>= lead_s - E), then every candidate at
  // or above L - E.  Phase 2 knows no exact score of the global leader: candidates at or above lead_s - 2E.
  float thr = lead_s - 2.f * E;
  if (!ext_lead) {
    for (int c0 = 0; c0 < n_cand; c0 += 32) {
      const unsigned long long mykey = (c0 + lane < n_cand) ? keys[c0 + lane] : 0ull;
      const unsigned hit = __ballot_sync(0xffffffffu, mykey == lead);
      if (hit) { rescore(lead, c0 + __ffs(hit) - 1); break; }
    }
    const unsigned long long b = warp_best();
    if (b) thr = fmaxf(thr, key_score(b) - E);
  }
  // 32 candidates at a time (one coalesced load), the few inside the band are then handled by the whole warp
  for (int c0 = 0; c0 < n_cand; c0 += 32) {
    const unsigned long long mykey = (c0 + lane < n_cand) ? keys[c0 + lane] : 0ull;
    unsigned hits = __ballot_sync(0xffffffffu, mykey != 0ull && !(key_score(mykey) < thr) && (ext_lead || mykey != lead));
    while (hits) {
      const int src = __ffs(hits) - 1;
      hits &= hits - 1;
      rescore(__shfl_sync(0xffffffffu, mykey, src), c0 + src);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long other = __shfl_xor_sync(0xffffffffu, best, o);
    best = other > best ? other : best;
  }
  if (lane == 0) {
    vals[m] = best ? key_score(best) : -INFINITY;
    items[m] = best ? (int64_t)key_col(best) + item_base : -1;
  }
}

// ---- phase 1 of the catalog-sharded arg-max: the shard's best tensor-core score per row ---------------------------------
__global__ void __launch_bounds__(256)
approx_leader_kernel(const unsigned long long* __restrict__ slice_keys, int n_cand, int M, const float* __restrict__ wmax2,
                     float* __restrict__ lead_out) {
  const int lane = threadIdx.x & 31;
  const int m = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (blockIdx.x == 0 && threadIdx.x == 0) lead_out[M] = wmax2 ? *wmax2 : 0.f;      // the shard's rounding-error scale
  if (m >= M) return;
  const unsigned long long* keys = slice_keys + (int64_t)m * n_cand;
  unsigned long long lead = 0ull;
  for (int c = lane; c < n_cand; c += 32) lead = keys[c] > lead ? keys[c] : lead;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long other = __shfl_xor_sync(0xffffffffu, lead, o);
    lead = other > lead ? other : lead;
  }
  if (lane == 0) lead_out[m] = lead ? key_score(lead) : -INFINITY;
}

// ---- log-sum-exp finalisation -----------------------------------------------------------------------------
// Combines the per-(split, column half) running (max, sum) pairs of a row into lse = max + ln(sum), and
// computes the selected logits EXACTLY (fp32 FMA chain, as the CUDA-core engine) -- the cross-entropy of a row
// is lse - logit[target], so only the lse carries the ~1e-5 tensor-core error.  One warp per row.
__global__ void __launch_bounds__(256)
lse_finalize_kernel(const float2* __restrict__ slice_ms, int n_part, const float* __restrict__ h, int64_t ld_h,
                    const float* __restrict__ W, const float* __restrict__ bias, int M, int64_t N, int d, int64_t item_base,
                    const int64_t* __restrict__ sel, int n_sel, float* __restrict__ lse, float* __restrict__ logit) {
  const int lane = threadIdx.x & 31;
  const int m = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (m >= M) return;
  const float2* ms = slice_ms + (int64_t)m * n_part;
  float mx = -INFINITY;
  for (int c = lane; c < n_part; c += 32) mx = fmaxf(mx, ms[c].x);
  mx = warp_max(mx);
  float sum = 0.f;
  for (int c = lane; c < n_part; c += 32) { const float2 v = ms[c]; if (v.x > -INFINITY) sum += v.y * expf(v.x - mx); }
  sum = warp_sum(sum);
  if (lane == 0) lse[m] = mx + logf(sum);
  const float* hr = h + (int64_t)m * ld_h;
  for (int t = 0; t < n_sel; ++t) {
    const int64_t col = sel[(int64_t)m * n_sel + t] - item_base;
    float acc = 0.f;
    if (col >= 0 && col < N) {
      for (int kk = lane; kk < d; kk += 32) acc = fmaf(hr[kk], __ldg(W + col * d + kk), acc);
    }
    acc = warp_sum(acc);
    if (lane == 0) logit[(int64_t)m * n_sel + t] = (col >= 0 && col < N) ? acc + (bias ? __ldg(bias + col) : 0.f) : 0.f;
  }
}

// ---- rank finalisation -------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
rank_label_score_kernel(const float* __restrict__ h, int64_t ld_h, const float* __restrict__ W, const float* __restrict__ bias,
                        const int64_t* __restrict__ label, int64_t item_base, int M, int64_t N, int d, float* __restrict__ out) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  const int64_t c = label[m] - item_base;
  float acc = NAN;
  if (c >= 0 && c < N) {                                  // the same sequential FMA chain as every exact re-score
    acc = 0.f;
    for (int kk = 0; kk < d; ++kk) acc = fmaf(h[(int64_t)m * ld_h + kk], W[c * d + kk], acc);
    acc = acc + (bias ? bias[c] : 0.f);
  }
  out[m] = acc;
}

// rank = 1 + (columns surely ahead) + (listed uncertain columns that are exactly ahead: score > label score, or equal and
// lower column); a slice whose list overflowed is counted exactly from scratch.  0 if the label is excluded / out of
// range.  One warp per row.
__global__ void __launch_bounds__(256)
rank_finalize_tc_kernel(const int* __restrict__ rank_above, const int* __restrict__ rank_unsure, int n_splits,
                        int64_t tiles_per_split, const float* __restrict__ label_score, const int64_t* __restrict__ label,
                        const float* __restrict__ h, int64_t ld_h, const float* __restrict__ W, const float* __restrict__ bias,
                        int M, int64_t N, int d, int64_t item_base, const int32_t* __restrict__ excl_sorted,
                        const int32_t* __restrict__ excl_count, int Lx, int64_t* __restrict__ rank,
                        int32_t* __restrict__ count_excluded /* non-null: COUNT mode of a catalog shard */) {
  const int lane = threadIdx.x & 31;
  const int m = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (m >= M) return;
  const int64_t l = label[m] - item_base;
  const int32_t* lst = excl_sorted ? excl_sorted + (int64_t)m * Lx : nullptr;
  const int ecnt = excl_sorted ? excl_count[m] : 0;
  const bool count_mode = count_excluded != nullptr;
  if (!count_mode) {
    if (l < 0 || l >= N || (lst && is_excluded(lst, ecnt, l))) { if (lane == 0) rank[m] = 0; return; }
  } else if (lane == 0) {
    // the label may live in another shard (l out of range): its score comes from outside, nothing is "the label" here
    count_excluded[m] = (l >= 0 && l < N && lst && is_excluded(lst, ecnt, l)) ? 1 : 0;
  }
  const float lab = label_score[m];
  const float* hr = h + (int64_t)m * ld_h;
  const bool vec = ((d & 3) == 0) && ((reinterpret_cast<uintptr_t>(W) & 15) == 0) && ((reinterpret_cast<uintptr_t>(hr) & 15) == 0);
  auto ahead_exact = [&](int64_t col) -> int {
    if (col == l || col >= N) return 0;
    float acc = 0.f;
    if (vec) {                                          // 16-byte loads, the SAME sequential FMA chain over k
      const float4* wr = reinterpret_cast<const float4*>(W + col * d);
      const float4* h4 = reinterpret_cast<const float4*>(hr);
      for (int k4 = 0; k4 < d / 4; ++k4) {
        const float4 w = __ldg(wr + k4), x = h4[k4];
        acc = fmaf(x.x, w.x, acc); acc = fmaf(x.y, w.y, acc); acc = fmaf(x.z, w.z, acc); acc = fmaf(x.w, w.w, acc);
      }
    } else {
      for (int kk = 0; kk < d; ++kk) acc = fmaf(hr[kk], __ldg(W + col * d + kk), acc);
    }
    acc = acc + (bias ? __ldg(bias + col) : 0.f);
    return (acc > lab || (acc == lab && col < l)) ? 1 : 0;
  };
  int total = 0;
  const int n_slices = n_splits * 2;
  for (int sl = 0; sl < n_slices; ++sl) {                   // warp-uniform loop
    const int64_t slot = (int64_t)m * n_slices + sl;
    const int* ul = rank_unsure + slot * (1 + RCAP);
    const int n = ul[0];
    if (n <= RCAP) {
      if (lane == 0) total += rank_above[slot];
      for (int i = lane; i < n; i += 32) total += ahead_exact(ul[1 + i]);
    } else {
      // overflow: count this (split, column half) slice exactly; half h owns columns [128 h, 128 h + 128) of every tile
      const int split = sl >> 1, half = sl & 1;
      const int64_t t0 = (int64_t)split * tiles_per_split, t1 = min(t0 + tiles_per_split, ceil_div(N, (int64_t)BN));
      for (int64_t t = t0; t < t1; ++t)
        for (int c = lane; c < BN / 2; c += 32) {
          const int64_t col = t * BN + half * (BN / 2) + c;
          if (col < N && !(lst && is_excluded(lst, ecnt, col))) total += ahead_exact(col);
        }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) total += __shfl_xor_sync(0xffffffffu, total, o);
  if (lane == 0) rank[m] = (int64_t)total + (count_mode ? 0 : 1);
}

// ---- top-k (k > 1) finalisation ---------------------------------------------------------------------------------------
// Input: the best single-MMA (hi*hi) score of every 32-column chunk of the row (MODE 3).  With E the bound on
// |s_hihi - s_fp32| of such a score, (2u + u^2) |h| max_j |W_j| plus accumulation, u = 2^-8 (single_mma_band() is 2E):
//   * tau = the k-th largest chunk maximum.  k distinct chunks hold a column scoring >= tau on the tensor core, i.e.
//     >= tau - E exactly, so the exact k-th best score T_k >= tau - E;
//   * a column of the exact top-k scores >= T_k, hence >= tau - 2E on the tensor core: it lives in a chunk whose maximum is
//     >= tau - 2E.  Those chunks (k plus a few) are re-scored column by column with the fp32 FMA chain of the CUDA-core
//     engine (same bits as irs_score_topk), keys below tau - 2E dropped, the rest sorted by (score desc, column asc).
// One CTA per row: 4-pass radix select over the chunk maxima, candidate list and key list in shared memory.  A row whose
// lists overflow (thousands of chunks inside the band: degenerate, tie-saturated scores) gets the engine's overflow marker
// (NaN, -2), like irs_score_topk.
constexpr int TK_CAND_CAP = 4096;
constexpr int TK_KEY_CAP = 2048;          // static shared memory: 16 KB keys + 16 KB candidate chunks
constexpr int TK_DMAX = KMAX_SINGLE;

__device__ __forceinline__ void bitonic_desc_256(unsigned long long* keys, int P) {
  for (int size = 2; size <= P; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      __syncthreads();
      for (int t = threadIdx.x; t < (P >> 1); t += blockDim.x) {
        const int lo = 2 * t - (t & (stride - 1));
        const int hi = lo + stride;
        const bool desc = ((lo & size) == 0);
        const unsigned long long a = keys[lo], b = keys[hi];
        if ((a < b) == desc) { keys[lo] = b; keys[hi] = a; }
      }
    }
  }
  __syncthreads();
}

__global__ void __launch_bounds__(256)
topk_select_kernel(const float* __restrict__ chunk_max, int64_t ld_cm, int64_t n_chunk, const float* __restrict__ h,
                   int64_t ld_h, const float* __restrict__ W, const float* __restrict__ bias, int M, int64_t N, int d,
                   int64_t item_base, float band_rel, const float* __restrict__ wmax2,
                   const int32_t* __restrict__ excl_sorted, const int32_t* __restrict__ excl_count, int Lx, int k,
                   float* __restrict__ vals, int64_t* __restrict__ items) {
  __shared__ unsigned long long s_keys[TK_KEY_CAP];
  __shared__ int s_cand[TK_CAND_CAP];
  __shared__ float s_h[TK_DMAX];
  __shared__ unsigned s_hist[256];
  __shared__ unsigned s_prefix;
  __shared__ int s_kk, s_ncand, s_nkeys;
  __shared__ float s_red[8];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int m = blockIdx.x;
  const float* cm = chunk_max + (int64_t)m * ld_cm;
  const float* hr = h + (int64_t)m * ld_h;
  float q = 0.f;
  for (int kk = tid; kk < d; kk += 256) { const float x = hr[kk]; s_h[kk] = x; q = fmaf(x, x, q); }
  q = warp_sum(q);
  if (lane == 0) s_red[warp] = q;
  if (tid == 0) { s_ncand = 0; s_nkeys = 0; }
  __syncthreads();
  float hn = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) hn += s_red[w];
  // ---- tau: k-th largest chunk maximum (exact, 4 x 8-bit radix select on order-preserving keys)
  float tau = -INFINITY;
  if (n_chunk >= k) {
    unsigned prefix = 0u, mask = 0u;
    int kk = k;
    for (int pass = 0; pass < 4; ++pass) {
      const int shift = 24 - 8 * pass;
      s_hist[tid] = 0u;
      __syncthreads();
      for (int64_t i = tid; i < n_chunk; i += 256) {
        const unsigned u = f32_orderable(cm[i]);
        if ((u & mask) == prefix) atomicAdd(&s_hist[(u >> shift) & 255u], 1u);
      }
      __syncthreads();
      if (tid == 0) {
        int cum = 0, b = 255;
        for (; b > 0; --b) { if (cum + (int)s_hist[b] >= kk) break; cum += (int)s_hist[b]; }
        s_prefix = prefix | ((unsigned)b << shift);
        s_kk = kk - cum;
      }
      __syncthreads();
      prefix = s_prefix; kk = s_kk; mask |= 0xffu << shift;
      __syncthreads();
    }
    tau = f32_from_orderable(prefix);
  }
  const bool all = !(tau > -INFINITY);                      // fewer than k live chunks: every live column is a candidate
  const float band = all ? 0.f : band_rel * fmaxf(1.0f, fabsf(tau)) + single_mma_band(hn, *wmax2);
  const float thr = all ? -INFINITY : tau - band;
  // ---- candidate chunks
  for (int64_t i = tid; i < n_chunk; i += 256) {
    const float v = cm[i];
    if (v > -INFINITY && v >= thr) {
      const int pos = atomicAdd(&s_ncand, 1);
      if (pos < TK_CAND_CAP) s_cand[pos] = (int)i;
    }
  }
  __syncthreads();
  const int n_cand = min(s_ncand, TK_CAND_CAP);
  bool overflow = s_ncand > TK_CAND_CAP;
  // ---- exact re-scoring: one warp per candidate chunk, one lane per column
  const int32_t* lst = excl_sorted ? excl_sorted + (int64_t)m * Lx : nullptr;
  const int ecnt = excl_sorted ? excl_count[m] : 0;
  const bool vec = ((d & 3) == 0) && ((reinterpret_cast<uintptr_t>(W) & 15) == 0);
  for (int c = warp; c < n_cand; c += 8) {
    const int64_t col = (int64_t)s_cand[c] * 32 + lane;
    if (col < N && !(lst && is_excluded(lst, ecnt, col))) {
      float acc = 0.f;
      if (vec) {
        const float4* wr = reinterpret_cast<const float4*>(W + col * d);
        for (int k4 = 0; k4 < d / 4; ++k4) {
          const float4 w = __ldg(wr + k4);
          acc = fmaf(s_h[4 * k4], w.x, acc); acc = fmaf(s_h[4 * k4 + 1], w.y, acc);
          acc = fmaf(s_h[4 * k4 + 2], w.z, acc); acc = fmaf(s_h[4 * k4 + 3], w.w, acc);
        }
      } else {
        for (int kk = 0; kk < d; ++kk) acc = fmaf(s_h[kk], __ldg(W + col * d + kk), acc);
      }
      acc = acc + (bias ? __ldg(bias + col) : 0.f);
      if (acc >= thr && acc > -INFINITY) {
        const int pos = atomicAdd(&s_nkeys, 1);
        if (pos < TK_KEY_CAP) s_keys[pos] = pack_key(acc, (uint32_t)col);
      }
    }
  }
  __syncthreads();
  overflow = overflow || s_nkeys > TK_KEY_CAP;
  const int n = min(s_nkeys, TK_KEY_CAP);
  int P = 1;
  while (P < n || P < k) P <<= 1;                             // k <= 1024 <= TK_KEY_CAP
  for (int t = n + tid; t < P; t += 256) s_keys[t] = 0ull;
  bitonic_desc_256(s_keys, P);
  for (int t = tid; t < k; t += 256) {
    const unsigned long long key = s_keys[t];
    float v; int64_t it;
    if (overflow) { v = NAN; it = -2; }                       // IRS_E_OVERFLOW marker, as irs_score_topk
    else if (key) { v = key_score(key); it = (int64_t)key_col(key) + item_base; }
    else { v = -INFINITY; it = -1; }                          // fewer than k live items
    vals[(int64_t)m * k + t] = v;
    items[(int64_t)m * k + t] = it;
  }
}

static void plan(int M, int64_t N, int& m_tiles, int64_t& n_tiles, int64_t& tiles_per_split, int& n_splits) {
  m_tiles = (int)ceil_div(M, BM);
  n_tiles = ceil_div(N, BN);
  // ~96 catalog tiles per CTA amortise the A staging and the pipeline fill; whole waves of 148 CTAs.
  int64_t ctas = ceil_div(ceil_div((int64_t)m_tiles * n_tiles, 96), kNumSMs) * kNumSMs;
  int64_t splits = ctas / m_tiles;
  if (splits < 1) splits = 1;
  if (splits > n_tiles) splits = n_tiles;
  tiles_per_split = ceil_div(n_tiles, splits);
  n_splits = (int)ceil_div(n_tiles, tiles_per_split);
}

}  // namespace tc
}  // namespace irs

using namespace irs;

static long long* g_scorer_timeline = nullptr;
/* debug hook (not in the public header): device buffer of 3*64*4 int64 receiving CTA 0's per-tile time stamps */
extern "C" void irs_scorer_debug_timeline(long long* buf) { g_scorer_timeline = buf; }

extern "C" size_t irs_scorer_prepared_bytes(int64_t N, int d) {
  if (N <= 0 || d <= 0 || d > tc::KMAX_SINGLE) return 0;      // d in (128, 256]: single-MMA consumers only (arg-max, top-k)
  const int n_chunks = (d + tc::KC - 1) / tc::KC;
  return (size_t)ceil_div(N, tc::BN) * n_chunks * tc::STAGE_BYTES + 256;      // + tail: max_j |W_j|^2
}

extern "C" int irs_scorer_prepare_weights(const float* W, int64_t N, int d, void* prepared, void* stream) {
  if (!W || !prepared || N <= 0 || d <= 0) return IRS_E_BADARG;
  if (d > tc::KMAX_SINGLE) return IRS_E_SHAPE;
  const int n_chunks = (d + tc::KC - 1) / tc::KC;
  tc::prepare_weights_kernel<<<kNumSMs * 8, 256, 0, (cudaStream_t)stream>>>(W, N, d, n_chunks, (uint4*)prepared);
  IRS_LAUNCHED();
  float* wmax2 = (float*)((char*)prepared + (size_t)ceil_div(N, tc::BN) * n_chunks * tc::STAGE_BYTES);
  IRS_CUDA(cudaMemsetAsync(wmax2, 0, 256, (cudaStream_t)stream));
  tc::weight_norm_kernel<<<kNumSMs * 4, 256, 0, (cudaStream_t)stream>>>(W, N, d, wmax2);
  IRS_LAUNCHED();
  return 0;
}

extern "C" size_t irs_score_argmax_tc_workspace_bytes(int M, int64_t N, int d) {
  if (M <= 0 || N <= 0 || d <= 0) return 0;
  int m_tiles, n_splits; int64_t n_tiles, tps;
  tc::plan(M, N, m_tiles, n_tiles, tps, n_splits);
  const size_t n_segs = (size_t)ceil_div(tps, (int64_t)tc::SEG_TILES);
  return (((size_t)M * n_splits * n_segs * 6 * 8 + 255) & ~(size_t)255) + 256;
}

// phase 0: score + re-score (one shard = the whole catalog); phase 1: score + per-row shard leader -> lead[M+1];
// phase 2: re-score against the global leaders lead[M+1] (lead[M] = max over shards of max_j |W_j|^2)
static int argmax_tc_run(int phase, const float* h, int64_t ld_h, const float* W, const void* prepared, const float* bias,
                         int64_t item_base, const int32_t* excl_sorted, const int32_t* excl_count, int Lx,
                         float* lead, float* vals, int64_t* items, int M, int64_t N, int d, int variant,
                         void* workspace, size_t workspace_bytes, void* stream) {
  if (!h || !W || !prepared || !workspace) return IRS_E_BADARG;
  if ((phase != 1 && (!vals || !items)) || (phase != 0 && !lead)) return IRS_E_BADARG;
  if (M <= 0 || N <= 0 || d <= 0) return IRS_E_BADARG;
  if (d > tc::KMAX_SINGLE || N > 0x7ffffffe) return IRS_E_SHAPE;
  if (d > tc::KMAX && !(variant & 2)) return IRS_E_SHAPE;       // 128 < d <= 256: single-MMA variant only (no lo image of h)
  if (excl_sorted && (!excl_count || Lx <= 0)) return IRS_E_BADARG;
  if (workspace_bytes < irs_score_argmax_tc_workspace_bytes(M, N, d)) return IRS_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  tc::Params p = {};
  p.h = h; p.ld_h = ld_h; p.Wt = (const uint4*)prepared; p.bias = bias; p.M = M; p.N = N; p.d = d;
  p.n_chunks = (d + tc::KC - 1) / tc::KC;
  p.excl_sorted = excl_sorted; p.excl_count = excl_count; p.Lx = Lx;
  tc::plan(M, N, p.m_tiles, p.n_tiles, p.tiles_per_split, p.n_splits);
  p.n_segs = (int)ceil_div(p.tiles_per_split, (int64_t)tc::SEG_TILES);
  p.slice_keys = (unsigned long long*)workspace;
  p.error_flag = (int*)((char*)workspace + (((size_t)M * p.n_splits * p.n_segs * 6 * 8 + 255) & ~(size_t)255));
  p.variant = variant;
  p.timeline = g_scorer_timeline;
  p.single = (variant & 2) ? 1 : 0;
  p.wmax2 = (const float*)((const char*)prepared + (size_t)ceil_div(N, tc::BN) * p.n_chunks * tc::STAGE_BYTES);
  // floor of the band, relative to the leader's score: covers the fp32 rounding of the bias addition in both scores
  p.band_rel = 1e-4f;
  const int n_cand = p.n_splits * p.n_segs * 6;
  if (phase != 2) {
    IRS_CUDA(cudaMemsetAsync(p.error_flag, 0, sizeof(int), s));
    static bool configured = false;
    if (!configured) {
      IRS_CUDA(cudaFuncSetAttribute(tc::score_tc_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::SMEM_BYTES));
      configured = true;
    }
    tc::score_tc_kernel<0><<<(unsigned)(p.m_tiles * p.n_splits), tc::THREADS, tc::SMEM_BYTES, s>>>(p);
    IRS_LAUNCHED();
  }
  if (phase == 1) {
    tc::approx_leader_kernel<<<(unsigned)ceil_div((int64_t)M * 32, 256), 256, 0, s>>>(p.slice_keys, n_cand, M, p.wmax2, lead);
    IRS_LAUNCHED();
    return 0;
  }
  // the error band of phase 2 uses the largest weight norm of ANY shard: the global leader may come from there
  const float* wmax2 = phase == 2 ? lead + M : p.wmax2;
  tc::rescore_finalize_kernel<<<(unsigned)ceil_div((int64_t)M * 32, 256), 256, 0, s>>>(
      p.slice_keys, n_cand, h, ld_h, W, bias, M, N, d, item_base, p.band_rel, wmax2, p.single,
      excl_sorted, excl_count, Lx, p.tiles_per_split, p.n_segs, phase == 2 ? lead : nullptr, vals, items);
  IRS_LAUNCHED();
  return 0;
}

extern "C" int irs_score_argmax_tc(const float* h, int64_t ld_h, const float* W, const void* prepared, const float* bias,
                                   int64_t item_base, const int32_t* excl_sorted, const int32_t* excl_count, int Lx,
                                   float* vals, int64_t* items, int M, int64_t N, int d, int variant,
                                   void* workspace, size_t workspace_bytes, void* stream) {
  return argmax_tc_run(0, h, ld_h, W, prepared, bias, item_base, excl_sorted, excl_count, Lx, nullptr, vals, items, M, N, d, variant,
                       workspace, workspace_bytes, stream);
}

extern "C" int irs_score_argmax_tc_phase1(const float* h, int64_t ld_h, const float* W, const void* prepared, const float* bias,
                                          int64_t item_base, const int32_t* excl_sorted, const int32_t* excl_count, int Lx,
                                          float* lead, int M, int64_t N, int d, int variant,
                                          void* workspace, size_t workspace_bytes, void* stream) {
  return argmax_tc_run(1, h, ld_h, W, prepared, bias, item_base, excl_sorted, excl_count, Lx, lead, nullptr, nullptr, M, N, d, variant,
                       workspace, workspace_bytes, stream);
}

extern "C" int irs_score_argmax_tc_phase2(const float* h, int64_t ld_h, const float* W, const void* prepared, const float* bias,
                                          int64_t item_base, const int32_t* excl_sorted, const int32_t* excl_count, int Lx,
                                          const float* lead_global, float* vals, int64_t* items, int M, int64_t N, int d, int variant,
                                          void* workspace, size_t workspace_bytes, void* stream) {
  return argmax_tc_run(2, h, ld_h, W, prepared, bias, item_base, excl_sorted, excl_count, Lx, const_cast<float*>(lead_global), vals,
                       items, M, N, d, variant, workspace, workspace_bytes, stream);
}

extern "C" size_t irs_score_lse_gather_tc_workspace_bytes(int M, int64_t N, int d) {
  if (M <= 0 || N <= 0 || d <= 0) return 0;
  int m_tiles, n_splits; int64_t n_tiles, tps;
  tc::plan(M, N, m_tiles, n_tiles, tps, n_splits);
  return (((size_t)M * n_splits * 2 * 8 + 255) & ~(size_t)255) + 256;
}

extern "C" int irs_score_lse_gather_tc(const float* h, int64_t ld_h, const float* W, const void* prepared, const float* bias,
                                       int64_t item_base, const int64_t* sel, int n_sel, float* lse, float* logit,
                                       int M, int64_t N, int d, void* workspace, size_t workspace_bytes, void* stream) {
  if (!h || !W || !prepared || !lse || !workspace) return IRS_E_BADARG;
  if (M <= 0 || N <= 0 || d <= 0 || n_sel < 0 || (n_sel > 0 && (!sel || !logit))) return IRS_E_BADARG;
  if (d > tc::KMAX || N > 0x7ffffffe) return IRS_E_SHAPE;
  if (workspace_bytes < irs_score_lse_gather_tc_workspace_bytes(M, N, d)) return IRS_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  tc::Params p = {};
  p.h = h; p.ld_h = ld_h; p.Wt = (const uint4*)prepared; p.bias = bias; p.M = M; p.N = N; p.d = d;
  p.n_chunks = (d + tc::KC - 1) / tc::KC;
  tc::plan(M, N, p.m_tiles, p.n_tiles, p.tiles_per_split, p.n_splits);
  p.slice_ms = (float2*)workspace;
  p.error_flag = (int*)((char*)workspace + (((size_t)M * p.n_splits * 2 * 8 + 255) & ~(size_t)255));
  IRS_CUDA(cudaMemsetAsync(p.error_flag, 0, sizeof(int), s));
  static bool configured = false;
  if (!configured) {
    IRS_CUDA(cudaFuncSetAttribute(tc::score_tc_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::SMEM_BYTES));
    configured = true;
  }
  tc::score_tc_kernel<1><<<(unsigned)(p.m_tiles * p.n_splits), tc::THREADS, tc::SMEM_BYTES, s>>>(p);
  IRS_LAUNCHED();
  tc::lse_finalize_kernel<<<(unsigned)ceil_div((int64_t)M * 32, 256), 256, 0, s>>>(
      p.slice_ms, p.n_splits * 2, h, ld_h, W, bias, M, N, d, item_base, sel, n_sel, lse, logit);
  IRS_LAUNCHED();
  return 0;
}

static size_t rank_ws_layout(int M, int n_splits, size_t& off_above, size_t& off_unsure, size_t& off_flag) {
  auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
  size_t o = al((size_t)M * 4);                                   // label scores
  off_above = o; o += al((size_t)M * n_splits * 2 * 4);
  off_unsure = o; o += al((size_t)M * n_splits * 2 * (1 + tc::RCAP) * 4);
  off_flag = o; o += 256;
  return o;
}

extern "C" size_t irs_score_rank_tc_workspace_bytes(int M, int64_t N, int d) {
  if (M <= 0 || N <= 0 || d <= 0) return 0;
  int m_tiles, n_splits; int64_t n_tiles, tps;
  tc::plan(M, N, m_tiles, n_tiles, tps, n_splits);
  size_t a, b, c;
  return rank_ws_layout(M, n_splits, a, b, c);
}

extern "C" int irs_score_rank_tc(const float* h, int64_t ld_h, const float* W, const void* prepared, const float* bias,
                                 int64_t item_base, const int64_t* label, const int32_t* excl_sorted, const int32_t* excl_count,
                                 int Lx, int64_t* rank, int M, int64_t N, int d,
                                 void* workspace, size_t workspace_bytes, void* stream) {
  if (!h || !W || !prepared || !label || !rank || !workspace) return IRS_E_BADARG;
  if (M <= 0 || N <= 0 || d <= 0) return IRS_E_BADARG;
  if (d > tc::KMAX || N > 0x7ffffffe) return IRS_E_SHAPE;
  if (excl_sorted && (!excl_count || Lx <= 0)) return IRS_E_BADARG;
  if (workspace_bytes < irs_score_rank_tc_workspace_bytes(M, N, d)) return IRS_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  tc::Params p = {};
  p.h = h; p.ld_h = ld_h; p.Wt = (const uint4*)prepared; p.bias = bias; p.M = M; p.N = N; p.d = d;
  p.n_chunks = (d + tc::KC - 1) / tc::KC;
  p.excl_sorted = excl_sorted; p.excl_count = excl_count; p.Lx = Lx;
  tc::plan(M, N, p.m_tiles, p.n_tiles, p.tiles_per_split, p.n_splits);
  size_t off_above, off_unsure, off_flag;
  rank_ws_layout(M, p.n_splits, off_above, off_unsure, off_flag);
  float* lab_s = (float*)workspace;
  p.label_score = lab_s;
  p.rank_above = (int*)((char*)workspace + off_above);
  p.rank_unsure = (int*)((char*)workspace + off_unsure);
  p.error_flag = (int*)((char*)workspace + off_flag);
  p.wmax2 = (const float*)((const char*)prepared + (size_t)ceil_div(N, tc::BN) * p.n_chunks * tc::STAGE_BYTES);
  IRS_CUDA(cudaMemsetAsync(p.error_flag, 0, sizeof(int), s));
  tc::rank_label_score_kernel<<<(unsigned)ceil_div(M, 256), 256, 0, s>>>(h, ld_h, W, bias, label, item_base, M, N, d, lab_s);
  IRS_LAUNCHED();
  static bool configured = false;
  if (!configured) {
    IRS_CUDA(cudaFuncSetAttribute(tc::score_tc_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::SMEM_BYTES));
    configured = true;
  }
  tc::score_tc_kernel<2><<<(unsigned)(p.m_tiles * p.n_splits), tc::THREADS, tc::SMEM_BYTES, s>>>(p);
  IRS_LAUNCHED();
  tc::rank_finalize_tc_kernel<<<(unsigned)ceil_div((int64_t)M * 32, 256), 256, 0, s>>>(
      p.rank_above, p.rank_unsure, p.n_splits, p.tiles_per_split, lab_s, label, h, ld_h, W, bias, M, N, d, item_base,
      excl_sorted, excl_count, Lx, rank, nullptr);
  IRS_LAUNCHED();
  return 0;
}

extern "C" int irs_score_count_ahead_tc(const float* h, int64_t ld_h, const float* W, const void* prepared, const float* bias,
                                        int64_t item_base, const int64_t* label, const float* label_score,
                                        const int32_t* excl_sorted, const int32_t* excl_count, int Lx,
                                        int64_t* count, int32_t* label_excluded, int M, int64_t N, int d,
                                        void* workspace, size_t workspace_bytes, void* stream) {
  if (!h || !W || !prepared || !label || !label_score || !count || !label_excluded || !workspace) return IRS_E_BADARG;
  if (M <= 0 || N <= 0 || d <= 0) return IRS_E_BADARG;
  if (d > tc::KMAX || N > 0x7ffffffe) return IRS_E_SHAPE;
  if (excl_sorted && (!excl_count || Lx <= 0)) return IRS_E_BADARG;
  if (workspace_bytes < irs_score_rank_tc_workspace_bytes(M, N, d)) return IRS_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  tc::Params p = {};
  p.h = h; p.ld_h = ld_h; p.Wt = (const uint4*)prepared; p.bias = bias; p.M = M; p.N = N; p.d = d;
  p.n_chunks = (d + tc::KC - 1) / tc::KC;
  p.excl_sorted = excl_sorted; p.excl_count = excl_count; p.Lx = Lx;
  tc::plan(M, N, p.m_tiles, p.n_tiles, p.tiles_per_split, p.n_splits);
  size_t off_above, off_unsure, off_flag;
  rank_ws_layout(M, p.n_splits, off_above, off_unsure, off_flag);
  p.label_score = label_score;                         // the owning shard's exact fp32 score, given from outside
  p.rank_above = (int*)((char*)workspace + off_above);
  p.rank_unsure = (int*)((char*)workspace + off_unsure);
  p.error_flag = (int*)((char*)workspace + off_flag);
  p.wmax2 = (const float*)((const char*)prepared + (size_t)ceil_div(N, tc::BN) * p.n_chunks * tc::STAGE_BYTES);
  IRS_CUDA(cudaMemsetAsync(p.error_flag, 0, sizeof(int), s));
  static bool configured = false;
  if (!configured) {
    IRS_CUDA(cudaFuncSetAttribute(tc::score_tc_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::SMEM_BYTES));
    configured = true;
  }
  tc::score_tc_kernel<2><<<(unsigned)(p.m_tiles * p.n_splits), tc::THREADS, tc::SMEM_BYTES, s>>>(p);
  IRS_LAUNCHED();
  tc::rank_finalize_tc_kernel<<<(unsigned)ceil_div((int64_t)M * 32, 256), 256, 0, s>>>(
      p.rank_above, p.rank_unsure, p.n_splits, p.tiles_per_split, label_score, label, h, ld_h, W, bias, M, N, d, item_base,
      excl_sorted, excl_count, Lx, count, label_excluded);
  IRS_LAUNCHED();
  return 0;
}


// ---- top-k (k > 1) on the tensor cores ----------------------------------------------------------------------------------
static size_t topk_tc_ws_layout(int M, int64_t N, size_t& off_flag, int64_t& ld_cm) {
  ld_cm = ceil_div(N, (int64_t)tc::BN) * (tc::BN / 32);
  size_t o = ((size_t)M * (size_t)ld_cm * 4 + 255) & ~(size_t)255;
  off_flag = o;
  return o + 256;
}

extern "C" size_t irs_score_topk_tc_workspace_bytes(int M, int64_t N, int d, int k) {
  if (M <= 0 || N <= 0 || d <= 0 || k <= 0) return 0;
  size_t off; int64_t ld;
  return topk_tc_ws_layout(M, N, off, ld);
}

extern "C" int irs_score_topk_tc(const float* h, int64_t ld_h, const float* W, const void* prepared, const float* bias,
                                 int64_t item_base, const int32_t* excl_sorted, const int32_t* excl_count, int Lx, int k,
                                 float* vals, int64_t* items, int M, int64_t N, int d,
                                 void* workspace, size_t workspace_bytes, void* stream) {
  if (!h || !W || !prepared || !vals || !items || !workspace) return IRS_E_BADARG;
  if (M <= 0 || N <= 0 || d <= 0 || k < 1 || k > 1024) return IRS_E_BADARG;
  if (d > tc::KMAX_SINGLE || N > 0x7ffffffe) return IRS_E_SHAPE;
  if (excl_sorted && (!excl_count || Lx <= 0)) return IRS_E_BADARG;
  if (workspace_bytes < irs_score_topk_tc_workspace_bytes(M, N, d, k)) return IRS_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  tc::Params p = {};
  p.h = h; p.ld_h = ld_h; p.Wt = (const uint4*)prepared; p.bias = bias; p.M = M; p.N = N; p.d = d;
  p.n_chunks = (d + tc::KC - 1) / tc::KC;
  p.excl_sorted = excl_sorted; p.excl_count = excl_count; p.Lx = Lx;
  tc::plan(M, N, p.m_tiles, p.n_tiles, p.tiles_per_split, p.n_splits);
  size_t off_flag;
  topk_tc_ws_layout(M, N, off_flag, p.ld_cm);
  p.chunk_max = (float*)workspace;
  p.error_flag = (int*)((char*)workspace + off_flag);
  p.single = 1;
  p.variant = 2;
  p.band_rel = 1e-4f;
  p.wmax2 = (const float*)((const char*)prepared + (size_t)ceil_div(N, tc::BN) * p.n_chunks * tc::STAGE_BYTES);
  IRS_CUDA(cudaMemsetAsync(p.error_flag, 0, sizeof(int), s));
  static bool configured = false;
  if (!configured) {
    IRS_CUDA(cudaFuncSetAttribute(tc::score_tc_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::SMEM_BYTES));
    configured = true;
  }
  tc::score_tc_kernel<3><<<(unsigned)(p.m_tiles * p.n_splits), tc::THREADS, tc::SMEM_BYTES, s>>>(p);
  IRS_LAUNCHED();
  tc::topk_select_kernel<<<(unsigned)M, 256, 0, s>>>(p.chunk_max, p.ld_cm, p.ld_cm, h, ld_h, W, bias, M, N, d, item_base,
                                                   p.band_rel, p.wmax2, excl_sorted, excl_count, Lx, k, vals, items);
  IRS_LAUNCHED();
  return 0;
}
