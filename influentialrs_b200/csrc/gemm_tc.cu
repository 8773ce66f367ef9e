// Decoder-body linear layers on the 5th-generation tensor cores, fp32-faithful:
//   C[R, Nout] = epilogue( A[R, K] . W[Nout, K]^T )        A, C fp32 row-major in HBM
// with the same bf16 hi/lo split and three accumulating tcgen05.mma as the catalog scorer
// (lo*hi + hi*lo + hi*hi, fp32 accumulation in TMEM), and fused epilogues:
//   EPI_BIAS       C = acc + bias                                   (in_proj of self-attention)
//   EPI_BIAS_RELU  C = relu(acc + bias)                             (linear1 of the FFN)
//   EPI_RESID_LN   C = LN(resid + acc + bias)  [ -> LN( . + c2) ]   (out_proj+norm1(+cross-attn const+norm2),
//                                                                    linear2+norm3)
// The layers are HBM-bound (K = 128..256, Nout = 128..256), so the kernel is organised around keeping
// loads in flight:  persistent CTAs, one 128-row activation tile at a time (UMMA M=128, TMEM lane =
// activation row), K streamed in 32-wide chunks through a 4-stage ring.  Per stage the A chunk is
// converted fp32 -> bf16 hi/lo by converter warps straight into the canonical K-major shared-memory
// image, and the weight chunk (re-tiled once, L2 resident) arrives as one cp.async.bulk.  Two TMEM
// accumulators double-buffer the MMA against two epilogue warpgroups that alternate tiles, so every
// epilogue thread owns complete output rows -- LayerNorm needs no cross-thread reduction.
// 14 warps: 0-3 epilogue group 0, 4-7 epilogue group 1, 8-11 converters, 12 bulk-copy producer,
// 13 MMA issuer + TMEM allocator.
//   reference: nn.TransformerDecoderLayer as configured at model/influentialRS.py:67-74
//   (self_attn.in_proj / out_proj, linear1, linear2, norm1..3), model/uRS.py:42-44.
#include "tc_common.cuh"

namespace irs {
namespace tcg {

using namespace irs::tc;

constexpr int BM = 128;
constexpr int KC = 32;
constexpr int STAGES = 4;
constexpr int NMAX = 256;
constexpr int KMAX_G = 256;
constexpr int CONV_WARPS = 4;
constexpr int WARP_CONV0 = 8, WARP_PROD = 12, WARP_MMA = 13;
constexpr int THREADS = 14 * 32;
constexpr uint32_t A_STAGE_BYTES = 2u * (KC / 8) * BM * 16;           // hi + lo : 16384
constexpr uint32_t A_HALF = A_STAGE_BYTES / 2;
constexpr uint32_t A_LBO = BM * 16;
constexpr uint32_t SBO = 128;
constexpr uint32_t B_STAGE_MAX = 2u * (KC / 8) * NMAX * 16;           // 32768
constexpr uint32_t OFF_A = 0;
constexpr uint32_t OFF_B = STAGES * A_STAGE_BYTES;                    // 65536
constexpr uint32_t OFF_VEC = OFF_B + STAGES * B_STAGE_MAX;            // 196608 : bias, g1, b1, c2, g2, b2  [6][NMAX] floats
constexpr uint32_t OFF_BARS = OFF_VEC + 6 * NMAX * 4;                 // full[4], empty[4], tfull[2], tempty[2]
constexpr uint32_t OFF_TMEM = OFF_BARS + (2 * STAGES + 4) * 8;
constexpr uint32_t SMEM_BYTES = OFF_TMEM + 16;
constexpr uint32_t TMEM_COLS = 512;

enum Epilogue { EPI_BIAS = 0, EPI_BIAS_RELU = 1, EPI_RESID_LN = 2 };

struct Params {
  const float* A; int64_t lda;
  const uint4* Wt;                 // prepared weights [chunk][hi|lo][slab][n_pad][8 bf16]
  const float* bias;               // [Nout] or null
  const float* resid; int64_t ldr; // EPI_RESID_LN
  const float* g1; const float* b1; const float* c2; const float* g2; const float* b2; float eps;
  float* C; int64_t ldc;
  int64_t R; int K; int Nout; int n_pad; int n_chunks;
  int64_t n_tiles;
  int* error_flag;
};

// W [Nout, K] fp32 -> [chunk][part][slab][n_pad rows][8 bf16]  (zero padded)
__global__ void __launch_bounds__(256)
prepare_linear_kernel(const float* __restrict__ W, int Nout, int K, int n_pad, int n_chunks, uint4* __restrict__ out) {
  const int total = n_chunks * 4 * n_pad;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    const int r = idx % n_pad;
    const int s = (idx / n_pad) % 4;
    const int c = idx / (n_pad * 4);
    const int k0 = c * KC + s * 8;
    float x[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) x[e] = (r < Nout && k0 + e < K) ? W[(int64_t)r * K + k0 + e] : 0.f;
    uint4 hi, lo;
    split8(x, hi, lo);
    const int base = c * 2 * 4 * n_pad;
    out[base + s * n_pad + r] = hi;
    out[base + (4 + s) * n_pad + r] = lo;
  }
}

// Chan's parallel-variance merge: fold the statistics of nb more values (mean mb, sum of squared deviations qb) into the
// running (n, mean, m2) of a row.  Each 32-column chunk is centred on its own mean before it is squared, so the row
// statistics stay accurate when the mean is large next to the spread (E[t^2] - mean^2 would cancel).
__device__ __forceinline__ void chan_merge(float& n, float& mean, float& m2, float nb, float mb, float qb) {
  const float nn = n + nb;
  const float delta = mb - mean;
  const float w = nb / nn;
  mean = fmaf(delta, w, mean);
  m2 += qb + delta * delta * (n * w);
  n = nn;
}

template <int EPI>
__global__ void __launch_bounds__(THREADS, 1)
linear_tc_kernel(const Params p) {
  extern __shared__ __align__(128) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n_chunks = p.n_chunks;
  const uint32_t b_stage_bytes = 2u * (KC / 8) * (uint32_t)p.n_pad * 16u;
  const uint32_t b_half = b_stage_bytes / 2;
  const uint32_t b_lbo = (uint32_t)p.n_pad * 16u;
  const uint32_t idesc = make_idesc_bf16(BM, p.n_pad);

  auto bar_full = [&](int s) { return sbase + OFF_BARS + 8u * s; };
  auto bar_empty = [&](int s) { return sbase + OFF_BARS + 8u * (STAGES + s); };
  auto bar_tfull = [&](int a) { return sbase + OFF_BARS + 8u * (2 * STAGES + a); };
  auto bar_tempty = [&](int a) { return sbase + OFF_BARS + 8u * (2 * STAGES + 2 + a); };
  volatile uint32_t* tmem_holder = reinterpret_cast<volatile uint32_t*>(smem + OFF_TMEM);
  float* vecs = reinterpret_cast<float*>(smem + OFF_VEC);

  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(bar_full(s), 2); mbar_init(bar_empty(s), 1); }   // converter + bulk producer
    for (int a = 0; a < 2; ++a) { mbar_init(bar_tfull(a), 1); mbar_init(bar_tempty(a), 128); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == WARP_MMA) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 :: "r"(sbase + OFF_TMEM), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  // per-column vectors of the epilogue
  for (int i = tid; i < NMAX; i += THREADS) {
    const bool ok = i < p.Nout;
    vecs[0 * NMAX + i] = (ok && p.bias) ? p.bias[i] : 0.f;
    vecs[1 * NMAX + i] = (ok && p.g1) ? p.g1[i] : 0.f;
    vecs[2 * NMAX + i] = (ok && p.b1) ? p.b1[i] : 0.f;
    vecs[3 * NMAX + i] = (ok && p.c2) ? p.c2[i] : 0.f;
    vecs[4 * NMAX + i] = (ok && p.g2) ? p.g2[i] : 0.f;
    vecs[5 * NMAX + i] = (ok && p.b2) ? p.b2[i] : 0.f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;
  const int64_t first_tile = blockIdx.x;
  const int64_t tile_step = gridDim.x;

  if (warp >= WARP_CONV0 && warp < WARP_CONV0 + CONV_WARPS) {
    // ===== converters: warp cw owns global stage numbers g with g % 4 == cw (many loads in flight) =====
    const int cw = warp - WARP_CONV0;
    int64_t g = 0;                                        // global stage counter of this CTA
    for (int64_t tile = first_tile; tile < p.n_tiles; tile += tile_step) {
      const int64_t r0 = tile * BM;
      for (int c = 0; c < n_chunks; ++c, ++g) {
        if ((int)(g % CONV_WARPS) != cw) continue;
        const int stage = (int)(g % STAGES);
        const uint32_t phase = (uint32_t)((g / STAGES) & 1);
        mbar_wait(bar_empty(stage), phase ^ 1u, p.error_flag, 11);
        uint8_t* dst = smem + OFF_A + stage * A_STAGE_BYTES;
        // 128 rows x 32 floats.  lane -> (row = 8*group + lane%8, 8-float slab = lane/8): every lane reads one
        // full 32-byte sector, and each quarter-warp writes 128 contiguous bytes of a core-matrix column
        // (conflict-free 16-byte shared stores).
        const int slab = lane >> 3;
        const int k0 = c * KC + slab * 8;
#pragma unroll 1
        for (int pass = 0; pass < 4; ++pass) {
          float x[4][8];
#pragma unroll
          for (int rep = 0; rep < 4; ++rep) {               // all loads of the pass first (memory-level parallelism)
            const int row = (pass * 4 + rep) * 8 + (lane & 7);
            const int64_t r = r0 + row;
            if (r < p.R && k0 + 8 <= p.K) {
              const float4 v0 = *reinterpret_cast<const float4*>(p.A + r * p.lda + k0);
              const float4 v1 = *reinterpret_cast<const float4*>(p.A + r * p.lda + k0 + 4);
              x[rep][0] = v0.x; x[rep][1] = v0.y; x[rep][2] = v0.z; x[rep][3] = v0.w;
              x[rep][4] = v1.x; x[rep][5] = v1.y; x[rep][6] = v1.z; x[rep][7] = v1.w;
            } else {
#pragma unroll
              for (int e = 0; e < 8; ++e) x[rep][e] = (r < p.R && k0 + e < p.K) ? p.A[r * p.lda + k0 + e] : 0.f;
            }
          }
#pragma unroll
          for (int rep = 0; rep < 4; ++rep) {
            const int row = (pass * 4 + rep) * 8 + (lane & 7);
            uint4 hi, lo;
            split8(x[rep], hi, lo);
            *reinterpret_cast<uint4*>(dst + slab * A_LBO + row * 16) = hi;
            *reinterpret_cast<uint4*>(dst + A_HALF + slab * A_LBO + row * 16) = lo;
          }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_full(stage));
      }
    }
  } else if (warp == WARP_PROD) {
    // ===== weight chunks: one bulk copy per stage (the prepared matrix is tiny and L2 resident) =====
    if (lane == 0) {
      int64_t g = 0;
      for (int64_t tile = first_tile; tile < p.n_tiles; tile += tile_step) {
        for (int c = 0; c < n_chunks; ++c, ++g) {
          const int stage = (int)(g % STAGES);
          const uint32_t phase = (uint32_t)((g / STAGES) & 1);
          mbar_wait(bar_empty(stage), phase ^ 1u, p.error_flag, 12);
          mbar_arrive_expect_tx(bar_full(stage), b_stage_bytes);
          bulk_g2s(sbase + OFF_B + stage * B_STAGE_MAX, p.Wt + (int64_t)c * (b_stage_bytes / 16), b_stage_bytes, bar_full(stage));
        }
      }
    }
  } else if (warp == WARP_MMA) {
    if (lane == 0) {
      int64_t g = 0;
      int it = 0;
      for (int64_t tile = first_tile; tile < p.n_tiles; tile += tile_step, ++it) {
        const int ab = it & 1;
        const uint32_t acc_phase = (uint32_t)(it >> 1) & 1u;
        mbar_wait(bar_tempty(ab), acc_phase ^ 1u, p.error_flag, 13);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(ab * NMAX);
        for (int c = 0; c < n_chunks; ++c, ++g) {
          const int stage = (int)(g % STAGES);
          const uint32_t phase = (uint32_t)((g / STAGES) & 1);
          mbar_wait(bar_full(stage), phase, p.error_flag, 14);
          tc_fence_after();
          const uint32_t as = sbase + OFF_A + stage * A_STAGE_BYTES;
          const uint32_t bs = sbase + OFF_B + stage * B_STAGE_MAX;
#pragma unroll
          for (int kk = 0; kk < KC / 16; ++kk) {
            const uint64_t a_hi = make_desc(as + (uint32_t)(kk * 2) * A_LBO, A_LBO, SBO);
            const uint64_t a_lo = make_desc(as + A_HALF + (uint32_t)(kk * 2) * A_LBO, A_LBO, SBO);
            const uint64_t b_hi = make_desc(bs + (uint32_t)(kk * 2) * b_lbo, b_lbo, SBO);
            const uint64_t b_lo = make_desc(bs + b_half + (uint32_t)(kk * 2) * b_lbo, b_lbo, SBO);
            tc_mma_bf16(d_tmem, a_lo, b_hi, idesc, (c | kk) != 0 ? 1u : 0u);
            tc_mma_bf16(d_tmem, a_hi, b_lo, idesc, 1u);
            tc_mma_bf16(d_tmem, a_hi, b_hi, idesc, 1u);
          }
          tc_commit(bar_empty(stage));
        }
        tc_commit(bar_tfull(ab));
      }
    }
  } else if (warp < 8) {
    // ===== epilogue: group (warp/4) takes every other tile; thread <-> output row =====
    const int group = warp >> 2, quad = warp & 3;
    const int row = quad * 32 + lane;
    const float* bias_s = vecs;
    int it = 0;
    for (int64_t tile = first_tile; tile < p.n_tiles; tile += tile_step, ++it) {
      if ((it & 1) != group) continue;
      const int ab = it & 1;
      const uint32_t acc_phase = (uint32_t)(it >> 1) & 1u;
      const int64_t r = tile * BM + row;
      const bool row_ok = r < p.R;
      mbar_wait(bar_tfull(ab), acc_phase, p.error_flag, 15);
      tc_fence_after();
      const uint32_t tbase = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(ab * NMAX);
      const int n_ch = (p.Nout + 31) / 32;
      if (EPI != EPI_RESID_LN) {
        for (int ch = 0; ch < n_ch; ++ch) {
          uint32_t v[32];
          tc_ld32(tbase + ch * 32, v);
          tc_wait_ld();
          if (row_ok) {
            float* dst = p.C + r * p.ldc + ch * 32;
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              float4 o;
              o.x = __uint_as_float(v[j]) + bias_s[ch * 32 + j];
              o.y = __uint_as_float(v[j + 1]) + bias_s[ch * 32 + j + 1];
              o.z = __uint_as_float(v[j + 2]) + bias_s[ch * 32 + j + 2];
              o.w = __uint_as_float(v[j + 3]) + bias_s[ch * 32 + j + 3];
              if (EPI == EPI_BIAS_RELU) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
              if (ch * 32 + j + 4 <= p.Nout) *reinterpret_cast<float4*>(dst + j) = o;
              else {
                const float oo[4] = {o.x, o.y, o.z, o.w};
                for (int e = 0; e < 4; ++e) if (ch * 32 + j + e < p.Nout) dst[j + e] = oo[e];
              }
            }
          }
        }
      } else {
        // pass 1: t = resid + acc + bias, written back into the accumulator (TMEM as row scratch); mean and squared
        // deviations of each chunk, merged into the row's.  pass 2 (optional): the same statistics of LN1(t)+c2.
        // pass 3: normalise, store.
        const float inv_n = 1.0f / (float)p.Nout;
        const float* rsd = p.resid + (row_ok ? r : 0) * p.ldr;
        float n1 = 0.f, mean1 = 0.f, q1 = 0.f;
        for (int ch = 0; ch < n_ch; ++ch) {
          uint32_t v[32];
          tc_ld32(tbase + ch * 32, v);
          float rr[32];
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
            if (ch * 32 + j + 4 <= p.Nout) q = *reinterpret_cast<const float4*>(rsd + ch * 32 + j);
            else { float* qq = reinterpret_cast<float*>(&q); for (int e = 0; e < 4; ++e) if (ch * 32 + j + e < p.Nout) qq[e] = rsd[ch * 32 + j + e]; }
            rr[j] = q.x; rr[j + 1] = q.y; rr[j + 2] = q.z; rr[j + 3] = q.w;
          }
          tc_wait_ld();
          const int nc = min(32, p.Nout - ch * 32);
          float cs[4] = {0.f, 0.f, 0.f, 0.f}, cq[4] = {0.f, 0.f, 0.f, 0.f};     // four partial sums: short dependent chains
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int n = ch * 32 + j;
            float t = 0.f;
            if (n < p.Nout) { t = __uint_as_float(v[j]) + bias_s[n] + rr[j]; cs[j & 3] += t; }
            v[j] = __float_as_uint(t);
          }
          tc_st32(tbase + ch * 32, v);
          const float cm = ((cs[0] + cs[1]) + (cs[2] + cs[3])) / (float)nc;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float e = __uint_as_float(v[j]) - cm;
            if (ch * 32 + j < p.Nout) cq[j & 3] = fmaf(e, e, cq[j & 3]);
          }
          chan_merge(n1, mean1, q1, (float)nc, cm, (cq[0] + cq[1]) + (cq[2] + cq[3]));
        }
        tc_wait_st();
        const float rstd1 = rsqrtf(q1 * inv_n + p.eps);
        float mean2 = 0.f, rstd2 = 1.f;
        const bool two = (p.g2 != nullptr);
        if (two) {
          float n2 = 0.f, q2 = 0.f;
          for (int ch = 0; ch < n_ch; ++ch) {
            uint32_t v[32];
            tc_ld32(tbase + ch * 32, v);
            tc_wait_ld();
            const int nc = min(32, p.Nout - ch * 32);
            float y[32], cs[4] = {0.f, 0.f, 0.f, 0.f}, cq[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const int n = ch * 32 + j;
              y[j] = 0.f;
              if (n < p.Nout) {
                y[j] = (__uint_as_float(v[j]) - mean1) * rstd1 * vecs[1 * NMAX + n] + vecs[2 * NMAX + n] + vecs[3 * NMAX + n];
                cs[j & 3] += y[j];
              }
            }
            const float cm = ((cs[0] + cs[1]) + (cs[2] + cs[3])) / (float)nc;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const float e = y[j] - cm;
              if (ch * 32 + j < p.Nout) cq[j & 3] = fmaf(e, e, cq[j & 3]);
            }
            chan_merge(n2, mean2, q2, (float)nc, cm, (cq[0] + cq[1]) + (cq[2] + cq[3]));
          }
          rstd2 = rsqrtf(q2 * inv_n + p.eps);
        }
        for (int ch = 0; ch < n_ch; ++ch) {
          uint32_t v[32];
          tc_ld32(tbase + ch * 32, v);
          tc_wait_ld();
          if (row_ok) {
            float* dst = p.C + r * p.ldc + ch * 32;
            float y[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const int n = ch * 32 + j;
              float yy = 0.f;
              if (n < p.Nout) {
                yy = (__uint_as_float(v[j]) - mean1) * rstd1 * vecs[1 * NMAX + n] + vecs[2 * NMAX + n];
                if (two) yy = (yy + vecs[3 * NMAX + n] - mean2) * rstd2 * vecs[4 * NMAX + n] + vecs[5 * NMAX + n];
              }
              y[j] = yy;
            }
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              if (ch * 32 + j + 4 <= p.Nout) *reinterpret_cast<float4*>(dst + j) = make_float4(y[j], y[j + 1], y[j + 2], y[j + 3]);
              else for (int e = 0; e < 4; ++e) if (ch * 32 + j + e < p.Nout) dst[j + e] = y[j + e];
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive(bar_tempty(ab));
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == WARP_MMA) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

}  // namespace tcg
}  // namespace irs

using namespace irs;

static int pad16(int n) { return (n + 15) & ~15; }

extern "C" size_t irs_linear_prepared_bytes(int Nout, int K) {
  if (Nout <= 0 || K <= 0 || Nout > tcg::NMAX || K > tcg::KMAX_G) return 0;
  const int n_chunks = (K + tcg::KC - 1) / tcg::KC;
  return (size_t)n_chunks * 2 * 4 * pad16(Nout) * 16;
}

extern "C" int irs_linear_prepare_weights(const float* W, int Nout, int K, void* prepared, void* stream) {
  if (!W || !prepared || Nout <= 0 || K <= 0) return IRS_E_BADARG;
  if (Nout > tcg::NMAX || K > tcg::KMAX_G) return IRS_E_SHAPE;
  const int n_chunks = (K + tcg::KC - 1) / tcg::KC;
  tcg::prepare_linear_kernel<<<32, 256, 0, (cudaStream_t)stream>>>(W, Nout, K, pad16(Nout), n_chunks, (uint4*)prepared);
  IRS_LAUNCHED();
  return 0;
}

extern "C" int irs_linear_tc(const float* A, int64_t lda, const void* prepared, const float* bias, int epilogue,
                             const float* resid, int64_t ldr, const float* g1, const float* b1,
                             const float* c2, const float* g2, const float* b2, float eps,
                             float* C, int64_t ldc, int64_t R, int K, int Nout, int* error_flag, void* stream) {
  if (!A || !prepared || !C) return IRS_E_BADARG;
  if (R < 0 || K <= 0 || Nout <= 0) return IRS_E_BADARG;
  if (R == 0) return 0;
  if (Nout > tcg::NMAX || K > tcg::KMAX_G) return IRS_E_SHAPE;
  if ((lda & 3) || (K & 3) || ((uintptr_t)A & 15) || (ldc & 3) || ((uintptr_t)C & 15)) return IRS_E_SHAPE;
  if (epilogue < 0 || epilogue > 2) return IRS_E_BADARG;
  if (epilogue == tcg::EPI_RESID_LN && (!resid || !g1 || !b1 || (g2 && !b2))) return IRS_E_BADARG;
  // epilogue 2 reads resid rows with float4 loads
  if (epilogue == tcg::EPI_RESID_LN && ((ldr & 3) || ((uintptr_t)resid & 15))) return IRS_E_SHAPE;
  cudaStream_t s = (cudaStream_t)stream;
  tcg::Params p = {};
  p.A = A; p.lda = lda; p.Wt = (const uint4*)prepared; p.bias = bias; p.resid = resid; p.ldr = ldr;
  p.g1 = g1; p.b1 = b1; p.c2 = c2; p.g2 = g2; p.b2 = b2; p.eps = eps; p.C = C; p.ldc = ldc;
  p.R = R; p.K = K; p.Nout = Nout; p.n_pad = pad16(Nout); p.n_chunks = (K + tcg::KC - 1) / tcg::KC;
  p.n_tiles = ceil_div(R, tcg::BM);
  p.error_flag = error_flag;
  const unsigned grid = (unsigned)(p.n_tiles < kNumSMs ? p.n_tiles : kNumSMs);
  void (*const kernels[])(tcg::Params) = {tcg::linear_tc_kernel<0>, tcg::linear_tc_kernel<1>, tcg::linear_tc_kernel<2>};
  const auto kernel = kernels[epilogue];
  IRS_CUDA(opt_in_smem(kernel, tcg::SMEM_BYTES));
  kernel<<<grid, tcg::THREADS, tcg::SMEM_BYTES, s>>>(p);
  IRS_LAUNCHED();
  return 0;
}
