// K3, persistent edition: PIM / causal self-attention for full windows of 129..223 positions with 32-wide
// heads (the BASELINE cfg3/cfg5 shape: L = 201, dh = 32) on the 5th-generation tensor cores.
//
// Input is the q/k/v projection in "operand image" form (qkv_image.cuh): per (batch, head) item one
// contiguous 88 KB block that already is the shared-memory image the MMAs consume.  One persistent CTA
// per SM walks over items:
//   * staging an item is three cp.async.bulk copies issued by one thread into a double buffer -- no
//     conversion, no register traffic, and the next item streams in while the current one is computed;
//   * the probabilities never touch shared memory: P = exp2(s - max) is written back IN PLACE over the
//     scores in TMEM as packed bf16 pairs (hi in 16 columns, lo in the next 16 of every 32-key block) and
//     the P.V product reads its A operand from TMEM; V is consumed as an MN-major B operand, so it needs
//     no transpose and shares K's layout;
//   * the causal triangle is balanced: the window is cut into 32-row chunks and the two softmax
//     warpgroups (two M = 128 tiles in flight, 256 TMEM columns each) take chunks such that every SM
//     sub-partition sees about the same number of visible key blocks (long rows paired with short rows).
// Arithmetic is that of attention_tc.cu: scores in the log2 domain, three bf16 MMAs per product
// (lo*hi + hi*lo + hi*hi) with fp32 accumulation, softmax in fp32.
// Warps: 0-3 softmax group 0, 4-7 softmax group 1 (TMEM lane quadrant = warp % 4), 8 bulk-copy producer
// + key-bias vector, 9 MMA issuer.
//   reference: model/influentialRS.py:139-151,171,189-193; torch multi_head_attention_forward; model/uRS.py:47-61.
#include <cstdlib>
#include "tc_common.cuh"
#include "qkv_image.cuh"

namespace irs {
namespace tcp {

using namespace irs::tc;
using namespace irs::img;

constexpr int PB = 32;
constexpr int THREADS = 10 * 32;
constexpr int WARP_PROD = 8, WARP_MMA = 9;
constexpr uint32_t SBO = 128;
constexpr uint32_t OFF_KB = ITEM_BYTES;                                     // float [224] key bias
constexpr uint32_t OFF_KSTAT = OFF_KB + KEYS * 4;                           // float: bound on |score| over the whole item
constexpr uint32_t BUF_BYTES = ((OFF_KSTAT + 16 + 127) / 128) * 128;       // 91136
constexpr float NO_SHIFT_SAFE = 80.f;   // log2 units: with every |score| below this, exp2(s) of a row needs no max subtraction
                                        // (p in [2^-80, 2^80]: normal fp32 / bf16 numbers, sums far from overflow)
enum Bars { B_KV_FULL = 0, B_KV_FREE = 2, B_S = 4, B_P = 6, B_P2 = 8, B_O = 10, B_KB = 12, B_COUNT = 14 };
constexpr uint32_t OFF_BARS = 2 * BUF_BYTES;
constexpr uint32_t OFF_TMEM = OFF_BARS + B_COUNT * 8;
constexpr uint32_t SMEM_BYTES = OFF_TMEM + 16;
// TMEM columns: group 0 (the long rows) S/P [0, 224) + O [224, 288); group 1 (short rows: at most 3 chunks + the PIM
// objective column = 112 columns) S/P [288, 400) + O [416, 480).  O is 64 wide: columns 0-31 accumulate P_hi.V_hi +
// P_lo.V_hi, columns 32-63 P_hi.V_lo (see issue_pv); the epilogue adds the two halves.
__device__ __forceinline__ uint32_t g_base(int g) { return g ? 288u : 0u; }
__device__ __forceinline__ uint32_t o_col(int g) { return g ? 128u : 224u; }

struct Params {
  const uint8_t* images;           // [B*H] items of ITEM_BYTES
  const int64_t* ids; const float* r_u; float w_h, w_obj; int mode;
  float* out; int B, L, H; int n_items;
  int q_row;                       // -1: all rows -> out [B, L, H*32]; otherwise only this row -> out [B, 1, H*32]
  int* error_flag;
  float no_shift_safe;             // NO_SHIFT_SAFE, or a negative number to force the exact row-max pass (A/B measurements)
  long long* timeline;             // debug: [8 items][4 roles][16 events] clock64 stamps of CTA 0 (null in production)
};

#define IRS_ATL(role, idx)                                                                        \
  do {                                                                                            \
    if (p.timeline && blockIdx.x == 0 && it < 8 && lane == 0)                                     \
      p.timeline[(it * 4 + (role)) * 16 + (idx)] = clock64();                                     \
  } while (0)

__device__ __forceinline__ void stg256(float* p, const float* a) {
  asm volatile("st.global.L1::no_allocate.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               :: "l"(p), "f"(a[0]), "f"(a[1]), "f"(a[2]), "f"(a[3]), "f"(a[4]), "f"(a[5]), "f"(a[6]), "f"(a[7]) : "memory");
}
__device__ __forceinline__ float ex2_approx(float x) {      // MUFU.EX2, flush-to-zero: exp2(-inf) = 0, exp2(NaN) = NaN
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ bool mbar_test(uint32_t bar, uint32_t parity) {      // non-blocking phase test
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\t"
               "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
               "selp.u32 %0, 1, 0, p;\n\t}"
               : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok != 0;
}
// D[tmem] (+)= A[tmem] . B[smem] : A operand = packed bf16 pairs, lane = row, column = k / 2.
__device__ __forceinline__ void tc_mma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile("{\n\t.reg .pred p;\n\t"
               "setp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
               :: "r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}

__global__ void __launch_bounds__(THREADS, 1)
pim_attn_persistent_kernel(const Params p) {
  extern __shared__ __align__(128) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  auto bar = [&](int i) { return sbase + OFF_BARS + 8u * (uint32_t)i; };
  volatile uint32_t* tmem_holder = reinterpret_cast<volatile uint32_t*>(smem + OFF_TMEM);
  const int L = p.L, H = p.H;
  const bool pim = (p.mode == IRS_MASK_PIM);
  const int koff = pim ? 1 : 0;                      // column c <-> key c - koff; column 0 <-> key L-1 in PIM mode
  const int n_chunks = (L + 31) / 32;                // 5..7
  const float l2e = 1.4426950408889634f;
  // columns each group's tile can see, padded to the MMA N granularity
  const int rem = n_chunks - 4;
  const int tcols_g0 = L, tcols_g1 = min(32 * rem, L - koff) + koff;
  auto tcols_of = [&](int g) { return g == 0 ? tcols_g0 : tcols_g1; };
  auto tpad_of = [&](int g) { return (tcols_of(g) + 15) & ~15; };
  // P.V is issued in two stages per tile so that it overlaps the second half of the softmax
  auto nblk_of = [&](int g) { return (tpad_of(g) + PB - 1) / PB; };
  auto split_of = [&](int g) { return (nblk_of(g) + 1) / 2; };

  if (tid == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar(B_KV_FULL + i), 1); mbar_init(bar(B_KV_FREE + i), 1); mbar_init(bar(B_KB + i), 1);
      mbar_init(bar(B_S + i), 1); mbar_init(bar(B_P + i), 128); mbar_init(bar(B_P2 + i), 128); mbar_init(bar(B_O + i), 1);
    }
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
  const int first = blockIdx.x, step = gridDim.x;

  if (warp == WARP_PROD) {
    // ===== producer: item `it` -> buffer it & 1 (three bulk copies) + the key-bias vector of the item =====
    int it = 0;
    for (int item = first; item < p.n_items; item += step, ++it) {
      const int b = item / H;
      const int bufi = it & 1;
      mbar_wait(bar(B_KV_FREE + bufi), (uint32_t)(((it >> 1) & 1) ^ 1), p.error_flag, 51);
      IRS_ATL(3, 0);
      if (lane == 0) {
        const uint8_t* src = p.images + (int64_t)item * ITEM_BYTES;
        const uint32_t dst = sbase + (uint32_t)bufi * BUF_BYTES;
        mbar_arrive_expect_tx(bar(B_KV_FULL + bufi), ITEM_BYTES);
        bulk_g2s(dst + OFF_Q, src + OFF_Q, 2 * Q_PART, bar(B_KV_FULL + bufi));
        bulk_g2s(dst + OFF_K, src + OFF_K, 2 * K_PART, bar(B_KV_FULL + bufi));
        bulk_g2s(dst + OFF_V, src + OFF_V, 2 * K_PART, bar(B_KV_FULL + bufi));
      }
      // per-column additive term of every row that can see the column: l2e * (mask weight + key padding)
      float* kb = reinterpret_cast<float*>(smem + bufi * BUF_BYTES + OFF_KB);
      const float obj = pim ? p.w_obj * p.r_u[b] : 0.f;
      int64_t idv[KEYS / 32];
#pragma unroll
      for (int j = 0; j < KEYS / 32; ++j) {                       // all loads first: one memory round trip
        const int c = lane + 32 * j;
        const int key = (pim && c == 0) ? L - 1 : c - koff;
        idv[j] = (c < L && p.mode != IRS_MASK_CAUSAL) ? p.ids[(int64_t)b * L + key] : 1;
      }
      float babs = -1.f;
#pragma unroll
      for (int j = 0; j < KEYS / 32; ++j) {
        const int c = lane + 32 * j;
        float bias = -INFINITY;                                   // padded columns never contribute
        if (c < L && idv[j] != 0) {
          bias = l2e * ((pim && c == 0) ? obj : (pim ? p.w_h : 0.f));
          babs = fmaxf(babs, fabsf(bias));
        }
        kb[c] = bias;
      }
      // Row-max shortcut of the softmax warps: |s_ij| <= max_i|q_i| max_j|k_j| + max|bias| (Cauchy-Schwarz); when that is
      // small the softmax of this item needs no shift at all (no pass over S for the row maxima).  The norms come from
      // the landed images (hi halves; the bound carries a 2 % margin for the lo halves and rounding).
      mbar_wait(bar(B_KV_FULL + bufi), (uint32_t)((it >> 1) & 1), p.error_flag, 58);
      auto max_norm2 = [&](const uint8_t* img, uint32_t lbo, int n_rows) {       // rows 16 B apart, slabs `lbo` apart
        float best = 0.f;
        for (int r = lane; r < n_rows; r += 32) {
          float a[SLABS];
#pragma unroll
          for (int sl = 0; sl < SLABS; ++sl) {
            const uint4 w = *reinterpret_cast<const uint4*>(img + sl * lbo + r * 16);
            const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
            float acc = 0.f;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float a0 = __uint_as_float(ww[e] << 16), a1 = __uint_as_float(ww[e] & 0xffff0000u);
              acc = fmaf(a0, a0, acc); acc = fmaf(a1, a1, acc);
            }
            a[sl] = acc;
          }
          best = fmaxf(best, (a[0] + a[1]) + (a[2] + a[3]));
        }
        return best;
      };
      const uint8_t* ib = smem + bufi * BUF_BYTES;
      float k2 = max_norm2(ib + OFF_K, K_LBO, KEYS);
      float q2 = fmaxf(max_norm2(ib + OFF_Q, Q_LBO, BM), max_norm2(ib + OFF_Q + Q_TILE, Q_LBO, BM));
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        k2 = fmaxf(k2, __shfl_xor_sync(0xffffffffu, k2, o));
        q2 = fmaxf(q2, __shfl_xor_sync(0xffffffffu, q2, o));
        babs = fmaxf(babs, __shfl_xor_sync(0xffffffffu, babs, o));
      }
      if (lane == 0) {
        float* ks = reinterpret_cast<float*>(smem + bufi * BUF_BYTES + OFF_KSTAT);
        // every key padded (no finite bias): +inf -> the exact pass runs and the rows come out NaN, as in torch
        ks[0] = babs >= 0.f ? 1.02f * sqrtf(q2 * k2) + babs : INFINITY;
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(bar(B_KB + bufi));
      IRS_ATL(3, 1);
    }
  } else if (warp == WARP_MMA) {
    if (lane == 0) {
      const uint32_t idesc_o = make_idesc_bf16(BM, DH) | (1u << 16);       // B operand (V) is MN-major
      const uint32_t idesc_o64 = make_idesc_bf16(BM, 2 * DH) | (1u << 16);
      auto issue_qk = [&](int g, int bufi) {
        const uint32_t bb = sbase + (uint32_t)bufi * BUF_BYTES;
        const uint32_t idesc_s = make_idesc_bf16(BM, tpad_of(g));
        const uint32_t d = tmem_base + g_base(g);
#pragma unroll
        for (int kk = 0; kk < DH / 16; ++kk) {
          const uint64_t q_hi = make_desc(bb + OFF_Q + (uint32_t)g * Q_TILE + (uint32_t)(kk * 2) * Q_LBO, Q_LBO, SBO);
          const uint64_t q_lo = make_desc(bb + OFF_Q + Q_PART + (uint32_t)g * Q_TILE + (uint32_t)(kk * 2) * Q_LBO, Q_LBO, SBO);
          const uint64_t k_hi = make_desc(bb + OFF_K + (uint32_t)(kk * 2) * K_LBO, K_LBO, SBO);
          const uint64_t k_lo = make_desc(bb + OFF_K + K_PART + (uint32_t)(kk * 2) * K_LBO, K_LBO, SBO);
          tc_mma_bf16(d, q_lo, k_hi, idesc_s, kk != 0 ? 1u : 0u);
          tc_mma_bf16(d, q_hi, k_lo, idesc_s, 1u);
          tc_mma_bf16(d, q_hi, k_hi, idesc_s, 1u);
        }
        tc_commit(bar(B_S + g));
      };
      auto issue_pv = [&](int g, int bufi, int blk0, int blk1) {
        const uint32_t bb = sbase + (uint32_t)bufi * BUF_BYTES;
        const uint32_t ts = tmem_base + g_base(g);
        const uint32_t to = ts + o_col(g);
        for (int blk = blk0; blk < blk1; ++blk) {
#pragma unroll
          for (int kk = 0; kk < PB / 16; ++kk) {
            const uint32_t a_hi = ts + (uint32_t)(blk * PB + kk * 8), a_lo = a_hi + 16u;
            // MN-major V: 16 keys x 32 head dims; keys 16 B apart (8-key groups 128 B apart: leading offset),
            // 8-wide head-dim slabs K_LBO apart (stride offset)
            const uint32_t vo = (uint32_t)(blk * PB + kk * 16) * 16u;
            // The lo half of V follows the hi half at the same slab stride (K_PART = 4 K_LBO), so ONE N = 64 MMA computes
            // P_hi.[V_hi | V_lo] into 64 columns.  With the A operand in tensor memory an MMA costs its A read (4 KB at
            // 64 B/clk) whatever N is: two MMAs per k-step instead of three is a third off the P.V time.
            const uint64_t v_hi = make_desc(bb + OFF_V + vo, 128u, K_LBO);
            tc_mma_bf16_ts(to, a_hi, v_hi, idesc_o64, (blk | kk) != 0 ? 1u : 0u);
            tc_mma_bf16_ts(to, a_lo, v_hi, idesc_o, 1u);
          }
        }
      };
      int it = 0;
      if (first < p.n_items) {
        mbar_wait(bar(B_KV_FULL + 0), 0u, p.error_flag, 52);
        tc_fence_after();
        issue_qk(0, 0);
        issue_qk(1, 0);
      }
      for (int item = first; item < p.n_items; item += step, ++it) {
        const int bufi = it & 1;
        const bool has_next = item + step < p.n_items;
        const uint32_t ph = (uint32_t)(it & 1);
        // event driven: serve whichever group is ready (0: first half of P.V, 1: second half, 2: S of the next item, 3: done)
        int state[2] = {0, 0};
        bool next_ready = false;
        const long long t0 = clock64();
        while (state[0] < 3 || state[1] < 3) {
#pragma unroll
          for (int g = 0; g < 2; ++g) {
            if (state[g] == 0 && mbar_test(bar(B_P + g), ph)) {               // (also: O of the previous item has been read)
              tc_fence_after();
              IRS_ATL(2, 1 + 5 * g);
              issue_pv(g, bufi, 0, split_of(g));
              state[g] = 1;
            } else if (state[g] == 1 && mbar_test(bar(B_P2 + g), ph)) {
              tc_fence_after();
              IRS_ATL(2, 2 + 5 * g);
              issue_pv(g, bufi, split_of(g), nblk_of(g));
              tc_commit(bar(B_O + g));
              state[g] = has_next ? 2 : 3;
            } else if (state[g] == 2 && (next_ready || mbar_test(bar(B_KV_FULL + (bufi ^ 1)), (uint32_t)(((it + 1) >> 1) & 1)))) {
              if (!next_ready) { tc_fence_after(); next_ready = true; }
              issue_qk(g, bufi ^ 1);                                         // S of the next item: runs behind this P.V in the pipe
              IRS_ATL(2, 4 + 5 * g);
              state[g] = 3;
            }
          }
          if (clock64() - t0 > 4000000000ll) {                                // protocol watchdog (see mbar_wait)
            if (p.error_flag) atomicExch(p.error_flag, 53);
            __threadfence_system();
            __trap();
          }
        }
        tc_commit(bar(B_KV_FREE + bufi));
      }
    }
  } else if (warp < 8) {
    // ===== softmax warps: thread <-> query row =====
    const int g = warp >> 2, quad = warp & 3;
    const int chunk = chunk_of(n_chunks, g, quad);
    const bool active = chunk >= 0;
    const int split = split_of(g);
    const int r_lo = chunk * 32;
    const int i = r_lo + lane;
    const int tcols = tcols_of(g), tcols_pad = tpad_of(g);
    const int nblk = (tcols_pad + PB - 1) / PB;
    const int vis_last = min(r_lo + 31 + koff, tcols - 1);         // last column any row of the warp sees
    const int nb_warp = vis_last / PB + 1;                         // blocks this warp must evaluate
    const int n_full = (r_lo + koff + 1) / PB;                     // blocks [0, n_full) are visible to every row
    const int my_last = i + koff;                                  // last visible column of this row
    const uint32_t trow = tmem_base + (((uint32_t)(quad * 32)) << 16) + g_base(g);
    const bool tl = (quad == (g == 0 ? 1 : 0));
    int it = 0;
    for (int item = first; item < p.n_items; item += step, ++it) {
      const int b = item / H, h = item % H;
      const float* kb = reinterpret_cast<const float*>(smem + (it & 1) * BUF_BYTES + OFF_KB);
      if (tl) IRS_ATL(g, 0);
      mbar_wait(bar(B_S + g), (uint32_t)(it & 1), p.error_flag, 55);
      tc_fence_after();
      if (tl) IRS_ATL(g, 1);
      float sum = 0.f;
      if (active) {
        mbar_wait(bar(B_KB + (it & 1)), (uint32_t)((it >> 1) & 1), p.error_flag, 57);      // key-bias vector of this item
        float mx = -INFINITY;
        // no pass over S for the row maxima when every score of the item is provably small (producer warp):
        // |s_ij| <= 1.02 max|q_i| max|k_j| + max|bias| <= NO_SHIFT_SAFE  ->  p = exp2(s) as it is (shift 0)
        const bool bound_ok = *reinterpret_cast<const float*>(smem + (it & 1) * BUF_BYTES + OFF_KSTAT) <= p.no_shift_safe;
        if (bound_ok) mx = 0.f;
        auto block_max = [&](const uint32_t (&v)[32], int blk) {
          const float4* cw4 = reinterpret_cast<const float4*>(kb + blk * PB);
          float m0 = -INFINITY, m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;
          if (blk < n_full) {
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) {
              const float4 w = cw4[j4];
              m0 = fmaxf(m0, __uint_as_float(v[4 * j4 + 0]) + w.x); m1 = fmaxf(m1, __uint_as_float(v[4 * j4 + 1]) + w.y);
              m2 = fmaxf(m2, __uint_as_float(v[4 * j4 + 2]) + w.z); m3 = fmaxf(m3, __uint_as_float(v[4 * j4 + 3]) + w.w);
            }
          } else {
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) {
              const float4 w = cw4[j4];
              const int c = blk * PB + 4 * j4;
              const bool firstc = pim && c == 0;                  // the objective column is visible to every row
              if (c + 0 <= my_last || firstc) m0 = fmaxf(m0, __uint_as_float(v[4 * j4 + 0]) + w.x);
              if (c + 1 <= my_last) m1 = fmaxf(m1, __uint_as_float(v[4 * j4 + 1]) + w.y);
              if (c + 2 <= my_last) m2 = fmaxf(m2, __uint_as_float(v[4 * j4 + 2]) + w.z);
              if (c + 3 <= my_last) m3 = fmaxf(m3, __uint_as_float(v[4 * j4 + 3]) + w.w);
            }
          }
          mx = fmaxf(mx, fmaxf(fmaxf(m0, m1), fmaxf(m2, m3)));
        };
        auto block_exp = [&](const uint32_t (&v)[32], int blk) {
          uint32_t pk[32];
          const float4* cw4 = reinterpret_cast<const float4*>(kb + blk * PB);
          const bool full = blk < n_full;
#pragma unroll
          for (int s8 = 0; s8 < PB / 8; ++s8) {
            float x[8];
#pragma unroll
            for (int hq = 0; hq < 2; ++hq) {
              const float4 w = cw4[s8 * 2 + hq];
              const int c = blk * PB + s8 * 8 + hq * 4;
              const float ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                // fully masked row: -inf - -inf = NaN, as torch's softmax
                float pv = ex2_approx(__uint_as_float(v[s8 * 8 + hq * 4 + e]) + ww[e] - mx);
                if (!full && !(c + e <= my_last || (pim && c + e == 0))) pv = 0.f;
                x[hq * 4 + e] = pv;
                sum += pv;
              }
            }
            uint4 hi, lo;
            split8(x, hi, lo);
            pk[s8 * 4 + 0] = hi.x; pk[s8 * 4 + 1] = hi.y; pk[s8 * 4 + 2] = hi.z; pk[s8 * 4 + 3] = hi.w;
            pk[16 + s8 * 4 + 0] = lo.x; pk[16 + s8 * 4 + 1] = lo.y; pk[16 + s8 * 4 + 2] = lo.z; pk[16 + s8 * 4 + 3] = lo.w;
          }
          tc_st32(trow + blk * PB, pk);              // P over S, in place: [hi: 16 columns | lo: 16 columns]
        };
        // both passes keep one TMEM load in flight behind the arithmetic (two register buffers)
        if (!bound_ok) {
          uint32_t va[32], vb[32];
          tc_ld32(trow, va);
          for (int blk = 0; blk < nb_warp; blk += 2) {
            tc_wait_ld();
            if (blk + 1 < nb_warp) tc_ld32(trow + (blk + 1) * PB, vb);
            block_max(va, blk);
            if (blk + 1 < nb_warp) {
              tc_wait_ld();
              if (blk + 2 < nb_warp) tc_ld32(trow + (blk + 2) * PB, va);
              block_max(vb, blk + 1);
            }
          }
        }
        if (tl) IRS_ATL(g, 2);
        bool stage1 = false;
        auto after_block = [&](int blk) {            // first half of P complete: let its P.V start
          if (blk + 1 == split) {
            tc_wait_st();
            tc_fence_before();
            mbar_arrive(bar(B_P + g));
            stage1 = true;
          }
        };
        {
          uint32_t va[32], vb[32];
          tc_ld32(trow, va);
          for (int blk = 0; blk < nb_warp; blk += 2) {
            tc_wait_ld();
            if (blk + 1 < nb_warp) tc_ld32(trow + (blk + 1) * PB, vb);
            block_exp(va, blk);
            after_block(blk);
            if (blk + 1 < nb_warp) {
              tc_wait_ld();
              if (blk + 2 < nb_warp) tc_ld32(trow + (blk + 2) * PB, va);
              block_exp(vb, blk + 1);
              after_block(blk + 1);
            }
          }
          uint32_t z[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) z[j] = 0u;
          for (int blk = nb_warp; blk < nblk; ++blk) { tc_st32(trow + blk * PB, z); after_block(blk); }
        }
        tc_wait_st();
        if (!stage1) { tc_fence_before(); mbar_arrive(bar(B_P + g)); }
      } else {
        mbar_arrive(bar(B_P + g));
      }
      tc_fence_before();
      mbar_arrive(bar(B_P2 + g));
      if (tl) IRS_ATL(g, 3);
      mbar_wait(bar(B_O + g), (uint32_t)(it & 1), p.error_flag, 56);
      tc_fence_after();
      if (tl) IRS_ATL(g, 4);
      if (active) {
        uint32_t v[32], v2[32];
        tc_ld32(trow + o_col(g), v);
        tc_ld32(trow + o_col(g) + 32u, v2);
        tc_wait_ld();
        if (i < L) {
          const float inv = 1.0f / sum;
          float o[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) o[j] = (__uint_as_float(v[j]) + __uint_as_float(v2[j])) * inv;
          float* dst = p.out + ((int64_t)b * L + i) * (H * DH) + h * DH;
#pragma unroll
          for (int q = 0; q < 4; ++q) stg256(dst + q * 8, &o[q * 8]);
        }
      }
      if (tl) IRS_ATL(g, 5);
      tc_fence_before();
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == WARP_MMA) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(512u) : "memory");
  }
}


// One query row per (batch, head) -- what generation reads from the last decoder layer.  A single row
// cannot fill an M = 128 MMA tile, and the work per item (2 x 201 x 32 MACs) is tiny next to streaming the
// item's K and V images (56 KB), so this is a bandwidth kernel on the CUDA cores: one warp per item, lane <->
// key column, every load a coalesced 512-byte run of 16-byte core-matrix rows straight from HBM
// (hi + lo gives back the fp32 value to 2^-17).  Scores stay in the log2 domain like the tensor-core path.
__global__ void __launch_bounds__(256)
pim_attn_row_kernel(const Params p) {
  const int lane = threadIdx.x & 31;
  const int warps_per_cta = blockDim.x >> 5;
  const int L = p.L, H = p.H;
  const bool pim = (p.mode == IRS_MASK_PIM);
  const int koff = pim ? 1 : 0;
  const int n_chunks = (L + 31) / 32;
  const float l2e = 1.4426950408889634f;
  const int slot = q_slot(n_chunks, p.q_row);
  const int my_last = p.q_row + koff;                       // last visible key column of the row
  auto bf2f = [](uint32_t w, float& a, float& b) { a = __uint_as_float(w << 16); b = __uint_as_float(w & 0xffff0000u); };
  auto unpack8 = [&](const uint4& hi, const uint4& lo, float (&x)[8]) {
    const uint32_t hw[4] = {hi.x, hi.y, hi.z, hi.w}, lw[4] = {lo.x, lo.y, lo.z, lo.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float h0, h1, l0, l1;
      bf2f(hw[e], h0, h1); bf2f(lw[e], l0, l1);
      x[2 * e] = h0 + l0; x[2 * e + 1] = h1 + l1;
    }
  };
  for (int item = blockIdx.x * warps_per_cta + (threadIdx.x >> 5); item < p.n_items; item += gridDim.x * warps_per_cta) {
    const int b = item / H, h = item % H;
    const uint8_t* blk = p.images + (int64_t)item * ITEM_BYTES;
    // the query row (already scaled by log2(e)/sqrt(dh)), replicated in every lane
    float q[DH];
    {
      const uint8_t* qp = blk + OFF_Q + (slot / BM) * Q_TILE + (slot % BM) * 16;
#pragma unroll
      for (int s = 0; s < SLABS; ++s) {
        const uint4 hi = __ldg(reinterpret_cast<const uint4*>(qp + s * Q_LBO));
        const uint4 lo = __ldg(reinterpret_cast<const uint4*>(qp + Q_PART + s * Q_LBO));
        unpack8(hi, lo, *reinterpret_cast<float(*)[8]>(&q[s * 8]));
      }
    }
    const float obj = pim ? p.w_obj * p.r_u[b] : 0.f;
    // scores of this lane's columns (c = lane + 32 j)
    float sc[KEYS / 32];
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < KEYS / 32; ++j) {
      const int c = lane + 32 * j;
      float s_ = -INFINITY;
      const bool vis = c < L && (c <= my_last || (pim && c == 0));
      if (vis) {
        const int key = (pim && c == 0) ? L - 1 : c - koff;
        const bool pad = (p.mode != IRS_MASK_CAUSAL && p.ids[(int64_t)b * L + key] == 0);
        if (!pad) {
          float acc = 0.f;
#pragma unroll
          for (int s = 0; s < SLABS; ++s) {
            const uint4 hi = __ldg(reinterpret_cast<const uint4*>(blk + OFF_K + s * K_LBO + c * 16));
            const uint4 lo = __ldg(reinterpret_cast<const uint4*>(blk + OFF_K + K_PART + s * K_LBO + c * 16));
            float kx[8];
            unpack8(hi, lo, kx);
#pragma unroll
            for (int e = 0; e < 8; ++e) acc = fmaf(q[s * 8 + e], kx[e], acc);
          }
          s_ = acc + l2e * ((pim && c == 0) ? obj : (pim ? p.w_h : 0.f));
        }
      }
      sc[j] = s_;
      mx = fmaxf(mx, s_);
    }
    mx = warp_max(mx);
    float o[DH];
#pragma unroll
    for (int e = 0; e < DH; ++e) o[e] = 0.f;
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < KEYS / 32; ++j) {
      const int c = lane + 32 * j;
      const float pv = exp2f(sc[j] - mx);                  // fully masked row: -inf - -inf = NaN, as torch's softmax
      if (sc[j] != -INFINITY || mx == -INFINITY) {
        sum += pv;
        if (c < L) {
#pragma unroll
          for (int s = 0; s < SLABS; ++s) {
            const uint4 hi = __ldg(reinterpret_cast<const uint4*>(blk + OFF_V + s * K_LBO + c * 16));
            const uint4 lo = __ldg(reinterpret_cast<const uint4*>(blk + OFF_V + K_PART + s * K_LBO + c * 16));
            float vx[8];
            unpack8(hi, lo, vx);
#pragma unroll
            for (int e = 0; e < 8; ++e) o[s * 8 + e] = fmaf(pv, vx[e], o[s * 8 + e]);
          }
        }
      }
    }
    sum = warp_sum(sum);
    // 32 lane-partial output vectors -> lane e holds o[e]: transpose-reduce in 5 halving steps
    float mine = 0.f;
#pragma unroll
    for (int e = 0; e < DH; ++e) {
      const float t = warp_sum(o[e]);
      if (lane == e) mine = t;
    }
    p.out[(int64_t)b * (H * DH) + h * DH + lane] = mine / sum;
  }
}

// fp32 packed projection [B*L, 3*H*32] (nn.MultiheadAttention in_proj layout) -> operand images.
// One thread per (token, head, q|k|v): 32 floats in, 4 x (hi, lo) 16-byte pieces out.
__global__ void __launch_bounds__(256)
qkv_to_images_kernel(const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
                     int64_t ld_q, int64_t ld_k, int64_t ld_v, uint8_t* __restrict__ images, int B, int L, int H, int mode) {
  const int64_t total = (int64_t)B * L * H * 3;
  const bool pim = (mode == IRS_MASK_PIM);
  const int n_chunks = (L + 31) / 32;
  const float qscale = 1.4426950408889634f / sqrtf((float)DH);
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    // consecutive threads = consecutive tokens: a warp writes 512 contiguous bytes per piece
    const int l = (int)(idx % L);
    const int64_t rest = idx / L;
    const int which = (int)(rest % 3);
    const int h = (int)((rest / 3) % H);
    const int b = (int)(rest / (3 * H));
    const float* src = (which == 0 ? q + ((int64_t)b * L + l) * ld_q : which == 1 ? k + ((int64_t)b * L + l) * ld_k
                                                                                  : v + ((int64_t)b * L + l) * ld_v) + h * DH;
    uint8_t* blk = images + ((int64_t)b * H + h) * ITEM_BYTES;
    uint8_t* dst; uint32_t part, lbo;
    if (which == 0) { const int s = q_slot(n_chunks, l); dst = blk + OFF_Q + (s / BM) * Q_TILE + (s % BM) * 16; part = Q_PART; lbo = Q_LBO; }
    else { dst = blk + (which == 1 ? OFF_K : OFF_V) + kv_col(pim, L, l) * 16; part = K_PART; lbo = K_LBO; }
#pragma unroll
    for (int s = 0; s < SLABS; ++s) {
      float x[8];
      const float4 a = *reinterpret_cast<const float4*>(src + s * 8), c = *reinterpret_cast<const float4*>(src + s * 8 + 4);
      x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = c.x; x[5] = c.y; x[6] = c.z; x[7] = c.w;
      if (which == 0) {
#pragma unroll
        for (int e = 0; e < 8; ++e) x[e] *= qscale;
      }
      uint4 hi, lo;
      split8(x, hi, lo);
      *reinterpret_cast<uint4*>(dst + s * lbo) = hi;
      *reinterpret_cast<uint4*>(dst + part + s * lbo) = lo;
    }
  }
}

}  // namespace tcp
}  // namespace irs

using namespace irs;

static long long* g_attn_timeline = nullptr;
/* debug hook (not in the public header): device buffer of 8*4*16 int64 */
extern "C" void irs_pim_attn_debug_timeline(long long* buf) { g_attn_timeline = buf; }

extern "C" int irs_pim_attn_img_supported(int L, int dh) { return (dh == img::DH && L > 128 && L <= img::KEYS - 1) ? 1 : 0; }

extern "C" size_t irs_qkv_images_bytes(int B, int L, int H, int dh) {
  if (!irs_pim_attn_img_supported(L, dh) || B <= 0 || H <= 0) return 0;
  return (size_t)B * H * img::ITEM_BYTES;
}

extern "C" int irs_qkv_to_images(const float* q, const float* k, const float* v, int64_t ld_q, int64_t ld_k, int64_t ld_v,
                                 void* images, int B, int L, int H, int dh, int mode, void* stream) {
  if (!q || !k || !v || !images || B <= 0 || H <= 0) return IRS_E_BADARG;
  if (mode < 0 || mode > 2) return IRS_E_BADARG;
  if (!irs_pim_attn_img_supported(L, dh)) return IRS_E_SHAPE;
  if ((ld_q & 3) || (ld_k & 3) || (ld_v & 3) || ((uintptr_t)q & 15) || ((uintptr_t)k & 15) || ((uintptr_t)v & 15) || ((uintptr_t)images & 15))
    return IRS_E_SHAPE;
  const int64_t total = (int64_t)B * L * H * 3;
  const unsigned grid = (unsigned)(ceil_div(total, 256) < 148 * 16 ? ceil_div(total, 256) : 148 * 16);
  tcp::qkv_to_images_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(q, k, v, ld_q, ld_k, ld_v, (uint8_t*)images, B, L, H, mode);
  IRS_LAUNCHED();
  return 0;
}

extern "C" int irs_pim_attn_fwd_img(const void* images, const int64_t* ids, const float* r_u, float w_h, float w_obj, int mode,
                                    float* out, int B, int L, int H, int dh, int q_row0, int n_q,
                                    int* error_flag, void* stream) {
  if (!images || !out) return IRS_E_BADARG;
  if (B <= 0 || L <= 0 || H <= 0 || q_row0 < 0 || n_q <= 0 || q_row0 + n_q > L) return IRS_E_BADARG;
  if (mode < 0 || mode > 2) return IRS_E_BADARG;
  if (mode != IRS_MASK_CAUSAL && !ids) return IRS_E_BADARG;
  if (mode == IRS_MASK_PIM && !r_u) return IRS_E_BADARG;
  if (!irs_pim_attn_img_supported(L, dh)) return IRS_E_SHAPE;
  if (!(n_q == L || n_q == 1)) return IRS_E_SHAPE;             // all rows, or exactly one
  if (((uintptr_t)images & 15) || ((uintptr_t)out & 31)) return IRS_E_SHAPE;
  tcp::Params p = {};
  p.images = (const uint8_t*)images; p.ids = ids; p.r_u = r_u; p.w_h = w_h; p.w_obj = w_obj; p.mode = mode;
  p.out = out; p.B = B; p.L = L; p.H = H; p.n_items = B * H; p.q_row = (n_q == L) ? -1 : q_row0;
  p.error_flag = error_flag;
  p.timeline = g_attn_timeline;
  { static int force = -1; if (force < 0) { const char* e = getenv("IRS_ATTN_EXACT_MAX"); force = (e && atoi(e)) ? 1 : 0; }
    p.no_shift_safe = force ? -1.f : tcp::NO_SHIFT_SAFE; }
  if (p.q_row >= 0) {
    const int64_t ctas = ceil_div(p.n_items, 8);
    tcp::pim_attn_row_kernel<<<(unsigned)(ctas < kNumSMs * 8 ? ctas : kNumSMs * 8), 256, 0, (cudaStream_t)stream>>>(p);
    IRS_LAUNCHED();
    return 0;
  }
  const unsigned grid = (unsigned)(p.n_items < kNumSMs ? p.n_items : kNumSMs);
  IRS_CUDA(opt_in_smem(tcp::pim_attn_persistent_kernel, tcp::SMEM_BYTES));
  tcp::pim_attn_persistent_kernel<<<grid, tcp::THREADS, tcp::SMEM_BYTES, (cudaStream_t)stream>>>(p);
  IRS_LAUNCHED();
  return 0;
}
