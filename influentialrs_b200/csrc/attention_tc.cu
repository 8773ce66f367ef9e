// K3 on the 5th-generation tensor cores: PIM / causal self-attention for head sizes that are
// multiples of 16 and windows of up to 223 positions (every BASELINE config: dh = 32, L <= 201).
//
// One CTA owns one (batch, head).  K and V^T of the head are staged once into shared memory as bf16
// hi/lo K-major "core matrix" images; the query rows are processed in tiles of 128 (UMMA M = 128,
// TMEM lane = query row, one softmax thread per row):
//     S = Q K^T          6 tcgen05.mma (bf16 hi/lo split: lo*hi + hi*lo + hi*hi), fp32 accumulators in TMEM
//     pass 1             row max of  S/sqrt(dh) + mask  (mask built in registers from (row, key, r_u, pad))
//     pass 2             P = exp(s - max) in 32-key blocks -> bf16 hi/lo A-operand image in shared memory,
//                        double buffered;  O += P V  (6 tcgen05.mma per block) overlaps the next block
//     epilogue           O / rowsum -> global
// Causality is used per tile (tile t only multiplies the keys it can see).  In PIM mode the objective
// key L-1, which EVERY row sees (model/influentialRS.py:149), is moved to column 0 so that it is
// inside every tile's key range.  ~104 KB of shared memory and 256 TMEM columns per CTA, so two CTAs
// share an SM: while one stages the next head's K/V the other computes.
// The fp32 CUDA-core kernel in attention.cu remains the path for other shapes and for the backward.
//   reference: model/influentialRS.py:139-151,171,189-193; torch multi_head_attention_forward;
//   model/uRS.py:47-61; model/sas.py:168-177.
#include "tc_common.cuh"

namespace irs {
namespace tca {

using namespace irs::tc;

constexpr int BM = 128;
constexpr int KEYS_MAX = 224;        // padded key columns (L <= 223)
constexpr int PB = 32;               // keys per P block
constexpr int THREADS = 160;         // warps 0-3 softmax (TMEM lane quadrant = warp), warp 4 MMA + restaging
constexpr uint32_t SBO = 128;
constexpr uint32_t TMEM_COLS = 256;
constexpr uint32_t O_COL = 224;

struct Layout {
  uint32_t off_k_hi, off_k_lo, off_v_hi, off_v_lo, off_q_hi, off_q_lo, off_p, p_buf_bytes, off_kb, off_bars, off_tmem, total;
};
__host__ __device__ inline Layout make_layout(int dh) {
  Layout l;
  const uint32_t kbytes = (uint32_t)KEYS_MAX * dh * 2;            // one part of K ( [dh/8][224][8] bf16 )
  const uint32_t qbytes = (uint32_t)BM * dh * 2;
  l.off_k_hi = 0; l.off_k_lo = kbytes;
  l.off_v_hi = 2 * kbytes; l.off_v_lo = 3 * kbytes;             // V^T : [224/8][dh][8]
  l.off_q_hi = 4 * kbytes; l.off_q_lo = 4 * kbytes + qbytes;
  l.off_p = 4 * kbytes + 2 * qbytes;
  l.p_buf_bytes = 2u * (PB / 8) * BM * 16;                       // hi + lo : 16384
  l.off_kb = l.off_p + 2 * l.p_buf_bytes;                        // float [224] key bias
  l.off_bars = l.off_kb + KEYS_MAX * 4;                          // s, o, oread, pfull[2], pfree[2], q
  l.off_tmem = l.off_bars + 8 * 8;
  l.total = l.off_tmem + 16;
  return l;
}

struct Params {
  const float* q; const float* k; const float* v; int64_t ld_q, ld_k, ld_v;
  const int64_t* ids; const float* r_u; float w_h, w_obj; int mode;
  float* out; int B, L, H, dh, q_row0, n_q;
  int* error_flag;
  float* lse;                      // optional [B,H,n_q]: natural-log log-sum-exp of the masked scores (for irs_pim_attn_bwd)
};

__global__ void __launch_bounds__(THREADS, 2)
pim_attn_tc_kernel(const Params p) {
  extern __shared__ __align__(128) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const Layout lay = make_layout(p.dh);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int b = blockIdx.x / p.H, h = blockIdx.x % p.H;
  const int L = p.L, dh = p.dh, slabs = dh / 8;
  const bool pim = (p.mode == IRS_MASK_PIM);
  const int koff = pim ? 1 : 0;                    // column c <-> key c - koff; column 0 <-> key L-1 in PIM mode
  const int ncols = L;                             // PIM: {L-1, 0..L-2};  otherwise 0..L-1
  // Scores are kept in the log2 domain: q is pre-scaled by log2(e)/sqrt(dh) and the additive mask by
  // log2(e), so the softmax numerator is a bare exp2(s' - max').
  const float l2e = 1.4426950408889634f;
  const float qscale = l2e / sqrtf((float)dh);
  const float obj = pim ? p.w_obj * p.r_u[b] : 0.f;
  const float base_w = pim ? p.w_h : 0.f;
  float* kb = reinterpret_cast<float*>(smem + lay.off_kb);

  const uint32_t bar_s = sbase + lay.off_bars, bar_o = bar_s + 8, bar_oread = bar_s + 16;
  auto bar_pfull = [&](int i) { return bar_s + 24 + 8u * i; };
  auto bar_pfree = [&](int i) { return bar_s + 40 + 8u * i; };
  const uint32_t bar_q = bar_s + 56;
  volatile uint32_t* tmem_holder = reinterpret_cast<volatile uint32_t*>(smem + lay.off_tmem);

  if (tid == 0) {
    mbar_init(bar_s, 1); mbar_init(bar_o, 1); mbar_init(bar_oread, 128); mbar_init(bar_q, 128);
    for (int i = 0; i < 2; ++i) { mbar_init(bar_pfull(i), 128); mbar_init(bar_pfree(i), 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 4) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 :: "r"(sbase + lay.off_tmem), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }

  auto key_of = [&](int c) { return (pim && c == 0) ? L - 1 : c - koff; };
  const int first_tile = p.q_row0 / BM;
  const int last_tile = (p.q_row0 + p.n_q - 1) / BM;
  // columns the last processed tile can see (causal) -> how much of K / V^T must be staged
  const int cols_needed = min(BM * (last_tile + 1), L - koff) + koff;
  const int cols_pad = (cols_needed + 15) & ~15;
  const uint32_t k_lbo = (uint32_t)KEYS_MAX * 16, v_lbo = (uint32_t)dh * 16, q_lbo = (uint32_t)BM * 16;

  // ---- stage K: rows = key columns, K-major (dh contiguous)
  const float* kbase = p.k + (int64_t)b * L * p.ld_k + h * dh;
  const float* vbase = p.v + (int64_t)b * L * p.ld_v + h * dh;
  for (int c = tid; c < cols_pad; c += THREADS) {                 // thread <-> key column, all of its slabs
    const bool ok = c < ncols && c < cols_needed;
    const float* src = kbase + (int64_t)(ok ? key_of(c) : 0) * p.ld_k;
    for (int s = 0; s < slabs; ++s) {
      float x[8];
      if (ok) {
        const float4 v0 = *reinterpret_cast<const float4*>(src + s * 8), v1 = *reinterpret_cast<const float4*>(src + s * 8 + 4);
        x[0] = v0.x; x[1] = v0.y; x[2] = v0.z; x[3] = v0.w; x[4] = v1.x; x[5] = v1.y; x[6] = v1.z; x[7] = v1.w;
      } else {
#pragma unroll
        for (int e = 0; e < 8; ++e) x[e] = 0.f;
      }
      uint4 hi, lo;
      split8(x, hi, lo);
      *reinterpret_cast<uint4*>(smem + lay.off_k_hi + s * k_lbo + c * 16) = hi;
      *reinterpret_cast<uint4*>(smem + lay.off_k_lo + s * k_lbo + c * 16) = lo;
    }
  }
  // ---- stage V^T: rows = head dims, K-major over key columns (register transpose: lane <-> head dim,
  //      warp <-> group of 8 keys; every load is a coalesced 128-byte row segment)
  const int vcols = (cols_pad + PB - 1) / PB * PB;               // P blocks are 32 keys wide: zero-fill up to the block edge
  for (int ks = warp; ks < vcols / 8; ks += THREADS / 32) {
    for (int c = lane; c < dh; c += 32) {
      float x[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int col = ks * 8 + e;
        x[e] = (col < ncols && col < cols_needed) ? vbase[(int64_t)key_of(col) * p.ld_v + c] : 0.f;
      }
      uint4 hi, lo;
      split8(x, hi, lo);
      *reinterpret_cast<uint4*>(smem + lay.off_v_hi + ks * v_lbo + c * 16) = hi;
      *reinterpret_cast<uint4*>(smem + lay.off_v_lo + ks * v_lbo + c * 16) = lo;
    }
  }
  for (int c = tid; c < KEYS_MAX; c += THREADS) {
    // per-column additive term of every row that can see the column: l2e * (mask weight + key padding)
    float bias = -INFINITY;                                   // padded columns never contribute
    if (c < ncols) {
      const bool pad = (p.mode != IRS_MASK_CAUSAL && p.ids[(int64_t)b * L + key_of(c)] == 0);
      bias = pad ? -INFINITY : l2e * ((pim && c == 0) ? obj : base_w);
    }
    kb[c] = bias;
  }
  // Q tile: thread r (< 128) owns query row r of the tile -- its dh floats are one contiguous segment.
  const float* qbase = p.q + (int64_t)b * L * p.ld_q + h * dh;
  auto load_q_slab = [&](int tile, int r, int s, float (&x)[8]) {
    const int i = tile * BM + r;
    if (i < L) {
      const float* src = qbase + (int64_t)i * p.ld_q + s * 8;
      const float4 v0 = *reinterpret_cast<const float4*>(src), v1 = *reinterpret_cast<const float4*>(src + 4);
      x[0] = v0.x * qscale; x[1] = v0.y * qscale; x[2] = v0.z * qscale; x[3] = v0.w * qscale;
      x[4] = v1.x * qscale; x[5] = v1.y * qscale; x[6] = v1.z * qscale; x[7] = v1.w * qscale;
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) x[e] = 0.f;
    }
  };
  auto store_q_slab = [&](int r, int s, const float (&x)[8]) {
    uint4 hi, lo;
    split8(x, hi, lo);
    *reinterpret_cast<uint4*>(smem + lay.off_q_hi + s * q_lbo + r * 16) = hi;
    *reinterpret_cast<uint4*>(smem + lay.off_q_lo + s * q_lbo + r * 16) = lo;
  };
  if (tid < BM) {
    for (int s = 0; s < slabs; ++s) {
      float x[8];
      load_q_slab(first_tile, tid, s, x);
      store_q_slab(tid, s, x);
    }
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  uint32_t ph_s = 0, ph_o = 0, ph_oread = 0, ph_q = 0, ph_pfull[2] = {0, 0}, ph_pfree[2] = {0, 0};

  if (warp == 4) {
    // ===== MMA issue (lane 0) + restaging of the next query tile (whole warp) =====
    for (int tile = first_tile; tile <= last_tile; ++tile) {
      const int tcols = min(BM * (tile + 1), L - koff) + koff;       // columns this tile can see
      const int tcols_pad = (tcols + 15) & ~15;
      const int nblk = (tcols_pad + PB - 1) / PB;
      if (tile > first_tile && lane == 0) {
        // the softmax threads re-filled the Q buffer (bar_q) and read the previous tile's O (bar_oread)
        mbar_wait(bar_q, ph_q, p.error_flag, 20); ph_q ^= 1u;
        mbar_wait(bar_oread, ph_oread, p.error_flag, 21); ph_oread ^= 1u;
      }
      if (lane == 0) {
        tc_fence_after();
        const uint32_t idesc_s = make_idesc_bf16(BM, tcols_pad);
        for (int kk = 0; kk < dh / 16; ++kk) {
          const uint64_t q_hi = make_desc(sbase + lay.off_q_hi + (uint32_t)(kk * 2) * q_lbo, q_lbo, SBO);
          const uint64_t q_lo = make_desc(sbase + lay.off_q_lo + (uint32_t)(kk * 2) * q_lbo, q_lbo, SBO);
          const uint64_t k_hi = make_desc(sbase + lay.off_k_hi + (uint32_t)(kk * 2) * k_lbo, k_lbo, SBO);
          const uint64_t k_lo = make_desc(sbase + lay.off_k_lo + (uint32_t)(kk * 2) * k_lbo, k_lbo, SBO);
          tc_mma_bf16(tmem_base, q_lo, k_hi, idesc_s, kk != 0 ? 1u : 0u);
          tc_mma_bf16(tmem_base, q_hi, k_lo, idesc_s, 1u);
          tc_mma_bf16(tmem_base, q_hi, k_hi, idesc_s, 1u);
        }
        tc_commit(bar_s);
        const uint32_t idesc_o = make_idesc_bf16(BM, dh);
        for (int blk = 0; blk < nblk; ++blk) {
          const int pb = blk & 1;
          mbar_wait(bar_pfull(pb), ph_pfull[pb], p.error_flag, 22);
          ph_pfull[pb] ^= 1u;
          tc_fence_after();
          const uint32_t ps = sbase + lay.off_p + pb * lay.p_buf_bytes;
#pragma unroll
          for (int kk = 0; kk < PB / 16; ++kk) {
            const uint64_t p_hi = make_desc(ps + (uint32_t)(kk * 2) * q_lbo, q_lbo, SBO);
            const uint64_t p_lo = make_desc(ps + lay.p_buf_bytes / 2 + (uint32_t)(kk * 2) * q_lbo, q_lbo, SBO);
            const uint32_t vo = (uint32_t)(blk * (PB / 8) + kk * 2) * v_lbo;
            const uint64_t v_hi = make_desc(sbase + lay.off_v_hi + vo, v_lbo, SBO);
            const uint64_t v_lo = make_desc(sbase + lay.off_v_lo + vo, v_lbo, SBO);
            tc_mma_bf16(tmem_base + O_COL, p_lo, v_hi, idesc_o, (blk | kk) != 0 ? 1u : 0u);
            tc_mma_bf16(tmem_base + O_COL, p_hi, v_lo, idesc_o, 1u);
            tc_mma_bf16(tmem_base + O_COL, p_hi, v_hi, idesc_o, 1u);
          }
          tc_commit(bar_pfree(pb));
        }
        tc_commit(bar_o);
      }
      __syncwarp();
    }
  } else {
    // ===== softmax warps: thread <-> query row =====
    // Column blocks (32 keys) are classified per WARP: fully visible to its 32 rows (no per-element
    // test), on the causal diagonal (per-element test), or invisible (skipped; P block zero-filled).
    const int row = warp * 32 + lane;
    const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16);
    for (int tile = first_tile; tile <= last_tile; ++tile) {
      const int i = tile * BM + row;
      const int tcols = min(BM * (tile + 1), L - koff) + koff;
      const int tcols_pad = (tcols + 15) & ~15;
      const int nblk = (tcols_pad + PB - 1) / PB;
      const int r_lo = tile * BM + warp * 32;                      // first row of this warp
      const int vis_last = min(r_lo + 31 + koff, tcols - 1);       // last column any row of the warp sees
      const int nb_warp = vis_last / PB + 1;                       // blocks this warp must evaluate
      const int n_full = (r_lo + koff + 1) / PB;                   // blocks [0, n_full) are visible to every row
      const int my_last = i + koff;                                // last visible column of this row
      mbar_wait(bar_s, ph_s, p.error_flag, 23);
      ph_s ^= 1u;
      tc_fence_after();
      if (tile < last_tile) {
        // S of this tile is complete, so the Q buffer is free: stage the next tile's query row of this
        // thread (the loads overlap pass 1) and tell the MMA warp.
        for (int s = 0; s < slabs; ++s) {
          float x[8];
          load_q_slab(tile + 1, row, s, x);
          store_q_slab(row, s, x);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_arrive(bar_q);
      }
      float mx = -INFINITY;
      for (int blk = 0; blk < nb_warp; ++blk) {
        uint32_t v[32];
        tc_ld32(trow + blk * PB, v);
        const float4* cw4 = reinterpret_cast<const float4*>(kb + blk * PB);
        tc_wait_ld();
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
            const bool first = pim && c == 0;                     // the objective column is visible to every row
            if (c + 0 <= my_last || first) m0 = fmaxf(m0, __uint_as_float(v[4 * j4 + 0]) + w.x);
            if (c + 1 <= my_last) m1 = fmaxf(m1, __uint_as_float(v[4 * j4 + 1]) + w.y);
            if (c + 2 <= my_last) m2 = fmaxf(m2, __uint_as_float(v[4 * j4 + 2]) + w.z);
            if (c + 3 <= my_last) m3 = fmaxf(m3, __uint_as_float(v[4 * j4 + 3]) + w.w);
          }
        }
        mx = fmaxf(mx, fmaxf(fmaxf(m0, m1), fmaxf(m2, m3)));
      }
      float sum = 0.f;
      for (int blk = 0; blk < nblk; ++blk) {
        const int pb = blk & 1;
        uint32_t v[32];
        const bool live = blk < nb_warp;
        if (live) tc_ld32(trow + blk * PB, v);
        if (blk >= 2) { mbar_wait(bar_pfree(pb), ph_pfree[pb], p.error_flag, 24); ph_pfree[pb] ^= 1u; }
        uint8_t* pdst = smem + lay.off_p + pb * lay.p_buf_bytes;
        if (live) {
          const float4* cw4 = reinterpret_cast<const float4*>(kb + blk * PB);
          tc_wait_ld();
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
                float pv = exp2f(__uint_as_float(v[s8 * 8 + hq * 4 + e]) + ww[e] - mx);
                if (!full && !(c + e <= my_last || (pim && c + e == 0))) pv = 0.f;
                x[hq * 4 + e] = pv;
                sum += pv;
              }
            }
            uint4 hi, lo;
            split8(x, hi, lo);
            *reinterpret_cast<uint4*>(pdst + s8 * q_lbo + row * 16) = hi;
            *reinterpret_cast<uint4*>(pdst + lay.p_buf_bytes / 2 + s8 * q_lbo + row * 16) = lo;
          }
        } else {
          const uint4 z = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
          for (int s8 = 0; s8 < PB / 8; ++s8) {
            *reinterpret_cast<uint4*>(pdst + s8 * q_lbo + row * 16) = z;
            *reinterpret_cast<uint4*>(pdst + lay.p_buf_bytes / 2 + s8 * q_lbo + row * 16) = z;
          }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        tc_fence_before();
        mbar_arrive(bar_pfull(pb));
      }
      // drain the pfree phases of this tile's last (up to two) blocks so the parity bookkeeping stays aligned
      for (int blk = max(nblk - 2, 0); blk < nblk; ++blk) {
        const int pb = blk & 1;
        mbar_wait(bar_pfree(pb), ph_pfree[pb], p.error_flag, 25);
        ph_pfree[pb] ^= 1u;
      }
      mbar_wait(bar_o, ph_o, p.error_flag, 26);
      ph_o ^= 1u;
      tc_fence_after();
      {
        const float inv = 1.0f / sum;
        const bool write = (i < L) && (i >= p.q_row0) && (i < p.q_row0 + p.n_q);
        float* dst = p.out + ((int64_t)b * p.n_q + (i - p.q_row0)) * (p.H * dh) + h * dh;
        // scores live in the log2 domain (q pre-scaled by log2(e)/sqrt(dh)): lse = ln 2 * (max + log2 sum)
        if (write && p.lse != nullptr)
          p.lse[((int64_t)b * p.H + h) * p.n_q + (i - p.q_row0)] = 0.6931471805599453f * (mx + log2f(sum));
        for (int c0 = 0; c0 < dh; c0 += 16) {
          uint32_t v[16];
          asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 "
                       "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                       : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                         "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                       : "r"(trow + O_COL + c0));
          tc_wait_ld();
          if (write) {
#pragma unroll
            for (int j = 0; j < 16; j += 4)
              *reinterpret_cast<float4*>(dst + c0 + j) = make_float4(__uint_as_float(v[j]) * inv, __uint_as_float(v[j + 1]) * inv,
                                                                     __uint_as_float(v[j + 2]) * inv, __uint_as_float(v[j + 3]) * inv);
          }
        }
      }
      tc_fence_before();
      mbar_arrive(bar_oread);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

}  // namespace tca

// ---------------------------------------------------------------------------------------------------------
// Key-blocked variant for windows of any length up to 2048.  One CTA per (batch, head, 128-row query tile);
// thread r (< 128) owns query row r of the tile (TMEM lane r), thread 0 also issues the MMAs.  Q is staged once;
// K and V^T stream through shared memory in blocks of KB = 128 keys, converted to the same bf16 hi/lo core-matrix
// images the resident kernel uses.  Tile t visits key blocks 0..t only (causality):
//   pass 1   S_blk = Q K_blk^T (TMEM columns [0,128)), running row max of the masked scores (no exp)
//   pass 2   S_blk again; P = exp2(s - max) as hi/lo 32-key sub-blocks (double buffered),
//            O += P V_blk (TMEM columns [128, 128+dh)) and the row sum
//   epilogue O / sum, lse
// The objective key L-1 of PIM mode is not in any block: each row adds it as an exact fp32 term
// (q_i . k_{L-1}, weight exp2(s_obj - max), v_{L-1} added in the epilogue), so no tile visits extra blocks.
// Shared memory: Q, K, V^T at most 32 KB each (dh = 64), P 32 KB, independent of L.  Two CTAs per SM for dh <= 48
// overlap one CTA's staging with the other's MMAs.
// ---------------------------------------------------------------------------------------------------------
namespace tcb {

using namespace irs::tc;

constexpr int BM = 128;
constexpr int KB = 128;              // keys per block
constexpr int PB = 32;               // keys per P sub-block
constexpr int THREADS = 128;
constexpr uint32_t SBO = 128;
constexpr uint32_t TMEM_COLS = 256;
constexpr uint32_t O_COL = KB;

struct Layout {
  uint32_t off_q_hi, off_q_lo, off_k_hi, off_k_lo, off_v_hi, off_v_lo, off_p, p_buf_bytes, off_kb, off_bars, off_tmem, total;
};
__host__ __device__ inline Layout make_layout(int dh) {
  Layout l;
  const uint32_t part = (uint32_t)BM * dh * 2;                  // one bf16 part of a [128][dh] operand
  l.off_q_hi = 0; l.off_q_lo = part;
  l.off_k_hi = 2 * part; l.off_k_lo = 3 * part;                  // K   : [dh/8][128 keys][8]
  l.off_v_hi = 4 * part; l.off_v_lo = 5 * part;                  // V^T : [128/8 key groups][dh][8]
  l.off_p = 6 * part;
  l.p_buf_bytes = 2u * (PB / 8) * BM * 16;                       // hi + lo of one 32-key sub-block: 16384
  l.off_kb = l.off_p + 2 * l.p_buf_bytes;                        // float [128] key bias of the block
  l.off_bars = l.off_kb + KB * 4;                                // s, v, pfree[2]
  l.off_tmem = l.off_bars + 4 * 8;
  l.total = l.off_tmem + 16;
  return l;
}

__global__ void __launch_bounds__(THREADS, 2)
pim_attn_tc_blocked_kernel(const tca::Params p) {
  extern __shared__ __align__(128) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const Layout lay = make_layout(p.dh);
  const int tid = threadIdx.x, warp = tid >> 5;
  const int b = blockIdx.x / p.H, h = blockIdx.x % p.H;
  const int tile = p.q_row0 / BM + blockIdx.y;
  const int L = p.L, dh = p.dh, slabs = dh / 8;
  const bool pim = (p.mode == IRS_MASK_PIM);
  const int Lk = pim ? L - 1 : L;                  // keys held in blocks (PIM: all but the objective key)
  const float l2e = 1.4426950408889634f;
  const float qscale = l2e / sqrtf((float)dh);
  const float base_w = l2e * (pim ? p.w_h : 0.f);
  float* kb = reinterpret_cast<float*>(smem + lay.off_kb);

  const uint32_t bar_s = sbase + lay.off_bars, bar_v = bar_s + 8;
  auto bar_pfree = [&](int i) { return bar_s + 16 + 8u * i; };
  volatile uint32_t* tmem_holder = reinterpret_cast<volatile uint32_t*>(smem + lay.off_tmem);
  if (tid == 0) {
    mbar_init(bar_s, 1); mbar_init(bar_v, 1); mbar_init(bar_pfree(0), 1); mbar_init(bar_pfree(1), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 :: "r"(sbase + lay.off_tmem), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }

  const uint32_t k_lbo = (uint32_t)KB * 16, v_lbo = (uint32_t)dh * 16, q_lbo = (uint32_t)BM * 16;
  const float* qbase = p.q + (int64_t)b * L * p.ld_q + h * dh;
  const float* kbase = p.k + (int64_t)b * L * p.ld_k + h * dh;
  const float* vbase = p.v + (int64_t)b * L * p.ld_v + h * dh;
  const int i = tile * BM + tid;                   // this thread's query row
  const bool row_ok = i < L;

  // Q tile, pre-scaled into the log2 domain; the objective score in fp32 from the same scaled q
  float s_obj = -INFINITY;
  {
    const float* qk = kbase + (int64_t)(L - 1) * p.ld_k;
    float dot = 0.f;
    for (int s = 0; s < slabs; ++s) {
      float x[8];
      if (row_ok) {
        const float* src = qbase + (int64_t)i * p.ld_q + s * 8;
        const float4 v0 = *reinterpret_cast<const float4*>(src), v1 = *reinterpret_cast<const float4*>(src + 4);
        x[0] = v0.x * qscale; x[1] = v0.y * qscale; x[2] = v0.z * qscale; x[3] = v0.w * qscale;
        x[4] = v1.x * qscale; x[5] = v1.y * qscale; x[6] = v1.z * qscale; x[7] = v1.w * qscale;
        if (pim) {
          const float4 k0 = *reinterpret_cast<const float4*>(qk + s * 8), k1 = *reinterpret_cast<const float4*>(qk + s * 8 + 4);
          dot = fmaf(x[0], k0.x, dot); dot = fmaf(x[1], k0.y, dot); dot = fmaf(x[2], k0.z, dot); dot = fmaf(x[3], k0.w, dot);
          dot = fmaf(x[4], k1.x, dot); dot = fmaf(x[5], k1.y, dot); dot = fmaf(x[6], k1.z, dot); dot = fmaf(x[7], k1.w, dot);
        }
      } else {
#pragma unroll
        for (int e = 0; e < 8; ++e) x[e] = 0.f;
      }
      uint4 hi, lo;
      split8(x, hi, lo);
      *reinterpret_cast<uint4*>(smem + lay.off_q_hi + s * q_lbo + tid * 16) = hi;
      *reinterpret_cast<uint4*>(smem + lay.off_q_lo + s * q_lbo + tid * 16) = lo;
    }
    if (pim && p.ids[(int64_t)b * L + L - 1] != 0) s_obj = dot + l2e * p.w_obj * p.r_u[b];
  }

  // blocks this tile visits: keys 0 .. min(last row of the tile, Lk - 1)
  const int nblk = (min(BM * (tile + 1), Lk) + KB - 1) / KB;
  auto stage_k = [&](int blk) {                                  // thread <-> key column of the block
    const int j = blk * KB + tid;
    const bool ok = j < Lk;
    const float* src = kbase + (int64_t)(ok ? j : 0) * p.ld_k;
    for (int s = 0; s < slabs; ++s) {
      float x[8];
      if (ok) {
        const float4 v0 = *reinterpret_cast<const float4*>(src + s * 8), v1 = *reinterpret_cast<const float4*>(src + s * 8 + 4);
        x[0] = v0.x; x[1] = v0.y; x[2] = v0.z; x[3] = v0.w; x[4] = v1.x; x[5] = v1.y; x[6] = v1.z; x[7] = v1.w;
      } else {
#pragma unroll
        for (int e = 0; e < 8; ++e) x[e] = 0.f;
      }
      uint4 hi, lo;
      split8(x, hi, lo);
      *reinterpret_cast<uint4*>(smem + lay.off_k_hi + s * k_lbo + tid * 16) = hi;
      *reinterpret_cast<uint4*>(smem + lay.off_k_lo + s * k_lbo + tid * 16) = lo;
    }
    kb[tid] = (!ok || (p.mode != IRS_MASK_CAUSAL && p.ids[(int64_t)b * L + j] == 0)) ? -INFINITY : base_w;
  };
  auto stage_v = [&](int blk) {                                  // warp <-> group of 8 keys, lane <-> head dim
    const int lane = tid & 31;
    for (int ks = warp; ks < KB / 8; ks += THREADS / 32) {
      for (int c = lane; c < dh; c += 32) {
        float x[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int j = blk * KB + ks * 8 + e;
          x[e] = (j < Lk) ? vbase[(int64_t)j * p.ld_v + c] : 0.f;
        }
        uint4 hi, lo;
        split8(x, hi, lo);
        *reinterpret_cast<uint4*>(smem + lay.off_v_hi + ks * v_lbo + c * 16) = hi;
        *reinterpret_cast<uint4*>(smem + lay.off_v_lo + ks * v_lbo + c * 16) = lo;
      }
    }
  };

  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;
  const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16);
  const uint32_t idesc_s = make_idesc_bf16(BM, KB);
  const uint32_t idesc_o = make_idesc_bf16(BM, dh);
  uint32_t ph_s = 0, ph_v = 0, ph_pfree[2] = {0, 0};

  // S_blk = Q K_blk^T once the K image of the block is in shared memory; every thread waits for it
  auto score_block = [&]() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      for (int kk = 0; kk < dh / 16; ++kk) {
        const uint64_t q_hi = make_desc(sbase + lay.off_q_hi + (uint32_t)(kk * 2) * q_lbo, q_lbo, SBO);
        const uint64_t q_lo = make_desc(sbase + lay.off_q_lo + (uint32_t)(kk * 2) * q_lbo, q_lbo, SBO);
        const uint64_t k_hi = make_desc(sbase + lay.off_k_hi + (uint32_t)(kk * 2) * k_lbo, k_lbo, SBO);
        const uint64_t k_lo = make_desc(sbase + lay.off_k_lo + (uint32_t)(kk * 2) * k_lbo, k_lbo, SBO);
        tc_mma_bf16(tmem_base, q_lo, k_hi, idesc_s, kk != 0 ? 1u : 0u);
        tc_mma_bf16(tmem_base, q_hi, k_lo, idesc_s, 1u);
        tc_mma_bf16(tmem_base, q_hi, k_hi, idesc_s, 1u);
      }
      tc_commit(bar_s);
    }
    mbar_wait(bar_s, ph_s, p.error_flag, 40);
    ph_s ^= 1u;
    tc_fence_after();
  };

  // ---- pass 1: row max
  float mx = s_obj;
  for (int blk = 0; blk < nblk; ++blk) {
    __syncthreads();                                             // every thread is done with the previous block's kb
    stage_k(blk);
    score_block();
    const bool full = (blk + 1) * KB <= min(tile * BM + 1, Lk);  // every key of the block visible to every row
    for (int sb = 0; sb < KB / PB; ++sb) {
      uint32_t v[32];
      tc_ld32(trow + sb * PB, v);
      const float4* cw4 = reinterpret_cast<const float4*>(kb + sb * PB);
      tc_wait_ld();
      const int c0 = blk * KB + sb * PB;
      float m0 = -INFINITY, m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;
      if (full) {
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
          const int c = c0 + 4 * j4;
          if (c + 0 <= i) m0 = fmaxf(m0, __uint_as_float(v[4 * j4 + 0]) + w.x);
          if (c + 1 <= i) m1 = fmaxf(m1, __uint_as_float(v[4 * j4 + 1]) + w.y);
          if (c + 2 <= i) m2 = fmaxf(m2, __uint_as_float(v[4 * j4 + 2]) + w.z);
          if (c + 3 <= i) m3 = fmaxf(m3, __uint_as_float(v[4 * j4 + 3]) + w.w);
        }
      }
      mx = fmaxf(mx, fmaxf(fmaxf(m0, m1), fmaxf(m2, m3)));
    }
  }

  // ---- pass 2: P and O += P V
  float sum = pim ? exp2f(s_obj - mx) : 0.f;                     // fully masked row: -inf - -inf = NaN, as torch
  for (int blk = 0; blk < nblk; ++blk) {
    if (blk > 0) { mbar_wait(bar_v, ph_v, p.error_flag, 41); ph_v ^= 1u; }   // the previous block's O MMAs read V and P
    __syncthreads();
    stage_k(blk);
    stage_v(blk);
    score_block();
    const bool full = (blk + 1) * KB <= min(tile * BM + 1, Lk);
    for (int sb = 0; sb < KB / PB; ++sb) {
      const int g = blk * (KB / PB) + sb, pb = g & 1;
      uint32_t v[32];
      tc_ld32(trow + sb * PB, v);
      if (g >= 2) { mbar_wait(bar_pfree(pb), ph_pfree[pb], p.error_flag, 42); ph_pfree[pb] ^= 1u; }
      uint8_t* pdst = smem + lay.off_p + pb * lay.p_buf_bytes;
      const float4* cw4 = reinterpret_cast<const float4*>(kb + sb * PB);
      tc_wait_ld();
      const int c0 = blk * KB + sb * PB;
#pragma unroll
      for (int s8 = 0; s8 < PB / 8; ++s8) {
        float x[8];
#pragma unroll
        for (int hq = 0; hq < 2; ++hq) {
          const float4 w = cw4[s8 * 2 + hq];
          const float ww[4] = {w.x, w.y, w.z, w.w};
          const int c = c0 + s8 * 8 + hq * 4;
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            float pv = exp2f(__uint_as_float(v[s8 * 8 + hq * 4 + e]) + ww[e] - mx);
            if (!full && c + e > i) pv = 0.f;
            x[hq * 4 + e] = pv;
            sum += pv;
          }
        }
        uint4 hi, lo;
        split8(x, hi, lo);
        *reinterpret_cast<uint4*>(pdst + s8 * q_lbo + tid * 16) = hi;
        *reinterpret_cast<uint4*>(pdst + lay.p_buf_bytes / 2 + s8 * q_lbo + tid * 16) = lo;
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      tc_fence_before();
      __syncthreads();
      if (tid == 0) {
        tc_fence_after();
        const uint32_t ps = sbase + lay.off_p + pb * lay.p_buf_bytes;
#pragma unroll
        for (int kk = 0; kk < PB / 16; ++kk) {
          const uint64_t p_hi = make_desc(ps + (uint32_t)(kk * 2) * q_lbo, q_lbo, SBO);
          const uint64_t p_lo = make_desc(ps + lay.p_buf_bytes / 2 + (uint32_t)(kk * 2) * q_lbo, q_lbo, SBO);
          const uint32_t vo = (uint32_t)(sb * (PB / 8) + kk * 2) * v_lbo;
          const uint64_t v_hi = make_desc(sbase + lay.off_v_hi + vo, v_lbo, SBO);
          const uint64_t v_lo = make_desc(sbase + lay.off_v_lo + vo, v_lbo, SBO);
          tc_mma_bf16(tmem_base + O_COL, p_lo, v_hi, idesc_o, (g | kk) != 0 ? 1u : 0u);
          tc_mma_bf16(tmem_base + O_COL, p_hi, v_lo, idesc_o, 1u);
          tc_mma_bf16(tmem_base + O_COL, p_hi, v_hi, idesc_o, 1u);
        }
        tc_commit(bar_pfree(pb));
        if (sb == KB / PB - 1) tc_commit(bar_v);
      }
    }
  }
  if (nblk > 0) { mbar_wait(bar_v, ph_v, p.error_flag, 43); ph_v ^= 1u; }
  tc_fence_after();

  // ---- epilogue: O / sum (+ the objective term), lse
  {
    const bool write = row_ok && (i >= p.q_row0) && (i < p.q_row0 + p.n_q);
    const float inv = 1.0f / sum;
    const float w_obj_row = pim ? exp2f(s_obj - mx) : 0.f;
    const float* vobj = vbase + (int64_t)(L - 1) * p.ld_v;
    float* dst = p.out + ((int64_t)b * p.n_q + (i - p.q_row0)) * (p.H * dh) + h * dh;
    if (write && p.lse != nullptr)
      p.lse[((int64_t)b * p.H + h) * p.n_q + (i - p.q_row0)] = 0.6931471805599453f * (mx + log2f(sum));
    for (int c0 = 0; c0 < dh; c0 += 16) {
      uint32_t v[16];
      if (nblk > 0) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 "
                     "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                     : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                       "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                     : "r"(trow + O_COL + c0));
        tc_wait_ld();
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = 0u;
      }
      if (write) {
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
          float4 o4 = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
          if (pim) {
            const float4 vo = *reinterpret_cast<const float4*>(vobj + c0 + j);
            o4.x = fmaf(w_obj_row, vo.x, o4.x); o4.y = fmaf(w_obj_row, vo.y, o4.y);
            o4.z = fmaf(w_obj_row, vo.z, o4.z); o4.w = fmaf(w_obj_row, vo.w, o4.w);
          }
          *reinterpret_cast<float4*>(dst + c0 + j) = make_float4(o4.x * inv, o4.y * inv, o4.z * inv, o4.w * inv);
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

}  // namespace tcb
}  // namespace irs

using namespace irs;

extern "C" int irs_pim_attn_tc_supported(int L, int dh) {
  return (dh % 16 == 0 && dh >= 16 && dh <= 64 && L >= 1 && L <= IRS_ATTN_MAX_L) ? 1 : 0;
}

static int attn_tc_check(const float* q, const float* k, const float* v, int64_t ld_q, int64_t ld_k, int64_t ld_v,
                         const int64_t* ids, const float* r_u, int mode, const float* out, int B, int L, int H, int dh,
                         int q_row0, int n_q) {
  if (!q || !k || !v || !out) return IRS_E_BADARG;
  if (B <= 0 || L <= 0 || H <= 0 || dh <= 0 || q_row0 < 0 || n_q <= 0 || q_row0 + n_q > L) return IRS_E_BADARG;
  if (mode < 0 || mode > 2) return IRS_E_BADARG;
  if (mode != IRS_MASK_CAUSAL && !ids) return IRS_E_BADARG;
  if (mode == IRS_MASK_PIM && !r_u) return IRS_E_BADARG;
  if (!irs_pim_attn_tc_supported(L, dh)) return IRS_E_SHAPE;
  if ((ld_q & 3) || (ld_k & 3) || (ld_v & 3) || ((uintptr_t)q & 15) || ((uintptr_t)k & 15) || ((uintptr_t)v & 15) ||
      ((uintptr_t)out & 15))
    return IRS_E_SHAPE;
  return 0;
}

static tca::Params attn_tc_params(const float* q, const float* k, const float* v, int64_t ld_q, int64_t ld_k, int64_t ld_v,
                                  const int64_t* ids, const float* r_u, float w_h, float w_obj, int mode,
                                  float* out, float* lse, int B, int L, int H, int dh, int q_row0, int n_q, int* error_flag) {
  tca::Params p = {};
  p.q = q; p.k = k; p.v = v; p.ld_q = ld_q; p.ld_k = ld_k; p.ld_v = ld_v; p.ids = ids; p.r_u = r_u;
  p.w_h = w_h; p.w_obj = w_obj; p.mode = mode; p.out = out; p.B = B; p.L = L; p.H = H; p.dh = dh;
  p.q_row0 = q_row0; p.n_q = n_q; p.error_flag = error_flag; p.lse = lse;
  return p;
}

static int attn_tc_blocked_launch(const tca::Params& p, void* stream) {
  const tcb::Layout lay = tcb::make_layout(p.dh);
  static uint32_t configured = 0;
  if (lay.total > configured) {
    IRS_CUDA(cudaFuncSetAttribute(tcb::pim_attn_tc_blocked_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lay.total));
    configured = lay.total;
  }
  const int tiles = (p.q_row0 + p.n_q - 1) / tcb::BM - p.q_row0 / tcb::BM + 1;
  dim3 grid((unsigned)(p.B * p.H), (unsigned)tiles);
  tcb::pim_attn_tc_blocked_kernel<<<grid, tcb::THREADS, lay.total, (cudaStream_t)stream>>>(p);
  IRS_LAUNCHED();
  return 0;
}

extern "C" int irs_pim_attn_fwd_tc(const float* q, const float* k, const float* v, int64_t ld_q, int64_t ld_k, int64_t ld_v,
                                   const int64_t* ids, const float* r_u, float w_h, float w_obj, int mode,
                                   float* out, float* lse, int B, int L, int H, int dh, int q_row0, int n_q,
                                   int* error_flag, void* stream) {
  const int rc = attn_tc_check(q, k, v, ld_q, ld_k, ld_v, ids, r_u, mode, out, B, L, H, dh, q_row0, n_q);
  if (rc) return rc;
  const tca::Params p = attn_tc_params(q, k, v, ld_q, ld_k, ld_v, ids, r_u, w_h, w_obj, mode, out, lse, B, L, H, dh,
                                       q_row0, n_q, error_flag);
  if (L > tca::KEYS_MAX - 1) return attn_tc_blocked_launch(p, stream);    // the head's K / V^T no longer fit on chip
  const tca::Layout lay = tca::make_layout(dh);
  static uint32_t configured = 0;
  if (lay.total > configured) {
    IRS_CUDA(cudaFuncSetAttribute(tca::pim_attn_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lay.total));
    configured = lay.total;
  }
  tca::pim_attn_tc_kernel<<<(unsigned)(B * H), tca::THREADS, lay.total, (cudaStream_t)stream>>>(p);
  IRS_LAUNCHED();
  return 0;
}

extern "C" int irs_pim_attn_fwd_tc_blocked(const float* q, const float* k, const float* v, int64_t ld_q, int64_t ld_k, int64_t ld_v,
                                           const int64_t* ids, const float* r_u, float w_h, float w_obj, int mode,
                                           float* out, float* lse, int B, int L, int H, int dh, int q_row0, int n_q,
                                           int* error_flag, void* stream) {
  const int rc = attn_tc_check(q, k, v, ld_q, ld_k, ld_v, ids, r_u, mode, out, B, L, H, dh, q_row0, n_q);
  if (rc) return rc;
  return attn_tc_blocked_launch(attn_tc_params(q, k, v, ld_q, ld_k, ld_v, ids, r_u, w_h, w_obj, mode, out, lse, B, L, H, dh,
                                               q_row0, n_q, error_flag), stream);
}
