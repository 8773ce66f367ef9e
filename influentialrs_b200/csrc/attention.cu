// K3 / K4: self-attention with the Personalized Impressionability Mask computed in-kernel
// (no [B*H,L,L] mask tensor ever exists).  fp32 CUDA-core version: K and V of one (batch, head)
// live in shared memory, a warp owns 4 query rows at a time, lanes split the keys for QK^T and the
// head dimension for PV.  Causality is exploited: row i only visits keys j <= i plus, in PIM mode,
// the objective column L-1 that every row sees.
//   reference: model/influentialRS.py:139-151 (PIM, keyword branch), :171 (key padding), :189-193
//   (decoder call), torch.nn.functional.multi_head_attention_forward (scores/softmax/PV);
//   model/uRS.py:47-61 (causal + padding), model/sas.py:168-177 (causal only).
#include "common.cuh"

namespace irs {

constexpr int kAttWarps = 8;
constexpr int kAttRows = 4;     // query rows a warp processes together

struct AttnSmem {
  int kstride;      // floats per K row (odd => conflict-free lane-per-key reads)
  int off_v, off_kb, off_warp, warp_floats, total_floats;
};

__host__ __device__ inline AttnSmem attn_smem_layout(int L, int dh) {
  AttnSmem s;
  s.kstride = dh | 1;
  s.off_v = (L * s.kstride + 3) & ~3;
  s.off_kb = s.off_v + ((L * dh + 3) & ~3);
  s.off_warp = s.off_kb + ((L + 3) & ~3);
  s.warp_floats = dh * kAttRows + L * kAttRows;      // q^T [dh][4] + p [L][4], both float4-aligned
  s.total_floats = s.off_warp + kAttWarps * s.warp_floats;
  return s;
}

// Attention-probability dropout (nn.MultiheadAttention(dropout=p) in train mode; model/influentialRS.py:67-74 builds the
// decoder layers with dropout=self.dropout): a counter-based keep mask, a pure function of (seed, batch*head, query, key),
// so the backward kernel regenerates exactly the mask of the forward.  Returns 0 or 1/(1-p).
__device__ __forceinline__ float drop_scale(unsigned long long seed, uint32_t thresh, float inv_keep, int bh, int i, int j, int L) {
  if (thresh == 0u) return 1.0f;
  unsigned long long x = seed + 0x9E3779B97F4A7C15ull * ((unsigned long long)(((long long)bh * L + i) * L + j) + 1ull);
  x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; x ^= x >> 33;   // murmur3 finaliser
  return ((uint32_t)(x >> 32) >= thresh) ? inv_keep : 0.0f;
}

__device__ __forceinline__ float mask_value(int mode, int i, int j, int L, float w_h, float obj) {
  if (mode == IRS_MASK_PIM) {
    if (j == L - 1) return obj;
    return (j <= i) ? w_h : -INFINITY;
  }
  return (j <= i) ? 0.f : -INFINITY;
}

__global__ void __launch_bounds__(kAttWarps * 32)
pim_attn_fwd_kernel(const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
                    int64_t ld_q, int64_t ld_k, int64_t ld_v, const int64_t* __restrict__ ids,
                    const float* __restrict__ r_u, float w_h, float w_obj, int mode,
                    float* __restrict__ out, float* __restrict__ lse,
                    int L, int H, int dh, int q_row0, int n_q, int rows_per_cta,
                    unsigned long long seed, uint32_t drop_thresh, float inv_keep) {
  extern __shared__ __align__(16) float smem[];
  const AttnSmem lay = attn_smem_layout(L, dh);
  float* Ks = smem;
  float* Vs = smem + lay.off_v;
  float* kb = smem + lay.off_kb;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* qs = smem + lay.off_warp + warp * lay.warp_floats;      // [dh][4]
  float* ps = qs + dh * kAttRows;                                // [L][4]

  const int b = blockIdx.x / H, h = blockIdx.x % H;
  const int q_begin = q_row0 + blockIdx.y * rows_per_cta;
  const int q_end = min(q_row0 + n_q, q_begin + rows_per_cta);
  if (q_begin >= q_end) return;
  const int d = H * dh;
  const float scale = 1.0f / sqrtf((float)dh);
  const float obj = (mode == IRS_MASK_PIM) ? w_obj * r_u[b] : 0.f;
  const bool pim = (mode == IRS_MASK_PIM);

  // Keys this CTA can touch: j <= q_end-1, plus the objective column.
  const int kmax = min(q_end - 1, L - 1);
  const float* kbase = k + (int64_t)b * L * ld_k + h * dh;
  const float* vbase = v + (int64_t)b * L * ld_v + h * dh;
  for (int idx = threadIdx.x; idx < L * dh; idx += blockDim.x) {
    const int j = idx / dh, c = idx - j * dh;
    if (j <= kmax || (pim && j == L - 1)) {
      Ks[j * lay.kstride + c] = kbase[(int64_t)j * ld_k + c];
      Vs[j * dh + c] = vbase[(int64_t)j * ld_v + c];
    }
  }
  for (int j = threadIdx.x; j < L; j += blockDim.x)
    kb[j] = (mode != IRS_MASK_CAUSAL && ids[(int64_t)b * L + j] == 0) ? -INFINITY : 0.f;
  __syncthreads();

  for (int i0 = q_begin + warp * kAttRows; i0 < q_end; i0 += kAttWarps * kAttRows) {
    const int nrows = min(kAttRows, q_end - i0);
    for (int idx = lane; idx < dh * kAttRows; idx += 32) {
      const int r = idx / dh, c = idx - r * dh;
      qs[c * kAttRows + r] = (r < nrows) ? q[((int64_t)b * L + i0 + r) * ld_q + h * dh + c] : 0.f;
    }
    __syncwarp();
    const int jmax = min(i0 + nrows - 1, L - 1);
    const int nslots = jmax + 1 + ((pim && jmax < L - 1) ? 1 : 0);
    float m[kAttRows];
#pragma unroll
    for (int r = 0; r < kAttRows; ++r) m[r] = -INFINITY;
    for (int t = lane; t < nslots; t += 32) {
      const int j = (t <= jmax) ? t : L - 1;
      const float* kr = Ks + j * lay.kstride;
      float acc[kAttRows] = {0.f, 0.f, 0.f, 0.f};
      for (int c = 0; c < dh; ++c) {
        const float kv = kr[c];
        const float4 q4 = *reinterpret_cast<const float4*>(qs + c * kAttRows);
        acc[0] = fmaf(q4.x, kv, acc[0]); acc[1] = fmaf(q4.y, kv, acc[1]);
        acc[2] = fmaf(q4.z, kv, acc[2]); acc[3] = fmaf(q4.w, kv, acc[3]);
      }
      float4 s4;
      float* sp = reinterpret_cast<float*>(&s4);
#pragma unroll
      for (int r = 0; r < kAttRows; ++r) {
        const float s = acc[r] * scale + (mask_value(mode, i0 + r, j, L, w_h, obj) + kb[j]);
        sp[r] = s;
        m[r] = fmaxf(m[r], s);
      }
      *reinterpret_cast<float4*>(ps + t * kAttRows) = s4;
    }
#pragma unroll
    for (int r = 0; r < kAttRows; ++r) m[r] = warp_max(m[r]);
    __syncwarp();
    float sum[kAttRows] = {0.f, 0.f, 0.f, 0.f};
    for (int t = lane; t < nslots; t += 32) {
      float4 s4 = *reinterpret_cast<const float4*>(ps + t * kAttRows);
      float* sp = reinterpret_cast<float*>(&s4);
#pragma unroll
      const int jd = (t <= jmax) ? t : L - 1;
      for (int r = 0; r < kAttRows; ++r) {
        const float p = expf(sp[r] - m[r]);    // fully masked row: -inf - -inf = NaN, as torch
        sum[r] += p;                           // the softmax normaliser is taken BEFORE dropout (F.dropout(softmax(s)))
        sp[r] = p * drop_scale(seed, drop_thresh, inv_keep, blockIdx.x, i0 + r, jd, L);
      }
      *reinterpret_cast<float4*>(ps + t * kAttRows) = s4;
    }
#pragma unroll
    for (int r = 0; r < kAttRows; ++r) sum[r] = warp_sum(sum[r]);
    __syncwarp();
    for (int c = lane; c < dh; c += 32) {
      float o[kAttRows] = {0.f, 0.f, 0.f, 0.f};
      for (int t = 0; t < nslots; ++t) {
        const int j = (t <= jmax) ? t : L - 1;
        const float vv = Vs[j * dh + c];
        const float4 p4 = *reinterpret_cast<const float4*>(ps + t * kAttRows);
        o[0] = fmaf(p4.x, vv, o[0]); o[1] = fmaf(p4.y, vv, o[1]);
        o[2] = fmaf(p4.z, vv, o[2]); o[3] = fmaf(p4.w, vv, o[3]);
      }
#pragma unroll
      for (int r = 0; r < kAttRows; ++r)
        if (r < nrows) out[((int64_t)b * n_q + (i0 + r - q_row0)) * d + h * dh + c] = o[r] / sum[r];
    }
    if (lse != nullptr && lane < nrows)
      lse[((int64_t)b * H + h) * n_q + (i0 + lane - q_row0)] = m[lane] + logf(sum[lane]);
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------------------
// backward.  Phase A (row-wise, warp per 4 query rows): D_i = dO_i . O_i and
//   dQ_i = scale * sum_j dS_ij K_j with dS_ij = P_ij (dO_i . V_j - D_i), P recomputed from lse.
// Phase B (column-wise, warp per 4 keys): dV_j = sum_i P_ij dO_i,  dK_j = scale * sum_i dS_ij Q_i,
//   and the PIM column's  d r_u[b] += w_obj * sum_{h,i} dS[i, L-1]  (one atomic per (b,h)).
// Recomputing P in both phases keeps everything in shared memory / registers (no L x L buffer, no
// atomics on dK/dV).
// ---------------------------------------------------------------------------------------------
struct AttnBwdSmem {
  int stride;   // odd row stride for Q,K,V,dO
  int off_k, off_v, off_do, off_kb, off_lse, off_D, off_warp, warp_floats, total_floats;
};
__host__ __device__ inline AttnBwdSmem attn_bwd_smem_layout(int L, int dh) {
  AttnBwdSmem s;
  s.stride = dh | 1;
  const int mat = (L * s.stride + 3) & ~3;
  s.off_k = mat; s.off_v = 2 * mat; s.off_do = 3 * mat;
  s.off_kb = 4 * mat;
  s.off_lse = s.off_kb + ((L + 3) & ~3);
  s.off_D = s.off_lse + ((L + 3) & ~3);
  s.off_warp = s.off_D + ((L + 3) & ~3);
  s.warp_floats = dh * kAttRows + 2 * L * kAttRows;    // x^T [dh][4], p [L][4], ds [L][4]
  s.total_floats = s.off_warp + kAttWarps * s.warp_floats;
  return s;
}

__global__ void __launch_bounds__(kAttWarps * 32)
pim_attn_bwd_kernel(const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
                    int64_t ld_q, int64_t ld_k, int64_t ld_v, const int64_t* __restrict__ ids,
                    const float* __restrict__ r_u, float w_h, float w_obj, int mode,
                    const float* __restrict__ o, const float* __restrict__ lse_g, const float* __restrict__ d_o,
                    float* __restrict__ d_q, float* __restrict__ d_k, float* __restrict__ d_v,
                    float* __restrict__ d_r_u, int L, int H, int dh,
                    unsigned long long seed, uint32_t drop_thresh, float inv_keep) {
  extern __shared__ __align__(16) float smem[];
  const AttnBwdSmem lay = attn_bwd_smem_layout(L, dh);
  float* Qs = smem;
  float* Ks = smem + lay.off_k;
  float* Vs = smem + lay.off_v;
  float* dOs = smem + lay.off_do;
  float* kb = smem + lay.off_kb;
  float* lses = smem + lay.off_lse;
  float* Ds = smem + lay.off_D;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* xs = smem + lay.off_warp + warp * lay.warp_floats;   // [dh][4]
  float* ps = xs + dh * kAttRows;                             // [L][4]
  float* dss = ps + L * kAttRows;                             // [L][4]
  const int st = lay.stride;

  const int b = blockIdx.x / H, h = blockIdx.x % H;
  const int d = H * dh;
  const float scale = 1.0f / sqrtf((float)dh);
  const bool pim = (mode == IRS_MASK_PIM);
  const float obj = pim ? w_obj * r_u[b] : 0.f;

  for (int idx = threadIdx.x; idx < L * dh; idx += blockDim.x) {
    const int j = idx / dh, c = idx - j * dh;
    const int64_t row = (int64_t)b * L + j;
    Qs[j * st + c] = q[row * ld_q + h * dh + c];
    Ks[j * st + c] = k[row * ld_k + h * dh + c];
    Vs[j * st + c] = v[row * ld_v + h * dh + c];
    dOs[j * st + c] = d_o[row * d + h * dh + c];
  }
  for (int j = threadIdx.x; j < L; j += blockDim.x) {
    kb[j] = (mode != IRS_MASK_CAUSAL && ids[(int64_t)b * L + j] == 0) ? -INFINITY : 0.f;
    lses[j] = lse_g[((int64_t)b * H + h) * L + j];
  }
  __syncthreads();
  // D_i = dO_i . O_i
  for (int i = warp; i < L; i += kAttWarps) {
    float acc = 0.f;
    for (int c = lane; c < dh; c += 32) acc += dOs[i * st + c] * o[((int64_t)b * L + i) * d + h * dh + c];
    acc = warp_sum(acc);
    if (lane == 0) Ds[i] = acc;
  }
  __syncthreads();

  // ---- Phase A: dQ
  for (int i0 = warp * kAttRows; i0 < L; i0 += kAttWarps * kAttRows) {
    const int nrows = min(kAttRows, L - i0);
    const int jmax = min(i0 + nrows - 1, L - 1);
    const int nslots = jmax + 1 + ((pim && jmax < L - 1) ? 1 : 0);
    for (int t = lane; t < nslots; t += 32) {
      const int j = (t <= jmax) ? t : L - 1;
      float4 ds4;
      float* dsp = reinterpret_cast<float*>(&ds4);
#pragma unroll
      for (int r = 0; r < kAttRows; ++r) {
        const int i = min(i0 + r, L - 1);
        float s = 0.f, dp = 0.f;
        for (int c = 0; c < dh; ++c) {
          const float kv = Ks[j * st + c];
          s = fmaf(Qs[i * st + c], kv, s);
          dp = fmaf(dOs[i * st + c], Vs[j * st + c], dp);
        }
        s = s * scale + (mask_value(mode, i0 + r, j, L, w_h, obj) + kb[j]);
        const float p = (r < nrows) ? expf(s - lses[i]) : 0.f;
        // with dropout O = (P o M) V: dP = (dO V^T) o M and D_i = dO_i . O_i still equals sum_j P_ij dP_ij
        dsp[r] = p * (dp * drop_scale(seed, drop_thresh, inv_keep, blockIdx.x, i, j, L) - Ds[i]);
      }
      *reinterpret_cast<float4*>(dss + t * kAttRows) = ds4;
    }
    __syncwarp();
    for (int c = lane; c < dh; c += 32) {
      float a[kAttRows] = {0.f, 0.f, 0.f, 0.f};
      for (int t = 0; t < nslots; ++t) {
        const int j = (t <= jmax) ? t : L - 1;
        const float kv = Ks[j * st + c];
        const float4 d4 = *reinterpret_cast<const float4*>(dss + t * kAttRows);
        a[0] = fmaf(d4.x, kv, a[0]); a[1] = fmaf(d4.y, kv, a[1]);
        a[2] = fmaf(d4.z, kv, a[2]); a[3] = fmaf(d4.w, kv, a[3]);
      }
#pragma unroll
      for (int r = 0; r < kAttRows; ++r)
        if (r < nrows) d_q[((int64_t)b * L + i0 + r) * ld_q + h * dh + c] = a[r] * scale;
    }
    __syncwarp();
  }

  // ---- Phase B: dK, dV (warp per 4 keys; lanes over query rows i >= j, or all rows for the
  //      objective column in PIM mode)
  float dru = 0.f;
  for (int j0 = warp * kAttRows; j0 < L; j0 += kAttWarps * kAttRows) {
    const int ncols = min(kAttRows, L - j0);
    const bool has_obj = pim && (j0 + ncols - 1 == L - 1);
    const int ibeg = has_obj ? 0 : j0;
    for (int i = ibeg + lane; i < L; i += 32) {
      float4 p4, ds4;
      float* pp = reinterpret_cast<float*>(&p4);
      float* dsp = reinterpret_cast<float*>(&ds4);
#pragma unroll
      for (int r = 0; r < kAttRows; ++r) {
        const int j = min(j0 + r, L - 1);
        float s = 0.f, dp = 0.f;
        for (int c = 0; c < dh; ++c) {
          s = fmaf(Qs[i * st + c], Ks[j * st + c], s);
          dp = fmaf(dOs[i * st + c], Vs[j * st + c], dp);
        }
        s = s * scale + (mask_value(mode, i, j, L, w_h, obj) + kb[j]);
        const float p = (r < ncols) ? expf(s - lses[i]) : 0.f;
        const float dm = drop_scale(seed, drop_thresh, inv_keep, blockIdx.x, i, j, L);
        pp[r] = p * dm;                         // dV_j = sum_i (P o M)_ij dO_i
        dsp[r] = p * (dp * dm - Ds[i]);
        if (pim && j0 + r == L - 1 && r < ncols) dru += dsp[r];
      }
      *reinterpret_cast<float4*>(ps + (i - ibeg) * kAttRows) = p4;
      *reinterpret_cast<float4*>(dss + (i - ibeg) * kAttRows) = ds4;
    }
    __syncwarp();
    for (int c = lane; c < dh; c += 32) {
      float ak[kAttRows] = {0.f, 0.f, 0.f, 0.f}, av[kAttRows] = {0.f, 0.f, 0.f, 0.f};
      for (int i = ibeg; i < L; ++i) {
        const float qv = Qs[i * st + c], dov = dOs[i * st + c];
        const float4 p4 = *reinterpret_cast<const float4*>(ps + (i - ibeg) * kAttRows);
        const float4 d4 = *reinterpret_cast<const float4*>(dss + (i - ibeg) * kAttRows);
        ak[0] = fmaf(d4.x, qv, ak[0]); ak[1] = fmaf(d4.y, qv, ak[1]);
        ak[2] = fmaf(d4.z, qv, ak[2]); ak[3] = fmaf(d4.w, qv, ak[3]);
        av[0] = fmaf(p4.x, dov, av[0]); av[1] = fmaf(p4.y, dov, av[1]);
        av[2] = fmaf(p4.z, dov, av[2]); av[3] = fmaf(p4.w, dov, av[3]);
      }
#pragma unroll
      for (int r = 0; r < kAttRows; ++r)
        if (r < ncols) {
          const int64_t row = (int64_t)b * L + j0 + r;
          d_k[row * ld_k + h * dh + c] = ak[r] * scale;
          d_v[row * ld_v + h * dh + c] = av[r];
        }
    }
    __syncwarp();
  }
  if (pim && d_r_u != nullptr) {
    dru = warp_sum(dru);
    if (lane == 0 && dru != 0.f) atomicAdd(d_r_u + b, w_obj * dru);
  }
}

// ---------------------------------------------------------------------------------------------
// Key-blocked fp32 kernels, for windows whose resident layout above exceeds 227 KB (L <= 2048,
// dh <= 256).  Shared memory holds one block of kBlk keys (or query rows) at a time, so its size does
// not depend on L.  A CTA owns 32 query rows (forward, dQ) or 32 keys (dK/dV); a warp owns 4 of them.
// Key slots: in PIM mode slot 0 is the objective key L-1, which every row sees, and slot s >= 1 is key
// s-1 < L-1; otherwise slot s is key s.  So a row tile visits only the slots of the keys it can see.
// The forward keeps an online softmax (running max, rescaled sum and output); the dropout keep mask is
// drop_scale of the same (b*H+h, i, j), so (p_drop, seed) drops exactly what the resident kernels drop.
// ---------------------------------------------------------------------------------------------
constexpr int kBlk = 64;
constexpr int kBlkRows = kAttWarps * kAttRows;     // 32 rows (or keys) per CTA
constexpr int kBlkMaxDh = 256;
constexpr int kBlkC = kBlkMaxDh / 32;              // head dims per lane

struct BlkSmem {
  int stride;       // odd row stride of the staged [kBlk][dh] blocks
  int off_b, off_kb, off_x, off_warp, warp_floats, total_floats;
};
// forward / dQ: A = K block, B = V block, kb = key padding bias, per warp x^T [dh][4] (+ y^T) and s [kBlk][4]
// dK/dV:        A = Q block, B = dO block, kb = lse, x = D, per warp k^T, v^T [dh][4] and p, ds [kBlk][4]
__host__ __device__ inline BlkSmem blk_smem_layout(int dh, int n_xt, int n_st) {
  BlkSmem s;
  s.stride = dh | 1;
  const int mat = (kBlk * s.stride + 3) & ~3;
  s.off_b = mat;
  s.off_kb = 2 * mat;
  s.off_x = s.off_kb + kBlk;
  s.off_warp = s.off_x + kBlk;
  s.warp_floats = n_xt * dh * kAttRows + n_st * kBlk * kAttRows;
  s.total_floats = s.off_warp + kAttWarps * s.warp_floats;
  return s;
}

__device__ __forceinline__ int slot_key(bool pim, int s, int L) { return pim ? (s == 0 ? L - 1 : s - 1) : s; }

__global__ void __launch_bounds__(kAttWarps * 32)
pim_attn_fwd_blocked_kernel(const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
                            int64_t ld_q, int64_t ld_k, int64_t ld_v, const int64_t* __restrict__ ids,
                            const float* __restrict__ r_u, float w_h, float w_obj, int mode,
                            float* __restrict__ out, float* __restrict__ lse, int L, int H, int dh, int q_row0, int n_q,
                            unsigned long long seed, uint32_t drop_thresh, float inv_keep) {
  extern __shared__ __align__(16) float smem[];
  const BlkSmem lay = blk_smem_layout(dh, 1, 1);
  const int st = lay.stride;
  float* Ks = smem;
  float* Vs = smem + lay.off_b;
  float* kb = smem + lay.off_kb;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* qs = smem + lay.off_warp + warp * lay.warp_floats;      // [dh][4]
  float* ps = qs + dh * kAttRows;                                // [kBlk][4]

  const int b = blockIdx.x / H, h = blockIdx.x % H;
  const int i_beg = q_row0 + blockIdx.y * kBlkRows;
  const int i_end = min(q_row0 + n_q, i_beg + kBlkRows);
  const int i0 = i_beg + warp * kAttRows;
  const int nrows = max(0, min(kAttRows, i_end - i0));
  const int d = H * dh;
  const float scale = 1.0f / sqrtf((float)dh);
  const bool pim = (mode == IRS_MASK_PIM);
  const float obj = pim ? w_obj * r_u[b] : 0.f;
  const int koff = pim ? 1 : 0;
  const int nslots = koff + min(i_end - 1, L - 1 - koff) + 1;    // slots the CTA's last row can see
  const float* kbase = k + (int64_t)b * L * ld_k + h * dh;
  const float* vbase = v + (int64_t)b * L * ld_v + h * dh;

  for (int idx = lane; idx < dh * kAttRows; idx += 32) {
    const int r = idx / dh, c = idx - r * dh;
    qs[c * kAttRows + r] = (r < nrows) ? q[((int64_t)b * L + i0 + r) * ld_q + h * dh + c] : 0.f;
  }
  float m[kAttRows], sum[kAttRows], o[kAttRows][kBlkC];
#pragma unroll
  for (int r = 0; r < kAttRows; ++r) {
    m[r] = -INFINITY; sum[r] = 0.f;
#pragma unroll
    for (int cc = 0; cc < kBlkC; ++cc) o[r][cc] = 0.f;
  }
  for (int s0 = 0; s0 < nslots; s0 += kBlk) {
    const int nb = min(kBlk, nslots - s0);
    __syncthreads();                                            // the previous block is consumed
    for (int idx = threadIdx.x; idx < nb * dh; idx += blockDim.x) {
      const int t = idx / dh, c = idx - t * dh;
      const int j = slot_key(pim, s0 + t, L);
      Ks[t * st + c] = kbase[(int64_t)j * ld_k + c];
      Vs[t * st + c] = vbase[(int64_t)j * ld_v + c];
    }
    for (int t = threadIdx.x; t < nb; t += blockDim.x)
      kb[t] = (mode != IRS_MASK_CAUSAL && ids[(int64_t)b * L + slot_key(pim, s0 + t, L)] == 0) ? -INFINITY : 0.f;
    __syncthreads();
    if (nrows == 0) continue;
    float bm[kAttRows] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
    for (int t = lane; t < nb; t += 32) {
      const int j = slot_key(pim, s0 + t, L);
      const float* kr = Ks + t * st;
      float acc[kAttRows] = {0.f, 0.f, 0.f, 0.f};
      for (int c = 0; c < dh; ++c) {
        const float kv = kr[c];
        const float4 q4 = *reinterpret_cast<const float4*>(qs + c * kAttRows);
        acc[0] = fmaf(q4.x, kv, acc[0]); acc[1] = fmaf(q4.y, kv, acc[1]);
        acc[2] = fmaf(q4.z, kv, acc[2]); acc[3] = fmaf(q4.w, kv, acc[3]);
      }
      float4 s4;
      float* sp = reinterpret_cast<float*>(&s4);
#pragma unroll
      for (int r = 0; r < kAttRows; ++r) {
        sp[r] = acc[r] * scale + (mask_value(mode, i0 + r, j, L, w_h, obj) + kb[t]);
        bm[r] = fmaxf(bm[r], sp[r]);
      }
      *reinterpret_cast<float4*>(ps + t * kAttRows) = s4;
    }
    float alpha[kAttRows];
#pragma unroll
    for (int r = 0; r < kAttRows; ++r) {
      const float mn = fmaxf(m[r], warp_max(bm[r]));
      alpha[r] = (mn == -INFINITY) ? 1.f : expf(m[r] - mn);      // a row that has seen no key yet keeps o = sum = 0
      m[r] = mn;
    }
    __syncwarp();
    float psum[kAttRows] = {0.f, 0.f, 0.f, 0.f};
    for (int t = lane; t < nb; t += 32) {
      const int j = slot_key(pim, s0 + t, L);
      float4 s4 = *reinterpret_cast<const float4*>(ps + t * kAttRows);
      float* sp = reinterpret_cast<float*>(&s4);
#pragma unroll
      for (int r = 0; r < kAttRows; ++r) {
        const float p = (m[r] == -INFINITY) ? 0.f : expf(sp[r] - m[r]);
        psum[r] += p;                          // the softmax normaliser is taken BEFORE dropout
        sp[r] = p * drop_scale(seed, drop_thresh, inv_keep, blockIdx.x, i0 + r, j, L);
      }
      *reinterpret_cast<float4*>(ps + t * kAttRows) = s4;
    }
#pragma unroll
    for (int r = 0; r < kAttRows; ++r) sum[r] = sum[r] * alpha[r] + warp_sum(psum[r]);
    __syncwarp();
#pragma unroll
    for (int cc = 0; cc < kBlkC; ++cc) {
      const int c = lane + 32 * cc;
      if (c < dh) {
        float a0 = o[0][cc] * alpha[0], a1 = o[1][cc] * alpha[1], a2 = o[2][cc] * alpha[2], a3 = o[3][cc] * alpha[3];
        for (int t = 0; t < nb; ++t) {
          const float vv = Vs[t * st + c];
          const float4 p4 = *reinterpret_cast<const float4*>(ps + t * kAttRows);
          a0 = fmaf(p4.x, vv, a0); a1 = fmaf(p4.y, vv, a1); a2 = fmaf(p4.z, vv, a2); a3 = fmaf(p4.w, vv, a3);
        }
        o[0][cc] = a0; o[1][cc] = a1; o[2][cc] = a2; o[3][cc] = a3;
      }
    }
  }
  // a row whose keys are all masked yields NaN, as torch's softmax (and the resident kernel) does
#pragma unroll
  for (int r = 0; r < kAttRows; ++r) {
    if (r >= nrows) continue;
    const bool dead = (m[r] == -INFINITY);
    const float inv = dead ? __int_as_float(0x7fc00000) : 1.0f / sum[r];
#pragma unroll
    for (int cc = 0; cc < kBlkC; ++cc) {
      const int c = lane + 32 * cc;
      if (c < dh) out[((int64_t)b * n_q + (i0 + r - q_row0)) * d + h * dh + c] = o[r][cc] * inv;
    }
    if (lse != nullptr && lane == 0)
      lse[((int64_t)b * H + h) * n_q + (i0 + r - q_row0)] = dead ? __int_as_float(0x7fc00000) : m[r] + logf(sum[r]);
  }
}

// Blocked backward, part 1 (CTA = 32 query rows, key blocks as the forward):
//   dQ_i = scale * sum_j dS_ij K_j,  dS_ij = P_ij (dP_ij M_ij - D_i),  D_i = dO_i . O_i,  P from lse;
//   the objective slot's dS gives  d r_u[b] += w_obj * sum_i dS[i, L-1]  (one atomic per warp).
__global__ void __launch_bounds__(kAttWarps * 32)
pim_attn_bwd_dq_blocked_kernel(const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
                               int64_t ld_q, int64_t ld_k, int64_t ld_v, const int64_t* __restrict__ ids,
                               const float* __restrict__ r_u, float w_h, float w_obj, int mode,
                               const float* __restrict__ o, const float* __restrict__ lse_g, const float* __restrict__ d_o,
                               float* __restrict__ d_q, float* __restrict__ d_r_u, int L, int H, int dh,
                               unsigned long long seed, uint32_t drop_thresh, float inv_keep) {
  extern __shared__ __align__(16) float smem[];
  const BlkSmem lay = blk_smem_layout(dh, 2, 1);
  const int st = lay.stride;
  float* Ks = smem;
  float* Vs = smem + lay.off_b;
  float* kb = smem + lay.off_kb;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* qs = smem + lay.off_warp + warp * lay.warp_floats;      // q^T  [dh][4]
  float* gs = qs + dh * kAttRows;                                // dO^T [dh][4]
  float* dss = gs + dh * kAttRows;                               // dS   [kBlk][4]

  const int b = blockIdx.x / H, h = blockIdx.x % H;
  const int i_beg = blockIdx.y * kBlkRows;
  const int i_end = min(L, i_beg + kBlkRows);
  const int i0 = i_beg + warp * kAttRows;
  const int nrows = max(0, min(kAttRows, i_end - i0));
  const int d = H * dh;
  const float scale = 1.0f / sqrtf((float)dh);
  const bool pim = (mode == IRS_MASK_PIM);
  const float obj = pim ? w_obj * r_u[b] : 0.f;
  const int koff = pim ? 1 : 0;
  const int nslots = koff + min(i_end - 1, L - 1 - koff) + 1;
  const float* kbase = k + (int64_t)b * L * ld_k + h * dh;
  const float* vbase = v + (int64_t)b * L * ld_v + h * dh;

  float D[kAttRows], ls[kAttRows];
#pragma unroll
  for (int r = 0; r < kAttRows; ++r) {
    const int i = min(i0 + r, L - 1);
    const int64_t row = (int64_t)b * L + i;
    float acc = 0.f;
    for (int c = lane; c < dh; c += 32) {
      const float g = d_o[row * d + h * dh + c];
      acc += g * o[row * d + h * dh + c];
      qs[c * kAttRows + r] = (r < nrows) ? q[row * ld_q + h * dh + c] : 0.f;
      gs[c * kAttRows + r] = (r < nrows) ? g : 0.f;
    }
    D[r] = warp_sum(acc);
    ls[r] = lse_g[((int64_t)b * H + h) * L + i];
  }
  float dq[kAttRows][kBlkC];
#pragma unroll
  for (int r = 0; r < kAttRows; ++r)
#pragma unroll
    for (int cc = 0; cc < kBlkC; ++cc) dq[r][cc] = 0.f;
  float dru = 0.f;
  for (int s0 = 0; s0 < nslots; s0 += kBlk) {
    const int nb = min(kBlk, nslots - s0);
    __syncthreads();
    for (int idx = threadIdx.x; idx < nb * dh; idx += blockDim.x) {
      const int t = idx / dh, c = idx - t * dh;
      const int j = slot_key(pim, s0 + t, L);
      Ks[t * st + c] = kbase[(int64_t)j * ld_k + c];
      Vs[t * st + c] = vbase[(int64_t)j * ld_v + c];
    }
    for (int t = threadIdx.x; t < nb; t += blockDim.x)
      kb[t] = (mode != IRS_MASK_CAUSAL && ids[(int64_t)b * L + slot_key(pim, s0 + t, L)] == 0) ? -INFINITY : 0.f;
    __syncthreads();
    if (nrows == 0) continue;
    for (int t = lane; t < nb; t += 32) {
      const int j = slot_key(pim, s0 + t, L);
      float s[kAttRows] = {0.f, 0.f, 0.f, 0.f}, dp[kAttRows] = {0.f, 0.f, 0.f, 0.f};
      for (int c = 0; c < dh; ++c) {
        const float kv = Ks[t * st + c], vv = Vs[t * st + c];
        const float4 q4 = *reinterpret_cast<const float4*>(qs + c * kAttRows);
        const float4 g4 = *reinterpret_cast<const float4*>(gs + c * kAttRows);
        s[0] = fmaf(q4.x, kv, s[0]); s[1] = fmaf(q4.y, kv, s[1]); s[2] = fmaf(q4.z, kv, s[2]); s[3] = fmaf(q4.w, kv, s[3]);
        dp[0] = fmaf(g4.x, vv, dp[0]); dp[1] = fmaf(g4.y, vv, dp[1]); dp[2] = fmaf(g4.z, vv, dp[2]); dp[3] = fmaf(g4.w, vv, dp[3]);
      }
      float4 ds4;
      float* dsp = reinterpret_cast<float*>(&ds4);
#pragma unroll
      for (int r = 0; r < kAttRows; ++r) {
        const float sc = s[r] * scale + (mask_value(mode, i0 + r, j, L, w_h, obj) + kb[t]);
        const float p = (r < nrows) ? expf(sc - ls[r]) : 0.f;
        dsp[r] = (r < nrows) ? p * (dp[r] * drop_scale(seed, drop_thresh, inv_keep, blockIdx.x, i0 + r, j, L) - D[r]) : 0.f;
      }
      if (pim && s0 + t == 0) dru += (dsp[0] + dsp[1]) + (dsp[2] + dsp[3]);
      *reinterpret_cast<float4*>(dss + t * kAttRows) = ds4;
    }
    __syncwarp();
#pragma unroll
    for (int cc = 0; cc < kBlkC; ++cc) {
      const int c = lane + 32 * cc;
      if (c < dh) {
        float a0 = dq[0][cc], a1 = dq[1][cc], a2 = dq[2][cc], a3 = dq[3][cc];
        for (int t = 0; t < nb; ++t) {
          const float kv = Ks[t * st + c];
          const float4 d4 = *reinterpret_cast<const float4*>(dss + t * kAttRows);
          a0 = fmaf(d4.x, kv, a0); a1 = fmaf(d4.y, kv, a1); a2 = fmaf(d4.z, kv, a2); a3 = fmaf(d4.w, kv, a3);
        }
        dq[0][cc] = a0; dq[1][cc] = a1; dq[2][cc] = a2; dq[3][cc] = a3;
      }
    }
    __syncwarp();
  }
#pragma unroll
  for (int r = 0; r < kAttRows; ++r) {
    if (r >= nrows) continue;
#pragma unroll
    for (int cc = 0; cc < kBlkC; ++cc) {
      const int c = lane + 32 * cc;
      if (c < dh) d_q[((int64_t)b * L + i0 + r) * ld_q + h * dh + c] = dq[r][cc] * scale;
    }
  }
  if (pim && d_r_u != nullptr) {
    dru = warp_sum(dru);
    if (lane == 0 && dru != 0.f) atomicAdd(d_r_u + b, w_obj * dru);
  }
}

// Blocked backward, part 2 (CTA = 32 keys, blocks of kBlk query rows staged in turn; a key's rows are i >= j,
// or all rows for the objective key in PIM mode):  dV_j = sum_i (P o M)_ij dO_i,  dK_j = scale * sum_i dS_ij Q_i.
__global__ void __launch_bounds__(kAttWarps * 32, 1)     // 2 x 4 x 8 accumulators per lane: give ptxas the registers
pim_attn_bwd_dkv_blocked_kernel(const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
                                int64_t ld_q, int64_t ld_k, int64_t ld_v, const int64_t* __restrict__ ids,
                                const float* __restrict__ r_u, float w_h, float w_obj, int mode,
                                const float* __restrict__ o, const float* __restrict__ lse_g, const float* __restrict__ d_o,
                                float* __restrict__ d_k, float* __restrict__ d_v, int L, int H, int dh,
                                unsigned long long seed, uint32_t drop_thresh, float inv_keep) {
  extern __shared__ __align__(16) float smem[];
  const BlkSmem lay = blk_smem_layout(dh, 2, 2);
  const int st = lay.stride;
  float* Qs = smem;
  float* Gs = smem + lay.off_b;                                  // dO rows
  float* lses = smem + lay.off_kb;
  float* Ds = smem + lay.off_x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* ks = smem + lay.off_warp + warp * lay.warp_floats;      // k^T [dh][4]
  float* vs = ks + dh * kAttRows;                                // v^T [dh][4]
  float* ps = vs + dh * kAttRows;                                // P o M [kBlk][4]
  float* dss = ps + kBlk * kAttRows;                             // dS    [kBlk][4]

  const int b = blockIdx.x / H, h = blockIdx.x % H;
  const int j_beg = blockIdx.y * kBlkRows;
  const int j_end = min(L, j_beg + kBlkRows);
  const int j0 = j_beg + warp * kAttRows;
  const int ncols = max(0, min(kAttRows, j_end - j0));
  const int d = H * dh;
  const float scale = 1.0f / sqrtf((float)dh);
  const bool pim = (mode == IRS_MASK_PIM);
  const float obj = pim ? w_obj * r_u[b] : 0.f;
  const int ibeg = (pim && j_end == L) ? 0 : j_beg;

  float kbias[kAttRows];
#pragma unroll
  for (int r = 0; r < kAttRows; ++r) {
    const int j = min(j0 + r, L - 1);
    const int64_t row = (int64_t)b * L + j;
    for (int c = lane; c < dh; c += 32) {
      ks[c * kAttRows + r] = (r < ncols) ? k[row * ld_k + h * dh + c] : 0.f;
      vs[c * kAttRows + r] = (r < ncols) ? v[row * ld_v + h * dh + c] : 0.f;
    }
    kbias[r] = (mode != IRS_MASK_CAUSAL && ids[row] == 0) ? -INFINITY : 0.f;
  }
  float dk[kAttRows][kBlkC], dv[kAttRows][kBlkC];
#pragma unroll
  for (int r = 0; r < kAttRows; ++r)
#pragma unroll
    for (int cc = 0; cc < kBlkC; ++cc) { dk[r][cc] = 0.f; dv[r][cc] = 0.f; }
  for (int r0 = ibeg; r0 < L; r0 += kBlk) {
    const int nr = min(kBlk, L - r0);
    __syncthreads();
    for (int idx = threadIdx.x; idx < nr * dh; idx += blockDim.x) {
      const int t = idx / dh, c = idx - t * dh;
      const int64_t row = (int64_t)b * L + r0 + t;
      Qs[t * st + c] = q[row * ld_q + h * dh + c];
      Gs[t * st + c] = d_o[row * d + h * dh + c];
    }
    for (int t = threadIdx.x; t < nr; t += blockDim.x) lses[t] = lse_g[((int64_t)b * H + h) * L + r0 + t];
    for (int t = warp; t < nr; t += kAttWarps) {                 // D_i = dO_i . O_i
      const int64_t row = (int64_t)b * L + r0 + t;
      float acc = 0.f;
      for (int c = lane; c < dh; c += 32) acc += d_o[row * d + h * dh + c] * o[row * d + h * dh + c];
      acc = warp_sum(acc);
      if (lane == 0) Ds[t] = acc;
    }
    __syncthreads();
    if (ncols == 0) continue;
    for (int t = lane; t < nr; t += 32) {
      const int i = r0 + t;
      float s[kAttRows] = {0.f, 0.f, 0.f, 0.f}, dp[kAttRows] = {0.f, 0.f, 0.f, 0.f};
      for (int c = 0; c < dh; ++c) {
        const float qv = Qs[t * st + c], gv = Gs[t * st + c];
        const float4 k4 = *reinterpret_cast<const float4*>(ks + c * kAttRows);
        const float4 v4 = *reinterpret_cast<const float4*>(vs + c * kAttRows);
        s[0] = fmaf(qv, k4.x, s[0]); s[1] = fmaf(qv, k4.y, s[1]); s[2] = fmaf(qv, k4.z, s[2]); s[3] = fmaf(qv, k4.w, s[3]);
        dp[0] = fmaf(gv, v4.x, dp[0]); dp[1] = fmaf(gv, v4.y, dp[1]); dp[2] = fmaf(gv, v4.z, dp[2]); dp[3] = fmaf(gv, v4.w, dp[3]);
      }
      float4 p4, ds4;
      float* pp = reinterpret_cast<float*>(&p4);
      float* dsp = reinterpret_cast<float*>(&ds4);
#pragma unroll
      for (int r = 0; r < kAttRows; ++r) {
        const int j = min(j0 + r, L - 1);
        const float sc = s[r] * scale + (mask_value(mode, i, j, L, w_h, obj) + kbias[r]);
        const float p = (r < ncols) ? expf(sc - lses[t]) : 0.f;
        const float dm = drop_scale(seed, drop_thresh, inv_keep, blockIdx.x, i, j, L);
        pp[r] = p * dm;
        dsp[r] = p * (dp[r] * dm - Ds[t]);
      }
      *reinterpret_cast<float4*>(ps + t * kAttRows) = p4;
      *reinterpret_cast<float4*>(dss + t * kAttRows) = ds4;
    }
    __syncwarp();
#pragma unroll
    for (int cc = 0; cc < kBlkC; ++cc) {
      const int c = lane + 32 * cc;
      if (c < dh) {
        float k0 = dk[0][cc], k1 = dk[1][cc], k2 = dk[2][cc], k3 = dk[3][cc];
        float v0 = dv[0][cc], v1 = dv[1][cc], v2 = dv[2][cc], v3 = dv[3][cc];
        for (int t = 0; t < nr; ++t) {
          const float qv = Qs[t * st + c], gv = Gs[t * st + c];
          const float4 p4 = *reinterpret_cast<const float4*>(ps + t * kAttRows);
          const float4 d4 = *reinterpret_cast<const float4*>(dss + t * kAttRows);
          k0 = fmaf(d4.x, qv, k0); k1 = fmaf(d4.y, qv, k1); k2 = fmaf(d4.z, qv, k2); k3 = fmaf(d4.w, qv, k3);
          v0 = fmaf(p4.x, gv, v0); v1 = fmaf(p4.y, gv, v1); v2 = fmaf(p4.z, gv, v2); v3 = fmaf(p4.w, gv, v3);
        }
        dk[0][cc] = k0; dk[1][cc] = k1; dk[2][cc] = k2; dk[3][cc] = k3;
        dv[0][cc] = v0; dv[1][cc] = v1; dv[2][cc] = v2; dv[3][cc] = v3;
      }
    }
    __syncwarp();
  }
#pragma unroll
  for (int r = 0; r < kAttRows; ++r) {
    if (r >= ncols) continue;
    const int64_t row = (int64_t)b * L + j0 + r;
#pragma unroll
    for (int cc = 0; cc < kBlkC; ++cc) {
      const int c = lane + 32 * cc;
      if (c < dh) {
        d_k[row * ld_k + h * dh + c] = dk[r][cc] * scale;
        d_v[row * ld_v + h * dh + c] = dv[r][cc];
      }
    }
  }
}

}  // namespace irs

static int attn_check(const float* q, const float* k, const float* v, const int64_t* ids, const float* r_u,
                      int mode, int B, int L, int H, int dh) {
  if (!q || !k || !v) return IRS_E_BADARG;
  if (B <= 0 || L <= 0 || H <= 0 || dh <= 0) return IRS_E_BADARG;
  if (mode < 0 || mode > 2) return IRS_E_BADARG;
  if (mode != IRS_MASK_CAUSAL && !ids) return IRS_E_BADARG;
  if (mode == IRS_MASK_PIM && !r_u) return IRS_E_BADARG;
  return 0;
}

static int attn_drop_args(float p_drop, uint32_t* thresh, float* inv_keep) {
  if (!(p_drop >= 0.f) || p_drop >= 1.f) return IRS_E_BADARG;
  *thresh = p_drop > 0.f ? (uint32_t)((double)p_drop * 4294967296.0) : 0u;
  *inv_keep = 1.0f / (1.0f - p_drop);
  return 0;
}

// The routed entry points stream the window in key blocks when it does not fit on chip; the _blocked ones always do.
static int attn_fwd(bool blocked, const float* q, const float* k, const float* v, int64_t ld_q, int64_t ld_k, int64_t ld_v,
                    const int64_t* ids, const float* r_u, float w_h, float w_obj, int mode,
                    float* out, float* lse, int B, int L, int H, int dh, int q_row0, int n_q,
                    float p_drop, unsigned long long seed, void* stream) {
  int rc = attn_check(q, k, v, ids, r_u, mode, B, L, H, dh);
  if (rc) return rc;
  if (!out || q_row0 < 0 || n_q <= 0 || q_row0 + n_q > L) return IRS_E_BADARG;
  uint32_t drop_thresh;
  float inv_keep;
  if ((rc = attn_drop_args(p_drop, &drop_thresh, &inv_keep))) return rc;
  if (L > IRS_ATTN_MAX_L) return IRS_E_SHAPE;
  const cudaStream_t s = (cudaStream_t)stream;
  const size_t bytes = (size_t)irs::attn_smem_layout(L, dh).total_floats * sizeof(float);
  if (blocked || bytes > 227 * 1024) {
    if (dh > irs::kBlkMaxDh) return IRS_E_SHAPE;
    const size_t bytes_blk = (size_t)irs::blk_smem_layout(dh, 1, 1).total_floats * sizeof(float);
    IRS_CUDA(irs::opt_in_smem(irs::pim_attn_fwd_blocked_kernel, bytes_blk));
    dim3 grid((unsigned)(B * H), (unsigned)((n_q + irs::kBlkRows - 1) / irs::kBlkRows));
    irs::pim_attn_fwd_blocked_kernel<<<grid, irs::kAttWarps * 32, bytes_blk, s>>>(
        q, k, v, ld_q, ld_k, ld_v, ids, r_u, w_h, w_obj, mode, out, lse, L, H, dh, q_row0, n_q, seed, drop_thresh, inv_keep);
    IRS_LAUNCHED();
    return 0;
  }
  IRS_CUDA(irs::opt_in_smem(irs::pim_attn_fwd_kernel, bytes));
  // Enough CTAs to fill the machine: split the query rows when B*H alone is too few.
  int chunks = 1;
  const int per_pass = irs::kAttWarps * irs::kAttRows;
  while ((int64_t)B * H * chunks < 2 * irs::kNumSMs && (n_q + chunks - 1) / chunks > per_pass) chunks *= 2;
  int rows_per_cta = (n_q + chunks - 1) / chunks;
  rows_per_cta = ((rows_per_cta + irs::kAttRows - 1) / irs::kAttRows) * irs::kAttRows;
  chunks = (n_q + rows_per_cta - 1) / rows_per_cta;
  dim3 grid((unsigned)(B * H), (unsigned)chunks);
  irs::pim_attn_fwd_kernel<<<grid, irs::kAttWarps * 32, bytes, s>>>(
      q, k, v, ld_q, ld_k, ld_v, ids, r_u, w_h, w_obj, mode, out, lse, L, H, dh, q_row0, n_q, rows_per_cta,
      seed, drop_thresh, inv_keep);
  IRS_LAUNCHED();
  return 0;
}

static int attn_bwd(bool blocked, const float* q, const float* k, const float* v, int64_t ld_q, int64_t ld_k, int64_t ld_v,
                    const int64_t* ids, const float* r_u, float w_h, float w_obj, int mode,
                    const float* out, const float* lse, const float* d_out,
                    float* d_q, float* d_k, float* d_v, float* d_r_u,
                    int B, int L, int H, int dh, float p_drop, unsigned long long seed, void* stream) {
  int rc = attn_check(q, k, v, ids, r_u, mode, B, L, H, dh);
  if (rc) return rc;
  if (!out || !lse || !d_out || !d_q || !d_k || !d_v) return IRS_E_BADARG;
  uint32_t drop_thresh;
  float inv_keep;
  if ((rc = attn_drop_args(p_drop, &drop_thresh, &inv_keep))) return rc;
  if (L > IRS_ATTN_MAX_L) return IRS_E_SHAPE;
  const cudaStream_t s = (cudaStream_t)stream;
  const size_t bytes = (size_t)irs::attn_bwd_smem_layout(L, dh).total_floats * sizeof(float);
  if (blocked || bytes > 227 * 1024) {
    if (dh > irs::kBlkMaxDh) return IRS_E_SHAPE;
    const size_t bytes_q = (size_t)irs::blk_smem_layout(dh, 2, 1).total_floats * sizeof(float);
    const size_t bytes_kv = (size_t)irs::blk_smem_layout(dh, 2, 2).total_floats * sizeof(float);
    IRS_CUDA(irs::opt_in_smem(irs::pim_attn_bwd_dq_blocked_kernel, bytes_q));
    IRS_CUDA(irs::opt_in_smem(irs::pim_attn_bwd_dkv_blocked_kernel, bytes_kv));
    dim3 grid((unsigned)(B * H), (unsigned)((L + irs::kBlkRows - 1) / irs::kBlkRows));
    irs::pim_attn_bwd_dq_blocked_kernel<<<grid, irs::kAttWarps * 32, bytes_q, s>>>(
        q, k, v, ld_q, ld_k, ld_v, ids, r_u, w_h, w_obj, mode, out, lse, d_out, d_q, d_r_u, L, H, dh, seed, drop_thresh, inv_keep);
    IRS_LAUNCHED();
    irs::pim_attn_bwd_dkv_blocked_kernel<<<grid, irs::kAttWarps * 32, bytes_kv, s>>>(
        q, k, v, ld_q, ld_k, ld_v, ids, r_u, w_h, w_obj, mode, out, lse, d_out, d_k, d_v, L, H, dh, seed, drop_thresh, inv_keep);
    IRS_LAUNCHED();
    return 0;
  }
  IRS_CUDA(irs::opt_in_smem(irs::pim_attn_bwd_kernel, bytes));
  irs::pim_attn_bwd_kernel<<<(unsigned)(B * H), irs::kAttWarps * 32, bytes, s>>>(
      q, k, v, ld_q, ld_k, ld_v, ids, r_u, w_h, w_obj, mode, out, lse, d_out, d_q, d_k, d_v, d_r_u, L, H, dh,
      seed, drop_thresh, inv_keep);
  IRS_LAUNCHED();
  return 0;
}

extern "C" int irs_pim_attn_fwd(const float* q, const float* k, const float* v, int64_t ld_q, int64_t ld_k, int64_t ld_v,
                                const int64_t* ids, const float* r_u, float w_h, float w_obj, int mode,
                                float* out, float* lse, int B, int L, int H, int dh, int q_row0, int n_q,
                                float p_drop, unsigned long long seed, void* stream) {
  return attn_fwd(false, q, k, v, ld_q, ld_k, ld_v, ids, r_u, w_h, w_obj, mode, out, lse, B, L, H, dh, q_row0, n_q,
                  p_drop, seed, stream);
}

extern "C" int irs_pim_attn_fwd_blocked(const float* q, const float* k, const float* v, int64_t ld_q, int64_t ld_k, int64_t ld_v,
                                        const int64_t* ids, const float* r_u, float w_h, float w_obj, int mode,
                                        float* out, float* lse, int B, int L, int H, int dh, int q_row0, int n_q,
                                        float p_drop, unsigned long long seed, void* stream) {
  return attn_fwd(true, q, k, v, ld_q, ld_k, ld_v, ids, r_u, w_h, w_obj, mode, out, lse, B, L, H, dh, q_row0, n_q,
                  p_drop, seed, stream);
}

extern "C" int irs_pim_attn_bwd(const float* q, const float* k, const float* v, int64_t ld_q, int64_t ld_k, int64_t ld_v,
                                const int64_t* ids, const float* r_u, float w_h, float w_obj, int mode,
                                const float* out, const float* lse, const float* d_out,
                                float* d_q, float* d_k, float* d_v, float* d_r_u,
                                int B, int L, int H, int dh, float p_drop, unsigned long long seed, void* stream) {
  return attn_bwd(false, q, k, v, ld_q, ld_k, ld_v, ids, r_u, w_h, w_obj, mode, out, lse, d_out, d_q, d_k, d_v, d_r_u,
                  B, L, H, dh, p_drop, seed, stream);
}

extern "C" int irs_pim_attn_bwd_blocked(const float* q, const float* k, const float* v, int64_t ld_q, int64_t ld_k, int64_t ld_v,
                                        const int64_t* ids, const float* r_u, float w_h, float w_obj, int mode,
                                        const float* out, const float* lse, const float* d_out,
                                        float* d_q, float* d_k, float* d_v, float* d_r_u,
                                        int B, int L, int H, int dh, float p_drop, unsigned long long seed, void* stream) {
  return attn_bwd(true, q, k, v, ld_q, ld_k, ld_v, ids, r_u, w_h, w_obj, mode, out, lse, d_out, d_q, d_k, d_v, d_r_u,
                  B, L, H, dh, p_drop, seed, stream);
}
