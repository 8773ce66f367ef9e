// K5b: backward of softmax cross-entropy over the catalog with the logits recomputed tile by tile
// (the [M,N] probability matrix never exists: 409 GB at cfg4).  fp32 CUDA-core version.
//   g[m,j] = (exp(s[m,j] - lse[m]) - [j == target[m]]) * gscale
//   d_h = g W          (kernel OWNER_M: a CTA owns 128 rows of h and sweeps the catalog)
//   d_W += g^T h, d_bias += colsum(g)   (kernel OWNER_N: a CTA owns 128 catalog rows and sweeps M)
// Each owner accumulates its 128 x d output tile in registers (one 128-row tile at a time, then into the
// running sum), so there are no global atomics and the result is deterministic.  Any of d_h, d_W, d_bias may be NULL.
//   reference: autograd of self.project + nn.CrossEntropyLoss, model/influentialRS.py:214,303,307.
#include "common.cuh"

namespace irs {

namespace ce {
constexpr int BM = 128, BN = 128, BK = 16, kThreads = 256, kPad = 4;
constexpr int DMAX = 128;

struct Smem {
  float As[2][BK][BM + kPad];
  float Bs[2][BK][BN + kPad];
  float Gs[128][128 + kPad];      // reduction-major copy of the gradient tile
  float Bt[128][DMAX + kPad];     // second-GEMM B operand: 128 rows of W (OWNER_M) or h (OWNER_N)
  float colsum[128];
};
}  // namespace ce

template <bool OWNER_M>
__global__ void __launch_bounds__(ce::kThreads, 1)
ce_bwd_kernel(const float* __restrict__ h, int64_t ld_h, const float* __restrict__ W, const float* __restrict__ bias,
              const int64_t* __restrict__ target, const float* __restrict__ lse, float gscale,
              float* __restrict__ d_h, float* __restrict__ d_W, float* __restrict__ d_bias,
              int M, int64_t N, int d) {
  using namespace ce;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  int rm[8], cn[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    rm[i] = (i < 4) ? ty * 4 + i : 64 + ty * 4 + (i - 4);
    cn[i] = (i < 4) ? tx * 4 + i : 64 + tx * 4 + (i - 4);
  }
  const int64_t m_tiles = ceil_div(M, BM), n_tiles = ceil_div(N, BN);
  const int64_t own0 = (int64_t)blockIdx.x * 128;
  const int64_t sweep_tiles = OWNER_M ? n_tiles : m_tiles;
  const int lrow = tid >> 2, lk = (tid & 3) * 4;
  const int k_slabs = (d + BK - 1) / BK;

  float acc2[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc2[i][j] = 0.f;
  if (tid < 128) sm.colsum[tid] = 0.f;

  for (int64_t sw = 0; sw < sweep_tiles; ++sw) {
    const int64_t m0 = OWNER_M ? own0 : sw * BM;
    const int64_t n0 = OWNER_M ? sw * BN : own0;
    // ---- S tile = h[m0:,:] W[n0:,:]^T  (same FMA chain as the forward scorer)
    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    float4 ra[2], rb[2];
    auto load_slab = [&](int k0) {
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        const int r = lrow + 64 * half;
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
        float* ap = reinterpret_cast<float*>(&a);
        float* bp = reinterpret_cast<float*>(&b);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          if (m0 + r < M && k0 + lk + e < d) ap[e] = h[(m0 + r) * ld_h + k0 + lk + e];
          if (n0 + r < N && k0 + lk + e < d) bp[e] = __ldg(W + (n0 + r) * d + k0 + lk + e);
        }
        ra[half] = a; rb[half] = b;
      }
    };
    auto store_slab = [&](int buf) {
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        const int r = lrow + 64 * half;
        sm.As[buf][lk + 0][r] = ra[half].x; sm.As[buf][lk + 1][r] = ra[half].y;
        sm.As[buf][lk + 2][r] = ra[half].z; sm.As[buf][lk + 3][r] = ra[half].w;
        sm.Bs[buf][lk + 0][r] = rb[half].x; sm.Bs[buf][lk + 1][r] = rb[half].y;
        sm.Bs[buf][lk + 2][r] = rb[half].z; sm.Bs[buf][lk + 3][r] = rb[half].w;
      }
    };
    load_slab(0);
    store_slab(0);
    // stage the second-GEMM operand tile (natural layout, zero padded)
    for (int idx = tid; idx < 128 * DMAX; idx += kThreads) {
      const int r = idx / DMAX, c = idx - r * DMAX;
      float v = 0.f;
      if (c < d) {
        if (OWNER_M) { if (n0 + r < N) v = __ldg(W + (n0 + r) * d + c); }
        else { if (m0 + r < M) v = h[(m0 + r) * ld_h + c]; }
      }
      sm.Bt[r][c] = v;
    }
    __syncthreads();
    for (int ks = 0; ks < k_slabs; ++ks) {
      const int buf = ks & 1;
      if (ks + 1 < k_slabs) load_slab((ks + 1) * BK);
#pragma unroll
      for (int kk = 0; kk < BK; ++kk) {
        const float4 a0 = *reinterpret_cast<const float4*>(&sm.As[buf][kk][ty * 4]);
        const float4 a1 = *reinterpret_cast<const float4*>(&sm.As[buf][kk][64 + ty * 4]);
        const float4 b0 = *reinterpret_cast<const float4*>(&sm.Bs[buf][kk][tx * 4]);
        const float4 b1 = *reinterpret_cast<const float4*>(&sm.Bs[buf][kk][64 + tx * 4]);
        const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
        const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
      }
      if (ks + 1 < k_slabs) store_slab(buf ^ 1);
      __syncthreads();
    }
    // ---- gradient tile into shared memory, reduction-major
    float csum[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int64_t m = m0 + rm[i];
      const bool row_ok = m < M;
      const int64_t tgt = row_ok ? target[m] : -1;
      const float l = (row_ok && tgt >= 0) ? lse[m] : 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int64_t n = n0 + cn[j];
        float g = 0.f;
        if (row_ok && tgt >= 0 && n < N) {
          const float s = acc[i][j] + (bias ? __ldg(bias + n) : 0.f);
          g = (expf(s - l) - (n == tgt ? 1.f : 0.f)) * gscale;
        }
        if (OWNER_M) sm.Gs[cn[j]][rm[i]] = g; else sm.Gs[rm[i]][cn[j]] = g;
        csum[j] += g;
      }
    }
    if (!OWNER_M) {
#pragma unroll
      for (int j = 0; j < 8; ++j) atomicAdd(&sm.colsum[cn[j]], csum[j]);
    }
    __syncthreads();
    // ---- second GEMM: acc2[owner, c] += sum_r Gs[r][owner] * Bt[r][c], the tile summed on its own first: added one by one
    // to a running sum over 500k items, the terms of tail items (p ~ 1e-6 and below) fall under half an ulp of it and are
    // rounded away -- the same way every time, ~1e-3 of |d_h| on a catalog whose embeddings share a direction
    float part[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) part[i][j] = 0.f;
#pragma unroll 4
    for (int r = 0; r < 128; ++r) {
      const float4 a0 = *reinterpret_cast<const float4*>(&sm.Gs[r][ty * 4]);
      const float4 a1 = *reinterpret_cast<const float4*>(&sm.Gs[r][64 + ty * 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&sm.Bt[r][tx * 4]);
      const float4 b1 = *reinterpret_cast<const float4*>(&sm.Bt[r][64 + tx * 4]);
      const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) part[i][j] = fmaf(a[i], b[j], part[i][j]);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc2[i][j] += part[i][j];
    __syncthreads();
  }

  // ---- write the owner tile
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int64_t o = own0 + rm[i];
    if (o >= (OWNER_M ? (int64_t)M : N)) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = cn[j];
      if (c >= d) continue;
      if (OWNER_M) d_h[o * d + c] = acc2[i][j];
      else if (d_W != nullptr) d_W[o * d + c] += acc2[i][j];
    }
  }
  if (!OWNER_M && d_bias != nullptr && tid < 128 && own0 + tid < N) d_bias[own0 + tid] += sm.colsum[tid];
}

}  // namespace irs

extern "C" int irs_score_ce_bwd(const float* h, int64_t ld_h, const float* W, const float* bias,
                                const int64_t* target, const float* lse, float gscale,
                                float* d_h, float* d_W, float* d_bias, int M, int64_t N, int d, void* stream) {
  using namespace irs;
  if (!h || !W || !target || !lse) return IRS_E_BADARG;
  if (M <= 0 || N <= 0 || d <= 0) return IRS_E_BADARG;
  if (d > ce::DMAX) return IRS_E_SHAPE;
  cudaStream_t s = (cudaStream_t)stream;
  const size_t bytes = sizeof(ce::Smem);
  static bool configured = false;
  if (!configured) {
    IRS_CUDA(cudaFuncSetAttribute(ce_bwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    IRS_CUDA(cudaFuncSetAttribute(ce_bwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    configured = true;
  }
  if (d_h != nullptr) {
    ce_bwd_kernel<true><<<(unsigned)ceil_div(M, 128), ce::kThreads, bytes, s>>>(
        h, ld_h, W, bias, target, lse, gscale, d_h, nullptr, nullptr, M, N, d);
    IRS_LAUNCHED();
  }
  if (d_W != nullptr || d_bias != nullptr) {             // d_bias comes out of the d_W pass
    ce_bwd_kernel<false><<<(unsigned)ceil_div(N, 128), ce::kThreads, bytes, s>>>(
        h, ld_h, W, bias, target, lse, gscale, nullptr, d_W, d_bias, M, N, d);
    IRS_LAUNCHED();
  }
  return 0;
}
