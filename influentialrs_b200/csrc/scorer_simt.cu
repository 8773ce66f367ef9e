// K5 (fp32 CUDA-core core): full-catalog scoring  s = h W^T + bias  fused with its consumers, so
// the [M,N] logits never reach HBM.  One 128x128x16 register-blocked tile engine, four epilogues:
//   MODE_MAX     per-(row, slice) best (score, column) under the exclusion lists   -> arg-max / threshold
//   MODE_COLLECT append every non-excluded (score, column) >= the row's threshold  -> exact top-k
//   MODE_LSE     online log-sum-exp per row + gather of selected logits            -> CE / log-prob
//   MODE_RANK    count of non-excluded items ahead of the label                    -> rank, Hit@k, MRR
// The dot product is a sequential fp32 FMA chain over k (same order in every mode and in the label
// prologue), so a score is bit-identical wherever it is recomputed.
//   reference: model/influentialRS.py:214 (project), :418-429 (softmax/topk/filter), :294-303 (CE),
//   :375-388 (sort/rank); model/evaluator.py:194-205,266-286; model/sas.py:224,380-386;
//   model/caser.py:176-179,291-298.
#include "scorer.cuh"

namespace irs {

constexpr int BM = 128, BN = 128, BK = 16;
constexpr int kThreads = 256;
constexpr int kPad = 4;   // smem row padding (floats)

template <int MODE>
__global__ void __launch_bounds__(kThreads)
score_simt_kernel(const ScoreParams p) {
  __shared__ __align__(16) float As[2][BK][BM + kPad];
  __shared__ __align__(16) float Bs[2][BK][BN + kPad];
  __shared__ uint32_t excl_bits[BM][BN / 32];
  __shared__ int excl_ptr[BM];
  __shared__ int label_excluded[BM];

  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int m_tile = blockIdx.x % p.m_tiles;
  const int split = blockIdx.x / p.m_tiles;
  const int m0 = m_tile * BM;
  const int64_t tile_begin = (int64_t)split * p.tiles_per_split;
  const int64_t tile_end = min(tile_begin + p.tiles_per_split, p.n_tiles);
  const bool use_excl = (p.excl_sorted != nullptr);

  // rows / cols owned by this thread inside a tile
  int rm[8], cn[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    rm[i] = (i < 4) ? ty * 4 + i : 64 + ty * 4 + (i - 4);
    cn[i] = (i < 4) ? tx * 4 + i : 64 + tx * 4 + (i - 4);
  }

  if (tid < BM) { excl_ptr[tid] = 0; label_excluded[tid] = 0; }
  if (use_excl && tid < BM && m0 + tid < p.M && tile_begin > 0) {
    // skip the part of the sorted list that lies before this split's first column
    const int32_t* lst = p.excl_sorted + (int64_t)(m0 + tid) * p.Lx;
    const int cnt = p.excl_count[m0 + tid];
    const int64_t first = tile_begin * BN;
    int lo = 0, hi = cnt;
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (lst[mid] < first) lo = mid + 1; else hi = mid; }
    excl_ptr[tid] = lo;
  }

  // per-thread epilogue state
  float best_v[8]; int best_c[8];            // MODE_MAX
  float run_m[8], run_s[8];                  // MODE_LSE
  int ahead[8];                              // MODE_RANK
  float thr_v[8]; uint32_t thr_c[8];         // MODE_COLLECT
  float lab_s[8]; int64_t lab_c[8];          // MODE_RANK
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    best_v[i] = -INFINITY; best_c[i] = -1; run_m[i] = -INFINITY; run_s[i] = 0.f; ahead[i] = 0;
    thr_v[i] = INFINITY; thr_c[i] = 0; lab_s[i] = 0.f; lab_c[i] = -1;
    const int m = m0 + rm[i];
    if (m < p.M) {
      if (MODE == MODE_COLLECT) {
        const unsigned long long t = p.thr_keys[m];      // 0 = "no threshold": collect every live column
        thr_v[i] = t ? key_score(t) : -INFINITY;
        thr_c[i] = t ? key_col(t) : 0xffffffffu;
      }
      if (MODE == MODE_RANK) { lab_s[i] = p.label_score[m]; lab_c[i] = p.label[m] - p.item_base; }
    }
  }

  // global -> register staging of one k-slab of the A (h) and B (W) tiles
  const int lrow = tid >> 2, lk = (tid & 3) * 4;     // rows lrow, lrow+64; 4 consecutive k
  float4 ra[2], rb[2];
  auto load_slab = [&](int64_t n0, int k0) {
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      const int r = lrow + 64 * half;
      const int m = m0 + r;
      const int64_t n = n0 + r;
      float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
      if (p.vec_ok) {
        if (m < p.M && k0 + lk < p.d) a = *reinterpret_cast<const float4*>(p.h + (int64_t)m * p.ld_h + k0 + lk);
        if (n < p.N && k0 + lk < p.d) b = __ldg(reinterpret_cast<const float4*>(p.W + n * p.d + k0 + lk));
      } else {
        float* ap = reinterpret_cast<float*>(&a);
        float* bp = reinterpret_cast<float*>(&b);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          if (m < p.M && k0 + lk + e < p.d) ap[e] = p.h[(int64_t)m * p.ld_h + k0 + lk + e];
          if (n < p.N && k0 + lk + e < p.d) bp[e] = __ldg(p.W + n * p.d + k0 + lk + e);
        }
      }
      ra[half] = a; rb[half] = b;
    }
  };
  auto store_slab = [&](int buf) {
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      const int r = lrow + 64 * half;
      As[buf][lk + 0][r] = ra[half].x; As[buf][lk + 1][r] = ra[half].y;
      As[buf][lk + 2][r] = ra[half].z; As[buf][lk + 3][r] = ra[half].w;
      Bs[buf][lk + 0][r] = rb[half].x; Bs[buf][lk + 1][r] = rb[half].y;
      Bs[buf][lk + 2][r] = rb[half].z; Bs[buf][lk + 3][r] = rb[half].w;
    }
  };

  const int k_slabs = (p.d + BK - 1) / BK;

  for (int64_t tile = tile_begin; tile < tile_end; ++tile) {
    const int64_t n0 = tile * BN;
    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

    // exclusion bitmap of this tile (row-owner threads walk their sorted lists once, in order)
    if (use_excl) {
      if (tid < BM) {
#pragma unroll
        for (int w = 0; w < BN / 32; ++w) excl_bits[tid][w] = 0u;
        const int m = m0 + tid;
        if (m < p.M) {
          const int32_t* lst = p.excl_sorted + (int64_t)m * p.Lx;
          const int cnt = p.excl_count[m];
          int ptr = excl_ptr[tid];
          const int64_t lab = (MODE == MODE_RANK) ? (p.label[m] - p.item_base) : -1;
          while (ptr < cnt && lst[ptr] < n0 + BN) {
            const int c = (int)(lst[ptr] - n0);
            if (c >= 0) excl_bits[tid][c >> 5] |= 1u << (c & 31);
            if (lst[ptr] == lab) label_excluded[tid] = 1;
            ++ptr;
          }
          excl_ptr[tid] = ptr;
        }
      }
    }

    load_slab(n0, 0);
    store_slab(0);
    __syncthreads();
    for (int ks = 0; ks < k_slabs; ++ks) {
      const int buf = ks & 1;
      if (ks + 1 < k_slabs) load_slab(n0, (ks + 1) * BK);
#pragma unroll
      for (int kk = 0; kk < BK; ++kk) {
        const float4 a0 = *reinterpret_cast<const float4*>(&As[buf][kk][ty * 4]);
        const float4 a1 = *reinterpret_cast<const float4*>(&As[buf][kk][64 + ty * 4]);
        const float4 b0 = *reinterpret_cast<const float4*>(&Bs[buf][kk][tx * 4]);
        const float4 b1 = *reinterpret_cast<const float4*>(&Bs[buf][kk][64 + tx * 4]);
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

    // ---- epilogue on the register tile
    float bj[8];
    bool col_ok[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int64_t n = n0 + cn[j];
      col_ok[j] = n < p.N;
      bj[j] = (p.bias != nullptr && col_ok[j]) ? __ldg(p.bias + n) : 0.f;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int m = m0 + rm[i];
      if (m >= p.M) continue;
      uint32_t bits_lo = 0u, bits_hi = 0u;
      if (use_excl) {   // columns cn[0..3] live in word tx/8, cn[4..7] in word 2 + tx/8
        bits_lo = excl_bits[rm[i]][tx >> 3] >> ((tx & 7) * 4);
        bits_hi = excl_bits[rm[i]][2 + (tx >> 3)] >> ((tx & 7) * 4);
      }
      float tile_max = -INFINITY;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float s = acc[i][j] + bj[j];
        const bool excluded = ((j < 4 ? bits_lo >> j : bits_hi >> (j - 4)) & 1u) != 0u;
        const bool live = col_ok[j] && !excluded;
        const int64_t n = n0 + cn[j];
        if (MODE == MODE_MAX) {
          // columns are visited in increasing order, so strict '>' keeps the lowest id among ties
          if (live && s > best_v[i]) { best_v[i] = s; best_c[i] = (int)n; }
        } else if (MODE == MODE_COLLECT) {
          if (live && (s > thr_v[i] || (s == thr_v[i] && (uint32_t)n <= thr_c[i]))) {
            const int pos = atomicAdd(p.cand_count + m, 1);
            if (pos < p.cand_cap) p.cand_keys[(int64_t)m * p.cand_cap + pos] = pack_key(s, (uint32_t)n);
          }
        } else if (MODE == MODE_LSE) {
          if (col_ok[j]) tile_max = fmaxf(tile_max, s);
          acc[i][j] = col_ok[j] ? s : -INFINITY;
        } else if (MODE == MODE_RANK) {
          if (live && n != lab_c[i] && (s > lab_s[i] || (s == lab_s[i] && n < lab_c[i]))) ++ahead[i];
        }
      }
      if (MODE == MODE_LSE) {
        if (tile_max > -INFINITY) {
          const float nm = fmaxf(run_m[i], tile_max);
          float add = 0.f;
#pragma unroll
          for (int j = 0; j < 8; ++j) add += expf(acc[i][j] - nm);
          run_s[i] = run_s[i] * expf(run_m[i] - nm) + add;
          run_m[i] = nm;
        }
        for (int t = 0; t < p.n_sel; ++t) {
          const int64_t c = p.sel[(int64_t)m * p.n_sel + t] - p.item_base - n0;
          if (c >= 0 && c < BN) {
            // an id past the catalog but inside its last partial tile keeps the 0.0 it was given (acc is -inf there)
#pragma unroll
            for (int j = 0; j < 8; ++j)
              if (c == cn[j] && col_ok[j]) p.sel_logit[(int64_t)m * p.n_sel + t] = acc[i][j];
          }
        }
      }
    }
    if (use_excl) __syncthreads();   // bitmap is rebuilt next tile
  }

  // ---- cross-thread reduction over the 16 threads (tx) that share each row, then write-out
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int m = m0 + rm[i];
    if (MODE == MODE_MAX) {
      unsigned long long key = (best_c[i] >= 0) ? pack_key(best_v[i], (uint32_t)best_c[i]) : 0ull;
      if (p.slices_per_split == 1) {
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) {
          const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
          key = other > key ? other : key;
        }
        if (tx == 0 && m < p.M) p.slice_keys[(int64_t)m * p.n_slices + split] = key;
      } else if (m < p.M) {
        p.slice_keys[(int64_t)m * p.n_slices + split * 16 + tx] = key;
      }
    } else if (MODE == MODE_LSE) {
      float mm = run_m[i], ss = run_s[i];
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) {
        const float om = __shfl_xor_sync(0xffffffffu, mm, o);
        const float os = __shfl_xor_sync(0xffffffffu, ss, o);
        const float nm = fmaxf(mm, om);
        if (nm > -INFINITY) ss = ss * expf(mm - nm) + os * expf(om - nm);
        mm = nm;
      }
      if (tx == 0 && m < p.M) {
        p.part_max[(int64_t)m * p.n_splits + split] = mm;
        p.part_sum[(int64_t)m * p.n_splits + split] = ss;
      }
    } else if (MODE == MODE_RANK) {
      int c = ahead[i];
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
      if (tx == 0 && m < p.M && c) atomicAdd(p.rank_count + m, c);
    }
  }
  if (MODE == MODE_RANK && use_excl) {
    __syncthreads();
    if (tid < BM && m0 + tid < p.M && label_excluded[tid]) p.rank_excluded[m0 + tid] = 1;
  }
}

int launch_score_simt(int mode, ScoreParams& p, cudaStream_t s) {
  p.m_tiles = (int)ceil_div(p.M, BM);
  p.n_tiles = ceil_div(p.N, BN);
  // grid ~ a whole number of waves of 148 SMs x 2 resident CTAs; adjacent CTAs share the same
  // catalog range (different user tiles) so W streams from HBM once and is re-served by L2.
  const int64_t target = (int64_t)kNumSMs * 2 * 2;
  int64_t splits = target / p.m_tiles;
  if (splits < 1) splits = 1;
  if (splits > p.n_tiles) splits = p.n_tiles;
  if (p.max_splits > 0 && splits > p.max_splits) splits = p.max_splits;
  p.tiles_per_split = ceil_div(p.n_tiles, splits);
  p.n_splits = (int)ceil_div(p.n_tiles, p.tiles_per_split);
  p.vec_ok = ((p.d & 3) == 0) && ((p.ld_h & 3) == 0) && (((uintptr_t)p.h & 15) == 0) && (((uintptr_t)p.W & 15) == 0);
  if (mode == MODE_MAX) p.n_slices = p.n_splits * p.slices_per_split;
  const unsigned grid = (unsigned)(p.m_tiles * p.n_splits);
  switch (mode) {
    case MODE_MAX: score_simt_kernel<MODE_MAX><<<grid, kThreads, 0, s>>>(p); break;
    case MODE_COLLECT: score_simt_kernel<MODE_COLLECT><<<grid, kThreads, 0, s>>>(p); break;
    case MODE_LSE: score_simt_kernel<MODE_LSE><<<grid, kThreads, 0, s>>>(p); break;
    case MODE_RANK: score_simt_kernel<MODE_RANK><<<grid, kThreads, 0, s>>>(p); break;
    default: return IRS_E_BADARG;
  }
  IRS_LAUNCHED();
  return 0;
}

int score_simt_max_splits(int M, int64_t N) {
  const int m_tiles = (int)ceil_div(M, BM);
  const int64_t n_tiles = ceil_div(N, BN);
  int64_t splits = (int64_t)kNumSMs * 2 * 2 / m_tiles;
  if (splits < 1) splits = 1;
  if (splits > n_tiles) splits = n_tiles;
  return (int)splits;
}

}  // namespace irs
