// Selection / finalisation kernels around the fused scorer and the C-ABI entry points that chain
// them: exclusion-list sorting, arg-max / threshold / candidate finalisers, log-sum-exp merge,
// rank finalise, multi-GPU shard merge, device-side window shift.
//   reference call sites are cited on each extern "C" function in include/irs_b200.h.
#include "scorer.cuh"

namespace irs {

// Block-wide bitonic sort of P (power of two) 64-bit keys in shared memory, DESCENDING.
__device__ void block_bitonic_desc(unsigned long long* keys, int P) {
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

__host__ __device__ inline int next_pow2(int x) { int p = 1; while (p < x) p <<= 1; return p; }

// ---- exclusion lists: ids -> sorted int32 columns -------------------------------------------------
__global__ void __launch_bounds__(256)
sort_exclusions_kernel(const int64_t* __restrict__ ids, int M, int Lx, int64_t item_base, int64_t N,
                       int32_t* __restrict__ out_sorted, int32_t* __restrict__ out_count, int P) {
  extern __shared__ unsigned long long sk[];
  __shared__ int s_count;
  const int m = blockIdx.x;
  if (threadIdx.x == 0) s_count = 0;
  for (int t = threadIdx.x; t < P; t += blockDim.x) {
    unsigned long long key = 0ull;                       // invalid sorts last in the descending order
    if (t < Lx) {
      const int64_t c = ids[(int64_t)m * Lx + t] - item_base;
      if (c >= 0 && c < N) key = ~(unsigned long long)c; // descending on ~c  ==  ascending on c
    }
    sk[t] = key;
  }
  block_bitonic_desc(sk, P);
  for (int t = threadIdx.x; t < Lx; t += blockDim.x) {
    const unsigned long long key = sk[t];
    out_sorted[(int64_t)m * Lx + t] = key ? (int32_t)(~key) : 0x7fffffff;
    if (key) atomicAdd(&s_count, 1);
  }
  __syncthreads();
  if (threadIdx.x == 0) out_count[m] = s_count;
}

// ---- exclusion lists: one window step = remove the id that slid out, insert the pick -------------------
// One warp per row.  The list stays sorted (duplicates allowed: a window may hold an id twice, one occurrence goes); ids
// outside this catalog shard [item_base, item_base + N) and PAD (0) are not in the list and are ignored here.
__global__ void __launch_bounds__(256)
exclusions_update_kernel(int32_t* __restrict__ sorted, int32_t* __restrict__ count, const int64_t* __restrict__ removed,
                         int64_t removed_stride, const int64_t* __restrict__ inserted, int M, int Lx, int64_t item_base, int64_t N) {
  extern __shared__ int32_t sh[];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int m = blockIdx.x * (blockDim.x >> 5) + w;
  if (m >= M) return;
  int32_t* buf = sh + (size_t)w * Lx;
  int32_t* row = sorted + (int64_t)m * Lx;
  const int cnt = count[m];
  const int64_t rc64 = removed[(int64_t)m * removed_stride] - item_base;
  const int64_t ic64 = inserted[m] - item_base;
  const bool do_rm = rc64 >= 0 && rc64 < N;
  const bool do_in = ic64 >= 0 && ic64 < N;
  const int32_t rc = (int32_t)rc64, ic = (int32_t)ic64;
  int rpos = 0x7fffffff;
  for (int j = lane; j < cnt; j += 32) {
    const int32_t v = row[j];
    buf[j] = v;
    if (do_rm && v == rc) rpos = min(rpos, j);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) rpos = min(rpos, __shfl_xor_sync(0xffffffffu, rpos, o));
  __syncwarp();
  const bool removed_one = rpos != 0x7fffffff;
  const int cnt1 = cnt - (removed_one ? 1 : 0);
  const bool ins = do_in && cnt1 < Lx;
  for (int j = lane; j < cnt; j += 32) {
    if (removed_one && j == rpos) continue;
    const int32_t v = buf[j];
    int idx = j - ((removed_one && j > rpos) ? 1 : 0);
    if (ins && v > ic) ++idx;                       // equal ids stay in front of the inserted one
    row[idx] = v;
  }
  if (ins) {
    int below = 0;                                  // position of the pick = number of remaining entries <= ic
    for (int j = lane; j < cnt; j += 32) if (!(removed_one && j == rpos) && buf[j] <= ic) ++below;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) below += __shfl_xor_sync(0xffffffffu, below, o);
    if (lane == 0) row[below] = ic;
  }
  const int cnt2 = cnt1 + (ins ? 1 : 0);
  if (lane == 0) {
    count[m] = cnt2;
    if (cnt2 < cnt) row[cnt2] = 0x7fffffff;         // the vacated tail slot
  }
}

// ---- k == 1 : best of the slices ------------------------------------------------------------------
__global__ void __launch_bounds__(256)
argmax_finalize_kernel(const unsigned long long* __restrict__ slice_keys, int n_slices, int M, int64_t item_base,
                       float* __restrict__ vals, int64_t* __restrict__ items) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  unsigned long long best = 0ull;
  for (int s = 0; s < n_slices; ++s) {
    const unsigned long long key = slice_keys[(int64_t)m * n_slices + s];
    best = key > best ? key : best;
  }
  vals[m] = best ? key_score(best) : -INFINITY;
  items[m] = best ? (int64_t)key_col(best) + item_base : -1;
}

// ---- k > 1, step 1 : k-th largest slice maximum = a lower bound of the k-th largest score ---------
__global__ void __launch_bounds__(256)
threshold_kernel(const unsigned long long* __restrict__ slice_keys, int n_slices, int k, int P,
                 unsigned long long* __restrict__ thr_keys, int* __restrict__ cand_count) {
  extern __shared__ unsigned long long sk[];
  const int m = blockIdx.x;
  for (int t = threadIdx.x; t < P; t += blockDim.x) sk[t] = (t < n_slices) ? slice_keys[(int64_t)m * n_slices + t] : 0ull;
  block_bitonic_desc(sk, P);
  if (threadIdx.x == 0) {
    thr_keys[m] = (k <= n_slices) ? sk[k - 1] : 0ull;   // 0 = collect everything
    cand_count[m] = 0;
  }
}

// ---- k > 1, step 3 : sort the collected candidates, emit the k best --------------------------------
__global__ void __launch_bounds__(256)
candidates_finalize_kernel(const unsigned long long* __restrict__ cand_keys, const int* __restrict__ cand_count,
                           int cap, int k, int64_t item_base, float* __restrict__ vals, int64_t* __restrict__ items) {
  extern __shared__ unsigned long long sk[];
  const int m = blockIdx.x;
  const int cnt = cand_count[m];
  const bool overflow = cnt > cap;
  const int n = overflow ? cap : cnt;
  const int P = next_pow2(n > k ? n : k);
  for (int t = threadIdx.x; t < P; t += blockDim.x) sk[t] = (t < n) ? cand_keys[(int64_t)m * cap + t] : 0ull;
  block_bitonic_desc(sk, P);
  for (int t = threadIdx.x; t < k; t += blockDim.x) {
    const unsigned long long key = sk[t];
    if (overflow) { vals[(int64_t)m * k + t] = NAN; items[(int64_t)m * k + t] = -2; }          // IRS_E_OVERFLOW marker
    else if (key) { vals[(int64_t)m * k + t] = key_score(key); items[(int64_t)m * k + t] = (int64_t)key_col(key) + item_base; }
    else { vals[(int64_t)m * k + t] = -INFINITY; items[(int64_t)m * k + t] = -1; }              // fewer than k live items
  }
}

// ---- log-sum-exp merge over catalog splits ----------------------------------------------------------
__global__ void __launch_bounds__(256)
lse_finalize_kernel(const float* __restrict__ part_max, const float* __restrict__ part_sum, int n_splits, int M,
                    float* __restrict__ lse) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  float mm = -INFINITY;
  for (int s = 0; s < n_splits; ++s) mm = fmaxf(mm, part_max[(int64_t)m * n_splits + s]);
  float ss = 0.f;
  for (int s = 0; s < n_splits; ++s) {
    const float pm = part_max[(int64_t)m * n_splits + s];
    if (pm > -INFINITY) ss += part_sum[(int64_t)m * n_splits + s] * expf(pm - mm);
  }
  lse[m] = mm + logf(ss);
}

// ---- rank: label score prologue (same FMA chain as the tile engine) and finalise --------------------
__global__ void __launch_bounds__(256)
label_score_kernel(const float* __restrict__ h, int64_t ld_h, const float* __restrict__ W, const float* __restrict__ bias,
                   const int64_t* __restrict__ label, int64_t item_base, int M, int64_t N, int d,
                   float* __restrict__ label_score, int* __restrict__ rank_count, int* __restrict__ rank_excluded) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  const int64_t c = label[m] - item_base;
  float acc = 0.f;
  if (c >= 0 && c < N) {
    for (int kk = 0; kk < d; ++kk) acc = fmaf(h[(int64_t)m * ld_h + kk], W[c * d + kk], acc);
    acc = acc + (bias ? bias[c] : 0.f);
  } else {
    acc = NAN;
  }
  label_score[m] = acc;
  rank_count[m] = 0;
  rank_excluded[m] = (c >= 0 && c < N) ? 0 : 1;
}

__global__ void __launch_bounds__(256)
rank_finalize_kernel(const int* __restrict__ rank_count, const int* __restrict__ rank_excluded, int M,
                     int64_t* __restrict__ rank) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  rank[m] = rank_excluded[m] ? 0 : (int64_t)rank_count[m] + 1;
}

// ---- shard merge --------------------------------------------------------------------------------------
// Row m of the [G, M, k] per-shard candidates as keys sorted by (score desc, item id asc) in sk[0..P); candidates with a
// negative item id or a NaN score become 0 (sorted last).  With `marker` non-null, *marker (shared) ends up 1 iff one of
// the row's candidates is the overflow marker (NaN, -2) of irs_score_topk.  Every thread of the block calls this.
__device__ void merge_row_candidates(const float* __restrict__ vals, const int64_t* __restrict__ items, int G, int M, int k,
                                     int P, int m, unsigned long long* sk, int* marker) {
  if (marker) {
    if (threadIdx.x == 0) *marker = 0;
    __syncthreads();
  }
  for (int t = threadIdx.x; t < P; t += blockDim.x) {
    unsigned long long key = 0ull;
    if (t < G * k) {
      const int g = t / k, j = t - g * k;
      const int64_t it = items[((int64_t)g * M + m) * k + j];
      const float v = vals[((int64_t)g * M + m) * k + j];
      if (it >= 0 && it <= 0xfffffffell && !(v != v)) key = pack_key(v, (uint32_t)it);   // item id as the column
      else if (marker && (it == -2 || v != v)) *marker = 1;   // racing threads all store 1; the sort's barriers publish it
    }
    sk[t] = key;
  }
  block_bitonic_desc(sk, P);                    // starts and ends with a barrier: *marker is final on return
}

__global__ void __launch_bounds__(256)
topk_merge_kernel(const float* __restrict__ vals, const int64_t* __restrict__ items, int G, int M, int k, int P,
                  float* __restrict__ out_vals, int64_t* __restrict__ out_items) {
  extern __shared__ unsigned long long sk[];
  const int m = blockIdx.x;
  merge_row_candidates(vals, items, G, M, k, P, m, sk, nullptr);
  for (int t = threadIdx.x; t < k; t += blockDim.x) {
    const unsigned long long key = sk[t];
    out_vals[(int64_t)m * k + t] = key ? key_score(key) : -INFINITY;
    out_items[(int64_t)m * k + t] = key ? (int64_t)key_col(key) : -1;
  }
}

// ---- top-k sampling (one draw from the softmax over the merged k best) -----------------------------------
__device__ __forceinline__ unsigned long long fmix64(unsigned long long x) {      // murmur3 finaliser
  x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; x ^= x >> 33;
  return x;
}

__global__ void __launch_bounds__(256)
topk_sample_kernel(const float* __restrict__ vals, const int64_t* __restrict__ items, int G, int M, int k, int P,
                   unsigned long long seed, int64_t step, const int64_t* __restrict__ row_key, int64_t* __restrict__ out_items) {
  extern __shared__ unsigned long long sk[];
  __shared__ int s_marker;
  const int m = blockIdx.x;
  merge_row_candidates(vals, items, G, M, k, P, m, sk, &s_marker);
  if (threadIdx.x != 0) return;
  if (s_marker) { out_items[m] = -2; return; }
  // the uniform: a pure function of (seed, step, row key); the header states the definition
  const unsigned long long phi = 0x9E3779B97F4A7C15ull;
  unsigned long long x = fmix64(seed + phi * ((unsigned long long)step + 1ull));
  x = fmix64(x + phi * ((unsigned long long)row_key[m] + 1ull));
  const double u = (double)(x >> 11) * 0x1.0p-53;
  // weights exp(v_i - v_0) of the finite survivors among the k best, summed one after another in sorted order
  double v0 = 0.0, total = 0.0;
  int n_live = 0;
  for (int t = 0; t < k; ++t) {
    const unsigned long long key = sk[t];
    if (!key) break;                                   // keys sort last: no survivor after the first empty slot
    const float v = key_score(key);
    if (!isfinite(v)) continue;
    if (n_live++ == 0) v0 = (double)v;
    total += exp((double)v - v0);
  }
  if (n_live == 0) { out_items[m] = -1; return; }      // every item excluded: what the arg-max returns
  const double target = u * total;
  double run = 0.0;
  int64_t pick = -1;
  for (int t = 0; t < k; ++t) {
    const unsigned long long key = sk[t];
    if (!key) break;
    const float v = key_score(key);
    if (!isfinite(v)) continue;
    pick = (int64_t)key_col(key);                      // rounding may leave no running sum above target: the last one
    run += exp((double)v - v0);
    if (run > target) break;
  }
  out_items[m] = pick;
}

// ---- window shift ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
window_shift_kernel(int64_t* __restrict__ seq, const int64_t* __restrict__ next, float* __restrict__ paths,
                    int B, int L, int P, int step) {
  const int lane = threadIdx.x & 31;
  const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (b >= B) return;
  int64_t* row = seq + (int64_t)b * L;
  const int64_t nx = next[b];
  // row[l] <- row[l+1] for l in [0, L-3]; row[L-2] <- next; row[L-1] (objective) stays
  for (int base = 0; base < L - 2; base += 32) {
    const int l = base + lane;
    int64_t v = 0;
    if (l < L - 2) v = row[l + 1];
    __syncwarp();
    if (l < L - 2) row[l] = v;
    __syncwarp();
  }
  if (lane == 0) {
    if (L >= 2) row[L - 2] = nx;
    if (paths != nullptr) paths[(int64_t)b * P + step] = (float)nx;
  }
}

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

}  // namespace irs

using namespace irs;

extern "C" int irs_sort_exclusions(const int64_t* excl_ids, int M, int Lx, int64_t item_base, int64_t N,
                                   int32_t* out_sorted, int32_t* out_count, void* stream) {
  if (!excl_ids || !out_sorted || !out_count) return IRS_E_BADARG;
  if (M <= 0 || Lx <= 0 || N <= 0) return IRS_E_BADARG;
  if (Lx > 2048 || N > 0x7ffffffe) return IRS_E_SHAPE;
  const int P = next_pow2(Lx);
  sort_exclusions_kernel<<<M, 256, (size_t)P * 8, (cudaStream_t)stream>>>(excl_ids, M, Lx, item_base, N, out_sorted, out_count, P);
  IRS_LAUNCHED();
  return 0;
}

extern "C" int irs_exclusions_update(int32_t* sorted, int32_t* count, const int64_t* removed_ids, int64_t removed_stride,
                                     const int64_t* inserted_ids, int M, int Lx, int64_t item_base, int64_t N, void* stream) {
  if (!sorted || !count || !removed_ids || !inserted_ids) return IRS_E_BADARG;
  if (M <= 0 || Lx <= 0 || N <= 0 || removed_stride <= 0) return IRS_E_BADARG;
  if (Lx > 2048 || N > 0x7ffffffe) return IRS_E_SHAPE;
  const int warps = 4;
  exclusions_update_kernel<<<(unsigned)ceil_div(M, warps), warps * 32, (size_t)warps * Lx * 4, (cudaStream_t)stream>>>(
      sorted, count, removed_ids, removed_stride, inserted_ids, M, Lx, item_base, N);
  IRS_LAUNCHED();
  return 0;
}

static int cand_cap_for(int k) {
  int c = next_pow2(4 * k);
  if (c < 512) c = 512;
  if (c > 4096) c = 4096;
  return c;
}

static int score_common_check(const float* h, const float* W, int M, int64_t N, int d) {
  if (!h || !W) return IRS_E_BADARG;
  if (M <= 0 || N <= 0 || d <= 0) return IRS_E_BADARG;
  if (N > 0x7ffffffe) return IRS_E_SHAPE;
  return 0;
}

extern "C" size_t irs_score_topk_workspace_bytes(int M, int64_t N, int d, int k) {
  (void)d;
  if (M <= 0 || N <= 0 || k <= 0) return 0;
  const int splits = score_simt_max_splits(M, N);
  if (k == 1) return align256((size_t)M * splits * 8);
  size_t b = align256((size_t)M * splits * 16 * 8);      // slice keys
  b += align256((size_t)M * 8);                          // thresholds
  b += align256((size_t)M * 4);                          // candidate counts
  b += align256((size_t)M * cand_cap_for(k) * 8);        // candidate keys
  return b;
}

extern "C" int irs_score_topk(const float* h, int64_t ld_h, const float* W, const float* bias, int64_t item_base,
                              const int32_t* excl_sorted, const int32_t* excl_count, int Lx, int k,
                              float* vals, int64_t* items, int M, int64_t N, int d,
                              void* workspace, size_t workspace_bytes, void* stream) {
  int rc = score_common_check(h, W, M, N, d);
  if (rc) return rc;
  if (!vals || !items || !workspace || k < 1 || k > 1024) return IRS_E_BADARG;
  if (excl_sorted && (!excl_count || Lx <= 0)) return IRS_E_BADARG;
  if (workspace_bytes < irs_score_topk_workspace_bytes(M, N, d, k)) return IRS_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  ScoreParams p = {};
  p.h = h; p.ld_h = ld_h; p.W = W; p.bias = bias; p.M = M; p.N = N; p.d = d; p.item_base = item_base;
  p.excl_sorted = excl_sorted; p.excl_count = excl_count; p.Lx = Lx;
  char* ws = (char*)workspace;
  const int splits = score_simt_max_splits(M, N);
  p.max_splits = splits;
  p.slice_keys = (unsigned long long*)ws;
  if (k == 1) {
    p.slices_per_split = 1;
    rc = launch_score_simt(MODE_MAX, p, s);
    if (rc) return rc;
    argmax_finalize_kernel<<<(unsigned)ceil_div(M, 256), 256, 0, s>>>(p.slice_keys, p.n_slices, M, item_base, vals, items);
    IRS_LAUNCHED();
    return 0;
  }
  ws += align256((size_t)M * splits * 16 * 8);
  unsigned long long* thr = (unsigned long long*)ws; ws += align256((size_t)M * 8);
  int* cnt = (int*)ws; ws += align256((size_t)M * 4);
  unsigned long long* cand = (unsigned long long*)ws;
  const int cap = cand_cap_for(k);
  p.slices_per_split = 16;
  if (p.max_splits > 256) p.max_splits = 256;       // the threshold kernel sorts <= 4096 slice keys per row (few rows x large catalog)
  rc = launch_score_simt(MODE_MAX, p, s);
  if (rc) return rc;
  const int P = next_pow2(p.n_slices);
  if (P > 4096) return IRS_E_SHAPE;
  threshold_kernel<<<M, 256, (size_t)P * 8, s>>>(p.slice_keys, p.n_slices, k, P, thr, cnt);
  IRS_LAUNCHED();
  p.thr_keys = thr; p.cand_keys = cand; p.cand_count = cnt; p.cand_cap = cap;
  rc = launch_score_simt(MODE_COLLECT, p, s);
  if (rc) return rc;
  candidates_finalize_kernel<<<M, 256, (size_t)cap * 8, s>>>(cand, cnt, cap, k, item_base, vals, items);
  IRS_LAUNCHED();
  return 0;
}

extern "C" size_t irs_score_lse_gather_workspace_bytes(int M, int64_t N, int d, int n_sel) {
  (void)d; (void)n_sel;
  if (M <= 0 || N <= 0) return 0;
  return 2 * align256((size_t)M * score_simt_max_splits(M, N) * 4);
}

extern "C" int irs_score_lse_gather(const float* h, int64_t ld_h, const float* W, const float* bias, int64_t item_base,
                                    const int64_t* sel, int n_sel, float* lse, float* logit,
                                    int M, int64_t N, int d, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = score_common_check(h, W, M, N, d);
  if (rc) return rc;
  if (!lse || !workspace || n_sel < 0 || (n_sel > 0 && (!sel || !logit))) return IRS_E_BADARG;
  if (workspace_bytes < irs_score_lse_gather_workspace_bytes(M, N, d, n_sel)) return IRS_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  ScoreParams p = {};
  p.h = h; p.ld_h = ld_h; p.W = W; p.bias = bias; p.M = M; p.N = N; p.d = d; p.item_base = item_base;
  const int splits = score_simt_max_splits(M, N);
  p.max_splits = splits;
  p.part_max = (float*)workspace;
  p.part_sum = (float*)((char*)workspace + align256((size_t)M * splits * 4));
  p.sel = sel; p.n_sel = n_sel; p.sel_logit = logit;
  if (n_sel > 0) IRS_CUDA(cudaMemsetAsync(logit, 0, (size_t)M * n_sel * 4, s));
  rc = launch_score_simt(MODE_LSE, p, s);
  if (rc) return rc;
  lse_finalize_kernel<<<(unsigned)ceil_div(M, 256), 256, 0, s>>>(p.part_max, p.part_sum, p.n_splits, M, lse);
  IRS_LAUNCHED();
  return 0;
}

extern "C" size_t irs_score_rank_workspace_bytes(int M, int64_t N, int d) {
  (void)N; (void)d;
  if (M <= 0) return 0;
  return 3 * align256((size_t)M * 4);
}

extern "C" int irs_score_rank(const float* h, int64_t ld_h, const float* W, const float* bias, int64_t item_base,
                              const int64_t* label, const int32_t* excl_sorted, const int32_t* excl_count, int Lx,
                              int64_t* rank, int M, int64_t N, int d,
                              void* workspace, size_t workspace_bytes, void* stream) {
  int rc = score_common_check(h, W, M, N, d);
  if (rc) return rc;
  if (!label || !rank || !workspace) return IRS_E_BADARG;
  if (excl_sorted && (!excl_count || Lx <= 0)) return IRS_E_BADARG;
  if (workspace_bytes < irs_score_rank_workspace_bytes(M, N, d)) return IRS_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  char* ws = (char*)workspace;
  float* lab_s = (float*)ws; ws += align256((size_t)M * 4);
  int* cnt = (int*)ws; ws += align256((size_t)M * 4);
  int* exc = (int*)ws;
  label_score_kernel<<<(unsigned)ceil_div(M, 256), 256, 0, s>>>(h, ld_h, W, bias, label, item_base, M, N, d, lab_s, cnt, exc);
  IRS_LAUNCHED();
  ScoreParams p = {};
  p.h = h; p.ld_h = ld_h; p.W = W; p.bias = bias; p.M = M; p.N = N; p.d = d; p.item_base = item_base;
  p.excl_sorted = excl_sorted; p.excl_count = excl_count; p.Lx = Lx;
  p.label = label; p.label_score = lab_s; p.rank_count = cnt; p.rank_excluded = exc;
  rc = launch_score_simt(MODE_RANK, p, s);
  if (rc) return rc;
  rank_finalize_kernel<<<(unsigned)ceil_div(M, 256), 256, 0, s>>>(cnt, exc, M, rank);
  IRS_LAUNCHED();
  return 0;
}

// ---- catalog-sharded rank / log-prob support (SURVEY 8e row 3) ------------------------------------------------------------
// exact scores of selected items with the tile engines' sequential fp32 FMA chain; -inf outside this shard / for PAD
__global__ void __launch_bounds__(256)
score_select_kernel(const float* __restrict__ h, int64_t ld_h, const float* __restrict__ W, const float* __restrict__ bias,
                    int64_t item_base, const int64_t* __restrict__ sel, int n_sel, float* __restrict__ out, int M, int64_t N, int d) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)M * n_sel) return;
  const int m = (int)(i / n_sel);
  const int64_t id = sel[i];
  const int64_t c = id - item_base;
  float acc = -INFINITY;
  if (id != 0 && c >= 0 && c < N) {
    acc = 0.f;
    for (int kk = 0; kk < d; ++kk) acc = fmaf(h[(int64_t)m * ld_h + kk], __ldg(W + c * d + kk), acc);
    acc = acc + (bias ? __ldg(bias + c) : 0.f);
  }
  out[i] = acc;
}

__global__ void __launch_bounds__(256)
count_finalize_kernel(const int* __restrict__ cnt, const int* __restrict__ exc, int M, int64_t* __restrict__ count,
                      int32_t* __restrict__ label_excluded) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  count[m] = (int64_t)cnt[m];
  label_excluded[m] = exc[m] ? 1 : 0;
}

extern "C" int irs_score_select(const float* h, int64_t ld_h, const float* W, const float* bias, int64_t item_base,
                                const int64_t* sel, int n_sel, float* out, int M, int64_t N, int d, void* stream) {
  int rc = score_common_check(h, W, M, N, d);
  if (rc) return rc;
  if (!sel || !out || n_sel <= 0) return IRS_E_BADARG;
  score_select_kernel<<<(unsigned)ceil_div((int64_t)M * n_sel, 256), 256, 0, (cudaStream_t)stream>>>(
      h, ld_h, W, bias, item_base, sel, n_sel, out, M, N, d);
  IRS_LAUNCHED();
  return 0;
}

extern "C" size_t irs_score_count_ahead_workspace_bytes(int M, int64_t N, int d) {
  (void)N; (void)d;
  return M > 0 ? 2 * align256((size_t)M * 4) : 0;
}

extern "C" int irs_score_count_ahead(const float* h, int64_t ld_h, const float* W, const float* bias, int64_t item_base,
                                     const int64_t* label, const float* label_score,
                                     const int32_t* excl_sorted, const int32_t* excl_count, int Lx,
                                     int64_t* count, int32_t* label_excluded, int M, int64_t N, int d,
                                     void* workspace, size_t workspace_bytes, void* stream) {
  int rc = score_common_check(h, W, M, N, d);
  if (rc) return rc;
  if (!label || !label_score || !count || !label_excluded || !workspace) return IRS_E_BADARG;
  if (excl_sorted && (!excl_count || Lx <= 0)) return IRS_E_BADARG;
  if (workspace_bytes < irs_score_count_ahead_workspace_bytes(M, N, d)) return IRS_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  char* ws = (char*)workspace;
  int* cnt = (int*)ws; ws += align256((size_t)M * 4);
  int* exc = (int*)ws;
  IRS_CUDA(cudaMemsetAsync(workspace, 0, 2 * align256((size_t)M * 4), s));
  ScoreParams p = {};
  p.h = h; p.ld_h = ld_h; p.W = W; p.bias = bias; p.M = M; p.N = N; p.d = d; p.item_base = item_base;
  p.excl_sorted = excl_sorted; p.excl_count = excl_count; p.Lx = Lx;
  p.label = label; p.label_score = label_score; p.rank_count = cnt; p.rank_excluded = exc;
  rc = launch_score_simt(MODE_RANK, p, s);
  if (rc) return rc;
  count_finalize_kernel<<<(unsigned)ceil_div(M, 256), 256, 0, s>>>(cnt, exc, M, count, label_excluded);
  IRS_LAUNCHED();
  return 0;
}

extern "C" int irs_topk_merge(const float* vals, const int64_t* items, int G, int M, int k,
                              float* out_vals, int64_t* out_items, void* stream) {
  if (!vals || !items || !out_vals || !out_items) return IRS_E_BADARG;
  if (G <= 0 || M <= 0 || k <= 0) return IRS_E_BADARG;
  if ((int64_t)G * k > 4096) return IRS_E_SHAPE;
  const int P = next_pow2(G * k);
  topk_merge_kernel<<<M, 256, (size_t)P * 8, (cudaStream_t)stream>>>(vals, items, G, M, k, P, out_vals, out_items);
  IRS_LAUNCHED();
  return 0;
}

extern "C" int irs_topk_sample(const float* vals, const int64_t* items, int G, int M, int k,
                               unsigned long long seed, int64_t step, const int64_t* row_key,
                               int64_t* out_items, void* stream) {
  if (!vals || !items || !row_key || !out_items) return IRS_E_BADARG;
  if (G <= 0 || M <= 0 || k <= 0) return IRS_E_BADARG;
  if ((int64_t)G * k > 4096) return IRS_E_SHAPE;
  const int P = next_pow2(G * k);
  int threads = next_pow2(P / 2);                       // one compare-exchange per thread and stage
  threads = threads < 32 ? 32 : (threads > 256 ? 256 : threads);
  topk_sample_kernel<<<M, threads, (size_t)P * 8, (cudaStream_t)stream>>>(vals, items, G, M, k, P, seed, step, row_key,
                                                                          out_items);
  IRS_LAUNCHED();
  return 0;
}

extern "C" int irs_window_shift(int64_t* seq, const int64_t* next, float* paths, int B, int L, int P, int step, void* stream) {
  if (!seq || !next) return IRS_E_BADARG;
  if (B <= 0 || L < 2) return IRS_E_BADARG;
  if (paths && (step < 0 || step >= P)) return IRS_E_BADARG;
  window_shift_kernel<<<(unsigned)ceil_div((int64_t)B * 32, 256), 256, 0, (cudaStream_t)stream>>>(seq, next, paths, B, L, P, step);
  IRS_LAUNCHED();
  return 0;
}
