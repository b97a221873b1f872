// Exact full-catalog top-K recommendation: for each user u the K items j in [1, V), j not excluded, with the largest
// canonical logits s(u,j) (score_full.cuh: k ascending, multiply and add rounded separately), ties broken by item id
// ascending.  Returned scores are those canonical logits bit for bit; fewer than K eligible items pad the tail with
// (id 0, -inf).
//
// Tensor-core path (mode 0): the tcgen05 3xTF32 pipeline of score_full is only a filter, with d = c_K |u| |e_j| the
// rigorous bound on |s~ - s|.
//   1. threshold pass   sf_umma_kernel<BoundEpi>: each epilogue thread keeps in registers the TK_R largest lower bounds
//                       s~ - d of eligible items over its (work unit, column half); every gathered bound belongs to a
//                       distinct eligible item and is <= its score, so the K-th largest gathered bound tau_u
//                       (tk_tau_kernel) is <= the K-th largest score (-inf when fewer than K bounds were gathered);
//   2. admission pass   sf_umma_kernel<AdmitEpi>: every eligible item with s~ + d >= tau_u goes to a per-user
//                       candidate buffer (integer atomics).  An item of the true top K has s >= tau_u and s~ + d >= s,
//                       so it is admitted, and so is every item tied with the K-th score;
//   3. select           tk_select_kernel: canonical dot per candidate, rank by (score desc, id asc), write the top K.
//                       A user whose buffer overflowed (or whose tau_u is -inf) takes the exact path instead.
// Exact path (mode 1, and the fallback): brute-force canonical dots with a block-wide running top K.
#include "score_full.cuh"

namespace cast {

constexpr int TK_R = 8;          // lower bounds kept per (epilogue thread, work unit) in the threshold pass
constexpr int TK_MAXK = 256;
constexpr int TK_THREADS = 128;  // select / exact kernels

static inline int tk_cap(int K) { return 2 * K + 256; }   // candidate buffer per user

__device__ __forceinline__ float tk_ninf() { return __int_as_float((int)0xff800000u); }

// is item j in the user's exclusion row (CSR, ids ascending; duplicates and out-of-range ids are harmless)
__device__ __forceinline__ bool tk_excluded(const int* __restrict__ eptr, const int* __restrict__ eidx, long u, int j) {
  if (!eptr) return false;
  int lo = eptr[u];
  const int end = eptr[u + 1];
  int hi = end;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (eidx[mid] < j) lo = mid + 1;
    else hi = mid;
  }
  return lo < end && eidx[lo] == j;
}

// result order: score descending, then id ascending (ids are distinct, so this is a strict total order)
__device__ __forceinline__ bool tk_before(float s, int i, float t, int j) { return s > t || (s == t && i < j); }

// m distinct entries (s, id) -> the K first in result order, each written at its rank (rank = entries before it)
__device__ __forceinline__ void tk_rank_scatter(const float* s, const int* id, int m, int K, float* os, int* oi) {
  for (int i = threadIdx.x; i < m; i += blockDim.x) {
    const float x = s[i];
    const int xi = id[i];
    int r = 0;
    for (int j = 0; j < m; ++j) r += tk_before(s[j], id[j], x, xi) ? 1 : 0;
    if (r < K) { os[r] = x; oi[r] = xi; }
  }
}

// Exact top K of user u by brute force (whole block).  Items arrive in id order, so a new item enters the list only
// with a score strictly above the current K-th.  smem: H floats, then two (score, id) arrays of K + blockDim entries.
__device__ void tk_exact_user(const float* __restrict__ urow, const float* __restrict__ table, int V, int H, int K,
                              const int* __restrict__ eptr, const int* __restrict__ eidx, long u,
                              unsigned char* smem, int* n_sh, int* add_sh, int* __restrict__ out_id,
                              float* __restrict__ out_s) {
  const int T = blockDim.x;
  float* us = reinterpret_cast<float*>(smem);
  float* as = us + ((H + 3) & ~3);
  int* ai = reinterpret_cast<int*>(as + K + T);
  float* bs = reinterpret_cast<float*>(ai + K + T);
  int* bi = reinterpret_cast<int*>(bs + K + T);
  for (int k = threadIdx.x; k < H; k += T) us[k] = urow[k];
  if (threadIdx.x == 0) { *n_sh = 0; *add_sh = 0; }
  __syncthreads();
  for (long base = 1; base < V; base += T) {
    const int n = *n_sh;
    const float kth = n == K ? as[K - 1] : tk_ninf();
    const long j = base + threadIdx.x;
    bool take = false;
    float s = 0.f;
    if (j < V && !tk_excluded(eptr, eidx, u, (int)j)) {
      s = canonical_dot(us, table + j * H, H);
      take = n < K || s > kth;
    }
    if (take) {
      const int p = atomicAdd(add_sh, 1);
      as[n + p] = s;
      ai[n + p] = (int)j;
    }
    __syncthreads();
    const int m = n + *add_sh;
    if (m > n) {   // merge the list and the newcomers into the other buffer, then swap
      tk_rank_scatter(as, ai, m, K, bs, bi);
      float* ts = as; as = bs; bs = ts;
      int* ti = ai; ai = bi; bi = ti;
    }
    __syncthreads();
    if (threadIdx.x == 0) { *n_sh = m < K ? m : K; *add_sh = 0; }
    __syncthreads();
  }
  const int n = *n_sh;
  for (int r = threadIdx.x; r < K; r += T) {
    out_id[r] = r < n ? ai[r] : 0;
    out_s[r] = r < n ? as[r] : tk_ninf();
  }
}

static size_t tk_exact_smem(int H, int K) { return (size_t)((H + 3) & ~3) * 4 + 4 * (size_t)(K + TK_THREADS) * 4; }

// mode 1: one CTA per user
__global__ void __launch_bounds__(TK_THREADS) tk_exact_kernel(const float* __restrict__ users, long ldu,
                                                               const float* __restrict__ table, int V, int H, int K,
                                                               const int* __restrict__ eptr,
                                                               const int* __restrict__ eidx, int* __restrict__ top_ids,
                                                               float* __restrict__ top_scores) {
  CAST_DYN_SMEM(unsigned char, sm);
  __shared__ int n_sh, add_sh;
  const long u = blockIdx.x;
  tk_exact_user(users + u * ldu, table, V, H, K, eptr, eidx, u, sm, &n_sh, &add_sh, top_ids + u * K,
                top_scores + u * K);
}

#ifndef CAST_EMU
// ------------------------------------------------------------------------------------------------ tensor-core path
// threshold pass: top-TK_R lower bounds s~ - d per (thread, work unit), written to lbs[user][split][half][TK_R]
struct BoundEpi {
  struct Params {
    const int* eptr;
    const int* eidx;
    float* lbs;
    int nslot;   // 2 * nsplit
  };
  const Params& p;
  const long me;
  const int je, slot;
  float d = 0.f;
  float top[TK_R];   // descending

  __device__ __forceinline__ BoundEpi(const SfPipe&, const Params& p_, long me_, bool, int sp, int chalf, int,
                                      int je_)
      : p(p_), me(me_), je(je_), slot(2 * sp + chalf) {
#pragma unroll
    for (int i = 0; i < TK_R; ++i) top[i] = tk_ninf();
  }

  __device__ __forceinline__ void tile(int, float d_) { d = d_; }

  __device__ __forceinline__ void chunk(const float (&v)[32], int j) {
    unsigned m = 0;
#pragma unroll
    for (int e = 0; e < 32; ++e) m |= (v[e] - d > top[TK_R - 1]) ? (1u << e) : 0u;
    while (m) {   // only values that would enter the list pay for the eligibility check
      const int e = __ffs((int)m) - 1;
      m &= m - 1;
      float x = v[0];
#pragma unroll
      for (int k = 1; k < 32; ++k) x = k == e ? v[k] : x;
      x = x - d;
      const int item = j + e;
      if (x > top[TK_R - 1] && item >= 1 && item < je && !tk_excluded(p.eptr, p.eidx, me, item)) {
#pragma unroll
        for (int i = 0; i < TK_R; ++i) {   // insert, dropping the smallest
          const float hi = fmaxf(top[i], x);
          x = fminf(top[i], x);
          top[i] = hi;
        }
      }
    }
  }

  __device__ __forceinline__ void finish() {
    float* o = p.lbs + ((size_t)me * p.nslot + slot) * TK_R;
#pragma unroll
    for (int i = 0; i < TK_R; ++i) o[i] = top[i];
  }
};

// admission pass: eligible items with s~ + d >= tau_u are appended to the user's candidate buffer
struct AdmitEpi {
  struct Params {
    const int* eptr;
    const int* eidx;
    const float* tau;
    int* cnt;
    int* cand;   // [U, cap]
    int cap;
  };
  const Params& p;
  const long me;
  const int je;
  const float tau;
  float d = 0.f;

  __device__ __forceinline__ AdmitEpi(const SfPipe&, const Params& p_, long me_, bool live, int, int, int, int je_)
      : p(p_), me(me_), je(je_), tau(live ? p_.tau[me_] : 0.f) {}

  __device__ __forceinline__ void tile(int, float d_) { d = d_; }

  __device__ __forceinline__ void chunk(const float (&v)[32], int j) {
    if (tau == tk_ninf()) return;   // the user is already on the exact path
    unsigned m = 0;
#pragma unroll
    for (int e = 0; e < 32; ++e) m |= (v[e] + d >= tau) ? (1u << e) : 0u;
    while (m) {
      const int e = __ffs((int)m) - 1;
      m &= m - 1;
      const int item = j + e;
      if (item < 1 || item >= je || tk_excluded(p.eptr, p.eidx, me, item)) continue;
      const int slot = atomicAdd(&p.cnt[me], 1);
      if (slot < p.cap) p.cand[(size_t)me * p.cap + slot] = item;
    }
  }

  __device__ __forceinline__ void finish() {}
};

// |u| bound per user (one warp per user)
__global__ void tk_unorm_kernel(const float* __restrict__ users, long ldu, int H, long U, float* __restrict__ unorm) {
  const int lane = threadIdx.x & 31;
  const long u = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (u >= U) return;
  const float* ur = users + u * ldu;
  float s = 0.f;
  for (int k = lane; k < H; k += 32) s = fmaf(ur[k], ur[k], s);
  s = warp_sum(s);
  if (lane == 0) unorm[u] = sqrtf(s) * NORM_SLACK;
}

__device__ __forceinline__ unsigned tk_key(float x) {   // order-preserving float -> unsigned
  const unsigned b = __float_as_uint(x);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

// tau_u = K-th largest of the user's gathered lower bounds (radix select on the ordered keys, one warp per user);
// fewer than K finite bounds: tau_u = -inf and the candidate count starts past the capacity (exact path)
__global__ void tk_tau_kernel(const float* __restrict__ lbs, int n, long U, int K, int cap, float* __restrict__ tau,
                              int* __restrict__ cnt) {
  const int lane = threadIdx.x & 31;
  const long u = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (u >= U) return;
  const float* x = lbs + (size_t)u * n;
  int fin = 0;
  for (int i = lane; i < n; i += 32) fin += x[i] > tk_ninf() ? 1 : 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) fin += __shfl_xor_sync(0xffffffffu, fin, o);
  if (fin < K) {
    if (lane == 0) { tau[u] = tk_ninf(); cnt[u] = cap + 1; }
    return;
  }
  unsigned prefix = 0;
  for (int bit = 31; bit >= 0; --bit) {
    const unsigned c = prefix | (1u << bit);
    int ge = 0;
    for (int i = lane; i < n; i += 32) ge += tk_key(x[i]) >= c ? 1 : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ge += __shfl_xor_sync(0xffffffffu, ge, o);
    if (ge >= K) prefix = c;
  }
  if (lane == 0) {
    tau[u] = __uint_as_float((prefix & 0x80000000u) ? (prefix & 0x7fffffffu) : ~prefix);
    cnt[u] = 0;
  }
}

// one CTA per user: canonical dots of the admitted candidates, ranked; overflowed users take the exact path
__global__ void __launch_bounds__(TK_THREADS) tk_select_kernel(const float* __restrict__ users, long ldu,
                                                                const float* __restrict__ table, int V, int H, int K,
                                                                const int* __restrict__ eptr,
                                                                const int* __restrict__ eidx,
                                                                const int* __restrict__ cnt,
                                                                const int* __restrict__ cand, int cap,
                                                                int* __restrict__ top_ids,
                                                                float* __restrict__ top_scores,
                                                                unsigned long long* __restrict__ stats) {
  CAST_DYN_SMEM(unsigned char, sm);
  __shared__ int n_sh, add_sh;
  const long u = blockIdx.x;
  const int c = cnt[u];
  int* oid = top_ids + u * K;
  float* osc = top_scores + u * K;
  if (c > cap) {
    if (stats && threadIdx.x == 0) atomicAdd(&stats[1], 1ull);
    tk_exact_user(users + u * ldu, table, V, H, K, eptr, eidx, u, sm, &n_sh, &add_sh, oid, osc);
    return;
  }
  if (stats && threadIdx.x == 0 && c) atomicAdd(&stats[0], (unsigned long long)c);
  float* cs = reinterpret_cast<float*>(sm);
  int* ci = reinterpret_cast<int*>(cs + cap);
  const float* ur = users + u * ldu;
  for (int i = threadIdx.x; i < c; i += blockDim.x) {
    const int j = cand[(size_t)u * cap + i];
    cs[i] = canonical_dot(ur, table + (long)j * H, H);
    ci[i] = j;
  }
  __syncthreads();
  tk_rank_scatter(cs, ci, c, K, osc, oid);
  for (int r = c + threadIdx.x; r < K; r += blockDim.x) {
    oid[r] = 0;
    osc[r] = tk_ninf();
  }
}
#endif  // !CAST_EMU

// threshold-pass splits: ~2 work units per SM, and 2 * TK_R * nsplit >= 2K bounds per user where the catalog has
// the tiles; the value is the split count the pipeline ends up with (sf_set_split keeps it unchanged)
static long tk_nsplit(long U, int V, int K) {
  const long ntiles = cdiv(V, 256);
  long n = cdiv(148L * 2, cdiv(U, 128));
  if (n < cdiv(K, TK_R)) n = cdiv(K, TK_R);
  if (n > ntiles) n = ntiles;
  if (n < 1) n = 1;
  return cdiv(V, cdiv(ntiles, n) * 256);
}

struct TkLayout {
  size_t inorm, tnorm, unorm, tau, cnt, lbs, cand, pre, total;
};

// workspace: [256-byte flag block | inorm V | tnorm | unorm U | tau U | cnt U | bounds | candidates | operand images]
static TkLayout tk_layout(long U, int V, int H, int K) {
  TkLayout l;
  size_t o = 256;
  l.inorm = o; o += sf_align((size_t)V * 4);
  l.tnorm = o; o += sf_align((size_t)(V / 256 + 2) * 4);
  l.unorm = o; o += sf_align((size_t)U * 4);
  l.tau = o; o += sf_align((size_t)U * 4);
  l.cnt = o; o += sf_align((size_t)U * 4);
  l.lbs = o; o += sf_align((size_t)U * 2 * tk_nsplit(U, V, K) * TK_R * 4);
  l.cand = o; o += sf_align((size_t)U * tk_cap(K) * 4);
  l.pre = o; o += sf_presplit_bytes(U, V, H, nullptr);
  l.total = o;
  return l;
}

}  // namespace cast

using namespace cast;

extern "C" size_t cast_topk_full_workspace_bytes(long U, int V, int H, int K) {
  if (U <= 0 || V <= 1 || H <= 0 || K < 1 || K > TK_MAXK) return 0;
  return tk_layout(U, V, H, K).total;
}

extern "C" int cast_topk_full(const float* seq_last, long ld, const float* table, int V, int H, long U, int K,
                              const int* excl_ptr, const int* excl_idx, int mode, int* top_ids, float* top_scores,
                              unsigned long long* stats, void* workspace, size_t workspace_bytes, void* stream) {
  if (K < 1 || K > TK_MAXK) return set_error(CAST_ERR_BAD_ARG, "topk_full: K must be in [1, 256]");
  if (!seq_last || !table || !top_ids || !top_scores || V <= 1 || H <= 0 || U <= 0 || ld < H ||
      (mode != 0 && mode != 1) || (excl_ptr && !excl_idx))
    return set_error(CAST_ERR_BAD_ARG, "topk_full");
  const TkLayout l = tk_layout(U, V, H, K);
  if (!workspace || workspace_bytes < l.total) return set_error(CAST_ERR_WORKSPACE, "topk_full: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  unsigned char* w = static_cast<unsigned char*>(workspace);
  int* err = reinterpret_cast<int*>(w);
  int rc;
  cudaMemsetAsync(err, 0, sizeof(int), st);
  if (stats) cudaMemsetAsync(stats, 0, 2 * sizeof(unsigned long long), st);
#ifdef CAST_EMU
  mode = 1;  // the host emulation has no tensor cores; the exact path defines the same result
#endif
  if (mode == 1) {
    CAST_LAUNCH(tk_exact_kernel, dim3((unsigned)U), dim3(TK_THREADS), tk_exact_smem(H, K), st, seq_last, ld, table, V,
                H, K, excl_ptr, excl_idx, top_ids, top_scores);
    return check_launch("topk_full(exact)");
  }
#ifndef CAST_EMU
  float* inorm = reinterpret_cast<float*>(w + l.inorm);
  float* tnorm = reinterpret_cast<float*>(w + l.tnorm);
  float* unorm = reinterpret_cast<float*>(w + l.unorm);
  float* tau = reinterpret_cast<float*>(w + l.tau);
  int* cnt = reinterpret_cast<int*>(w + l.cnt);
  float* lbs = reinterpret_cast<float*>(w + l.lbs);
  int* cand = reinterpret_cast<int*>(w + l.cand);
  SfPipe a;
  if ((rc = sf_prepare(a, seq_last, ld, table, V, H, U, w + l.pre, inorm, tnorm, st, "topk_full(prepare)"))) return rc;
  tk_unorm_kernel<<<dim3((unsigned)cdiv(U, 4)), dim3(128), 0, st>>>(seq_last, ld, H, U, unorm);
  a.unorm = unorm;
  a.err = err;
  const long nsplit = tk_nsplit(U, V, K);
  sf_set_split(a, nsplit);
  if (a.nsplit != nsplit) return set_error(CAST_ERR_BAD_ARG, "topk_full: split plan mismatch");
  BoundEpi::Params bp{excl_ptr, excl_idx, lbs, 2 * a.nsplit};
  if ((rc = sf_launch<BoundEpi>(a, bp, st, "topk_full(threshold)"))) return rc;
  const int cap = tk_cap(K);
  tk_tau_kernel<<<dim3((unsigned)cdiv(U, 4)), dim3(128), 0, st>>>(lbs, 2 * a.nsplit * TK_R, U, K, cap, tau, cnt);
  if ((rc = check_launch("topk_full(tau)"))) return rc;
  AdmitEpi::Params ap{excl_ptr, excl_idx, tau, cnt, cand, cap};
  if ((rc = sf_launch<AdmitEpi>(a, ap, st, "topk_full(admit)"))) return rc;
  size_t smem = tk_exact_smem(H, K);
  if (smem < (size_t)cap * 8) smem = (size_t)cap * 8;
  tk_select_kernel<<<dim3((unsigned)U), dim3(TK_THREADS), smem, st>>>(seq_last, ld, table, V, H, K, excl_ptr, excl_idx,
                                                                      cnt, cand, cap, top_ids, top_scores, stats);
  return check_launch("topk_full(select)");
#else
  return CAST_OK;
#endif
}

// 0 = ok; non-zero = a tensor-core pass timed out waiting for its MMAs (never expected; results invalid)
extern "C" int cast_topk_full_status(const void* workspace, long U, int V, int H, int K, int* host_flag,
                                     void* stream) {
  (void)U; (void)V; (void)H; (void)K;   // the flag sits at the start of the workspace
  if (!workspace || !host_flag) return set_error(CAST_ERR_BAD_ARG, "topk_full_status");
  const int* err = static_cast<const int*>(workspace);
#ifdef CAST_EMU
  *host_flag = *err;
  (void)stream;
#else
  if (cudaMemcpyAsync(host_flag, err, sizeof(int), cudaMemcpyDeviceToHost, (cudaStream_t)stream) != cudaSuccess)
    return set_error(CAST_ERR_CUDA, "topk_full_status");
  cudaStreamSynchronize((cudaStream_t)stream);
#endif
  return CAST_OK;
}
