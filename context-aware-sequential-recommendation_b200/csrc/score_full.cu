// K9 (full-catalog mode): rank of the target item among ALL items the user has not interacted with — the
// user-tile x item-tile GEMM of models/sasrec.py:93-97 (test_logits = seq_emb . item_emb^T, last position) fused with
// the rank-of-target count of util.py:318-321, with integer ranks that are exact.
//
//   canonical logit   s(u,j) = sum_k u[k]*e_j[k], k ascending, multiply and add rounded separately (fp32, no FMA) —
//                     the same arithmetic as cast_score_rank_cand and the oracle, so logits are bit-reproducible;
//   count_greater[u]  = #{ j in [1,V) : j != target(u), j not rated by u, s(u,j) >  s(u,target) }
//   count_equal[u]    = #{ ... same set ...                            s(u,j) == s(u,target) }
//
// Tensor-core path (mode 0).  The U x V x H contraction runs on the 5th-generation tensor cores: tcgen05.mma
// kind::tf32, a 128-user x 256-item fp32 accumulator tile in tensor memory, operands split in shared memory into
// tf32 hi + lo parts (3 MMAs per k-step: lo*hi + hi*lo + hi*hi, "3xTF32") so the tile is accurate to
// ~K * 2^-22 * |u||e_j|.  The epilogue (tcgen05.ld, one thread per user row) never trusts that approximation for a
// decision it could get wrong: with d = c_K * |u| * |e_j| a rigorous bound on its error, an item counts as greater
// when s~ > t + d, is dropped when s~ < t - d, and anything inside the band is re-scored with the canonical fp32 dot.
// Only integers leave the kernel (integer atomics => deterministic).  Rated items are subtracted afterwards by an
// exact gather kernel, so the tensor-core pass needs no per-user mask.
//
// Exact path (mode 1): the same counts by brute-force canonical dots (small catalogs, validation of mode 0).
#include "score_full.cuh"

namespace cast {

// per user: |u|_2 bound and the canonical target score (target id outside [1,V) scores 0 like the zero-pad row)
__global__ void user_prep_kernel(const float* __restrict__ users, long ldu, const float* __restrict__ table, int V,
                                 int H, long U, const int* __restrict__ target,
                                 const float* __restrict__ tscore_in, float* __restrict__ unorm,
                                 float* __restrict__ tscore) {
  const int lane = threadIdx.x & 31;
  const long u = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (u >= U) return;
  const float* ur = users + u * ldu;
  float s = 0.f;
  for (int k = lane; k < H; k += 32) s = fmaf(ur[k], ur[k], s);
  s = warp_sum(s);
  if (lane == 0) {
    unorm[u] = sqrtf(s) * NORM_SLACK;
    const int t = target[u];
    // tscore_in: the target lives in another rank's shard of the table; its canonical score was computed there
    tscore[u] = tscore_in ? tscore_in[u] : ((t > 0 && t < V) ? canonical_dot(ur, table + (long)t * H, H) : 0.f);
  }
}

// mode 1 / emulation: brute force over an item range per CTA row (blockIdx.y = user)
__global__ void score_full_exact_kernel(const float* __restrict__ users, long ldu, const float* __restrict__ table,
                                        int V, int H, const int* __restrict__ target,
                                        const float* __restrict__ tscore, long items_per_cta, int* __restrict__ cgt,
                                        int* __restrict__ ceq) {
  CAST_DYN_SMEM(float, us);
  const long u = blockIdx.y;
  for (int k = threadIdx.x; k < H; k += blockDim.x) us[k] = users[u * ldu + k];
  __syncthreads();
  const float t = tscore[u];
  const int tid = target[u];
  long j0 = (long)blockIdx.x * items_per_cta;
  long j1 = j0 + items_per_cta < V ? j0 + items_per_cta : V;
  if (j0 < 1) j0 = 1;
  int gt = 0, eq = 0;
  for (long j = j0 + threadIdx.x; j < j1; j += blockDim.x) {
    if (j == tid) continue;
    const float s = canonical_dot(us, table + j * H, H);
    gt += s > t ? 1 : 0;
    eq += s == t ? 1 : 0;
  }
  if (gt) atomicAdd(&cgt[u], gt);
  if (eq) atomicAdd(&ceq[u], eq);
}

// subtract the user's rated items (CSR, ids unique per user) that the catalog-wide pass counted
__global__ void rated_subtract_kernel(const float* __restrict__ users, long ldu, const float* __restrict__ table,
                                      int V, int H, long U, const int* __restrict__ target,
                                      const float* __restrict__ tscore, const int* __restrict__ rptr,
                                      const int* __restrict__ ridx, int* __restrict__ cgt, int* __restrict__ ceq) {
  const int lane = threadIdx.x & 31;
  const long u = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (u >= U) return;
  const float t = tscore[u];
  const int tid = target[u];
  int gt = 0, eq = 0;
  for (int p = rptr[u] + lane; p < rptr[u + 1]; p += 32) {
    const int j = ridx[p];
    if (j < 1 || j >= V || j == tid) continue;
    const float s = canonical_dot(users + u * ldu, table + (long)j * H, H);
    gt += s > t ? 1 : 0;
    eq += s == t ? 1 : 0;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    gt += __shfl_xor_sync(0xffffffffu, gt, o);
    eq += __shfl_xor_sync(0xffffffffu, eq, o);
  }
  if (lane == 0) {
    cgt[u] -= gt;
    ceq[u] -= eq;
  }
}

#ifndef CAST_EMU
// Deferred exact decisions: one thread per (user, item) pair that the tensor-core pass could not classify.  The
// canonical dot is a sequential chain, so the parallelism is across pairs (inline in the epilogue it would stall a
// whole warp per pair: measured 9 ms -> see profiles/r01e).
__global__ void band_rescore_kernel(const float* __restrict__ users, long ldu, const float* __restrict__ table, int H,
                                    const float* __restrict__ tscore, const int2* __restrict__ pairs,
                                    const unsigned long long* __restrict__ count, unsigned long long cap,
                                    int* __restrict__ cgt, int* __restrict__ ceq) {
  unsigned long long n = *count;
  if (n > cap) n = cap;
  for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (unsigned long long)gridDim.x * blockDim.x) {
    const int2 p = pairs[i];
    const float ex = canonical_dot(users + (long)p.x * ldu, table + (long)p.y * H, H);
    const float t = tscore[p.x];
    if (ex > t) atomicAdd(&cgt[p.x], 1);
    else if (ex == t) atomicAdd(&ceq[p.x], 1);
  }
}

// Epilogue of the tensor-core pass (sf_umma_kernel<CountEpi>): two compares per element against per-(user, tile)
// thresholds, band pairs appended to a list.
struct CountEpi {
  struct Params {
    const float* tscore;
    const int* target;
    int* cgt;
    int* ceq;
    unsigned long long* stats;        // [0] band candidates re-scored exactly  (optional)
    unsigned long long* band_count;   // device counter of deferred band pairs
    int2* band_pairs;                 // (user, item) pairs inside the error band, re-scored by band_rescore_kernel
    unsigned long long band_cap;
  };
  const SfPipe& a;
  const Params& p;
  const long me;
  const int je;
  const float tsc;
  const int tgt;
  int gt = 0;
  unsigned band = 0;
  float hi = 0.f, lo = 0.f;
  bool interior = false;

  __device__ __forceinline__ CountEpi(const SfPipe& a_, const Params& p_, long me_, bool live, int, int, int,
                                      int je_)
      : a(a_), p(p_), me(me_), je(je_), tsc(live ? p_.tscore[me_] : 0.f), tgt(live ? p_.target[me_] : -1) {}

  // above `hi` is certainly greater, below `lo` certainly smaller, in between the canonical fp32 logit decides
  // (deferred)
  __device__ __forceinline__ void tile(int j0, float d) {
    hi = tsc + d;
    lo = tsc - d;
    interior = j0 >= 1 && j0 + SF_N <= je && (tgt < j0 || tgt >= j0 + SF_N);  // no per-item exclusions
  }

  __device__ __forceinline__ void chunk(const float (&v)[32], int j) {
    unsigned inband = 0;
    if (interior) {
#pragma unroll
      for (int e = 0; e < 32; ++e) {
        gt += v[e] > hi ? 1 : 0;
        inband |= (v[e] >= lo && !(v[e] > hi)) ? (1u << e) : 0u;
      }
    } else {
#pragma unroll
      for (int e = 0; e < 32; ++e) {
        const int item = j + e;
        const bool valid = item >= 1 && item < je && item != tgt;
        gt += (valid && v[e] > hi) ? 1 : 0;
        inband |= (valid && v[e] >= lo && !(v[e] > hi)) ? (1u << e) : 0u;
      }
    }
    while (inband) {  // rare: hand the pair to band_rescore_kernel
      const int e = __ffs((int)inband) - 1;
      inband &= inband - 1;
      const int item = j + e;
      const unsigned long long slot = atomicAdd(p.band_count, 1ull);
      if (slot < p.band_cap) {
        p.band_pairs[slot] = make_int2((int)me, item);
      } else {  // list full: decide here (slow path)
        const float ex = canonical_dot(a.users + me * a.ldu, a.table + (long)item * a.H, a.H);
        if (ex > tsc) ++gt;
        else if (ex == tsc) atomicAdd(&p.ceq[me], 1);
      }
      ++band;
    }
  }

  __device__ __forceinline__ void finish() {
    if (gt) atomicAdd(&p.cgt[me], gt);
    if (p.stats && band) atomicAdd(&p.stats[0], (unsigned long long)band);
  }
};
#endif  // !CAST_EMU

}  // namespace cast

using namespace cast;

// capacity of the deferred band list: 0.5 % of the (user, item) pairs, at least 64k (overflow is handled inline)
static unsigned long long sf_band_cap(long U, int V) {
  unsigned long long c = (unsigned long long)U * (unsigned long long)V / 200ull;
  if (c < 65536ull) c = 65536ull;
  if (c > (1ull << 28)) c = 1ull << 28;
  return c;
}

extern "C" size_t cast_score_rank_full_workspace_bytes(long U, int V, int H) {
  return sf_align((size_t)V * 4) + 2 * sf_align((size_t)U * 4) + 256 + sf_presplit_bytes(U, V, H, nullptr) +
         sf_align((size_t)sf_band_cap(U, V) * sizeof(int2)) + sf_align((size_t)(V / 256 + 2) * 4);
}

extern "C" int cast_score_rank_full(const float* seq_last, long ld, const float* table, int V, int H, long U,
                                    const int* target, const float* target_score, const int* rated_ptr,
                                    const int* rated_idx, int mode,
                                    int* count_greater, int* count_equal, unsigned long long* stats, void* workspace,
                                    size_t workspace_bytes, void* stream) {
  if (!seq_last || !table || !target || !count_greater || !count_equal || V <= 1 || H <= 0 || U <= 0 ||
      (mode != 0 && mode != 1) || (rated_ptr && !rated_idx))
    return set_error(CAST_ERR_BAD_ARG, "score_rank_full");
  if (!workspace || workspace_bytes < cast_score_rank_full_workspace_bytes(U, V, H))
    return set_error(CAST_ERR_WORKSPACE, "score_rank_full: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  unsigned char* w = static_cast<unsigned char*>(workspace);
  float* inorm = reinterpret_cast<float*>(w);
  float* tscore = reinterpret_cast<float*>(w + sf_align((size_t)V * 4));
  float* unorm = reinterpret_cast<float*>(w + sf_align((size_t)V * 4) + sf_align((size_t)U * 4));
  int* err = reinterpret_cast<int*>(w + sf_align((size_t)V * 4) + 2 * sf_align((size_t)U * 4));
  int rc;
  cudaMemsetAsync(count_greater, 0, (size_t)U * sizeof(int), st);
  cudaMemsetAsync(count_equal, 0, (size_t)U * sizeof(int), st);
  cudaMemsetAsync(err, 0, sizeof(int), st);
  if (stats) cudaMemsetAsync(stats, 0, 2 * sizeof(unsigned long long), st);
  CAST_LAUNCH(user_prep_kernel, dim3((unsigned)cdiv(U, 4)), dim3(128), 0, st, seq_last, ld, table, V, H, U, target,
              target_score, unorm, tscore);
  if ((rc = check_launch("score_full(user_prep)"))) return rc;
#ifdef CAST_EMU
  mode = 1;  // the host emulation has no tensor cores; the exact path defines the same integers
#endif
  if (mode == 1) {
    const long per = 2048;
    CAST_LAUNCH(score_full_exact_kernel, dim3((unsigned)cdiv(V, per), (unsigned)U), dim3(128), H * sizeof(float), st,
                seq_last, ld, table, V, H, target, (const float*)tscore, per, count_greater, count_equal);
    if ((rc = check_launch("score_full(exact)"))) return rc;
  } else {
#ifndef CAST_EMU
    SfPipe a;
    unsigned char* pre = w + sf_align((size_t)V * 4) + 2 * sf_align((size_t)U * 4) + 256;
    CountEpi::Params ep;
    ep.band_pairs = reinterpret_cast<int2*>(pre + sf_presplit_bytes(U, V, H, nullptr));
    ep.band_cap = sf_band_cap(U, V);
    ep.band_count = reinterpret_cast<unsigned long long*>(err + 2);   // inside the 256-byte flag block
    cudaMemsetAsync(ep.band_count, 0, sizeof(unsigned long long), st);
    float* tnorm = reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(ep.band_pairs) +
                                            sf_align((size_t)ep.band_cap * sizeof(int2)));
    if ((rc = sf_prepare(a, seq_last, ld, table, V, H, U, pre, inorm, tnorm, st, "score_full(prepare)"))) return rc;
    a.unorm = unorm; a.err = err;
    sf_set_split(a, cdiv(148L * 2, cdiv(U, SF_M)));   // ~2 work units per SM
    ep.tscore = tscore; ep.target = target; ep.cgt = count_greater; ep.ceq = count_equal; ep.stats = stats;
    if ((rc = sf_launch<CountEpi>(a, ep, st, "score_full(umma)"))) return rc;
    band_rescore_kernel<<<dim3(148 * 8), dim3(256), 0, st>>>(seq_last, ld, table, H, (const float*)tscore,
                                                             (const int2*)ep.band_pairs, ep.band_count, ep.band_cap,
                                                             count_greater, count_equal);
    if ((rc = check_launch("score_full(band)"))) return rc;
#endif
  }
  if (rated_ptr) {
    CAST_LAUNCH(rated_subtract_kernel, dim3((unsigned)cdiv(U, 4)), dim3(128), 0, st, seq_last, ld, table, V, H, U,
                target, (const float*)tscore, rated_ptr, rated_idx, count_greater, count_equal);
    if ((rc = check_launch("score_full(rated)"))) return rc;
  }
  return CAST_OK;
}

// 0 = ok; non-zero = the tensor-core pass timed out waiting for its MMAs (never expected; results invalid)
extern "C" int cast_score_rank_full_status(const void* workspace, long U, int V, int* host_flag, void* stream) {
  // (the flag sits right after the norm / score arrays; H does not move it)
  if (!workspace || !host_flag) return set_error(CAST_ERR_BAD_ARG, "score_rank_full_status");
  const unsigned char* w = static_cast<const unsigned char*>(workspace);
  const int* err = reinterpret_cast<const int*>(w + sf_align((size_t)V * 4) + 2 * sf_align((size_t)U * 4));
#ifdef CAST_EMU
  *host_flag = *err;
  (void)stream;
#else
  if (cudaMemcpyAsync(host_flag, err, sizeof(int), cudaMemcpyDeviceToHost, (cudaStream_t)stream) != cudaSuccess)
    return set_error(CAST_ERR_CUDA, "score_rank_full_status");
  cudaStreamSynchronize((cudaStream_t)stream);
#endif
  return CAST_OK;
}
