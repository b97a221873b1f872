// K7: deterministic sparse embedding gradient.  TF's autodiff of `tf.nn.embedding_lookup` sums duplicate ids
// with unsorted_segment_sum (atomics, order not reproducible — SURVEY a9); here the (id, entry) pairs are put
// through a stable LSD radix sort (digits of <= 8 bits sized to the table, one warp per 256-key chunk, ranks by warp
// match/ballot) and each table row then sums its own segment in ascending entry order — no float atomics,
// bit-reproducible.  Entries enumerate up to 4 gradient sources of N positions each (item table: the input-sequence
// lookup x sqrt(H), the positive-item lookup and the negative-item lookup, models/sasrec.py:27,89-90).
#include "cast_rt.cuh"

namespace cast {

constexpr int RS_WARPS = 8;     // warps per CTA
constexpr int RS_CHUNK = 256;   // keys ranked by one warp

// counts of each digit per chunk: hist[digit * nchunks + chunk]
__global__ void radix_hist_kernel(const unsigned* __restrict__ keys, long n, int shift, unsigned mask, int nchunks,
                                  unsigned* __restrict__ hist) {
  __shared__ unsigned cnt[RS_WARPS][256];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int chunk = blockIdx.x * RS_WARPS + w;
  for (int i = lane; i <= (int)mask; i += 32) cnt[w][i] = 0u;
  __syncwarp();
  if (chunk < nchunks) {
    const long beg = (long)chunk * RS_CHUNK;
    const long end = beg + RS_CHUNK < n ? beg + RS_CHUNK : n;
    for (long i = beg + lane; i < end; i += 32) atomicAdd(&cnt[w][(keys[i] >> shift) & mask], 1u);
  }
  __syncwarp();
  if (chunk < nchunks)
    for (int i = lane; i <= (int)mask; i += 32) hist[(long)i * nchunks + chunk] = cnt[w][i];
}

// exclusive scan of `total` counters in place (single CTA of 1024 threads, integer => order-free)
__global__ void __launch_bounds__(1024) radix_scan_kernel(unsigned* __restrict__ hist, long total) {
  __shared__ unsigned wsum[32];
  const int t = threadIdx.x, lane = t & 31, w = t >> 5;
  const long per = (total + blockDim.x - 1) / blockDim.x;
  const long beg = (long)t * per;
  const long end = beg + per < total ? beg + per : total;
  unsigned s = 0;
  for (long i = beg; i < end; ++i) s += hist[i];
  unsigned inc = s;  // inclusive scan inside the warp
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned v = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += v;
  }
  if (lane == 31) wsum[w] = inc;
  __syncthreads();
  if (w == 0) {
    unsigned v = wsum[lane], vi = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned u = __shfl_up_sync(0xffffffffu, vi, o);
      if (lane >= o) vi += u;
    }
    wsum[lane] = vi - v;  // exclusive warp offsets
  }
  __syncthreads();
  unsigned run = wsum[w] + inc - s;
  for (long i = beg; i < end; ++i) {
    const unsigned v = hist[i];
    hist[i] = run;
    run += v;
  }
}

__global__ void radix_scatter_kernel(const unsigned* __restrict__ keys_in, const unsigned* __restrict__ pay_in, long n,
                                     int shift, unsigned mask, int nchunks, const unsigned* __restrict__ offs,
                                     unsigned* __restrict__ keys_out, unsigned* __restrict__ pay_out) {
  __shared__ unsigned base[RS_WARPS][256];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int chunk = blockIdx.x * RS_WARPS + w;
  if (chunk >= nchunks) return;  // warp-uniform; no block barriers below
  for (int i = lane; i <= (int)mask; i += 32) base[w][i] = offs[(long)i * nchunks + chunk];
  __syncwarp();
  const long beg = (long)chunk * RS_CHUNK;
  const long end = beg + RS_CHUNK < n ? beg + RS_CHUNK : n;
  for (long i0 = beg; i0 < end; i0 += 32) {
    const long i = i0 + lane;
    const bool valid = i < end;
    const unsigned k = valid ? keys_in[i] : 0u;
    const unsigned pay = valid ? (pay_in ? pay_in[i] : (unsigned)i) : 0u;
    const unsigned dgt = valid ? ((k >> shift) & mask) : (256u + lane);
    const unsigned peers = __match_any_sync(0xffffffffu, dgt);
    const int rank = __popc(peers & ((1u << lane) - 1u));
    const int leader = __ffs((int)peers) - 1;
    unsigned b = 0u;
    if (valid && lane == leader) {
      b = base[w][dgt];
      base[w][dgt] = b + (unsigned)__popc(peers);
    }
    b = __shfl_sync(0xffffffffu, b, leader);
    if (valid) {
      const unsigned p = b + (unsigned)rank;
      keys_out[p] = k;
      pay_out[p] = pay;
    }
    __syncwarp();
  }
}

struct ScatterSrc {
  const float* rows[4];
  const float* rowscale[4];
  float scale[4];
};

// sorted entries walked by one warp: 32 (one per lane: short walks, many warps in flight — sparse tables, remote rows)
// or 64 (heavily duplicated ids: half as many chunk partials to stitch per popular row).  0 = choose per call from
// the mean run length (entries per table row); cast_scatter_set_chunk forces one.
static int g_seg_chunk = 0;
// entries whose row loads are in flight together (NV = columns per lane): bounded so the staging registers stay <= 64

// Stage 1: every warp walks SEG_CHUNK consecutive sorted entries, lanes own columns.  Each lane first resolves two
// entries (key, scale factor, source row) in parallel; the walk then broadcasts them by shuffle, so the serial part
// only waits on the row loads (SEG_U rows in flight).  Segments (runs of equal key) inside the chunk are summed in
// entry order and written straight to dtable; a run that crosses a chunk boundary leaves a partial: part[w][0]
// ("head": the run began in an earlier chunk) and/or part[w][1] ("tail": the run begins here and continues).  Stage 2
// stitches the pieces of each crossing run in chunk order.  Work per warp is bounded by the chunk size however
// skewed the id distribution is (popular items own thousands of entries).
// Lazy form (LAZY = true; the dense form compiles without it): stamp[r] == *epoch marks a table row that already holds a gradient of the current backward
// pass.  The first segment sum that reaches row r in a pass writes it and stamps it, later ones (the other sources of
// the owner pull) add to it, so the table needs no zeroing pass and rows no batch touches are never written.  Each
// row is written by one warp per call and calls are stream-ordered: every lane reads the stamp before lane 0 moves it.
template <bool LAZY>
__device__ __forceinline__ bool row_adds(const unsigned* stamp, unsigned row, unsigned ep, int accumulate) {
  if (LAZY) return stamp[row] == ep;
  return accumulate != 0;
}
template <bool LAZY>
__device__ __forceinline__ void stamp_row(unsigned* stamp, unsigned row, unsigned ep, int lane) {
  if (!LAZY) return;
  __syncwarp();
  if (lane == 0) stamp[row] = ep;
}

template <int NV, int SEG_CHUNK, bool LAZY>
__global__ void segment_partial_kernel(const unsigned* __restrict__ skeys, const unsigned* __restrict__ spay,
                                       long total, long N, ScatterSrc src, unsigned klo, unsigned khi, int H,
                                       float* __restrict__ dtable, float* __restrict__ part, int* __restrict__ pkey,
                                       int accumulate, unsigned* __restrict__ stamp, const unsigned* __restrict__ epoch) {
  constexpr int SEG_Q = SEG_CHUNK / 32;
  cast_pdl_wait();
  cast_pdl_trigger();
  const int lane = threadIdx.x & 31;
  const long w = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const long beg = w * SEG_CHUNK;
  if (beg >= total) return;
  const long end = beg + SEG_CHUNK < total ? beg + SEG_CHUNK : total;
  const int cnt = (int)(end - beg);
  const unsigned ep = LAZY ? *epoch : 0u;
  constexpr int SEG_U = NV <= 2 ? 16 : (NV <= 8 ? 8 : (NV <= 16 ? 4 : 2));
  // ---- this lane's two entries
  unsigned mk[SEG_Q];
  float mf[SEG_Q];
  const float* mrow[SEG_Q];
#pragma unroll
  for (int q = 0; q < SEG_Q; ++q) {
    const long e = beg + lane + 32 * q;
    mk[q] = e < end ? skeys[e] : 0xffffffffu;
    mf[q] = 0.f;
    mrow[q] = nullptr;
    if (e < end && mk[q] != 0u && mk[q] >= klo && mk[q] < khi) {
      const unsigned p = spay ? spay[e] : (unsigned)e;
      const int s = (int)(p / N);
      const long n = (long)p - (long)s * N;
      mf[q] = src.scale[s] * (src.rowscale[s] ? src.rowscale[s][n] : 1.0f);
      mrow[q] = src.rows[s] + n * H;
    }
  }
  const unsigned last_key = __shfl_sync(0xffffffffu, mk[SEG_Q == 1 ? 0 : ((cnt - 1) >> 5)], (cnt - 1) & 31);
  const unsigned first_key = __shfl_sync(0xffffffffu, mk[0], 0);
  // sorted => the whole chunk is padding (id 0) or lies outside the key range of this call: contributes nothing
  if (last_key == 0u || last_key < klo || first_key >= khi) {
    if (lane == 0) { pkey[w * 2 + 0] = -1; pkey[w * 2 + 1] = -1; }
    return;
  }
  float acc[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) acc[i] = 0.f;
  unsigned cur = __shfl_sync(0xffffffffu, mk[0], 0);
  const bool first_open = beg > 0 && skeys[beg - 1] == cur;
  bool is_first = true;
  int head_key = -1, tail_key = -1;
  for (int e0 = 0; e0 < cnt; e0 += SEG_U) {
    unsigned k[SEG_U];
    float f[SEG_U];
    float val[SEG_U][NV];
#pragma unroll
    for (int u = 0; u < SEG_U; ++u) {
      const int e = e0 + u;  // < 64; entries >= cnt carry key 0xffffffff / null row
      const int q = SEG_Q == 1 ? 0 : (e >> 5), sl = e & 31;
      const unsigned kk = __shfl_sync(0xffffffffu, mk[q], sl);
      const float ff = __shfl_sync(0xffffffffu, mf[q], sl);
      const unsigned long long rp = __shfl_sync(0xffffffffu, (unsigned long long)mrow[q], sl);
      const float* row = reinterpret_cast<const float*>(rp);
      k[u] = kk;
      f[u] = ff;
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const int c = lane + 32 * i;
        val[u][i] = (row && c < H) ? row[c] : 0.f;
      }
    }
#pragma unroll
    for (int u = 0; u < SEG_U; ++u) {
      if (e0 + u >= cnt) break;
      if (k[u] != cur) {  // run of `cur` ends inside this chunk
        if (is_first && first_open) {
          head_key = (int)cur;
#pragma unroll
          for (int i = 0; i < NV; ++i) {
            const int c = lane + 32 * i;
            if (c < H) part[(w * 2 + 0) * H + c] = acc[i];
          }
        } else if (cur != 0u && cur >= klo && cur < khi) {
          const bool add = row_adds<LAZY>(stamp, cur - klo, ep, accumulate);
#pragma unroll
          for (int i = 0; i < NV; ++i) {
            const int c = lane + 32 * i;
            const long o = (long)(cur - klo) * H + c;
            if (c < H) dtable[o] = add ? dtable[o] + acc[i] : acc[i];
          }
          stamp_row<LAZY>(stamp, cur - klo, ep, lane);
        }
#pragma unroll
        for (int i = 0; i < NV; ++i) acc[i] = 0.f;
        cur = k[u];
        is_first = false;
      }
#pragma unroll
      for (int i = 0; i < NV; ++i) acc[i] = fmaf(val[u][i], f[u], acc[i]);
    }
  }
  const bool last_open = end < total && skeys[end] == cur;
  if (is_first && first_open) {
    head_key = (int)cur;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = lane + 32 * i;
      if (c < H) part[(w * 2 + 0) * H + c] = acc[i];
    }
  } else if (last_open) {
    tail_key = (int)cur;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = lane + 32 * i;
      if (c < H) part[(w * 2 + 1) * H + c] = acc[i];
    }
  } else if (cur != 0u && cur >= klo && cur < khi) {
    const bool add = row_adds<LAZY>(stamp, cur - klo, ep, accumulate);
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = lane + 32 * i;
      const long o = (long)(cur - klo) * H + c;
      if (c < H) dtable[o] = add ? dtable[o] + acc[i] : acc[i];
    }
    stamp_row<LAZY>(stamp, cur - klo, ep, lane);
  }
  if (lane == 0) {
    pkey[w * 2 + 0] = head_key;
    pkey[w * 2 + 1] = tail_key;
  }
}

// Stage 2: the chunk where a crossing run begins adds the following chunks' heads.  The run length is found 32 chunks
// per ballot; the sum uses ST_U interleaved accumulators (chunk j goes to accumulator j mod ST_U, each in ascending
// chunk order) folded in a fixed order at the end => still a fixed summation tree, with ST_U loads in flight.
template <int NV, bool LAZY>
__global__ void segment_stitch_kernel(const float* __restrict__ part, const int* __restrict__ pkey, long nchunks,
                                      unsigned klo, unsigned khi, int H, float* __restrict__ dtable, int accumulate,
                                      unsigned* __restrict__ stamp, const unsigned* __restrict__ epoch) {
  cast_pdl_wait();
  cast_pdl_trigger();
  const int lane = threadIdx.x & 31;
  const long w = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (w >= nchunks) return;
  const int key = pkey[w * 2 + 1];
  if (key <= 0 || (unsigned)key < klo || (unsigned)key >= khi) return;
  constexpr int ST_U = NV <= 2 ? 16 : (NV <= 4 ? 8 : (NV <= 8 ? 4 : 2));
  const unsigned ep = LAZY ? *epoch : 0u;
  long L = 0;  // chunks w+1 .. w+L continue the run
  for (;;) {
    const long w2 = w + 1 + L + lane;
    const bool cont = w2 < nchunks && pkey[w2 * 2 + 0] == key;
    const unsigned m = __ballot_sync(0xffffffffu, cont);
    if (m == 0xffffffffu) { L += 32; continue; }
    L += __ffs((int)~m) - 1;
    break;
  }
  float acc[ST_U][NV];
#pragma unroll
  for (int u = 0; u < ST_U; ++u)
#pragma unroll
    for (int i = 0; i < NV; ++i) acc[u][i] = 0.f;
  for (long j0 = 0; j0 < L; j0 += ST_U) {
    // all ST_U loads of the batch are issued before the first add (the run's chunks are summed by ONE warp: the walk
    // is a chain of L2 round trips unless the loads are in flight together); partial j goes to accumulator j mod ST_U
    float val[ST_U][NV];
#pragma unroll
    for (int u = 0; u < ST_U; ++u) {
      const long j = j0 + u;
      const float* src = part + ((w + 1 + (j < L ? j : 0)) * 2 + 0) * H;
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const int c = lane + 32 * i;
        val[u][i] = (j < L && c < H) ? src[c] : 0.f;
      }
    }
#pragma unroll
    for (int u = 0; u < ST_U; ++u)
#pragma unroll
      for (int i = 0; i < NV; ++i) acc[u][i] += val[u][i];
  }
  const bool add = row_adds<LAZY>(stamp, (unsigned)key - klo, ep, accumulate);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = lane + 32 * i;
    if (c < H) {
      float s = part[(w * 2 + 1) * H + c];
#pragma unroll
      for (int u = 0; u < ST_U; ++u) s += acc[u][i];
      const long o = (long)((unsigned)key - klo) * H + c;
      dtable[o] = add ? dtable[o] + s : s;
    }
  }
  stamp_row<LAZY>(stamp, (unsigned)key - klo, ep, lane);
}

// row-sharded table (TableRef, cast_rt.cuh): id -> owner-major key  (id % n) * R + id / n (+ 1 on shards 1..n-1), so
// that the sorted entries are grouped by owning rank and, inside a rank, by local row; ids outside (0, V) -> 0 = padding
__global__ void shard_keys_kernel(const int* __restrict__ ids, long total, int V, int n, int R,
                                  unsigned* __restrict__ out) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int id = ids[i];
    unsigned k = 0u;
    if (id > 0 && id < V) {
      const int o = id % n;
      k = (unsigned)o * (unsigned)R + (unsigned)(id / n + (o ? 1 : 0));
    }
    out[i] = k;
  }
}

// Owner pull, first half: the entries of a peer's sorted arrays whose key lies in [klo, khi) are fetched — one warp
// per entry, thousands of independent rows in flight over NVLink — into local staging (row e of `stage`, factor
// stage_f[e]); the segment sums then walk local memory.  (Walking the peer's rows directly serialises on NVLink
// latency: 450 us instead of 40 us for 38k rows of 1 KB.)
__global__ void pull_gather_kernel(const unsigned* __restrict__ skeys, const unsigned* __restrict__ spay, long total,
                                   long N, ScatterSrc src, unsigned klo, unsigned khi, int H,
                                   float* __restrict__ stage, float* __restrict__ stage_f) {
  const int lane = threadIdx.x & 31;
  const long e = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (e >= total) return;
  const unsigned k = skeys[e];
  if (k == 0u || k < klo || k >= khi) return;
  const unsigned p = spay[e];
  const int s = (int)(p / N);
  const long n = (long)p - (long)s * N;
  const float* row = src.rows[s] + n * H;
  float* out = stage + e * H;
  if ((H & 3) == 0) {
    for (int c = 4 * lane; c < H; c += 128) *reinterpret_cast<float4*>(out + c) = *reinterpret_cast<const float4*>(row + c);
  } else {
    for (int c = lane; c < H; c += 32) out[c] = row[c];
  }
  if (lane == 0) stage_f[e] = src.scale[s] * (src.rowscale[s] ? src.rowscale[s][n] : 1.0f);
}

// number of radix passes and digit width for a table of V rows (ids < V)
static inline void key_plan(int V, int* passes, int* dbits) {
  int bits = 1;
  while ((1L << bits) < (long)V) ++bits;
  *passes = (bits + 7) / 8;
  *dbits = (bits + *passes - 1) / *passes;
}

}  // namespace cast

using namespace cast;

// per-call scratch of the reduce half: chunk partials [nseg][2][H] followed by their keys [nseg][2]
extern "C" size_t cast_scatter_partial_bytes(long N, int nsrc, int H) {
  return (size_t)cdiv(N * nsrc, 32) * 2 * ((size_t)H * sizeof(float) + sizeof(int));   // (sized for 32-entry chunks)
}

extern "C" size_t cast_scatter_workspace_bytes(long N, int nsrc, int V) {
  const long total = N * nsrc;
  const long nchunks = cdiv(total, RS_CHUNK);
  (void)V;
  const long nseg = cdiv(total, 32);
  return (size_t)(5 * total + 256 * nchunks) * sizeof(unsigned) + (size_t)nseg * 2 * sizeof(int) + 64;
}

// Sort half of the scatter: depends on the ids only, so the engine runs it on a side stream at the start of the step,
// concurrently with the forward pass; the sorted (key, entry) arrays stay in the workspace for cast_scatter_apply.
static int scatter_sort_impl(const int* keys, int nsrc, long N, int V, int nshards, int rows_per_shard,
                             void* workspace, size_t workspace_bytes, void* stream) {
  if (!keys || nsrc < 1 || nsrc > 4 || N <= 0 || V <= 0) return set_error(CAST_ERR_BAD_ARG, "scatter_sort");
  const long total = N * nsrc;
  if (total >= (1L << 32)) return set_error(CAST_ERR_UNSUPPORTED, "scatter_sort: too many entries");
  if (!workspace || workspace_bytes < cast_scatter_workspace_bytes(N, nsrc, V))
    return set_error(CAST_ERR_WORKSPACE, "scatter_sort: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  const int nchunks = (int)cdiv(total, RS_CHUNK);
  unsigned* base = static_cast<unsigned*>(workspace);
  unsigned* bufK[2] = {base, base + total};
  unsigned* bufP[2] = {base + 2 * total, base + 3 * total};
  unsigned* hist = base + 5 * total;
  const unsigned* kin = reinterpret_cast<const unsigned*>(keys);
  const unsigned* pin = nullptr;
  int passes, dbits, rc;
  if (nshards > 1) {  // sort by (owner, local row)
    if ((long)nshards * rows_per_shard < V) return set_error(CAST_ERR_BAD_ARG, "scatter_sort: shards do not cover V");
    unsigned* tk = base + 4 * total;
    CAST_LAUNCH(shard_keys_kernel, dim3((unsigned)cdiv(total, 256) < 1184u ? (unsigned)cdiv(total, 256) : 1184u),
                dim3(256), 0, st, keys, total, V, nshards, rows_per_shard, tk);
    if ((rc = check_launch("shard_keys"))) return rc;
    kin = tk;
    V = nshards * rows_per_shard;
  }
  key_plan(V, &passes, &dbits);
  const unsigned mask = (1u << dbits) - 1u;
  const int nblk = (int)cdiv(nchunks, RS_WARPS);
  for (int p = 0; p < passes; ++p) {
    unsigned* kout = bufK[p & 1];
    unsigned* pout = bufP[p & 1];
    CAST_LAUNCH(radix_hist_kernel, dim3(nblk), dim3(32 * RS_WARPS), 0, st, kin, total, dbits * p, mask, nchunks, hist);
    if ((rc = check_launch("radix_hist"))) return rc;
    CAST_LAUNCH(radix_scan_kernel, dim3(1), dim3(1024), 0, st, hist, (long)(mask + 1) * nchunks);
    if ((rc = check_launch("radix_scan"))) return rc;
    CAST_LAUNCH(radix_scatter_kernel, dim3(nblk), dim3(32 * RS_WARPS), 0, st, kin, pin, total, dbits * p, mask, nchunks,
                (const unsigned*)hist, kout, pout);
    if ((rc = check_launch("radix_scatter"))) return rc;
    kin = kout;
    pin = pout;
  }
  return CAST_OK;
}

/* tuning hook: sorted entries per warp in the segment sums (32 or 64) */
extern "C" int cast_scatter_set_chunk(int entries) {
  if (entries != 0 && entries != 32 && entries != 64) return set_error(CAST_ERR_BAD_ARG, "scatter_set_chunk: 0, 32 or 64");
  g_seg_chunk = entries;
  return CAST_OK;
}

extern "C" int cast_scatter_sort(const int* keys, int nsrc, long N, int V, void* workspace, size_t workspace_bytes,
                                 void* stream) {
  return scatter_sort_impl(keys, nsrc, N, V, 1, 0, workspace, workspace_bytes, stream);
}

/* the same sort on owner-major keys (row-sharded table: nshards ranks x rows_per_shard local rows, TableRef) */
extern "C" int cast_scatter_sort_sharded(const int* keys, int nsrc, long N, int V, int nshards, int rows_per_shard,
                                         void* workspace, size_t workspace_bytes, void* stream) {
  if (nshards < 1 || rows_per_shard < 1) return set_error(CAST_ERR_BAD_ARG, "scatter_sort_sharded");
  return scatter_sort_impl(keys, nsrc, N, V, nshards, rows_per_shard, workspace, workspace_bytes, stream);
}

/* byte offsets, inside a sort workspace for (N, nsrc, key range Vkeys), of the sorted keys and of their payloads */
extern "C" int cast_scatter_sorted_offsets(long N, int nsrc, int Vkeys, size_t* keys_offset, size_t* payload_offset) {
  if (N <= 0 || nsrc < 1 || Vkeys <= 0 || !keys_offset || !payload_offset)
    return set_error(CAST_ERR_BAD_ARG, "scatter_sorted_offsets");
  const long total = N * nsrc;
  int passes, dbits;
  key_plan(Vkeys, &passes, &dbits);
  const int last = (passes - 1) & 1;   // buffer pair the final pass wrote
  *keys_offset = ((size_t)last * total) * sizeof(unsigned);
  *payload_offset = (2 * (size_t)total + (size_t)last * total) * sizeof(unsigned);
  return CAST_OK;
}

// Reduce half: fixed-order segment sums of the rows whose sorted key lies in [klo, khi), written to dtable row key - klo
static int scatter_apply_impl(int nsrc, long N, const float* const* rows, const float* const* rowscale,
                              const float* scale, int H, float* dtable, long dtable_rows, const unsigned* kin,
                              const unsigned* pin, unsigned klo, unsigned khi, void* partial, size_t partial_bytes,
                              int accumulate, unsigned* stamp, const unsigned* epoch, void* stream) {
  if (!rows || !scale || !dtable || !kin || nsrc < 1 || nsrc > 4 || N <= 0 || H <= 0 || H > 1024 || khi <= klo ||
      (stamp && !epoch))
    return set_error(CAST_ERR_BAD_ARG, "scatter_apply");
  const long total = N * nsrc;
  if (!partial || partial_bytes < cast_scatter_partial_bytes(N, nsrc, H))
    return set_error(CAST_ERR_WORKSPACE, "scatter_apply: partial buffer too small");
  cudaStream_t st = (cudaStream_t)stream;
  int rc;
  ScatterSrc src;
  for (int s = 0; s < 4; ++s) {
    src.rows[s] = s < nsrc ? rows[s] : nullptr;
    src.rowscale[s] = (s < nsrc && rowscale) ? rowscale[s] : nullptr;
    src.scale[s] = s < nsrc ? scale[s] : 0.f;
  }
  // rows nobody touches (and row 0) must read as zero: dense-gradient semantics of the reference
  // (accumulate: dtable already holds the sum of an earlier call over other sources; every row is written at most
  // once per call, so adding to it is race-free and keeps a fixed summation order)
  // (lazy form: no zeroing; the stamps tell which rows hold this pass's gradient)
  if (!accumulate && !stamp) cudaMemsetAsync(dtable, 0, (size_t)dtable_rows * H * sizeof(float), st);
  const int chunk = g_seg_chunk ? g_seg_chunk : (total >= 8 * ((long)khi - (long)klo) ? 64 : 32);
  const long nseg = cdiv(total, chunk);
  float* part = static_cast<float*>(partial);
  int* pkey = reinterpret_cast<int*>(part + (size_t)nseg * 2 * H);
  const int wpb = 4;
  const dim3 grid((unsigned)cdiv(nseg, wpb)), block(32 * wpb);
#define CAST_SEG(NV, LZ)                                                                                        \
  {                                                                                                             \
    if (chunk == 32) {                                                                                          \
      CAST_LAUNCH_DEP((segment_partial_kernel<NV, 32, LZ>), grid, block, 0, st, kin, pin, total, N, src, klo, khi, \
                  H, dtable, part, pkey, accumulate, stamp, epoch);                                             \
    } else {                                                                                                    \
      CAST_LAUNCH_DEP((segment_partial_kernel<NV, 64, LZ>), grid, block, 0, st, kin, pin, total, N, src, klo, khi, \
                  H, dtable, part, pkey, accumulate, stamp, epoch);                                             \
    }                                                                                                           \
    if ((rc = check_launch("segment_partial"))) return rc;                                                      \
    CAST_LAUNCH_DEP((segment_stitch_kernel<NV, LZ>), grid, block, 0, st, (const float*)part, (const int*)pkey,  \
                nseg, klo, khi, H, dtable, accumulate, stamp, epoch);                                           \
  }
#define CAST_SEG_H(LZ)                                                                                          \
  if (H <= 64) CAST_SEG(2, LZ)                                                                                  \
  else if (H <= 128) CAST_SEG(4, LZ)                                                                            \
  else if (H <= 256) CAST_SEG(8, LZ)                                                                            \
  else if (H <= 512) CAST_SEG(16, LZ)                                                                           \
  else CAST_SEG(32, LZ)
  if (stamp) {
    CAST_SEG_H(true)
  } else {
    CAST_SEG_H(false)
  }
#undef CAST_SEG_H
#undef CAST_SEG
  return check_launch("segment_stitch");
}

// ... over the arrays cast_scatter_sort left in the workspace, whole table
extern "C" int cast_scatter_apply(int nsrc, long N, const float* const* rows, const float* const* rowscale,
                                  const float* scale, int V, int H, float* dtable, void* workspace,
                                  size_t workspace_bytes, void* partial, size_t partial_bytes, int accumulate,
                                  void* stream) {
  if (N <= 0 || nsrc < 1 || V <= 0) return set_error(CAST_ERR_BAD_ARG, "scatter_apply");
  if (!workspace || workspace_bytes < cast_scatter_workspace_bytes(N, nsrc, V))
    return set_error(CAST_ERR_WORKSPACE, "scatter_apply: workspace too small");
  size_t ko, po;
  cast_scatter_sorted_offsets(N, nsrc, V, &ko, &po);
  const unsigned char* w = static_cast<const unsigned char*>(workspace);
  return scatter_apply_impl(nsrc, N, rows, rowscale, scale, H, dtable, V, reinterpret_cast<const unsigned*>(w + ko),
                            reinterpret_cast<const unsigned*>(w + po), 0u, (unsigned)V, partial, partial_bytes,
                            accumulate, nullptr, nullptr, stream);
}

/* cast_scatter_apply's lazy form (optimizer "lazy_adam"): no zeroing pass over the table; a row the batch touches is
 * written (stamp[row] != *epoch) or added to (== *epoch) and then stamped, a row it does not touch keeps stale data
 * and its old stamp.  stamp [V] and epoch are device memory; the epoch advances once per backward pass. */
extern "C" int cast_scatter_apply_lazy(int nsrc, long N, const float* const* rows, const float* const* rowscale,
                                       const float* scale, int V, int H, float* dtable, void* workspace,
                                       size_t workspace_bytes, void* partial, size_t partial_bytes, unsigned* stamp,
                                       const unsigned* epoch, void* stream) {
  if (N <= 0 || nsrc < 1 || V <= 0 || !stamp || !epoch) return set_error(CAST_ERR_BAD_ARG, "scatter_apply_lazy");
  if (!workspace || workspace_bytes < cast_scatter_workspace_bytes(N, nsrc, V))
    return set_error(CAST_ERR_WORKSPACE, "scatter_apply_lazy: workspace too small");
  size_t ko, po;
  cast_scatter_sorted_offsets(N, nsrc, V, &ko, &po);
  const unsigned char* w = static_cast<const unsigned char*>(workspace);
  return scatter_apply_impl(nsrc, N, rows, rowscale, scale, H, dtable, V, reinterpret_cast<const unsigned*>(w + ko),
                            reinterpret_cast<const unsigned*>(w + po), 0u, (unsigned)V, partial, partial_bytes, 0,
                            stamp, epoch, stream);
}

/* Owner side of the row-sharded embedding gradient (SURVEY §8e): fold the entries of ONE rank's sorted arrays
 * (sorted_keys / sorted_payload: device pointers, possibly that rank's memory read over NVLink; made by
 * cast_scatter_sort_sharded for N x nsrc entries) whose owner-major key lies in [key_lo, key_hi) — this rank's rows —
 * into dtable [key_hi - key_lo, H] (row = key - key_lo).  rows / rowscale are that rank's source tensors.  Called once
 * per rank in rank order (accumulate = 0 for the first) the sum over ranks has a fixed order: bit-reproducible. */
extern "C" int cast_scatter_apply_range(int nsrc, long N, const float* const* rows, const float* const* rowscale,
                                        const float* scale, int H, float* dtable, const void* sorted_keys,
                                        const void* sorted_payload, unsigned key_lo, unsigned key_hi, void* partial,
                                        size_t partial_bytes, int accumulate, void* stream) {
  return scatter_apply_impl(nsrc, N, rows, rowscale, scale, H, dtable, (long)key_hi - (long)key_lo,
                            static_cast<const unsigned*>(sorted_keys), static_cast<const unsigned*>(sorted_payload),
                            key_lo, key_hi, partial, partial_bytes, accumulate, nullptr, nullptr, stream);
}

/* lazy form of cast_scatter_apply_range (stamps of dtable's rows, see cast_scatter_apply_lazy): every rank's call
 * writes or adds by the stamps, so the rank-ordered calls need no accumulate flag and no zeroing pass */
extern "C" int cast_scatter_apply_range_lazy(int nsrc, long N, const float* const* rows, const float* const* rowscale,
                                             const float* scale, int H, float* dtable, const void* sorted_keys,
                                             const void* sorted_payload, unsigned key_lo, unsigned key_hi,
                                             void* partial, size_t partial_bytes, unsigned* stamp,
                                             const unsigned* epoch, void* stream) {
  if (!stamp || !epoch) return set_error(CAST_ERR_BAD_ARG, "scatter_apply_range_lazy");
  return scatter_apply_impl(nsrc, N, rows, rowscale, scale, H, dtable, (long)key_hi - (long)key_lo,
                            static_cast<const unsigned*>(sorted_keys), static_cast<const unsigned*>(sorted_payload),
                            key_lo, key_hi, partial, partial_bytes, 0, stamp, epoch, stream);
}

/* cast_scatter_apply_range for a PEER's entries: its in-range rows are first gathered into `stage`
 * (cast_scatter_stage_bytes: N*nsrc rows + factors, local memory) with one warp per entry, then summed locally with
 * the same arithmetic (bit-identical to cast_scatter_apply_range on the same data). */
extern "C" size_t cast_scatter_stage_bytes(long N, int nsrc, int H) {
  return (size_t)N * nsrc * ((size_t)H + 1) * sizeof(float) + 256;
}

static int scatter_pull_range_impl(int nsrc, long N, const float* const* rows, const float* const* rowscale,
                                   const float* scale, int H, float* dtable, const void* sorted_keys,
                                   const void* sorted_payload, unsigned key_lo, unsigned key_hi, void* stage,
                                   size_t stage_bytes, void* partial, size_t partial_bytes, int accumulate,
                                   unsigned* stamp, const unsigned* epoch, void* stream) {
  if (!rows || !scale || !sorted_keys || !sorted_payload || nsrc < 1 || nsrc > 4 || N <= 0 || H <= 0)
    return set_error(CAST_ERR_BAD_ARG, "scatter_pull_range");
  if (!stage || stage_bytes < cast_scatter_stage_bytes(N, nsrc, H))
    return set_error(CAST_ERR_WORKSPACE, "scatter_pull_range: staging buffer too small");
  const long total = N * nsrc;
  ScatterSrc src;
  for (int s = 0; s < 4; ++s) {
    src.rows[s] = s < nsrc ? rows[s] : nullptr;
    src.rowscale[s] = (s < nsrc && rowscale) ? rowscale[s] : nullptr;
    src.scale[s] = s < nsrc ? scale[s] : 0.f;
  }
  float* st_rows = static_cast<float*>(stage);
  float* st_f = st_rows + (size_t)total * H;
  const int wpb = 8;
  CAST_LAUNCH(pull_gather_kernel, dim3((unsigned)cdiv(total, wpb)), dim3(32 * wpb), 0, (cudaStream_t)stream,
              static_cast<const unsigned*>(sorted_keys), static_cast<const unsigned*>(sorted_payload), total, N, src,
              key_lo, key_hi, H, st_rows, st_f);
  int rc = check_launch("pull_gather");
  if (rc) return rc;
  const float* lrows[1] = {st_rows};
  const float* lscale_rows[1] = {st_f};
  const float one[1] = {1.0f};
  return scatter_apply_impl(1, total, lrows, lscale_rows, one, H, dtable, (long)key_hi - (long)key_lo,
                            static_cast<const unsigned*>(sorted_keys), nullptr, key_lo, key_hi, partial, partial_bytes,
                            accumulate, stamp, epoch, stream);
}

extern "C" int cast_scatter_pull_range(int nsrc, long N, const float* const* rows, const float* const* rowscale,
                                       const float* scale, int H, float* dtable, const void* sorted_keys,
                                       const void* sorted_payload, unsigned key_lo, unsigned key_hi, void* stage,
                                       size_t stage_bytes, void* partial, size_t partial_bytes, int accumulate,
                                       void* stream) {
  return scatter_pull_range_impl(nsrc, N, rows, rowscale, scale, H, dtable, sorted_keys, sorted_payload, key_lo,
                                 key_hi, stage, stage_bytes, partial, partial_bytes, accumulate, nullptr, nullptr,
                                 stream);
}

/* lazy form of cast_scatter_pull_range (stamps of dtable's rows, see cast_scatter_apply_lazy) */
extern "C" int cast_scatter_pull_range_lazy(int nsrc, long N, const float* const* rows, const float* const* rowscale,
                                            const float* scale, int H, float* dtable, const void* sorted_keys,
                                            const void* sorted_payload, unsigned key_lo, unsigned key_hi, void* stage,
                                            size_t stage_bytes, void* partial, size_t partial_bytes, unsigned* stamp,
                                            const unsigned* epoch, void* stream) {
  if (!stamp || !epoch) return set_error(CAST_ERR_BAD_ARG, "scatter_pull_range_lazy");
  return scatter_pull_range_impl(nsrc, N, rows, rowscale, scale, H, dtable, sorted_keys, sorted_payload, key_lo,
                                 key_hi, stage, stage_bytes, partial, partial_bytes, 0, stamp, epoch, stream);
}

extern "C" int cast_scatter_rows(const int* keys, int nsrc, long N, const float* const* rows,
                                 const float* const* rowscale, const float* scale, int V, int H, float* dtable,
                                 void* workspace, size_t workspace_bytes, void* partial, size_t partial_bytes,
                                 void* stream) {
  int rc = cast_scatter_sort(keys, nsrc, N, V, workspace, workspace_bytes, stream);
  if (rc) return rc;
  return cast_scatter_apply(nsrc, N, rows, rowscale, scale, V, H, dtable, workspace, workspace_bytes, partial,
                            partial_bytes, 0, stream);
}
