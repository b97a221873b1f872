// K8: tf.train.AdamOptimizer(learning_rate=lr, beta2=0.98) (models/sasrec.py:120-121) as one fused pass over the
// flat parameter buffer.  TF-1.15 semantics: lr_t = lr*sqrt(1-beta2^t)/(1-beta1^t); m,v updated on EVERY element of
// every variable (the embedding tables too: the zero-pad concat makes their gradient dense, SURVEY a10), epsilon
// added to sqrt(v) outside the root.  beta powers are fp32 state multiplied after the update, like TF's
// beta1_power / beta2_power variables.  HBM-bound: 16 B read + 12 B written per parameter.
#include "cast_rt.cuh"

namespace cast {

struct AdamState {
  float b1p, b2p;
  unsigned long long step;
};

__global__ void adam_init_kernel(AdamState* st, float b1, float b2) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    st->b1p = b1;
    st->b2p = b2;
    st->step = 0ull;
  }
}

// One element of the update.  The contractions are written out (fmaf) so that every kernel below — scalar, 16-byte
// and the peer-summing form — rounds identically: a data-parallel run stays bit-comparable with a single-process one.
// CLIP (global-norm clipping) multiplies the gradient, l2 term included, by the step's scale; x * 1.0f == x, so a step
// below the threshold gives the bits of the unclipped update.
template <bool CLIP = false>
__device__ __forceinline__ void adam_elem(float& w, float& m, float& v, float g, bool decay, float l2, float b1,
                                          float omb1, float b2, float omb2, float lr_t, float eps, float scale = 1.0f) {
  if (decay) g = fmaf(l2, w, g);
  if (CLIP) g = g * scale;
  m = fmaf(b1, m, omb1 * g);
  v = fmaf(b2, v, (omb2 * g) * g);
  w = w - (lr_t * m) / (sqrtf(v) + eps);
}

// the kernels below come in two forms, plain and CLIP (the scale read from clip[0]); both share one body
template <bool CLIP>
__device__ __forceinline__ void adam_step_body(float* __restrict__ w, const float* __restrict__ grad,
                                               float* __restrict__ m, float* __restrict__ v, long n, float lr, float b1,
                                               float b2, float eps, const float* __restrict__ gdenom, float l2,
                                               long l2_lo, long l2_hi, const AdamState* __restrict__ st,
                                               const float* __restrict__ clip) {
  cast_pdl_wait();
  cast_pdl_trigger();
  const float gs = gdenom ? 1.0f / *gdenom : 1.0f;
  const float sc = CLIP ? clip[0] : 1.0f;
  const float lr_t = lr * sqrtf(1.0f - st->b2p) / (1.0f - st->b1p);
  const float omb1 = 1.0f - b1, omb2 = 1.0f - b2;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    float wi = w[i], mi = m[i], vi = v[i];
    adam_elem<CLIP>(wi, mi, vi, grad[i] * gs, i >= l2_lo && i < l2_hi, l2, b1, omb1, b2, omb2, lr_t, eps, sc);
    m[i] = mi;
    v[i] = vi;
    w[i] = wi;
  }
}

__global__ void adam_step_kernel(float* __restrict__ w, const float* __restrict__ grad, float* __restrict__ m,
                                 float* __restrict__ v, long n, float lr, float b1, float b2, float eps,
                                 const float* __restrict__ gdenom, float l2, long l2_lo, long l2_hi,
                                 const AdamState* __restrict__ st) {
  adam_step_body<false>(w, grad, m, v, n, lr, b1, b2, eps, gdenom, l2, l2_lo, l2_hi, st, nullptr);
}

__global__ void adam_step_clip_kernel(float* __restrict__ w, const float* __restrict__ grad, float* __restrict__ m,
                                      float* __restrict__ v, long n, float lr, float b1, float b2, float eps,
                                      const float* __restrict__ gdenom, float l2, long l2_lo, long l2_hi,
                                      const AdamState* __restrict__ st, const float* __restrict__ clip) {
  adam_step_body<true>(w, grad, m, v, n, lr, b1, b2, eps, gdenom, l2, l2_lo, l2_hi, st, clip);
}

// same update, four elements per thread (16-byte loads/stores); n4 = n/4, pointers 16-byte aligned
template <bool CLIP>
__device__ __forceinline__ void adam_step_vec4_body(float4* __restrict__ w, const float4* __restrict__ grad,
                                                    float4* __restrict__ m, float4* __restrict__ v, long n4, float lr,
                                                    float b1, float b2, float eps, const float* __restrict__ gdenom,
                                                    float l2, long l2_lo, long l2_hi,
                                                    const AdamState* __restrict__ st, const float* __restrict__ clip) {
  cast_pdl_wait();
  cast_pdl_trigger();
  const float gs = gdenom ? 1.0f / *gdenom : 1.0f;
  const float sc = CLIP ? clip[0] : 1.0f;
  const float lr_t = lr * sqrtf(1.0f - st->b2p) / (1.0f - st->b1p);
  const float omb1 = 1.0f - b1, omb2 = 1.0f - b2;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    const float4 wi = w[i], gi = grad[i], mi = m[i], vi = v[i];
    float wv[4] = {wi.x, wi.y, wi.z, wi.w}, gv[4] = {gi.x, gi.y, gi.z, gi.w};
    float mv[4] = {mi.x, mi.y, mi.z, mi.w}, vv[4] = {vi.x, vi.y, vi.z, vi.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const long idx = 4 * i + e;
      adam_elem<CLIP>(wv[e], mv[e], vv[e], gv[e] * gs, idx >= l2_lo && idx < l2_hi, l2, b1, omb1, b2, omb2, lr_t,
                      eps, sc);
    }
    m[i] = make_float4(mv[0], mv[1], mv[2], mv[3]);
    v[i] = make_float4(vv[0], vv[1], vv[2], vv[3]);
    w[i] = make_float4(wv[0], wv[1], wv[2], wv[3]);
  }
}

__global__ void adam_step_vec4_kernel(float4* __restrict__ w, const float4* __restrict__ grad, float4* __restrict__ m,
                                      float4* __restrict__ v, long n4, float lr, float b1, float b2, float eps,
                                      const float* __restrict__ gdenom, float l2, long l2_lo, long l2_hi,
                                      const AdamState* __restrict__ st) {
  adam_step_vec4_body<false>(w, grad, m, v, n4, lr, b1, b2, eps, gdenom, l2, l2_lo, l2_hi, st, nullptr);
}

__global__ void adam_step_vec4_clip_kernel(float4* __restrict__ w, const float4* __restrict__ grad,
                                           float4* __restrict__ m, float4* __restrict__ v, long n4, float lr, float b1,
                                           float b2, float eps, const float* __restrict__ gdenom, float l2, long l2_lo,
                                           long l2_hi, const AdamState* __restrict__ st,
                                           const float* __restrict__ clip) {
  adam_step_vec4_body<true>(w, grad, m, v, n4, lr, b1, b2, eps, gdenom, l2, l2_lo, l2_hi, st, clip);
}

// Data-parallel form: the gradient of element i is the sum over the n ranks' buffers in rank order (own buffer + peer
// mappings read over NVLink), formed inside the optimizer pass instead of by a separate reduction launch.  The loads
// of one element group from all ranks are issued together (a serial walk pays one NVLink round trip per rank).  The
// buffers hold `np` gradient numerators followed by `tail` >= 3 sums [loss_sum, auc_sum, count, ...]: the reduced
// count is the gradient denominator; every reduced element is also written to g_red (loss read-back, diagnostics).
constexpr int ADAM_PEER_BATCH = 8;
__global__ void adam_step_peers_kernel(float* __restrict__ w, const float* const* __restrict__ g, int n,
                                       float* __restrict__ g_red, float* __restrict__ m, float* __restrict__ v,
                                       long lo, long np, long tail, float lr, float b1, float b2, float eps, float l2,
                                       long l2_lo, long l2_hi, const AdamState* __restrict__ st) {
  __shared__ float s_count;
  cast_pdl_wait();
  cast_pdl_trigger();
  if (threadIdx.x == 0) {
    float c = g[0][np + 2];
    for (int r = 1; r < n; ++r) c += g[r][np + 2];
    s_count = c;
  }
  __syncthreads();
  const float gs = 1.0f / s_count;
  const float lr_t = lr * sqrtf(1.0f - st->b2p) / (1.0f - st->b1p);
  const float omb1 = 1.0f - b1, omb2 = 1.0f - b2;
  const long total = np + tail;
  // elements below `lo` are neither reduced nor updated (lo = 0 but for the lazy optimizer, whose row pass owns them);
  // groups of 4 stay aligned to the buffers, the one that straddles `lo` goes element by element
  for (long i0 = (lo & ~3L) + 4 * ((long)blockIdx.x * blockDim.x + threadIdx.x); i0 < total;
       i0 += 4 * (long)gridDim.x * blockDim.x) {
    float gv[4] = {0.f, 0.f, 0.f, 0.f};
    const int cnt = total - i0 < 4 ? (int)(total - i0) : 4;
    const int e0 = i0 < lo ? (int)(lo - i0) : 0;
    if (cnt == 4 && e0 == 0) {
      for (int r0 = 0; r0 < n; r0 += ADAM_PEER_BATCH) {
        float4 q[ADAM_PEER_BATCH];
#pragma unroll
        for (int u = 0; u < ADAM_PEER_BATCH; ++u)
          if (r0 + u < n) q[u] = *reinterpret_cast<const float4*>(g[r0 + u] + i0);
#pragma unroll
        for (int u = 0; u < ADAM_PEER_BATCH; ++u)
          if (r0 + u < n) {
            if (r0 + u == 0) {
              gv[0] = q[u].x; gv[1] = q[u].y; gv[2] = q[u].z; gv[3] = q[u].w;
            } else {
              gv[0] += q[u].x; gv[1] += q[u].y; gv[2] += q[u].z; gv[3] += q[u].w;
            }
          }
      }
      *reinterpret_cast<float4*>(g_red + i0) = make_float4(gv[0], gv[1], gv[2], gv[3]);
    } else {
      for (int e = e0; e < cnt; ++e) {
        float sacc = g[0][i0 + e];
        for (int r = 1; r < n; ++r) sacc += g[r][i0 + e];
        gv[e] = sacc;
        g_red[i0 + e] = sacc;
      }
    }
    const int na = np - i0 >= 4 ? 4 : (np - i0 > 0 ? (int)(np - i0) : 0);  // elements of this group that are parameters
    if (na == 4 && e0 == 0) {
      const float4 wi = *reinterpret_cast<const float4*>(w + i0), mi = *reinterpret_cast<const float4*>(m + i0),
                   vi = *reinterpret_cast<const float4*>(v + i0);
      float wv[4] = {wi.x, wi.y, wi.z, wi.w}, mv[4] = {mi.x, mi.y, mi.z, mi.w}, vv[4] = {vi.x, vi.y, vi.z, vi.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const long idx = i0 + e;
        adam_elem(wv[e], mv[e], vv[e], gv[e] * gs, idx >= l2_lo && idx < l2_hi, l2, b1, omb1, b2, omb2, lr_t, eps);
      }
      *reinterpret_cast<float4*>(m + i0) = make_float4(mv[0], mv[1], mv[2], mv[3]);
      *reinterpret_cast<float4*>(v + i0) = make_float4(vv[0], vv[1], vv[2], vv[3]);
      *reinterpret_cast<float4*>(w + i0) = make_float4(wv[0], wv[1], wv[2], wv[3]);
    } else {
      for (int e = e0; e < na; ++e) {
        const long idx = i0 + e;
        float wi = w[idx], mi = m[idx], vi = v[idx];
        adam_elem(wi, mi, vi, gv[e] * gs, idx >= l2_lo && idx < l2_hi, l2, b1, omb1, b2, omb2, lr_t, eps);
        m[idx] = mi;
        v[idx] = vi;
        w[idx] = wi;
      }
    }
  }
}

// ---- lazy TF-Adam (optimizer "lazy_adam", tf.contrib.opt.LazyAdamOptimizer on the item table)
// A table row is updated iff this backward pass wrote its gradient (stamp[r] == *epoch, see cast_scatter_apply_lazy);
// every other row keeps w, m and v bit for bit.  The element arithmetic is adam_elem with the dense pass's lr_t and
// 1/count, so a touched row gets exactly the bits the dense kernel would give it.  One warp per `rpw` <= 32 consecutive
// rows: the lanes read the rpw stamps at once, then the warp updates the touched rows one by one, lanes over columns.
// rpw is 32 for a large table (one coalesced stamp read per 32 rows) and shrinks until a small table still gives every
// SM warps to run (rows_per_warp).
__global__ void grad_epoch_advance_kernel(unsigned* epoch) {
  cast_pdl_wait();
  cast_pdl_trigger();
  if (threadIdx.x == 0 && blockIdx.x == 0) *epoch += 1u;
}

template <bool CLIP = false>
__device__ __forceinline__ void adam_row(float* __restrict__ w, float* __restrict__ m, float* __restrict__ v,
                                         const float* __restrict__ g, int H, bool vec, float gs, float b1, float omb1,
                                         float b2, float omb2, float lr_t, float eps, int lane, float sc = 1.0f) {
  if (vec) {
    for (int c = 4 * lane; c < H; c += 128) {
      const float4 wi = *reinterpret_cast<const float4*>(w + c), gi = *reinterpret_cast<const float4*>(g + c),
                   mi = *reinterpret_cast<const float4*>(m + c), vi = *reinterpret_cast<const float4*>(v + c);
      float wv[4] = {wi.x, wi.y, wi.z, wi.w}, gv[4] = {gi.x, gi.y, gi.z, gi.w};
      float mv[4] = {mi.x, mi.y, mi.z, mi.w}, vv[4] = {vi.x, vi.y, vi.z, vi.w};
#pragma unroll
      for (int e = 0; e < 4; ++e)
        adam_elem<CLIP>(wv[e], mv[e], vv[e], gv[e] * gs, false, 0.f, b1, omb1, b2, omb2, lr_t, eps, sc);
      *reinterpret_cast<float4*>(m + c) = make_float4(mv[0], mv[1], mv[2], mv[3]);
      *reinterpret_cast<float4*>(v + c) = make_float4(vv[0], vv[1], vv[2], vv[3]);
      *reinterpret_cast<float4*>(w + c) = make_float4(wv[0], wv[1], wv[2], wv[3]);
    }
  } else {
    for (int c = lane; c < H; c += 32) {
      float wi = w[c], mi = m[c], vi = v[c];
      adam_elem<CLIP>(wi, mi, vi, g[c] * gs, false, 0.f, b1, omb1, b2, omb2, lr_t, eps, sc);
      m[c] = mi;
      v[c] = vi;
      w[c] = wi;
    }
  }
}

template <bool CLIP>
__device__ __forceinline__ void adam_rows_body(float* __restrict__ w, const float* __restrict__ grad,
                                               float* __restrict__ m, float* __restrict__ v, long rows, int rpw, int H,
                                               int vec, float lr, float b1, float b2, float eps,
                                               const float* __restrict__ gdenom, const unsigned* __restrict__ stamp,
                                               const unsigned* __restrict__ epoch, const AdamState* __restrict__ st,
                                               const float* __restrict__ clip) {
  cast_pdl_wait();
  cast_pdl_trigger();
  const float gs = gdenom ? 1.0f / *gdenom : 1.0f;
  const float sc = CLIP ? clip[0] : 1.0f;
  const float lr_t = lr * sqrtf(1.0f - st->b2p) / (1.0f - st->b1p);
  const float omb1 = 1.0f - b1, omb2 = 1.0f - b2;
  const unsigned ep = *epoch;
  const int lane = threadIdx.x & 31;
  const long nwarps = (long)gridDim.x * (blockDim.x >> 5);
  for (long r0 = rpw * ((long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)); r0 < rows; r0 += rpw * nwarps) {
    const long r = r0 + lane;
    unsigned todo = __ballot_sync(0xffffffffu, lane < rpw && r > 0 && r < rows && stamp[r] == ep);
    while (todo) {
      const long q = r0 + __ffs((int)todo) - 1;
      todo &= todo - 1u;
      const long o = q * H;
      adam_row<CLIP>(w + o, m + o, v + o, grad + o, H, vec, gs, b1, omb1, b2, omb2, lr_t, eps, lane, sc);
    }
  }
}

__global__ void adam_rows_kernel(float* __restrict__ w, const float* __restrict__ grad, float* __restrict__ m,
                                 float* __restrict__ v, long rows, int rpw, int H, int vec, float lr, float b1, float b2,
                                 float eps, const float* __restrict__ gdenom, const unsigned* __restrict__ stamp,
                                 const unsigned* __restrict__ epoch, const AdamState* __restrict__ st) {
  adam_rows_body<false>(w, grad, m, v, rows, rpw, H, vec, lr, b1, b2, eps, gdenom, stamp, epoch, st, nullptr);
}

__global__ void adam_rows_clip_kernel(float* __restrict__ w, const float* __restrict__ grad, float* __restrict__ m,
                                      float* __restrict__ v, long rows, int rpw, int H, int vec, float lr, float b1,
                                      float b2, float eps, const float* __restrict__ gdenom,
                                      const unsigned* __restrict__ stamp, const unsigned* __restrict__ epoch,
                                      const AdamState* __restrict__ st, const float* __restrict__ clip) {
  adam_rows_body<true>(w, grad, m, v, rows, rpw, H, vec, lr, b1, b2, eps, gdenom, stamp, epoch, st, clip);
}

// replicated data parallelism: row r's gradient is the rank-ordered sum over the ranks that touched it (stamps[q][r] ==
// *epochs[q], each rank against its own counter) with +0 for the others — what the dense peer pass reads from a rank
// whose zeroed row the batch missed — and the denominator is the rank-ordered sum of the ranks' counts (grads[q][np+2])
constexpr int ADAM_MAX_RANKS = 32;
template <bool CLIP>
__device__ __forceinline__ void adam_rows_peers_body(float* __restrict__ w, const float* const* __restrict__ g,
                                                     const unsigned* const* __restrict__ stamps,
                                                     const unsigned* const* __restrict__ epochs, int n,
                                                     float* __restrict__ m, float* __restrict__ v, long rows, int rpw,
                                                     int H, long np, float lr, float b1, float b2, float eps,
                                                     const AdamState* __restrict__ st,
                                                     const float* __restrict__ clip) {
  __shared__ float s_count;
  cast_pdl_wait();
  cast_pdl_trigger();
  if (threadIdx.x == 0) {
    float c = g[0][np + 2];
    for (int q = 1; q < n; ++q) c += g[q][np + 2];
    s_count = c;
  }
  __syncthreads();
  const float gs = 1.0f / s_count;
  const float sc = CLIP ? clip[0] : 1.0f;
  const float lr_t = lr * sqrtf(1.0f - st->b2p) / (1.0f - st->b1p);
  const float omb1 = 1.0f - b1, omb2 = 1.0f - b2;
  const int lane = threadIdx.x & 31;
  const long nwarps = (long)gridDim.x * (blockDim.x >> 5);
  for (long r0 = rpw * ((long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)); r0 < rows; r0 += rpw * nwarps) {
    const long r = r0 + lane;
    unsigned mine = 0u;        // ranks that touched row r (bit q)
    if (lane < rpw && r > 0 && r < rows)
      for (int q = 0; q < n; ++q) mine |= (stamps[q][r] == *epochs[q] ? 1u : 0u) << q;
    unsigned todo = __ballot_sync(0xffffffffu, mine != 0u);
    while (todo) {
      const int l = __ffs((int)todo) - 1;
      todo &= todo - 1u;
      const long o = (r0 + l) * H;
      const unsigned who = __shfl_sync(0xffffffffu, mine, l);
      for (int c = lane; c < H; c += 32) {
        float gsum = (who & 1u) ? g[0][o + c] : 0.f;
        for (int q = 1; q < n; ++q) gsum += ((who >> q) & 1u) ? g[q][o + c] : 0.f;
        float wi = w[o + c], mi = m[o + c], vi = v[o + c];
        adam_elem<CLIP>(wi, mi, vi, gsum * gs, false, 0.f, b1, omb1, b2, omb2, lr_t, eps, sc);
        m[o + c] = mi;
        v[o + c] = vi;
        w[o + c] = wi;
      }
    }
  }
}

__global__ void adam_rows_peers_kernel(float* __restrict__ w, const float* const* __restrict__ g,
                                       const unsigned* const* __restrict__ stamps,
                                       const unsigned* const* __restrict__ epochs, int n, float* __restrict__ m,
                                       float* __restrict__ v, long rows, int rpw, int H, long np, float lr, float b1,
                                       float b2,
                                       float eps, const AdamState* __restrict__ st) {
  adam_rows_peers_body<false>(w, g, stamps, epochs, n, m, v, rows, rpw, H, np, lr, b1, b2, eps, st, nullptr);
}

__global__ void adam_rows_peers_clip_kernel(float* __restrict__ w, const float* const* __restrict__ g,
                                            const unsigned* const* __restrict__ stamps,
                                            const unsigned* const* __restrict__ epochs, int n, float* __restrict__ m,
                                            float* __restrict__ v, long rows, int rpw, int H, long np, float lr,
                                            float b1, float b2, float eps, const AdamState* __restrict__ st,
                                            const float* __restrict__ clip) {
  adam_rows_peers_body<true>(w, g, stamps, epochs, n, m, v, rows, rpw, H, np, lr, b1, b2, eps, st, clip);
}

// rows scanned per warp of the lazy row pass: 32 unless that leaves fewer than 32 warps per SM (148 SMs)
static inline int rows_per_warp(long rows) {
  const long per = rows / (148L * 32);
  int rpw = 1;
  while (rpw < 32 && rpw < per) rpw <<= 1;
  return rpw;
}

// ---- global-norm gradient clipping (args.clip_grad, threshold args.max_norm; tf.clip_by_global_norm on the gradient
// Adam consumes).  Sum-of-squares passes write CLIP_PARTS fp64 partials each: block b's sum (threads' grid-stride sums
// folded by a fixed tree) in slot b, zeros in the slots past the grid, which depends on the shape only.  The finalize
// pass folds the partials in slot order (and, with a row-sharded table, every rank's shard partials in rank order)
// and writes {scale, norm}; the CLIP Adam kernels read the scale from device memory.  No atomics: same bits every run,
// and on every rank, since every rank folds the same values in the same order.
constexpr int CLIP_PARTS = 1024;
constexpr int CLIP_THREADS = 256;

// block-wide sum of one value per thread, fixed tree; the result is returned to every thread
__device__ __forceinline__ double clip_block_sum(double a) {
  __shared__ double s[CLIP_THREADS];
  s[threadIdx.x] = a;
  __syncthreads();
  for (int o = CLIP_THREADS / 2; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
    __syncthreads();
  }
  const double r = s[0];
  __syncthreads();
  return r;
}

__device__ __forceinline__ void clip_store_part(double acc, double* __restrict__ parts) {
  const double b = clip_block_sum(acc);
  if (threadIdx.x == 0) parts[blockIdx.x] = b;
  if (blockIdx.x == 0)
    for (int i = gridDim.x + threadIdx.x; i < CLIP_PARTS; i += blockDim.x) parts[i] = 0.0;
}

// sum over i < n of g_i^2, g_i = grad[i] / *gdenom (+ l2 * w[i] on [l2_lo, l2_hi)): the g of adam_step_body.  Four
// loads in flight per thread; the accumulation order is the plain grid-stride order.
__global__ void clip_sumsq_range_kernel(const float* __restrict__ grad, const float* __restrict__ w, long n,
                                        const float* __restrict__ gdenom, float l2, long l2_lo, long l2_hi,
                                        double* __restrict__ parts) {
  cast_pdl_wait();
  cast_pdl_trigger();
  const float gs = gdenom ? 1.0f / *gdenom : 1.0f;
  const long stride = (long)gridDim.x * blockDim.x;
  double acc = 0.0;
  long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  for (; i + 3 * stride < n; i += 4 * stride) {
    float g[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) g[e] = grad[i + e * stride] * gs;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const long k = i + e * stride;
      if (k >= l2_lo && k < l2_hi) g[e] = fmaf(l2, w[k], g[e]);
      acc += (double)g[e] * (double)g[e];
    }
  }
  for (; i < n; i += stride) {
    float g = grad[i] * gs;
    if (i >= l2_lo && i < l2_hi) g = fmaf(l2, w[i], g);
    acc += (double)g * (double)g;
  }
  clip_store_part(acc, parts);
}

// lazy_adam: the rows [1, rows) of a [rows, H] table gradient stamped in this backward pass (adam_rows_body's rows);
// every other row counts as 0
__global__ void clip_sumsq_rows_kernel(const float* __restrict__ grad, long rows, int rpw, int H,
                                       const float* __restrict__ gdenom, const unsigned* __restrict__ stamp,
                                       const unsigned* __restrict__ epoch, double* __restrict__ parts) {
  cast_pdl_wait();
  cast_pdl_trigger();
  const float gs = gdenom ? 1.0f / *gdenom : 1.0f;
  const unsigned ep = *epoch;
  const int lane = threadIdx.x & 31;
  const long nwarps = (long)gridDim.x * (blockDim.x >> 5);
  double acc = 0.0;
  for (long r0 = rpw * ((long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)); r0 < rows; r0 += rpw * nwarps) {
    const long r = r0 + lane;
    unsigned todo = __ballot_sync(0xffffffffu, lane < rpw && r > 0 && r < rows && stamp[r] == ep);
    while (todo) {
      const long o = (r0 + __ffs((int)todo) - 1) * H;
      todo &= todo - 1u;
      for (int c = lane; c < H; c += 32) {
        const float g = grad[o + c] * gs;
        acc += (double)g * (double)g;
      }
    }
  }
  clip_store_part(acc, parts);
}

// lazy_adam under replicated data parallelism: the rank-ordered sum over the touching ranks of each row any rank
// touched (adam_rows_peers_body's gradient)
__global__ void clip_sumsq_rows_peers_kernel(const float* const* __restrict__ g,
                                             const unsigned* const* __restrict__ stamps,
                                             const unsigned* const* __restrict__ epochs, int n, long rows, int rpw,
                                             int H, long np, double* __restrict__ parts) {
  __shared__ float s_count;
  cast_pdl_wait();
  cast_pdl_trigger();
  if (threadIdx.x == 0) {
    float c = g[0][np + 2];
    for (int q = 1; q < n; ++q) c += g[q][np + 2];
    s_count = c;
  }
  __syncthreads();
  const float gs = 1.0f / s_count;
  const int lane = threadIdx.x & 31;
  const long nwarps = (long)gridDim.x * (blockDim.x >> 5);
  double acc = 0.0;
  for (long r0 = rpw * ((long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)); r0 < rows; r0 += rpw * nwarps) {
    const long r = r0 + lane;
    unsigned mine = 0u;
    if (lane < rpw && r > 0 && r < rows)
      for (int q = 0; q < n; ++q) mine |= (stamps[q][r] == *epochs[q] ? 1u : 0u) << q;
    unsigned todo = __ballot_sync(0xffffffffu, mine != 0u);
    while (todo) {
      const int l = __ffs((int)todo) - 1;
      todo &= todo - 1u;
      const long o = (r0 + l) * H;
      const unsigned who = __shfl_sync(0xffffffffu, mine, l);
      for (int c = lane; c < H; c += 32) {
        float gsum = (who & 1u) ? g[0][o + c] : 0.f;
        for (int q = 1; q < n; ++q) gsum += ((who >> q) & 1u) ? g[q][o + c] : 0.f;
        const float gv = gsum * gs;
        acc += (double)gv * (double)gv;
      }
    }
  }
  clip_store_part(acc, parts);
}

// replicated data parallelism: the reduction of adam_step_peers_kernel without the update — g_red[i] = sum_r g[r][i]
// (rank order) for i in [lo, np + tail) — plus the squares of the parameters' gradients g_red[i] / count (+ l2 * w[i]).
// Groups of 4 stay aligned to the buffers; the group that straddles `lo` goes element by element.
__global__ void clip_reduce_sumsq_peers_kernel(const float* const* __restrict__ g, int n, float* __restrict__ g_red,
                                               const float* __restrict__ w, long lo, long np, long tail, float l2,
                                               long l2_lo, long l2_hi, double* __restrict__ parts) {
  __shared__ float s_count;
  cast_pdl_wait();
  cast_pdl_trigger();
  if (threadIdx.x == 0) {
    float c = g[0][np + 2];
    for (int r = 1; r < n; ++r) c += g[r][np + 2];
    s_count = c;
  }
  __syncthreads();
  const float gs = 1.0f / s_count;
  const long total = np + tail;
  double acc = 0.0;
  for (long i0 = (lo & ~3L) + 4 * ((long)blockIdx.x * blockDim.x + threadIdx.x); i0 < total;
       i0 += 4 * (long)gridDim.x * blockDim.x) {
    float gv[4] = {0.f, 0.f, 0.f, 0.f};
    const int cnt = total - i0 < 4 ? (int)(total - i0) : 4;
    const int e0 = i0 < lo ? (int)(lo - i0) : 0;
    if (cnt == 4 && e0 == 0) {
      for (int r0 = 0; r0 < n; r0 += ADAM_PEER_BATCH) {
        float4 q[ADAM_PEER_BATCH];
#pragma unroll
        for (int u = 0; u < ADAM_PEER_BATCH; ++u)
          if (r0 + u < n) q[u] = *reinterpret_cast<const float4*>(g[r0 + u] + i0);
#pragma unroll
        for (int u = 0; u < ADAM_PEER_BATCH; ++u)
          if (r0 + u < n) {
            if (r0 + u == 0) {
              gv[0] = q[u].x; gv[1] = q[u].y; gv[2] = q[u].z; gv[3] = q[u].w;
            } else {
              gv[0] += q[u].x; gv[1] += q[u].y; gv[2] += q[u].z; gv[3] += q[u].w;
            }
          }
      }
      *reinterpret_cast<float4*>(g_red + i0) = make_float4(gv[0], gv[1], gv[2], gv[3]);
    } else {
      for (int e = e0; e < cnt; ++e) {
        float sacc = g[0][i0 + e];
        for (int r = 1; r < n; ++r) sacc += g[r][i0 + e];
        gv[e] = sacc;
        g_red[i0 + e] = sacc;
      }
    }
    const int na = np - i0 >= 4 ? 4 : (np - i0 > 0 ? (int)(np - i0) : 0);
    for (int e = e0; e < na; ++e) {
      const long idx = i0 + e;
      float x = gv[e] * gs;
      if (idx >= l2_lo && idx < l2_hi) x = fmaf(l2, w[idx], x);
      acc += (double)x * (double)x;
    }
  }
  clip_store_part(acc, parts);
}

// norm = sqrt(sum of the shard partials of ranks 0..n_ranks-1 (each folded, then added in rank order) + sum of the
// local partials); scale = norm > max_norm ? max_norm / norm : 1, NaN for a non-finite norm.  out = {scale, norm}.
__global__ void clip_finalize_kernel(const double* __restrict__ parts, int nparts, const double* const* __restrict__ peer,
                                     int n_ranks, double max_norm, float* __restrict__ out) {
  cast_pdl_wait();
  cast_pdl_trigger();
  double a = 0.0;
  for (int i = threadIdx.x; i < nparts; i += blockDim.x) a += parts[i];
  double tot = clip_block_sum(a);
  if (peer) {
    double shards = 0.0;
    for (int r = 0; r < n_ranks; ++r) {
      double b = 0.0;
      for (int i = threadIdx.x; i < CLIP_PARTS; i += blockDim.x) b += peer[r][i];
      b = clip_block_sum(b);
      shards = r == 0 ? b : shards + b;
    }
    tot = shards + tot;
  }
  if (threadIdx.x == 0) {
    const double norm = sqrt(tot);
    float scale = 1.0f;
    if (!(norm <= 1.7976931348623157e308))   // inf or NaN
      scale = nanf("");
    else if (norm > max_norm)
      scale = (float)(max_norm / norm);
    out[0] = scale;
    out[1] = (float)norm;
  }
}

__global__ void adam_advance_kernel(AdamState* st, float b1, float b2) {
  cast_pdl_wait();
  cast_pdl_trigger();
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    st->b1p *= b1;
    st->b2p *= b2;
    st->step += 1ull;
  }
}

}  // namespace cast

using namespace cast;

extern "C" int cast_adam_init_state(void* state, float beta1, float beta2, void* stream) {
  if (!state) return set_error(CAST_ERR_BAD_ARG, "adam_init_state");
  CAST_LAUNCH(adam_init_kernel, dim3(1), dim3(32), 0, (cudaStream_t)stream, static_cast<AdamState*>(state), beta1,
              beta2);
  return check_launch("adam_init");
}

// the update of one contiguous range; `advance` != 0 also steps the beta powers / step counter afterwards (callers that
// update several ranges of one model — a row shard of the item table plus the replicated weights — advance once)
extern "C" int cast_adam_tf_range(float* w, const float* grad, float* m, float* v, long n, float lr, float beta1,
                                  float beta2, float eps, const float* gdenom, float l2, long l2_lo, long l2_hi,
                                  void* state, int advance, void* stream) {
  if (!w || !grad || !m || !v || !state || n <= 0) return set_error(CAST_ERR_BAD_ARG, "adam_tf_range");
  const bool vec = (n % 4 == 0) && ((((uintptr_t)w | (uintptr_t)grad | (uintptr_t)m | (uintptr_t)v) & 15) == 0);
  int rc;
  if (vec) {
    long g = cdiv(n / 4, 256);
    if (g > 148 * 8) g = 148 * 8;
    CAST_LAUNCH_DEP(adam_step_vec4_kernel, dim3((unsigned)g), dim3(256), 0, (cudaStream_t)stream,
                reinterpret_cast<float4*>(w), reinterpret_cast<const float4*>(grad), reinterpret_cast<float4*>(m),
                reinterpret_cast<float4*>(v), n / 4, lr, beta1, beta2, eps, gdenom, l2, l2_lo, l2_hi,
                static_cast<const AdamState*>(state));
  } else {
    long g = cdiv(n, 256);
    if (g > 148 * 8) g = 148 * 8;
    CAST_LAUNCH_DEP(adam_step_kernel, dim3((unsigned)g), dim3(256), 0, (cudaStream_t)stream, w, grad, m, v, n, lr, beta1,
                beta2, eps, gdenom, l2, l2_lo, l2_hi, static_cast<const AdamState*>(state));
  }
  if ((rc = check_launch("adam_step"))) return rc;
  if (advance) {
    CAST_LAUNCH_DEP(adam_advance_kernel, dim3(1), dim3(32), 0, (cudaStream_t)stream, static_cast<AdamState*>(state),
                beta1, beta2);
    return check_launch("adam_advance");
  }
  return CAST_OK;
}

extern "C" int cast_adam_tf_step(float* w, const float* grad, float* m, float* v, long n, float lr, float beta1,
                                 float beta2, float eps, const float* gdenom, float l2, long l2_lo, long l2_hi,
                                 void* state, void* stream) {
  return cast_adam_tf_range(w, grad, m, v, n, lr, beta1, beta2, eps, gdenom, l2, l2_lo, l2_hi, state, 1, stream);
}

/* Data-parallel TF-Adam: grads is a DEVICE array of n_ranks pointers (this rank's buffer and the peer mappings of the
 * others, each 16-byte aligned, n + tail floats: gradient numerators then [loss_sum, auc_sum, count, ...]); the update
 * uses sum_r grads[r][i] (rank order) / sum_r count_r and the reduced buffer is left in g_red[n + tail].  Replaces
 * cast_peer_reduce + cast_adam_tf_step; the caller brackets it with cast_peer_barrier as for cast_peer_reduce. */
extern "C" int cast_adam_tf_step_peers(float* w, const void* const* grads, int n_ranks, float* g_red, float* m, float* v,
                                       long n, long tail, float lr, float beta1, float beta2, float eps, float l2,
                                       long l2_lo, long l2_hi, void* state, void* stream) {
  if (!w || !grads || !g_red || !m || !v || !state || n <= 0 || tail < 3 || n_ranks < 1)
    return set_error(CAST_ERR_BAD_ARG, "adam_tf_step_peers");
  if ((((uintptr_t)w | (uintptr_t)g_red | (uintptr_t)m | (uintptr_t)v) & 15) != 0)
    return set_error(CAST_ERR_BAD_ARG, "adam_tf_step_peers: buffers must be 16-byte aligned");
  long g = cdiv(cdiv(n + tail, 4), 256);
  if (g > 148 * 8) g = 148 * 8;
  CAST_LAUNCH_DEP(adam_step_peers_kernel, dim3((unsigned)g), dim3(256), 0, (cudaStream_t)stream, w,
              reinterpret_cast<const float* const*>(grads), n_ranks, g_red, m, v, 0L, n, tail, lr, beta1, beta2, eps,
              l2, l2_lo, l2_hi, static_cast<const AdamState*>(state));
  int rc;
  if ((rc = check_launch("adam_step_peers"))) return rc;
  CAST_LAUNCH_DEP(adam_advance_kernel, dim3(1), dim3(32), 0, (cudaStream_t)stream, static_cast<AdamState*>(state), beta1,
              beta2);
  return check_launch("adam_advance");
}

/* One-thread kernel: the next backward pass's gradient epoch (*epoch += 1).  The counter is never rewound, so a
 * stamp left by any earlier pass (an eager warm-up, a rewound optimizer state) can never look current. */
extern "C" int cast_grad_epoch_advance(unsigned* epoch, void* stream) {
  if (!epoch) return set_error(CAST_ERR_BAD_ARG, "grad_epoch_advance");
  CAST_LAUNCH_DEP(grad_epoch_advance_kernel, dim3(1), dim3(32), 0, (cudaStream_t)stream, epoch);
  return check_launch("grad_epoch_advance");
}

/* Lazy TF-Adam over a row table [rows, H] (the item table or this rank's shard of it): updates row r only if
 * stamp[r] == *epoch (its gradient was written in this backward pass); row 0 never.  Does not advance the beta
 * powers: the caller's cast_adam_tf_range over the dense remainder does, once. */
extern "C" int cast_adam_tf_rows(float* w, const float* grad, float* m, float* v, long rows, int H, float lr,
                                 float beta1, float beta2, float eps, const float* gdenom, const unsigned* stamp,
                                 const unsigned* epoch, void* state, void* stream) {
  if (!w || !grad || !m || !v || !stamp || !epoch || !state || rows <= 0 || H <= 0)
    return set_error(CAST_ERR_BAD_ARG, "adam_tf_rows");
  const int vec = (H % 4 == 0) && ((((uintptr_t)w | (uintptr_t)grad | (uintptr_t)m | (uintptr_t)v) & 15) == 0);
  const int rpw = rows_per_warp(rows);
  long g = cdiv(cdiv(rows, rpw), 8);
  if (g > 148 * 8) g = 148 * 8;
  CAST_LAUNCH_DEP(adam_rows_kernel, dim3((unsigned)g), dim3(256), 0, (cudaStream_t)stream, w, grad, m, v, rows, rpw, H,
                  vec,
                  lr, beta1, beta2, eps, gdenom, stamp, epoch, static_cast<const AdamState*>(state));
  return check_launch("adam_rows");
}

/* cast_adam_tf_rows under replicated data parallelism: grads / stamps / epochs are DEVICE arrays of n_ranks pointers
 * (own buffer + peer mappings; grads as for cast_adam_tf_step_peers, np = parameter count before the tail sums).  Row
 * r is updated if any rank touched it, with the rank-ordered sum of the touching ranks' rows.  No advance. */
extern "C" int cast_adam_tf_rows_peers(float* w, const void* const* grads, const void* const* stamps,
                                       const void* const* epochs, int n_ranks, float* m, float* v, long rows, int H,
                                       long np, float lr, float beta1, float beta2, float eps, void* state,
                                       void* stream) {
  if (!w || !grads || !stamps || !epochs || !m || !v || !state || rows <= 0 || H <= 0 || np < rows * H ||
      n_ranks < 1 || n_ranks > ADAM_MAX_RANKS)
    return set_error(CAST_ERR_BAD_ARG, "adam_tf_rows_peers");
  const int rpw = rows_per_warp(rows);
  long g = cdiv(cdiv(rows, rpw), 8);
  if (g > 148 * 8) g = 148 * 8;
  CAST_LAUNCH_DEP(adam_rows_peers_kernel, dim3((unsigned)g), dim3(256), 0, (cudaStream_t)stream, w,
                  reinterpret_cast<const float* const*>(grads), reinterpret_cast<const unsigned* const*>(stamps),
                  reinterpret_cast<const unsigned* const*>(epochs), n_ranks, m, v, rows, rpw, H, np, lr, beta1, beta2, eps,
                  static_cast<const AdamState*>(state));
  return check_launch("adam_rows_peers");
}

/* cast_adam_tf_step_peers over the elements [lo, n) only (elements below lo are neither reduced into g_red nor
 * updated): the dense remainder behind the lazy row pass of cast_adam_tf_rows_peers.  Advances the beta powers. */
extern "C" int cast_adam_tf_range_peers(float* w, const void* const* grads, int n_ranks, float* g_red, float* m,
                                        float* v, long lo, long n, long tail, float lr, float beta1, float beta2,
                                        float eps, void* state, void* stream) {
  if (!w || !grads || !g_red || !m || !v || !state || lo < 0 || n <= lo || tail < 3 || n_ranks < 1)
    return set_error(CAST_ERR_BAD_ARG, "adam_tf_range_peers");
  if ((((uintptr_t)w | (uintptr_t)g_red | (uintptr_t)m | (uintptr_t)v) & 15) != 0)
    return set_error(CAST_ERR_BAD_ARG, "adam_tf_range_peers: buffers must be 16-byte aligned");
  long g = cdiv(cdiv(n + tail - (lo & ~3L), 4), 256);
  if (g > 148 * 8) g = 148 * 8;
  CAST_LAUNCH_DEP(adam_step_peers_kernel, dim3((unsigned)g), dim3(256), 0, (cudaStream_t)stream, w,
                  reinterpret_cast<const float* const*>(grads), n_ranks, g_red, m, v, lo, n, tail, lr, beta1, beta2,
                  eps, 0.f, 0L, 0L, static_cast<const AdamState*>(state));
  int rc;
  if ((rc = check_launch("adam_step_peers"))) return rc;
  CAST_LAUNCH_DEP(adam_advance_kernel, dim3(1), dim3(32), 0, (cudaStream_t)stream, static_cast<AdamState*>(state), beta1,
                  beta2);
  return check_launch("adam_advance");
}

// ---------------------------------------------------------------------------------------------------------------------
// global-norm gradient clipping (include/cast_b200.h)
static inline unsigned clip_grid(long work) {
  const long g = cdiv(work, CLIP_THREADS);
  return (unsigned)(g < 1 ? 1 : (g > CLIP_PARTS ? CLIP_PARTS : g));
}

extern "C" int cast_clip_parts(void) { return CLIP_PARTS; }

extern "C" int cast_clip_sumsq_range(const float* grad, const float* w, long n, const float* gdenom, float l2,
                                     long l2_lo, long l2_hi, double* parts, void* stream) {
  if (!grad || !parts || n <= 0 || (l2_hi > l2_lo && !w)) return set_error(CAST_ERR_BAD_ARG, "clip_sumsq_range");
  CAST_LAUNCH_DEP(clip_sumsq_range_kernel, dim3(clip_grid(cdiv(n, 4))), dim3(CLIP_THREADS), 0, (cudaStream_t)stream,
                  grad, w, n, gdenom, l2, l2_lo, l2_hi, parts);
  return check_launch("clip_sumsq_range");
}

extern "C" int cast_clip_sumsq_rows(const float* grad, long rows, int H, const float* gdenom, const unsigned* stamp,
                                    const unsigned* epoch, double* parts, void* stream) {
  if (!grad || !stamp || !epoch || !parts || rows <= 0 || H <= 0) return set_error(CAST_ERR_BAD_ARG, "clip_sumsq_rows");
  const int rpw = rows_per_warp(rows);
  CAST_LAUNCH_DEP(clip_sumsq_rows_kernel, dim3(clip_grid(cdiv(rows, rpw) * 32)), dim3(CLIP_THREADS), 0,
                  (cudaStream_t)stream, grad, rows, rpw, H, gdenom, stamp, epoch, parts);
  return check_launch("clip_sumsq_rows");
}

extern "C" int cast_clip_sumsq_rows_peers(const void* const* grads, const void* const* stamps,
                                          const void* const* epochs, int n_ranks, long rows, int H, long np,
                                          double* parts, void* stream) {
  if (!grads || !stamps || !epochs || !parts || rows <= 0 || H <= 0 || np < rows * H || n_ranks < 1 ||
      n_ranks > ADAM_MAX_RANKS)
    return set_error(CAST_ERR_BAD_ARG, "clip_sumsq_rows_peers");
  const int rpw = rows_per_warp(rows);
  CAST_LAUNCH_DEP(clip_sumsq_rows_peers_kernel, dim3(clip_grid(cdiv(rows, rpw) * 32)), dim3(CLIP_THREADS), 0,
                  (cudaStream_t)stream, reinterpret_cast<const float* const*>(grads),
                  reinterpret_cast<const unsigned* const*>(stamps), reinterpret_cast<const unsigned* const*>(epochs),
                  n_ranks, rows, rpw, H, np, parts);
  return check_launch("clip_sumsq_rows_peers");
}

extern "C" int cast_clip_reduce_sumsq_peers(const void* const* grads, int n_ranks, float* g_red, const float* w,
                                            long lo, long n, long tail, float l2, long l2_lo, long l2_hi,
                                            double* parts, void* stream) {
  if (!grads || !g_red || !w || !parts || lo < 0 || n <= lo || tail < 3 || n_ranks < 1)
    return set_error(CAST_ERR_BAD_ARG, "clip_reduce_sumsq_peers");
  if (((uintptr_t)g_red & 15) != 0) return set_error(CAST_ERR_BAD_ARG, "clip_reduce_sumsq_peers: g_red alignment");
  CAST_LAUNCH_DEP(clip_reduce_sumsq_peers_kernel, dim3(clip_grid(cdiv(n + tail - (lo & ~3L), 4))), dim3(CLIP_THREADS),
                  0, (cudaStream_t)stream, reinterpret_cast<const float* const*>(grads), n_ranks, g_red, w, lo, n,
                  tail, l2, l2_lo, l2_hi, parts);
  return check_launch("clip_reduce_sumsq_peers");
}

extern "C" int cast_clip_finalize(const double* parts, int nparts, const void* const* peer_parts, int n_ranks,
                                  double max_norm, float* out, void* stream) {
  if (!parts || !out || nparts <= 0 || (peer_parts && n_ranks < 1) || !(max_norm > 0.0))
    return set_error(CAST_ERR_BAD_ARG, "clip_finalize");
  CAST_LAUNCH_DEP(clip_finalize_kernel, dim3(1), dim3(CLIP_THREADS), 0, (cudaStream_t)stream, parts, nparts,
                  reinterpret_cast<const double* const*>(peer_parts), n_ranks, max_norm, out);
  return check_launch("clip_finalize");
}

extern "C" int cast_adam_tf_range_clip(float* w, const float* grad, float* m, float* v, long n, float lr, float beta1,
                                       float beta2, float eps, const float* gdenom, float l2, long l2_lo, long l2_hi,
                                       const float* clip, void* state, int advance, void* stream) {
  if (!w || !grad || !m || !v || !clip || !state || n <= 0) return set_error(CAST_ERR_BAD_ARG, "adam_tf_range_clip");
  const bool vec = (n % 4 == 0) && ((((uintptr_t)w | (uintptr_t)grad | (uintptr_t)m | (uintptr_t)v) & 15) == 0);
  int rc;
  if (vec) {
    long g = cdiv(n / 4, 256);
    if (g > 148 * 8) g = 148 * 8;
    CAST_LAUNCH_DEP(adam_step_vec4_clip_kernel, dim3((unsigned)g), dim3(256), 0, (cudaStream_t)stream,
                    reinterpret_cast<float4*>(w), reinterpret_cast<const float4*>(grad), reinterpret_cast<float4*>(m),
                    reinterpret_cast<float4*>(v), n / 4, lr, beta1, beta2, eps, gdenom, l2, l2_lo, l2_hi,
                    static_cast<const AdamState*>(state), clip);
  } else {
    long g = cdiv(n, 256);
    if (g > 148 * 8) g = 148 * 8;
    CAST_LAUNCH_DEP(adam_step_clip_kernel, dim3((unsigned)g), dim3(256), 0, (cudaStream_t)stream, w, grad, m, v, n, lr,
                    beta1, beta2, eps, gdenom, l2, l2_lo, l2_hi, static_cast<const AdamState*>(state), clip);
  }
  if ((rc = check_launch("adam_step_clip"))) return rc;
  if (advance) {
    CAST_LAUNCH_DEP(adam_advance_kernel, dim3(1), dim3(32), 0, (cudaStream_t)stream, static_cast<AdamState*>(state),
                    beta1, beta2);
    return check_launch("adam_advance");
  }
  return CAST_OK;
}

extern "C" int cast_adam_tf_rows_clip(float* w, const float* grad, float* m, float* v, long rows, int H, float lr,
                                      float beta1, float beta2, float eps, const float* gdenom, const unsigned* stamp,
                                      const unsigned* epoch, const float* clip, void* state, void* stream) {
  if (!w || !grad || !m || !v || !stamp || !epoch || !clip || !state || rows <= 0 || H <= 0)
    return set_error(CAST_ERR_BAD_ARG, "adam_tf_rows_clip");
  const int vec = (H % 4 == 0) && ((((uintptr_t)w | (uintptr_t)grad | (uintptr_t)m | (uintptr_t)v) & 15) == 0);
  const int rpw = rows_per_warp(rows);
  long g = cdiv(cdiv(rows, rpw), 8);
  if (g > 148 * 8) g = 148 * 8;
  CAST_LAUNCH_DEP(adam_rows_clip_kernel, dim3((unsigned)g), dim3(256), 0, (cudaStream_t)stream, w, grad, m, v, rows,
                  rpw, H, vec, lr, beta1, beta2, eps, gdenom, stamp, epoch, static_cast<const AdamState*>(state), clip);
  return check_launch("adam_rows_clip");
}

extern "C" int cast_adam_tf_rows_peers_clip(float* w, const void* const* grads, const void* const* stamps,
                                            const void* const* epochs, int n_ranks, float* m, float* v, long rows,
                                            int H, long np, float lr, float beta1, float beta2, float eps,
                                            const float* clip, void* state, void* stream) {
  if (!w || !grads || !stamps || !epochs || !m || !v || !clip || !state || rows <= 0 || H <= 0 || np < rows * H ||
      n_ranks < 1 || n_ranks > ADAM_MAX_RANKS)
    return set_error(CAST_ERR_BAD_ARG, "adam_tf_rows_peers_clip");
  const int rpw = rows_per_warp(rows);
  long g = cdiv(cdiv(rows, rpw), 8);
  if (g > 148 * 8) g = 148 * 8;
  CAST_LAUNCH_DEP(adam_rows_peers_clip_kernel, dim3((unsigned)g), dim3(256), 0, (cudaStream_t)stream, w,
                  reinterpret_cast<const float* const*>(grads), reinterpret_cast<const unsigned* const*>(stamps),
                  reinterpret_cast<const unsigned* const*>(epochs), n_ranks, m, v, rows, rpw, H, np, lr, beta1, beta2,
                  eps, static_cast<const AdamState*>(state), clip);
  return check_launch("adam_rows_peers_clip");
}
