// Fused row-tile kernels for one transformer block when hidden_units <= 64 (BASELINE configs 1-3, H = 50):
//   ln_qkv_fwd : LN(x) -> Q = LN(x)Wq+bq, K = xWk+bk, V = xWv+bv, key/query masks       (modules.py:74-78, :203-205, :222, :248)
//   ln_ffn_fwd : LN(y) -> relu(.W1+b1) -> dropout -> .W2+b2 -> dropout -> + LN(y) -> *mask (sasrec.py:81-83, modules.py:298-313)
//   ffn_bwd    : backward of ln_ffn_fwd incl. dW1, dW2, db1, db2, dgamma, dbeta
//   qkv_bwd    : backward of ln_qkv_fwd incl. dWq, dWk, dWv, biases, dgamma, dbeta (and the attention residual)
// One CTA works on 64-row tiles with all H columns; the kernels themselves (fused_mma.cuh) contract on the tensor cores
// (mma.sync 3xTF32).  The whole weight matrix (H*H*4 <= 16 KB) sits in shared memory; activations make exactly one HBM
// round trip per kernel instead of one per op.  Backward kernels are persistent (one CTA per SM loops over row tiles)
// and keep their weight-gradient partials in registers; a fixed-order second stage sums the per-CTA partials straight
// into the flat gradient buffer => deterministic.
// Gradient layout contract (flat, contiguous, see engine.param_shapes):
//   qkv_bwd -> [ln1.beta H | ln1.gamma H | q.w H*H | q.b H | k.w H*H | k.b H | v.w H*H | v.b H]
//   ffn_bwd -> [ln2.beta H | ln2.gamma H | ffn1.w H*H | ffn1.b H | ffn2.w H*H | ffn2.b H]
#include "cast_rt.cuh"

namespace cast {

int launch_reduce_partials(const float* partial, int nparts, long count, float* out0, long split, float* out1,
                           cudaStream_t stream);

constexpr int FR = 64;        // rows per tile
constexpr int FT = 256;       // threads

struct FDims {
  long N;
  int H, HP4, HS;
};

static FDims fdims(long N, int H) {
  FDims d;
  d.N = N;
  d.H = H;
  d.HP4 = (H + 3) & ~3;
  d.HS = (d.HP4 % 32 == 0) ? d.HP4 + 4 : d.HP4;
  return d;
}

// LN of the rows of Xs (row-major smem tile) -> Ns (smem) and optionally global y / stats / zero-sum flags
__device__ __forceinline__ void f_layernorm_rows(const float* __restrict__ Xs, float* __restrict__ Ns,
                                                 const float* __restrict__ gamma, const float* __restrict__ beta,
                                                 float eps, long row0, const FDims& d, float* __restrict__ y,
                                                 float* __restrict__ mean_out, float* __restrict__ rstd_out,
                                                 float* __restrict__ xnz, float* __restrict__ ynz) {
  const int lane = threadIdx.x & 31;
  const int c0 = lane, c1 = lane + 32;
  const float g0 = c0 < d.H ? gamma[c0] : 0.f, g1 = c1 < d.H ? gamma[c1] : 0.f;
  const float b0 = c0 < d.H ? beta[c0] : 0.f, b1 = c1 < d.H ? beta[c1] : 0.f;
  for (int r = threadIdx.x >> 5; r < FR; r += FT / 32) {
    const long row = row0 + r;
    const float v0 = c0 < d.H ? Xs[r * d.HS + c0] : 0.f;
    const float v1 = c1 < d.H ? Xs[r * d.HS + c1] : 0.f;
    const float s = warp_sum(v0 + v1);
    const float mean = s / (float)d.H;
    const float d0 = c0 < d.H ? v0 - mean : 0.f, d1 = c1 < d.H ? v1 - mean : 0.f;
    const float var = warp_sum(d0 * d0 + d1 * d1) / (float)d.H;
    const float stdv = sqrtf(var + eps);
    const float o0 = c0 < d.H ? g0 * (d0 / stdv) + b0 : 0.f;
    const float o1 = c1 < d.H ? g1 * (d1 / stdv) + b1 : 0.f;
    const float ys = warp_sum(o0 + o1);
    if (c0 < d.HP4) Ns[r * d.HS + c0] = o0;
    if (c1 < d.HP4) Ns[r * d.HS + c1] = o1;
    if (row < d.N) {
      if (y) {
        if (c0 < d.H) y[row * d.H + c0] = o0;
        if (c1 < d.H) y[row * d.H + c1] = o1;
      }
      if (lane == 0) {
        if (mean_out) mean_out[row] = mean;
        if (rstd_out) rstd_out[row] = 1.0f / stdv;
        if (xnz) xnz[row] = (s != 0.f) ? 1.f : 0.f;
        if (ynz) ynz[row] = (ys != 0.f) ? 1.f : 0.f;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// kernel arguments (the kernels are in fused_mma.cuh)
struct LnQkvArgs {
  const float *x, *gamma, *beta, *W[3], *b[3];
  float eps;
  float *qn, *out[3], *mean, *rstd, *kmask, *qmask;
};

struct LnFfnArgs {
  const float *y, *gamma, *beta, *W1, *b1, *W2, *b2;
  const int* ids;
  float eps, rate;
  unsigned long long seed;
  const unsigned long long* step;
  int site_h, site_o;
  float *zn, *h1d, *xout, *mean, *rstd;
};

// Optional last step on the dx rows the LayerNorm backward writes: the gradient of `dropout(emb) * mask` at the tower input
// (sasrec.py:58-62), so that block 0's backward kernel emits the embedding gradient directly.
struct LnOutFx {
  const int* ids;  // row mask (ids[row] == 0 => 0), may be null
  Drop drop;
  bool on;
};
__device__ __forceinline__ LnOutFx ln_out_none() {
  LnOutFx f;
  f.ids = nullptr;
  f.drop.k0 = f.drop.k1 = f.drop.thresh = 0u;
  f.drop.scale = 1.f;
  f.on = false;
  return f;
}

struct FfnBwdArgs {
  const float *dx, *zn, *h1d, *y, *mean, *rstd, *gamma, *W1, *W2;
  const int* ids;
  float rate;
  unsigned long long seed;
  const unsigned long long* step;
  int site_o;
  float* dy;
  float* partial;  // [gridDim.x][2H + 2(H*H + H)]
  long ntiles;
};

struct QkvBwdArgs {
  const float *dQ, *dK, *dV, *dres, *x, *qn, *mean, *rstd, *gamma, *Wq, *Wk, *Wv;
  float* dx;
  float* partial;  // [gridDim.x][2H + 3(H*H + H)]
  long ntiles;
  // block 0 of a tower whose input is dropout(embedding) * mask: dx *= mask(out_ids) * dropout(out_rate, out_site)
  const int* out_ids;
  float out_rate;
  unsigned long long seed;
  const unsigned long long* step;
  int out_site;
  int out_fx;
};
__device__ __forceinline__ LnOutFx qkv_out_fx(const QkvBwdArgs& a) {
  LnOutFx f = ln_out_none();
  if (a.out_fx) {
    f.ids = a.out_ids;
    f.drop = make_drop(a.out_rate, a.seed, a.step, a.out_site);
    f.on = true;
  }
  return f;
}

}  // namespace cast
#include "fused_mma.cuh"
namespace cast {

// persistent grids: one wave of resident CTAs on the 148 SMs of a B200 (the backward kernels run one 512-thread CTA
// per SM), so no CTA waits for a slot and the number of weight-gradient partials stays minimal
constexpr int NUM_SMS = 148;
static int bwd_grid(long ntiles, int ctas_per_sm) {
  const long cap = (long)NUM_SMS * ctas_per_sm;
  return (int)(ntiles < cap ? ntiles : cap);
}

}  // namespace cast

using namespace cast;

#define CAST_FUSED_SMEM(kernel, bytes)                                                          \
  {                                                                                             \
    static size_t configured = 48 * 1024;                                                       \
    if ((bytes) > configured) {                                                                 \
      cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes));  \
      configured = (bytes);                                                                     \
    }                                                                                           \
  }

extern "C" int cast_fused_supported(int H) { return H > 0 && H <= 64; }

template <int KS>
static void launch_qkv_bwd_mma(const QkvBwdArgs& a, FDims d, int grid, cudaStream_t stream) {
  d.HS = 8 * KS + 4;
  const size_t smem = qkv_bwd_mma_smem<KS>();
  auto kf = qkv_bwd_mma_kernel<KS, RM_BWD_NG>;
  CAST_FUSED_SMEM(kf, smem)
  CAST_LAUNCH_DEP(kf, dim3(grid), dim3(128 * RM_BWD_NG), smem, stream, a, d);
}
template <int KS>
static void launch_ffn_bwd_mma(const FfnBwdArgs& a, FDims d, int grid, cudaStream_t stream) {
  d.HS = 8 * KS + 4;
  const size_t smem = ffn_bwd_mma_smem<KS>();
  auto kf = ffn_bwd_mma_kernel<KS, RM_BWD_NG>;
  CAST_FUSED_SMEM(kf, smem)
  CAST_LAUNCH_DEP(kf, dim3(grid), dim3(128 * RM_BWD_NG), smem, stream, a, d);
}
template <int KS>
static void launch_ln_qkv_fwd_mma(const LnQkvArgs& a, FDims d, cudaStream_t stream) {
  d.HS = 8 * KS + 4;
  const long ntiles = cdiv(d.N, FR);
  const size_t smem = ln_qkv_fwd_mma_smem<KS>();
  auto kf = ln_qkv_fwd_mma_kernel<KS>;
  CAST_FUSED_SMEM(kf, smem)
  CAST_LAUNCH(kf, dim3((unsigned)ntiles), dim3(FT), smem, stream, a, d);
}
template <int KS>
static void launch_ln_ffn_fwd_mma(const LnFfnArgs& a, FDims d, cudaStream_t stream) {
  d.HS = 8 * KS + 4;
  const long ntiles = cdiv(d.N, FR);
  const size_t smem = ln_ffn_fwd_mma_smem<KS>();
  auto kf = ln_ffn_fwd_mma_kernel<KS>;
  CAST_FUSED_SMEM(kf, smem)
  CAST_LAUNCH(kf, dim3((unsigned)ntiles), dim3(FT), smem, stream, a, d);
}
#define CAST_KS_SWITCH(H, CALL)                                                          \
  switch (((H) + 7) / 8) {                                                               \
    case 1: CALL(1); break; case 2: CALL(2); break; case 3: CALL(3); break; case 4: CALL(4); break; \
    case 5: CALL(5); break; case 6: CALL(6); break; case 7: CALL(7); break; default: CALL(8); break; \
  }

extern "C" int cast_ln_qkv_fwd(const float* x, const float* gamma, const float* beta, const float* Wq, const float* bq,
                               const float* Wk, const float* bk, const float* Wv, const float* bv, long N, int H,
                               float eps, float* qn, float* Q, float* K, float* V, float* mean, float* rstd,
                               float* kmask, float* qmask, void* stream) {
  if (!x || !gamma || !beta || !Wq || !bq || !Wk || !bk || !Wv || !bv || !qn || !Q || !K || !V || N <= 0)
    return set_error(CAST_ERR_BAD_ARG, "ln_qkv_fwd");
  if (!cast_fused_supported(H)) return set_error(CAST_ERR_UNSUPPORTED, "ln_qkv_fwd: H > 64");
  const FDims d = fdims(N, H);
  LnQkvArgs a{x, gamma, beta, {Wq, Wk, Wv}, {bq, bk, bv}, eps, qn, {Q, K, V}, mean, rstd, kmask, qmask};
#define CAST_CALL(K) launch_ln_qkv_fwd_mma<K>(a, d, (cudaStream_t)stream)
  CAST_KS_SWITCH(H, CAST_CALL)
#undef CAST_CALL
  return check_launch("ln_qkv_fwd");
}

extern "C" int cast_ln_ffn_fwd(const float* y, const float* gamma, const float* beta, const float* W1, const float* b1,
                               const float* W2, const float* b2, const int* ids, float drop_rate,
                               unsigned long long seed, const unsigned long long* step, int site_hidden, int site_out,
                               long N, int H, float eps, float* zn, float* h1d, float* xout, float* mean, float* rstd,
                               void* stream) {
  if (!y || !gamma || !beta || !W1 || !b1 || !W2 || !b2 || !zn || !h1d || !xout || N <= 0)
    return set_error(CAST_ERR_BAD_ARG, "ln_ffn_fwd");
  if (!cast_fused_supported(H)) return set_error(CAST_ERR_UNSUPPORTED, "ln_ffn_fwd: H > 64");
  if (drop_rate < 0.f || drop_rate >= 1.f) return set_error(CAST_ERR_BAD_ARG, "ln_ffn_fwd: drop_rate");
  const FDims d = fdims(N, H);
  LnFfnArgs a{y, gamma, beta, W1, b1, W2, b2, ids, eps, drop_rate, seed, step, site_hidden, site_out,
              zn, h1d, xout, mean, rstd};
#define CAST_CALL(K) launch_ln_ffn_fwd_mma<K>(a, d, (cudaStream_t)stream)
  CAST_KS_SWITCH(H, CAST_CALL)
#undef CAST_CALL
  return check_launch("ln_ffn_fwd");
}

/* number of per-CTA partial blocks cast_ffn_bwd / cast_qkv_bwd leave in their workspace for N rows */
extern "C" int cast_block_bwd_parts(long N, int which) {  // which: 0 = cast_ffn_bwd, 1 = cast_qkv_bwd
  (void)which;  // both kernels run the same grid
  return bwd_grid(cdiv(N, FR), 1);
}

// sized for up to two CTAs per SM, twice what the kernels use: callers size their buffers with this value, so it stays
extern "C" size_t cast_block_bwd_workspace_bytes(long N, int H) {
  const long ntiles = cdiv(N, FR);
  return (size_t)bwd_grid(ntiles, 2) * (size_t)(2L * H + 3L * ((long)H * H + H)) * sizeof(float);
}

extern "C" int cast_ffn_bwd(const float* dx, const int* ids, const float* zn, const float* h1d, const float* y,
                            const float* mean, const float* rstd, const float* gamma, const float* W1, const float* W2,
                            float drop_rate, unsigned long long seed, const unsigned long long* step, int site_out,
                            long N, int H, float* dy, float* grads_out, void* workspace, size_t workspace_bytes,
                            void* stream) {
  if (!dx || !zn || !h1d || !y || !mean || !rstd || !gamma || !W1 || !W2 || !dy || N <= 0)
    return set_error(CAST_ERR_BAD_ARG, "ffn_bwd");
  if (!cast_fused_supported(H)) return set_error(CAST_ERR_UNSUPPORTED, "ffn_bwd: H > 64");
  if (!workspace || workspace_bytes < cast_block_bwd_workspace_bytes(N, H))
    return set_error(CAST_ERR_WORKSPACE, "ffn_bwd: workspace too small");
  const FDims d = fdims(N, H);
  const long ntiles = cdiv(N, FR);
  const int grid = bwd_grid(ntiles, 1);
  FfnBwdArgs a{dx, zn, h1d, y, mean, rstd, gamma, W1, W2, ids, drop_rate, seed, step, site_out, dy,
               static_cast<float*>(workspace), ntiles};
#define CAST_CALL(K) launch_ffn_bwd_mma<K>(a, d, grid, (cudaStream_t)stream)
  CAST_KS_SWITCH(H, CAST_CALL)
#undef CAST_CALL
  int rc = check_launch("ffn_bwd");
  if (rc || !grads_out) return rc;  // grads_out == null: partials stay in the workspace (cast_reduce_partials_batch)
  const long count = 2L * H + 2L * ((long)H * H + H);
  return launch_reduce_partials(static_cast<float*>(workspace), grid, count, grads_out, count, (float*)nullptr,
                                (cudaStream_t)stream);
}

// out_fx != 0: dx is also multiplied by the padding mask of out_ids (may be null) and by the dropout keep/scale of
// (out_rate, seed, *step, out_site) at flat index row*H + col — the gradient of `dropout(emb) * mask` (sasrec.py:58-62)
static int qkv_bwd_impl(const float* dQ, const float* dK, const float* dV, const float* dres, const float* x,
                        const float* qn, const float* mean, const float* rstd, const float* gamma, const float* Wq,
                        const float* Wk, const float* Wv, long N, int H, float* dx, float* grads_out, void* workspace,
                        size_t workspace_bytes, int out_fx, const int* out_ids, float out_rate, unsigned long long seed,
                        const unsigned long long* step, int out_site, void* stream) {
  if (!dQ || !dK || !dV || !dres || !x || !qn || !mean || !rstd || !gamma || !Wq || !Wk || !Wv || !dx || N <= 0)
    return set_error(CAST_ERR_BAD_ARG, "qkv_bwd");
  if (!cast_fused_supported(H)) return set_error(CAST_ERR_UNSUPPORTED, "qkv_bwd: H > 64");
  if (!workspace || workspace_bytes < cast_block_bwd_workspace_bytes(N, H))
    return set_error(CAST_ERR_WORKSPACE, "qkv_bwd: workspace too small");
  const FDims d = fdims(N, H);
  const long ntiles = cdiv(N, FR);
  const int grid = bwd_grid(ntiles, 1);
  QkvBwdArgs a{dQ, dK, dV, dres, x, qn, mean, rstd, gamma, Wq, Wk, Wv, dx, static_cast<float*>(workspace), ntiles,
               out_ids, out_rate, seed, step, out_site, out_fx};
#define CAST_CALL(K) launch_qkv_bwd_mma<K>(a, d, grid, (cudaStream_t)stream)
  CAST_KS_SWITCH(H, CAST_CALL)
#undef CAST_CALL
  int rc = check_launch("qkv_bwd");
  if (rc || !grads_out) return rc;
  const long count = 2L * H + 3L * ((long)H * H + H);
  return launch_reduce_partials(static_cast<float*>(workspace), grid, count, grads_out, count, (float*)nullptr,
                                (cudaStream_t)stream);
}

extern "C" int cast_qkv_bwd(const float* dQ, const float* dK, const float* dV, const float* dres, const float* x,
                            const float* qn, const float* mean, const float* rstd, const float* gamma, const float* Wq,
                            const float* Wk, const float* Wv, long N, int H, float* dx, float* grads_out,
                            void* workspace, size_t workspace_bytes, void* stream) {
  return qkv_bwd_impl(dQ, dK, dV, dres, x, qn, mean, rstd, gamma, Wq, Wk, Wv, N, H, dx, grads_out, workspace,
                      workspace_bytes, 0, nullptr, 0.f, 0ull, nullptr, 0, stream);
}

extern "C" int cast_qkv_bwd_embed(const float* dQ, const float* dK, const float* dV, const float* dres, const float* x,
                                  const float* qn, const float* mean, const float* rstd, const float* gamma,
                                  const float* Wq, const float* Wk, const float* Wv, long N, int H,
                                  const int* mask_ids, float drop_rate, unsigned long long seed,
                                  const unsigned long long* step, int site, float* dx, float* grads_out,
                                  void* workspace, size_t workspace_bytes, void* stream) {
  return qkv_bwd_impl(dQ, dK, dV, dres, x, qn, mean, rstd, gamma, Wq, Wk, Wv, N, H, dx, grads_out, workspace,
                      workspace_bytes, 1, mask_ids, drop_rate, seed, step, site, stream);
}
