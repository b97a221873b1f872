// Backward row-tile kernels of one transformer block when hidden_units <= 64 (BASELINE configs 1-3, H = 50):
//   ffn_bwd : backward of LN(y) -> relu(.W1+b1) -> dropout -> .W2+b2 -> dropout -> + LN(y) -> *mask
//             (sasrec.py:81-83, modules.py:298-313) incl. dW1, dW2, db1, db2, dgamma, dbeta
//   qkv_bwd : backward of LN(x) -> Q = LN(x)Wq+bq, K = xWk+bk, V = xWv+bv (modules.py:74-78, :203-205)
//             incl. dWq, dWk, dWv, biases, dgamma, dbeta (and the attention residual)
// Their forward halves are the tcgen05 row kernels of row_umma.cu.  One CTA works on 64-row tiles with all H columns;
// the kernels themselves (fused_mma.cuh) contract on the tensor cores (mma.sync 3xTF32).  The whole weight matrix
// (H*H*4 <= 16 KB) sits in shared memory; activations make exactly one HBM round trip per kernel instead of one per op.
// The kernels are persistent (one CTA per SM loops over row tiles) and keep their weight-gradient partials in
// registers; a fixed-order second stage sums the per-CTA partials straight into the flat gradient buffer =>
// deterministic.
// Gradient layout contract (flat, contiguous, see engine.param_shapes):
//   qkv_bwd -> [ln1.beta H | ln1.gamma H | q.w H*H | q.b H | k.w H*H | k.b H | v.w H*H | v.b H]
//   ffn_bwd -> [ln2.beta H | ln2.gamma H | ffn1.w H*H | ffn1.b H | ffn2.w H*H | ffn2.b H]
#include "cast_rt.cuh"

namespace cast {

int launch_reduce_partials(const float* partial, int nparts, long count, float* out0, long split, float* out1,
                           cudaStream_t stream);

constexpr int FR = 64;        // rows per tile

struct FDims {
  long N;
  int H;
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

static bool bwd_supported(int H) { return H > 0 && H <= 64; }

template <int KS>
static void launch_qkv_bwd_mma(const QkvBwdArgs& a, FDims d, int grid, cudaStream_t stream) {
  const size_t smem = qkv_bwd_mma_smem<KS>();
  auto kf = qkv_bwd_mma_kernel<KS, RM_BWD_NG>;
  CAST_FUSED_SMEM(kf, smem)
  CAST_LAUNCH_DEP(kf, dim3(grid), dim3(128 * RM_BWD_NG), smem, stream, a, d);
}
template <int KS>
static void launch_ffn_bwd_mma(const FfnBwdArgs& a, FDims d, int grid, cudaStream_t stream) {
  const size_t smem = ffn_bwd_mma_smem<KS>();
  auto kf = ffn_bwd_mma_kernel<KS, RM_BWD_NG>;
  CAST_FUSED_SMEM(kf, smem)
  CAST_LAUNCH_DEP(kf, dim3(grid), dim3(128 * RM_BWD_NG), smem, stream, a, d);
}
#define CAST_KS_SWITCH(H, CALL)                                                          \
  switch (((H) + 7) / 8) {                                                               \
    case 1: CALL(1); break; case 2: CALL(2); break; case 3: CALL(3); break; case 4: CALL(4); break; \
    case 5: CALL(5); break; case 6: CALL(6); break; case 7: CALL(7); break; default: CALL(8); break; \
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
  if (!bwd_supported(H)) return set_error(CAST_ERR_UNSUPPORTED, "ffn_bwd: H > 64");
  if (!workspace || workspace_bytes < cast_block_bwd_workspace_bytes(N, H))
    return set_error(CAST_ERR_WORKSPACE, "ffn_bwd: workspace too small");
  const FDims d{N, H};
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
  if (!bwd_supported(H)) return set_error(CAST_ERR_UNSUPPORTED, "qkv_bwd: H > 64");
  if (!workspace || workspace_bytes < cast_block_bwd_workspace_bytes(N, H))
    return set_error(CAST_ERR_WORKSPACE, "qkv_bwd: workspace too small");
  const FDims d{N, H};
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
