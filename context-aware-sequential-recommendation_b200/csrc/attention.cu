// K4 dispatch: see attention.cuh for the kernels.  The per-head-width instantiations live in attention_w*.cu so that
// they compile in parallel.
#include "attention.cuh"

namespace cast {

extern template int dispatch_att<4>(int, const AttnFwdArgs*, const AttnBwdArgs*, const AttnDims&, cudaStream_t);
extern template int dispatch_att<8>(int, const AttnFwdArgs*, const AttnBwdArgs*, const AttnDims&, cudaStream_t);
extern template int dispatch_att<12>(int, const AttnFwdArgs*, const AttnBwdArgs*, const AttnDims&, cudaStream_t);
extern template int dispatch_att<16>(int, const AttnFwdArgs*, const AttnBwdArgs*, const AttnDims&, cudaStream_t);
extern template int dispatch_att<20>(int, const AttnFwdArgs*, const AttnBwdArgs*, const AttnDims&, cudaStream_t);
extern template int dispatch_att<24>(int, const AttnFwdArgs*, const AttnBwdArgs*, const AttnDims&, cudaStream_t);
extern template int dispatch_att<28>(int, const AttnFwdArgs*, const AttnBwdArgs*, const AttnDims&, cudaStream_t);
extern template int dispatch_att<32>(int, const AttnFwdArgs*, const AttnBwdArgs*, const AttnDims&, cudaStream_t);
extern template int dispatch_att<36>(int, const AttnFwdArgs*, const AttnBwdArgs*, const AttnDims&, cudaStream_t);
extern template int dispatch_att<40>(int, const AttnFwdArgs*, const AttnBwdArgs*, const AttnDims&, cudaStream_t);
extern template int dispatch_att<44>(int, const AttnFwdArgs*, const AttnBwdArgs*, const AttnDims&, cudaStream_t);
extern template int dispatch_att<48>(int, const AttnFwdArgs*, const AttnBwdArgs*, const AttnDims&, cudaStream_t);
extern template int dispatch_att<52>(int, const AttnFwdArgs*, const AttnBwdArgs*, const AttnDims&, cudaStream_t);
extern template int dispatch_att<56>(int, const AttnFwdArgs*, const AttnBwdArgs*, const AttnDims&, cudaStream_t);
extern template int dispatch_att<60>(int, const AttnFwdArgs*, const AttnBwdArgs*, const AttnDims&, cudaStream_t);
extern template int dispatch_att<64>(int, const AttnFwdArgs*, const AttnBwdArgs*, const AttnDims&, cudaStream_t);
extern template int dispatch_att<100>(int, const AttnFwdArgs*, const AttnBwdArgs*, const AttnDims&, cudaStream_t);
extern template int dispatch_att<128>(int, const AttnFwdArgs*, const AttnBwdArgs*, const AttnDims&, cudaStream_t);
extern template int dispatch_att<256>(int, const AttnFwdArgs*, const AttnBwdArgs*, const AttnDims&, cudaStream_t);

bool attn_mma_supported(const AttnDims& dm);
int dispatch_att_mma(int which, const AttnFwdArgs* fa, const AttnBwdArgs* ba, const float* out, const float* resid,
                     float* pbuf, float* dbuf, const AttnDims& dm, cudaStream_t stream);

static int dispatch_by_width(int which, const AttnFwdArgs* fa, const AttnBwdArgs* ba, const AttnDims& dm,
                             cudaStream_t stream) {
  switch (dm.dpad) {
#define CAST_W(D) case D: return dispatch_att<D>(which, fa, ba, dm, stream);
    CAST_W(4) CAST_W(8) CAST_W(12) CAST_W(16) CAST_W(20) CAST_W(24) CAST_W(28) CAST_W(32) CAST_W(36) CAST_W(40)
    CAST_W(44) CAST_W(48) CAST_W(52) CAST_W(56) CAST_W(60) CAST_W(64) CAST_W(100) CAST_W(128) CAST_W(256)
#undef CAST_W
    default:
      return set_error(CAST_ERR_UNSUPPORTED,
                       "attention: head width not instantiated (supported: d <= 64, 97..100, 125..128, 253..256)");
  }
}

}  // namespace cast

using namespace cast;

extern "C" size_t cast_attn_bwd_workspace_bytes(int B, int T, int h) {
  return 2 * (size_t)B * h * T * T * sizeof(float);
}

extern "C" int cast_attn_fwd(const float* Q, long ldq, const float* K, long ldk, const float* V, long ldv,
                             const float* queries, const float* kmask, const float* qmask, int B, int T, int H, int h,
                             float drop_rate, unsigned long long seed, const unsigned long long* step, int site,
                             const int* skip_ids, float* out, float* attn_weights, float* row_max, float* row_linv,
                             void* stream) {
  if (!Q || !K || !V || !queries || !kmask || !qmask || !out || B <= 0 || T <= 0 || H <= 0 || h <= 0 || H % h)
    return set_error(CAST_ERR_BAD_ARG, "attn_fwd");
  if (drop_rate < 0.f || drop_rate >= 1.f) return set_error(CAST_ERR_BAD_ARG, "attn_fwd: drop_rate");
  const AttnDims dm = make_dims(B, T, H, h);
  AttnFwdArgs args{Q, K, V, ldq, ldk, ldv, queries, kmask, qmask, out, skip_ids, attn_weights, row_max, row_linv,
                   drop_rate, seed, step, site};
  // tensor-core path (attention_mma.cu) unless the [h*B,T,T] weights are wanted or the head is wider than 64
  int rc = (!attn_weights && attn_mma_supported(dm))
               ? dispatch_att_mma(0, &args, nullptr, nullptr, nullptr, nullptr, nullptr, dm, (cudaStream_t)stream)
               : dispatch_by_width(0, &args, nullptr, dm, (cudaStream_t)stream);
  if (rc) return rc;
  return check_launch("attn_fwd");
}

extern "C" int cast_attn_bwd(const float* Q, long ldq, const float* K, long ldk, const float* V, long ldv,
                             const float* dO, const float* kmask, const float* qmask, const float* row_max,
                             const float* row_linv, const int* skip_ids, float* rowD, int B, int T, int H, int h,
                             float drop_rate, unsigned long long seed, const unsigned long long* step, int site,
                             float* dQ, long lddq,
                             float* dK, long lddk, float* dV, long lddv, const float* out, const float* queries,
                             void* workspace, size_t workspace_bytes, void* stream) {
  if (!Q || !K || !V || !dO || !kmask || !qmask || !row_max || !row_linv || !rowD || !dQ || !dK || !dV || B <= 0 ||
      T <= 0 || H <= 0 || h <= 0 || H % h)
    return set_error(CAST_ERR_BAD_ARG, "attn_bwd");
  const AttnDims dm = make_dims(B, T, H, h);
  AttnBwdArgs args{Q, K, V, ldq, ldk, ldv, dO, kmask, qmask, row_max, row_linv, skip_ids, rowD, dQ, dK, dV, lddq, lddk,
                   lddv,
                   drop_rate, seed, step, site};
  const bool mma = out && queries && attn_mma_supported(dm);
  // with a [2][h*B,T,T] workspace the dQ kernel stores P~ and dS and the dK/dV kernel does not recompute them
  const size_t half = (size_t)B * h * T * T * sizeof(float);
  float* pbuf = (mma && workspace && workspace_bytes >= 2 * half) ? static_cast<float*>(workspace) : nullptr;
  float* dbuf = pbuf ? pbuf + (size_t)B * h * T * T : nullptr;
  int rc = mma ? dispatch_att_mma(1, nullptr, &args, out, queries, pbuf, dbuf, dm, (cudaStream_t)stream)
               : dispatch_by_width(1, nullptr, &args, dm, (cudaStream_t)stream);
  if (rc) return rc;
  if ((rc = check_launch("attn_bwd_dq"))) return rc;
  rc = mma ? dispatch_att_mma(2, nullptr, &args, out, queries, pbuf, dbuf, dm, (cudaStream_t)stream)
           : dispatch_by_width(2, nullptr, &args, dm, (cudaStream_t)stream);
  if (rc) return rc;
  return check_launch("attn_bwd_dkv");
}
