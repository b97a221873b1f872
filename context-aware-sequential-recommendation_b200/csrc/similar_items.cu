// Exact item-to-item retrieval: for each query item q the K items j in [1, V) of the table, j != q (the caller's
// exclusion rows), with the largest canonical score, ties broken by item id ascending.  The scorer is cast_topk_full
// (topk_full.cu) unchanged; this file only prepares its two operands:
//   - the query operand [U, H]: the rows of the query ids, read from the local table or from the owners' shards of a
//     row-sharded table (TableRef), and
//   - under the cosine metric, the normalised table ê [V, H] of the local table or shard.
// Canonical normalisation (the same bits for a row wherever it is read): n = sqrt_rn(sum_k e_k * e_k), k ascending,
// multiply and add rounded separately (as canonical_dot); ê_k = e_k / n (IEEE division); n == 0 -> the zero vector.
// Scores are then canonical_dot(ê_q, ê_j) (cosine) or canonical_dot(e_q, e_j) (dot), so both tensor-core filter and
// brute force return those bits.  cast_similar_items_biased adds a per-item offset b_j (local rows) to every score
// exactly as cast_topk_full_biased does.
#include "cast_rt.cuh"

namespace cast {

constexpr int SI_WARPS = 8;   // rows per CTA of item_rows_kernel (one warp per row)

// out[i] = row ids[i] of the table (ids == nullptr: row i), normalised when `normalize`; ids outside [0, V) give a
// zero row.  One warp per row: the row is staged in shared memory, every lane runs the same sequential norm over it.
__global__ void __launch_bounds__(32 * SI_WARPS) item_rows_kernel(const int* __restrict__ ids, long n, TableRef table,
                                                                  int V, int H, int normalize, float* __restrict__ out) {
  CAST_DYN_SMEM(float, sm);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const long i = (long)blockIdx.x * SI_WARPS + w;
  if (i >= n) return;
  float* srow = sm + (size_t)w * H;
  const long id = ids ? (long)ids[i] : i;
  const bool live = id >= 0 && id < V;
  const float* r = table.row(live ? (int)id : 0, H);
  for (int k = lane; k < H; k += 32) srow[k] = live ? r[k] : 0.f;
  __syncwarp();
  float nrm = 1.f;
  if (normalize) {
    float n2 = 0.f;
    for (int k = 0; k < H; ++k) n2 = __fadd_rn(n2, __fmul_rn(srow[k], srow[k]));
    nrm = __fsqrt_rn(n2);
  }
  float* o = out + i * H;
  for (int k = lane; k < H; k += 32) {
    const float x = srow[k];
    o[k] = !normalize ? x : (nrm == 0.f ? 0.f : __fdiv_rn(x, nrm));
  }
}

static int launch_item_rows(const int* ids, long n, TableRef t, int V, int H, int normalize, float* out,
                            cudaStream_t st) {
  CAST_LAUNCH(item_rows_kernel, dim3((unsigned)cdiv(n, SI_WARPS)), dim3(32 * SI_WARPS),
              (size_t)SI_WARPS * H * sizeof(float), st, ids, n, t, V, H, normalize, out);
  return check_launch("item_rows");
}

struct SiLayout {
  size_t topk, q, ehat, total;
};

// workspace: [cast_topk_full workspace (its watchdog flag first) | query rows U x H | ê V x H (cosine only)]
static SiLayout si_layout(long U, int V, int H, int K, int metric) {
  SiLayout l;
  l.topk = 0;
  size_t o = (cast_topk_full_workspace_bytes(U, V, H, K) + 255) & ~(size_t)255;
  l.q = o; o += ((size_t)U * H * 4 + 255) & ~(size_t)255;
  l.ehat = o; if (metric == CAST_SIM_COSINE) o += ((size_t)V * H * 4 + 255) & ~(size_t)255;
  l.total = o;
  return l;
}

}  // namespace cast

using namespace cast;

extern "C" int cast_item_rows(const int* ids, long n, const float* table, const float* const* shards, int nshards,
                              int V, int H, int normalize, float* out, void* stream) {
  if (n <= 0 || V <= 0 || H <= 0 || !out || (!table && !shards) || (shards && nshards < 1) ||
      (size_t)SI_WARPS * H * sizeof(float) > 48 * 1024)
    return set_error(CAST_ERR_BAD_ARG, "item_rows");
  const TableRef t = shards ? table_ref(shards, nshards) : table_ref(table);
  return launch_item_rows(ids, n, t, V, H, normalize ? 1 : 0, out, (cudaStream_t)stream);
}

extern "C" size_t cast_similar_items_workspace_bytes(long U, int V, int H, int K, int metric) {
  if ((metric != CAST_SIM_DOT && metric != CAST_SIM_COSINE) || cast_topk_full_workspace_bytes(U, V, H, K) == 0)
    return 0;
  return si_layout(U, V, H, K, metric).total;
}

extern "C" int cast_similar_items_biased(const int* ids, long U, const float* table, int V, const float* const* shards,
                                         int nshards, int V_items, int H, int K, int metric, const int* excl_ptr,
                                         const int* excl_idx, const float* item_bias, int mode, int* top_ids,
                                         float* top_scores, unsigned long long* stats, void* workspace,
                                         size_t workspace_bytes, void* stream) {
  if (K < 1 || K > 256) return set_error(CAST_ERR_BAD_ARG, "similar_items: K must be in [1, 256]");
  if (metric != CAST_SIM_DOT && metric != CAST_SIM_COSINE)
    return set_error(CAST_ERR_BAD_ARG, "similar_items: metric must be CAST_SIM_DOT or CAST_SIM_COSINE");
  if (!ids || !table || U <= 0 || V <= 1 || H <= 0 || (shards && (nshards < 1 || V_items <= 1)) ||
      (size_t)SI_WARPS * H * sizeof(float) > 48 * 1024)
    return set_error(CAST_ERR_BAD_ARG, "similar_items");
  if ((uintptr_t)item_bias % 16 != 0)
    return set_error(CAST_ERR_BAD_ARG, "similar_items: item_bias must be 16-byte aligned");
  const SiLayout l = si_layout(U, V, H, K, metric);
  if (!workspace || workspace_bytes < l.total)
    return set_error(CAST_ERR_WORKSPACE, "similar_items: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  unsigned char* w = static_cast<unsigned char*>(workspace);
  float* q = reinterpret_cast<float*>(w + l.q);
  const int cos = metric == CAST_SIM_COSINE ? 1 : 0;
  const TableRef src = shards ? table_ref(shards, nshards) : table_ref(table);
  int rc;
  if ((rc = launch_item_rows(ids, U, src, shards ? V_items : V, H, cos, q, st))) return rc;
  const float* scored = table;
  if (cos) {
    float* ehat = reinterpret_cast<float*>(w + l.ehat);
    if ((rc = launch_item_rows(nullptr, V, table_ref(table), V, H, 1, ehat, st))) return rc;
    scored = ehat;
  }
  return cast_topk_full_biased(q, H, scored, V, H, U, K, excl_ptr, excl_idx, item_bias, mode, top_ids, top_scores,
                               stats, w + l.topk, l.q - l.topk, stream);
}

extern "C" int cast_similar_items(const int* ids, long U, const float* table, int V, const float* const* shards,
                                  int nshards, int V_items, int H, int K, int metric, const int* excl_ptr,
                                  const int* excl_idx, int mode, int* top_ids, float* top_scores,
                                  unsigned long long* stats, void* workspace, size_t workspace_bytes, void* stream) {
  return cast_similar_items_biased(ids, U, table, V, shards, nshards, V_items, H, K, metric, excl_ptr, excl_idx,
                                   nullptr, mode, top_ids, top_scores, stats, workspace, workspace_bytes, stream);
}

extern "C" int cast_similar_items_status(const void* workspace, long U, int V, int H, int K, int* host_flag,
                                         void* stream) {
  return cast_topk_full_status(workspace, U, V, H, K, host_flag, stream);   // its workspace sits at the start
}
