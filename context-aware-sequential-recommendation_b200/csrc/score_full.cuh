// Shared pieces of the full-catalog scorers (score_full.cu: rank of a target; topk_full.cu: exact top-K): the canonical
// fp32 dot, the item / tile norm kernels that feed the rigorous error bound, and the tcgen05 user-tile x item-tile
// pipeline, templated on its epilogue.  Kernels defined here are static or templates, so every translation unit that
// includes this header emits its own copies and no host stub is defined twice.
#pragma once
#include "cast_rt.cuh"
#ifndef CAST_EMU
#include "umma.cuh"
#endif

namespace cast {

// canonical logit: sequential k, separately rounded multiply and add
__device__ __forceinline__ float canonical_dot(const float* __restrict__ u, const float* __restrict__ e, int H) {
  float acc = 0.f;
  for (int k = 0; k < H; ++k) acc = __fadd_rn(acc, __fmul_rn(u[k], e[k]));
  return acc;
}

constexpr float NORM_SLACK = 1.0001f;  // fp32 norm evaluation error, folded into the bound

// inorm[j] >= |e_j|_2 (row 0 is the zero-pad row of the lookup table: never a candidate)
static __global__ void item_norm_kernel(const float* __restrict__ table, int V, int H, float* __restrict__ inorm) {
  const int lane = threadIdx.x & 31;
  const long j = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (j >= V) return;
  float s = 0.f;
  for (int k = lane; k < H; k += 32) {
    const float x = table[j * H + k];
    s = fmaf(x, x, s);
  }
  s = warp_sum(s);
  if (lane == 0) inorm[j] = sqrtf(s) * NORM_SLACK;
}

// tnorm[t] = max of inorm over the 256 items of tile t (one warp per tile)
static __global__ void tile_norm_kernel(const float* __restrict__ inorm, int V, int tile, float* __restrict__ tnorm) {
  const int lane = threadIdx.x & 31;
  const long t = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (t * tile >= V) return;
  float m = 0.f;
  for (long j = t * tile + lane; j < (t + 1) * tile && j < V; j += 32) m = fmaxf(m, inorm[j]);
  m = warp_max(m);
  if (lane == 0) tnorm[t] = m;
}

// |s~ - s| <= sf_cbound(kpad) * |u| * |e_j| for the 3xTF32 tile: three dropped/rounded split terms (3 * 2^-22) plus
// one accumulation error of at most 2^-22 * sum|u_k e_k| per MMA (3 * kpad/8 MMAs per tile); doubled for slack
static inline float sf_cbound(int kpad) { return 2.0f * (3.0f + 3.0f * (float)kpad / 8.0f) * 2.384185791015625e-07f; }

static inline size_t sf_align(size_t x) { return (x + 255) & ~(size_t)255; }

constexpr int SF_EPI_WARPS = 8;                // two warps per TMEM lane quarter (each takes half of the columns)
constexpr int SF_THREADS = 64 + 32 * SF_EPI_WARPS;
constexpr int SF_M = 128;                      // users per tile  (UMMA M)
constexpr int SF_N = 256;                      // items per tile  (UMMA N); 2 accumulators = all 512 TMEM columns
constexpr int SF_KC = 32;                      // K elements per pipeline chunk
constexpr int SF_SLABS = SF_KC / 4;
constexpr int SF_A_PITCH = SF_M * 16 + 16;     // bytes between K slabs of the user tile
constexpr int SF_B_PITCH = SF_N * 16 + 16;     // bytes between K slabs of the item tile
constexpr int SF_ABYTES = 2 * SF_SLABS * SF_A_PITCH;   // one user-tile chunk: hi slabs then lo slabs
constexpr int SF_BBYTES = 2 * SF_SLABS * SF_B_PITCH;   // one item-tile chunk
constexpr int SF_STAGES = 2;
constexpr size_t SF_SMEM = (size_t)SF_STAGES * (SF_ABYTES + SF_BBYTES) + 128;

// pre-split operand images (users: 128-row tiles, items: 256-row tiles)
static inline size_t sf_presplit_bytes(long U, int V, int H, size_t* a_bytes) {
#ifndef CAST_EMU
  const int kpad = (H + 7) & ~7;
  const size_t nkc = (size_t)cdiv(kpad, SF_KC);
  const size_t ab = (size_t)cdiv(U, SF_M) * nkc * SF_ABYTES;
  const size_t bb = (size_t)cdiv(V, SF_N) * nkc * SF_BBYTES;
  if (a_bytes) *a_bytes = sf_align(ab);
  return sf_align(ab) + sf_align(bb);
#else
  (void)U; (void)V; (void)H;
  if (a_bytes) *a_bytes = 0;
  return 0;
#endif
}

#ifndef CAST_EMU
// ------------------------------------------------------------------------------------------------ tensor-core path
// Warp-specialised pipeline, one persistent CTA per SM:
//   warp 0 (one lane)  producer : TMA 1-D bulk copies (cp.async.bulk) of pre-split operand chunks into a 2-stage
//                                 shared-memory ring, completion counted on `full[s]` as transaction bytes
//   warp 1 (one lane)  MMA      : waits full[s], issues 3 x tcgen05.mma per 8 K-elements into one of TWO TMEM
//                                 accumulators (2 x 256 columns), tcgen05.commit -> empty[s] (stage free) and, after the
//                                 last K chunk of a tile, -> tfull[acc]
//   warps 2-9          epilogue : wait tfull[acc], tcgen05.ld the 128 x 256 tile (thread <-> user row, two warps per
//                                 lane quarter split the columns), hand each 32-column chunk to the epilogue policy
//                                 `Epi`, then arrive on tempty[acc]
// so the copy of chunk k+1, the MMAs of chunk k and the epilogue of the previous tile overlap.  Operands are split
// into tf32 hi/lo ONCE by presplit_kernel into the exact shared-memory image of a chunk (K-major slabs, see umma.cuh),
// so the hot loop executes no conversion instructions at all: the item table is static for a whole evaluation.

// X [R, ld] row-major fp32 -> out[tile][kchunk][hi|lo][slab][TR rows x 16 B (+16 B pad)]; zero beyond R rows / H cols
template <int TR>
__global__ void presplit_kernel(const float* __restrict__ X, long ld, long R, int H, int nkc,
                                unsigned char* __restrict__ out) {
  constexpr int PITCH = TR * 16 + 16;
  constexpr int CBYTES = 2 * SF_SLABS * PITCH;
  const long tile = blockIdx.x;
  const int kc = blockIdx.y;
  unsigned char* dst = out + ((size_t)tile * nkc + kc) * CBYTES;
  for (int idx = threadIdx.x; idx < TR * SF_SLABS; idx += blockDim.x) {
    const int r = idx / SF_SLABS, c = idx - r * SF_SLABS;
    const long row = tile * TR + r;
    const int k = kc * SF_KC + 4 * c;
    float x[4] = {0.f, 0.f, 0.f, 0.f};
    if (row < R) {
#pragma unroll
      for (int e = 0; e < 4; ++e)
        if (k + e < H) x[e] = __ldg(X + row * ld + k + e);
    }
    float4 h, l;
    umma::split_tf32(x[0], h.x, l.x);
    umma::split_tf32(x[1], h.y, l.y);
    umma::split_tf32(x[2], h.z, l.z);
    umma::split_tf32(x[3], h.w, l.w);
    *reinterpret_cast<float4*>(dst + (size_t)c * PITCH + r * 16) = h;
    *reinterpret_cast<float4*>(dst + (size_t)(SF_SLABS + c) * PITCH + r * 16) = l;
  }
}

// what the pipeline itself needs; the epilogue policy brings its own parameters
struct SfPipe {
  const float* users;
  long ldu;
  const float* table;
  const unsigned char* apre;   // pre-split user tiles
  const unsigned char* bpre;   // pre-split item tiles
  const float* tnorm;          // per item tile: max of |e_j| over the tile
  const float* unorm;          // per user: |u|
  int V, H;
  long U;
  int nkc;               // K chunks of SF_KC elements
  int kpad;              // H rounded up to 8
  long items_per_split;  // multiple of SF_N
  int nsplit;
  long nunits;           // user tiles x nsplit
  float cbound;
  int* err;              // watchdog flag: an mbarrier wait timed out
};

// Work unit `unit` = (user tile, item split).  The epilogue policy is constructed once per (thread, unit):
//   Epi(const SfPipe&, const Epi::Params&, long user, bool live, int split, int column_half, int jb, int je)
//   tile(j0, d)      before the tile at item j0; d >= |s~ - s| for every item of the tile
//   chunk(v, j)      32 accumulator values of items j .. j+31 (live threads only)
//   finish()         after the unit's last tile (live threads, pipeline not failed)
template <class Epi>
__global__ void __launch_bounds__(SF_THREADS, 1) sf_umma_kernel(SfPipe a, typename Epi::Params ep) {
  extern __shared__ __align__(128) unsigned char sf_smem[];
  __shared__ __align__(8) uint64_t full[SF_STAGES], empty[SF_STAGES], tfull[2], tempty[2], afull, adone;
  __shared__ uint32_t tmem_slot;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  // small K: the user tile stays resident (loaded once per work unit) and the ring holds item chunks only
  const bool a_res = a.nkc <= SF_STAGES;
  unsigned char* Ares = sf_smem;
  unsigned char* ring = a_res ? sf_smem + (size_t)SF_STAGES * SF_ABYTES : sf_smem;
  const int stage_bytes = a_res ? SF_BBYTES : SF_ABYTES + SF_BBYTES;
  if (warp == 1) umma::tmem_alloc(&tmem_slot, 2 * SF_N);
  if (t == 0) {
    for (int i = 0; i < SF_STAGES; ++i) { umma::mbar_init(&full[i], 1); umma::mbar_init(&empty[i], 1); }
    for (int i = 0; i < 2; ++i) { umma::mbar_init(&tfull[i], 1); umma::mbar_init(&tempty[i], SF_EPI_WARPS); }
    umma::mbar_init(&afull, 1);
    umma::mbar_init(&adone, 1);
  }
  umma::fence_before_sync();
  __syncthreads();
  umma::fence_after_sync();
  const uint32_t tmem = tmem_slot;
  bool failed = false;

  if (warp == 0) {
    // ================================================================== producer
    if (lane == 0) {
      uint32_t it = 0;          // ring position counter
      uint32_t units_done = 0;
      for (long unit = blockIdx.x; unit < a.nunits && !failed; unit += gridDim.x, ++units_done) {
        const long ut = unit / a.nsplit;
        const int sp = (int)(unit - ut * a.nsplit);
        const long jb = (long)sp * a.items_per_split;
        const long je = jb + a.items_per_split < a.V ? jb + a.items_per_split : a.V;
        const unsigned char* asrc = a.apre + (size_t)ut * a.nkc * SF_ABYTES;
        if (a_res) {
          if (units_done > 0 && !umma::mbar_wait(&adone, (units_done - 1) & 1)) { failed = true; break; }
          umma::mbar_arrive_expect_tx(&afull, (uint32_t)(a.nkc * SF_ABYTES));
          for (int kc = 0; kc < a.nkc; ++kc) umma::bulk_g2s(Ares + (size_t)kc * SF_ABYTES, asrc + (size_t)kc * SF_ABYTES,
                                                            SF_ABYTES, &afull);
        }
        for (long j0 = jb; j0 < je && !failed; j0 += SF_N) {
          const unsigned char* bsrc = a.bpre + (size_t)(j0 / SF_N) * a.nkc * SF_BBYTES;
          for (int kc = 0; kc < a.nkc; ++kc, ++it) {
            const int s = it % SF_STAGES;
            const uint32_t round = it / SF_STAGES;
            if (!umma::mbar_wait(&empty[s], (round & 1) ^ 1)) { failed = true; break; }
            unsigned char* dst = ring + (size_t)s * stage_bytes;
            if (a_res) {
              umma::mbar_arrive_expect_tx(&full[s], SF_BBYTES);
              umma::bulk_g2s(dst, bsrc + (size_t)kc * SF_BBYTES, SF_BBYTES, &full[s]);
            } else {
              umma::mbar_arrive_expect_tx(&full[s], SF_ABYTES + SF_BBYTES);
              umma::bulk_g2s(dst, asrc + (size_t)kc * SF_ABYTES, SF_ABYTES, &full[s]);
              umma::bulk_g2s(dst + SF_ABYTES, bsrc + (size_t)kc * SF_BBYTES, SF_BBYTES, &full[s]);
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================================================================== MMA issuer
    if (lane == 0) {
      const uint32_t idesc = umma::idesc_tf32(SF_M, SF_N);
      // descriptors are built once; inside the loops a k-step costs four 64-bit adds and three MMAs (the issuing
      // thread is latency-bound on its own instruction stream)
      uint64_t dA[SF_STAGES], dB[SF_STAGES];
#pragma unroll
      for (int s = 0; s < SF_STAGES; ++s) {
        const unsigned char* st = ring + (size_t)s * stage_bytes;
        dA[s] = umma::smem_desc(umma::smem_u32(a_res ? Ares + (size_t)s * SF_ABYTES : st), SF_A_PITCH, 128);
        dB[s] = umma::smem_desc(umma::smem_u32(a_res ? st : st + SF_ABYTES), SF_B_PITCH, 128);
      }
      uint32_t it = 0, tile_no = 0, units_done = 0;
      for (long unit = blockIdx.x; unit < a.nunits && !failed; unit += gridDim.x, ++units_done) {
        const long ut = unit / a.nsplit;
        const int sp = (int)(unit - ut * a.nsplit);
        const long jb = (long)sp * a.items_per_split;
        const long je = jb + a.items_per_split < a.V ? jb + a.items_per_split : a.V;
        if (a_res && !umma::mbar_wait(&afull, units_done & 1)) { failed = true; break; }
        for (long j0 = jb; j0 < je && !failed; j0 += SF_N, ++tile_no) {
          const uint32_t acc = tile_no & 1;
          if (!umma::mbar_wait(&tempty[acc], ((tile_no >> 1) & 1) ^ 1)) { failed = true; break; }
          umma::fence_after_sync();
          const uint32_t dcol = tmem + acc * SF_N;
          for (int kc = 0; kc < a.nkc; ++kc, ++it) {
            const int s = it % SF_STAGES;
            if (!umma::mbar_wait(&full[s], (it / SF_STAGES) & 1)) { failed = true; break; }
            umma::fence_after_sync();
            // resident user tile: chunk kc lives in slot kc (nkc <= SF_STAGES); streamed: in the ring stage
            const uint64_t dah = a_res ? (kc == 0 ? dA[0] : dA[1]) : (s == 0 ? dA[0] : dA[1]);
            const uint64_t dbh = s == 0 ? dB[0] : dB[1];
            const int kleft = a.kpad - kc * SF_KC;
            const int ksteps = (kleft < SF_KC ? kleft : SF_KC) / 8;
#pragma unroll
            for (int ks = 0; ks < SF_KC / 8; ++ks) {
              if (ks < ksteps) {
                const uint64_t ah = umma::desc_advance(dah, 2 * ks * SF_A_PITCH);
                const uint64_t al = umma::desc_advance(dah, (SF_SLABS + 2 * ks) * SF_A_PITCH);
                const uint64_t bh = umma::desc_advance(dbh, 2 * ks * SF_B_PITCH);
                const uint64_t bl = umma::desc_advance(dbh, (SF_SLABS + 2 * ks) * SF_B_PITCH);
                umma::mma_tf32(dcol, al, bh, idesc, (kc > 0 || ks > 0) ? 1u : 0u);
                umma::mma_tf32(dcol, ah, bl, idesc, 1u);
                umma::mma_tf32(dcol, ah, bh, idesc, 1u);
              }
            }
            umma::mma_commit(&empty[s]);   // stage s may be refilled once these MMAs have read it
          }
          if (!failed) umma::mma_commit(&tfull[acc]);
        }
        if (a_res && !failed) umma::mma_commit(&adone);
      }
    }
  } else {
    // ================================================================== epilogue (warps 2..9, thread <-> user row)
    const uint32_t q = warp & 3;               // TMEM lane quarter this warp may read
    const int chalf = (warp - 2) >> 2;         // which half of the 256 columns it takes
    uint32_t tile_no = 0;
    for (long unit = blockIdx.x; unit < a.nunits && !failed; unit += gridDim.x) {
      const long ut = unit / a.nsplit;
      const int sp = (int)(unit - ut * a.nsplit);
      const int jb = (int)((long)sp * a.items_per_split);
      const int je = (long)jb + a.items_per_split < a.V ? (int)(jb + a.items_per_split) : a.V;
      const long me = ut * SF_M + q * 32 + lane;
      const bool live = me < a.U;
      const float nu = live ? a.unorm[me] * a.cbound : 0.f;
      Epi epi(a, ep, me, live, sp, chalf, jb, je);
      for (int j0 = jb; j0 < je && !failed; j0 += SF_N, ++tile_no) {
        const uint32_t acc = tile_no & 1;
        const bool ok = umma::mbar_wait(&tfull[acc], (tile_no >> 1) & 1);
        if (!__all_sync(0xffffffffu, ok)) { failed = true; break; }
        umma::fence_after_sync();
        // |s~ - s| <= nu * |e_j| <= d for every item of the tile
        epi.tile(j0, nu * __ldg(a.tnorm + j0 / SF_N));
#pragma unroll 1
        for (int cb = chalf * (SF_N / 2); cb < (chalf + 1) * (SF_N / 2); cb += 32) {
          float v[32];
          umma::tmem_ld32(tmem + ((q * 32u) << 16) + acc * SF_N + (uint32_t)cb, v);
          if (!live) continue;
          epi.chunk(v, j0 + cb);
        }
        umma::fence_before_sync();
        __syncwarp();
        if (lane == 0) umma::mbar_arrive(&tempty[acc]);   // this warp's share of the accumulator is free
      }
      if (live && !failed) epi.finish();
    }
  }
  if (failed) atomicExch(a.err, 1);
  __syncthreads();
  if (warp == 1) umma::tmem_free(tmem, 2 * SF_N);
}

// Everything before the pipeline launch: operand images into `pre` (sf_presplit_bytes), item norms (inorm [V]),
// per-tile norms (tnorm [V/256 + 2]).  The caller fills users / unorm / err and the split (sf_set_split).
static inline int sf_prepare(SfPipe& a, const float* users, long ldu, const float* table, int V, int H, long U,
                             unsigned char* pre, float* inorm, float* tnorm, cudaStream_t st, const char* what) {
  a.users = users; a.ldu = ldu; a.table = table; a.V = V; a.H = H; a.U = U;
  a.kpad = (H + 7) & ~7;
  a.nkc = (int)cdiv(a.kpad, SF_KC);
  a.cbound = sf_cbound(a.kpad);
  CAST_LAUNCH(item_norm_kernel, dim3((unsigned)cdiv(V, 8)), dim3(256), 0, st, table, V, H, inorm);
  size_t a_bytes = 0;
  sf_presplit_bytes(U, V, H, &a_bytes);
  presplit_kernel<SF_M><<<dim3((unsigned)cdiv(U, SF_M), (unsigned)a.nkc), 256, 0, st>>>(users, ldu, U, H, a.nkc, pre);
  presplit_kernel<SF_N><<<dim3((unsigned)cdiv(V, SF_N), (unsigned)a.nkc), 256, 0, st>>>(table, H, V, H, a.nkc,
                                                                                      pre + a_bytes);
  tile_norm_kernel<<<dim3((unsigned)cdiv(cdiv(V, SF_N), 8)), dim3(256), 0, st>>>(inorm, V, SF_N, tnorm);
  a.apre = pre;
  a.bpre = pre + a_bytes;
  a.tnorm = tnorm;
  return check_launch(what);
}

// item range of each work unit: `nsplit` splits of whole tiles (clamped to the tile count)
static inline void sf_set_split(SfPipe& a, long nsplit) {
  const long ntile_items = cdiv(a.V, SF_N);
  if (nsplit > ntile_items) nsplit = ntile_items;
  if (nsplit < 1) nsplit = 1;
  a.items_per_split = cdiv(ntile_items, nsplit) * SF_N;
  a.nsplit = (int)cdiv(a.V, a.items_per_split);
  a.nunits = cdiv(a.U, SF_M) * a.nsplit;
}

template <class Epi>
static inline int sf_launch(const SfPipe& a, const typename Epi::Params& ep, cudaStream_t st, const char* what) {
  static bool configured = false;
  if (!configured) {
    cudaFuncSetAttribute(sf_umma_kernel<Epi>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SF_SMEM);
    configured = true;
  }
  const long grid = a.nunits < 148 ? a.nunits : 148;
  sf_umma_kernel<Epi><<<dim3((unsigned)grid), dim3(SF_THREADS), SF_SMEM, st>>>(a, ep);
  return check_launch(what);
}
#endif  // !CAST_EMU

}  // namespace cast
