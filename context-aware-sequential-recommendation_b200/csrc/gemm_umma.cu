// Dense projections on the 5th-generation tensor cores: the strided GEMM of cast_gemm (tf.layers.dense / conv1d(k=1)
// of modules.py:203-205, :298-306, :333-334 and their gradients) as tcgen05.mma kind::tf32 with the 3xTF32 operand
// split (hi*hi + hi*lo + lo*hi => ~2^-22 relative to sum|a||b|: fp32-grade results, parity tolerance 1e-4 holds).
// Used for the blocks of the wide models (hidden_units > 64: BASELINE configs 4 and 5) and of any width outside the
// row kernels' 8 <= H <= 52; the blocks of configs 1-3 (H = 50) run the row kernels.
//
// Persistent, warp-specialised CTAs (one per SM) over work units = (128-row tile, <=256-column tile, K range):
//   warps 0-3  producers : split the fp32 A chunk (and, for weight gradients, the B chunk) into tf32 hi/lo and store it
//                          in the K-major slab layout of umma.cuh; arrive on full[s]
//   warp  4    B copy    : forward / data-gradient GEMMs read the weight operand from an image pre-split once per call
//                          (presplit_b_kernel) with one cp.async.bulk per chunk (transaction bytes on full[s])
//   warp  5    MMA       : one lane waits full[s], issues 12 tcgen05.mma per 32-element K chunk into one of two TMEM
//                          accumulators, tcgen05.commit -> empty[s]; after the last chunk -> tfull[acc]
//   warps 6-9  epilogue  : tcgen05.ld (thread <-> output row), bias / ReLU / dropout / ReLU-backward mask / residual /
//                          padding-row mask in registers (same order as gemm.cu), 16-byte stores; arrive tempty[acc]
// so staging of chunk k+1, the MMAs of chunk k and the epilogue of the previous unit overlap.
#include "cast_rt.cuh"
#ifndef CAST_EMU
#include "umma.cuh"

namespace cast {

int launch_reduce_partials(const float* partial, int nparts, long count, float* out0, long split, float* out1,
                           cudaStream_t stream);

constexpr int UG_PROD_THREADS = 128;
constexpr int UG_THREADS = 320;
constexpr int UG_M = 128, UG_N = 256;
constexpr int UG_KC = 16;                      // K elements per pipeline stage
constexpr int UG_STAGES = 3;
constexpr int UG_EPI_PITCH = 33;               // floats per row of a warp's 32 x 32 transpose buffer
constexpr int UG_EPI_BYTES = 4 * 32 * UG_EPI_PITCH * 4;
constexpr int UG_A_PITCH = UG_M * 16 + 16, UG_B_PITCH = UG_N * 16 + 16, UG_SLABS = UG_KC / 4;
constexpr int UG_ABYTES = 2 * UG_SLABS * UG_A_PITCH;   // hi slabs then lo slabs
constexpr int UG_BBYTES = 2 * UG_SLABS * UG_B_PITCH;
constexpr size_t UG_SMEM = (size_t)UG_STAGES * (UG_ABYTES + UG_BBYTES) + UG_EPI_BYTES + 128;

struct UGemmEpi {
  const float* bias;
  int relu;
  float drop_rate;
  unsigned long long seed;
  const unsigned long long* step;
  int site;
  const float* act;
  long ld_act;
  float act_scale;
  const float* resid;
  long ldr;
  const int* row_ids;
};

struct UGemmArgs {
  const float* A;
  long sam, sak;
  const float* B;
  long sbk, sbn;
  const unsigned char* bpre;   // pre-split B image [ntile][K chunk][UG_BBYTES] or null (B staged by the producers)
  float* C;
  long ldc;
  long M;
  int N;
  long K, klen;
  int ntile;        // output columns per unit (<= UG_N, multiple of 16)
  int mtiles, ntiles, zs;
  int kchunks;      // ceil(K / UG_KC): chunks per column tile in the image
  UGemmEpi epi;
  float* partials;  // split-K: raw sums [z][M][N]
  int* err;
};

// B[k*sbk + n*sbn] (n < N rows of the operand, k < K) -> image[ntile][kchunk][hi|lo][slab][UG_N rows x 16 B (+pad)]
__global__ void presplit_b_kernel(const float* __restrict__ B, long sbk, long sbn, int N, long K, int ntile,
                                  int kchunks, unsigned char* __restrict__ out) {
  const int nt = blockIdx.x, kc = blockIdx.y;
  unsigned char* dst = out + ((size_t)nt * kchunks + kc) * UG_BBYTES;
  const bool kfast = (sbk == 1);
  for (int idx = threadIdx.x; idx < ntile * UG_SLABS; idx += blockDim.x) {
    int r, c;
    if (kfast) { r = idx / UG_SLABS; c = idx % UG_SLABS; } else { c = idx / ntile; r = idx % ntile; }
    const long n = (long)nt * ntile + r;
    const long k = (long)kc * UG_KC + 4 * c;
    float x[4] = {0.f, 0.f, 0.f, 0.f};
    if (n < N) {
#pragma unroll
      for (int e = 0; e < 4; ++e)
        if (k + e < K) x[e] = __ldg(B + (k + e) * sbk + n * sbn);
    }
    float4 h, l;
    umma::split_tf32(x[0], h.x, l.x);
    umma::split_tf32(x[1], h.y, l.y);
    umma::split_tf32(x[2], h.z, l.z);
    umma::split_tf32(x[3], h.w, l.w);
    *reinterpret_cast<float4*>(dst + (size_t)c * UG_B_PITCH + r * 16) = h;
    *reinterpret_cast<float4*>(dst + (size_t)(UG_SLABS + c) * UG_B_PITCH + r * 16) = l;
  }
}

// Per-thread staging plan of one operand for the 128 producer threads: ITEMS (row, 4-element K slab) pairs whose
// source pointer advances by one K chunk per pipeline step; all index arithmetic happens once per work unit.
// KFAST: the source is contiguous along K; otherwise along the operand's rows (transposed operand).
template <int R_MAX, bool KFAST>
struct StagePlan {
  static constexpr int ITEMS = R_MAX * UG_SLABS / UG_PROD_THREADS;
  const float* ptr[ITEMS];
  int off[ITEMS];        // byte offset of the pair inside the hi slabs (lo slabs follow UG_SLABS pitches later)
  int mode[ITEMS];       // 0 = row beyond the staged tile (nothing stored), 1 = row beyond the operand (zeros), 2 = load
  int kofs[ITEMS];
  long sk;

  __device__ __forceinline__ void init(const float* src, long sr, long sk_, long row0, long rows_total, int R,
                                       long kbeg, int pitch) {
    sk = sk_;
#pragma unroll
    for (int i = 0; i < ITEMS; ++i) {
      const int idx = threadIdx.x + i * UG_PROD_THREADS;
      int r, c;
      if (KFAST) { r = idx / UG_SLABS; c = idx % UG_SLABS; } else { c = idx / R_MAX; r = idx % R_MAX; }
      const long row = row0 + r;
      kofs[i] = 4 * c;
      off[i] = c * pitch + r * 16;
      mode[i] = (r >= R) ? 0 : (row >= rows_total ? 1 : 2);
      ptr[i] = src + (row < rows_total ? row : 0) * sr + (kbeg + 4 * c) * sk;
    }
  }

  // issue the global loads of the next chunk (registers x); the source pointers advance by one chunk
  template <bool VEC4>
  __device__ __forceinline__ void load(float (&x)[ITEMS][4], long kleft) {
    const bool full = kleft >= UG_KC;
#pragma unroll
    for (int i = 0; i < ITEMS; ++i) {
#pragma unroll
      for (int e = 0; e < 4; ++e) x[i][e] = 0.f;
      if (mode[i] == 2) {
        if (full) {
          if (KFAST && VEC4) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(ptr[i]));
            x[i][0] = v.x; x[i][1] = v.y; x[i][2] = v.z; x[i][3] = v.w;
          } else {
#pragma unroll
            for (int e = 0; e < 4; ++e) x[i][e] = __ldg(ptr[i] + e * sk);
          }
        } else if (kleft > 0) {
#pragma unroll
          for (int e = 0; e < 4; ++e)
            if (kofs[i] + e < kleft) x[i][e] = __ldg(ptr[i] + e * sk);
        }
      }
      ptr[i] += UG_KC * sk;
    }
  }

  // split the loaded values into tf32 hi / lo and store them into a pipeline stage
  __device__ __forceinline__ void store(const float (&x)[ITEMS][4], unsigned char* __restrict__ base, int pitch) {
#pragma unroll
    for (int i = 0; i < ITEMS; ++i) {
      if (mode[i] == 0) continue;
      float4 h, l;
      umma::split_tf32(x[i][0], h.x, l.x);
      umma::split_tf32(x[i][1], h.y, l.y);
      umma::split_tf32(x[i][2], h.z, l.z);
      umma::split_tf32(x[i][3], h.w, l.w);
      *reinterpret_cast<float4*>(base + off[i]) = h;
      *reinterpret_cast<float4*>(base + (size_t)UG_SLABS * pitch + off[i]) = l;
    }
  }
};

#ifdef CAST_UMMA_TRACE
__device__ long long g_trace[4][64];
#define UG_TRACE(role, slot) do { if (blockIdx.x == 0 && (slot) < 64) g_trace[role][slot] = clock64(); } while (0)
#else
#define UG_TRACE(role, slot) do { } while (0)
#endif

struct UnitCoord {
  long i0;
  int j0, nN, npad;
  long kbeg, kend;
  int nch, z, nt;
};

__device__ __forceinline__ UnitCoord unit_coord(const UGemmArgs& a, long unit) {
  UnitCoord u;
  const int mt = (int)(unit % a.mtiles);
  const long rest = unit / a.mtiles;
  u.nt = (int)(rest % a.ntiles);
  u.z = (int)(rest / a.ntiles);
  u.i0 = (long)mt * UG_M;
  u.j0 = u.nt * a.ntile;
  u.nN = a.N - u.j0 < a.ntile ? a.N - u.j0 : a.ntile;
  u.npad = (u.nN + 15) & ~15;
  u.kbeg = (long)u.z * a.klen;
  u.kend = u.kbeg + a.klen < a.K ? u.kbeg + a.klen : a.K;
  u.nch = (int)((u.kend - u.kbeg + UG_KC - 1) / UG_KC);
  return u;
}

template <bool A_KFAST, bool B_STAGED, bool B_KFAST, bool VEC4>
__global__ void __launch_bounds__(UG_THREADS, 1) gemm_umma_kernel(UGemmArgs a) {
  extern __shared__ __align__(128) unsigned char ug_smem[];
  __shared__ __align__(8) uint64_t full[UG_STAGES], empty[UG_STAGES], tfull[2], tempty[2];
  __shared__ uint32_t tmem_slot;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  if (warp == 5) umma::tmem_alloc(&tmem_slot, 2 * UG_N);
  if (t == 0) {
    // full[s]: 4 producer warps (+ the bulk-copy thread's expect_tx arrival when B comes from the image)
    for (int i = 0; i < UG_STAGES; ++i) { umma::mbar_init(&full[i], B_STAGED ? 4 : 5); umma::mbar_init(&empty[i], 1); }
    for (int i = 0; i < 2; ++i) { umma::mbar_init(&tfull[i], 1); umma::mbar_init(&tempty[i], 4); }
  }
  umma::fence_before_sync();
  __syncthreads();
  umma::fence_after_sync();
  const uint32_t tmem = tmem_slot;
  const long nunits = (long)a.mtiles * a.ntiles * a.zs;
  bool failed = false;

  if (warp < 4) {
    // ================================================================== producers (128 threads)
    uint32_t it = 0;
    for (long unit = blockIdx.x; unit < nunits && !failed; unit += gridDim.x) {
      const UnitCoord u = unit_coord(a, unit);
      StagePlan<UG_M, A_KFAST> pa;
      pa.init(a.A, a.sam, a.sak, u.i0, a.M, UG_M, u.kbeg, UG_A_PITCH);
      StagePlan<B_STAGED ? UG_N : UG_PROD_THREADS / UG_SLABS, B_KFAST> pb;   // (dummy 16-row plan when unused)
      if (B_STAGED) pb.init(a.B, a.sbn, a.sbk, u.j0, a.N, u.npad, u.kbeg, UG_B_PITCH);
      // software pipeline: the loads of the next PF-1 chunks are in flight while chunk ch is converted and stored
      using PA = StagePlan<UG_M, A_KFAST>;
      using PB = StagePlan<B_STAGED ? UG_N : UG_PROD_THREADS / UG_SLABS, B_KFAST>;
      constexpr int PF = B_STAGED ? 2 : 3;
      float xa[PF][PA::ITEMS][4];
      float xb[PF][PB::ITEMS][4];
#pragma unroll
      for (int h = 0; h < PF - 1; ++h) {
        const long kl = u.kend - (u.kbeg + (long)h * UG_KC);
        pa.template load<VEC4>(xa[h], kl);
        if (B_STAGED) pb.template load<VEC4>(xb[h], kl);
      }
#pragma unroll 1
      for (int ch = 0; ch < u.nch; ch += PF) {
#pragma unroll
        for (int h = 0; h < PF; ++h) {
          const int c = ch + h;
          if (c >= u.nch) break;
          const long knext = u.kend - (u.kbeg + (long)(c + PF - 1) * UG_KC);   // <= 0 past the end: loads nothing
          pa.template load<VEC4>(xa[(h + PF - 1) % PF], knext);
          if (B_STAGED) pb.template load<VEC4>(xb[(h + PF - 1) % PF], knext);
          const int s = it % UG_STAGES;
          const bool ok = umma::mbar_wait(&empty[s], ((it / UG_STAGES) & 1) ^ 1);
          if (!__all_sync(0xffffffffu, ok)) { failed = true; break; }
          if (t == 0) UG_TRACE(0, 2 * (int)it);
          unsigned char* st = ug_smem + (size_t)s * (UG_ABYTES + UG_BBYTES);
          pa.store(xa[h], st, UG_A_PITCH);
          if (B_STAGED) pb.store(xb[h], st + UG_ABYTES, UG_B_PITCH);
          umma::fence_smem_to_async();
          __syncwarp();
          if (lane == 0) umma::mbar_arrive(&full[s]);
          if (t == 0) UG_TRACE(0, 2 * (int)it + 1);
          ++it;
        }
        if (failed) break;
      }
    }
  } else if (warp == 4) {
    // ================================================================== weight-image bulk copies
    if (!B_STAGED && lane == 0) {
      uint32_t it = 0;
      for (long unit = blockIdx.x; unit < nunits && !failed; unit += gridDim.x) {
        const UnitCoord u = unit_coord(a, unit);
        const unsigned char* src = a.bpre + ((size_t)u.nt * a.kchunks + (size_t)(u.kbeg / UG_KC)) * UG_BBYTES;
        for (int ch = 0; ch < u.nch; ++ch, ++it) {
          const int s = it % UG_STAGES;
          if (!umma::mbar_wait(&empty[s], ((it / UG_STAGES) & 1) ^ 1)) { failed = true; break; }
          unsigned char* st = ug_smem + (size_t)s * (UG_ABYTES + UG_BBYTES) + UG_ABYTES;
          umma::mbar_arrive_expect_tx(&full[s], UG_BBYTES);
          umma::bulk_g2s(st, src + (size_t)ch * UG_BBYTES, UG_BBYTES, &full[s]);
        }
      }
    }
  } else if (warp == 5) {
    // ================================================================== MMA issuer
    if (lane == 0) {
      // descriptors of every stage are built once; inside the loops a k-step costs four 64-bit adds and three MMAs
      uint64_t dA[UG_STAGES], dB[UG_STAGES];
#pragma unroll
      for (int s = 0; s < UG_STAGES; ++s) {
        const uint32_t ab = umma::smem_u32(ug_smem + (size_t)s * (UG_ABYTES + UG_BBYTES));
        dA[s] = umma::smem_desc(ab, UG_A_PITCH, 128);
        dB[s] = umma::smem_desc(ab + UG_ABYTES, UG_B_PITCH, 128);
      }
      uint32_t it = 0, un = 0;
      int s = 0;
      uint32_t fph = 0;   // parity to wait for on full[s]: flips every time the ring wraps
      for (long unit = blockIdx.x; unit < nunits && !failed; unit += gridDim.x, ++un) {
        const UnitCoord u = unit_coord(a, unit);
        const uint32_t idesc = umma::idesc_tf32(UG_M, u.npad);
        const uint32_t acc = un & 1;
        if (!umma::mbar_wait(&tempty[acc], ((un >> 1) & 1) ^ 1)) { failed = true; break; }
        umma::fence_after_sync();
        const uint32_t dcol = tmem + acc * UG_N;
        for (int ch = 0; ch < u.nch; ++ch, ++it) {
          if (!umma::mbar_wait(&full[s], fph)) { failed = true; break; }
          UG_TRACE(1, 2 * (int)it);
          umma::fence_after_sync();
          uint64_t dah, dbh;
#pragma unroll
          for (int q = 0; q < UG_STAGES; ++q)
            if (q == s) { dah = dA[q]; dbh = dB[q]; }
#pragma unroll
          for (int ks = 0; ks < UG_KC / 8; ++ks) {  // a short last chunk is zero padded to UG_KC
            const uint64_t ah = umma::desc_advance(dah, 2 * ks * UG_A_PITCH);
            const uint64_t al = umma::desc_advance(dah, (UG_SLABS + 2 * ks) * UG_A_PITCH);
            const uint64_t bh = umma::desc_advance(dbh, 2 * ks * UG_B_PITCH);
            const uint64_t bl = umma::desc_advance(dbh, (UG_SLABS + 2 * ks) * UG_B_PITCH);
            umma::mma_tf32(dcol, al, bh, idesc, (ch == 0 && ks == 0) ? 0u : 1u);
            umma::mma_tf32(dcol, ah, bl, idesc, 1u);
            umma::mma_tf32(dcol, ah, bh, idesc, 1u);
          }
          umma::mma_commit(&empty[s]);
          UG_TRACE(1, 2 * (int)it + 1);
          if (++s == UG_STAGES) { s = 0; fph ^= 1u; }
        }
        if (!failed) umma::mma_commit(&tfull[acc]);
      }
    }
  } else {
    // ================================================================== epilogue (warps 6..9, thread <-> output row)
    const uint32_t q = warp & 3;
    const UGemmEpi& e = a.epi;
    const Drop d = make_drop(e.drop_rate, e.seed, e.step, e.site);
    const bool has_drop = d.thresh != 0u;
    const bool plain = !e.bias && !e.relu && !has_drop && !e.act && !e.resid && !e.row_ids;
    uint32_t un = 0;
    for (long unit = blockIdx.x; unit < nunits && !failed; unit += gridDim.x, ++un) {
      const UnitCoord u = unit_coord(a, unit);
      const uint32_t acc = un & 1;
      const bool ok = umma::mbar_wait(&tfull[acc], (un >> 1) & 1);
      if (!__all_sync(0xffffffffu, ok)) { failed = true; break; }
      if (warp == 6 && lane == 0) UG_TRACE(2, 2 * (int)un);
      umma::fence_after_sync();
      // each warp owns 32 accumulator rows; every 32 x 32 block goes through the warp's shared-memory buffer so that
      // the global side (bias / act / resid reads, C stores) is 128 contiguous bytes per warp instruction
      float* tb = reinterpret_cast<float*>(ug_smem + (size_t)UG_STAGES * (UG_ABYTES + UG_BBYTES)) +
                  (warp - 6) * 32 * UG_EPI_PITCH;
      const long row0 = u.i0 + q * 32;
      const int rows = a.M - row0 < 32 ? (int)(a.M - row0) : 32;   // may be <= 0 for the last tile
#pragma unroll 1
      for (int cb = 0; cb < u.npad; cb += 32) {
        // The epilogue warps are latency-bound on their own instruction stream (one warp per scheduler): the global
        // loads of the whole 32-row block (residual, ReLU-backward mask, row ids) are issued first, so their latency
        // overlaps the TMEM load and the transposition, and the row loop only increments pointers.
        const int cc = cb + lane;          // this lane's column within the unit
        const bool col_ok = cc < u.nN && rows > 0;
        const int gj = u.j0 + cc;
        float rv[32], av[32];
        int myid = 1;
        if (!plain && !a.partials) {
          if (e.row_ids && lane < rows) myid = e.row_ids[row0 + lane];
          if (e.resid && col_ok) {
            const float* rrow = e.resid + row0 * e.ldr + gj;
#pragma unroll
            for (int k = 0; k < 32; ++k) rv[k] = k < rows ? rrow[(long)k * e.ldr] : 0.f;
          }
          if (e.act && col_ok) {
            const float* arow = e.act + row0 * e.ld_act + gj;
#pragma unroll
            for (int k = 0; k < 32; ++k) av[k] = k < rows ? arow[(long)k * e.ld_act] : 1.f;
          }
        }
        float v[32];
        umma::tmem_ld32(tmem + ((q * 32u) << 16) + acc * UG_N + (uint32_t)cb, v);
#pragma unroll
        for (int x = 0; x < 32; ++x) tb[lane * UG_EPI_PITCH + x] = v[x];
        __syncwarp();
        const float* tcol = tb + lane;
        if (a.partials) {
          if (col_ok) {
            float* prow = a.partials + ((long)u.z * a.M + row0) * a.N + gj;
#pragma unroll 8
            for (int rr = 0; rr < rows; ++rr, prow += a.N) *prow = tcol[rr * UG_EPI_PITCH];
          }
        } else if (plain) {
          if (col_ok) {
            float* orow = a.C + row0 * a.ldc + gj;
#pragma unroll 8
            for (int rr = 0; rr < rows; ++rr, orow += a.ldc) *orow = tcol[rr * UG_EPI_PITCH];
          }
        } else {
          const float bj = (e.bias && col_ok) ? __ldg(e.bias + gj) : 0.f;
          float* orow = a.C + row0 * a.ldc + gj;
          unsigned long long didx = (unsigned long long)(row0 * a.N + gj);
#pragma unroll
          for (int k = 0; k < 32; ++k) {
            const int idk = __shfl_sync(0xffffffffu, myid, k);   // all lanes take part
            if (k < rows && col_ok) {
              float c = tcol[k * UG_EPI_PITCH] + bj;
              if (e.relu) c = fmaxf(c, 0.f);
              if (has_drop) c *= drop_mul(d, didx);
              if (e.act) c *= (av[k] > 0.f) ? e.act_scale : 0.f;
              if (e.resid) c += rv[k];
              if (idk == 0) c = 0.f;
              *orow = c;
            }
            orow += a.ldc;
            didx += (unsigned long long)a.N;
          }
        }
        __syncwarp();
      }
      umma::fence_before_sync();
      __syncwarp();
      if (lane == 0) umma::mbar_arrive(&tempty[acc]);
      if (warp == 6 && lane == 0) UG_TRACE(2, 2 * (int)un + 1);
    }
  }
  if (failed) atomicExch(a.err, 1);
  __syncthreads();
  if (warp == 5) umma::tmem_free(tmem, 2 * UG_N);
}

// device-side watchdog flag shared by all tensor-core GEMM launches of the process (0 = ok)
__device__ int g_umma_gemm_err = 0;

template <bool AK, bool BS, bool BK, bool V4>
static void launch_inst(const UGemmArgs& a, int grid, cudaStream_t stream) {
  static bool configured = false;
  if (!configured) {
    cudaFuncSetAttribute(gemm_umma_kernel<AK, BS, BK, V4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)UG_SMEM);
    configured = true;
  }
  gemm_umma_kernel<AK, BS, BK, V4><<<dim3((unsigned)grid), dim3(UG_THREADS), UG_SMEM, stream>>>(a);
}

// bytes of the pre-split weight image for an N x K operand (forward / data-gradient GEMMs)
size_t gemm_umma_image_bytes(int N, long K) {
  return (size_t)cdiv(N, 64) * (size_t)cdiv(K, UG_KC) * UG_BBYTES + 256;
}

int gemm_umma_launch(const float* A, long sam, long sak, const float* B, long sbk, long sbn, float* C, long ldc, long M,
                     int N, long K, const UGemmEpi& epi, int splits, float* partials, void* image, size_t image_bytes,
                     cudaStream_t stream) {
  static int* err_ptr = nullptr;
  if (!err_ptr) cudaGetSymbolAddress(reinterpret_cast<void**>(&err_ptr), g_umma_gemm_err);
  UGemmArgs a;
  a.A = A; a.sam = sam; a.sak = sak; a.B = B; a.sbk = sbk; a.sbn = sbn; a.C = C; a.ldc = ldc; a.M = M; a.N = N;
  a.K = K; a.epi = epi; a.partials = partials; a.err = err_ptr;
  a.mtiles = (int)cdiv(M, UG_M);
  // column tile: 256 wide unless that leaves most of the 148 SMs idle (short M: C4-sized batches)
  int ntile = UG_N;
  if (splits == 1)
    while (ntile > 64 && (long)a.mtiles * cdiv(N, ntile) < 148) ntile /= 2;
  a.ntile = ntile;
  a.ntiles = (int)cdiv(N, ntile);
  if (splits > 1) {  // about two waves of CTAs over the reduction dimension are enough (fewer partials to reduce)
    long want = cdiv(296, (long)a.mtiles * a.ntiles);
    if (want < 1) want = 1;
    if (want < splits) splits = (int)want;
  }
  long klen = cdiv(K, splits);
  klen = cdiv(klen, UG_KC) * UG_KC;
  a.klen = klen;
  a.zs = (int)cdiv(K, klen);
  a.kchunks = (int)cdiv(K, UG_KC);
  const long nunits = (long)a.mtiles * a.ntiles * a.zs;
  const int grid = (int)(nunits < 148 ? nunits : 148);
  const bool ak = (sak == 1), bk = (sbk == 1);
  // the weight operand of forward / data-gradient GEMMs is re-read by every row tile: split it once into an image
  const bool use_image = splits == 1 && image && image_bytes >= gemm_umma_image_bytes(N, K) && a.mtiles >= 2;
  a.bpre = nullptr;
  if (use_image) {
    unsigned char* img = static_cast<unsigned char*>(image);
    img += (256 - (reinterpret_cast<uintptr_t>(img) & 255)) & 255;
    presplit_b_kernel<<<dim3((unsigned)a.ntiles, (unsigned)a.kchunks), 256, 0, stream>>>(B, sbk, sbn, N, K, ntile,
                                                                                        a.kchunks, img);
    a.bpre = img;
  }
  const bool v4 = (!ak || (sam % 4 == 0 && (reinterpret_cast<uintptr_t>(A) & 15) == 0)) &&
                  (use_image || !bk || (sbn % 4 == 0 && (reinterpret_cast<uintptr_t>(B) & 15) == 0));
  if (use_image) {
    if (ak) { if (v4) launch_inst<true, false, false, true>(a, grid, stream); else launch_inst<true, false, false, false>(a, grid, stream); }
    else launch_inst<false, false, false, false>(a, grid, stream);
  } else if (ak && bk) {
    if (v4) launch_inst<true, true, true, true>(a, grid, stream); else launch_inst<true, true, true, false>(a, grid, stream);
  } else if (ak) {
    if (v4) launch_inst<true, true, false, true>(a, grid, stream); else launch_inst<true, true, false, false>(a, grid, stream);
  } else if (bk) {
    if (v4) launch_inst<false, true, true, true>(a, grid, stream); else launch_inst<false, true, true, false>(a, grid, stream);
  } else {
    launch_inst<false, true, false, false>(a, grid, stream);
  }
  int rc = check_launch("gemm(umma)");
  if (rc) return rc;
  if (partials)
    return launch_reduce_partials(partials, a.zs, M * (long)N, C, M * (long)N, (float*)nullptr, stream);
  return CAST_OK;
}

}  // namespace cast

#ifdef CAST_UMMA_TRACE
extern "C" int cast_gemm_trace(long long* host_buf /* [4][64] */) {
  cudaDeviceSynchronize();
  return cudaMemcpyFromSymbol(host_buf, cast::g_trace, sizeof(long long) * 4 * 64) == cudaSuccess ? 0 : -1;
}
#endif

extern "C" int cast_gemm_tensor_status(int* host_flag, void* stream) {
  if (!host_flag) return cast::set_error(CAST_ERR_BAD_ARG, "gemm_tensor_status");
  cudaStreamSynchronize((cudaStream_t)stream);
  if (cudaMemcpyFromSymbol(host_flag, cast::g_umma_gemm_err, sizeof(int)) != cudaSuccess)
    return cast::set_error(CAST_ERR_CUDA, "gemm_tensor_status");
  return CAST_OK;
}
#else
#include <stddef.h>
extern "C" int cast_gemm_tensor_status(int* host_flag, void* stream) {
  (void)stream;
  if (host_flag) *host_flag = 0;
  return 0;
}
#endif
