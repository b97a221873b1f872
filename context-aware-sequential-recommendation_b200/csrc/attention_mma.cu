// K4 on the tensor cores: causal multi-head attention (modules.py:208-269) forward and backward for head widths
// d <= 64, as register-resident warp tiles of mma.sync m16n8k8 3xTF32 (mma_tf32.cuh).  Same mask semantics as the
// FFMA kernels of attention.cuh (which remain for d > 64 and for the `attention_weights` output):
//
//   S = Q K^T / sqrt(d);  S = where(key masked | k > q, -2^32+1, S);  P = softmax(S) over all T keys;
//   P *= query mask;  P = dropout(P);  O = P V + queries.
//
// Layout: CTA = 8 warps on 64 rows of one (batch element, head); warps w and w + 4 own the same 16 rows and each
// takes one 32-column half of every 64-row chunk of the other operand, streamed through a two-stage cp.async pipeline
// in shared memory (the next chunk is in flight while the current one is multiplied); the two halves' partial results
// are merged through shared memory at the end.  Scores live only in the accumulator fragments: the forward pass keeps a
// running row max / row sum (rescaling O when the max moves), and the C fragment of S is fed straight back as the A
// fragment of P.V by relabelling the contraction index inside each k-step (mma_tf32.cuh), so probabilities never
// touch shared memory.  Row tiles are aligned to the END of the sequence (sequences are left-padded: the ragged tile
// is the cheap, mostly padded first one); the grid is tile-major, heaviest tiles first, so that the block scheduler's
// round-robin fill hands every SM one tile of each weight.
//
// Backward = two deterministic kernels, no float atomics:
//   dQ  per query tile:  S, dP = dO V^T -> dS = P (dP~ - D) / sqrt(d) -> dQ += dS K
//   dKV per key tile:    S^T = K Q^T, dP^T = V dO^T -> dV += P~^T dO, dK += dS^T Q
// with P recomputed from the saved row max / 1/rowsum and D_i = sum_j P_ij dP~_ij = dO_i . (out_i - queries_i)
// (P~ V = out - queries), computed by the dQ kernel's prologue and handed to the dKV kernel through rowD.
#include "attention.cuh"
#include "mma_tf32.cuh"

namespace cast {

constexpr int AM_THREADS = 256;  // 8 warps: 4 row blocks of 16 rows x 2 key (or query) groups
constexpr int AM_T = 64;         // rows per CTA
constexpr int AM_NT = 4;         // n-tiles of 8 rows a warp takes from each staged 64-row chunk (its half)

// first kept key (kmask != 0) and first query (ids != 0; 0 without ids) of the sequence, T when there is none.
// One pass, one barrier: strided scan (a thread's first hit is its minimum), warp minimum by shuffles, one slot per
// warp in s2[64] (first keys | first queries), every thread folds the slots.
constexpr int AM_FIRST_SLOTS = 64;
__device__ __forceinline__ void am_first2(const float* __restrict__ kmask_b, const int* __restrict__ ids_b, int T,
                                          int* s2, int& first_key, int& qstart) {
  int mk = T, mq = ids_b ? T : 0;
  for (int j = threadIdx.x; j < T; j += (int)blockDim.x) {
    const float kv = kmask_b[j];
    const int iv = ids_b ? ids_b[j] : 0;
    if (mk == T && kv != 0.f) mk = j;
    if (ids_b && mq == T && iv != 0) mq = j;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const int ok = __shfl_xor_sync(0xffffffffu, mk, o), oq = __shfl_xor_sync(0xffffffffu, mq, o);
    mk = ok < mk ? ok : mk;
    mq = oq < mq ? oq : mq;
  }
  const int w = threadIdx.x >> 5, nw = ((int)blockDim.x + 31) >> 5;
  if ((threadIdx.x & 31) == 0) {
    s2[w] = mk;
    s2[32 + w] = mq;
  }
  __syncthreads();
  first_key = s2[0];
  qstart = s2[32];
  for (int i = 1; i < nw; ++i) {
    first_key = s2[i] < first_key ? s2[i] : first_key;
    qstart = s2[32 + i] < qstart ? s2[32 + i] : qstart;
  }
}

// asynchronous tile load: dst[r][c] = src[(row0 + r) * ld + c] for 0 <= row0 + r < T and c < d, zero rows outside the
// sequence; columns d.. of dst are left alone (zeroed once by am_zero_pad).  Warp w copies rows w, w+4, ..; lane l the
// 8-byte column pair l (vec2: d even, rows 8-byte aligned), else 4-byte copies.
template <int NROWS, int DS, int NW = 4>
__device__ __forceinline__ void am_load_rows_async(float* __restrict__ dst, const float* __restrict__ src, long ld,
                                                   int row0, int T, int d, bool vec2) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (vec2) {
    if (2 * lane < d) {
      float* o = dst + warp * DS + 2 * lane;
      int row = row0 + warp;
      const float* s = src + (long)row * ld + 2 * lane;
#pragma unroll
      for (int k = 0; k < NROWS / NW; ++k) {
        const bool ok = (unsigned)row < (unsigned)T;
        cp_async<8>(o, ok ? s : src, ok);
        o += NW * DS;
        s += NW * ld;
        row += NW;
      }
    }
  } else {
    for (int r = warp; r < NROWS; r += NW) {
      const int row = row0 + r;
      const bool ok = (unsigned)row < (unsigned)T;
      const float* s = src + (long)(ok ? row : 0) * ld;
      for (int c = lane; c < d; c += 32) cp_async<4>(dst + r * DS + c, s + c, ok);
    }
  }
}

__device__ __forceinline__ bool am_vec2_ok(const void* p, long ld, int d, int hh) {
  return ((d | (int)(ld & 1)) & 1) == 0 && ((reinterpret_cast<uintptr_t>(p) + (uintptr_t)hh * d * 4) & 7) == 0;
}

// zero the columns d..DP-1 of `rows` consecutive tile rows (row stride DS)
template <int DP, int DS>
__device__ __forceinline__ void am_zero_pad(float* __restrict__ buf, int rows, int d) {
  for (int r = threadIdx.x; r < rows; r += (int)blockDim.x)
    for (int c = d; c < DP; ++c) buf[r * DS + c] = 0.f;
}

// acc[nt] (16 x 8 each, nt < NT) += A[16 x 8KS] * B[8NT x 8KS]^T for the n-tiles nt_lo <= nt < nt_hi (warp-uniform).
// The three TF32 passes run across all n-tiles before the next pass, so dependent MMAs are NT instructions apart.
template <int KS, int NT, int DS>
__device__ __forceinline__ void am_rows_x_cols(float (&acc)[NT][4], const float* __restrict__ As,
                                               const float* __restrict__ Bs, int nt_lo, int nt_hi, int lane) {
#pragma unroll
  for (int ks = 0; ks < KS; ++ks) {
    unsigned af[4], ah[4], al[4];
    ldsm_a<DS>(af, As, ks * 8, lane);
    tf32_split_n(af, ah, al);
    unsigned bh[NT][2], bl[NT][2];
#pragma unroll
    for (int np = 0; np < NT / 2; ++np) {
      if (2 * np + 1 >= nt_lo && 2 * np < nt_hi) {
        unsigned bf[4];
        ldsm_b2<DS>(bf, Bs + np * 16 * DS, ks * 8, lane);
        tf32_split(__uint_as_float(bf[0]), bh[2 * np][0], bl[2 * np][0]);
        tf32_split(__uint_as_float(bf[1]), bh[2 * np][1], bl[2 * np][1]);
        tf32_split(__uint_as_float(bf[2]), bh[2 * np + 1][0], bl[2 * np + 1][0]);
        tf32_split(__uint_as_float(bf[3]), bh[2 * np + 1][1], bl[2 * np + 1][1]);
      }
    }
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
      if (nt >= nt_lo && nt < nt_hi) mma_tf32(acc[nt], al, bh[nt][0], bh[nt][1]);
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
      if (nt >= nt_lo && nt < nt_hi) mma_tf32(acc[nt], ah, bl[nt][0], bl[nt][1]);
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
      if (nt >= nt_lo && nt < nt_hi) mma_tf32(acc[nt], ah, bh[nt][0], bh[nt][1]);
  }
}

// out[no] (16 x 8 each, no < NTO) += P[16 x 8NT] * M[8NT x 8NTO], P given as C fragments p[kk] (kk = k-step = n-tile
// of the product that made it), M row-major [k][n] in shared memory; k-steps kk_lo <= kk < kk_hi (warp-uniform)
template <int NTO, int NT, int DS>
__device__ __forceinline__ void am_frag_x_rows(float (&out)[NTO][4], const float (&p)[NT][4],
                                               const float* __restrict__ Ms, int kk_lo, int kk_hi, int g, int tig) {
#pragma unroll
  for (int kk = 0; kk < NT; ++kk) {
    if (kk >= kk_lo && kk < kk_hi) {
      unsigned ah[4], al[4];
      tf32_split(p[kk][0], ah[0], al[0]);  // (row g,   k-slot tig)     <- column 2 tig
      tf32_split(p[kk][2], ah[1], al[1]);  // (row g+8, k-slot tig)
      tf32_split(p[kk][1], ah[2], al[2]);  // (row g,   k-slot tig + 4) <- column 2 tig + 1
      tf32_split(p[kk][3], ah[3], al[3]);  // (row g+8, k-slot tig + 4)
      const float* m0 = Ms + (kk * 8 + 2 * tig) * DS + g;
      unsigned bh[NTO][2], bl[NTO][2];
#pragma unroll
      for (int no = 0; no < NTO; ++no) {
        tf32_split(m0[no * 8], bh[no][0], bl[no][0]);
        tf32_split(m0[DS + no * 8], bh[no][1], bl[no][1]);
      }
#pragma unroll
      for (int no = 0; no < NTO; ++no) mma_tf32(out[no], al, bh[no][0], bh[no][1]);
#pragma unroll
      for (int no = 0; no < NTO; ++no) mma_tf32(out[no], ah, bl[no][0], bl[no][1]);
#pragma unroll
      for (int no = 0; no < NTO; ++no) mma_tf32(out[no], ah, bh[no][0], bh[no][1]);
    }
  }
}

// row tiles / chunks of `width` rows aligned to the end of the sequence: index 0 starts at T - n*width (may be < 0)
__device__ __forceinline__ int am_row0(int T, int n, int idx, int width) { return T - (n - idx) * width; }

// grid = (B*h, ntile): blockIdx.x -> (b, head), blockIdx.y = 0 is the LAST (heaviest) row tile
__device__ __forceinline__ void am_block(const AttnDims& dm, int& b, int& hh, int& ntile, int& tile) {
  b = (int)blockIdx.x / dm.h;
  hh = (int)blockIdx.x - b * dm.h;
  ntile = (int)gridDim.y;
  tile = ntile - 1 - (int)blockIdx.y;
}

// the same for key tiles (dK/dV): blockIdx.y = 0 is the FIRST key tile, the heaviest one -- keys are reached by every
// later query, so the early live key tiles loop over the most query chunks and must be scheduled first
__device__ __forceinline__ void am_block_keys(const AttnDims& dm, int& b, int& hh, int& ntile, int& tile) {
  b = (int)blockIdx.x / dm.h;
  hh = (int)blockIdx.x - b * dm.h;
  ntile = (int)gridDim.y;
  tile = (int)blockIdx.y;
}

// ------------------------------------------------------------------------------------------------ forward
// Warps w and w+4 own the same 16 rows and split every staged chunk of 64 keys in halves (each keeps its own running
// max / sum / O), merged through shared memory at the end -- the critical path of the late (long) row tiles halves.
template <int KS>
__global__ void __launch_bounds__(AM_THREADS, KS <= 7 ? 2 : 1) attn_fwd_mma_kernel(AttnFwdArgs a, AttnDims dm) {
  cast_pdl_wait();
  // every CTA signals at once: the next kernel of the chain (a row kernel: weights, shared-memory set-up, tensor-memory
  // allocation before its own wait) may take the SMs this grid leaves idle in its long tail (DESIGN.md 4c)
  cast_pdl_trigger();
  constexpr int DP = 8 * KS, DS = DP + 4, NTO = KS, NT = AM_NT, TW = 8 * NT, TC = 2 * TW;
  constexpr int NTHR = AM_THREADS, NW = NTHR / 32;
  CAST_DYN_SMEM(float, sm);
  __shared__ int s_first[AM_FIRST_SLOTS];
  float* Qs = sm;                         // [64][DS]
  float* Kst = Qs + AM_T * DS;            // [2][TC][DS]
  float* Vst = Kst + 2 * TC * DS;         // [2][TC][DS]
  float* kms = Vst + 2 * TC * DS;         // [2][TC] key mask of the chunk (0 outside the sequence)
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5, warp = wid & 3, kg = wid >> 2, g = lane >> 2, tig = lane & 3;
  const int T = dm.T, d = dm.d;
  int b, hh, ntile, tile;
  am_block(dm, b, hh, ntile, tile);
  const int q0 = am_row0(T, ntile, tile, AM_T);
  const long rowbase = (long)b * T;
  // the query tile starts moving before the scan for the sequence's first key / first query (one round trip, not two)
  am_load_rows_async<AM_T, DS, NW>(Qs, a.Q + rowbase * a.ldq + hh * d, a.ldq, q0, T, d, am_vec2_ok(a.Q, a.ldq, d, hh));
  int first_key, qstart;
  am_first2(a.kmask + rowbase, a.skip_ids ? a.skip_ids + rowbase : nullptr, T, s_first, first_key, qstart);
  const long sbase = ((long)b * dm.h + hh) * T;
  if (q0 + AM_T <= qstart) {  // every row of this tile is padding: output = residual only (block-uniform exit)
    cp_async_commit();
    cp_async_wait<0>();
    for (int idx = t; idx < AM_T * d; idx += NTHR) {
      const int i = q0 + idx / d, c = idx % d;
      if (i >= 0) {
        const long off = (rowbase + i) * dm.H + hh * d + c;
        a.out[off] = a.resid[off];
      }
    }
    for (int r = t; r < AM_T; r += NTHR) {
      const int i = q0 + r;
      if (i >= 0) {
        if (a.row_max) a.row_max[sbase + i] = 0.f;
        if (a.row_linv) a.row_linv[sbase + i] = 0.f;
      }
    }
    return;
  }
  const int qlo = q0 > qstart ? q0 : qstart;
  const bool uni = qlo < first_key;  // tile holds fully-masked rows: they are uniform over all T keys
  const int kend = uni ? T : q0 + AM_T;
  const int kbeg = uni ? 0 : (first_key / TC) * TC;
  const int nch = (kend - kbeg + TC - 1) / TC;
  const int r0 = q0 + warp * 16;
  const int iA = r0 + g, iB = iA + 8;
  const bool wact = r0 + 16 > qstart;
  const bool wuni = (r0 > qstart ? r0 : qstart) < first_key;
  const int wkend = wuni ? T : r0 + 16;

  const float* Kg = a.K + rowbase * a.ldk + hh * d;
  const float* Vg = a.V + rowbase * a.ldv + hh * d;
  const bool vk = am_vec2_ok(a.K, a.ldk, d, hh), vv = am_vec2_ok(a.V, a.ldv, d, hh);
  auto issue = [&](int j0, int st) {
    am_load_rows_async<TC, DS, NW>(Kst + st * TC * DS, Kg, a.ldk, j0, T, d, vk);
    am_load_rows_async<TC, DS, NW>(Vst + st * TC * DS, Vg, a.ldv, j0, T, d, vv);
    if (t < TC) cp_async<4>(kms + st * TC + t, a.kmask + rowbase + (j0 + t < T ? j0 + t : 0), j0 + t < T);
    cp_async_commit();
  };
  issue(kbeg, 0);   // (the query tile issued above rides in this first group)
  am_zero_pad<DP, DS>(sm, AM_T + 4 * TC, d);

  const Drop dr = make_drop(a.rate, a.seed, a.step, a.site);
  const unsigned long long ibA = ((unsigned long long)((long)hh * dm.B + b) * T + (unsigned long long)(long)iA) * T;
  const unsigned long long ibB = ibA + 8ull * T;
  float mA = -INFINITY, mB = -INFINITY, lA = 0.f, lB = 0.f;
  float o[NTO][4];
#pragma unroll
  for (int no = 0; no < NTO; ++no)
#pragma unroll
    for (int c = 0; c < 4; ++c) o[no][c] = 0.f;

  // the residual tile (queries) rides in the K stage that is free during the last chunk -- the epilogue then reads it
  // from shared memory
  static_assert(TC == AM_T, "a K stage holds the residual tile");
  const float* Rg = a.resid + rowbase * dm.H + hh * d;
  const bool vr = am_vec2_ok(a.resid, dm.H, d, hh);
  const int rst = nch & 1;  // stage not used by the last chunk
  float* resS = Kst + rst * TC * DS;
  for (int ci = 0; ci < nch; ++ci) {
    const int j0s = kbeg + ci * TC, st = ci & 1;
    const int j0 = j0s + kg * TW;  // this warp's part of the staged chunk
    if (ci + 1 < nch) {
      issue(j0s + TC, st ^ 1);
    } else {
      am_load_rows_async<AM_T, DS, NW>(resS, Rg, dm.H, q0, T, d, vr);
      cp_async_commit();
    }
    cp_async_wait<1>();
    __syncthreads();
    if (wact && j0 < wkend) {
      const float* Ks = Kst + (st * TC + kg * TW) * DS;
      const float* Vs = Vst + (st * TC + kg * TW) * DS;
      const float* km_s = kms + st * TC + kg * TW;
      int ntl = (wkend - j0 + 7) >> 3;
      if (ntl > NT) ntl = NT;
      float s[NT][4];
#pragma unroll
      for (int nt = 0; nt < NT; ++nt)
#pragma unroll
        for (int c = 0; c < 4; ++c) s[nt][c] = 0.f;
      am_rows_x_cols<KS, NT, DS>(s, Qs + warp * 16 * DS, Ks, 0, ntl, lane);
      // ---- masks + running max
      float cmA = -INFINITY, cmB = -INFINITY;
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        if (nt < ntl) {
          const int jl = nt * 8 + 2 * tig;
          const float2 km = *reinterpret_cast<const float2*>(km_s + jl);
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const int j = j0 + jl + (c & 1), i = (c < 2) ? iA : iB;
            const bool keep = ((c & 1) ? km.y : km.x) != 0.f && j <= i;
            float v = keep ? s[nt][c] * dm.inv_sqrt_d : CAST_NEG_FILL;
            if (j >= T) v = -INFINITY;
            s[nt][c] = v;
            if (c < 2) cmA = fmaxf(cmA, v); else cmB = fmaxf(cmB, v);
          }
        }
      }
      cmA = quad_max(cmA);
      cmB = quad_max(cmB);
      const float nmA = fmaxf(mA, cmA), nmB = fmaxf(mB, cmB);
      const float alA = __expf(mA - nmA), alB = __expf(mB - nmB);  // first chunk: exp(-inf) = 0
      mA = nmA;
      mB = nmB;
      lA *= alA;
      lB *= alB;
#pragma unroll
      for (int no = 0; no < NTO; ++no) {
        o[no][0] *= alA; o[no][1] *= alA; o[no][2] *= alB; o[no][3] *= alB;
      }
      // ---- exp, row sums (per-thread partials), dropout
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        if (nt < ntl) {
          const int j = j0 + nt * 8 + 2 * tig;
          float dA0, dA1, dB0, dB1;
          drop_mul2(dr, ibA + j, dA0, dA1);
          drop_mul2(dr, ibB + j, dB0, dB1);
          const float e0 = __expf(s[nt][0] - mA), e1 = __expf(s[nt][1] - mA);
          const float e2 = __expf(s[nt][2] - mB), e3 = __expf(s[nt][3] - mB);
          lA += e0 + e1;
          lB += e2 + e3;
          s[nt][0] = e0 * dA0; s[nt][1] = e1 * dA1; s[nt][2] = e2 * dB0; s[nt][3] = e3 * dB1;
        }
      }
      am_frag_x_rows<NTO, NT, DS>(o, s, Vs, 0, ntl, g, tig);
    }
    __syncthreads();  // stage st is free for the copy issued two iterations later
  }
  // ---- normalise, query mask, heads merged + residual (outputs += queries)
  cp_async_wait<0>();
  __syncthreads();
  lA = quad_sum(lA);
  lB = quad_sum(lB);
  {  // fold the second key group's (max, sum, O) into the first through the K / V stage the last chunk used
    // (kg - 1 == 0 here and the V-stage arm of rrow below is never taken; written this way they keep the register
    // allocation this kernel was measured with; the plain forms move it by up to 5 registers and 32 instructions)
    float* mo = Kst + ((nch - 1) & 1) * TC * DS;  // [128 threads][4 * NTO]
    float* ml = Vst + ((nch - 1) & 1) * TC * DS;  // [128 threads][4]
    static_assert(128 * 4 * NTO <= TC * DS && 128 * 4 <= TC * DS, "merge space");
    const int slot = warp * 32 + lane;
    if (kg > 0) {
      float* mog = mo + (kg - 1) * 128 * 4 * NTO;
#pragma unroll
      for (int no = 0; no < NTO; ++no)
        *reinterpret_cast<float4*>(mog + (slot * NTO + no) * 4) = make_float4(o[no][0], o[no][1], o[no][2], o[no][3]);
      *reinterpret_cast<float4*>(ml + ((kg - 1) * 128 + slot) * 4) = make_float4(mA, mB, lA, lB);
    }
    __syncthreads();
    if (kg > 0) return;
    const float4 st1 = *reinterpret_cast<const float4*>(ml + slot * 4);
    const float nmA = fmaxf(mA, st1.x), nmB = fmaxf(mB, st1.y);
    // a group that saw no chunk has max = -inf, sum = 0: its factor is exp(-inf) = 0 (nm is finite for live rows)
    const float a0A = nmA == -INFINITY ? 0.f : __expf(mA - nmA), a1A = nmA == -INFINITY ? 0.f : __expf(st1.x - nmA);
    const float a0B = nmB == -INFINITY ? 0.f : __expf(mB - nmB), a1B = nmB == -INFINITY ? 0.f : __expf(st1.y - nmB);
    lA = lA * a0A + st1.z * a1A;
    lB = lB * a0B + st1.w * a1B;
    mA = nmA;
    mB = nmB;
#pragma unroll
    for (int no = 0; no < NTO; ++no) {
      const float4 o1 = *reinterpret_cast<const float4*>(mo + (slot * NTO + no) * 4);
      o[no][0] = o[no][0] * a0A + o1.x * a1A;
      o[no][1] = o[no][1] * a0A + o1.y * a1A;
      o[no][2] = o[no][2] * a0B + o1.z * a1B;
      o[no][3] = o[no][3] * a0B + o1.w * a1B;
    }
  }
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    const int i = half ? iB : iA;
    if (i < 0) continue;
    const int rr = warp * 16 + g + half * 8;
    const float* rrow = (rr < TC ? resS + rr * DS : Vst + rst * TC * DS + (rr - TC) * DS);
    const bool live = wact && i >= qstart;
    const float l = half ? lB : lA, m = half ? mB : mA;
    const float linv = live ? 1.0f / l : 0.f;
    const float f = live ? a.qmask[rowbase + i] * linv : 0.f;
    if (tig == 0) {
      if (a.row_max) a.row_max[sbase + i] = live ? m : 0.f;
      if (a.row_linv) a.row_linv[sbase + i] = linv;
    }
    const long obase = (rowbase + i) * dm.H + hh * d;
    const bool pair_ok = ((dm.H | d) & 1) == 0 && (reinterpret_cast<uintptr_t>(a.out) & 7) == 0;
#pragma unroll
    for (int no = 0; no < NTO; ++no) {
      const int c = no * 8 + 2 * tig;
      if (c >= d) continue;
      const float v0 = o[no][half * 2] * f + rrow[c];
      if (pair_ok) {  // d even => c + 1 < d
        *reinterpret_cast<float2*>(a.out + obase + c) = make_float2(v0, o[no][half * 2 + 1] * f + rrow[c + 1]);
      } else {
        a.out[obase + c] = v0;
        if (c + 1 < d) a.out[obase + c + 1] = o[no][half * 2 + 1] * f + rrow[c + 1];
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ backward: dQ
struct AttnBwdMmaArgs {
  AttnBwdArgs b;
  const float* out;    // forward output (P~ V + queries) [B*T, H]
  const float* resid;  // queries = LN(x) [B*T, H]
  float* pbuf;         // optional [h*B, T, T]: P~ (dropped, query-masked probabilities) written by the dQ kernel
  float* dbuf;         // optional [h*B, T, T]: dS, so that the dK/dV kernel is two products and no recomputation
};

// ST: also store P~ and dS of every computed score to aa.pbuf / aa.dbuf (then fully-masked "uniform" rows, whose P~
// reaches all T keys, are walked over the whole key range like in the forward pass)
template <int KS, bool ST>
__global__ void __launch_bounds__(AM_THREADS, KS <= 7 ? 2 : 1) attn_bwd_dq_mma_kernel(AttnBwdMmaArgs aa, AttnDims dm) {
  constexpr int DP = 8 * KS, DS = DP + 4, NTO = KS, NT = AM_NT, TW = 8 * NT, TC = 2 * TW;
  constexpr int NTHR = AM_THREADS, NW = NTHR / 32;
  const AttnBwdArgs& a = aa.b;
  CAST_DYN_SMEM(float, sm);
  __shared__ int s_first[AM_FIRST_SLOTS];
  float* Qs = sm;                   // [64][DS]
  float* dOs = Qs + AM_T * DS;      // [64][DS]
  float* Kst = dOs + AM_T * DS;     // [2][TC][DS]
  float* Vst = Kst + 2 * TC * DS;   // [2][TC][DS]
  float* kms = Vst + 2 * TC * DS;   // [2][TC]
  float* Dsm = kms + 2 * TC;        // [64] D_i of the tile's rows
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5, warp = wid & 3, kg = wid >> 2, g = lane >> 2, tig = lane & 3;
  const int T = dm.T, d = dm.d;
  int b, hh, ntile, tile;
  am_block(dm, b, hh, ntile, tile);
  const int q0 = am_row0(T, ntile, tile, AM_T);
  const long rowbase = (long)b * T;
  const long sbase = ((long)b * dm.h + hh) * T;
  // The tile's own rows (Q, dO and, for D_i, out and queries — parked in the second K/V stage, which the chunk loop
  // does not touch before its first iteration) start moving before anything is known about the sequence: the scan for
  // its first key / first query below then costs no extra round trip.
  // Of this kernel's inputs only dO is produced by the kernel before it in the chain (the FFN backward kernel): the
  // query tile, out / queries, the sequence scan and the first K/V chunk are requested before the wait on that kernel.
  am_load_rows_async<AM_T, DS, NW>(Qs, a.Q + rowbase * a.ldq + hh * d, a.ldq, q0, T, d, am_vec2_ok(a.Q, a.ldq, d, hh));
  static_assert(TC == AM_T, "a K/V stage holds a whole row tile");
  float* outS = Kst + TC * DS;
  float* resS = Vst + TC * DS;
  am_load_rows_async<AM_T, DS, NW>(outS, aa.out + rowbase * dm.H + hh * d, dm.H, q0, T, d,
                                   am_vec2_ok(aa.out, dm.H, d, hh));
  am_load_rows_async<AM_T, DS, NW>(resS, aa.resid + rowbase * dm.H + hh * d, dm.H, q0, T, d,
                                   am_vec2_ok(aa.resid, dm.H, d, hh));
  cp_async_commit();
  int first_key, qstart;
  am_first2(a.kmask + rowbase, a.skip_ids ? a.skip_ids + rowbase : nullptr, T, s_first, first_key, qstart);
  if (q0 + AM_T <= qstart) {  // padding-only tile: zero gradient
    cp_async_wait<0>();
    cast_pdl_wait();
    for (int idx = t; idx < AM_T * d; idx += NTHR) {
      const int i = q0 + idx / d, c = idx % d;
      if (i >= 0) a.dQ[(rowbase + i) * a.lddq + hh * d + c] = 0.f;
    }
    for (int r = t; r < AM_T; r += NTHR)
      if (q0 + r >= 0) a.rowD[sbase + q0 + r] = 0.f;
    return;
  }
  // only kept keys (first_key <= j <= i) carry dS; fully-masked (uniform) rows have dS == 0
  const int qlo = q0 > qstart ? q0 : qstart;
  const bool uni = ST && qlo < first_key;
  const int kend = uni ? T : q0 + AM_T;
  const int kbeg = uni ? 0 : (first_key / TC) * TC;
  const int nch = kend > kbeg ? (kend - kbeg + TC - 1) / TC : 0;
  const int r0 = q0 + warp * 16;
  const int iA = r0 + g, iB = iA + 8;
  const int rlive = qstart > first_key ? qstart : first_key;  // rows below have zero dQ
  const bool wuni = ST && (r0 > qstart ? r0 : qstart) < first_key;
  const bool wact = ST ? (r0 + 16 > qstart) : (r0 + 16 > rlive);
  const int wkend = wuni ? T : r0 + 16;

  const float* Kg = a.K + rowbase * a.ldk + hh * d;
  const float* Vg = a.V + rowbase * a.ldv + hh * d;
  const bool vk = am_vec2_ok(a.K, a.ldk, d, hh), vv = am_vec2_ok(a.V, a.ldv, d, hh);
  auto issue = [&](int j0, int st) {
    am_load_rows_async<TC, DS, NW>(Kst + st * TC * DS, Kg, a.ldk, j0, T, d, vk);
    am_load_rows_async<TC, DS, NW>(Vst + st * TC * DS, Vg, a.ldv, j0, T, d, vv);
    if (t < TC) cp_async<4>(kms + st * TC + t, a.kmask + rowbase + (j0 + t < T ? j0 + t : 0), j0 + t < T);
    cp_async_commit();
  };
  if (nch > 0) issue(kbeg, 0); else cp_async_commit();
  am_zero_pad<DP, DS>(sm, 2 * AM_T + 4 * TC, d);
  cast_pdl_wait();
  // every CTA signals at once (after its own wait, so that whatever precedes the previous kernel is complete when a
  // dependent starts): the dK/dV kernel may take the SMs this grid leaves idle in its long tail (DESIGN.md 4c)
  cast_pdl_trigger();
  am_load_rows_async<AM_T, DS, NW>(dOs, a.dO + rowbase * dm.H + hh * d, dm.H, q0, T, d, am_vec2_ok(a.dO, dm.H, d, hh));
  cp_async_commit();
  cp_async_wait<0>();   // the tile's rows and the first chunk have landed
  __syncthreads();
  // D_i = dO_i . (out_i - queries_i) over this head's columns, from the staged rows: one warp per row
  {
    constexpr int RW = AM_T / NW;
#pragma unroll
    for (int k = 0; k < RW; ++k) {
      const int r = wid + k * NW, i = q0 + r;
      float acc = 0.f;
      if (i >= qstart && i >= 0) {
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int c = lane + 32 * u;
          if (c >= d) continue;
          acc = fmaf(dOs[r * DS + c], outS[r * DS + c] - resS[r * DS + c], acc);
        }
      }
      const float v = warp_sum(acc);
      if (lane == 0) {
        Dsm[r] = v;
        if (i >= 0) a.rowD[sbase + i] = v;
      }
    }
  }
  __syncthreads();      // Dsm is complete; the parked tiles may be overwritten by the second chunk
  const Drop dr = make_drop(a.rate, a.seed, a.step, a.site);
  const unsigned long long ibA = ((unsigned long long)((long)hh * dm.B + b) * T + (unsigned long long)(long)iA) * T;
  const unsigned long long ibB = ibA + 8ull * T;
  const bool okA = iA >= (ST ? qstart : rlive), okB = iB >= (ST ? qstart : rlive);  // (qstart, rlive >= 0)
  const float mxA = okA ? a.row_max[sbase + iA] : 0.f, mxB = okB ? a.row_max[sbase + iB] : 0.f;
  const float liA = okA ? a.row_linv[sbase + iA] : 0.f, liB = okB ? a.row_linv[sbase + iB] : 0.f;
  const float qmA = okA ? a.qmask[rowbase + iA] : 0.f, qmB = okB ? a.qmask[rowbase + iB] : 0.f;
  float o[NTO][4];
#pragma unroll
  for (int no = 0; no < NTO; ++no)
#pragma unroll
    for (int c = 0; c < 4; ++c) o[no][c] = 0.f;

  for (int ci = 0; ci < nch; ++ci) {
    const int j0s = kbeg + ci * TC, st = ci & 1;
    const int j0 = j0s + kg * TW;  // this warp's half of the staged chunk
    if (ci + 1 < nch) {
      issue(j0s + TC, st ^ 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    if (wact && j0 < wkend) {
      const float* Ks = Kst + (st * TC + kg * TW) * DS;
      const float* Vs = Vst + (st * TC + kg * TW) * DS;
      const float* km_s = kms + st * TC + kg * TW;
      int ntl = (wkend - j0 + 7) >> 3;
      if (ntl > NT) ntl = NT;
      float s[NT][4], dp[NT][4];
#pragma unroll
      for (int nt = 0; nt < NT; ++nt)
#pragma unroll
        for (int c = 0; c < 4; ++c) s[nt][c] = dp[nt][c] = 0.f;
      am_rows_x_cols<KS, NT, DS>(s, Qs + warp * 16 * DS, Ks, 0, ntl, lane);
      am_rows_x_cols<KS, NT, DS>(dp, dOs + warp * 16 * DS, Vs, 0, ntl, lane);
      const float DA = Dsm[warp * 16 + g], DB = Dsm[warp * 16 + g + 8];
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        if (nt < ntl) {
          const int jl = nt * 8 + 2 * tig;
          const float2 km = *reinterpret_cast<const float2*>(km_s + jl);
          float dm0[4];
          drop_mul2(dr, ibA + j0 + jl, dm0[0], dm0[1]);
          drop_mul2(dr, ibB + j0 + jl, dm0[2], dm0[3]);
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const int j = j0 + jl + (c & 1), i = (c < 2) ? iA : iB;
            const bool keep = ((c & 1) ? km.y : km.x) != 0.f && j <= i && i >= rlive;
            const float mx = (c < 2) ? mxA : mxB, li = (c < 2) ? liA : liB, qm = (c < 2) ? qmA : qmB;
            const float D = (c < 2) ? DA : DB;
            const float mul = qm * dm0[c];
            const float dpt = dp[nt][c] * mul;
            if (ST) {
              const bool okr = (c < 2) ? okA : okB;
              const float sv = keep ? s[nt][c] * dm.inv_sqrt_d : CAST_NEG_FILL;
              const float p = okr ? __expf(sv - mx) * li : 0.f;  // uniform rows: exp(fill - fill) / T
              dp[nt][c] = p * mul;                                  // P~
              s[nt][c] = keep ? p * (dpt - D) * dm.inv_sqrt_d : 0.f;
            } else {
              const float p = __expf(s[nt][c] * dm.inv_sqrt_d - mx) * li;
              s[nt][c] = keep ? p * (dpt - D) * dm.inv_sqrt_d : 0.f;
            }
          }
          if (ST) {
            const int j = j0 + jl;
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {
              if (!(hf ? okB : okA) || j >= T) continue;
              const unsigned long long e = (hf ? ibB : ibA) + (unsigned long long)j;
              if (((T | j) & 1) == 0) {
                *reinterpret_cast<float2*>(aa.pbuf + e) = make_float2(dp[nt][2 * hf], dp[nt][2 * hf + 1]);
                *reinterpret_cast<float2*>(aa.dbuf + e) = make_float2(s[nt][2 * hf], s[nt][2 * hf + 1]);
              } else {
                aa.pbuf[e] = dp[nt][2 * hf];
                aa.dbuf[e] = s[nt][2 * hf];
                if (j + 1 < T) {
                  aa.pbuf[e + 1] = dp[nt][2 * hf + 1];
                  aa.dbuf[e + 1] = s[nt][2 * hf + 1];
                }
              }
            }
          }
        }
      }
      am_frag_x_rows<NTO, NT, DS>(o, s, Ks, 0, ntl, g, tig);
    }
    __syncthreads();
  }
  cp_async_wait<0>();
  {  // dQ = sum of the two key groups' partial products
    __syncthreads();
    float* mo = Kst;  // [128 threads][4 * NTO] (both K stages are free now)
    static_assert(128 * 4 * NTO <= 2 * TC * DS, "merge space");
    const int slot = warp * 32 + lane;
    if (kg > 0) {
#pragma unroll
      for (int no = 0; no < NTO; ++no)
        *reinterpret_cast<float4*>(mo + (slot * NTO + no) * 4) = make_float4(o[no][0], o[no][1], o[no][2], o[no][3]);
    }
    __syncthreads();
    if (kg > 0) return;
#pragma unroll
    for (int no = 0; no < NTO; ++no) {
      const float4 o1 = *reinterpret_cast<const float4*>(mo + (slot * NTO + no) * 4);
      o[no][0] += o1.x; o[no][1] += o1.y; o[no][2] += o1.z; o[no][3] += o1.w;
    }
  }
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    const int i = half ? iB : iA;
    if (i < 0) continue;
    const bool live = wact && i >= rlive;
    const long obase = (rowbase + i) * a.lddq + hh * d;
    const bool pair_ok = (((int)(a.lddq & 1) | d) & 1) == 0 && (reinterpret_cast<uintptr_t>(a.dQ) & 7) == 0;
#pragma unroll
    for (int no = 0; no < NTO; ++no) {
      const int c = no * 8 + 2 * tig;
      if (c >= d) continue;
      const float v0 = live ? o[no][half * 2] : 0.f, v1 = live ? o[no][half * 2 + 1] : 0.f;
      if (pair_ok) {
        *reinterpret_cast<float2*>(a.dQ + obase + c) = make_float2(v0, v1);
      } else {
        a.dQ[obase + c] = v0;
        if (c + 1 < d) a.dQ[obase + c + 1] = v1;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ backward: dK, dV
template <int KS>
__global__ void __launch_bounds__(AM_THREADS, KS <= 7 ? 2 : 1) attn_bwd_dkv_mma_kernel(AttnBwdMmaArgs aa, AttnDims dm) {
  cast_pdl_wait();
  constexpr int DP = 8 * KS, DS = DP + 4, NTO = KS, NT = AM_NT, TW = 8 * NT, TC = 2 * TW;
  constexpr int NTHR = AM_THREADS, NW = NTHR / 32;
  const AttnBwdArgs& a = aa.b;
  CAST_DYN_SMEM(float, sm);
  __shared__ int s_first[AM_FIRST_SLOTS];
  float* Ks = sm;                    // [64][DS]
  float* Vs = Ks + AM_T * DS;        // [64][DS]
  float* Qst = Vs + AM_T * DS;       // [2][TC][DS]
  float* dOst = Qst + 2 * TC * DS;   // [2][TC][DS]
  float* stat = dOst + 2 * TC * DS;  // [2][4][TC]: row max, 1/rowsum, D, query mask of the chunk's queries
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5, warp = wid & 3, kg = wid >> 2, g = lane >> 2, tig = lane & 3;
  const int T = dm.T, d = dm.d;
  int b, hh, ntile, tile;
  am_block_keys(dm, b, hh, ntile, tile);
  const int k0 = am_row0(T, ntile, tile, AM_T);
  const long rowbase = (long)b * T;
  const long sbase = ((long)b * dm.h + hh) * T;
  int first_key, qstart;
  am_first2(a.kmask + rowbase, a.skip_ids ? a.skip_ids + rowbase : nullptr, T, s_first, first_key, qstart);
  const bool has_uniform = qstart < first_key;  // some computed (non-padding) row is fully masked
  if (k0 + AM_T <= first_key && !has_uniform) {
    // every key of this tile is masked and no row is uniform: P == 0 on the whole tile => zero gradients
    for (int idx = t; idx < AM_T * d; idx += NTHR) {
      const int j = k0 + idx / d, c = idx % d;
      if (j >= 0) {
        a.dK[(rowbase + j) * a.lddk + hh * d + c] = 0.f;
        a.dV[(rowbase + j) * a.lddv + hh * d + c] = 0.f;
      }
    }
    return;
  }
  const Drop dr = make_drop(a.rate, a.seed, a.step, a.site);
  // query chunks (TC rows, aligned to the end of the sequence) this key tile needs: those that hold queries >= k0, and
  // those that hold uniform rows (which reach every key)
  const int nchunk = (T + TC - 1) / TC;
  auto needed = [&](int cc) {
    const int c0 = am_row0(T, nchunk, cc, TC);
    if (c0 + TC <= qstart) return false;                       // padding rows only
    const bool cuni = has_uniform && c0 < first_key;
    return cuni || c0 + TC > k0;
  };
  const float* Qg = a.Q + rowbase * a.ldq + hh * d;
  const float* dOg = a.dO + rowbase * dm.H + hh * d;
  const bool vq = am_vec2_ok(a.Q, a.ldq, d, hh), vo = am_vec2_ok(a.dO, dm.H, d, hh);
  auto issue = [&](int cc, int st) {
    const int c0 = am_row0(T, nchunk, cc, TC);
    am_load_rows_async<TC, DS, NW>(Qst + st * TC * DS, Qg, a.ldq, c0, T, d, vq);
    am_load_rows_async<TC, DS, NW>(dOst + st * TC * DS, dOg, dm.H, c0, T, d, vo);
    if (t < TC) {
      const int i = c0 + t;
      const bool ok = i >= qstart && i >= 0;
      const long si = sbase + (ok ? i : 0), ri = rowbase + (ok ? i : 0);
      float* sp = stat + st * 4 * TC + t;
      cp_async<4>(sp, a.row_max + si, ok);
      cp_async<4>(sp + TC, a.row_linv + si, ok);
      cp_async<4>(sp + 2 * TC, a.rowD + si, ok);
      cp_async<4>(sp + 3 * TC, a.qmask + ri, ok);
    }
    cp_async_commit();
  };
  auto next_needed = [&](int cc) {
    while (cc < nchunk && !needed(cc)) ++cc;
    return cc;
  };
  am_load_rows_async<AM_T, DS, NW>(Ks, a.K + rowbase * a.ldk + hh * d, a.ldk, k0, T, d, am_vec2_ok(a.K, a.ldk, d, hh));
  am_load_rows_async<AM_T, DS, NW>(Vs, a.V + rowbase * a.ldv + hh * d, a.ldv, k0, T, d, am_vec2_ok(a.V, a.ldv, d, hh));
  int cc = next_needed(0);
  if (cc < nchunk) issue(cc, 0); else cp_async_commit();
  am_zero_pad<DP, DS>(sm, 2 * AM_T + 4 * TC, d);

  const int r0 = k0 + warp * 16;
  const int jA = r0 + g, jB = jA + 8;
  const bool kmA = jA >= 0 && a.kmask[rowbase + jA] != 0.f, kmB = jB >= 0 && a.kmask[rowbase + jB] != 0.f;
  const int qs0 = qstart > 0 ? qstart : 0;
  const unsigned long long hb = (unsigned long long)((long)hh * dm.B + b) * T;
  float gk[NTO][4], gv[NTO][4];
#pragma unroll
  for (int no = 0; no < NTO; ++no)
#pragma unroll
    for (int c = 0; c < 4; ++c) gk[no][c] = gv[no][c] = 0.f;

  for (int it = 0; cc < nchunk; ++it) {
    const int st = it & 1;
    const int c0s = am_row0(T, nchunk, cc, TC);
    const int c0 = c0s + kg * TW;                      // this warp's half of the staged query chunk
    const bool cuni = has_uniform && c0s < first_key;  // chunk holds uniform rows: they reach every key
    const int cn = next_needed(cc + 1);
    if (cn < nchunk) {
      issue(cn, st ^ 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    // queries before the warp's first key see none of its keys unless they are uniform rows
    int nt0 = cuni ? 0 : (r0 - c0) >> 3;
    if (nt0 < 0) nt0 = 0;
    if (r0 + 16 > 0 && nt0 < NT) {
      const float* Qc = Qst + (st * TC + kg * TW) * DS;
      const float* dOc = dOst + (st * TC + kg * TW) * DS;
      const float* sp = stat + st * 4 * TC + kg * TW;
      float s[NT][4], dp[NT][4];
#pragma unroll
      for (int nt = 0; nt < NT; ++nt)
#pragma unroll
        for (int c = 0; c < 4; ++c) s[nt][c] = dp[nt][c] = 0.f;
      am_rows_x_cols<KS, NT, DS>(s, Ks + warp * 16 * DS, Qc, nt0, NT, lane);
      am_rows_x_cols<KS, NT, DS>(dp, Vs + warp * 16 * DS, dOc, nt0, NT, lane);
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        if (nt >= nt0) {
          const int il = nt * 8 + 2 * tig;
          const float2 mx = *reinterpret_cast<const float2*>(sp + il);
          const float2 li = *reinterpret_cast<const float2*>(sp + TC + il);
          const float2 DD = *reinterpret_cast<const float2*>(sp + 2 * TC + il);
          const float2 qm = *reinterpret_cast<const float2*>(sp + 3 * TC + il);
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const int i = c0 + il + (c & 1), j = (c < 2) ? jA : jB;
            const bool keep = ((c < 2) ? kmA : kmB) && j <= i;
            const float sv = keep ? s[nt][c] * dm.inv_sqrt_d : CAST_NEG_FILL;
            // skipped rows (padding / before the sequence) carry nothing: never exp() them (inf * 0)
            const float p = i >= qs0 ? __expf(sv - ((c & 1) ? mx.y : mx.x)) * ((c & 1) ? li.y : li.x) : 0.f;
            const unsigned long long eidx = (hb + (unsigned long long)(long)i) * T + (unsigned long long)(long)j;
            const float mul = ((c & 1) ? qm.y : qm.x) * drop_mul(dr, eidx);
            const float dpt = dp[nt][c] * mul;
            s[nt][c] = p * mul;
            dp[nt][c] = keep ? p * (dpt - ((c & 1) ? DD.y : DD.x)) * dm.inv_sqrt_d : 0.f;
          }
        }
      }
      am_frag_x_rows<NTO, NT, DS>(gv, s, dOc, nt0, NT, g, tig);
      am_frag_x_rows<NTO, NT, DS>(gk, dp, Qc, nt0, NT, g, tig);
    }
    __syncthreads();
    cc = cn;
  }
  cp_async_wait<0>();
  {  // dK, dV = sums of the two query groups' partial products
    __syncthreads();
    float* mk = Qst;   // [128 threads][4 * NTO]
    float* mv = dOst;
    const int slot = warp * 32 + lane;
    if (kg == 1) {
#pragma unroll
      for (int no = 0; no < NTO; ++no) {
        *reinterpret_cast<float4*>(mk + (slot * NTO + no) * 4) = make_float4(gk[no][0], gk[no][1], gk[no][2], gk[no][3]);
        *reinterpret_cast<float4*>(mv + (slot * NTO + no) * 4) = make_float4(gv[no][0], gv[no][1], gv[no][2], gv[no][3]);
      }
    }
    __syncthreads();
    if (kg == 1) return;
#pragma unroll
    for (int no = 0; no < NTO; ++no) {
      const float4 k1 = *reinterpret_cast<const float4*>(mk + (slot * NTO + no) * 4);
      const float4 v1 = *reinterpret_cast<const float4*>(mv + (slot * NTO + no) * 4);
      gk[no][0] += k1.x; gk[no][1] += k1.y; gk[no][2] += k1.z; gk[no][3] += k1.w;
      gv[no][0] += v1.x; gv[no][1] += v1.y; gv[no][2] += v1.z; gv[no][3] += v1.w;
    }
  }
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    const int j = half ? jB : jA;
    if (j < 0) continue;
    const long kb = (rowbase + j) * a.lddk + hh * d, vb = (rowbase + j) * a.lddv + hh * d;
    const bool pair_ok = (((int)((a.lddk | a.lddv) & 1) | d) & 1) == 0 &&
                         ((reinterpret_cast<uintptr_t>(a.dK) | reinterpret_cast<uintptr_t>(a.dV)) & 7) == 0;
#pragma unroll
    for (int no = 0; no < NTO; ++no) {
      const int c = no * 8 + 2 * tig;
      if (c >= d) continue;
      if (pair_ok) {
        *reinterpret_cast<float2*>(a.dK + kb + c) = make_float2(gk[no][half * 2], gk[no][half * 2 + 1]);
        *reinterpret_cast<float2*>(a.dV + vb + c) = make_float2(gv[no][half * 2], gv[no][half * 2 + 1]);
      } else {
        a.dK[kb + c] = gk[no][half * 2];
        a.dV[vb + c] = gv[no][half * 2];
        if (c + 1 < d) {
          a.dK[kb + c + 1] = gk[no][half * 2 + 1];
          a.dV[vb + c + 1] = gv[no][half * 2 + 1];
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ backward: dK, dV from
// the P~ / dS the dQ kernel stored: dV += P~^T dO, dK += dS^T Q, nothing recomputed.  CTA = 64 keys, 8 warps: warp
// (w & 3) owns 16 keys, (w >> 2) one 16-query half of each staged 32-query chunk; A^T fragments come straight from
// the row-major [query][key] tiles (a0 = P~[q0+tig][k0+g]), masked to the entries the dQ kernel actually wrote.
constexpr int AW_TQ = 32, AW_PS = 72, AW_THREADS = 256;

template <int KS>
__global__ void __launch_bounds__(AW_THREADS, 2) attn_bwd_dkv_ws_kernel(AttnBwdMmaArgs aa, AttnDims dm) {
  constexpr int DP = 8 * KS, NTO = KS, TQ = AW_TQ, PS = AW_PS, NW = AW_THREADS / 32;
  const AttnBwdArgs& a = aa.b;
  CAST_DYN_SMEM(float, sm);
  __shared__ int s_first[AM_FIRST_SLOTS];
  float* Pst = sm;                     // [2][TQ][PS]  P~ rows of the chunk's queries, columns = this tile's keys
  float* Dst = Pst + 2 * TQ * PS;      // [2][TQ][PS]  dS
  float* Qst = Dst + 2 * TQ * PS;      // [2][TQ][PS]  Q  (row stride PS: conflict-free [k][n] fragment loads)
  float* dOst = Qst + 2 * TQ * PS;     // [2][TQ][PS]  dO
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5, warp = wid & 3, qg = wid >> 2, g = lane >> 2, tig = lane & 3;
  const int T = dm.T, d = dm.d;
  int b, hh, ntile, tile;
  am_block_keys(dm, b, hh, ntile, tile);
  const int k0 = am_row0(T, ntile, tile, AM_T);
  const long rowbase = (long)b * T;
  int first_key, qstart;
  am_first2(a.kmask + rowbase, a.skip_ids ? a.skip_ids + rowbase : nullptr, T, s_first, first_key, qstart);
  const bool has_uniform = qstart < first_key;
  // Up to here only forward-pass data was read (key mask, ids): the scan ran while the dQ kernel, whose P~ / dS tiles
  // this kernel consumes, may still be draining.  Nothing is written and no dQ-kernel output is read before the wait.
  cast_pdl_wait();
  cast_pdl_trigger();   // (after the wait: whatever precedes the dQ kernel is complete when a dependent starts)
  if (k0 + AM_T <= first_key && !has_uniform) {
    for (int idx = t; idx < AM_T * d; idx += AW_THREADS) {
      const int j = k0 + idx / d, c = idx % d;
      if (j >= 0) {
        a.dK[(rowbase + j) * a.lddk + hh * d + c] = 0.f;
        a.dV[(rowbase + j) * a.lddv + hh * d + c] = 0.f;
      }
    }
    return;
  }
  const int nchunk = (T + TQ - 1) / TQ;
  auto needed = [&](int cc) {
    const int c0 = am_row0(T, nchunk, cc, TQ);
    if (c0 + TQ <= qstart) return false;
    const bool cuni = has_uniform && c0 < first_key;
    return cuni || c0 + TQ > k0;
  };
  auto next_needed = [&](int cc) {
    while (cc < nchunk && !needed(cc)) ++cc;
    return cc;
  };
  const float* Qg = a.Q + rowbase * a.ldq + hh * d;
  const float* dOg = a.dO + rowbase * dm.H + hh * d;
  const bool vq = am_vec2_ok(a.Q, a.ldq, d, hh), vo = am_vec2_ok(a.dO, dm.H, d, hh);
  const unsigned long long hb = (unsigned long long)((long)hh * dm.B + b) * T;
  const bool vp = ((T | k0) & 1) == 0 && (reinterpret_cast<uintptr_t>(aa.pbuf) & 7) == 0 &&
                  (reinterpret_cast<uintptr_t>(aa.dbuf) & 7) == 0;
  auto issue = [&](int cc, int st) {
    const int c0 = am_row0(T, nchunk, cc, TQ);
    am_load_rows_async<TQ, PS, NW>(Qst + st * TQ * PS, Qg, a.ldq, c0, T, d, vq);
    am_load_rows_async<TQ, PS, NW>(dOst + st * TQ * PS, dOg, dm.H, c0, T, d, vo);
    for (int r = wid; r < TQ; r += NW) {
      const int i = c0 + r;
      const bool okr = i >= 0;  // (i < T by construction)
      const unsigned long long e = (hb + (unsigned long long)(okr ? i : 0)) * T;
      float* pd = Pst + (st * TQ + r) * PS;
      float* dd = Dst + (st * TQ + r) * PS;
      if (vp) {
        const int j = k0 + 2 * lane;
        const bool ok = okr && j >= 0 && j < T;
        const unsigned long long ej = e + (unsigned long long)(ok ? j : 0);
        cp_async<8>(pd + 2 * lane, aa.pbuf + ej, ok);
        cp_async<8>(dd + 2 * lane, aa.dbuf + ej, ok);
      } else {
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int j = k0 + lane + 32 * u;
          const bool ok = okr && j >= 0 && j < T;
          const unsigned long long ej = e + (unsigned long long)(ok ? j : 0);
          cp_async<4>(pd + lane + 32 * u, aa.pbuf + ej, ok);
          cp_async<4>(dd + lane + 32 * u, aa.dbuf + ej, ok);
        }
      }
    }
    cp_async_commit();
  };
  int cc = next_needed(0);
  if (cc < nchunk) issue(cc, 0); else cp_async_commit();
  am_zero_pad<DP, PS>(Qst, 4 * TQ, d);

  const int r0 = k0 + warp * 16;
  const int jA = r0 + g, jB = jA + 8;
  const int qs0 = qstart > 0 ? qstart : 0;
  float gk[NTO][4], gv[NTO][4];
#pragma unroll
  for (int no = 0; no < NTO; ++no)
#pragma unroll
    for (int c = 0; c < 4; ++c) gk[no][c] = gv[no][c] = 0.f;
  // entry (i, j) was written by the dQ kernel iff row i is computed and either uniform (all keys) or j is a kept-range key
  auto valid = [&](int i, int j) { return i >= qs0 && j >= 0 && (i < first_key || (j <= i && j >= first_key)); };

  for (int it = 0; cc < nchunk; ++it) {
    const int st = it & 1;
    const int c0 = am_row0(T, nchunk, cc, TQ);
    const bool cuni = has_uniform && c0 < first_key;
    const int cn = next_needed(cc + 1);
    if (cn < nchunk) {
      issue(cn, st ^ 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const int ql0 = qg * 16;  // this warp's 16 queries of the chunk
    if (r0 + 16 > 0 && (cuni || c0 + ql0 + 16 > r0)) {
      const float* Pc = Pst + st * TQ * PS + warp * 16 + g;
      const float* Dc = Dst + st * TQ * PS + warp * 16 + g;
      const float* Qc = Qst + st * TQ * PS + g;
      const float* dOc = dOst + st * TQ * PS + g;
#pragma unroll
      for (int ks = 0; ks < 2; ++ks) {
        const int ql = ql0 + ks * 8 + tig;
        const int i0 = c0 + ql, i1 = i0 + 4;
        const bool v00 = valid(i0, jA), v01 = valid(i0, jB), v10 = valid(i1, jA), v11 = valid(i1, jB);
        unsigned ph[4], pl[4], dh[4], dl[4];
        tf32_split(v00 ? Pc[ql * PS] : 0.f, ph[0], pl[0]);
        tf32_split(v01 ? Pc[ql * PS + 8] : 0.f, ph[1], pl[1]);
        tf32_split(v10 ? Pc[(ql + 4) * PS] : 0.f, ph[2], pl[2]);
        tf32_split(v11 ? Pc[(ql + 4) * PS + 8] : 0.f, ph[3], pl[3]);
        tf32_split(v00 ? Dc[ql * PS] : 0.f, dh[0], dl[0]);
        tf32_split(v01 ? Dc[ql * PS + 8] : 0.f, dh[1], dl[1]);
        tf32_split(v10 ? Dc[(ql + 4) * PS] : 0.f, dh[2], dl[2]);
        tf32_split(v11 ? Dc[(ql + 4) * PS + 8] : 0.f, dh[3], dl[3]);
        {
          unsigned bh[NTO][2], bl[NTO][2];
#pragma unroll
          for (int no = 0; no < NTO; ++no) {
            tf32_split(dOc[ql * PS + no * 8], bh[no][0], bl[no][0]);
            tf32_split(dOc[(ql + 4) * PS + no * 8], bh[no][1], bl[no][1]);
          }
#pragma unroll
          for (int no = 0; no < NTO; ++no) mma_tf32(gv[no], pl, bh[no][0], bh[no][1]);
#pragma unroll
          for (int no = 0; no < NTO; ++no) mma_tf32(gv[no], ph, bl[no][0], bl[no][1]);
#pragma unroll
          for (int no = 0; no < NTO; ++no) mma_tf32(gv[no], ph, bh[no][0], bh[no][1]);
        }
        {
          unsigned bh[NTO][2], bl[NTO][2];
#pragma unroll
          for (int no = 0; no < NTO; ++no) {
            tf32_split(Qc[ql * PS + no * 8], bh[no][0], bl[no][0]);
            tf32_split(Qc[(ql + 4) * PS + no * 8], bh[no][1], bl[no][1]);
          }
#pragma unroll
          for (int no = 0; no < NTO; ++no) mma_tf32(gk[no], dl, bh[no][0], bh[no][1]);
#pragma unroll
          for (int no = 0; no < NTO; ++no) mma_tf32(gk[no], dh, bl[no][0], bl[no][1]);
#pragma unroll
          for (int no = 0; no < NTO; ++no) mma_tf32(gk[no], dh, bh[no][0], bh[no][1]);
        }
      }
    }
    __syncthreads();
    cc = cn;
  }
  cp_async_wait<0>();
  {  // dK, dV = sums of the two query halves
    __syncthreads();
    float* mk = Pst;  // [128 threads][4 * NTO]
    float* mv = Dst;
    const int slot = warp * 32 + lane;
    if (qg == 1) {
#pragma unroll
      for (int no = 0; no < NTO; ++no) {
        *reinterpret_cast<float4*>(mk + (slot * NTO + no) * 4) = make_float4(gk[no][0], gk[no][1], gk[no][2], gk[no][3]);
        *reinterpret_cast<float4*>(mv + (slot * NTO + no) * 4) = make_float4(gv[no][0], gv[no][1], gv[no][2], gv[no][3]);
      }
    }
    __syncthreads();
    if (qg == 1) return;
#pragma unroll
    for (int no = 0; no < NTO; ++no) {
      const float4 k1 = *reinterpret_cast<const float4*>(mk + (slot * NTO + no) * 4);
      const float4 v1 = *reinterpret_cast<const float4*>(mv + (slot * NTO + no) * 4);
      gk[no][0] += k1.x; gk[no][1] += k1.y; gk[no][2] += k1.z; gk[no][3] += k1.w;
      gv[no][0] += v1.x; gv[no][1] += v1.y; gv[no][2] += v1.z; gv[no][3] += v1.w;
    }
  }
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    const int j = half ? jB : jA;
    if (j < 0) continue;
    const long kb = (rowbase + j) * a.lddk + hh * d, vb = (rowbase + j) * a.lddv + hh * d;
    const bool pair_ok = (((int)((a.lddk | a.lddv) & 1) | d) & 1) == 0 &&
                         ((reinterpret_cast<uintptr_t>(a.dK) | reinterpret_cast<uintptr_t>(a.dV)) & 7) == 0;
#pragma unroll
    for (int no = 0; no < NTO; ++no) {
      const int c = no * 8 + 2 * tig;
      if (c >= d) continue;
      if (pair_ok) {
        *reinterpret_cast<float2*>(a.dK + kb + c) = make_float2(gk[no][half * 2], gk[no][half * 2 + 1]);
        *reinterpret_cast<float2*>(a.dV + vb + c) = make_float2(gv[no][half * 2], gv[no][half * 2 + 1]);
      } else {
        a.dK[kb + c] = gk[no][half * 2];
        a.dV[vb + c] = gv[no][half * 2];
        if (c + 1 < d) {
          a.dK[kb + c + 1] = gk[no][half * 2 + 1];
          a.dV[vb + c + 1] = gv[no][half * 2 + 1];
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ dispatch
template <int KS>
static int launch_mma(int which, const AttnFwdArgs* fa, const AttnBwdMmaArgs* ba, const AttnDims& dm,
                      cudaStream_t stream) {
  constexpr int DS = 8 * KS + 4, TC = 2 * 8 * AM_NT;  // TC: rows of a staged chunk (both key groups)
  static size_t cfg[3] = {48 * 1024, 48 * 1024, 48 * 1024};
  const int ntile = (int)cdiv(dm.T, AM_T);
  const dim3 grid((unsigned)(dm.B * dm.h), (unsigned)ntile);
  const size_t row = sizeof(float) * DS;
  if (which == 0) {
    const size_t smem = (AM_T + 4 * TC) * row + sizeof(float) * 2 * TC;
    auto kf = attn_fwd_mma_kernel<KS>;
    if (smem > cfg[0]) {
      cudaFuncSetAttribute(kf, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      cfg[0] = smem;
    }
    CAST_LAUNCH_DEP(kf, grid, dim3(AM_THREADS), smem, stream, *fa, dm);
  } else if (which == 1) {
    const size_t smem = (2 * AM_T + 4 * TC) * row + sizeof(float) * (2 * TC + AM_T);
    if (ba->pbuf) {
      static size_t cfgs = 48 * 1024;
      auto kf = attn_bwd_dq_mma_kernel<KS, true>;
      if (smem > cfgs) {
        cudaFuncSetAttribute(kf, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cfgs = smem;
      }
      CAST_LAUNCH_DEP(kf, grid, dim3(AM_THREADS), smem, stream, *ba, dm);
      return CAST_OK;
    }
    auto kf = attn_bwd_dq_mma_kernel<KS, false>;
    if (smem > cfg[1]) {
      cudaFuncSetAttribute(kf, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      cfg[1] = smem;
    }
    CAST_LAUNCH_DEP(kf, grid, dim3(AM_THREADS), smem, stream, *ba, dm);
  } else {
    if (ba->pbuf) {
      static size_t cfgw = 48 * 1024;
      const size_t smemw = sizeof(float) * 8 * AW_TQ * AW_PS;
      auto kw = attn_bwd_dkv_ws_kernel<KS>;
      if (smemw > cfgw) {
        cudaFuncSetAttribute(kw, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemw);
        cfgw = smemw;
      }
      CAST_LAUNCH_DEP(kw, grid, dim3(AW_THREADS), smemw, stream, *ba, dm);
      return CAST_OK;
    }
    const size_t smem = (2 * AM_T + 4 * TC) * row + sizeof(float) * 8 * TC;
    auto kf = attn_bwd_dkv_mma_kernel<KS>;
    if (smem > cfg[2]) {
      cudaFuncSetAttribute(kf, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      cfg[2] = smem;
    }
    CAST_LAUNCH_DEP(kf, grid, dim3(AM_THREADS), smem, stream, *ba, dm);
  }
  return CAST_OK;
}

bool attn_mma_supported(const AttnDims& dm) { return dm.d >= 1 && dm.d <= 64 && (long)dm.B * dm.h < 2147483647L; }

// which: 0 = forward (fa), 1 = backward dQ, 2 = backward dK/dV (ba + out/resid)
int dispatch_att_mma(int which, const AttnFwdArgs* fa, const AttnBwdArgs* ba, const float* out, const float* resid,
                     float* pbuf, float* dbuf, const AttnDims& dm, cudaStream_t stream) {
  AttnBwdMmaArgs bm{};
  if (ba) { bm.b = *ba; bm.out = out; bm.resid = resid; bm.pbuf = pbuf; bm.dbuf = dbuf; }
  switch ((dm.d + 7) / 8) {
#define CAST_K(K) case K: return launch_mma<K>(which, fa, &bm, dm, stream);
    CAST_K(1) CAST_K(2) CAST_K(3) CAST_K(4) CAST_K(5) CAST_K(6) CAST_K(7) CAST_K(8)
#undef CAST_K
  }
  return set_error(CAST_ERR_UNSUPPORTED, "attention (mma): head width > 64");
}

}  // namespace cast
