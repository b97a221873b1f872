// The backward row-tile kernels of fused.cu (included from there, after its helpers and argument structs):
// contractions as mma.sync m16n8k8 3xTF32 (mma_tf32.cuh), tiles streamed through a two-stage cp.async pipeline so the
// next 64-row tile loads while the current one is multiplied.
//
//   CTA = 16 warps (RM_BWD_NG = 4 column groups x 4 row blocks) on one 64-row tile; warp w owns the 16-row block
//   (w & 3) and the 16-column group (w >> 2) of every 64 x H product, and the same block of every H x H weight
//   gradient.
//   Tiles are row-major with stride S = 8*ceil(H/8) + 4 floats (16-byte rows, S/4 odd: ldmatrix conflict-free);
//   weights sit in shared memory in their natural [in][out] layout:
//     dgrad    dX = dY W^T  : B^T[n'][k] = W[n'][k]        -> ldmatrix fragments (contraction along a weight row)
//     wgrad    dW = X^T dY  : A^T and B straight from the two row-major tiles (contraction over the 64 rows)
#pragma once
#include "mma_tf32.cuh"

namespace cast {

// asynchronous copy of the 64-row tile starting at row0 of a row-major [N, H] tensor into dst (stride S); rows >= N
// are zero-filled, columns >= H untouched (zeroed once at kernel start).  Warp w of NW copies rows w, w+NW, ...
template <int S, int NW>
__device__ __forceinline__ void rm_load_tile_async(float* __restrict__ dst, const float* __restrict__ src, long row0,
                                                   long N, int H, bool vec2) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (vec2) {
    if (2 * lane < H) {
      float* o = dst + warp * S + 2 * lane;
      long row = row0 + warp;
      const float* s = src + row * H + 2 * lane;
#pragma unroll
      for (int k = 0; k < FR / NW; ++k) {
        const bool ok = row < N;
        cp_async<8>(o, ok ? s : src, ok);
        o += NW * S;
        s += NW * (long)H;
        row += NW;
      }
    }
  } else {
    for (int r = warp; r < FR; r += NW) {
      const long row = row0 + r;
      const bool ok = row < N;
      const float* s = src + (ok ? row : 0) * H;
      for (int c = lane; c < H; c += 32) cp_async<4>(dst + r * S + c, s + c, ok);
    }
  }
}

__device__ __forceinline__ bool rm_vec2_ok(const void* p, int H) {
  return (H & 1) == 0 && (reinterpret_cast<uintptr_t>(p) & 7) == 0;
}

// zero the padding columns H..HP8-1 of `rows` tile rows
template <int HP8, int S>
__device__ __forceinline__ void rm_zero_pad(float* __restrict__ buf, int rows, int H) {
  for (int r = threadIdx.x; r < rows; r += (int)blockDim.x)
    for (int c = H; c < HP8; ++c) buf[r * S + c] = 0.f;
}

// W[H][H] row-major (global) -> Ws[k][n] stride S through cp.async (joins the caller's next commit group: the weights
// arrive with the first row tile)
template <int S>
__device__ __forceinline__ void rm_load_w_async(float* __restrict__ Ws, const float* __restrict__ W, int H) {
  for (int idx = threadIdx.x; idx < H * H; idx += (int)blockDim.x) {
    const int k = idx / H, n = idx - k * H;
    cp_async<4>(Ws + k * S + n, W + idx, true);
  }
}

// LayerNorm backward over the FR rows of a tile, BT / FR threads per row (8 with 512 threads): thread `sub` of a row
// owns the float4 column groups (j * TPR + sub) * 4, so that a row's threads read 128 contiguous bytes of shared memory
// per request and write dx in row-contiguous pieces; row sums by xor shuffles inside the row's threads.
//   a = G * gamma, xhat = (x - mu) * rs, s1 = mean(a), s2 = mean(a * xhat), dx = rs * (a - s1 - xhat * s2) (+ Add)
// gam: gamma of this thread's columns (loaded once per kernel).  rowstat[r] = {mu, rs, s1, s2} for the column sums.
template <int S, int BT>
struct RmLnRows {
  static constexpr int TPR = BT / FR, NJ = 64 / (4 * TPR);
  static_assert(TPR == 4 || TPR == 8, "row threads");
  float gam[NJ][4];
  __device__ __forceinline__ void load_gamma(const float* __restrict__ gamma, int H) {
    const int sub = threadIdx.x % TPR;
#pragma unroll
    for (int j = 0; j < NJ; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int c = (j * TPR + sub) * 4 + e;
        gam[j][e] = c < H ? gamma[c] : 0.f;
      }
  }
  __device__ __forceinline__ void run(const float* __restrict__ Gs, const float* __restrict__ Xr,
                                      const float* __restrict__ Add, const float* __restrict__ mean,
                                      const float* __restrict__ rstd, float* __restrict__ rowstat, long row0,
                                      const FDims& d, float* __restrict__ dx, const LnOutFx& fx) const {
    const int t = threadIdx.x, r = t / TPR, sub = t % TPR;
    const long row = row0 + r;
    const bool live = row < d.N;
    const float mu = live ? mean[row] : 0.f, rs = live ? rstd[row] : 0.f;
    float av[NJ][4], xh[NJ][4];
    float p1 = 0.f, p2 = 0.f;
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      const int c4 = (j * TPR + sub) * 4;
      if (c4 < 8 * ((S - 4) / 8)) {   // inside the tile's (zero padded) column range
        const float4 gq = *reinterpret_cast<const float4*>(Gs + r * S + c4);
        const float4 xq = *reinterpret_cast<const float4*>(Xr + r * S + c4);
        const float gg[4] = {gq.x, gq.y, gq.z, gq.w}, xx[4] = {xq.x, xq.y, xq.z, xq.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const bool in = c4 + e < d.H;
          av[j][e] = in ? gg[e] * gam[j][e] : 0.f;
          xh[j][e] = in ? (xx[e] - mu) * rs : 0.f;
          p1 += av[j][e];
          p2 += av[j][e] * xh[j][e];
        }
      } else {
#pragma unroll
        for (int e = 0; e < 4; ++e) av[j][e] = xh[j][e] = 0.f;
      }
    }
#pragma unroll
    for (int o = 1; o < TPR; o <<= 1) {
      p1 += __shfl_xor_sync(0xffffffffu, p1, o);
      p2 += __shfl_xor_sync(0xffffffffu, p2, o);
    }
    const float s1 = p1 / (float)d.H, s2 = p2 / (float)d.H;
    if (sub == 0) {
      rowstat[r * 4 + 0] = mu;
      rowstat[r * 4 + 1] = rs;
      rowstat[r * 4 + 2] = s1;
      rowstat[r * 4 + 3] = s2;
    }
    if (!live) return;
    const float fm = (fx.on && fx.ids && fx.ids[row] == 0) ? 0.f : 1.f;
    const bool pair = (d.H & 1) == 0 && (reinterpret_cast<uintptr_t>(dx) & 7) == 0;
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      const int c4 = (j * TPR + sub) * 4;
      if (c4 >= d.H) continue;
      float o[4];
      float ad[4] = {0.f, 0.f, 0.f, 0.f};
      if (Add) {
        const float4 aq = *reinterpret_cast<const float4*>(Add + r * S + c4);
        ad[0] = aq.x; ad[1] = aq.y; ad[2] = aq.z; ad[3] = aq.w;
      }
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        o[e] = rs * (av[j][e] - s1 - xh[j][e] * s2);
        if (Add) o[e] += ad[e];
      }
      if (fx.on) {
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (c4 + e < d.H) o[e] = o[e] * fm * drop_mul(fx.drop, (unsigned long long)(row * d.H + c4 + e));
      }
      float* dst = dx + row * d.H + c4;
      if (pair) {   // H even => c4 + 1 < H whenever c4 < H, and (row * H + c4) * 4 bytes is a multiple of 8
        *reinterpret_cast<float2*>(dst) = make_float2(o[0], o[1]);
        if (c4 + 2 < d.H) *reinterpret_cast<float2*>(dst + 2) = make_float2(o[2], o[3]);
      } else {
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (c4 + e < d.H) dst[e] = o[e];
      }
    }
  }
};

// acc[nt] += A[16 x 8KS] * Bt^T, Bt[n][k] row-major (k contiguous), n-tiles nt < nact (warp-uniform, <= 4)
template <int KS, int S, int NTW = 4>
__device__ __forceinline__ void rm_mm_bt(float (&acc)[NTW][4], const float* __restrict__ As,
                                         const float* __restrict__ Bt, int nact, int lane) {
#pragma unroll
  for (int ks = 0; ks < KS; ++ks) {
    unsigned af[4], ah[4], al[4];
    ldsm_a<S>(af, As, ks * 8, lane);
    tf32_split_n(af, ah, al);
    unsigned bh[NTW][2], bl[NTW][2];
#pragma unroll
    for (int np = 0; np < NTW / 2; ++np) {
      if (2 * np < nact) {
        unsigned bf[4];
        ldsm_b2<S>(bf, Bt + np * 16 * S, ks * 8, lane);
        tf32_split(__uint_as_float(bf[0]), bh[2 * np][0], bl[2 * np][0]);
        tf32_split(__uint_as_float(bf[1]), bh[2 * np][1], bl[2 * np][1]);
        tf32_split(__uint_as_float(bf[2]), bh[2 * np + 1][0], bl[2 * np + 1][0]);
        tf32_split(__uint_as_float(bf[3]), bh[2 * np + 1][1], bl[2 * np + 1][1]);
      }
    }
#pragma unroll
    for (int nt = 0; nt < NTW; ++nt)
      if (nt < nact) mma_tf32(acc[nt], al, bh[nt][0], bh[nt][1]);
#pragma unroll
    for (int nt = 0; nt < NTW; ++nt)
      if (nt < nact) mma_tf32(acc[nt], ah, bl[nt][0], bl[nt][1]);
#pragma unroll
    for (int nt = 0; nt < NTW; ++nt)
      if (nt < nact) mma_tf32(acc[nt], ah, bh[nt][0], bh[nt][1]);
  }
}

// weight gradients: acc_j[nt][.] += sum_{r<64} X[r][m0 + .] * G_j[r][n0 + 8nt + .] for NB gradient tiles sharing X.
// Fragments come straight from the row-major tiles (A^T: a0 = X[r0+tig][m0+g], ...).
template <int NB, int S, int NTW = 4>
__device__ __forceinline__ void rm_wgrad(float (&acc)[NB][NTW][4], const float* __restrict__ X, int m0,
                                         const float* const (&G)[NB], int n0, int nact, int lane) {
  const int g = lane >> 2, tig = lane & 3;
#pragma unroll 2
  for (int r0 = 0; r0 < FR; r0 += 8) {
    const float* xa = X + (r0 + tig) * S + m0 + g;
    unsigned ah[4], al[4];
    tf32_split(xa[0], ah[0], al[0]);
    tf32_split(xa[8], ah[1], al[1]);
    tf32_split(xa[4 * S], ah[2], al[2]);
    tf32_split(xa[4 * S + 8], ah[3], al[3]);
#pragma unroll
    for (int j = 0; j < NB; ++j) {
      const float* gb = G[j] + (r0 + tig) * S + n0 + g;
      unsigned bh[NTW][2], bl[NTW][2];
#pragma unroll
      for (int nt = 0; nt < NTW; ++nt) {
        if (nt < nact) {
          tf32_split(gb[nt * 8], bh[nt][0], bl[nt][0]);
          tf32_split(gb[4 * S + nt * 8], bh[nt][1], bl[nt][1]);
        }
      }
#pragma unroll
      for (int nt = 0; nt < NTW; ++nt)
        if (nt < nact) mma_tf32(acc[j][nt], al, bh[nt][0], bh[nt][1]);
#pragma unroll
      for (int nt = 0; nt < NTW; ++nt)
        if (nt < nact) mma_tf32(acc[j][nt], ah, bl[nt][0], bl[nt][1]);
#pragma unroll
      for (int nt = 0; nt < NTW; ++nt)
        if (nt < nact) mma_tf32(acc[j][nt], ah, bh[nt][0], bh[nt][1]);
    }
  }
}

// Column sums spread over the whole CTA: thread t owns column t & 63 of the row slice t >> 6 (64 / SL rows); partial
// sums stay in the thread's registers across all tiles and are folded over the SL slices, in slice order, once at the
// end of the kernel (rm_fold_cols) -- instead of 64 threads walking all 64 rows of every tile.
template <int SL, int S>
__device__ __forceinline__ float rm_colsum_slice(const float* __restrict__ Ts) {
  const int c = threadIdx.x & 63, sl = threadIdx.x >> 6;
  constexpr int R = FR / SL;
  float s = 0.f;
#pragma unroll
  for (int r = 0; r < R; ++r) s += Ts[(sl * R + r) * S + c];
  return s;
}
// dgamma / dbeta slice sums of the LayerNorm backward: sum_r G[r][c] * xhat[r][c] and sum_r G[r][c]
template <int SL, int S>
__device__ __forceinline__ void rm_ln_cols_slice(const float* __restrict__ Gs, const float* __restrict__ Xr,
                                                 const float* __restrict__ rowstat, float& dgam, float& dbet) {
  const int c = threadIdx.x & 63, sl = threadIdx.x >> 6;
  constexpr int R = FR / SL;
  float sg = 0.f, sb = 0.f;
#pragma unroll
  for (int r0 = 0; r0 < R; ++r0) {
    const int r = sl * R + r0;
    const float gv = Gs[r * S + c];
    sg += gv * ((Xr[r * S + c] - rowstat[r * 4]) * rowstat[r * 4 + 1]);
    sb += gv;
  }
  dgam += sg;
  dbet += sb;
}
// out[c] = sum over the SL slices (fixed order) of the per-thread partials; scratch: [SL][64] floats
template <int SL>
__device__ __forceinline__ void rm_fold_cols(float v, float* __restrict__ scratch, float* __restrict__ out, int H) {
  const int c = threadIdx.x & 63, sl = threadIdx.x >> 6;
  __syncthreads();
  scratch[sl * 64 + c] = v;
  __syncthreads();
  if (sl == 0 && c < H) {
    float s = scratch[c];
#pragma unroll
    for (int k = 1; k < SL; ++k) s += scratch[k * 64 + c];
    out[c] = s;
  }
}

template <int NTW>
__device__ __forceinline__ void rm_zero(float (&acc)[NTW][4]) {
#pragma unroll
  for (int i = 0; i < NTW; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
}

// per-CTA weight-gradient partial from the warp's fragment block: P[k * H + n]
template <int NTW>
__device__ __forceinline__ void rm_store_wpartial(float* __restrict__ P, const float (&acc)[NTW][4], int m0, int n0,
                                                  int nact, int H, int lane) {
  const int g = lane >> 2, tig = lane & 3;
#pragma unroll
  for (int nt = 0; nt < NTW; ++nt) {
    if (nt >= nact) continue;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int k = m0 + g + (e >> 1) * 8, n = n0 + nt * 8 + 2 * tig + (e & 1);
      if (k < H && n < H) P[k * H + n] = acc[nt][e];
    }
  }
}

// ------------------------------------------------------------------------------------------------ qkv backward
// NG column groups per row block: 2 => 8 warps x (16 rows x 32 columns), 4 => 16 warps x (16 x 16)
template <int KS, int NG>
__global__ void __launch_bounds__(128 * NG, 1) qkv_bwd_mma_kernel(QkvBwdArgs a, FDims d) {
  constexpr int S = 8 * KS + 4, TILE = FR * S, STAGE = 5 * TILE, BT = 128 * NG, NW = 4 * NG, NTW = 8 / NG;
  CAST_DYN_SMEM(float, sm);
  float* Wsm = sm + 2 * STAGE;      // Wq | Wk | Wv, each [64][S] natural layout, zero padded
  float* rowstat = Wsm + 3 * TILE;  // [FR][4]
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5, g = lane >> 2, tig = lane & 3;
  const int mt = warp & 3, nh = warp >> 2;
  const int H = d.H;
  int nact = KS - NTW * nh;
  nact = nact < 0 ? 0 : (nact > NTW ? NTW : nact);
  const int m0 = mt * 16, n0 = nh * NTW * 8;
  for (int i = t; i < 3 * TILE; i += BT) Wsm[i] = 0.f;      // weights: zero padded to [64][S]
  rm_zero_pad<8 * KS, S>(sm, 10 * FR, H);                   // K-padding columns of the ten stage tiles
  __syncthreads();
  rm_load_w_async<S>(Wsm, a.Wq, H);   // (committed with the first tile's group below, or by the lone commit)
  rm_load_w_async<S>(Wsm + TILE, a.Wk, H);
  rm_load_w_async<S>(Wsm + 2 * TILE, a.Wv, H);
  RmLnRows<S, BT> lnr;
  lnr.load_gamma(a.gamma, H);
  const bool v0 = rm_vec2_ok(a.dQ, H), v1 = rm_vec2_ok(a.dK, H), v2 = rm_vec2_ok(a.dV, H), v3 = rm_vec2_ok(a.x, H),
             v4 = rm_vec2_ok(a.qn, H);
  auto issue = [&](long tile, int st) {
    float* b = sm + st * STAGE;
    const long row0 = tile * FR;
    rm_load_tile_async<S, NW>(b, a.dQ, row0, d.N, H, v0);
    rm_load_tile_async<S, NW>(b + TILE, a.dK, row0, d.N, H, v1);
    rm_load_tile_async<S, NW>(b + 2 * TILE, a.dV, row0, d.N, H, v2);
    rm_load_tile_async<S, NW>(b + 3 * TILE, a.x, row0, d.N, H, v3);
    rm_load_tile_async<S, NW>(b + 4 * TILE, a.qn, row0, d.N, H, v4);
    cp_async_commit();
  };
  const LnOutFx ofx = qkv_out_fx(a);
  float gWq[1][NTW][4], gWkv[2][NTW][4];
  rm_zero(gWq[0]);
  rm_zero(gWkv[0]);
  rm_zero(gWkv[1]);
  constexpr int SL = BT / 64;  // row slices of the column sums
  float vbq = 0.f, vbk = 0.f, vbv = 0.f;  // bias gradients, dgamma, dbeta: this thread's (column, row slice) partials
  float dgam = 0.f, dbet = 0.f;
  // The kernel before this one in the chain is the attention dK/dV kernel: of the first tile only dK and dV are its
  // output (dQ, x, LN(x), the weights and gamma were complete before it started), so everything else is requested
  // before the wait and arrives while that kernel drains.
  if ((long)blockIdx.x < a.ntiles) {
    const long row0 = (long)blockIdx.x * FR;
    rm_load_tile_async<S, NW>(sm, a.dQ, row0, d.N, H, v0);
    rm_load_tile_async<S, NW>(sm + 3 * TILE, a.x, row0, d.N, H, v3);
    rm_load_tile_async<S, NW>(sm + 4 * TILE, a.qn, row0, d.N, H, v4);
  }
  cp_async_commit();
  cast_pdl_wait();
  if ((long)blockIdx.x < a.ntiles) {
    const long row0 = (long)blockIdx.x * FR;
    rm_load_tile_async<S, NW>(sm + TILE, a.dK, row0, d.N, H, v1);
    rm_load_tile_async<S, NW>(sm + 2 * TILE, a.dV, row0, d.N, H, v2);
  }
  cp_async_commit();
  int it = 0;
  for (long tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x, ++it) {
    const int st = it & 1;
    float* Gq = sm + st * STAGE;
    float* Gk = Gq + TILE;
    float* Gv = Gk + TILE;
    float* X = Gv + TILE;
    float* Qn = X + TILE;
    const long row0 = tile * FR;
    __syncthreads();  // the other stage is free (its last readers finished the previous tile)
    if (tile + gridDim.x < a.ntiles) {
      issue(tile + gridDim.x, st ^ 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    // gradient of `outputs += queries` for this thread's fragment of dqn (fetched early, consumed after the products)
    float dres[NTW][4];
#pragma unroll
    for (int nt = 0; nt < NTW; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const long row = row0 + m0 + g + (e >> 1) * 8;
        const int c = n0 + nt * 8 + 2 * tig + (e & 1);
        dres[nt][e] = (nt < nact && c < H && row < d.N) ? a.dres[row * H + c] : 0.f;
      }
    {
      const float* const gq[1] = {Gq};
      rm_wgrad<1, S, NTW>(gWq, Qn, m0, gq, n0, nact, lane);
      const float* const gkv[2] = {Gk, Gv};
      rm_wgrad<2, S, NTW>(gWkv, X, m0, gkv, n0, nact, lane);
    }
    float accq[NTW][4], acck[NTW][4];
    rm_zero(accq);
    rm_zero(acck);
    rm_mm_bt<KS, S, NTW>(accq, Gq + m0 * S, Wsm + n0 * S, nact, lane);             // dqn (without the residual)
    rm_mm_bt<KS, S, NTW>(acck, Gk + m0 * S, Wsm + TILE + n0 * S, nact, lane);      // dx through K ...
    rm_mm_bt<KS, S, NTW>(acck, Gv + m0 * S, Wsm + 2 * TILE + n0 * S, nact, lane);  // ... and V
    vbq += rm_colsum_slice<SL, S>(Gq);
    vbk += rm_colsum_slice<SL, S>(Gk);
    vbv += rm_colsum_slice<SL, S>(Gv);
    __syncthreads();
#pragma unroll
    for (int nt = 0; nt < NTW; ++nt) {
      if (nt >= nact) continue;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int r = m0 + g + (e >> 1) * 8, c = n0 + nt * 8 + 2 * tig + (e & 1);
        const bool ok = c < H && row0 + r < d.N;
        Gq[r * S + c] = ok ? accq[nt][e] + dres[nt][e] : 0.f;
        Gk[r * S + c] = ok ? acck[nt][e] : 0.f;
      }
    }
    __syncthreads();
    lnr.run(Gq, X, Gk, a.mean, a.rstd, rowstat, row0, d, a.dx, ofx);
    __syncthreads();
    rm_ln_cols_slice<SL, S>(Gq, X, rowstat, dgam, dbet);
  }
  float* P = a.partial + (long)blockIdx.x * (2L * H + 3L * (H * H + H));
  rm_fold_cols<SL>(dgam, sm, P + H, H);
  rm_fold_cols<SL>(dbet, sm, P, H);
  rm_fold_cols<SL>(vbq, sm, P + 2 * H + H * H, H);
  rm_fold_cols<SL>(vbk, sm, P + 2 * H + (H * H + H) + H * H, H);
  rm_fold_cols<SL>(vbv, sm, P + 2 * H + 2 * (H * H + H) + H * H, H);
  rm_store_wpartial(P + 2 * H, gWq[0], m0, n0, nact, H, lane);
  rm_store_wpartial(P + 2 * H + (H * H + H), gWkv[0], m0, n0, nact, H, lane);
  rm_store_wpartial(P + 2 * H + 2 * (H * H + H), gWkv[1], m0, n0, nact, H, lane);
}

// ------------------------------------------------------------------------------------------------ ffn backward
template <int KS, int NG>
__global__ void __launch_bounds__(128 * NG, 1) ffn_bwd_mma_kernel(FfnBwdArgs a, FDims d) {
  constexpr int S = 8 * KS + 4, TILE = FR * S, STAGE = 4 * TILE, BT = 128 * NG, NW = 4 * NG, NTW = 8 / NG;
  CAST_DYN_SMEM(float, sm);
  float* Gd = sm + 2 * STAGE;  // dx * mask * dropout, later dzn
  float* Dh = Gd + TILE;       // gradient at the FFN hidden pre-activation
  float* W1s = Dh + TILE;      // [64][S] natural
  float* W2s = W1s + TILE;
  float* rowstat = W2s + TILE;  // [FR][4]
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5, g = lane >> 2, tig = lane & 3;
  const int mt = warp & 3, nh = warp >> 2;
  const int H = d.H;
  int nact = KS - NTW * nh;
  nact = nact < 0 ? 0 : (nact > NTW ? NTW : nact);
  const int m0 = mt * 16, n0 = nh * NTW * 8;
  const float scale = a.rate > 0.f ? 1.0f / (1.0f - a.rate) : 1.0f;
  const Drop dout = make_drop(a.rate, a.seed, a.step, a.site_o);
  for (int i = t; i < 4 * TILE; i += BT) Gd[i] = 0.f;       // Gd, Dh and the two weight tiles
  rm_zero_pad<8 * KS, S>(sm, 8 * FR, H);                    // K-padding columns of the eight stage tiles
  __syncthreads();
  rm_load_w_async<S>(W1s, a.W1, H);   // (committed with the first tile's group below, or by the lone commit)
  rm_load_w_async<S>(W2s, a.W2, H);
  RmLnRows<S, BT> lnr;
  lnr.load_gamma(a.gamma, H);
  const bool v0 = rm_vec2_ok(a.dx, H), v1 = rm_vec2_ok(a.zn, H), v2 = rm_vec2_ok(a.h1d, H), v3 = rm_vec2_ok(a.y, H);
  auto issue = [&](long tile, int st) {
    float* b = sm + st * STAGE;
    const long row0 = tile * FR;
    rm_load_tile_async<S, NW>(b, a.dx, row0, d.N, H, v0);
    rm_load_tile_async<S, NW>(b + TILE, a.zn, row0, d.N, H, v1);
    rm_load_tile_async<S, NW>(b + 2 * TILE, a.h1d, row0, d.N, H, v2);
    rm_load_tile_async<S, NW>(b + 3 * TILE, a.y, row0, d.N, H, v3);
    cp_async_commit();
  };
  float gW1[1][NTW][4], gW2[1][NTW][4];
  rm_zero(gW1[0]);
  rm_zero(gW2[0]);
  constexpr int SL = BT / 64;  // row slices of the column sums
  float vb1 = 0.f, vb2 = 0.f;  // bias gradients, dgamma, dbeta: this thread's (column, row slice) partials
  float dgam = 0.f, dbet = 0.f;
  // Of the first tile only dx is the previous kernel's output (the loss tail or the block above's qkv backward kernel);
  // LN(y), the hidden activations and y are forward-pass data: requested before the wait, with the weights and gamma.
  if ((long)blockIdx.x < a.ntiles) {
    const long row0 = (long)blockIdx.x * FR;
    rm_load_tile_async<S, NW>(sm + TILE, a.zn, row0, d.N, H, v1);
    rm_load_tile_async<S, NW>(sm + 2 * TILE, a.h1d, row0, d.N, H, v2);
    rm_load_tile_async<S, NW>(sm + 3 * TILE, a.y, row0, d.N, H, v3);
  }
  cp_async_commit();
  cast_pdl_wait();
  cast_pdl_trigger();  // the attention dQ kernel that follows has a long prologue that does not depend on this kernel
  if ((long)blockIdx.x < a.ntiles) rm_load_tile_async<S, NW>(sm, a.dx, (long)blockIdx.x * FR, d.N, H, v0);
  cp_async_commit();
  // row mask of a tile (padding positions and rows past N get 0): fetched one tile ahead by threads 0..FR-1 and handed
  // over through shared memory (the first FR words of rowstat, free until the LayerNorm pass at the end of the tile)
  auto row_mask = [&](long tile) -> float {
    const long row = tile * FR + t;
    return (t < FR && row < d.N && (!a.ids || a.ids[row] != 0)) ? 1.f : 0.f;
  };
  float mcur = (long)blockIdx.x < a.ntiles ? row_mask(blockIdx.x) : 0.f;
  float* rowm = rowstat;
  int it = 0;
  for (long tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x, ++it) {
    const int st = it & 1;
    float* Gm = sm + st * STAGE;  // dx, masked in place
    float* Zn = Gm + TILE;
    float* Hd = Zn + TILE;
    float* Yr = Hd + TILE;
    const long row0 = tile * FR;
    __syncthreads();
    float mnext = 0.f;
    if (tile + gridDim.x < a.ntiles) {
      mnext = row_mask(tile + gridDim.x);
      issue(tile + gridDim.x, st ^ 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    if (t < FR) rowm[t] = mcur;
    mcur = mnext;
    __syncthreads();
    // masked / dropped upstream gradient: one (row, column pair) task per thread and pass, one dropout hash word each
    {
      const int PW = (H + 1) >> 1;
#pragma unroll 4
      for (int p = t; p < FR * PW; p += BT) {
        const int r = p / PW, c = 2 * (p - r * PW);
        const long row = row0 + r;
        const bool ok = row < d.N;
        const float m = rowm[r];
        float dm2[2];
        drop_mul2(dout, (unsigned long long)(row * H + c), dm2[0], dm2[1]);
        const float g0 = Gm[r * S + c] * m;
        Gm[r * S + c] = g0;
        Gd[r * S + c] = ok ? g0 * dm2[0] : 0.f;
        if (c + 1 < H) {
          const float g1 = Gm[r * S + c + 1] * m;
          Gm[r * S + c + 1] = g1;
          Gd[r * S + c + 1] = ok ? g1 * dm2[1] : 0.f;
        }
      }
    }
    __syncthreads();
    // dW2 += h1d^T Gd ; db2 += colsum(Gd) ; dh = (Gd W2^T) * relu/dropout mask
    {
      const float* const gb[1] = {Gd};
      rm_wgrad<1, S, NTW>(gW2, Hd, m0, gb, n0, nact, lane);
      float acc[NTW][4];
      rm_zero(acc);
      rm_mm_bt<KS, S, NTW>(acc, Gd + m0 * S, W2s + n0 * S, nact, lane);
#pragma unroll
      for (int nt = 0; nt < NTW; ++nt) {
        if (nt >= nact) continue;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int r = m0 + g + (e >> 1) * 8, c = n0 + nt * 8 + 2 * tig + (e & 1);
          Dh[r * S + c] = (c < H && Hd[r * S + c] > 0.f) ? acc[nt][e] * scale : 0.f;
        }
      }
    }
    vb2 += rm_colsum_slice<SL, S>(Gd);
    __syncthreads();
    // dW1 += zn^T Dh ; db1 += colsum(Dh) ; dzn = Dh W1^T + Gm  (stored over Gd)
    {
      const float* const gb[1] = {Dh};
      rm_wgrad<1, S, NTW>(gW1, Zn, m0, gb, n0, nact, lane);
      float acc[NTW][4];
      rm_zero(acc);
      rm_mm_bt<KS, S, NTW>(acc, Dh + m0 * S, W1s + n0 * S, nact, lane);
#pragma unroll
      for (int nt = 0; nt < NTW; ++nt) {
        if (nt >= nact) continue;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int r = m0 + g + (e >> 1) * 8, c = n0 + nt * 8 + 2 * tig + (e & 1);
          Gd[r * S + c] = c < H ? acc[nt][e] + Gm[r * S + c] : 0.f;
        }
      }
    }
    vb1 += rm_colsum_slice<SL, S>(Dh);
    __syncthreads();
    lnr.run(Gd, Yr, nullptr, a.mean, a.rstd, rowstat, row0, d, a.dy, ln_out_none());
    __syncthreads();
    rm_ln_cols_slice<SL, S>(Gd, Yr, rowstat, dgam, dbet);
  }
  float* P = a.partial + (long)blockIdx.x * (2L * H + 2L * (H * H + H));
  rm_fold_cols<SL>(dgam, sm, P + H, H);
  rm_fold_cols<SL>(dbet, sm, P, H);
  rm_fold_cols<SL>(vb1, sm, P + 2 * H + H * H, H);
  rm_fold_cols<SL>(vb2, sm, P + 2 * H + H * H + H + H * H, H);
  rm_store_wpartial(P + 2 * H, gW1[0], m0, n0, nact, H, lane);
  rm_store_wpartial(P + 2 * H + H * H + H, gW2[0], m0, n0, nact, H, lane);
}

constexpr int RM_BWD_NG = 4;  // column groups (x4 row blocks = 16 warps) of the backward row kernels

template <int KS>
static size_t qkv_bwd_mma_smem() { return sizeof(float) * ((size_t)(10 + 3) * FR * (8 * KS + 4) + FR * 4); }
template <int KS>
static size_t ffn_bwd_mma_smem() { return sizeof(float) * ((size_t)(8 + 4) * FR * (8 * KS + 4) + FR * 4); }

}  // namespace cast
