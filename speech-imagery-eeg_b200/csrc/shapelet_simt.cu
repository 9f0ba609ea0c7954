// CUDA-core (FP32 pipe) shapelet distance + pooling, forward and backward, all distance modes.
//
// This is the engine for IGN_DIST_L1 (the reference default, Shapelet.py:74 — it has no cross term, so
// it can never run on tensor cores; its roofline is the FP32 ALU pipe) and the exact-fp32 engine
// (IGN_PREC_FP32) for the cross-term modes.  Reference semantics: Shapelet.py:60-84, :96-111.
//
// Data layout
//   xn     [B,M,Tp]   one series row per (sample, channel), time contiguous
//   W      [K,M,L]
//   dstore [B,M,K,Tw] all window distances (training only), time contiguous
//   pooled outputs [B,K,M]
//
// Forward.  One CTA owns a channel m, a block of KB shapelets and a chunk of the batch; the shapelets of
// that channel stay in shared memory for the CTA's lifetime, series rows stream through NB at a time.
//   phase 1  register-tiled distance: each thread owns TT consecutive windows x KK shapelets and slides
//            along the lag axis with a 12-register ring (1 LDS.128 of x + KK broadcast LDS.128 of w per
//            4 lags for 4*TT*KK accumulate pairs).  The epilogue stays in registers: raw sum -> distance
//            (norm terms from the prefix pass), coalesced store of d for backward, per-thread min/argmin.
//   phase 2  one warp per (sample, shapelet) row reduces the per-tile candidates with shuffles (first
//            index on ties) and applies the pooling non-linearity once per row:
//            max_t exp(-(eps d_t)^2) = exp(-(eps min_t d_t)^2), so no exp per window is needed.
// Strides > 1 (only when seq_len >= 3000, Shapelet.py:162) are handled by de-interleaving series and
// shapelet into `stride` residue classes: sum_l f(x[t*s+l], w[l]) = sum_r sum_q f(x_r[t+q], w_r[q]),
// i.e. `stride` unit-stride correlations, so the same sliding-window code runs for every stride.
//
// Backward (stored-d), four kernels per length group:
//   pooling backward (pool_bwd_reg_kernel, HBM-bound): one warp per saved distance row recomputes the soft-max
//            statistics (Z, S1, arg-max of p with first-index ties — exactly the reference's hard one-hot,
//            Shapelet.py:79) and writes a_t = dLoss/dd_t (times the mode's norm factor) to the coefficient workspace
//   tie pre-check (L1): which series rows can hold a value equal to one of the CTA's shapelet values
//   contraction (shapelet_bwd_kernel): one CTA owns a channel, a block of shapelets, a block of lags and a batch
//            chunk; each thread owns 8 lags of ONE shapelet in registers for the whole chunk and slides along the window
//            axis with the same 12-register ring:
//              L1 : dW[l] = -(1/L) sum_t a_t sign(x[t+l]-w[l])     (sign(0)=0, exact)
//              dot: G[l]  = sum_t a_t x[t+l], then dW from G and two per-shapelet scalars (finalize)
//   finalize: per-chunk partials summed in a fixed order, closed-form scalar terms
// Partial sums are combined in a fixed order (shared memory, then a per-chunk workspace, then the finalize
// kernel) so the result is bit-reproducible run to run — no float atomics.
#include "ign_common.cuh"

#include <math.h>
#include <stdlib.h>

#include <map>
#include <mutex>
#include <tuple>
#include <type_traits>
#include <vector>
#include <utility>

namespace ign {
namespace {

constexpr int OP_L1 = 0;
constexpr int OP_DOT = 1;
constexpr int kMaxThreads = 256;
// Lags per thread in the backward contraction: 8 (16 was measured slower: fewer items, lower occupancy) or 10, whichever
// fills the thread block and the lag axis better (plan_bwd): L = 100 with K = 5 is 13 tiles x 5 shapelets = 65 threads
// per slot at 8 lags (195 of 224 lanes, 104 lags computed for 100) and 10 x 5 = 50 at 10 lags (250 of 256, no lag padding).

struct Geo {  // geometry shared by forward and backward
  int B, M, T, Tp, K, L, s;
  int Tw;      // number of windows
  int Ts;      // pitch of dstore rows (Tw rounded to 4)
  int DP;      // pitch of smem d/c rows (Tw rounded to 8)
  int CP;      // backward: pitch of coefficient rows in smem, DP skewed to 12 mod 32 words (conflict-free
               // LDS.128 when consecutive lanes read consecutive shapelets' rows)
  int XQ;      // pitch of one residue row of x in smem
  int LQ;      // pitch of one residue row of w in smem (ceil(L/s) rounded to 8; backward: to its lag tile LT)
  int LT;      // backward: lags per thread (8, 10 or 12)
  int KK, KB, nkb;
  int NB;      // series rows resident per pass
  int dbuf;    // forward: series rows double buffered (cp.async one pass ahead)
  int nchunk, cbase, cextra;   // batch chunks (grid z): chunk c walks cbase (+1 if c < cextra) passes of NB rows
  int dist, pool;
  float eps;
};

// samples [bbeg, bend) of batch chunk c: balanced chunks, the longer ones first (they are dispatched first)
__device__ __forceinline__ void chunk_range(const Geo& g, int c, int& bbeg, int& bend) {
  const int u0 = c * g.cbase + min(c, g.cextra);
  const int nu = g.cbase + (c < g.cextra ? 1 : 0);
  bbeg = min(g.B, u0 * g.NB);
  bend = min(g.B, (u0 + nu) * g.NB);
}

struct FwdArgs {
  const float* xn; const float* st0; const float* W; const float* thr;   // st0: window statistics [B,M,SP]
  float* p; float* dmin; int* argmin; float* dstore;
  int SP;
};

struct BwdArgs {
  const float* xn; const float* W;
  const float* coef;    // [B][M][K][Ts] per-window coefficients a_t written by pool_bwd_kernel
  float* part;          // [nchunk][K][M][L]
  int nseg, nlb, tlb;   // t-segments per row, l-blocks, l-tiles per l-block
  const unsigned char* tie;   // L1 only: [B][M][nkb] 1 = this row may contain x == w (exact path); NULL = always exact
};

struct PoolArgs {
  const float* g; int gK, gk0;   // upstream gradient [B,gK,M]; this launch's shapelets are gk0 .. gk0+K-1 of it (recompute chunks)
  const float* dstore; const float* dmin; const int* argmin;
  const float* st0; const float* st1; int SP; const float* wstat;   // window stats [B,M,SP]; wstat [K][M]: sum (w-mean)^2 (pearson)
  float* coef;          // [B][M][K][Ts]
  float* rowsc;         // [B][M][K][2] per-row scalars for the finalize kernel
  const float* gd;      // NULL, or dLoss/d(min_t d) [B,gK,M] indexed like g: added at the window `argmin` names
};


// ------------------------------------------------------------------------------------------------
// shared-memory staging helpers
// ------------------------------------------------------------------------------------------------

// Shapelet slab for channel m, shapelets [k0,k0+KB): ws[kl][r][q] = W[k0+kl][m][q*s+r] (centred for
// pearson), zero padded; wstat[kl] = mode-specific shapelet statistic.
__device__ void load_shapelets(const Geo& g, const float* __restrict__ W, int m, int k0, float* ws,
                               float* wstat) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  const int rowlen = g.s * g.LQ;
  for (int kl = warp; kl < g.KB; kl += nwarp) {
    const int k = k0 + kl;
    float* dst = ws + (size_t)kl * rowlen;
    for (int i = lane; i < rowlen; i += 32) dst[i] = 0.f;
    float stat = 0.f;
    if (k < g.K) {
      const float* src = W + ((size_t)k * g.M + m) * g.L;
      float s1 = 0.f, s2 = 0.f;
      for (int l = lane; l < g.L; l += 32) { float w = __ldg(src + l); s1 += w; s2 = fmaf(w, w, s2); }
#pragma unroll
      for (int o = 16; o; o >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); }
      float mean = 0.f;
      if (g.dist == IGN_DIST_PEARSON) {
        mean = s1 / (float)g.L;
        float c2 = 0.f;
        for (int l = lane; l < g.L; l += 32) { float w = __ldg(src + l) - mean; c2 = fmaf(w, w, c2); }
#pragma unroll
        for (int o = 16; o; o >>= 1) c2 += __shfl_xor_sync(0xffffffffu, c2, o);
        stat = sqrtf(c2);                            // ||w-mean||
      } else if (g.dist == IGN_DIST_COSINE) {
        stat = 1.f / fmaxf(sqrtf(s2), 1e-8f);        // 1/max(||w||,eps)
      } else {
        stat = s2;                                   // ||w||^2 (sql2)
      }
      __syncwarp();
      for (int l = lane; l < g.L; l += 32) {
        const int r = l % g.s, q = l / g.s;
        dst[r * g.LQ + q] = __ldg(src + l) - mean;
      }
    }
    if (lane == 0) wstat[kl] = stat;
  }
}

// Series rows for samples [b0,b0+nb) of channel m, de-interleaved by residue; window statistics rows.
__device__ void load_series(const Geo& g, const float* __restrict__ xn, const float* __restrict__ stat, int SP,
                            int m, int b0, int nb, float* xs, float* st0) {
  const int rowlen = g.s * g.XQ;
  const int total = g.NB * rowlen;
  const int nthr = blockDim.x;
  if (g.s == 1) {
    for (int i = threadIdx.x * 4; i < total; i += nthr * 4) {   // XQ % 4 == 0
      const int bl = i / rowlen, q = i - bl * rowlen;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (bl < nb && q < g.Tp) v = *reinterpret_cast<const float4*>(xn + ((size_t)(b0 + bl) * g.M + m) * g.Tp + q);
      *reinterpret_cast<float4*>(xs + i) = v;
    }
  } else {
    for (int i = threadIdx.x; i < total; i += nthr) {
      const int bl = i / rowlen, rem = i - bl * rowlen;
      const int r = rem / g.XQ, q = rem - r * g.XQ;
      const int t = q * g.s + r;
      float v = 0.f;
      if (bl < nb && t < g.T) v = __ldg(xn + ((size_t)(b0 + bl) * g.M + m) * g.Tp + t);
      xs[i] = v;
    }
  }
  if (st0) {   // cross-term distances: per-window norm terms from the window-statistics pass (SP % 16 == 0)
    const int rowv = g.DP / 4;
    for (int i = threadIdx.x; i < g.NB * rowv; i += nthr) {
      const int bl = i / rowv, t = (i - bl * rowv) * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (bl < nb && t < SP) v = *reinterpret_cast<const float4*>(stat + ((size_t)(b0 + bl) * g.M + m) * SP + t);
      *reinterpret_cast<float4*>(st0 + bl * g.DP + t) = v;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// phase 1: register-tiled sliding distance
// ------------------------------------------------------------------------------------------------
template <int OP>
__device__ __forceinline__ float acc_op(float acc, float x, float w) {
  if (OP == OP_L1) return acc + fabsf(x - w);
  return fmaf(x, w, acc);
}

template <int OP, int KK, int TT>
__device__ __forceinline__ void distance_item(const Geo& g, const float* __restrict__ xrow,
                                              const float* __restrict__ wbase, int t0, float (&acc)[TT][KK]) {
  constexpr int RING = TT + 4;
#pragma unroll
  for (int j = 0; j < TT; ++j)
#pragma unroll
    for (int k = 0; k < KK; ++k) acc[j][k] = 0.f;
  const int wpitch = g.s * g.LQ;

  for (int r = 0; r < g.s; ++r) {
    const int Lr = (g.L - r + g.s - 1) / g.s;
    const float* xr = xrow + r * g.XQ + t0;
    const float* wr = wbase + r * g.LQ;
    float xv[RING];
#pragma unroll
    for (int j = 0; j < TT; j += 4) {
      float4 v = *reinterpret_cast<const float4*>(xr + j);
      xv[j] = v.x; xv[j + 1] = v.y; xv[j + 2] = v.z; xv[j + 3] = v.w;
    }
    const int Lr4 = Lr & ~3;
    int q = 0;
#define IGN_FWD_STEP(BASE, QQ)                                                              \
    {                                                                                       \
      float4 nx = *reinterpret_cast<const float4*>(xr + (QQ) + TT);                         \
      xv[((BASE) + TT + 0) % RING] = nx.x; xv[((BASE) + TT + 1) % RING] = nx.y;             \
      xv[((BASE) + TT + 2) % RING] = nx.z; xv[((BASE) + TT + 3) % RING] = nx.w;             \
      float4 w4[KK];                                                                        \
      _Pragma("unroll") for (int k = 0; k < KK; ++k)                                        \
        w4[k] = *reinterpret_cast<const float4*>(wr + k * wpitch + (QQ));                   \
      _Pragma("unroll") for (int j = 0; j < TT; ++j) {                                      \
        _Pragma("unroll") for (int k = 0; k < KK; ++k) {                                    \
          acc[j][k] = acc_op<OP>(acc[j][k], xv[((BASE) + j + 0) % RING], w4[k].x);          \
          acc[j][k] = acc_op<OP>(acc[j][k], xv[((BASE) + j + 1) % RING], w4[k].y);          \
          acc[j][k] = acc_op<OP>(acc[j][k], xv[((BASE) + j + 2) % RING], w4[k].z);          \
          acc[j][k] = acc_op<OP>(acc[j][k], xv[((BASE) + j + 3) % RING], w4[k].w);          \
        }                                                                                   \
      }                                                                                     \
    }
    if (TT == 8) {
      for (; q + 12 <= Lr4; q += 12) {
        IGN_FWD_STEP(0, q) IGN_FWD_STEP(4, q + 4) IGN_FWD_STEP(8, q + 8)
      }
      if (q + 4 <= Lr4) { IGN_FWD_STEP(0, q) q += 4; if (q + 4 <= Lr4) { IGN_FWD_STEP(4, q) q += 4; } }
    } else {
      for (; q + 8 <= Lr4; q += 8) {
        IGN_FWD_STEP(0, q) IGN_FWD_STEP(4, q + 4)
      }
      if (q + 4 <= Lr4) { IGN_FWD_STEP(0, q) q += 4; }
    }
#undef IGN_FWD_STEP
    for (; q < Lr; ++q) {   // scalar tail (< 4 lags)
#pragma unroll
      for (int k = 0; k < KK; ++k) {
        const float w = wr[k * wpitch + q];
#pragma unroll
        for (int j = 0; j < TT; ++j) acc[j][k] = acc_op<OP>(acc[j][k], xr[q + j], w);
      }
    }
  }
}

// raw accumulator -> distance
template <int OP>
__device__ __forceinline__ float finish_distance(int dist, float raw, float invL, float xstat, float wstat) {
  // (multiplication by 1/L and __fdividef differ from the reference's true divisions by <= 2 ulp and avoid the
  //  IEEE-division slow path, which zero numerators on padded windows would otherwise take warp-wide)
  if (OP == OP_L1) return raw * invL;
  if (dist == IGN_DIST_SQL2) return fmaxf((xstat + wstat - 2.f * raw) * invL, 0.f);
  if (dist == IGN_DIST_COSINE) return 1.f - raw * xstat * wstat;
  return 1.f - __fdividef(raw, xstat * wstat + 1e-8f);   // xstat = ||x_w-mu||, wstat = ||w-mean|| (sqrt hoisted)
}

// ex2.approx.ftz: 2 ulp, flushes denormals (p < 1e-38 -> 0); used only for backward soft-max weights
__device__ __forceinline__ float fast_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
constexpr float kLog2e = 1.4426950408889634f;

struct ArgVal { float v; int i; };
__device__ __forceinline__ ArgVal warp_argmax_first(float v, int i) {
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    float ov = __shfl_xor_sync(0xffffffffu, v, o);
    int oi = __shfl_xor_sync(0xffffffffu, i, o);
    if (ov > v || (ov == v && oi < i)) { v = ov; i = oi; }
  }
  return {v, i};
}
__device__ __forceinline__ ArgVal warp_argmin_first(float v, int i) {
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    float ov = __shfl_xor_sync(0xffffffffu, v, o);
    int oi = __shfl_xor_sync(0xffffffffu, i, o);
    if (ov < v || (ov == v && oi < i)) { v = ov; i = oi; }
  }
  return {v, i};
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async4(void* dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit_wait_all() {
  asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}


// ------------------------------------------------------------------------------------------------
// forward kernel
// ------------------------------------------------------------------------------------------------
template <int OP, int KK, int TT>
__global__ void __launch_bounds__(kMaxThreads, 2) shapelet_fwd_kernel(const Geo g, const FwdArgs a) {
  extern __shared__ __align__(16) float smem[];
  const int m = blockIdx.x, k0 = blockIdx.y * g.KB;
  int bbeg, bend;
  chunk_range(g, blockIdx.z, bbeg, bend);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;

  const int ntile = g.DP / TT;
  const int nkc = g.KB / KK;
  float* xs = smem;
  float* ws = xs + g.NB * g.s * g.XQ;
  float* st0 = ws + g.KB * g.s * g.LQ;
  float* wstat = st0 + (OP != OP_L1 ? g.NB * g.DP : 0);
  float* cand_d = wstat + g.KB;                                   // [NB][KB][ntile]
  int* cand_i = reinterpret_cast<int*>(cand_d + g.NB * g.KB * ntile);

  load_shapelets(g, a.W, m, k0, ws, wstat);

  const int nitem = g.NB * ntile * nkc;
  const float Lf = 1.f / (float)g.L;   // 1/L

  // Series (and window-statistics) rows are double buffered and fetched with cp.async one pass ahead (strided groups
  // de-interleave with 4-byte copies), so the load of pass i+1 hides under the distance loop of pass i (the exposed load + barrier phases cost short
  // shapelets ~8 %: FMA pipe 74 % at L=100 against 82 % at L=500 before this change).
  const bool dbuf = g.dbuf != 0;
  const int xs_sz = g.NB * g.s * g.XQ;
  float* xs1 = smem + round_up((int)(cand_d - smem) + 2 * g.NB * g.KB * ntile, 4);   // second buffers, 16-byte aligned, behind the candidates
  float* st1 = xs1 + (dbuf ? xs_sz : 0);
  auto prefetch = [&](int b0, int buf) {
    const int nb = min(g.NB, bend - b0);
    float* xd = buf ? xs1 : xs;
    const int xrow = g.Tp / 4;
    if (g.s == 1) {
      for (int i = threadIdx.x; i < nb * xrow; i += blockDim.x) {
        const int rbl = i / xrow, c = i - rbl * xrow;
        cp_async16(xd + rbl * g.XQ + c * 4, a.xn + ((size_t)(b0 + rbl) * g.M + m) * g.Tp + c * 4);
      }
    } else {                                            // de-interleave: sample t -> residue row t % s, slot t / s
      const int nthr = blockDim.x;
      const int dq = nthr / g.s, dr = nthr - dq * g.s;
      for (int rbl = 0; rbl < nb; ++rbl) {
        const float* xsrc = a.xn + ((size_t)(b0 + rbl) * g.M + m) * g.Tp;
        float* xdst = xd + (size_t)rbl * g.s * g.XQ;
        int q = threadIdx.x / g.s, r = threadIdx.x - q * g.s;
        for (int t = threadIdx.x; t < g.T; t += nthr) {
          cp_async4(xdst + r * g.XQ + q, xsrc + t);
          q += dq; r += dr;
          if (r >= g.s) { r -= g.s; ++q; }
        }
      }
    }
    if (OP != OP_L1) {
      float* sd = buf ? st1 : st0;
      const int srow = g.DP / 4;                                     // DP <= SP: whole 16-byte chunks of the statistics row
      for (int i = threadIdx.x; i < nb * srow; i += blockDim.x) {
        const int rbl = i / srow, c = i - rbl * srow;
        cp_async16(sd + rbl * g.DP + c * 4, a.st0 + ((size_t)(b0 + rbl) * g.M + m) * a.SP + c * 4);
      }
    }
  };
  if (dbuf) {   // zero once: the pad columns behind Tp are never written by the prefetch
    for (int i = threadIdx.x; i < xs_sz; i += blockDim.x) { xs[i] = 0.f; xs1[i] = 0.f; }
    __syncthreads();
    if (bbeg < bend) prefetch(bbeg, 0);
  }
  int buf = 0;

  for (int b0 = bbeg; b0 < bend; b0 += g.NB) {
    const int nb = min(g.NB, bend - b0);
    if (dbuf) {
      cp_async_commit_wait_all();
      __syncthreads();   // this pass's rows landed; everyone is done with the other buffer and with the candidates
      if (b0 + g.NB < bend) prefetch(b0 + g.NB, buf ^ 1);
    } else {
      __syncthreads();   // previous pass finished with xs/cand (and ws is written on the first pass)
      load_series(g, a.xn, a.st0, a.SP, m, b0, nb, xs, OP != OP_L1 ? st0 : nullptr);
      __syncthreads();
    }
    const float* xcur = (dbuf && buf) ? xs1 : xs;
    const float* stcur = (dbuf && buf) ? st1 : st0;
    // ---- phase 1: distances + register epilogue ----
    for (int item = threadIdx.x; item < nitem; item += blockDim.x) {
      const int tt = item % ntile;
      const int rest = item / ntile;
      const int bl = rest % g.NB, kc = rest / g.NB;
      if (bl >= nb || k0 + kc * KK >= g.K) continue;
      const int t0 = tt * TT;
      float acc[TT][KK];
      distance_item<OP, KK, TT>(g, xcur + bl * g.s * g.XQ, ws + kc * KK * g.s * g.LQ, t0, acc);
      float xst[TT];
#pragma unroll
      for (int j = 0; j < TT; ++j) xst[j] = (OP != OP_L1) ? stcur[bl * g.DP + t0 + j] : 0.f;
      const int b = b0 + bl;
#pragma unroll
      for (int k = 0; k < KK; ++k) {
        const int kl = kc * KK + k, kk = k0 + kl;
        if (kk >= g.K) break;
        const float wst = wstat[kl];
        float best = INFINITY; int bi = 0x7fffffff;
        float dv[TT];
#pragma unroll
        for (int j = 0; j < TT; ++j) {
          const float d = finish_distance<OP>(g.dist, acc[j][k], Lf, xst[j], wst);
          const bool valid = t0 + j < g.Tw;
          dv[j] = valid ? d : 0.f;
          if (valid && d < best) { best = d; bi = t0 + j; }
        }
        if (a.dstore) {
          float* dg = a.dstore + (((size_t)b * g.M + m) * g.K + kk) * g.Ts + t0;
#pragma unroll
          for (int j = 0; j < TT; j += 4)
            if (t0 + j < g.Ts) *reinterpret_cast<float4*>(dg + j) = make_float4(dv[j], dv[j + 1], dv[j + 2], dv[j + 3]);
        }
        cand_d[(bl * g.KB + kl) * ntile + tt] = best;
        cand_i[(bl * g.KB + kl) * ntile + tt] = bi;
      }
    }
    __syncthreads();
    // ---- phase 2: one warp per (sample, shapelet) row reduces the tile candidates ----
    for (int row = warp; row < g.NB * g.KB; row += nwarp) {
      const int bl = row / g.KB, kl = row - bl * g.KB;
      const int b = b0 + bl, k = k0 + kl;
      if (bl >= nb || k >= g.K) continue;
      float dmn = INFINITY; int imn = 0x7fffffff;
      for (int tt = lane; tt < ntile; tt += 32) {
        const float d = cand_d[row * ntile + tt];
        if (d < dmn) { dmn = d; imn = cand_i[row * ntile + tt]; }
      }
      ArgVal mn = warp_argmin_first(dmn, imn);
      if (lane == 0) {
        const size_t o = ((size_t)b * g.K + k) * g.M + m;
        float pv;
        if (g.pool == IGN_POOL_RBF_MAX) {
          const float ed = g.eps * mn.v;
          pv = expf(-(ed * ed));                              // Shapelet.py:77 at the best window
        } else {
          pv = 1.f / (1.f + expf(-(a.thr[(size_t)k * g.M + m] - mn.v)));   // Shapelet.py:109
        }
        a.p[o] = pv; a.dmin[o] = mn.v;
        if (a.argmin) a.argmin[o] = mn.i;
      }
    }
    buf ^= 1;
  }
  if (dbuf) cp_async_commit_wait_all();
}

// ------------------------------------------------------------------------------------------------
// backward kernel
// ------------------------------------------------------------------------------------------------
// L1 backward accumulates A[l] = sum_t c_t ([x>w] + 0.5 [x==w]); the finalize kernel forms
// sum_t c_t sign(x-w) = 2 A[l] - sum_t c_t  (sign(0) = 0 exactly, as torch's abs backward).
// Exact ties x == w are impossible for a series row that shares no value with the CTA's shapelets; that is
// decided per row by tie_check_kernel, and such rows take the 2-instruction path (FSETP + predicated FADD).
// (An FFMA.SAT-built indicator on the FMA pipe was measured at the same speed — both forms are issue-bound at
//  two instructions per element — and is inexact for |x-w| < 2^-60, so the compare form is kept.)
template <int OP, bool EXACT>
__device__ __forceinline__ float bwd_op(float acc, float c, float hc, float x, float w) {
  if (OP == OP_L1) {
    if (x > w) acc += c;
    if (EXACT) { if (x == w) acc += hc; }
    return acc;
  }
  return fmaf(c, x, acc);
}

constexpr unsigned kHashEmpty = 0x7fc00001u;   // a NaN payload: never equal to a series value
// 2^18-bit (32 KB) two-hash Bloom filter in front of the exact hash set.  A false hit sends the whole warp through the
// probe loop, so what matters is the rate per 32 elements: 2500 values (K = 5, L = 500) give 0.04 % per element with two
// hashes (1 % per warp step) against 1 % (26 %) with one; 20000 values (L = 2000, strided groups) 2 % against 7 %.
constexpr int kTieBitmapLog2 = 18;
constexpr int kTieBitmapWords = (1 << kTieBitmapLog2) / 32;
__device__ __forceinline__ unsigned hash_key(float v) {
  unsigned b = __float_as_uint(v);
  return b == 0x80000000u ? 0u : b;            // -0 == +0
}
__device__ __forceinline__ unsigned hash_slot(unsigned key, unsigned mask) {
  return ((key * 0x9E3779B1u) >> 7) & mask;
}

// ---- pooling backward: elementwise over all (sample, channel, shapelet, window), HBM-bound ----
// One warp per saved distance row d[b,m,k,:]: soft-max statistics of the row (Z, S1 and the reference's
// hard one-hot = first arg-max of p, Shapelet.py:79 | for lts_min the forward's argmin, :105), then the
// coefficient a_t = dLoss/dd_t times the distance mode's norm factor, written to `coef`; two per-row
// scalars go to `rowsc` for the finalize kernel.
// GD (a.gd != NULL): the layer's second output min_t d (Shapelet.py:84 | :111) has a gradient too.  It is the hard min,
// so its whole gradient lands on ONE window, the forward's argmin (first index on ties) — for rbf_max not necessarily
// the arg-max of p that the straight-through one-hot selects (every p underflows to 0: arg-max 0, the min elsewhere).
// The training path never differentiates it and runs the GD = false instantiations, which are the kernels without it.
__device__ __forceinline__ void cp_async16_pool(void* dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}

// Persistent warps: every warp walks rows  w, w + nwarps_total, ...  with the NEXT row's distances already in flight
// (cp.async into the other half of its shared-memory slot) while it works on the current one — the kernel is
// bound by how many bytes it keeps in flight, not by instructions (issue 70 %, 4.0 TB/s before this change).
template <int DIST>
__device__ __forceinline__ float pool_emit(float c, float d, float s0, float s1, float wst, float& sc0, float& sc1);

// c0..c3, the coefficients of windows t0 .. t0+3: + v on window i (nothing when i is outside them)
__device__ __forceinline__ void add_at4(float& c0, float& c1, float& c2, float& c3, int i, int t0, float v) {
  const int h = i - t0;
  if ((unsigned)h < 4u) { c0 += h == 0 ? v : 0.f; c1 += h == 1 ? v : 0.f; c2 += h == 2 ? v : 0.f; c3 += h == 3 ? v : 0.f; }
}

template <int POOL, int DIST, bool GD>
__global__ void __launch_bounds__(256) pool_bwd_kernel(const Geo g, const PoolArgs a, int rows) {
  extern __shared__ __align__(16) float prow[];          // [warps][2][DP]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  const int wstride = gridDim.x * nwarp;
  float* slot = prow + (size_t)warp * 2 * g.DP;
  auto prefetch = [&](int r, int buf) {
    const float* src = a.dstore + (size_t)r * g.Ts;
    float* dstp = slot + (size_t)buf * g.DP;
    for (int t = lane * 4; t < g.Ts; t += 128) cp_async16_pool(dstp + t, src + t);
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  int row = blockIdx.x * nwarp + warp;
  if (row < rows) prefetch(row, 0);
  int buf = 0;
  for (; row < rows; row += wstride, buf ^= 1) {
  const int nxt = row + wstride;
  if (nxt < rows) { prefetch(nxt, buf ^ 1); asm volatile("cp.async.wait_group 1;" ::: "memory"); }
  else asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncwarp();
  float* dr = slot + (size_t)buf * g.DP;
  const int k = row % g.K, bm = row / g.K;
  const int m = bm % g.M, b = bm / g.M;
  const size_t o = ((size_t)b * g.K + k) * g.M + m;
  const float gk = a.g[((size_t)b * a.gK + a.gk0 + k) * g.M + m];
  const float eps = g.eps;
  const float qscale = -eps * eps * kLog2e;              // p = exp(-(eps d)^2) = 2^(qscale d^2)
  float Zs = 0.f, S1s = 0.f, shift = 0.f;
  int ih;
  if (POOL == IGN_POOL_LTS_MIN) { shift = a.dmin[o]; ih = a.argmin[o]; }
  float gdv = 0.f;
  int idm = -1;
  if (GD) { gdv = a.gd[((size_t)b * a.gK + a.gk0 + k) * g.M + m]; idm = a.argmin[o]; }
  __syncwarp();
  // Both passes walk the row in float4 chunks (lane owns chunks lane, lane + 32, ...): 128-bit shared-memory reads and
  // global stores, and in pass 2 the window-statistics loads of kPoolUnroll chunks are issued before any of them is
  // used.  (Element-wise loops with one statistics load per window left 14 dependent L2 round trips per row: the cosine
  // instantiation ran at 1.0-1.3 TB/s for T' = 1401 ... 1801, against 4.6 TB/s for L1, which loads no statistics.)
  const float4* dr4 = reinterpret_cast<const float4*>(dr);
  const int nvf = g.Tw >> 2;                             // whole chunks; chunk nvf (if Tw % 4) is masked
  const int nv = g.Ts >> 2;
  if (POOL == IGN_POOL_RBF_MAX) {
    float pmx = -1.f; int imx = 0x7fffffff;
    auto ev = [&](float d, int t) {
      const float p = fast_ex2(qscale * d * d);
      const float e = fast_ex2(p * kLog2e);
      Zs += e; S1s = fmaf(e, p, S1s);
      if (p > pmx) { pmx = p; imx = t; }
    };
#pragma unroll 2
    for (int c = lane; c < nvf; c += 32) {
      const float4 d = dr4[c];
      ev(d.x, 4 * c); ev(d.y, 4 * c + 1); ev(d.z, 4 * c + 2); ev(d.w, 4 * c + 3);
    }
    if (nvf < nv && lane == (nvf & 31)) {                // the lane that owns the partial chunk (it comes last in its order)
      const float4 d = dr4[nvf];
      const int t = 4 * nvf;
      ev(d.x, t);
      if (t + 1 < g.Tw) ev(d.y, t + 1);
      if (t + 2 < g.Tw) ev(d.z, t + 2);
    }
    ih = warp_argmax_first(pmx, imx).i;
  } else {
    auto ev = [&](float d) {
      const float e = fast_ex2((shift - d) * kLog2e);
      Zs += e; S1s = fmaf(e, d, S1s);
    };
#pragma unroll 2
    for (int c = lane; c < nvf; c += 32) {
      const float4 d = dr4[c];
      ev(d.x); ev(d.y); ev(d.z); ev(d.w);
    }
    if (nvf < nv && lane == (nvf & 31)) {
      const float4 d = dr4[nvf];
      const int t = 4 * nvf;
      ev(d.x);
      if (t + 1 < g.Tw) ev(d.y);
      if (t + 2 < g.Tw) ev(d.z);
    }
  }
  Zs = warp_sum(Zs); S1s = warp_sum(S1s);
  const float invZ = 1.f / Zs, bar = S1s * invZ;
  const float wst = (DIST == IGN_DIST_PEARSON) ? a.wstat[(size_t)k * g.M + m] : 0.f;
  const size_t srow = (size_t)bm * a.SP;                 // SP % 16 == 0: float4-aligned rows
  const float4* s0r4 = reinterpret_cast<const float4*>(a.st0 + srow);
  const float4* s1r4 = reinterpret_cast<const float4*>(a.st1 + srow);
  float* dst = a.coef + (size_t)row * g.Ts;
  // constants folded once per row: c_t = gk * (hard_t + soft_t (p_t - bar)) * p_t * (-2 eps^2 d_t)   (rbf_max)
  //                                c_t = gk * (hard_t - soft_t (d_t - bar))                             (lts_min)
  const float gm = gk * (-2.f * eps * eps);
  float sc0 = 0.f, sc1 = 0.f;
  auto emit = [&](float d, int t, float sxn, float mu) -> float {
    float c;
    if (POOL == IGN_POOL_RBF_MAX) {
      const float p = fast_ex2(qscale * d * d);
      const float soft = fast_ex2(p * kLog2e) * invZ;
      c = fmaf(soft, p - bar, t == ih ? 1.f : 0.f) * (p * d) * gm;
    } else {
      const float soft = fast_ex2((shift - d) * kLog2e) * invZ;
      c = gk * fmaf(-soft, d - bar, t == ih ? 1.f : 0.f);
    }
    if (GD && t == idm) c += gdv;
    return pool_emit<DIST>(c, d, sxn, mu, wst, sc0, sc1);
  };
  constexpr bool kS0 = DIST == IGN_DIST_COSINE || DIST == IGN_DIST_PEARSON;
  constexpr bool kS1 = DIST == IGN_DIST_PEARSON;
  constexpr int kPoolUnroll = 4;
  for (int c0 = lane; c0 < nvf; c0 += 32 * kPoolUnroll) {
    float4 s0[kPoolUnroll], s1[kPoolUnroll];
#pragma unroll
    for (int u = 0; u < kPoolUnroll; ++u) {
      const int c = min(c0 + 32 * u, nv - 1);            // clamped: in range, ignored below
      s0[u] = kS0 ? __ldg(s0r4 + c) : make_float4(0.f, 0.f, 0.f, 0.f);
      s1[u] = kS1 ? __ldg(s1r4 + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int u = 0; u < kPoolUnroll; ++u) {
      const int c = c0 + 32 * u;
      if (c < nvf) {
        const float4 d = dr4[c];
        float4 o;
        o.x = emit(d.x, 4 * c, s0[u].x, s1[u].x);
        o.y = emit(d.y, 4 * c + 1, s0[u].y, s1[u].y);
        o.z = emit(d.z, 4 * c + 2, s0[u].z, s1[u].z);
        o.w = emit(d.w, 4 * c + 3, s0[u].w, s1[u].w);
        *reinterpret_cast<float4*>(dst + 4 * c) = o;
      }
    }
  }
  if (nvf < nv && lane == (nvf & 31)) {                  // partial chunk: pad windows (at most 3) get 0
    const float4 d = dr4[nvf];
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 s0 = kS0 ? __ldg(s0r4 + nvf) : z, s1 = kS1 ? __ldg(s1r4 + nvf) : z;
    const int t = 4 * nvf;
    float4 o = z;
    o.x = emit(d.x, t, s0.x, s1.x);
    if (t + 1 < g.Tw) o.y = emit(d.y, t + 1, s0.y, s1.y);
    if (t + 2 < g.Tw) o.z = emit(d.z, t + 2, s0.z, s1.z);
    *reinterpret_cast<float4*>(dst + t) = o;
  }
  sc0 = warp_sum(sc0); sc1 = warp_sum(sc1);
  if (lane == 0) { a.rowsc[(size_t)row * 2] = sc0; a.rowsc[(size_t)row * 2 + 1] = sc1; }
  __syncwarp();                                         // everyone is done reading this slot half before it is refilled
  }
}

// Register-resident variant for rows of at most NCH*128 windows (every geometry with T' <= 1024, i.e. all BASELINE
// configs below T = 2000).  The generic kernel above spends 37 issue slots per element — two passes that each
// evaluate both exponentials — and is issue-bound at 65 % of HBM peak.  Here each lane owns NCH float4 chunks of the
// row; pass 1 evaluates the exponentials once and keeps (U_t, V_t) in registers with
//     c_t = Kc * U_t * (V_t - vbar) + [t == ih] * fix  (+ [t == argmin] * gd when GD)
//   rbf_max: V = p' = log2(e) p_t,  U = e^{p_t} p' d_t,  vbar = sum(e^p p')/Z,  Kc = -2 eps^2 g / (Z log2(e)^2),  fix = -2 eps^2 g p_ih d_ih
//   lts_min: V = d_t,  U = e^{dmin - d_t},  vbar = sum(U d)/Z,  Kc = -g/Z,  fix = g
// so pass 2 is three FP32 instructions per element over registers, all shared-memory and global accesses are
// 128-bit, and the arg-max is tracked per chunk (3 FMNMX + one compare per four elements, the position inside the
// chunk is resolved once per row).  Rows are prefetched two ahead (three cp.async stages per warp).
constexpr int kPoolStages = 3;
constexpr float kLog2Log2e = 0.5287663729448977f;     // log2(log2(e))

__device__ __forceinline__ float rbf_pprime(float d, float q) {   // log2(e) * exp(-(eps d)^2), q = -eps^2 log2(e)
  return fast_ex2(__fmaf_rn(__fmul_rn(d, q), d, kLog2Log2e));
}

// mode factor of one coefficient (the pool-independent part of the generic kernel's inner loop)
template <int DIST>
__device__ __forceinline__ float pool_emit(float c, float d, float s0, float s1, float wst, float& sc0, float& sc1) {
  if (DIST == IGN_DIST_L1 || DIST == IGN_DIST_SQL2) { sc0 += c; return c; }
  if (DIST == IGN_DIST_COSINE) { sc0 = fmaf(c, 1.f - d, sc0); return c * s0; }
  const float D = s0 * wst + 1e-8f;                      // s0 = ||x_w-mu||, s1 = mu, wst = ||w-mean||
  const float coef = __fdividef(c, D);
  sc0 = fmaf(coef, s1, sc0);
  sc1 += __fdividef(c * (1.f - d) * s0, wst * D);
  return coef;
}

// Lane layout of a row: `nfull` whole 128-window chunks (lane owns the float4 at (j*32+lane)*4), then the remaining
// < 128 windows, kept in the last register slot, either as ONE more float4 chunk with per-element validity (64 or more
// tail windows: T' = 501 has 117, and four scalar sub-chunks with their scalar loads cost it a third of the row's time)
// or in scalar sub-chunks of 32 (lane owns window tail0 + s*32 + lane) — a nearly empty float4 chunk would cost the
// whole warp four element times (T' = 901, 5 tail windows: 14 % of the row's work).
//
// Row order.  Cosine: a warp walks one contiguous range of rows, i.e. the K shapelet rows of a (sample, channel) group
// one after the other — the factor 1/||x_w|| depends on (sample, channel, window) only, so its row is fetched into
// registers once per group instead of once per shapelet (T' = 701: 4.05 -> 4.48 TB/s, T' = 501: 3.73 -> 3.98).  The
// other instantiations keep rows strided over the grid's warps (all warps stream neighbouring rows: measured 3 % faster
// than contiguous ranges when nothing is reused).
constexpr int pool_reg_min_blocks(int NCH) { return NCH <= 4 ? 3 : 2; }   // short rows are latency-bound: a third CTA per SM

template <int POOL, int DIST, int NCH, bool GD>
__global__ void __launch_bounds__(256, pool_reg_min_blocks(NCH)) pool_bwd_reg_kernel(const Geo g, const PoolArgs a, int rows) {
  extern __shared__ __align__(16) float prow[];          // [warps][kPoolStages][DP]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  const int nw = gridDim.x * nwarp, wid = blockIdx.x * nwarp + warp;
  const int per_warp = ceil_div(rows, nw);
  constexpr bool kContig = DIST == IGN_DIST_COSINE;
  const int rstep = kContig ? 1 : nw;
  const int rbeg = kContig ? min(rows, wid * per_warp) : wid, rend = kContig ? min(rows, rbeg + per_warp) : rows;
  float* slot = prow + (size_t)warp * kPoolStages * g.DP;
  int pf_row = rbeg;                                     // prefetch cursor
  auto prefetch_next = [&](int buf) {                    // always commits a group, possibly empty
    if (pf_row < rend) {
      const int r = pf_row;
      pf_row += rstep;
      const float* src = a.dstore + (size_t)r * g.Ts;
      float* dstp = slot + (size_t)buf * g.DP;
      for (int t = lane * 4; t < g.Ts; t += 128) cp_async16_pool(dstp + t, src + t);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  const float eps = g.eps;
  const float q = -eps * eps * kLog2e;
  const int nfull = g.Tw >> 7, tail0 = nfull << 7;                          // nfull + (tail > 0) <= NCH
  const bool vtail = g.Tw - tail0 >= 64;                                    // the tail as one masked float4 chunk
  const int ntail = vtail ? 0 : g.Tw - tail0;                               // windows handled by the scalar sub-chunks
  const int tt = tail0 + lane;
  const int tv0 = tail0 + 4 * lane;                                         // this lane's first window of the masked chunk
  prefetch_next(0);
  prefetch_next(1);
  int buf = 0;
  constexpr int NS = DIST == IGN_DIST_COSINE ? NCH : 1;
  float4 S[NS];
  int sbm = -1;                                          // the group whose factors S holds
  for (int row = rbeg; row < rend; row += rstep, buf = buf == kPoolStages - 1 ? 0 : buf + 1) {
    const int bm = row / g.K, k = row - bm * g.K;
    prefetch_next(buf >= 1 ? buf - 1 : kPoolStages - 1);   // stage (buf + 2) % 3
    asm volatile("cp.async.wait_group 2;" ::: "memory");
    __syncwarp();
    const float* dr = slot + (size_t)buf * g.DP;
    const float4* d4 = reinterpret_cast<const float4*>(dr);
    const int m = bm % g.M, b = bm / g.M;
    const size_t o = ((size_t)b * g.K + k) * g.M + m;
    const float gk = a.g[((size_t)b * a.gK + a.gk0 + k) * g.M + m];
    float sl2 = 0.f;
    int ih = 0;
    if (POOL == IGN_POOL_LTS_MIN) { sl2 = a.dmin[o] * kLog2e; ih = a.argmin[o]; }
    float gdv = 0.f;                                       // GD: + gdv on window idm (the forward's argmin)
    int idm = -1;
    if (GD) { gdv = a.gd[((size_t)b * a.gK + a.gk0 + k) * g.M + m]; idm = a.argmin[o]; }

    // ---- pass 1: exponentials once, (U, V) to registers, soft-max statistics, chunk-wise arg-max
    float4 U[NCH], V[NCH];
    // cosine: the row's window-norm factors are fetched now and used in pass 2 (issued per chunk there, each 16-byte
    // load sat on the critical path: 0.36 ms per group against 0.17 ms for the L1 instantiation)
    const float* s0r = a.st0 + (size_t)bm * a.SP;          // SP % 16 == 0: float4-aligned rows
    const float* s1r = a.st1 + (size_t)bm * a.SP;
    if (DIST == IGN_DIST_COSINE && bm != sbm) {            // once per (sample, channel) group
      sbm = bm;
#pragma unroll
      for (int j = 0; j < NCH; ++j)
        if (j < nfull) S[j] = __ldg(reinterpret_cast<const float4*>(s0r + (j * 32 + lane) * 4));
      if (vtail && tv0 < g.Ts) S[NS - 1] = __ldg(reinterpret_cast<const float4*>(s0r + tv0));   // Ts <= SP
    }
    float Zs = 0.f, S1s = 0.f, pmx = 0.f;
    int jmx = -1;
    auto eval = [&](float d, float& u, float& v) {
      if (POOL == IGN_POOL_RBF_MAX) {
        v = rbf_pprime(d, q);
        const float e = fast_ex2(v);
        Zs += e; S1s = fmaf(e, v, S1s);
        u = e * v * d;
      } else {
        u = fast_ex2(fmaf(d, -kLog2e, sl2));
        v = d;
        Zs += u; S1s = fmaf(u, d, S1s);
      }
    };
#pragma unroll
    for (int j = 0; j < NCH; ++j) {
      U[j] = make_float4(0.f, 0.f, 0.f, 0.f);
      V[j] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (j < nfull) {
        const float4 d = d4[j * 32 + lane];
        eval(d.x, U[j].x, V[j].x); eval(d.y, U[j].y, V[j].y); eval(d.z, U[j].z, V[j].z); eval(d.w, U[j].w, V[j].w);
        if (POOL == IGN_POOL_RBF_MAX) {
          const float m4 = fmaxf(fmaxf(V[j].x, V[j].y), fmaxf(V[j].z, V[j].w));
          if (jmx < 0 || m4 > pmx) { pmx = m4; jmx = j; }
        }
      }
    }
#define IGN_POOL_TAIL1(S, UC, VC)                                                              \
    if ((S) * 32 < ntail && tt + (S) * 32 < g.Tw) {                                            \
      eval(dr[tt + (S) * 32], UC, VC);                                                         \
      if (POOL == IGN_POOL_RBF_MAX) { if (jmx < 0 || VC > pmx) { pmx = VC; jmx = NCH + (S); } } \
    }
    IGN_POOL_TAIL1(0, U[NCH - 1].x, V[NCH - 1].x)
    IGN_POOL_TAIL1(1, U[NCH - 1].y, V[NCH - 1].y)
    IGN_POOL_TAIL1(2, U[NCH - 1].z, V[NCH - 1].z)
    IGN_POOL_TAIL1(3, U[NCH - 1].w, V[NCH - 1].w)
#undef IGN_POOL_TAIL1
    if (vtail && tv0 < g.Tw) {                             // masked float4 tail chunk -> the last register slot
      const float4 d = d4[nfull * 32 + lane];
      float m4;
      eval(d.x, U[NCH - 1].x, V[NCH - 1].x); m4 = V[NCH - 1].x;
      if (tv0 + 1 < g.Tw) { eval(d.y, U[NCH - 1].y, V[NCH - 1].y); m4 = fmaxf(m4, V[NCH - 1].y); }
      if (tv0 + 2 < g.Tw) { eval(d.z, U[NCH - 1].z, V[NCH - 1].z); m4 = fmaxf(m4, V[NCH - 1].z); }
      if (tv0 + 3 < g.Tw) { eval(d.w, U[NCH - 1].w, V[NCH - 1].w); m4 = fmaxf(m4, V[NCH - 1].w); }
      if (POOL == IGN_POOL_RBF_MAX) { if (jmx < 0 || m4 > pmx) { pmx = m4; jmx = 2 * NCH; } }
    }
    float fix;
    if (POOL == IGN_POOL_RBF_MAX) {
      // first arg-max of p (the reference's hard one-hot, Shapelet.py:79): position inside the lane's best chunk, then
      // across lanes (largest p, smallest index).  p' >= 0, so its bit pattern orders like the value.
      int imx = 0x7fffffff;
      if (jmx == 2 * NCH) {                                // inside the masked tail chunk
        const float4 d = d4[nfull * 32 + lane];
        if (tv0 + 3 < g.Tw && rbf_pprime(d.w, q) == pmx) imx = tv0 + 3;
        if (tv0 + 2 < g.Tw && rbf_pprime(d.z, q) == pmx) imx = tv0 + 2;
        if (tv0 + 1 < g.Tw && rbf_pprime(d.y, q) == pmx) imx = tv0 + 1;
        if (rbf_pprime(d.x, q) == pmx) imx = tv0;
      } else if (jmx >= NCH) {
        imx = tt + (jmx - NCH) * 32;
      } else if (jmx >= 0) {
        const int t0 = (jmx * 32 + lane) * 4;
        const float4 d = d4[jmx * 32 + lane];
        if (rbf_pprime(d.w, q) == pmx) imx = t0 + 3;
        if (rbf_pprime(d.z, q) == pmx) imx = t0 + 2;
        if (rbf_pprime(d.y, q) == pmx) imx = t0 + 1;
        if (rbf_pprime(d.x, q) == pmx) imx = t0;
      }
      const unsigned bits = __float_as_uint(pmx);
      const unsigned vmax = __reduce_max_sync(0xffffffffu, bits);
      ih = (int)__reduce_min_sync(0xffffffffu, bits == vmax ? (unsigned)imx : 0x7fffffffu);
      const float dh = dr[ih];
      fix = gk * (-2.f * eps * eps) * (rbf_pprime(dh, q) * (1.f / kLog2e)) * dh;
    } else {
      fix = gk;
    }
    Zs = warp_sum(Zs); S1s = warp_sum(S1s);
    const float invZ = 1.f / Zs, vbar = S1s * invZ;
    const float Kc = POOL == IGN_POOL_RBF_MAX ? gk * (-2.f * eps * eps) * invZ * (1.f / (kLog2e * kLog2e)) : -gk * invZ;

    // ---- pass 2: coefficients from registers, mode factor, 128-bit stores
    const float wst = (DIST == IGN_DIST_PEARSON) ? a.wstat[(size_t)k * g.M + m] : 0.f;
    float* dst = a.coef + (size_t)row * g.Ts;
    float sc0 = 0.f, sc1 = 0.f;
    constexpr bool kStats = DIST == IGN_DIST_COSINE || DIST == IGN_DIST_PEARSON;
#pragma unroll
    for (int j = 0; j < NCH; ++j) {
      if (j < nfull) {
        const int t0 = (j * 32 + lane) * 4;
        float c0 = Kc * U[j].x * (V[j].x - vbar), c1 = Kc * U[j].y * (V[j].y - vbar);
        float c2 = Kc * U[j].z * (V[j].z - vbar), c3 = Kc * U[j].w * (V[j].w - vbar);
        const int hc = ih - t0;
        if ((unsigned)hc < 4u) {
          c0 += hc == 0 ? fix : 0.f; c1 += hc == 1 ? fix : 0.f; c2 += hc == 2 ? fix : 0.f; c3 += hc == 3 ? fix : 0.f;
        }
        if (GD) add_at4(c0, c1, c2, c3, idm, t0, gdv);
        float4 d = make_float4(0.f, 0.f, 0.f, 0.f), s0 = d, s1 = d;
        if (kStats) d = d4[j * 32 + lane];
        if (DIST == IGN_DIST_COSINE) s0 = S[j < NS ? j : 0];
        if (DIST == IGN_DIST_PEARSON) s0 = *reinterpret_cast<const float4*>(s0r + t0);
        if (DIST == IGN_DIST_PEARSON) s1 = *reinterpret_cast<const float4*>(s1r + t0);
        float4 out;
        out.x = pool_emit<DIST>(c0, d.x, s0.x, s1.x, wst, sc0, sc1);
        out.y = pool_emit<DIST>(c1, d.y, s0.y, s1.y, wst, sc0, sc1);
        out.z = pool_emit<DIST>(c2, d.z, s0.z, s1.z, wst, sc0, sc1);
        out.w = pool_emit<DIST>(c3, d.w, s0.w, s1.w, wst, sc0, sc1);
        *reinterpret_cast<float4*>(dst + t0) = out;
      }
    }
#define IGN_POOL_TAIL2(S, UC, VC)                                                              \
    if ((S) * 32 < ntail && tt + (S) * 32 < g.Tw) {                                            \
      const int t = tt + (S) * 32;                                                             \
      float c = Kc * UC * (VC - vbar);                                                         \
      if (t == ih) c += fix;                                                                   \
      if (GD && t == idm) c += gdv;                                                            \
      dst[t] = pool_emit<DIST>(c, kStats ? dr[t] : 0.f, kStats ? s0r[t] : 0.f,                 \
                               DIST == IGN_DIST_PEARSON ? s1r[t] : 0.f, wst, sc0, sc1);        \
    }
    IGN_POOL_TAIL2(0, U[NCH - 1].x, V[NCH - 1].x)
    IGN_POOL_TAIL2(1, U[NCH - 1].y, V[NCH - 1].y)
    IGN_POOL_TAIL2(2, U[NCH - 1].z, V[NCH - 1].z)
    IGN_POOL_TAIL2(3, U[NCH - 1].w, V[NCH - 1].w)
#undef IGN_POOL_TAIL2
    if (vtail && tv0 < g.Ts) {                             // masked float4 tail chunk: pad windows (t >= T') get 0
      const float4 uu = U[NCH - 1], vv = V[NCH - 1];
      float cc[4] = {Kc * uu.x * (vv.x - vbar), Kc * uu.y * (vv.y - vbar), Kc * uu.z * (vv.z - vbar), Kc * uu.w * (vv.w - vbar)};
      const int hc = ih - tv0;
      if ((unsigned)hc < 4u) {
        cc[0] += hc == 0 ? fix : 0.f; cc[1] += hc == 1 ? fix : 0.f; cc[2] += hc == 2 ? fix : 0.f; cc[3] += hc == 3 ? fix : 0.f;
      }
      if (GD) add_at4(cc[0], cc[1], cc[2], cc[3], idm, tv0, gdv);
      float4 d = make_float4(0.f, 0.f, 0.f, 0.f), s0 = d, s1 = d;
      if (kStats) d = d4[nfull * 32 + lane];
      if (DIST == IGN_DIST_COSINE) s0 = S[NS - 1];
      if (DIST == IGN_DIST_PEARSON) { s0 = *reinterpret_cast<const float4*>(s0r + tv0); s1 = *reinterpret_cast<const float4*>(s1r + tv0); }
      float4 out = make_float4(0.f, 0.f, 0.f, 0.f);
      if (tv0 < g.Tw) out.x = pool_emit<DIST>(cc[0], d.x, s0.x, s1.x, wst, sc0, sc1);
      if (tv0 + 1 < g.Tw) out.y = pool_emit<DIST>(cc[1], d.y, s0.y, s1.y, wst, sc0, sc1);
      if (tv0 + 2 < g.Tw) out.z = pool_emit<DIST>(cc[2], d.z, s0.z, s1.z, wst, sc0, sc1);
      if (tv0 + 3 < g.Tw) out.w = pool_emit<DIST>(cc[3], d.w, s0.w, s1.w, wst, sc0, sc1);
      *reinterpret_cast<float4*>(dst + tv0) = out;
    }
    if (!vtail && lane < g.Ts - g.Tw) dst[g.Tw + lane] = 0.f;        // pad windows (at most 3)
    sc0 = warp_sum(sc0);
    if (DIST == IGN_DIST_PEARSON) sc1 = warp_sum(sc1);
    if (lane == 0) { a.rowsc[(size_t)row * 2] = sc0; a.rowsc[(size_t)row * 2 + 1] = sc1; }
    __syncwarp();                                       // everyone is done with this stage before it is refilled
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
}

// ||w - mean|| per (k, m) shapelet row (pearson backward).  One warp per row.
__global__ void __launch_bounds__(256) shapelet_centred_norm_kernel(const float* __restrict__ W,
                                                                   float* __restrict__ wstat, int rows, int L) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float* w = W + (size_t)row * L;
  float s = 0.f;
  for (int l = lane; l < L; l += 32) s += w[l];
  const float mean = warp_sum(s) / (float)L;
  float c2 = 0.f;
  for (int l = lane; l < L; l += 32) { const float v = w[l] - mean; c2 = fmaf(v, v, c2); }
  c2 = warp_sum(c2);
  if (lane == 0) wstat[row] = sqrtf(c2);
}

// L1 only.  Exact ties x == w are impossible for a series row that shares no value with the shapelet block
// it is contracted against; this pre-pass decides that per (sample, channel, shapelet block) with a hash set
// of the block's shapelet values in shared memory, so the hot kernel can take the 2-instruction path.
__global__ void __launch_bounds__(256) tie_check_kernel(const float* __restrict__ xn, const float* __restrict__ W,
                                                        unsigned char* __restrict__ tie, int B, int M, int T, int Tp,
                                                        int K, int L, int KB, int nkb, int hcap, int bsplit) {
  extern __shared__ unsigned hset[];                       // [hcap] exact set, then [kTieBitmapWords] bitmap filter
  unsigned* bitmap = hset + hcap;
  const int m = blockIdx.x, kblk = blockIdx.y;
  const int k0 = kblk * KB;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  for (int i = threadIdx.x; i < hcap; i += blockDim.x) hset[i] = kHashEmpty;
  for (int i = threadIdx.x; i < kTieBitmapWords; i += blockDim.x) bitmap[i] = 0u;
  __syncthreads();
  const unsigned mask = hcap - 1;
  for (int i = threadIdx.x; i < KB * L; i += blockDim.x) {
    const int hk = i / L, l = i - hk * L;
    if (k0 + hk >= K) continue;
    const unsigned key = hash_key(__ldg(W + ((size_t)(k0 + hk) * M + m) * L + l));
    const unsigned hb = (key * 0x85EBCA6Bu) >> (32 - kTieBitmapLog2), hb2 = (key * 0xC2B2AE35u) >> (32 - kTieBitmapLog2);
    atomicOr(&bitmap[hb >> 5], 1u << (hb & 31));
    atomicOr(&bitmap[hb2 >> 5], 1u << (hb2 & 31));
    unsigned h = hash_slot(key, mask);
    while (true) {
      const unsigned old = atomicCAS(&hset[h], kHashEmpty, key);
      if (old == kHashEmpty || old == key) break;
      h = (h + 1) & mask;
    }
  }
  __syncthreads();
  const int per = ceil_div(B, bsplit);
  const int bbeg = blockIdx.z * per, bend = min(B, bbeg + per);
  for (int b = bbeg + warp; b < bend; b += nwarp) {
    const float4* xr = reinterpret_cast<const float4*>(xn + ((size_t)b * M + m) * Tp);   // pad samples are 0: a
    int hit = 0;                                                                          // spurious hit is harmless
    // eight 16-byte loads in flight per lane (a whole row for T <= 1024): with one load per lane the scan was bound by
    // DRAM latency (1.2 TB/s); indices past the row end are clamped — re-testing a sample is harmless
    constexpr int UN = 8;
    const int nv = Tp / 4;
    for (int t4 = lane; t4 < nv; t4 += 32 * UN) {
      float4 vq[UN];
#pragma unroll
      for (int u = 0; u < UN; ++u) vq[u] = __ldg(xr + min(t4 + u * 32, nv - 1));
#pragma unroll
      for (int u = 0; u < UN; ++u) {
        const float vv[4] = {vq[u].x, vq[u].y, vq[u].z, vq[u].w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const unsigned key = hash_key(vv[e]);
          const unsigned hb = (key * 0x85EBCA6Bu) >> (32 - kTieBitmapLog2), hb2 = (key * 0xC2B2AE35u) >> (32 - kTieBitmapLog2);
          if ((bitmap[hb >> 5] >> (hb & 31)) & (bitmap[hb2 >> 5] >> (hb2 & 31)) & 1u) {   // rare: confirm in the exact set
            unsigned h = hash_slot(key, mask);
            while (true) {
              const unsigned q = hset[h];
              if (q == key) { hit = 1; break; }
              if (q == kHashEmpty) break;
              h = (h + 1) & mask;
            }
          }
        }
      }
    }
    hit = __any_sync(0xffffffffu, hit);
    if (lane == 0) tie[((size_t)b * M + m) * nkb + kblk] = (unsigned char)hit;
  }
}

// ---- contraction kernel: dW partials from the coefficients and the series (pure FP32-pipe work) ----
template <int OP, int LT>
// 8-lag tiles fit 64 registers (four 256-thread CTAs per SM: L = 300 2.68 -> 2.55 ms); 10-lag tiles spill there and
// run slower with four CTAs than with three at 80 registers (L = 100 1.15 -> 1.19 ms)
__global__ void __launch_bounds__(kMaxThreads, LT == 8 ? 4 : 3) shapelet_bwd_kernel(const Geo g, const BwdArgs a) {
  extern __shared__ __align__(16) float smem[];
  const int m = blockIdx.x;
  const int kblk = blockIdx.y / a.nlb, lblk = blockIdx.y - kblk * a.nlb;
  const int k0 = kblk * g.KB;
  const int chunk = blockIdx.z;
  int bbeg, bend;
  chunk_range(g, chunk, bbeg, bend);
  const int nthr = blockDim.x;

  const int ntl_all = g.s * g.LQ / LT;                    // l-tiles over all residues
  const int lt_beg = lblk * a.tlb;
  const int ntl = min(a.tlb, ntl_all - lt_beg);           // l-tiles of this CTA
  const int nslot = g.NB * a.nseg;
  const int nitem = nslot * ntl * g.KB;                   // <= blockDim.x by construction

  // series and coefficient rows are double-buffered and prefetched with cp.async one pass ahead (strided groups
  // de-interleave the series with 4-byte copies); single-buffered only when two buffers do not fit shared memory
  const bool dbuf = g.dbuf != 0;
  const int xs_sz = g.NB * g.s * g.XQ;
  const int cb_sz = max(g.NB * g.KB * g.CP, dbuf ? 0 : kMaxThreads * LT);
  float* xs0 = smem;
  float* cb0 = xs0 + (dbuf ? 2 : 1) * xs_sz;
  if (dbuf) {   // zero once: pad columns (series tail, DP - Ts) are never written by the prefetch
    for (int i = threadIdx.x; i < 2 * xs_sz; i += nthr) xs0[i] = 0.f;
    for (int i = threadIdx.x; i < 2 * cb_sz; i += nthr) cb0[i] = 0.f;
  }

  // this thread's fixed tile: LT lags of one shapelet, one (sample slot, t-segment)
  const bool active = threadIdx.x < nitem;
  int lt = 0, kl = 0, seg = 0, bl = 0;
  if (active) {
    int it = threadIdx.x;          // shapelet index fastest: neighbouring lanes share the x address (broadcast)
    kl = it % g.KB; it /= g.KB;
    lt = it % ntl; it /= ntl;
    seg = it % a.nseg; bl = it / a.nseg;
  }
  const int ltg = lt_beg + lt;
  const int tiles_per_res = g.LQ / LT;
  const int r = ltg / tiles_per_res, q0 = (ltg - r * tiles_per_res) * LT;
  const int seg_len = round_up(ceil_div(g.DP, a.nseg), 4);
  const int ta = min(seg * seg_len, g.DP), tb = min(ta + seg_len, g.DP);

  float acc[LT], wreg[LT];
#pragma unroll
  for (int i = 0; i < LT; ++i) { acc[i] = 0.f; wreg[i] = 0.f; }
  if (OP == OP_L1 && active && k0 + kl < g.K) {           // this thread's LT shapelet values, once per CTA, straight from global
    const float* wrow = a.W + ((size_t)(k0 + kl) * g.M + m) * g.L;
#pragma unroll
    for (int i = 0; i < LT; ++i) {
      const int l = (q0 + i) * g.s + r;
      wreg[i] = l < g.L ? __ldg(wrow + l) : 0.f;
    }
  }
  __syncthreads();

  auto prefetch = [&](int b0, int buf) {
    const int nb = min(g.NB, bend - b0);
    float* xd = xs0 + buf * xs_sz;
    float* cd = cb0 + buf * cb_sz;
    // row by row (a handful of rows per pass): no index division per 16-byte copy — the flat loop spent ~40 issue
    // slots per copy, 5 % of the kernel's instructions at L = 100
    const int xrow = g.Tp / 4, crow = g.Ts / 4;
    const int kvalid = min(g.KB, g.K - k0);
    for (int rbl = 0; rbl < nb; ++rbl) {
      const float* xsrc = a.xn + ((size_t)(b0 + rbl) * g.M + m) * g.Tp;
      if (g.s == 1) {
        float* xdst = xd + rbl * g.XQ;
        for (int c = threadIdx.x; c < xrow; c += nthr) cp_async16(xdst + c * 4, xsrc + c * 4);
      } else {                                          // sample t -> residue row t % s, slot t / s
        float* xdst = xd + (size_t)rbl * g.s * g.XQ;
        int q = threadIdx.x / g.s, r = threadIdx.x - q * g.s;
        const int dq = nthr / g.s, dr = nthr - dq * g.s;
        for (int t = threadIdx.x; t < g.T; t += nthr) {
          cp_async4(xdst + r * g.XQ + q, xsrc + t);
          q += dq; r += dr;
          if (r >= g.s) { r -= g.s; ++q; }
        }
      }
      const float* csrc = a.coef + (((size_t)(b0 + rbl) * g.M + m) * g.K + k0) * g.Ts;
      float* cdst = cd + (size_t)rbl * g.KB * g.CP;
      for (int rkl = 0; rkl < kvalid; ++rkl)
        for (int c = threadIdx.x; c < crow; c += nthr) cp_async16(cdst + rkl * g.CP + c * 4, csrc + (size_t)rkl * g.Ts + c * 4);
    }
  };

  int buf = 0;
  if (dbuf && bbeg < bend) prefetch(bbeg, 0);
  for (int b0 = bbeg; b0 < bend; b0 += g.NB) {
    const int nb = min(g.NB, bend - b0);
    if (dbuf) {
      cp_async_commit_wait_all();
      __syncthreads();                    // pass data visible; everyone is done with the other buffer
      if (b0 + g.NB < bend) prefetch(b0 + g.NB, buf ^ 1);
    } else {
      __syncthreads();
      load_series(g, a.xn, nullptr, 0, m, b0, nb, xs0, nullptr);
      const int rowv = g.DP / 4, tot = g.NB * g.KB * rowv;
      for (int i = threadIdx.x; i < tot; i += nthr) {
        const int row = i / rowv, c4 = (i - row * rowv) * 4;
        const int rbl = row / g.KB, rkl = row - rbl * g.KB;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (rbl < nb && k0 + rkl < g.K && c4 < g.Ts)
          v = *reinterpret_cast<const float4*>(a.coef + (((size_t)(b0 + rbl) * g.M + m) * g.K + k0 + rkl) * g.Ts + c4);
        *reinterpret_cast<float4*>(cb0 + (size_t)row * g.CP + c4) = v;
      }
      __syncthreads();
    }
    const float* xs = xs0 + buf * xs_sz;
    const float* cbuf = cb0 + buf * cb_sz;
    // ---- contraction over windows, sliding along t with a ring of LT + 4 registers of x: step j of a revolution
    // (4 windows) reads the ring at base 4 j mod RING and refills the four slots it frees
    if (active && bl < nb && ta < tb && k0 + kl < g.K) {
      const float* xr = xs + ((size_t)bl * g.s + r) * g.XQ + q0;
      const float* cb = cbuf + ((size_t)bl * g.KB + kl) * g.CP;
      const bool exact = OP == OP_L1 && (a.tie == nullptr || a.tie[((size_t)(b0 + bl) * g.M + m) * g.nkb + kblk] != 0);
      constexpr int RING = LT + 4;
      constexpr int NSTEP = RING % 4 == 0 ? RING / 4 : RING / 2;    // steps per ring revolution: 3 (LT = 8), 7 (LT = 10)
      static_assert(LT % 2 == 0 && (4 * NSTEP) % RING == 0, "ring revolution");
      float xv[RING];
      if (LT % 4 == 0) {
#pragma unroll
        for (int i = 0; i < LT; i += 4) {
          const float4 v = *reinterpret_cast<const float4*>(xr + ta + i);
          xv[i] = v.x; xv[i + 1] = v.y; xv[i + 2] = v.z; xv[i + 3] = v.w;
        }
      } else {                                          // q0 is a multiple of LT: 8-byte aligned only
#pragma unroll
        for (int i = 0; i < LT; i += 2) {
          const float2 v = *reinterpret_cast<const float2*>(xr + ta + i);
          xv[i] = v.x; xv[i + 1] = v.y;
        }
      }
      auto step = [&](auto ex, int base, int tq) {       // `base` is a constant after unrolling: xv stays in registers
        constexpr bool EX = decltype(ex)::value;
        float n0, n1, n2, n3;
        if (LT % 4 == 0) {
          const float4 nx = *reinterpret_cast<const float4*>(xr + tq + LT);
          n0 = nx.x; n1 = nx.y; n2 = nx.z; n3 = nx.w;
        } else {
          const float2 na = *reinterpret_cast<const float2*>(xr + tq + LT);
          const float2 nb2 = *reinterpret_cast<const float2*>(xr + tq + LT + 2);
          n0 = na.x; n1 = na.y; n2 = nb2.x; n3 = nb2.y;
        }
        xv[(base + LT) % RING] = n0; xv[(base + LT + 1) % RING] = n1;
        xv[(base + LT + 2) % RING] = n2; xv[(base + LT + 3) % RING] = n3;
        const float4 c4 = *reinterpret_cast<const float4*>(cb + tq);
        const float4 h4 = make_float4(0.5f * c4.x, 0.5f * c4.y, 0.5f * c4.z, 0.5f * c4.w);
#pragma unroll
        for (int i = 0; i < LT; ++i) {
          acc[i] = bwd_op<OP, EX>(acc[i], c4.x, h4.x, xv[(base + i + 0) % RING], wreg[i]);
          acc[i] = bwd_op<OP, EX>(acc[i], c4.y, h4.y, xv[(base + i + 1) % RING], wreg[i]);
          acc[i] = bwd_op<OP, EX>(acc[i], c4.z, h4.z, xv[(base + i + 2) % RING], wreg[i]);
          acc[i] = bwd_op<OP, EX>(acc[i], c4.w, h4.w, xv[(base + i + 3) % RING], wreg[i]);
        }
      };
      auto sweep = [&](auto ex) {
        int t = ta;
        for (; t + 4 * NSTEP <= tb; t += 4 * NSTEP) {
#pragma unroll
          for (int j = 0; j < NSTEP; ++j) step(ex, (4 * j) % RING, t + 4 * j);
        }
#pragma unroll
        for (int j = 0; j < NSTEP - 1; ++j)             // segment lengths are multiples of 4
          if (t + 4 * (j + 1) <= tb) step(ex, (4 * j) % RING, t + 4 * j);
      };
      if (exact) sweep(std::true_type{}); else sweep(std::false_type{});
    }
    if (dbuf) buf ^= 1;
  }

  // ---- fixed-order reduction over (sample slot, t-segment), then one partial per chunk ----
  if (dbuf) cp_async_commit_wait_all();
  __syncthreads();
  float* red = cb0;
  if (active) {
    const int slot = bl * a.nseg + seg;
    float* dst = red + (((size_t)(kl * ntl + lt)) * nslot + slot) * LT;
#pragma unroll
    for (int i = 0; i < LT; ++i) dst[i] = acc[i];
  }
  __syncthreads();
  const int nout = g.KB * ntl * LT;
  for (int oidx = threadIdx.x; oidx < nout; oidx += nthr) {
    const int i = oidx % LT;
    const int tile = oidx / LT;                   // kl*ntl + lt
    const int okl = tile / ntl, olt = tile - okl * ntl;
    const float* src = red + (size_t)tile * nslot * LT + i;
    float s = 0.f;
    for (int sl = 0; sl < nslot; ++sl) s += src[(size_t)sl * LT];
    const int oltg = lt_beg + olt;
    const int orr = oltg / tiles_per_res, oq = (oltg - orr * tiles_per_res) * LT + i;
    const int l = oq * g.s + orr;
    const int k = k0 + okl;
    if (k < g.K && l < g.L && oq < (g.L - orr + g.s - 1) / g.s)
      a.part[(((size_t)chunk * g.K + k) * g.M + m) * g.L + l] = s;
  }
}

// dW[k,m,:] from the per-chunk partial contractions and the per-row scalars.  One warp per (k,m) row and block of 128
// lags (gridDim.y blocks); the chunk partials are summed in chunk order, eight loads in flight (one dependent load
// per chunk left L = 500 with its 29 chunks at 0.5 TB/s).
__global__ void __launch_bounds__(256) shapelet_bwd_finalize(const float* __restrict__ W,
                                                            const float* __restrict__ part,
                                                            const float* __restrict__ rowsc,
                                                            float* __restrict__ dW, int B, int K, int M, int L,
                                                            int nchunk, int dist) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= K * M) return;
  const int k = row / M, m = row - k * M;
  const float* w = W + (size_t)row * L;
  float s0 = 0.f, s1 = 0.f;
  for (int b = lane; b < B; b += 32) {            // fixed order: bit-reproducible
    const size_t r = (((size_t)b * M + m) * K + k) * 2;
    s0 += rowsc[r]; s1 += rowsc[r + 1];
  }
  s0 = warp_sum(s0); s1 = warp_sum(s1);
  float mean = 0.f, inv_nw = 0.f;
  if (dist == IGN_DIST_COSINE || dist == IGN_DIST_PEARSON) {
    float a = 0.f, b2 = 0.f;
    for (int l = lane; l < L; l += 32) { float v = w[l]; a += v; b2 = fmaf(v, v, b2); }
    a = warp_sum(a); b2 = warp_sum(b2);
    mean = a / (float)L;
    inv_nw = 1.f / fmaxf(sqrtf(b2), 1e-8f);
  }
  const float Lf = (float)L;
  const int lbeg = blockIdx.y * 128, lend = min(L, lbeg + 128);
  for (int l = lbeg + lane; l < lend; l += 32) {
    float G = 0.f;
    const float* pl = part + (size_t)row * L + l;
    const size_t cstride = (size_t)K * M * L;
    for (int c = 0; c < nchunk; c += 8) {
      float v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = c + u < nchunk ? __ldg(pl + (size_t)(c + u) * cstride) : 0.f;
#pragma unroll
      for (int u = 0; u < 8; ++u) G += v[u];         // chunk order; + 0.f past the end changes nothing
    }
    float o;
    if (dist == IGN_DIST_L1) o = -(2.f * G - s0) / Lf;
    else if (dist == IGN_DIST_SQL2) o = (2.f / Lf) * (w[l] * s0 - G);
    else if (dist == IGN_DIST_COSINE) o = -G * inv_nw + w[l] * s0 * inv_nw * inv_nw;
    else o = -(G - s0) + (w[l] - mean) * s1;
    dW[(size_t)row * L + l] = o;
  }
}

// ------------------------------------------------------------------------------------------------
// host-side planning
// ------------------------------------------------------------------------------------------------
int pick_kk(int K) {
  if (K % 5 == 0) return 5;
  if (K % 4 == 0 || K < 4) return 4;
  return (round_up(K, 5) - K <= round_up(K, 4) - K) ? 5 : 4;
}

bool base_geo(const ign_shapelet_desc& d, Geo& g) {
  g.B = d.B; g.M = d.M; g.T = d.T; g.Tp = d.Tp; g.K = d.K; g.L = d.L; g.s = d.stride;
  g.Tw = num_windows(d.T, d.L, d.stride);
  g.Ts = round_up(g.Tw, 4);
  g.DP = round_up(g.Tw, 8);
  g.CP = g.DP + ((12 - g.DP % 32) + 32) % 32;
  const int Lq = ceil_div(d.L, d.stride);
  g.LQ = round_up(Lq, 8);
  g.LT = 8;
  g.XQ = round_up(max(g.DP + g.LQ + 8, ceil_div(d.T, d.stride) + 8), 4);   // covers t + LT + 3 + q0 < DP + LQ
  g.KK = pick_kk(d.K);
  g.dist = d.dist; g.pool = d.pool; g.eps = d.eps;
  return g.Tw > 0;
}

// Resident CTAs per SM of `kern` at this block size and dynamic shared memory (host API, cached; IGN_DEBUG_PLAN output).
template <typename Kern>
int occupancy(Kern kern, int threads, size_t smem) {
  static std::mutex mu;
  static std::map<std::tuple<const void*, int, size_t>, int> cache;
  const auto key = std::make_tuple(reinterpret_cast<const void*>(kern), threads, smem);
  std::lock_guard<std::mutex> lock(mu);
  auto it = cache.find(key);
  if (it != cache.end()) return it->second;
  int n = 0;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess ||
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kern, threads, smem) != cudaSuccess) {
    cudaGetLastError();
    n = 1;
  }
  n = max(n, 1);
  cache[key] = n;
  return n;
}

// Batch chunking: about kTargetCtasPerSm CTAs per SM, in balanced chunks (sizes differ by at most one pass).
// Measured on B200 (profiles/r1e_plan_sweep.txt): fewer, longer CTAs sized to an exact number of resident "waves" are
// SLOWER (L1 backward 11.9 -> 12.6 ms at ~3 waves) — a CTA that is alone on its SM runs several times faster, so a
// short last wave costs little, while many CTAs in different phases hide each other's pass barriers.
constexpr int kTargetCtasPerSm = 24;
void plan_chunks(Geo& g, int ctas_per_chunk, int NB) {
  static const int target_env = getenv("IGN_PLAN_CTAS_PER_SM") ? atoi(getenv("IGN_PLAN_CTAS_PER_SM")) : 0;
  const int target = (target_env > 0 ? target_env : kTargetCtasPerSm) * sm_count();
  const int units = ceil_div(g.B, NB);
  int nc = max(1, ceil_div(target, max(1, ctas_per_chunk)));
  nc = min(nc, units);
  g.nchunk = nc; g.cbase = units / nc; g.cextra = units % nc;
}

size_t fwd_smem_floats(const Geo& g, int NB, int KB, int ntile) {
  const size_t mult = g.dbuf ? 2 : 1;         // series / statistics rows double buffered
  size_t f = mult * (size_t)NB * g.s * g.XQ + (size_t)KB * g.s * g.LQ + KB + (size_t)2 * NB * KB * ntile;
  if (g.dist != IGN_DIST_L1) f += mult * (size_t)NB * g.DP;
  return f + 4;                                // alignment slack of the second buffers
}

struct FwdPlan { int threads; size_t smem_bytes; };
using FwdKernel = void (*)(const Geo, const FwdArgs);
using BwdKernel = void (*)(const Geo, const BwdArgs);

bool plan_fwd(Geo& g, int TT, FwdPlan& fp) {
  g.dbuf = 0;
  const size_t cap_soft = 111 * 1024, cap_hard = (size_t)max_optin_smem() - 1024;   // two CTAs per SM
  const int Kpad = round_up(g.K, g.KK);
  const int ntile = g.DP / TT;
  int KB = min(Kpad, 8 * g.KK);
  while (KB > g.KK && fwd_smem_floats(g, 1, KB, ntile) * 4 > cap_soft) KB -= g.KK;
  if (fwd_smem_floats(g, 1, KB, ntile) * 4 > cap_hard) return false;
  // (no balancing of the shapelet blocks here, unlike plan_bwd: the items of a short last block are whole rounds of
  //  the item loop that are simply not run — K = 100 as 40 + 40 + 20 measured 10 % FASTER at L = 500 than 35 + 35 + 30)
  const size_t cap = fwd_smem_floats(g, 1, KB, ntile) * 4 > cap_soft ? cap_hard : cap_soft;
  const int nkc = KB / g.KK;
  // resident rows: fill whole rounds of the thread block (idle lanes in the last round are the waste).  Double
  // buffering the rows is taken only when it costs no lane efficiency (it halves the rows that fit).
  int best = 1, bthr = 32; double beff = -1.0;
  auto search = [&](int& obest, int& othr, double& oeff) {
    obest = 1; othr = 32; oeff = -1.0;
    for (int NB = 1; NB <= min(g.B, 64); ++NB) {
      if (fwd_smem_floats(g, NB, KB, ntile) * 4 > cap) break;
      const int nitem = NB * ntile * nkc;
      static const int thr_env = getenv("IGN_FWD_MAXTHR") ? atoi(getenv("IGN_FWD_MAXTHR")) : 0;   // experiments
      const int thr = min(thr_env > 0 ? thr_env : kMaxThreads, round_up(nitem, 32));
      // CTAs whose warp count is not a multiple of four load the SM's schedulers unevenly (see plan_bwd_cand)
      static const double kWarpShape[4] = {1.0, 0.80, 0.95, 0.87};
      const double e = (double)nitem / (double)(ceil_div(nitem, thr) * thr) * kWarpShape[(thr / 32) & 3];
      if (e > oeff + 0.01) { oeff = e; obest = NB; othr = thr; }
    }
  };
  g.dbuf = 0;
  search(best, bthr, beff);
  {
    int b2, t2; double e2;
    g.dbuf = 1;
    search(b2, t2, e2);
    if (fwd_smem_floats(g, 1, KB, ntile) * 4 <= cap && e2 >= beff - 0.015) { best = b2; bthr = t2; beff = e2; }
    else g.dbuf = 0;
  }
  g.KB = KB; g.nkb = ceil_div(Kpad, KB); g.NB = best;
  fp.threads = bthr;
  fp.smem_bytes = fwd_smem_floats(g, best, KB, ntile) * 4;
  plan_chunks(g, g.M * g.nkb, best);
  return true;
}

struct BwdPlan { int nseg, nlb, tlb, nchunk, threads, hcap; size_t smem_bytes; };

int bwd_hash_cap(const Geo& g, int KB) {
  if (g.dist != IGN_DIST_L1) return 0;
  size_t need = 2 * (size_t)KB * g.L, cap = 256;   // load factor <= 1/2; the set is probed only after a filter hit
  while (cap < need) cap <<= 1;
  return cap <= 32768 ? (int)cap : 0;      // larger slabs: skip the check, always take the exact path (128 KB + 32 KB smem)
}

size_t bwd_smem_floats(const Geo& g, int NB, int KB) {
  const size_t mult = g.dbuf ? 2 : 1;         // rows double-buffered
  const size_t xs = (size_t)NB * g.s * g.XQ, cb = (size_t)NB * KB * g.CP;
  size_t cbt = mult * cb;
  if (cbt < (size_t)kMaxThreads * g.LT) cbt = (size_t)kMaxThreads * g.LT;
  return mult * xs + cbt;
}

// One candidate (lag tile LT, shapelet block KB).  `cost` = estimated seconds for contraction + tie pre-check.
bool plan_bwd_cand(Geo& g, BwdPlan& bp, int LT, int KB, double& cost) {
  const size_t cap = (size_t)max_optin_smem() - 1024;
  const size_t cap_soft = 56 * 1024;     // more than one series row per pass only while >= 4 CTAs per SM still fit
  g.LT = LT;
  g.LQ = round_up(ceil_div(g.L, g.s), LT);
  g.XQ = round_up(max(g.DP + g.LQ + 8, ceil_div(g.T, g.s) + 8), 4);   // covers t + LT + 3 + q0 < DP + LQ
  const int ntl_all = g.s * g.LQ / LT;
  g.dbuf = 1;
  if (bwd_smem_floats(g, 1, KB) * 4 > cap) {          // very long series: one buffer, loads between two barriers
    g.dbuf = 0;
    if (bwd_smem_floats(g, 1, KB) * 4 > cap) return false;
  }
  // shapelet block and lag block: KB * tlb threads cover one (sample, segment) slot
  int tlb = min(ntl_all, kMaxThreads / KB);
  const int nlb = ceil_div(ntl_all, tlb);
  tlb = ceil_div(ntl_all, nlb);          // balance the lag blocks
  const int per_slot = tlb * KB;
  const int slots = max(1, kMaxThreads / per_slot);
  // rows per pass x t-segments: fill the thread block (idle lanes in the last warp are the waste).  Scoring candidates
  // by the scheduler balance of the resident warps as well (tools/ubench_f32x2.cu shows the effect in isolation: 21 or
  // 25 warps per SM run at 7/8 of the rate of 20 or 24) picked 160 threads x 4 CTAs over 224 x 3 at L=100 and measured
  // 3.5 % SLOWER (1.65 vs 1.59 ms) — the longer t-segments lose more than the balance gains — so it is not used.
  int bestNB = 1, bestSeg = 1; double beff = -1.0;
  for (int NB = 1; NB <= min(min(g.B, slots), 16); ++NB) {
    if (bwd_smem_floats(g, NB, KB) * 4 > (NB == 1 ? cap : cap_soft)) break;
    int nseg = max(1, slots / NB);
    nseg = min(nseg, max(1, g.DP / 48));             // keep segments >= 48 windows
    const int nitem = NB * nseg * per_slot;
    const double e = (double)nitem / (double)round_up(nitem, 32) + 1e-3 * NB;   // prefer more rows per pass on ties
    if (e > beff + 0.01) { beff = e; bestNB = NB; bestSeg = nseg; }
  }
  g.KB = KB; g.nkb = ceil_div(g.K, KB); g.NB = bestNB;
  bp.nseg = bestSeg; bp.nlb = nlb; bp.tlb = tlb;
  bp.threads = round_up(bestNB * bestSeg * per_slot, 32);
  bp.hcap = bwd_hash_cap(g, KB);
  bp.smem_bytes = bwd_smem_floats(g, bestNB, KB) * 4;
  plan_chunks(g, g.M * g.nkb * nlb, bestNB);
  bp.nchunk = g.nchunk;
  // Estimated time.  Useful share of the launched lane x lag slots: idle lanes of the last warp, lags padded to the
  // tile, shapelet slots of a short last block (K = 10 in blocks of 3 is 10 of 12).  Splitting the lag axis over CTAs
  // costs more than its lane count says (T = 4000, L = 2000, K = 10: 14.3 ms in blocks of 5 x 4 lag blocks against
  // 11.9 ms in blocks of 1 with every lag in one CTA), fewer than 16 resident warps do not hide the pass barriers, and
  // every shapelet block pays one tie pre-check scan of the series (L1).
  const int lags_done = g.s == 1 ? nlb * tlb * LT : g.s * g.LQ;
  double eff = (double)(bestNB * bestSeg * per_slot) / bp.threads * (double)g.L / (double)lags_done *
               (double)g.K / (double)(g.nkb * KB);
  if (nlb > 1) eff *= 0.83;
  // CTAs whose warp count is not a multiple of four load the SM's four schedulers unevenly (measured at equal lane
  // efficiency, T = 2000, L = 600, K = 10: 5-warp CTAs 21.4 TFLOP/s, 8-warp CTAs 26.7; config 2, L = 100: 7 warps 14 %
  // below what their lane count predicts; 6 warps ~5 %)
  static const double kWarpShape[4] = {1.0, 0.80, 0.95, 0.87};
  eff *= kWarpShape[(bp.threads / 32) & 3];
  // one FFMA per element leaves the cross-term form closer to the shared-memory limit: lanes of one shapelet block
  // share (broadcast) the series reads, so small blocks cost it more than they cost L1
  if (g.dist != IGN_DIST_L1) eff *= 0.88 + 0.03 * min(KB, 4);
  const int ctas = max(1, min((int)(((size_t)max_smem_per_sm()) / (bp.smem_bytes + 1024)), 65536 / ((LT == 8 ? 64 : 80) * bp.threads)));
  const double warps = (double)ctas * bp.threads / 32.0;
  if (warps < 16.0) eff *= warps / 16.0;
  const double E = (double)g.B * g.M * g.K * g.Tw * g.L;
  cost = 2.0 * E / (25e12 * eff);
  if (g.dist == IGN_DIST_L1) {
    if (bp.hcap) cost += (double)g.nkb * g.B * g.M * g.Tp * 4.0 / 3.4e12;
    else cost *= 2.0;                                  // no pre-check (block too large for the hash set): always the exact 4-instruction path
  }
  return true;
}

// Lag tile (8, 10 or 12 lags per thread) and shapelet block (1..8) by estimated time; on ties the larger block (fewer tie
// scans, more reuse of a staged series row).  IGN_BWD_LT=8|10|12 and IGN_BWD_KB=n force one (experiments).
bool plan_bwd(Geo& g, BwdPlan& bp) {
  static const int lt_env = getenv("IGN_BWD_LT") ? atoi(getenv("IGN_BWD_LT")) : 0;
  static const int kb_env = getenv("IGN_BWD_KB") ? atoi(getenv("IGN_BWD_KB")) : 0;
  bool found = false; double best = 0.0;
  Geo gb = g; BwdPlan bb{};
  for (int KB = min(g.K, 8); KB >= 1; --KB) {
    if (kb_env > 0 && KB != min(g.K, kb_env)) continue;
    if (kb_env <= 0 && ceil_div(g.K, ceil_div(g.K, KB)) != KB) continue;   // only balanced block sizes (K = 10: 8, 7, 6 are 5 + 5 anyway)
    for (int LT = 8; LT <= 12; LT += 2) {
      if (lt_env != 0 && LT != lt_env) continue;
      Geo gc = g; BwdPlan bc{}; double c = 0.0;
      if (!plan_bwd_cand(gc, bc, LT, KB, c)) continue;
      if (!found || c < best * 0.99) { found = true; best = c; gb = gc; bb = bc; }
    }
  }
  if (found) { g = gb; bp = bb; }
  return found;
}

template <typename Kern>
int set_smem(Kern kern, size_t bytes) {
  IGN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  return IGN_OK;
}

int run_fwd(FwdKernel kern, const Geo& g, const FwdArgs& a, const FwdPlan& fp, cudaStream_t st) {
  int rc = set_smem(kern, fp.smem_bytes);
  if (rc) return rc;
  dim3 grid(g.M, g.nkb, g.nchunk);
  kern<<<grid, fp.threads, fp.smem_bytes, st>>>(g, a);
  IGN_CUDA(cudaGetLastError());
  return IGN_OK;
}

int run_bwd(BwdKernel kern, const Geo& g, const BwdArgs& a, const BwdPlan& bp, cudaStream_t st) {
  int rc = set_smem(kern, bp.smem_bytes);
  if (rc) return rc;
  dim3 grid(g.M, g.nkb * bp.nlb, bp.nchunk);
  kern<<<grid, bp.threads, bp.smem_bytes, st>>>(g, a);
  IGN_CUDA(cudaGetLastError());
  return IGN_OK;
}

FwdKernel fwd_kernel(bool l1, int KK, int TT) {
  if (l1) {
    if (KK == 5) return TT == 8 ? shapelet_fwd_kernel<OP_L1, 5, 8> : shapelet_fwd_kernel<OP_L1, 5, 4>;
    return TT == 8 ? shapelet_fwd_kernel<OP_L1, 4, 8> : shapelet_fwd_kernel<OP_L1, 4, 4>;
  }
  if (KK == 5) return TT == 8 ? shapelet_fwd_kernel<OP_DOT, 5, 8> : shapelet_fwd_kernel<OP_DOT, 5, 4>;
  return TT == 8 ? shapelet_fwd_kernel<OP_DOT, 4, 8> : shapelet_fwd_kernel<OP_DOT, 4, 4>;
}

BwdKernel bwd_kernel(int dist, int LT) {
  if (LT == 10) return dist == IGN_DIST_L1 ? shapelet_bwd_kernel<OP_L1, 10> : shapelet_bwd_kernel<OP_DOT, 10>;
  if (LT == 12) return dist == IGN_DIST_L1 ? shapelet_bwd_kernel<OP_L1, 12> : shapelet_bwd_kernel<OP_DOT, 12>;
  return dist == IGN_DIST_L1 ? shapelet_bwd_kernel<OP_L1, 8> : shapelet_bwd_kernel<OP_DOT, 8>;
}

bool debug_plan_on() {
  static const bool on = getenv("IGN_DEBUG_PLAN") != nullptr;
  return on;
}

void debug_plan(const char* what, const Geo& g, int threads, size_t smem, int occ, int extra0, int extra1) {
  fprintf(stderr, "[ign plan] %s L=%d Tw=%d K=%d: threads=%d smem=%zu occ=%d NB=%d KB=%d nkb=%d nchunk=%d (base %d, +1 x %d) grid=%d waves=%.2f  [%d %d]\n",
          what, g.L, g.Tw, g.K, threads, smem, occ, g.NB, g.KB, g.nkb, g.nchunk, g.cbase, g.cextra,
          g.M * g.nkb * g.nchunk * max(1, extra1), (double)g.M * g.nkb * g.nchunk * max(1, extra1) / (sm_count() * occ), extra0, extra1);
}

// ---- optional per-phase CUDA-event timing of the backward (bench.py's per-kernel rooflines) ----
enum { PH_POOL = 0, PH_TIE, PH_CONTRACT, PH_FINALIZE, PH_COUNT };
struct PhaseRec { int phase; cudaEvent_t e0, e1; };
std::mutex g_phase_mu;
bool g_phase_on = false;
std::vector<PhaseRec> g_phase;
struct PhaseScope {
  cudaStream_t st; cudaEvent_t e1 = nullptr;
  PhaseScope(int phase, cudaStream_t s) : st(s) {
    std::lock_guard<std::mutex> lock(g_phase_mu);
    if (!g_phase_on) return;
    cudaEvent_t e0;
    if (cudaEventCreate(&e0) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess) { e1 = nullptr; return; }
    cudaEventRecord(e0, st);
    g_phase.push_back({phase, e0, e1});
  }
  ~PhaseScope() { if (e1) cudaEventRecord(e1, st); }
};

}  // namespace

int launch_shapelet_fwd_simt(const ign_shapelet_desc& d, const float* xn, const float* st0,
                             const float* W, const float* thr, float* p, float* dmin,
                             int* argmin, float* dstore, cudaStream_t st) {
  Geo g;
  if (!base_geo(d, g)) { set_error("shapelet_forward: T=%d < L=%d (unfold would raise)", d.T, d.L); return IGN_ERR_INVALID; }
  const int TT = g.Tw >= 64 ? 8 : 4;
  FwdPlan fp;
  const FwdKernel kern = fwd_kernel(d.dist == IGN_DIST_L1, g.KK, TT);
  if (!plan_fwd(g, TT, fp)) { set_error("shapelet_forward: problem does not fit shared memory (T=%d L=%d)", d.T, d.L); return IGN_ERR_UNSUPPORTED; }
  if (debug_plan_on()) debug_plan("fwd", g, fp.threads, fp.smem_bytes, occupancy(kern, fp.threads, fp.smem_bytes), TT, 1);
  FwdArgs a{xn, st0, W, thr, p, dmin, argmin, dstore, stats_pitch(d.T, d.L, d.stride)};
  return run_fwd(kern, g, a, fp, st);
}

struct BwdWorkspace { size_t part, coef, rowsc, wstat, tie, total; };   // offsets/size in floats

BwdWorkspace bwd_workspace(const ign_shapelet_desc& d, const Geo& g, const BwdPlan& bp) {
  BwdWorkspace w;
  w.part = 0;
  const int nchunk = shapelet_bwd_tc_supported(d) ? max(bp.nchunk, shapelet_bwd_tc_chunks(d)) : bp.nchunk;
  w.coef = (size_t)nchunk * d.K * d.M * d.L;
  w.coef = (w.coef + 3) / 4 * 4;                         // 16-byte aligned rows
  w.rowsc = w.coef + (size_t)d.B * d.M * d.K * g.Ts;
  w.wstat = w.rowsc + (size_t)d.B * d.M * d.K * 2;
  w.tie = w.wstat + (size_t)d.K * d.M;
  w.total = w.tie + ((size_t)d.B * d.M * g.nkb + 3) / 4;   // bytes, rounded up to floats
  return w;
}

// where the pooling backward leaves the per-window coefficients inside the workspace (floats from its start)
bool shapelet_bwd_coef_offset(const ign_shapelet_desc& d, size_t* off_floats, size_t* total_bytes) {
  Geo g; BwdPlan bp;
  if (!base_geo(d, g) || !plan_bwd(g, bp)) return false;
  const BwdWorkspace w = bwd_workspace(d, g, bp);
  *off_floats = w.coef; *total_bytes = w.total * sizeof(float);
  return true;
}

size_t shapelet_bwd_workspace_simt(const ign_shapelet_desc& d) {
  Geo g; BwdPlan bp;
  if (!base_geo(d, g) || !plan_bwd(g, bp)) return 0;
  return bwd_workspace(d, g, bp).total * sizeof(float);
}

int launch_shapelet_bwd_simt(const ign_shapelet_desc& d, const float* xn, const float* st0,
                             const float* st1, const float* W, const float* gr, const float* gdmin, int gK, int gk0,
                             const float* dstore, const float* dmin, const int* argmin, float* dW, void* ws,
                             size_t ws_bytes, cudaStream_t st) {
  Geo g; BwdPlan bp;
  if (!base_geo(d, g)) { set_error("shapelet_backward: T=%d < L=%d", d.T, d.L); return IGN_ERR_INVALID; }
  if (!plan_bwd(g, bp)) { set_error("shapelet_backward: problem does not fit shared memory (T=%d L=%d)", d.T, d.L); return IGN_ERR_UNSUPPORTED; }
  const BwdKernel kern = bwd_kernel(d.dist, g.LT);
  const BwdWorkspace wo = bwd_workspace(d, g, bp);
  if (ws_bytes < wo.total * sizeof(float)) { set_error("shapelet_backward: workspace %zu < %zu bytes", ws_bytes, wo.total * sizeof(float)); return IGN_ERR_INVALID; }
  if (((uintptr_t)ws & 15) != 0) { set_error("shapelet_backward: workspace must be 16-byte aligned"); return IGN_ERR_INVALID; }
  float* base = reinterpret_cast<float*>(ws);
  const bool use_tc = shapelet_bwd_tc_supported(d);
  const bool use_tie = dW && !use_tc && d.dist == IGN_DIST_L1 && bp.hcap;   // the tie flags serve the contraction only
  unsigned char* tflags = reinterpret_cast<unsigned char*>(base + wo.tie);
  // 1. pooling backward (elementwise, HBM-bound): d -> per-window coefficients + per-row scalars
  if (d.dist == IGN_DIST_PEARSON) {
    shapelet_centred_norm_kernel<<<ceil_div(d.K * d.M, 8), 256, 0, st>>>(W, base + wo.wstat, d.K * d.M, d.L);
    IGN_CUDA(cudaGetLastError());
  }
  {
    PhaseScope ph(PH_POOL, st);
    const int rows = d.B * d.M * d.K;
    // recompute mode passes dstore == NULL: the distances were just recomputed INTO the coefficient buffer and are
    // converted in place (every row is read into shared memory / registers by its own warp before it is rewritten)
    PoolArgs pa{gr, gK, gk0, dstore ? dstore : base + wo.coef, dmin, argmin, st0, st1, stats_pitch(d.T, d.L, d.stride), base + wo.wstat, base + wo.coef, base + wo.rowsc, gdmin};
    const bool in_regs = g.Tw <= 1024;       // rows that fit NCH float4 chunks per lane (pool_bwd_reg_kernel)
    int warps = 8;
    const int stages = in_regs ? kPoolStages : 2;
    while (warps > 1 && (size_t)warps * stages * g.DP * sizeof(float) > (in_regs ? 100 : 72) * 1024) warps >>= 1;
    const size_t smem = (size_t)warps * stages * g.DP * sizeof(float);
    if (smem > (size_t)max_optin_smem() - 1024) { set_error("shapelet_backward: %d windows per series do not fit shared memory", g.Tw); return IGN_ERR_UNSUPPORTED; }
    int per_sm = max(1, min(2048 / (warps * 32), (int)(((size_t)max_smem_per_sm()) / (smem + 1024))));
    const int nch = g.Tw > 768 ? 8 : g.Tw > 512 ? 6 : g.Tw > 256 ? 4 : 2;
    if (in_regs) per_sm = min(per_sm, pool_reg_min_blocks(nch));    // its __launch_bounds__
    const dim3 pgrid(min(ceil_div(rows, warps), sm_count() * per_sm)), pblock(warps * 32);
#define IGN_POOL_LAUNCH_K(KERN)                                                         \
    { int rc = set_smem(KERN, smem); if (rc) return rc;                                 \
      KERN<<<pgrid, pblock, smem, st>>>(g, pa, rows); }
#define IGN_POOL_LAUNCH_G(PV, DV, GV)                                                   \
    { if (!in_regs) IGN_POOL_LAUNCH_K((pool_bwd_kernel<PV, DV, GV>))                    \
      else if (g.Tw > 768) IGN_POOL_LAUNCH_K((pool_bwd_reg_kernel<PV, DV, 8, GV>))      \
      else if (g.Tw > 512) IGN_POOL_LAUNCH_K((pool_bwd_reg_kernel<PV, DV, 6, GV>))      \
      else if (g.Tw > 256) IGN_POOL_LAUNCH_K((pool_bwd_reg_kernel<PV, DV, 4, GV>))      \
      else IGN_POOL_LAUNCH_K((pool_bwd_reg_kernel<PV, DV, 2, GV>)) }
#define IGN_POOL_LAUNCH(PV, DV)                                                         \
    { if (gdmin) IGN_POOL_LAUNCH_G(PV, DV, true) else IGN_POOL_LAUNCH_G(PV, DV, false) }
    if (d.pool == IGN_POOL_RBF_MAX) {
      switch (d.dist) {
        case IGN_DIST_L1: IGN_POOL_LAUNCH(IGN_POOL_RBF_MAX, IGN_DIST_L1) break;
        case IGN_DIST_SQL2: IGN_POOL_LAUNCH(IGN_POOL_RBF_MAX, IGN_DIST_SQL2) break;
        case IGN_DIST_COSINE: IGN_POOL_LAUNCH(IGN_POOL_RBF_MAX, IGN_DIST_COSINE) break;
        default: IGN_POOL_LAUNCH(IGN_POOL_RBF_MAX, IGN_DIST_PEARSON) break;
      }
    } else {
      if (d.dist == IGN_DIST_L1) IGN_POOL_LAUNCH(IGN_POOL_LTS_MIN, IGN_DIST_L1)
      else IGN_POOL_LAUNCH(IGN_POOL_LTS_MIN, IGN_DIST_SQL2)
    }
#undef IGN_POOL_LAUNCH
#undef IGN_POOL_LAUNCH_G
#undef IGN_POOL_LAUNCH_K
    IGN_CUDA(cudaGetLastError());
  }
  if (use_tie) {     // L1: which series rows can hold a value equal to one of their shapelet block's values
    PhaseScope ph(PH_TIE, st);
    const size_t hs = ((size_t)bp.hcap + kTieBitmapWords) * sizeof(unsigned);
    // one warp walks a series row per load round trip: the scan is latency-bound, so it wants about three CTAs per SM
    // (each CTA rebuilds the filter and the set: more, shorter CTAs lose to that setup — 0.063 ms at six per SM against
    // 0.052 at three, L = 100) and never a second, nearly empty wave (L = 500: 500 CTAs on 444 slots 0.091 ms, 375 CTAs
    // 0.066 ms)
    static const int tie_env = getenv("IGN_TIE_PER_SM") ? atoi(getenv("IGN_TIE_PER_SM")) : 0;   // experiments
    const int resident = max(1, min(8, (int)((size_t)max_smem_per_sm() / (hs + 1024))));
    const int target = min(tie_env > 0 ? tie_env : 3, resident);
    const int cols = d.M * g.nkb;
    const int bsplit = max(1, min(min(ceil_div(d.B, 8), ceil_div(target * sm_count(), cols)),
                                  max(1, resident * sm_count() / cols)));
    int rc0 = set_smem(tie_check_kernel, hs);
    if (rc0) return rc0;
    tie_check_kernel<<<dim3(d.M, g.nkb, bsplit), 256, hs, st>>>(xn, W, tflags, d.B, d.M, d.T, d.Tp, d.K, d.L, g.KB,
                                                               g.nkb, bp.hcap, bsplit);
    IGN_CUDA(cudaGetLastError());
  }
  if (!dW) return IGN_OK;     // input gradient only: the coefficients are what launch_shapelet_dx reads
  // 2. contraction with the series into per-chunk partials: tensor pipe for the cross-term modes in the tcgen05
  //    precisions (shapelet_tc_bwd.cu), FP32 pipe otherwise
  if (use_tc) {
    int rc;
    { PhaseScope ph(PH_CONTRACT, st); rc = launch_shapelet_bwd_tc(d, xn, base + wo.coef, base + wo.part, st); }
    if (rc) return rc;
    PhaseScope ph(PH_FINALIZE, st);
    shapelet_bwd_finalize<<<dim3(ceil_div(d.K * d.M, 8), ceil_div(d.L, 128)), 256, 0, st>>>(W, base + wo.part, base + wo.rowsc, dW, d.B, d.K,
                                                                d.M, d.L, shapelet_bwd_tc_chunks(d), d.dist);
    IGN_CUDA(cudaGetLastError());
    return IGN_OK;
  }
  const unsigned char* tie = use_tie ? tflags : nullptr;
  BwdArgs a{xn, W, base + wo.coef, base + wo.part, bp.nseg, bp.nlb, bp.tlb, tie};
  if (debug_plan_on()) debug_plan("bwd", g, bp.threads, bp.smem_bytes, occupancy(kern, bp.threads, bp.smem_bytes), bp.nseg, bp.nlb);
  int rc;
  { PhaseScope ph(PH_CONTRACT, st); rc = run_bwd(kern, g, a, bp, st); }
  if (rc) return rc;
  // 3. combine
  PhaseScope ph(PH_FINALIZE, st);
  shapelet_bwd_finalize<<<dim3(ceil_div(d.K * d.M, 8), ceil_div(d.L, 128)), 256, 0, st>>>(W, base + wo.part, base + wo.rowsc, dW, d.B, d.K,
                                                              d.M, d.L, bp.nchunk, d.dist);
  IGN_CUDA(cudaGetLastError());
  return IGN_OK;
}

// ---- recompute mode: nothing saved by the forward; bounded workspace, shapelets walked in chunks --------------------
namespace {
struct RecomputeLayout { int Kc; size_t bwd_bytes, out_off, fws_off, fws_bytes, dist_off, total; };

size_t align128(size_t v) { return (v + 127) / 128 * 128; }

// The input gradient of cosine / pearson reads the window distances next to the coefficients (launch_shapelet_dx's
// beta terms), so with dx the chunk's distances get a buffer of their own instead of being converted in place.
bool dx_keeps_distances(const ign_shapelet_desc& d, bool dx) {
  return dx && (d.dist == IGN_DIST_COSINE || d.dist == IGN_DIST_PEARSON);
}

bool recompute_layout(const ign_shapelet_desc& d, int Kc, RecomputeLayout& r, bool dx) {
  ign_shapelet_desc dc = d;
  dc.K = Kc;
  Geo g; BwdPlan bp;
  if (!base_geo(dc, g) || !plan_bwd(g, bp)) return false;
  r.Kc = Kc;
  r.bwd_bytes = align128(bwd_workspace(dc, g, bp).total * sizeof(float));
  r.out_off = r.bwd_bytes;                                            // p | dmin | argmin of the chunk, [B,Kc,M] each
  r.fws_off = r.out_off + align128((size_t)3 * d.B * Kc * d.M * sizeof(float));
  r.fws_bytes = shapelet_forward_workspace_bytes(dc);
  r.dist_off = r.fws_off + align128(r.fws_bytes);                     // [B,M,Kc,Tw] distances (dx_keeps_distances)
  r.total = r.dist_off;
  if (dx_keeps_distances(d, dx)) r.total += align128((size_t)d.B * d.M * Kc * g.Ts * sizeof(float));
  return true;
}

// largest chunk whose workspace fits `bytes` (a whole number of 8-shapelet blocks unless K itself is smaller), then
// balanced over the resulting number of chunks
int recompute_chunk(const ign_shapelet_desc& d, size_t bytes, bool dx) {
  RecomputeLayout r;
  int fit = 0;
  for (int Kc = d.K; Kc >= 1; Kc = (Kc > 8 ? (Kc - 1) / 8 * 8 : Kc - 1)) {
    if (recompute_layout(d, Kc, r, dx) && r.total <= bytes) { fit = Kc; break; }
  }
  if (fit == 0) fit = min(d.K, 8);                                    // budget too small: the minimum chunk
  const int n = ceil_div(d.K, fit);
  int bal = ceil_div(d.K, n);
  if (bal > 8) bal = min(fit, round_up(bal, 8));
  return bal;
}
}  // namespace

size_t shapelet_bwd_recompute_workspace(const ign_shapelet_desc& d, size_t budget, bool dx) {
  RecomputeLayout r;
  if (!recompute_layout(d, recompute_chunk(d, budget, dx), r, dx)) return 0;
  return r.total;
}

int launch_shapelet_bwd_recompute(const ign_shapelet_desc& d, const float* xn, const float* st0, const float* st1,
                                  const float* W, const float* thr, const float* gr, const float* gdmin, float* dW,
                                  float* dxn, void* ws, size_t ws_bytes, cudaStream_t st) {
  const bool dx = dxn != nullptr;
  if (((uintptr_t)ws & 127) != 0) { set_error("shapelet_backward(recompute): workspace must be 128-byte aligned"); return IGN_ERR_INVALID; }
  const int Kc = recompute_chunk(d, ws_bytes, dx);
  RecomputeLayout r;
  if (!recompute_layout(d, Kc, r, dx)) { set_error("shapelet_backward(recompute): problem does not fit shared memory (T=%d L=%d)", d.T, d.L); return IGN_ERR_UNSUPPORTED; }
  if (r.total > ws_bytes) { set_error("shapelet_backward(recompute): workspace %zu < %zu bytes (%s)", ws_bytes, r.total, dx ? "ign_shapelet_backward_recompute_input_workspace" : "ign_shapelet_backward_recompute_workspace"); return IGN_ERR_INVALID; }
  uint8_t* base8 = reinterpret_cast<uint8_t*>(ws);
  for (int k0 = 0; k0 < d.K; k0 += Kc) {
    ign_shapelet_desc dc = d;
    dc.K = min(Kc, d.K - k0);
    RecomputeLayout rc;
    if (!recompute_layout(dc, dc.K, rc, dx) || rc.total > ws_bytes) { set_error("shapelet_backward(recompute): internal chunk layout"); return IGN_ERR_INVALID; }
    Geo g; BwdPlan bp;
    base_geo(dc, g); plan_bwd(g, bp);
    const BwdWorkspace wo = bwd_workspace(dc, g, bp);
    float* dbuf = reinterpret_cast<float*>(base8) + wo.coef;            // distances now, coefficients after the pooling pass
    float* dkeep = dx_keeps_distances(d, dx) ? reinterpret_cast<float*>(base8 + rc.dist_off) : nullptr;
    float* outp = reinterpret_cast<float*>(base8 + rc.out_off);
    const size_t no = (size_t)d.B * dc.K * d.M;
    const size_t wofs = (size_t)k0 * d.M * d.L;
    // 1. the forward of this chunk again (same kernels, same engine as the real forward): window distances -> dbuf, or
    //    -> dkeep when the input gradient reads them after the pooling pass
    int rc1 = shapelet_forward_dispatch(dc, xn, st0, W + wofs, thr ? thr + (size_t)k0 * d.M : nullptr, outp, outp + no,
                                        reinterpret_cast<int*>(outp + 2 * no), dkeep ? dkeep : dbuf, base8 + rc.fws_off,
                                        rc.fws_bytes, st);
    if (rc1) return rc1;
    // 2. pooling backward (in place, or dkeep -> dbuf), contraction, finalize -> dW[k0 .. k0+Kc) (dW == NULL: the
    //    pooling backward alone); gdmin is read like gr, at the chunk's shapelets, and lands on the recomputed argmin of
    //    the chunk (the same kernels give the forward's index)
    rc1 = launch_shapelet_bwd_simt(dc, xn, st0, st1, W + wofs, gr, gdmin, d.K, k0, dkeep, outp + no,
                                   reinterpret_cast<const int*>(outp + 2 * no), dW ? dW + wofs : nullptr, ws,
                                   rc.bwd_bytes, st);
    if (rc1) return rc1;
    // 3. dxn += this chunk's shapelets' share.  Every dxn row belongs to one CTA, which adds the shapelets in k order:
    //    chunk after chunk on one stream, the sum over k runs in the stored mode's order.
    if (dx) {
      rc1 = launch_shapelet_dx(dc, xn, st0, st1, W + wofs, dbuf, dkeep, dxn, st);
      if (rc1) return rc1;
    }
  }
  return IGN_OK;
}

int bwd_phase_timing(int enable) {
  std::lock_guard<std::mutex> lock(g_phase_mu);
  g_phase_on = enable != 0;
  return IGN_OK;
}

// total milliseconds and launch count per phase since the last read; waits for the recorded events
int bwd_phase_read(float* ms, int* count) {
  std::lock_guard<std::mutex> lock(g_phase_mu);
  for (int i = 0; i < PH_COUNT; ++i) { ms[i] = 0.f; count[i] = 0; }
  for (auto& r : g_phase) {
    float t = 0.f;
    IGN_CUDA(cudaEventSynchronize(r.e1));
    IGN_CUDA(cudaEventElapsedTime(&t, r.e0, r.e1));
    ms[r.phase] += t; count[r.phase] += 1;
    cudaEventDestroy(r.e0); cudaEventDestroy(r.e1);
  }
  g_phase.clear();
  return IGN_OK;
}

}  // namespace ign
