// Instance norm + layout change, and the sliding-window prefix-sum pass.  Both HBM-bound.
//
//   instnorm_kernel : x[B,T,M] (channels last) -> xn[B,M,Tp] (time contiguous, 16-byte rows)
//                     reference: Shapelet.py:186-187  (x-mean_T)/(std_T(unbiased)+1e-8)
//   window_stats_kernel : fp64 prefix sums of xn and xn^2 per series, from which every window's sum / squared
//                     norm is one subtraction, turned into the norm terms of cosine/pearson/sql2
//                     (Shapelet.py:11-19,28,64-66) for several length groups at once
#include "ign_common.cuh"

#include <cooperative_groups.h>

namespace ign {

namespace {

#include "tc_ptx.cuh"

namespace cg = cooperative_groups;

constexpr int kNormThreads = 256;
constexpr int kNormWarps = kNormThreads / 32;
constexpr int kMaxCluster = 8;          // portable maximum.  16 (opt-in on sm_100) was measured SLOWER: 0.131 ms vs 0.079 ms at
                                        // config 2 — 16 co-scheduled CTAs leave the GPC's other SMs waiting

// ---- cluster variant (the default whenever it applies): one thread-block cluster per sample, CTA `rank` owns the
// time rows [rank*R, rank*R + R).  In the [B,T,M] batch layout those rows are ONE contiguous byte range, so the CTA's
// whole tile is fetched by 1-D bulk TMA copies (fully coalesced DRAM reads, no per-thread address arithmetic, no
// register staging); per-channel sums are combined across the cluster through distributed shared memory (two-pass
// mean / squared deviations, as the reference's std), and each warp then writes one channel's R-sample segment with
// 128-byte stores.  The dense [R][M] tile is read column-wise in the drain, which is bank-conflict free when M is odd
// (stride M words: CHISCO's 125 channels); layouts with gcd(M, 32) > 2 keep the padded-tile kernel below.
__global__ void __launch_bounds__(kNormThreads) instnorm_cluster_kernel(const float* __restrict__ x,
                                                                        float* __restrict__ xn,
                                                                        float* __restrict__ mean_out,
                                                                        float* __restrict__ rstd_out, int T, int M,
                                                                        int Tp, int R) {
  extern __shared__ __align__(128) unsigned char smraw[];
  const int Mp = round_up(M, 32);
  float* tile = reinterpret_cast<float*>(smraw);          // [R][M], byte image of x[b, t_lo : t_lo + rows, :]
  float* part = tile + (size_t)R * M;                      // [2][warps][Mp] per-warp partial sums / sums of squares
  float* csum = part + 2 * kNormWarps * Mp;                // [2][Mp] this CTA's partials, read by the cluster peers
  float* stat = csum + 2 * Mp;                             // [2][Mp] mean, 1 / (std + 1e-8)
  uint64_t* bar = reinterpret_cast<uint64_t*>(stat + 2 * Mp);
  cg::cluster_group cluster = cg::this_cluster();
  const int CS = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
  const int b = blockIdx.x / CS;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int t_lo = rank * R, rows = max(0, min(R, T - t_lo));

  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    fence_proxy_async_smem();
    if (rows > 0) {
      const uint32_t bytes = (uint32_t)rows * M * sizeof(float);        // multiple of 16: rows % 4 == 0 or T*M % 4 == 0
      mbar_arrive_expect_tx(bar, bytes);
      const unsigned char* src = reinterpret_cast<const unsigned char*>(x + ((size_t)b * T + t_lo) * M);
      for (uint32_t off = 0; off < bytes; off += 32768u)
        tma_bulk_g2s(smraw + off, src + off, min(32768u, bytes - off), bar);
    }
  }
  __syncthreads();
  if (rows > 0) mbar_wait(bar, 0);

  // One pass over the tile: per-channel sum and sum of squares of (x - x[b,0,c]) — shifting by a sample of the series
  // keeps the one-pass variance as accurate as the two-pass form (|mean - shift| ~ std) and every CTA of the cluster
  // can fetch the same shift.  Lanes = consecutive channels (conflict-free), four rows in flight per thread.
  const float* x0 = x + (size_t)b * T * M;
  for (int c = lane; c < Mp; c += 32) {
    float a0 = 0.f, a1 = 0.f, q0 = 0.f, q1 = 0.f;
    if (c < M) {
      const float sh = __ldg(x0 + c);
      int t = warp;
      for (; t + kNormWarps < rows; t += 2 * kNormWarps) {
        const float v0 = tile[t * M + c] - sh, v1 = tile[(t + kNormWarps) * M + c] - sh;
        a0 += v0; q0 = fmaf(v0, v0, q0);
        a1 += v1; q1 = fmaf(v1, v1, q1);
      }
      if (t < rows) { const float v0 = tile[t * M + c] - sh; a0 += v0; q0 = fmaf(v0, v0, q0); }
    }
    part[warp * Mp + c] = a0 + a1;
    part[(kNormWarps + warp) * Mp + c] = q0 + q1;
  }
  __syncthreads();
  for (int c = threadIdx.x; c < 2 * Mp; c += kNormThreads) {
    const int h = c >= Mp ? 1 : 0, cc = c - h * Mp;
    float sacc = 0.f;
#pragma unroll
    for (int w = 0; w < kNormWarps; ++w) sacc += part[(h * kNormWarps + w) * Mp + cc];
    csum[c] = sacc;                                        // [2][Mp]: sums, sums of squares
  }
  cluster.sync();
  for (int c = threadIdx.x; c < M; c += kNormThreads) {
    float ps[kMaxCluster], pq[kMaxCluster];
#pragma unroll
    for (int r = 0; r < kMaxCluster; ++r) {                // independent remote loads
      const float* peer = cluster.map_shared_rank(csum, r < CS ? r : 0);
      ps[r] = r < CS ? peer[c] : 0.f;
      pq[r] = r < CS ? peer[Mp + c] : 0.f;
    }
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int r = 0; r < kMaxCluster; ++r) { s1 += ps[r]; s2 += pq[r]; }
    const float dm = s1 / (float)T;                        // mean - shift
    const float mu = __ldg(x0 + c) + dm;
    const float var = fmaxf(s2 - s1 * dm, 0.f) / (float)(T - 1);   // unbiased, as torch.std
    const float den = sqrtf(var) + 1e-8f;
    stat[c] = mu; stat[Mp + c] = 1.f / den;
    if (rank == 0) {
      if (mean_out) mean_out[(size_t)b * M + c] = mu;
      if (rstd_out) rstd_out[(size_t)b * M + c] = 1.f / den;
    }
  }
  cluster.sync();                                          // no CTA may exit while a peer still reads its csum

  // drain: one warp per channel, 128 contiguous bytes per store instruction
  const bool last = rows > 0 && t_lo + rows == T;
  for (int ch = warp; ch < M; ch += kNormWarps) {
    const float mu = stat[ch], rden = stat[Mp + ch];       // multiplication by 1/(std+1e-8): <= 1 ulp from the division
    float* dst = xn + ((size_t)b * M + ch) * Tp + t_lo;
    for (int i = lane; i < rows; i += 32) dst[i] = (tile[i * M + ch] - mu) * rden;
    if (last && lane < Tp - T) dst[rows + lane] = 0.f;     // row padding (at most 3 samples)
  }
}

// ---- single-read instance norm: the whole (T x CT-channel) tile of one sample is staged in shared memory,
// so DRAM sees exactly one read of x and one write of xn.  CT = 8 keeps the tile at ~36 KB for T = 1000
// (6 CTAs per SM: one CTA's loads overlap the others' statistics and stores; 32-byte row segments = one sector).  The tile is stored [t][CT+1] so both the
// channel-major fill (lanes = channels) and the time-major drain (lanes = time) are bank-conflict free.
template <int CT>
__global__ void __launch_bounds__(kNormThreads) instnorm_tile_kernel(const float* __restrict__ x,
                                                                     float* __restrict__ xn,
                                                                     float* __restrict__ mean_out,
                                                                     float* __restrict__ rstd_out, int T,
                                                                     int M, int Tp) {
  extern __shared__ __align__(16) float tile[];            // [T][CT+1]
  __shared__ float s_mean[CT], s_den[CT];
  constexpr int P = CT + 1;
  constexpr int TPW = 32 / CT;                             // time rows covered by one warp load
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int m0 = blockIdx.x * CT, b = blockIdx.y;
  const int c = lane % CT, dt = lane / CT;
  const bool mv = m0 + c < M;
  const float* xb = x + (size_t)b * T * M + m0 + c;

  // fill: each warp instruction reads TPW rows x CT channels (CT*4 contiguous bytes per row)
  const int rows_per_iter = kNormWarps * TPW;
  constexpr int UN = 16;                                   // loads in flight per thread (fills the DRAM pipe)
  for (int t0 = warp * TPW + dt; t0 < T; t0 += rows_per_iter * UN) {
    float v[UN];
#pragma unroll
    for (int u = 0; u < UN; ++u) {
      const int t = t0 + u * rows_per_iter;
      v[u] = (mv && t < T) ? __ldg(xb + (size_t)t * M) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < UN; ++u) {
      const int t = t0 + u * rows_per_iter;
      if (t < T) tile[t * P + c] = v[u];
    }
  }
  __syncthreads();
  // statistics: 256/CT threads per channel, two passes over shared memory (mean, then squared deviations)
  constexpr int TPC = kNormThreads / CT;
  const int sc = threadIdx.x / TPC, si = threadIdx.x % TPC;
  float acc = 0.f;
  for (int t = si; t < T; t += TPC) acc += tile[t * P + sc];
#pragma unroll
  for (int o = TPC / 2; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  const float mu = acc / (float)T;
  acc = 0.f;
  for (int t = si; t < T; t += TPC) { const float d = tile[t * P + sc] - mu; acc = fmaf(d, d, acc); }
#pragma unroll
  for (int o = TPC / 2; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (si == 0) {
    const float sd = sqrtf(acc / (float)(T - 1));          // unbiased, as torch.std; T==1 -> NaN
    s_mean[sc] = mu; s_den[sc] = sd + 1e-8f;
    if (m0 + sc < M) {
      if (mean_out) mean_out[(size_t)b * M + m0 + sc] = mu;
      if (rstd_out) rstd_out[(size_t)b * M + m0 + sc] = 1.f / (sd + 1e-8f);
    }
  }
  __syncthreads();
  // drain: one warp per channel row, 128 B per store instruction
  for (int ch = warp; ch < CT; ch += kNormWarps) {
    if (m0 + ch >= M) continue;
    const float mu_c = s_mean[ch], den = s_den[ch];
    float* dst = xn + ((size_t)b * M + m0 + ch) * Tp;
    for (int t = lane; t < Tp; t += 32) dst[t] = t < T ? (tile[t * P + ch] - mu_c) / den : 0.f;
  }
}

// Fallback for very long series (tile does not fit shared memory): three passes over x, passes 2 and 3
// mostly from L2.
__global__ void __launch_bounds__(kNormThreads) instnorm_kernel(const float* __restrict__ x,
                                                                float* __restrict__ xn,
                                                                float* __restrict__ mean_out,
                                                                float* __restrict__ rstd_out, int T, int M,
                                                                int Tp) {
  __shared__ float part[kNormWarps][32];
  __shared__ float s_mean[32], s_den[32];
  __shared__ float tile[kNormWarps][32][33];

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int m0 = blockIdx.x * 32, b = blockIdx.y;
  const int m = m0 + lane;
  const bool mv = m < M;
  const float* xb = x + (size_t)b * T * M;

  float acc = 0.f;
  for (int t = warp; t < T; t += kNormWarps) acc += mv ? __ldg(xb + (size_t)t * M + m) : 0.f;
  part[warp][lane] = acc;
  __syncthreads();
  if (warp == 0) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < kNormWarps; ++w) s += part[w][lane];
    s_mean[lane] = s / (float)T;
  }
  __syncthreads();
  const float mu = s_mean[lane];
  acc = 0.f;
  for (int t = warp; t < T; t += kNormWarps) {
    float v = mv ? __ldg(xb + (size_t)t * M + m) - mu : 0.f;
    acc = fmaf(v, v, acc);
  }
  __syncthreads();
  part[warp][lane] = acc;
  __syncthreads();
  if (warp == 0) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < kNormWarps; ++w) s += part[w][lane];
    float sd = sqrtf(s / (float)(T - 1));
    s_den[lane] = sd + 1e-8f;
    if (mv) {
      if (mean_out) mean_out[(size_t)b * M + m] = mu;
      if (rstd_out) rstd_out[(size_t)b * M + m] = 1.f / (sd + 1e-8f);
    }
  }
  __syncthreads();
  const int ntile = (Tp + 31) / 32;
  for (int tt = warp; tt < ntile; tt += kNormWarps) {
    const int t0 = tt * 32;
#pragma unroll 8
    for (int i = 0; i < 32; ++i) {
      int t = t0 + i;
      float v = (mv && t < T) ? __ldg(xb + (size_t)t * M + m) : 0.f;
      tile[warp][i][lane] = v;
    }
    __syncwarp();
    const int t = t0 + lane;
#pragma unroll 8
    for (int i = 0; i < 32; ++i) {
      int mm = m0 + i;
      if (mm < M && t < Tp) {
        float v = tile[warp][lane][i];
        float o = (t < T) ? (v - s_mean[i]) / s_den[i] : 0.f;
        xn[((size_t)b * M + mm) * Tp + t] = o;
      }
    }
    __syncwarp();
  }
}

__device__ __forceinline__ double warp_incl_scan(double v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    double n = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += n;
  }
  return v;
}

// Sliding-window statistics for all length groups in one pass: per series row an fp64 prefix scan of x and
// x^2 in shared memory, then for every group g and window t the norm term its distance needs, as fp32:
//   sql2    st0 = ||x_w||^2            cosine  st0 = 1/max(||x_w||,1e-8)
//   pearson st0 = sqrt(sum (x_w-mu)^2), st1 = mu
// Rows are written with pitch SP_g (windows rounded up to 16; pad slots carry an ignore marker).  One warp per row.
//
// Scan: lane l owns the C consecutive samples [l*C, l*C + C) (C = the power of two >= ceil(T/32)): a lane-local running
// sum, ONE warp scan of the 32 lane totals, then P[j] = base_l + local_j.  (The first version scanned every
// 128-sample chunk across the warp — eight dependent 64-bit shuffle scans per row, ~1700 instructions per row.)
// Slot j of a prefix row lives at j + j/C (a shift): the pad double per C slots makes both the lane-strided writes of the scan
// (stride C+1, odd) and the window-strided reads of the statistics conflict-free.
// Statistics (unit stride): a lane produces four consecutive windows per step and stores them with one 16-byte
// store; strides > 1 (seq_len >= 3000) keep the scalar loop.
// The square root / reciprocal use the MUFU approximations (rsqrt.approx / sqrt.approx: relative error <= 2^-22.9 /
// 2^-23, i.e. as good as the correctly rounded sequences to the 2e-5 the distances are tested to).  The IEEE forms
// (sqrtf + 1.f/x, fp64 sqrt and division) compiled to ~25 instructions with three slow-path branches per window and made
// this HBM-bound kernel issue-bound (52 instructions per output, 0.26 ms for the four groups of config 2).
// (.ftz: a denormal window energy flushes to 0 and lands on the same 1e8 clamp / 0 as the exact value would)
__device__ __forceinline__ float rsqrt_approx(float x) { float y; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float sqrt_approx(float x) { float y; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
template <int dist>
__device__ __forceinline__ float stat_value(double sxx, double sx, double invL, float& mean_out) {
  if (dist == IGN_DIST_SQL2) return (float)sxx;
  if (dist == IGN_DIST_COSINE) return fminf(rsqrt_approx((float)sxx), 1e8f);     // 1 / max(||x_w||, 1e-8)
  const double mu = sx * invL;
  mean_out = (float)mu;
  return sqrt_approx((float)fmax(sxx - sx * mu, 0.0));
}

template <int dist>
__global__ void __launch_bounds__(256, 3) window_stats_kernel(const float* __restrict__ xn, const StatGroups G,
                                                              int rows, int T, int Tp, int csh, int PS) {
  constexpr bool need1 = dist == IGN_DIST_PEARSON;
  extern __shared__ __align__(16) double pbuf[];          // [warps][nseq][PS]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int wstride = gridDim.x * (blockDim.x >> 5);       // persistent warps: rows w, w + wstride, ...
  int row = blockIdx.x * (blockDim.x >> 5) + warp;
  if (row >= rows) return;
  constexpr int nseq = need1 ? 2 : 1;
  double* P2 = pbuf + (size_t)warp * nseq * PS;
  double* P1 = P2 + PS;
  const int C = 1 << csh;                                  // samples per lane, a power of two
  auto slot = [&](int j) { return j + (j >> csh); };
  const int i0 = lane * C;
  constexpr int UN = 8;
  float4 keep[UN];                                         // the lane's first 32 samples (all of them for T <= 1024)
  auto fetch = [&](int r) {                                // samples at or beyond Tp read as 0 (Tp - T pads are 0 already)
    const float* xq = xn + (size_t)r * Tp;
#pragma unroll
    for (int u = 0; u < UN; ++u) {
      const int i = i0 + 4 * u;
      keep[u] = (4 * u < C && i < Tp) ? __ldg(reinterpret_cast<const float4*>(xq + i)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  fetch(row);
  for (; row < rows; row += wstride) {
  const float* xr = xn + (size_t)row * Tp;

  // pass 1: lane totals
  double t1 = 0.0, t2 = 0.0;
  for (int c0 = 0; c0 < C; c0 += 4 * UN) {
    float4 v[UN];
#pragma unroll
    for (int u = 0; u < UN; ++u) {
      const int i = i0 + c0 + 4 * u;
      if (c0 == 0) v[u] = keep[u];
      else v[u] = (c0 + 4 * u < C && i < Tp) ? __ldg(reinterpret_cast<const float4*>(xr + i)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int u = 0; u < UN; ++u) {
      const double a = v[u].x, b = v[u].y, c = v[u].z, d = v[u].w;
      t2 += (a * a + b * b) + (c * c + d * d);
      if (need1) t1 += (a + b) + (c + d);
    }
  }
  const double b2 = warp_incl_scan(t2, lane) - t2;         // exclusive: prefix in front of this lane's samples
  const double b1 = need1 ? warp_incl_scan(t1, lane) - t1 : 0.0;
  if (lane == 0) { P2[0] = 0.0; if (need1) P1[0] = 0.0; }

  // pass 2: P[j+1] = base + running local sum.  Two levels keep the fp64 dependency chain short (the kernel is
  // latency-bound: 24 warps per SM, one row per warp): the prefix inside each float4 (eight independent 3-deep chains),
  // an 8-step scan of the float4 totals, then four independent adds per float4.
  double r1 = 0.0, r2 = 0.0;                                // carry across groups of four float4
  auto group = [&](int c0, const float4 (&v)[4]) {
    double q2[4][4], q1[need1 ? 4 : 1][4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const double a = v[u].x, b = v[u].y, c = v[u].z, d = v[u].w;
      q2[u][0] = a * a; q2[u][1] = q2[u][0] + b * b; q2[u][2] = q2[u][1] + c * c; q2[u][3] = q2[u][2] + d * d;
      if (need1) { q1[u][0] = a; q1[u][1] = a + b; q1[u][2] = q1[u][1] + c; q1[u][3] = q1[u][2] + d; }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + c0 + 4 * u;
      const double o2 = b2 + r2, o1 = b1 + r1;
      r2 += q2[u][3];
      if (need1) r1 += q1[u][3];
      if (c0 + 4 * u >= C || i >= T) continue;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        if (i + e < T) {
          const int sl = slot(i + e + 1);
          P2[sl] = o2 + q2[u][e];
          if (need1) P1[sl] = o1 + q1[u][e];
        }
      }
    }
  };
  {
    const float4 g0[4] = {keep[0], keep[1], keep[2], keep[3]};
    group(0, g0);
    if (C > 16) { const float4 g1[4] = {keep[4], keep[5], keep[6], keep[7]}; group(16, g1); }
  }
  for (int c0 = 32; c0 < C; c0 += 16) {                      // longer series: re-read (L1 / L2 hits)
    float4 gv[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + c0 + 4 * u;
      gv[u] = i < Tp ? __ldg(reinterpret_cast<const float4*>(xr + i)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    group(c0, gv);
  }
  __syncwarp();
  // the next row's samples are fetched now, so that their DRAM latency hides under the statistics stage below (with one
  // row per warp and nothing in flight during that stage the kernel sat at 2.5 TB/s)
  if (row + wstride < rows) fetch(row + wstride);

  for (int gi = 0; gi < G.n; ++gi) {
    const int L = G.L[gi], st = G.s[gi], Tw = G.Tw[gi], SP = G.SP[gi];
    float* o0 = G.st0[gi] + (size_t)row * SP;
    float* o1 = need1 ? G.st1[gi] + (size_t)row * SP : nullptr;
    // Pad windows (t >= Tw) carry an "ignore me" marker instead of a norm term, so that the distance kernels need
    // no per-window validity logic: +inf for SQL2 (distance +inf), NaN for COSINE / PEARSON (distance NaN, which
    // the min reductions — FMNMX returns the non-NaN operand — skip).
    const float pad = dist == IGN_DIST_SQL2 ? INFINITY : __int_as_float(0x7fc00000);
    const double invL = 1.0 / (double)L;
    if (st == 1) {
#pragma unroll 2
      for (int t0 = lane * 4; t0 < SP; t0 += 128) {        // SP % 16 == 0: whole float4s, 16-byte aligned rows
        float av[4] = {pad, pad, pad, pad}, bv[4] = {0.f, 0.f, 0.f, 0.f};
        // t0 % 4 == 0 and C >= 4 is a power of two: the four low slots share one pad offset; so do the four high ones
        // unless (t0 + L) sits in the last three slots of a C-block
        if (t0 + 4 <= Tw && ((t0 + L) & (C - 1)) <= C - 4) {
          const double* lo2 = P2 + slot(t0), * hi2 = P2 + slot(t0 + L);
          const double* lo1 = P1 + slot(t0), * hi1 = P1 + slot(t0 + L);
#pragma unroll
          for (int e = 0; e < 4; ++e)
            av[e] = stat_value<dist>(hi2[e] - lo2[e], need1 ? hi1[e] - lo1[e] : 0.0, invL, bv[e]);
        } else {
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int t = t0 + e;
            if (t < Tw) {
              const int lo = slot(t), hi = slot(t + L);
              av[e] = stat_value<dist>(P2[hi] - P2[lo], need1 ? P1[hi] - P1[lo] : 0.0, invL, bv[e]);
            }
          }
        }
        *reinterpret_cast<float4*>(o0 + t0) = make_float4(av[0], av[1], av[2], av[3]);
        if (o1) *reinterpret_cast<float4*>(o1 + t0) = make_float4(bv[0], bv[1], bv[2], bv[3]);
      }
    } else {
      for (int t = lane; t < SP; t += 32) {
        float a = pad, b = 0.f;
        if (t < Tw) {
          const int lo = slot(t * st), hi = slot(t * st + L);
          a = stat_value<dist>(P2[hi] - P2[lo], need1 ? P1[hi] - P1[lo] : 0.0, invL, b);
        }
        o0[t] = a;
        if (o1) o1[t] = b;
      }
    }
  }
  __syncwarp();                                            // all lanes are done with this row's prefix sums
  }
}

}  // namespace

int gcd_int(int a, int b) { while (b) { const int t = a % b; a = b; b = t; } return a; }

int launch_instnorm(const float* x, float* xn, float* mean, float* rstd, int B, int T, int M,
                    cudaStream_t st) {
  const int Tp = padded_len(T);
  // cluster + bulk-TMA kernel: needs 16-byte aligned sample slabs and a conflict-free column read of the dense tile
  if (((size_t)T * M) % 4 == 0 && gcd_int(M, 32) <= 2 && (((uintptr_t)x) & 15) == 0 && T > 1) {
    const int Mp = round_up(M, 32);
    const size_t extra = (size_t)(2 * kNormWarps + 4) * Mp * sizeof(float) + 16;
    // smallest cluster whose tiles leave room for 3 CTAs per SM: the per-CTA chain TMA -> statistics -> cluster
    // exchange -> drain is latency-bound, so several CTAs per SM have to overlap it
    static int max_cluster = kMaxCluster;
    for (;;) {
      int CS = 0, R = 0;
      for (int cs = 1; cs <= max_cluster; cs *= 2) {
        const int r = round_up(ceil_div(T, cs), 4);
        const size_t bytes = (size_t)r * M * sizeof(float) + extra;
        if (bytes <= 74 * 1024 || (cs == max_cluster && bytes <= (size_t)max_optin_smem() - 1024)) { CS = cs; R = r; break; }
      }
      if (!CS) break;
      const size_t smem = (size_t)R * M * sizeof(float) + extra;
      IGN_CUDA(cudaFuncSetAttribute(instnorm_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      if (CS > 8) IGN_CUDA(cudaFuncSetAttribute(instnorm_cluster_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(B * CS); cfg.blockDim = dim3(kNormThreads); cfg.dynamicSmemBytes = smem; cfg.stream = st;
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = CS; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
      cfg.attrs = attr; cfg.numAttrs = 1;
      const cudaError_t e = cudaLaunchKernelEx(&cfg, instnorm_cluster_kernel, x, xn, mean, rstd, T, M, Tp, R);
      if (e == cudaSuccess) return IGN_OK;
      cudaGetLastError();
      if (CS > 8 && max_cluster > 8) { max_cluster = 8; continue; }   // this device / partition cannot co-schedule 16 CTAs
      set_error("instnorm: cluster launch failed: %s", cudaGetErrorString(e));
      return IGN_ERR_CUDA;
    }
  }
#ifndef IGN_NORM_CT
#define IGN_NORM_CT 8      // measured on B200 at config 2: CT=4 1.56 TB/s, 8 2.94 TB/s, 16 2.29 TB/s, 32 1.27 TB/s
#endif
  constexpr int CT = IGN_NORM_CT;
  const size_t tile16 = (size_t)T * (CT + 1) * sizeof(float);
  if (tile16 + 2048 <= (size_t)max_optin_smem()) {
    static bool configured = false;
    if (!configured) {
      IGN_CUDA(cudaFuncSetAttribute(instnorm_tile_kernel<CT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    max_optin_smem() - 2048));
      configured = true;
    }
    dim3 grid(ceil_div(M, CT), B);
    instnorm_tile_kernel<CT><<<grid, kNormThreads, tile16, st>>>(x, xn, mean, rstd, T, M, Tp);
  } else {
    dim3 grid(ceil_div(M, 32), B);
    instnorm_kernel<<<grid, kNormThreads, 0, st>>>(x, xn, mean, rstd, T, M, Tp);
  }
  IGN_CUDA(cudaGetLastError());
  return IGN_OK;
}

int launch_window_stats(const float* xn, const StatGroups& G, int B, int M, int T, int dist, cudaStream_t st) {
  const int rows = B * M;
  int csh = 2;                                             // samples per lane: the power of two >= ceil(T / 32), >= 4
  while ((32 << csh) < T) ++csh;
  const int PS = round_up(T + 1 + ((T + 1) >> csh) + 1, 2); // prefix row pitch in doubles (one pad slot per 2^csh)
  const size_t per_warp = (size_t)(dist == IGN_DIST_PEARSON ? 2 : 1) * PS * sizeof(double);
  int warps = 8;
  while (warps > 1 && warps * per_warp > 72 * 1024) warps >>= 1;
  const size_t smem = warps * per_warp;
  if (smem > (size_t)max_optin_smem() - 1024) { set_error("window_stats: series of %d samples do not fit shared memory", T); return IGN_ERR_UNSUPPORTED; }
  const int per_sm = max(1, min(3, (int)((size_t)max_smem_per_sm() / (smem + 1024))));
  const int grid = min(ceil_div(rows, warps), sm_count() * per_sm);
#define IGN_WS_LAUNCH(DV)                                                                                         \
  { IGN_CUDA(cudaFuncSetAttribute(window_stats_kernel<DV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    window_stats_kernel<DV><<<grid, warps * 32, smem, st>>>(xn, G, rows, T, padded_len(T), csh, PS); }
  if (dist == IGN_DIST_PEARSON) IGN_WS_LAUNCH(IGN_DIST_PEARSON)
  else if (dist == IGN_DIST_COSINE) IGN_WS_LAUNCH(IGN_DIST_COSINE)
  else IGN_WS_LAUNCH(IGN_DIST_SQL2)
#undef IGN_WS_LAUNCH
  IGN_CUDA(cudaGetLastError());
  return IGN_OK;
}

}  // namespace ign
