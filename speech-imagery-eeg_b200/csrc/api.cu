// extern "C" entry points of libign_b200.so — see include/ign_b200.h for the contract.
#include "ign_common.cuh"

#include <string.h>
#include <vector>

namespace ign {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int max_optin_smem() {
  static int cached = 0;
  if (!cached) {
    int dev = 0, v = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) == cudaSuccess && v > 0)
      cached = v;
    else { cudaGetLastError(); return 227 * 1024; }   // B200 value; used for planning without a device
  }
  return cached;
}

int max_smem_per_sm() {
  static int cached = 0;
  if (!cached) {
    int dev = 0, v = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev) == cudaSuccess && v > 0)
      cached = v;
    else { cudaGetLastError(); return 228 * 1024; }
  }
  return cached;
}

int sm_count() {
  static int cached = 0;
  if (!cached) {
    int dev = 0, v = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && v > 0)
      cached = v;
    else { cudaGetLastError(); return 148; }
  }
  return cached;
}

static int check_desc(const ign_shapelet_desc* d, const char* who) {
  IGN_REQUIRE(d != nullptr, "%s: null descriptor", who);
  IGN_REQUIRE(d->B > 0 && d->M > 0 && d->T > 0 && d->K > 0 && d->L > 0 && d->stride > 0,
              "%s: non-positive dimension (B=%d M=%d T=%d K=%d L=%d stride=%d)", who, d->B, d->M, d->T,
              d->K, d->L, d->stride);
  IGN_REQUIRE(d->Tp == padded_len(d->T), "%s: Tp=%d must equal ign_padded_len(T)=%d", who, d->Tp, padded_len(d->T));
  IGN_REQUIRE(d->T >= d->L, "%s: maximum size for tensor at dimension 2 is %d but size is %d (T < L)", who, d->T, d->L);
  IGN_REQUIRE(d->dist >= IGN_DIST_L1 && d->dist <= IGN_DIST_PEARSON, "%s: bad dist %d", who, d->dist);
  IGN_REQUIRE(d->pool == IGN_POOL_RBF_MAX || d->pool == IGN_POOL_LTS_MIN, "%s: bad pool %d", who, d->pool);
  IGN_REQUIRE(d->precision >= IGN_PREC_FP32 && d->precision <= IGN_PREC_TF32, "%s: bad precision %d", who, d->precision);
  IGN_REQUIRE(d->B <= 65535 * 64, "%s: batch too large", who);
  return IGN_OK;
}

size_t shapelet_forward_workspace_bytes(const ign_shapelet_desc& d) {
  return (d.precision != IGN_PREC_FP32 && shapelet_fwd_tc_supported(d)) ? shapelet_fwd_tc_workspace(d) : 0;
}

// tcgen05 engine for the cross-term distances in the tensor-core precisions; everything else (L1, IGN_PREC_FP32 and
// the geometries shapelet_fwd_tc_supported rejects) on the exact-fp32 CUDA-core engine — ign_shapelet_engine reports
// which one a descriptor gets
int shapelet_forward_dispatch(const ign_shapelet_desc& d, const float* xn, const float* st0, const float* W,
                              const float* thr, float* p, float* dmin, int* argmin, float* dstore, void* ws,
                              size_t ws_bytes, cudaStream_t st) {
  if (d.precision != IGN_PREC_FP32 && shapelet_fwd_tc_supported(d))
    return launch_shapelet_fwd_tc(d, xn, st0, W, thr, p, dmin, argmin, dstore, ws, ws_bytes, st);
  return launch_shapelet_fwd_simt(d, xn, st0, W, thr, p, dmin, argmin, dstore, st);
}

}  // namespace ign

using namespace ign;

extern "C" {

int32_t ign_abi_version(void) { return IGN_ABI_VERSION; }
const char* ign_last_error(void) { return g_err; }

int32_t ign_device_check(int32_t device) {
  int dev = device;
  if (dev < 0) IGN_CUDA(cudaGetDevice(&dev));
  int major = 0;
  IGN_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  if (major != 10) { set_error("device %d is compute capability %d.x; libign_b200 is built for sm_100a only", dev, major); return IGN_ERR_ARCH; }
  return IGN_OK;
}

int32_t ign_debug_bwd_phase_timing(int32_t enable) { return bwd_phase_timing(enable); }
int32_t ign_debug_bwd_phase_read(float* ms4, int32_t* count4) {
  IGN_REQUIRE(ms4 != nullptr && count4 != nullptr, "ign_debug_bwd_phase_read: null output");
  return bwd_phase_read(ms4, count4);
}
int32_t ign_debug_tc_trace(int64_t* host, int32_t n) { return tc_trace_read(reinterpret_cast<long long*>(host), n); }
int32_t ign_debug_tc_profile(uint64_t* host16, int32_t reset) {
  if (reset & 2) return bwd_tc_profile_read(reinterpret_cast<unsigned long long*>(host16), reset & 1);   // backward kernel's counters
  return tc_profile_read(reinterpret_cast<unsigned long long*>(host16), reset);
}
int32_t ign_padded_len(int32_t T) { return padded_len(T); }
int32_t ign_num_windows(int32_t T, int32_t L, int32_t stride) { return (L <= 0 || stride <= 0) ? 0 : num_windows(T, L, stride); }
int32_t ign_padded_windows(int32_t T, int32_t L, int32_t stride) { return (L <= 0 || stride <= 0) ? 0 : padded_windows(T, L, stride); }

int32_t ign_instnorm_forward(const float* x, float* xn, float* mean, float* rstd, int32_t B, int32_t T,
                             int32_t M, void* stream) {
  IGN_REQUIRE(x && xn, "instnorm_forward: null pointer");
  IGN_REQUIRE(B > 0 && T > 0 && M > 0 && B <= 65535, "instnorm_forward: bad shape B=%d T=%d M=%d", B, T, M);
  return launch_instnorm(x, xn, mean, rstd, B, T, M, (cudaStream_t)stream);
}

int32_t ign_stats_pitch(int32_t T, int32_t L, int32_t stride) { return (L <= 0 || stride <= 0) ? 0 : stats_pitch(T, L, stride); }

int32_t ign_window_stats(const float* xn, int32_t B, int32_t M, int32_t T, int32_t G, const int32_t* L,
                         const int32_t* stride, int32_t dist, float* const* st0, float* const* st1, void* stream) {
  IGN_REQUIRE(xn && L && stride && st0, "window_stats: null pointer");
  IGN_REQUIRE(B > 0 && M > 0 && T > 0, "window_stats: bad shape B=%d T=%d M=%d", B, T, M);
  IGN_REQUIRE(G > 0 && G <= kMaxStatGroups, "window_stats: 1..%d groups per call (got %d)", kMaxStatGroups, G);
  IGN_REQUIRE(dist >= IGN_DIST_SQL2 && dist <= IGN_DIST_PEARSON, "window_stats: dist %d has no norm term", dist);
  IGN_REQUIRE(dist != IGN_DIST_PEARSON || st1, "window_stats: PEARSON needs st1");
  StatGroups sg;
  sg.n = G;
  for (int g = 0; g < G; ++g) {
    IGN_REQUIRE(L[g] > 0 && stride[g] > 0 && T >= L[g] && st0[g], "window_stats: bad group %d (L=%d stride=%d)", g, L[g], stride[g]);
    IGN_REQUIRE(dist != IGN_DIST_PEARSON || st1[g], "window_stats: PEARSON needs st1[%d]", g);
    sg.L[g] = L[g]; sg.s[g] = stride[g]; sg.Tw[g] = num_windows(T, L[g], stride[g]);
    sg.SP[g] = stats_pitch(T, L[g], stride[g]); sg.st0[g] = st0[g]; sg.st1[g] = st1 ? st1[g] : nullptr;
  }
  return launch_window_stats(xn, sg, B, M, T, dist, (cudaStream_t)stream);
}

int32_t ign_shapelet_engine(const ign_shapelet_desc* d, int32_t backward) {
  if (check_desc(d, "shapelet_engine")) return -1;
  if (d->precision == IGN_PREC_FP32) return IGN_ENGINE_FP32;
  return (backward ? shapelet_bwd_tc_supported(*d) : shapelet_fwd_tc_supported(*d)) ? IGN_ENGINE_TCGEN05 : IGN_ENGINE_FP32;
}

size_t ign_shapelet_forward_workspace(const ign_shapelet_desc* d) {
  if (check_desc(d, "shapelet_forward_workspace")) return 0;
  return shapelet_forward_workspace_bytes(*d);
}

int32_t ign_shapelet_forward(const ign_shapelet_desc* d, const float* xn, const float* st0, const float* W,
                             const float* thr, float* p, float* dmin, int32_t* argmin, float* dstore,
                             void* ws, size_t ws_bytes, void* stream) {
  int rc = check_desc(d, "shapelet_forward");
  if (rc) return rc;
  IGN_REQUIRE(xn && W && p && dmin, "shapelet_forward: null pointer");
  IGN_REQUIRE(d->dist == IGN_DIST_L1 || st0, "shapelet_forward: dist %d needs the window statistics (ign_window_stats)", d->dist);
  IGN_REQUIRE(d->pool != IGN_POOL_LTS_MIN || thr, "shapelet_forward: LTS pooling needs threshold");
  IGN_REQUIRE(d->pool != IGN_POOL_LTS_MIN || d->dist <= IGN_DIST_SQL2,
              "shapelet_forward: DistThresholdShapelet ignores distance_func (Shapelet.py:100-103); use L1 or SQL2");
  return shapelet_forward_dispatch(*d, xn, st0, W, thr, p, dmin, argmin, dstore, ws, ws_bytes, (cudaStream_t)stream);
}

size_t ign_shapelet_backward_workspace(const ign_shapelet_desc* d) {
  if (check_desc(d, "shapelet_backward_workspace")) return 0;
  return shapelet_bwd_workspace_simt(*d);
}

size_t ign_shapelet_dstore_bytes(const ign_shapelet_desc* d) {
  if (check_desc(d, "shapelet_dstore_bytes")) return 0;
  return (size_t)d->B * d->M * d->K * padded_windows(d->T, d->L, d->stride) * sizeof(float);
}

size_t ign_shapelet_backward_recompute_workspace(const ign_shapelet_desc* d, size_t budget_bytes) {
  if (check_desc(d, "shapelet_backward_recompute_workspace")) return 0;
  return shapelet_bwd_recompute_workspace(*d, budget_bytes, false);
}

size_t ign_shapelet_backward_recompute_input_workspace(const ign_shapelet_desc* d, size_t budget_bytes) {
  if (check_desc(d, "shapelet_backward_recompute_input_workspace")) return 0;
  return shapelet_bwd_recompute_workspace(*d, budget_bytes, true);
}

int32_t ign_shapelet_backward_dmin(const ign_shapelet_desc* d, const float* xn, const float* st0, const float* st1,
                                   const float* W, const float* thr, const float* g, const float* gdmin,
                                   const float* dstore, const float* dmin, const int32_t* argmin, float* dW, void* ws,
                                   size_t ws_bytes, void* stream) {
  int rc = check_desc(d, "shapelet_backward");
  if (rc) return rc;
  IGN_REQUIRE(xn && W && g && ws, "shapelet_backward: null pointer");
  IGN_REQUIRE(d->dist == IGN_DIST_L1 || st0, "shapelet_backward: dist %d needs the window statistics", d->dist);
  IGN_REQUIRE(d->dist != IGN_DIST_PEARSON || st1, "shapelet_backward: PEARSON needs st1 (window means)");
  if (!dstore) {   // recompute mode: nothing was kept by the forward
    IGN_REQUIRE(dW, "shapelet_backward(recompute): dW is required (dW == NULL needs the stored distances)");
    IGN_REQUIRE(d->pool != IGN_POOL_LTS_MIN || thr, "shapelet_backward(recompute): lts_min needs the threshold again");
    return launch_shapelet_bwd_recompute(*d, xn, st0, st1, W, thr, g, gdmin, dW, nullptr, ws, ws_bytes,
                                         (cudaStream_t)stream);
  }
  IGN_REQUIRE(d->pool != IGN_POOL_LTS_MIN || (dmin && argmin), "shapelet_backward: lts_min needs the forward's dmin and argmin");
  IGN_REQUIRE(!gdmin || argmin, "shapelet_backward: gdmin needs the forward's argmin (the window it lands on)");
  return launch_shapelet_bwd_simt(*d, xn, st0, st1, W, g, gdmin, d->K, 0, dstore, dmin, argmin, dW, ws, ws_bytes,
                                  (cudaStream_t)stream);
}

int32_t ign_shapelet_backward(const ign_shapelet_desc* d, const float* xn, const float* st0, const float* st1,
                              const float* W, const float* thr, const float* g, const float* dstore,
                              const float* dmin, const int32_t* argmin, float* dW, void* ws, size_t ws_bytes,
                              void* stream) {
  return ign_shapelet_backward_dmin(d, xn, st0, st1, W, thr, g, nullptr, dstore, dmin, argmin, dW, ws, ws_bytes, stream);
}

int32_t ign_shapelet_backward_input(const ign_shapelet_desc* d, const float* xn, const float* st0, const float* st1,
                                    const float* W, const float* dstore, float* dxn, const void* ws, size_t ws_bytes,
                                    void* stream) {
  int rc = check_desc(d, "shapelet_backward_input");
  if (rc) return rc;
  IGN_REQUIRE(xn && W && dxn && ws, "shapelet_backward_input: null pointer");
  IGN_REQUIRE(dstore, "shapelet_backward_input: stored-distance mode only (dstore from the forward is required)");
  IGN_REQUIRE(d->dist < IGN_DIST_COSINE || st0, "shapelet_backward_input: dist %d needs the window statistics", d->dist);
  IGN_REQUIRE(d->dist != IGN_DIST_PEARSON || st1, "shapelet_backward_input: PEARSON needs st1 (window means)");
  size_t off = 0, total = 0;
  if (!shapelet_bwd_coef_offset(*d, &off, &total)) { set_error("shapelet_backward_input: T=%d < L=%d or the problem does not fit shared memory", d->T, d->L); return IGN_ERR_INVALID; }
  IGN_REQUIRE(ws_bytes >= total, "shapelet_backward_input: workspace %zu < %zu bytes (pass the workspace ign_shapelet_backward used)", ws_bytes, total);
  return launch_shapelet_dx(*d, xn, st0, st1, W, reinterpret_cast<const float*>(ws) + off, dstore, dxn, (cudaStream_t)stream);
}

int32_t ign_shapelet_backward_recompute_input(const ign_shapelet_desc* d, const float* xn, const float* st0,
                                              const float* st1, const float* W, const float* thr, const float* g,
                                              const float* gdmin, float* dW, float* dxn, void* ws, size_t ws_bytes,
                                              void* stream) {
  int rc = check_desc(d, "shapelet_backward_recompute_input");
  if (rc) return rc;
  IGN_REQUIRE(xn && W && g && dxn && ws, "shapelet_backward_recompute_input: null pointer");
  IGN_REQUIRE(d->dist == IGN_DIST_L1 || st0, "shapelet_backward_recompute_input: dist %d needs the window statistics", d->dist);
  IGN_REQUIRE(d->dist != IGN_DIST_PEARSON || st1, "shapelet_backward_recompute_input: PEARSON needs st1 (window means)");
  IGN_REQUIRE(d->pool != IGN_POOL_LTS_MIN || thr, "shapelet_backward_recompute_input: lts_min needs the threshold again");
  return launch_shapelet_bwd_recompute(*d, xn, st0, st1, W, thr, g, gdmin, dW, dxn, ws, ws_bytes, (cudaStream_t)stream);
}

int32_t ign_diversity_partials(int32_t K) { return K <= 0 ? 0 : diversity_blocks(K) * diversity_blocks(K); }

int32_t ign_diversity_forward(const float* W, float* coef, float* partial, int32_t K, int32_t M, int32_t L, void* stream) {
  IGN_REQUIRE(W && coef && partial, "diversity_forward: null pointer");
  IGN_REQUIRE(K > 0 && M > 0 && L > 0, "diversity_forward: bad shape K=%d M=%d L=%d", K, M, L);
  return launch_diversity_fwd(W, coef, partial, K, M, L, (cudaStream_t)stream);
}

int32_t ign_diversity_backward(const float* W, const float* coef, const float* gout, float* dW, int32_t K, int32_t M,
                               int32_t L, void* stream) {
  IGN_REQUIRE(W && coef && gout && dW, "diversity_backward: null pointer");
  IGN_REQUIRE(K > 0 && M > 0 && L > 0, "diversity_backward: bad shape K=%d M=%d L=%d", K, M, L);
  return launch_diversity_bwd(W, coef, gout, dW, K, M, L, (cudaStream_t)stream);
}

int32_t ign_gate_forward(const float* s, const float* z, float* out, float* eta, int32_t B, int32_t C,
                         int32_t use_gate, float gv, void* stream) {
  IGN_REQUIRE(s && z && out && eta, "gate_forward: null pointer");
  IGN_REQUIRE(B > 0 && C > 1, "gate_forward: bad shape B=%d C=%d (needs C>1)", B, C);
  return launch_gate_fwd(s, z, out, eta, B, C, use_gate, gv, (cudaStream_t)stream);
}

int32_t ign_gate_backward(const float* s, const float* z, const float* go, const float* ge, float* gs, float* gz,
                          int32_t B, int32_t C, int32_t use_gate, float gv, void* stream) {
  IGN_REQUIRE(s && z && go && gs && gz, "gate_backward: null pointer");
  IGN_REQUIRE(B > 0 && C > 1, "gate_backward: bad shape B=%d C=%d (needs C>1)", B, C);
  return launch_gate_bwd(s, z, go, ge, gs, gz, B, C, use_gate, gv, (cudaStream_t)stream);
}

int32_t ign_sbm_transform_host(const float* x_host, int32_t B, int32_t T, int32_t M, int32_t G,
                               const float* const* W_host, const int32_t* K, const int32_t* L, const int32_t* stride,
                               float eps, int32_t dist, int32_t precision, float* probs_host, float* dists_host) {
  IGN_REQUIRE(x_host && W_host && K && L && stride && probs_host && dists_host, "sbm_transform_host: null pointer");
  IGN_REQUIRE(B > 0 && T > 0 && M > 0 && G > 0, "sbm_transform_host: bad shape");
  IGN_REQUIRE(G <= kMaxStatGroups, "sbm_transform_host: at most %d groups", kMaxStatGroups);
  int rc = ign_device_check(-1);
  if (rc) return rc;
  const int Tp = padded_len(T);
  int F = 0, Kmax = 0;
  size_t wmax = 0;
  for (int g = 0; g < G; ++g) {
    IGN_REQUIRE(K[g] > 0 && L[g] > 0 && stride[g] > 0 && T >= L[g], "sbm_transform_host: bad group %d", g);
    F += K[g] * M; Kmax = K[g] > Kmax ? K[g] : Kmax;
    size_t w = (size_t)K[g] * M * L[g];
    wmax = w > wmax ? w : wmax;
  }
  cudaStream_t st;
  IGN_CUDA(cudaStreamCreate(&st));
  float *x = nullptr, *xn = nullptr, *W = nullptr, *out = nullptr;
  void* pre = nullptr;
  void* fws = nullptr;
  const size_t nx = (size_t)B * T * M, nxn = (size_t)B * M * Tp, nf = (size_t)B * Kmax * M;
  auto cleanup = [&]() {
    cudaFree(x); cudaFree(xn); cudaFree(W); cudaFree(out); cudaFree(pre); cudaFree(fws);
    cudaStreamDestroy(st);
  };
#define IGN_TRY(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) { set_error("%s failed: %s", #call, cudaGetErrorString(e__)); cleanup(); return IGN_ERR_CUDA; } } while (0)
  IGN_TRY(cudaMalloc(&x, nx * 4));
  IGN_TRY(cudaMalloc(&xn, nxn * 4));
  IGN_TRY(cudaMalloc(&W, wmax * 4));
  IGN_TRY(cudaMalloc(&out, nf * 2 * 4));
  size_t fws_bytes = 0;
  for (int g = 0; g < G; ++g) {
    ign_shapelet_desc dd{B, M, T, Tp, K[g], L[g], stride[g], eps, dist, IGN_POOL_RBF_MAX, precision};
    const size_t nb = ign_shapelet_forward_workspace(&dd);
    fws_bytes = nb > fws_bytes ? nb : fws_bytes;
  }
  if (fws_bytes) IGN_TRY(cudaMalloc(&fws, fws_bytes));
  size_t soff[kMaxStatGroups + 1] = {0};
  if (dist != IGN_DIST_L1) {
    for (int g = 0; g < G; ++g) soff[g + 1] = soff[g] + (size_t)B * M * stats_pitch(T, L[g], stride[g]);
    IGN_TRY(cudaMalloc(&pre, soff[G] * 2 * sizeof(float)));
  }
  IGN_TRY(cudaMemcpyAsync(x, x_host, nx * 4, cudaMemcpyHostToDevice, st));
  rc = launch_instnorm(x, xn, nullptr, nullptr, B, T, M, st);
  float* sbase = reinterpret_cast<float*>(pre);
  if (!rc && pre) {
    float* p0[kMaxStatGroups]; float* p1[kMaxStatGroups];
    for (int g = 0; g < G; ++g) { p0[g] = sbase + soff[g]; p1[g] = sbase + soff[G] + soff[g]; }
    rc = ign_window_stats(xn, B, M, T, G, L, stride, dist, p0, p1, st);
  }
  std::vector<float> hp, hd;
  int col = 0;
  for (int g = 0; g < G && !rc; ++g) {
    ign_shapelet_desc d{B, M, T, Tp, K[g], L[g], stride[g], eps, dist, IGN_POOL_RBF_MAX, precision};
    const size_t n = (size_t)B * K[g] * M;
    IGN_TRY(cudaMemcpyAsync(W, W_host[g], (size_t)K[g] * M * L[g] * 4, cudaMemcpyHostToDevice, st));
    rc = ign_shapelet_forward(&d, xn, pre ? sbase + soff[g] : nullptr, W, nullptr, out, out + nf, nullptr, nullptr, fws, fws_bytes, st);
    if (rc) break;
    hp.resize(n); hd.resize(n);
    IGN_TRY(cudaMemcpyAsync(hp.data(), out, n * 4, cudaMemcpyDeviceToHost, st));
    IGN_TRY(cudaMemcpyAsync(hd.data(), out + nf, n * 4, cudaMemcpyDeviceToHost, st));
    IGN_TRY(cudaStreamSynchronize(st));
    const int w = K[g] * M;
    for (int b = 0; b < B; ++b) {   // torch.cat(dim=-1) over groups (Shapelet.py:195-196)
      memcpy(probs_host + (size_t)b * F + col, hp.data() + (size_t)b * w, (size_t)w * 4);
      memcpy(dists_host + (size_t)b * F + col, hd.data() + (size_t)b * w, (size_t)w * 4);
    }
    col += w;
  }
  if (!rc) IGN_TRY(cudaStreamSynchronize(st));
#undef IGN_TRY
  cleanup();
  return rc;
}

}  // extern "C"
