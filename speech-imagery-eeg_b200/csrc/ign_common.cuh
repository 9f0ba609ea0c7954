// Shared declarations for libign_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/ign_b200.h"

namespace ign {

void set_error(const char* fmt, ...);

#define IGN_REQUIRE(cond, ...)                         \
  do {                                                 \
    if (!(cond)) {                                     \
      ::ign::set_error(__VA_ARGS__);                   \
      return IGN_ERR_INVALID;                          \
    }                                                  \
  } while (0)

#define IGN_CUDA(call)                                                                   \
  do {                                                                                   \
    cudaError_t e__ = (call);                                                            \
    if (e__ != cudaSuccess) {                                                            \
      ::ign::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, \
                       __LINE__);                                                        \
      return IGN_ERR_CUDA;                                                               \
    }                                                                                    \
  } while (0)

__host__ __device__ inline int round_up(int a, int b) { return (a + b - 1) / b * b; }
__host__ __device__ inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

inline int padded_len(int T) { return round_up(T, 4); }
inline int num_windows(int T, int L, int s) { return T < L ? 0 : (T - L) / s + 1; }
inline int padded_windows(int T, int L, int s) { return round_up(num_windows(T, L, s), 4); }
// per-group fp32 window statistics: row pitch = windows rounded up to 16 (zero padded)
inline int stats_pitch(int T, int L, int s) { return round_up(num_windows(T, L, s), 16); }
constexpr int kMaxStatGroups = 8;
struct StatGroups { int n; int L[kMaxStatGroups], s[kMaxStatGroups], Tw[kMaxStatGroups], SP[kMaxStatGroups]; float* st0[kMaxStatGroups]; float* st1[kMaxStatGroups]; };

// ---- launchers implemented in the .cu files (all asynchronous on `st`) ----
int launch_instnorm(const float* x, float* xn, float* mean, float* rstd, int B, int T, int M,
                    cudaStream_t st);
int launch_window_stats(const float* xn, const StatGroups& G, int B, int M, int T, int dist, cudaStream_t st);
int launch_shapelet_fwd_simt(const ign_shapelet_desc& d, const float* xn, const float* st0,
                             const float* W, const float* thr, float* p, float* dmin,
                             int* argmin, float* dstore, cudaStream_t st);
size_t shapelet_bwd_workspace_simt(const ign_shapelet_desc& d);
// g [B,gK,M]: the launch's K shapelets are gk0 .. gk0+K-1 of it; gdmin: NULL, or dLoss/d(min_t d) indexed like g (it
// is added at the window argmin names); dstore == NULL: the distances sit in the coefficient buffer of the workspace
// already (recompute mode) and are converted in place; dW == NULL: the preparation alone (the coefficients for
// launch_shapelet_dx), no contraction
int launch_shapelet_bwd_simt(const ign_shapelet_desc& d, const float* xn, const float* st0,
                             const float* st1, const float* W, const float* g, const float* gdmin, int gK, int gk0,
                             const float* dstore, const float* dmin, const int* argmin, float* dW, void* ws,
                             size_t ws_bytes, cudaStream_t st);
bool shapelet_bwd_coef_offset(const ign_shapelet_desc& d, size_t* off_floats, size_t* total_bytes);
int launch_shapelet_dx(const ign_shapelet_desc& d, const float* xn, const float* st0, const float* st1, const float* W,
                       const float* coef, const float* dstore, float* dxn, cudaStream_t st);
// dx: the layout of the input-gradient walk (dxn != NULL below), which keeps cosine / pearson distances apart
size_t shapelet_bwd_recompute_workspace(const ign_shapelet_desc& d, size_t budget, bool dx);
// dW == NULL: weights frozen (needs dxn); dxn == NULL: dW only; dxn != NULL: dxn += the input gradient, chunk by chunk
int launch_shapelet_bwd_recompute(const ign_shapelet_desc& d, const float* xn, const float* st0, const float* st1,
                                  const float* W, const float* thr, const float* g, const float* gdmin, float* dW,
                                  float* dxn, void* ws, size_t ws_bytes, cudaStream_t st);
// engine selection + launch shared by ign_shapelet_forward and the recompute backward (api.cu)
size_t shapelet_forward_workspace_bytes(const ign_shapelet_desc& d);
int shapelet_forward_dispatch(const ign_shapelet_desc& d, const float* xn, const float* st0, const float* W,
                              const float* thr, float* p, float* dmin, int* argmin, float* dstore, void* ws,
                              size_t ws_bytes, cudaStream_t st);
int bwd_phase_timing(int enable);
int bwd_phase_read(float* ms4, int* count4);
int tc_profile_read(unsigned long long* host16, int reset);
int tc_trace_read(long long* host, int n);
int bwd_tc_profile_read(unsigned long long* host16, int reset);
bool shapelet_fwd_tc_supported(const ign_shapelet_desc& d);
size_t shapelet_fwd_tc_workspace(const ign_shapelet_desc& d);
int launch_shapelet_fwd_tc(const ign_shapelet_desc& d, const float* xn, const float* st0,
                           const float* W, const float* thr, float* p, float* dmin, int* argmin, float* dstore,
                           void* ws, size_t ws_bytes, cudaStream_t st);
bool shapelet_bwd_tc_supported(const ign_shapelet_desc& d);
int shapelet_bwd_tc_chunks(const ign_shapelet_desc& d);
int launch_shapelet_bwd_tc(const ign_shapelet_desc& d, const float* xn, const float* coef, float* part, cudaStream_t st);
int launch_gate_fwd(const float* s, const float* z, float* out, float* eta, int B, int C, int use_gate,
                    float gv, cudaStream_t st);
int launch_gate_bwd(const float* s, const float* z, const float* go, const float* ge, float* gs,
                    float* gz, int B, int C, int use_gate, float gv, cudaStream_t st);

int diversity_blocks(int K);
int launch_diversity_fwd(const float* W, float* coef, float* partial, int K, int M, int L, cudaStream_t st);
int launch_diversity_bwd(const float* W, const float* coef, const float* gout, float* dW, int K, int M, int L,
                         cudaStream_t st);

int max_optin_smem();  // per-block opt-in shared memory of the current device (cached)
int max_smem_per_sm();  // shared memory of one SM (each resident CTA also reserves 1 KB of it)
int sm_count();

}  // namespace ign
