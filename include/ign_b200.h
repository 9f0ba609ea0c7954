/*
 * ign_b200.h — C ABI of the B200-native InterpGN shapelet hot path (libign_b200.so).
 *
 * Drop-in boundary for the reference path
 *   InterpretGatedNetwork/model/Shapelet.py:46-238   (Shapelet, DistThresholdShapelet, ShapeBottleneckModel)
 *   InterpretGatedNetwork/model/InterpGN.py:39-60    (Gini gate + mixture)
 * The reference has no FFI (it is eager PyTorch); these entry points are what a ctypes binding for that
 * path binds (INTEGRATION.md shows the stub).  Plain pointers and sizes only, no torch types.
 *
 * Conventions
 *   - Pointers named *_dev are CUDA device pointers on the current device; the caller owns all memory.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Calls are asynchronous
 *     on that stream, allocate nothing, and are re-entrant per device.
 *   - Every function returns ign_status_t; on failure ign_last_error() gives a thread-local message.
 *   - The library is CUDA-only by design (sm_100a): there is no CPU fallback.
 *   - Shapes use the reference's names: B batch, T seq_len, M channels (enc_in), K shapelets per length,
 *     L shapelet length, stride, T' = (T-L)/stride + 1 windows, C classes.
 *     Pooled outputs are [B,K,M] row-major, i.e. feature index k*M+m of Shapelet.py:84 after flatten.
 */
#ifndef IGN_B200_H_
#define IGN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IGN_ABI_VERSION 3

typedef enum {
  IGN_OK = 0,
  IGN_ERR_INVALID = 1,     /* bad shape / null pointer / bad enum (reference: torch raises RuntimeError) */
  IGN_ERR_CUDA = 2,        /* a CUDA runtime call failed */
  IGN_ERR_UNSUPPORTED = 3, /* combination not implemented */
  IGN_ERR_ARCH = 4         /* device is not sm_100 */
} ign_status_t;

/* distance arithmetic, as dispatched by Shapelet.forward (Shapelet.py:64-74) */
typedef enum {
  IGN_DIST_L1 = 0,      /* distance_func='euclidean': mean_l |x-w|            Shapelet.py:74 */
  IGN_DIST_SQL2 = 1,    /* 'euclidean' + memory_efficient: mean_l (w-x)^2     Shapelet.py:28 */
  IGN_DIST_COSINE = 2,  /* 1 - cos(x_w, w), per-vector norm clamp 1e-8        Shapelet.py:64-66 */
  IGN_DIST_PEARSON = 3  /* 1 - corr(x_w, w), +1e-8 on the denominator         Shapelet.py:11-19,67-69 */
} ign_dist_t;

/* pooling over time */
typedef enum {
  IGN_POOL_RBF_MAX = 0, /* p=exp(-(eps d)^2); straight-through soft/hard max  Shapelet.py:77-84 */
  IGN_POOL_LTS_MIN = 1  /* straight-through soft/hard min; sigmoid(thr-min)   Shapelet.py:105-111 */
} ign_pool_t;

/* engine / operand precision of the cross term <x_w, w> (ignored for IGN_DIST_L1, which has none) */
typedef enum {
  IGN_PREC_FP32 = 0,    /* CUDA-core FFMA, exact fp32 products                                     */
  IGN_PREC_3XTF32 = 1,  /* tcgen05 kind::tf32, hi*hi + hi*lo + lo*hi split: fp32-equivalent         */
  IGN_PREC_TF32 = 2     /* tcgen05 kind::tf32 single pass (own, looser tolerance)                   */
} ign_precision_t;

/* which kernels a call runs on (ign_shapelet_engine) */
typedef enum {
  IGN_ENGINE_FP32 = 0,    /* CUDA-core kernels (shapelet_simt.cu): exact fp32 products, any geometry          */
  IGN_ENGINE_TCGEN05 = 1  /* tensor-core kernels (shapelet_tc.cu / shapelet_tc_bwd.cu)                        */
} ign_engine_t;

typedef struct {
  int32_t B, M, T;      /* batch, channels, series length                                          */
  int32_t Tp;           /* row pitch of xn in floats, = ign_padded_len(T)                          */
  int32_t K, L, stride; /* shapelets per channel, shapelet length, window stride (Shapelet.py:47)  */
  float eps;            /* RBF width  (Shapelet.eps)                                               */
  int32_t dist;         /* ign_dist_t                                                              */
  int32_t pool;         /* ign_pool_t                                                              */
  int32_t precision;    /* ign_precision_t                                                         */
} ign_shapelet_desc;

int32_t ign_abi_version(void);
const char* ign_last_error(void);
/* IGN_OK iff `device` (or the current device when < 0) is compute capability 10.x */
int32_t ign_device_check(int32_t device);

/* debug / measurement: CUDA events around the four phases of ign_shapelet_backward (0 pooling backward, 1 tie
 * pre-check, 2 contraction, 3 finalize), recorded on the call's stream while enabled.  ign_debug_bwd_phase_read waits
 * for the recorded events and returns total milliseconds and launch counts per phase since the last read. */
int32_t ign_debug_bwd_phase_timing(int32_t enable);
int32_t ign_debug_bwd_phase_read(float* ms4_host, int32_t* count4_host);
/* debug: role-level cycle counters of the tcgen05 kernel (only in builds with -DIGN_TC_PROFILE) */
int32_t ign_debug_tc_profile(uint64_t* host16, int32_t reset);
/* debug: clock64() event trace of CTA 0 of the last tcgen05 launch, [12 roles][32 tiles][4 events] (same builds) */
int32_t ign_debug_tc_trace(int64_t* host, int32_t n);

/* pitch (floats) of one normalised series row: T rounded up to a multiple of 4 (16-byte rows) */
int32_t ign_padded_len(int32_t T);
/* number of windows T' (0 when T < L: the reference's unfold raises there) and its padded pitch */
int32_t ign_num_windows(int32_t T, int32_t L, int32_t stride);
int32_t ign_padded_windows(int32_t T, int32_t L, int32_t stride);

/* ShapeBottleneckModel.forward instance norm (Shapelet.py:186-187):
 *   x_dev [B,T,M] -> xn_dev [B,M,Tp],  xn = (x-mean_T)/(std_T(unbiased)+1e-8), pad columns zeroed.
 *   Optional (may be NULL) per-series statistics mean_dev/rstd_dev [B,M] (rstd = 1/(std+1e-8)). */
int32_t ign_instnorm_forward(const float* x_dev, float* xn_dev, float* mean_dev, float* rstd_dev,
                             int32_t B, int32_t T, int32_t M, void* stream);

/* pitch (floats) of one window-statistics row: T' rounded up to a multiple of 16 */
int32_t ign_stats_pitch(int32_t T, int32_t L, int32_t stride);

/* Sliding-window statistics for the norm terms of cosine / pearson / sql2: for G (<= 8) length groups at
 * once, per series row an fp64 prefix scan of xn and xn^2 in shared memory, then per window the fp32 norm term
 *   SQL2: st0 = ||x_w||^2      COSINE: st0 = 1/max(||x_w||,1e-8)      PEARSON: st0 = ||x_w-mu||, st1 = mu
 * The pad slots t >= T' of st0 hold an ignore marker (+inf for SQL2, NaN for COSINE / PEARSON: the resulting
 * distance is +inf / NaN and never wins the min over time); st1 pads are 0.
 * L / stride are HOST arrays of G ints; st0_dev / st1_dev are HOST arrays of G device pointers, each
 * [B,M,ign_stats_pitch(T,L[g],stride[g])] (st1_dev may be NULL unless dist == PEARSON).
 * Reference: the norm / mean terms inside cosine_similarity, pearson_corrcoef and ShapeletDistanceFunc
 * (Shapelet.py:11-19, :28, :64-69). */
int32_t ign_window_stats(const float* xn_dev, int32_t B, int32_t M, int32_t T, int32_t G, const int32_t* L,
                         const int32_t* stride, int32_t dist, float* const* st0_dev, float* const* st1_dev,
                         void* stream);

/* The engine ign_shapelet_forward (backward == 0) or the contraction of ign_shapelet_backward (backward != 0) runs
 * on for this descriptor.  `precision` is a request: IGN_DIST_L1 has no cross term and always runs on the FP32
 * engine; the tensor-core kernels tile every other geometry (any stride, up to 32768 windows per series; DESIGN.md
 * 3.2).  Callers that report an engine (bench.py, tools/sweep.py) must ask, not assume.
 * Returns an ign_engine_t, or -1 for an invalid descriptor. */
int32_t ign_shapelet_engine(const ign_shapelet_desc* desc, int32_t backward);

/* Shapelet.forward / DistThresholdShapelet.forward for one length group.
 *   xn_dev [B,M,Tp]; st0_dev [B,M,SP] window statistics of this group from ign_window_stats (required unless
 *   dist==L1); W_dev [K,M,L]; threshold_dev [K,M] (required for LTS_MIN).
 * Outputs, all [B,K,M]:
 *   p_dev       pooled predicate: max_t exp(-(eps d_t)^2) = exp(-(eps min_t d_t)^2)   Shapelet.py:77-82
 *               | sigmoid(thr - min_t d_t)                                            Shapelet.py:105-109
 *   dmin_dev    min_t d_t                                                             Shapelet.py:84
 *   argmin_dev  argmin_t d_t, first index on ties (may be NULL).  It is also the arg-max of p barring
 *               ties of p in fp32; backward re-derives the reference's arg-max-of-p one-hot itself.
 *   dstore_dev  optional [B,M,K,Tw] (Tw = ign_padded_windows) all window distances, kept for backward
 *               (the soft-max statistics are recomputed from it); NULL in inference.
 * Engine: precision FP32 -> CUDA-core kernels; 3XTF32 / TF32 -> tcgen05 kernels (any stride, up to 32768 windows per
 * series; ign_shapelet_engine tells which one a descriptor gets).  The tcgen05 engine needs ign_shapelet_forward_workspace(desc)
 * bytes of 128-byte-aligned scratch (the pre-swizzled shifted-shapelet tiles); 0 bytes / NULL otherwise. */
size_t ign_shapelet_forward_workspace(const ign_shapelet_desc* desc);
int32_t ign_shapelet_forward(const ign_shapelet_desc* desc, const float* xn_dev, const float* st0_dev,
                             const float* W_dev, const float* threshold_dev, float* p_dev, float* dmin_dev,
                             int32_t* argmin_dev, float* dstore_dev, void* workspace_dev, size_t workspace_bytes,
                             void* stream);

/* bytes of scratch ign_shapelet_backward needs for this problem in the stored-distance mode (dstore_dev given) */
size_t ign_shapelet_backward_workspace(const ign_shapelet_desc* desc);

/* bytes of the saved window distances [B,M,K,Tw] the stored-distance mode keeps between forward and backward */
size_t ign_shapelet_dstore_bytes(const ign_shapelet_desc* desc);

/* Recompute mode (dstore_dev == NULL in ign_shapelet_backward): nothing is kept from the forward; the backward
 * walks the K shapelets in chunks and, per chunk, recomputes the window distances into the workspace, turns them
 * in place into the per-window coefficients and contracts them — so its memory is bounded by the workspace, not by
 * B*M*K*T' (116 GB + 116 GB at K = 1000, B = 256, L = 100 in the stored mode).  This returns the workspace size for
 * the largest shapelet chunk that fits `budget_bytes` (at least one shapelet block: the result can exceed a budget
 * that is too small).  Pass the same number of bytes to ign_shapelet_backward: the chunking is derived from it. */
size_t ign_shapelet_backward_recompute_workspace(const ign_shapelet_desc* desc, size_t budget_bytes);

/* Gradient of the pooled output w.r.t. the shapelets, through the straight-through soft/hard pooling
 * (Shapelet.py:79-82 | :105-108): every window receives soft_t*(p_t - pbar) (+1 at the hard index).
 *   g_dev [B,K,M] = dLoss/d(max_p)  (rbf_max)   or   dLoss/d(min_d)  (lts_min; the caller folds the
 *   sigmoid: g_min = -g_p * p * (1-p), dthreshold = sum_b g_p * p * (1-p))
 *   st0_dev / st1_dev: window statistics as for forward (st1 only for PEARSON; both NULL for L1).
 *   dstore_dev [B,M,K,Tw] as written by ign_shapelet_forward on the same inputs, or NULL: recompute mode (above;
   then the threshold of lts_min is needed again: threshold_dev below, NULL otherwise allowed).
 *   dmin_dev / argmin_dev [B,K,M]: the forward's outputs; required for lts_min (its hard index and soft-min
 *   shift), ignored (may be NULL) for rbf_max, whose arg-max-of-p one-hot is re-derived from dstore.
 *   dW_dev [K,M,L] is overwritten (not accumulated).  Deterministic (no float atomics).
 *   dW_dev == NULL (weights frozen, only the input gradient wanted): runs the preparation alone — the pooling backward
 *   and, for PEARSON, the shapelet norms — which leaves in the workspace the coefficients ign_shapelet_backward_input
 *   reads; the contraction is skipped.  Stored-distance mode only (dstore_dev != NULL). */
int32_t ign_shapelet_backward(const ign_shapelet_desc* desc, const float* xn_dev, const float* st0_dev,
                              const float* st1_dev, const float* W_dev, const float* threshold_dev,
                              const float* g_dev, const float* dstore_dev, const float* dmin_dev,
                              const int32_t* argmin_dev, float* dW_dev, void* workspace_dev,
                              size_t workspace_bytes, void* stream);

/* ign_shapelet_backward with a gradient on the second output as well, min_t d (dmin_dev of the forward,
 * Shapelet.py:84 | :111), for losses that use it (ShapeBottleneckModel's ModelInfo.d):
 *   gdmin_dev [B,K,M] = dLoss/d(min_t d), or NULL (exactly ign_shapelet_backward, which forwards here with NULL).
 * min_t d is the hard minimum in both poolings, so gdmin_dev[b,k,m] is added to the coefficient of ONE window,
 * argmin_t d with the first index on ties — the forward's argmin_dev.  For rbf_max that is not always the window the
 * straight-through arg-max of p picks (where every p underflows to 0 the arg-max is window 0).
 *   Stored-distance mode: argmin_dev is required whenever gdmin_dev is given (for rbf_max too).  Recompute mode: the
 *   index is recomputed with the distances; argmin_dev is not read.
 *   g_dev stays required: pass zeros when only min_t d carries a gradient.
 * Every other argument, the workspace and the dW_dev == NULL case are as for ign_shapelet_backward, and
 * ign_shapelet_backward_input then gives the input gradient of both outputs. */
int32_t ign_shapelet_backward_dmin(const ign_shapelet_desc* desc, const float* xn_dev, const float* st0_dev,
                                   const float* st1_dev, const float* W_dev, const float* threshold_dev,
                                   const float* g_dev, const float* gdmin_dev, const float* dstore_dev,
                                   const float* dmin_dev, const int32_t* argmin_dev, float* dW_dev,
                                   void* workspace_dev, size_t workspace_bytes, void* stream);

/* Gradient w.r.t. the normalised input series — what autograd gives a user of the reference who asks for input
 * gradients (saliency, gradcheck) through Shapelet.forward; the training loop never does
 * (experiment_classification.py:315).  Call AFTER ign_shapelet_backward (with or without dW_dev) of the same group
 * with the same workspace: it reads the per-window coefficients that call left there.
 *   dxn_dev [B,M,Tp] += sum_k sum_t dLoss/dd[b,k,t] * d d_t / d xn[b,m,t*stride + l]     (ADDED: zero it once, call per group)
 * L1 (Shapelet.py:74, sign(0) = 0), cosine (:64-66), pearson (:11-19,:67-69).  SQL2: nothing is added — the
 * reference's ShapeletDistanceFunc.backward returns zeros for its input (Shapelet.py:40).  Stored-distance mode only;
 * recompute mode: ign_shapelet_backward_recompute_input below. */
int32_t ign_shapelet_backward_input(const ign_shapelet_desc* desc, const float* xn_dev, const float* st0_dev,
                                    const float* st1_dev, const float* W_dev, const float* dstore_dev, float* dxn_dev,
                                    const void* workspace_dev, size_t workspace_bytes, void* stream);

/* The input gradient in recompute mode, where no chunk's coefficients outlive the chunk: one call does what
 * ign_shapelet_backward_dmin (dstore_dev == NULL) and ign_shapelet_backward_input do in the stored mode.  Per shapelet
 * chunk it recomputes the window distances, runs the pooling backward, contracts into dW_dev (unless NULL) and adds
 * the chunk's share of the input gradient into dxn_dev.  Each dxn row adds its shapelets in k order, chunk after
 * chunk, as ign_shapelet_backward_input adds them in one pass.
 *   g_dev / gdmin_dev (may be NULL) / threshold_dev (required for lts_min) as for ign_shapelet_backward_dmin.
 *   dW_dev [K,M,L] is overwritten, or NULL when the weights are frozen: the contraction is skipped.
 *   dxn_dev [B,M,Tp] += dLoss/dxn, as ign_shapelet_backward_input (ADDED; nothing for SQL2).
 * The workspace (128-byte aligned, ign_shapelet_backward_recompute_input_workspace(desc, budget) bytes; the chunking
 * is derived from workspace_bytes) holds, per chunk: the coefficient workspace of ign_shapelet_backward, the chunk's
 * p / dmin / argmin, the forward's tcgen05 scratch and, for COSINE / PEARSON only, the chunk's window distances
 * [B,M,Kc,Tw].  The input gradient of those two modes reads the distances after the pooling backward has turned them
 * into coefficients, so they cannot be converted in place: at the same budget their chunks hold fewer shapelets than
 * those of ign_shapelet_backward_recompute_workspace.  For L1 and SQL2 both queries return the same size.  At least
 * one shapelet block, as for ign_shapelet_backward_recompute_workspace: the result can exceed a budget that is too
 * small. */
size_t ign_shapelet_backward_recompute_input_workspace(const ign_shapelet_desc* desc, size_t budget_bytes);
int32_t ign_shapelet_backward_recompute_input(const ign_shapelet_desc* desc, const float* xn_dev, const float* st0_dev,
                                              const float* st1_dev, const float* W_dev, const float* threshold_dev,
                                              const float* g_dev, const float* gdmin_dev, float* dW_dev,
                                              float* dxn_dev, void* workspace_dev, size_t workspace_bytes,
                                              void* stream);

/* InterpGN gate + mixture (InterpGN.py:44-52): q=softmax(s), eta=(C*sum q^2-1)/(C-1),
 * if use_gate: eta=1 where eta>gating_value; out=eta*s+(1-eta)*z.  s,z,out [B,C]; eta [B]. */
int32_t ign_gate_forward(const float* sbm_out_dev, const float* deep_out_dev, float* out_dev,
                         float* eta_dev, int32_t B, int32_t C, int32_t use_gate, float gating_value,
                         void* stream);
/* Backward of the above (eta is NOT detached in the reference).  g_eta_dev may be NULL. */
int32_t ign_gate_backward(const float* sbm_out_dev, const float* deep_out_dev, const float* g_out_dev,
                          const float* g_eta_dev, float* g_sbm_dev, float* g_deep_dev, int32_t B,
                          int32_t C, int32_t use_gate, float gating_value, void* stream);

/* Shapelet diversity regulariser of ShapeBottleneckModel.loss (Shapelet.py:223-230) for one length group:
 *   div = (1/(M K K)) * sum_{m, a != b} exp(-|| W[b,m,:] - W[a,m,:] + 1e-6 ||_2)
 * forward writes coef_dev [M,K,K] (= exp(-d)/d, 0 on the diagonal; the backward's input) and
 * ign_diversity_partials(K) * M partial sums to partial_dev; div = sum(partial) / (M K K), summed by the caller.
 * backward: dW_dev [K,M,L] = gout * d div / dW (overwritten); gout_dev points to ONE float on the device. */
int32_t ign_diversity_partials(int32_t K);
int32_t ign_diversity_forward(const float* W_dev, float* coef_dev, float* partial_dev, int32_t K, int32_t M,
                              int32_t L, void* stream);
int32_t ign_diversity_backward(const float* W_dev, const float* coef_dev, const float* gout_dev, float* dW_dev,
                               int32_t K, int32_t M, int32_t L, void* stream);

/* Host-buffer convenience call (inference): the whole shapelet transform of ShapeBottleneckModel.forward
 * (Shapelet.py:186-196) for G length groups with HOST pointers; copies in, launches, copies out and
 * synchronises.  x_host [B,T,M]; W_host[g] [K[g],M,L[g]]; probs_host/dists_host [B, sum_g K[g]*M]. */
int32_t ign_sbm_transform_host(const float* x_host, int32_t B, int32_t T, int32_t M, int32_t G,
                               const float* const* W_host, const int32_t* K, const int32_t* L,
                               const int32_t* stride, float eps, int32_t dist, int32_t precision,
                               float* probs_host, float* dists_host);

#ifdef __cplusplus
}
#endif
#endif /* IGN_B200_H_ */
