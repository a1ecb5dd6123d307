/* nlml_hpe_b200 -- C ABI of the B200-native NLML_HPE inference hot path.
 *
 * The reference (MahdiGhafoorian/NLML_HPE) is pure Python and has no FFI of its own; the
 * "operator interface" of the hot path is two Python callables:
 *
 *   TD_Tester.optimize_with_sgd(W, x, u_id, u_id_shape, params_y, params_p, params_r,
 *                               learning_rate=0.001, num_iterations=3000)      TD_Tester.py:127-159
 *       (entry point TD_Tester.Test(...), TD_Tester.py:162-291, called from TD_Inference.py:56-58)
 *   CombinedAnglePredictionModel.forward(x[B,1404]) -> (yaw[B,1], pitch[B,1], roll[B,1])
 *                                                                 NLML_HPE_Model_Builder.py:115-126
 *       (called from NLML_HPE_Test.py:272,327,411 and generatePose_on_video.py:210)
 *
 * Each entry point below is what a ctypes binding on the reference side would call in place of
 * those two callables (INTEGRATION.md shows the stubs).  Plain pointers and sizes only; no
 * torch / numpy types.  All functions return 0 on success and a non-zero code on failure
 * (positive = cudaError_t, negative = NLML_E_*); nlml_last_error() returns a thread-local
 * human-readable message for the last failure.  There is no CPU fallback: every compute entry
 * point fails with NLML_E_NO_DEVICE when no sm_100 device is usable.
 */
#ifndef NLML_HPE_B200_H
#define NLML_HPE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NLML_ABI_VERSION 1

#define NLML_E_INVALID (-1)     /* bad argument (null pointer, non-positive size, unsupported rank) */
#define NLML_E_NO_DEVICE (-2)   /* no usable CUDA device */
#define NLML_E_UNSUPPORTED (-3) /* valid request this build cannot serve (e.g. core too large) */

int nlml_abi_version(void);
const char* nlml_last_error(void);

/* ------------------------------------------------------------------------------------------
 * Tucker fit  (replaces TD_Tester.optimize_with_sgd, TD_Tester.py:127-159, batched over samples)
 * ------------------------------------------------------------------------------------------ */
typedef struct nlml_tucker_plan nlml_tucker_plan;

/* One-time preparation for a Tucker tensor W[r_id][r_y][r_p][r_r][F] (C-contiguous float32, HOST
 * pointer; the array TD_Inference.py:47 loads from Trained_data.npz) and the cosine rows
 * optimized_{yaw,pitch,roll}[0:r,:] (HOST, row-major [r][4] doubles = (a,b,c,d), TD_Inference.py:43-45,
 * :56-57).  Uploads W, builds the folded Gram tensor on `device`, keeps both resident. */
int nlml_tucker_plan_create(const float* W_host, int r_id, int r_y, int r_p, int r_r, int F,
                            const double* rows_y, const double* rows_p, const double* rows_r,
                            int device, nlml_tucker_plan** plan_out);
void nlml_tucker_plan_destroy(nlml_tucker_plan* plan);

/* Fit N samples.  X: DEVICE float32 [N][ldx] (first F columns used).  P_out: DEVICE float32
 * [N][ldp], ldp >= 3 + r_id: (w_yaw, w_pitch, w_roll) in radians followed by the identity
 * coefficients, exactly the vector optimize_with_sgd returns (TD_Tester.py:159).
 * iters / lr / clip are num_iterations, learning_rate (TD_Tester.py:127) and the max_norm of :150.
 * Asynchronous on `stream` (a cudaStream_t passed as void*; NULL = legacy default stream).
 * kernel_hint: 0 = choose by N and ranks, 1 = thread-per-sample kernel (throughput, ranks 5,3,3,3),
 * 2 = CTA-per-sample kernel (run-time ranks), 3 = warp-per-sample kernel (latency, ranks 5,3,3,3),
 * 4 = thread-per-sample kernel with q resident in tensor memory (12 warps per SM; measured equal to 1),
 * 5 = tensor-core iteration kernel (FP16 hi/lo tcgen05 GEMMs, FP32-grade, for the folded-Gram contractions; the default
 *     from 1536 samples: one wave of up to 128 samples per SM takes 4.4-4.7 ms at T = 3000 whatever its size),
 * 6 = run-time-rank tensor-core kernel (any ranks up to 16 per mode with a roll rank <= 8; the folded Gram tensor is
 *     streamed through a shared-memory ring by TMA when it exceeds one tile; the default for every rank set other than
 *     (5,3,3,3), i.e. the enlarged cores of BASELINE.json configs[4]; the reference takes the ranks from the arrays,
 *     TD_Inference.py:56-57). */
int nlml_tucker_fit_f32(nlml_tucker_plan* plan, const float* X_dev, int64_t N, int64_t ldx,
                        int iters, float lr, float clip, float* P_out_dev, int64_t ldp,
                        int kernel_hint, void* stream);

/* Same with HOST buffers: chunks the batch, overlaps H2D copy / kernel / D2H copy on two internal
 * streams with pinned staging, returns when P_out_host is complete. */
int nlml_tucker_fit_host_f32(nlml_tucker_plan* plan, const float* X_host, int64_t N, int64_t ldx,
                             int iters, float lr, float clip, float* P_out_host, int64_t ldp);

/* Converged fit: what TD_Tester.Test ships by default is a scipy Powell search over the same objective from
 * p = 0 (/root/reference/TD_Tester.py:164, :191-199).  This entry point reaches the local minimum of that basin
 * with a damped Newton iteration on the exact Hessian (csrc/tucker_math.h tucker_lm_solve), one thread per
 * sample, data-dependent number of evaluations (max_evals; 0 = default 64).  Ranks (5,3,3,3) only
 * (NLML_E_UNSUPPORTED otherwise).  P_out as nlml_tucker_fit_f32 (radians + identity coefficients);
 * evals_out_dev: optional DEVICE int32 [N], evaluations used per sample.  Asynchronous on `stream`. */
int nlml_tucker_solve_f32(nlml_tucker_plan* plan, const float* X_dev, int64_t N, int64_t ldx, int max_evals,
                          float* P_out_dev, int64_t ldp, int32_t* evals_out_dev, void* stream);
/* Same with HOST buffers (pipelined like nlml_tucker_fit_host_f32). */
int nlml_tucker_solve_host_f32(nlml_tucker_plan* plan, const float* X_host, int64_t N, int64_t ldx,
                               int max_evals, float* P_out_host, int64_t ldp);

/* TD_Tester.Test as the reference SHIPS it (/root/reference/TD_Tester.py:162-199): scipy.optimize.minimize(method="Powell")
 * over the float64 objective of :31-58 from p = 0.  scipy is an unpinned third-party dependency of the reference; the
 * algorithm is restated from scipy 1.18.1 (csrc/powell_math.h: bracket, Brent, _linesearch_powell, _minimize_powell with
 * the defaults the reference leaves in place) and the objective is evaluated in the reference's own operation order
 * (np.einsum accumulation order, numpy's pairwise np.sum), so the result equals the reference's BIT FOR BIT, including the
 * number of function evaluations (pinned by tests/golden/powell_golden.npz, 96 outputs of the real reference).
 * One CTA per sample; float64-pipe bound.  P_out: DEVICE float64 [N][ldp] = result.x (radians + identity coefficients);
 * fun_out / nfev_out: optional DEVICE [N] (result.fun, result.nfev).  Asynchronous on `stream`. */
int nlml_tucker_powell_f64(nlml_tucker_plan* plan, const float* X_dev, int64_t N, int64_t ldx, double* P_out_dev,
                           int64_t ldp, double* fun_out_dev, int32_t* nfev_out_dev, void* stream);

/* The Tucker entry points on RAW MediaPipe landmarks: LM holds x,y,z of landmark i at columns 3i..3i+2 (column f =
 * coordinate f % 3 of landmark f / 3), and every kernel's read of a row applies the normalisation of
 * Read_Landmarks_and_Normalizing_using_IPD (/root/reference/helpers/FeatureExtractor.py:30-66, with the nose-tip reference
 * point of :89-90 and the .float() of :105): subtract landmark 1, divide by ||landmark 33 - landmark 263|| (1e-6 when
 * zero), in float64, rounded to float32 -- the same device code as nlml_mlp_forward_landmarks_f32.  Each call computes
 * exactly what its feature twin computes on the normalised rows, bit for bit; kernel_hint, dispatch, asynchrony and the
 * stride rules are the twin's.  The plan needs F >= 792 (landmark 263); NLML_E_INVALID otherwise.  Filtering the
 * all-zero "no face" rows of the reference's callers stays the caller's job.  nlml_tucker_powell_landmarks_f64 equals the
 * reference's FE.get_feature_vector(..., normalize=True) -> TD_Tester.Test chain bit for bit. */
int nlml_tucker_fit_landmarks_f32(nlml_tucker_plan* plan, const float* LM_dev, int64_t N, int64_t ldx,
                                  int iters, float lr, float clip, float* P_out_dev, int64_t ldp,
                                  int kernel_hint, void* stream);
int nlml_tucker_fit_landmarks_host_f32(nlml_tucker_plan* plan, const float* LM_host, int64_t N, int64_t ldx,
                                       int iters, float lr, float clip, float* P_out_host, int64_t ldp);
int nlml_tucker_solve_landmarks_f32(nlml_tucker_plan* plan, const float* LM_dev, int64_t N, int64_t ldx, int max_evals,
                                    float* P_out_dev, int64_t ldp, int32_t* evals_out_dev, void* stream);
int nlml_tucker_solve_landmarks_host_f32(nlml_tucker_plan* plan, const float* LM_host, int64_t N, int64_t ldx,
                                         int max_evals, float* P_out_host, int64_t ldp);
int nlml_tucker_powell_landmarks_f64(nlml_tucker_plan* plan, const float* LM_dev, int64_t N, int64_t ldx, double* P_out_dev,
                                     int64_t ldp, double* fun_out_dev, int32_t* nfev_out_dev, void* stream);

/* Test hook: phase A of the (5,3,3,3) kernels as the tensor-core GEMM the converged solve uses from 4096 samples on
 * (3xTF32 tcgen05, raw FP32 X tiles by TMA): q = W2 x, CTA-blocked, Q_out_dev [ceil(N/128)][136][128]
 * (q[r] of sample s at ((s / 128) * 136 + r) * 128 + s % 128).  Synchronous. */
int nlml_debug_project_tc(nlml_tucker_plan* plan, const float* X_dev, int64_t N, int64_t ldx, float* Q_out_dev);

/* Test hook: TD_Tester.objective of ONE sample x_dev [F] at npts parameter points pts_dev [npts][3 + r_id] (float64),
 * evaluated by the Powell kernel's cooperative objective -> vals_dev [npts]. */
int nlml_debug_powell_objective(nlml_tucker_plan* plan, const float* x_dev, const double* pts_dev, int npts, double* vals_dev);

/* Offline steps that produce the hot path's constants (SURVEY.md section 8f row 4).
 * nlml_cosine_fit_f64 = TD_Trainer.Train for one factor matrix (/root/reference/TD_Trainer.py:232-351): per column the
 * Fourier initial guess of est_params_by_Uniform_Fourier (:125-148), then scipy Powell on the least-squares objective
 * (:38-43, :60-93), float64, one GPU thread per column.  U_host [n_rows][n_cols] row-major (rows = angle bins), w_deg_host
 * [n_rows] the bins in degrees; params_out_host [n_cols][4] = (a, b, c, d); optional init_out_host [n_cols][4],
 * fun_out_host [n_cols], nfev_out_host [n_cols].  HOST pointers (the matrices are tiny).  Synchronous. */
int nlml_cosine_fit_f64(const double* U_host, int n_rows, int n_cols, const double* w_deg_host, double* params_out_host,
                        double* init_out_host, double* fun_out_host, int32_t* nfev_out_host, int device);
/* nlml_core_times_features_f32 = W = core x_5 U_feat (/root/reference/TD_main.py:231-238): core_host [R][M] (R = product of
 * the four mode ranks, M = feature rank), U_feat_host [F][M] -> W_out_host [R][F].  HOST pointers.  Synchronous. */
int nlml_core_times_features_f32(const float* core_host, const float* U_feat_host, int64_t R, int M, int F, float* W_out_host,
                                 int device);

/* Number of kernel launches issued by this plan so far (for bench.py's gpu_launches). */
int64_t nlml_tucker_launch_count(const nlml_tucker_plan* plan);

/* ------------------------------------------------------------------------------------------
 * Encoder + yaw/pitch/roll heads  (replaces CombinedAnglePredictionModel.forward,
 * NLML_HPE_Model_Builder.py:115-126)
 * ------------------------------------------------------------------------------------------ */
typedef struct nlml_mlp_plan nlml_mlp_plan;

#define NLML_MLP_ENCODER_LAYERS 6 /* NLML_HPE_Model_Builder.py:33-53 */
#define NLML_MLP_HEAD_LAYERS 5    /* NLML_HPE_Model_Builder.py:76-92 */
#define NLML_MLP_NUM_TENSORS (NLML_MLP_ENCODER_LAYERS + 3 * NLML_MLP_HEAD_LAYERS) /* 21 Linear layers */

/* weights[i] / biases[i]: HOST float32, nn.Linear layout weight[out][in], bias[out]; order =
 * encoder.{0,2,4,6,8,10}, yaw model.{0,2,4,6,8}, pitch model.{...}, roll model.{...}
 * (the state_dicts loaded at NLML_HPE_Model_Builder.py:202,214-216).  out_dims/in_dims give each
 * layer's shape; the chain must be consistent (encoder out = 3 * head in).  Activations are fixed by
 * the reference: encoder ReLU x4, Tanh, none; heads ReLU x4, none. */
int nlml_mlp_plan_create(const float* const* weights, const float* const* biases,
                         const int* out_dims, const int* in_dims, int device,
                         nlml_mlp_plan** plan_out);
void nlml_mlp_plan_destroy(nlml_mlp_plan* plan);

/* X: DEVICE float32 [N][ldx]; YPR_out: DEVICE float32 [N][3] = (yaw, pitch, roll) radians.
 * Asynchronous on `stream`.
 * Range: the default (tensor-core) path carries every activation as two FP16 planes, so inputs and hidden
 * activations must stay within +-65504 (IPD-normalised landmarks are O(1)).  Beyond that the hi plane
 * overflows and the affected rows come back NON-FINITE -- never finite-but-wrong; nlml_mlp_set_path(plan, 1)
 * (FP32 CUDA-core chain, the reference's arithmetic) serves such inputs.  Pinned by
 * tests/test_mlp_gpu.py::test_out_of_range_inputs_fail_loudly. */
int nlml_mlp_forward_f32(nlml_mlp_plan* plan, const float* X_dev, int64_t N, int64_t ldx,
                         float* YPR_out_dev, void* stream);
/* HOST buffers, chunked and pipelined like nlml_tucker_fit_host_f32. */
int nlml_mlp_forward_host_f32(nlml_mlp_plan* plan, const float* X_host, int64_t N, int64_t ldx,
                              float* YPR_out_host);
/* Feature-side pre/post steps of the reference's callers (SURVEY.md section 8f row 3).
 *
 * nlml_mlp_forward_landmarks_f32: like nlml_mlp_forward_f32, but LM_dev holds RAW MediaPipe landmarks
 * (x,y,z of landmark i at columns 3i..3i+2) and the normalisation of
 * Read_Landmarks_and_Normalizing_using_IPD (/root/reference/helpers/FeatureExtractor.py:30-66, with the nose-tip
 * reference point of :89-90 and the .float() of :105) is fused into the first kernel's load stage: subtract
 * landmark 1, divide by ||landmark 33 - landmark 263|| (1e-6 when zero), in float64, rounded to float32.
 * Tensor-core path only (NLML_E_UNSUPPORTED after nlml_mlp_set_path(plan, 1)). */
int nlml_mlp_forward_landmarks_f32(nlml_mlp_plan* plan, const float* LM_dev, int64_t N, int64_t ldx,
                                   float* YPR_out_dev, void* stream);
/* The same with HOST buffers (MediaPipe delivers its landmarks on the host), pipelined like nlml_mlp_forward_host_f32. */
int nlml_mlp_forward_landmarks_host_f32(nlml_mlp_plan* plan, const float* LM_host, int64_t N, int64_t ldx,
                                        float* YPR_out_host);
/* nlml_pose_postprocess_f64: YPR_dev float32 [N][3] radians -> DEG_out_dev float64 [N][3]:
 * round(np.degrees(t.item()), decimals) as NLML_HPE_Test.py:273 (decimals 3) / generatePose_on_video.py:210
 * (decimals 2) and, when 0 < ema_alpha < 1, the exponential smoothing over consecutive rows (= video frames) of
 * generatePose_on_video.py:215-224 (alpha 0.4 there).  Bit-identical to the Python statements. */
int nlml_pose_postprocess_f64(const float* YPR_dev, int64_t N, int decimals, double ema_alpha,
                              double* DEG_out_dev, void* stream);
/* Encoder output only: LAT_out DEVICE float32 [N][latent] (for stage-wise parity checks). */
int nlml_mlp_latent_f32(nlml_mlp_plan* plan, const float* X_dev, int64_t N, int64_t ldx,
                        float* LAT_out_dev, void* stream);
int64_t nlml_mlp_launch_count(const nlml_mlp_plan* plan);
/* Kernel generation used for the wide layers: 0 (default) = tcgen05 tensor-core chain (FP16 hi/lo operand
 * split, 3 MMAs per MAC, FP32 TMEM accumulation) wherever a layer is a real dense contraction; 1 = FP32
 * CUDA-core chain for every layer (the exact-arithmetic path the tensor-core chain is validated against). */
int nlml_mlp_set_path(nlml_mlp_plan* plan, int path);

/* ------------------------------------------------------------------------------------------
 * Measurement helper: sustained FP32 FMA rate of the device (TFLOP/s), used by bench.py as the
 * denominator of the Tucker-fit kernel's FP32-pipe roofline.  Runs a register-only FFMA loop.
 * ------------------------------------------------------------------------------------------ */
int nlml_measure_fp32_tflops(int device, double* tflops_out);
/* Same loop with three run-time register operands per FFMA (no immediates): the register-file-limited rate
 * that bounds an FMA stream whose multiplier and addend both change, like the fit kernel's inner loop. */
int nlml_measure_fp32_tflops_3reg(int device, double* tflops_out);

/* Dense TF32 tensor-core rate (TFLOP/s): back-to-back tcgen05.mma.kind::tf32 128x256x8 from shared-memory operands on
 * every SM.  The denominator of the Tucker-fit kernels' tensor roofline (bench.py measures it live). */
int nlml_measure_tf32_tflops(int device, double* tflops_out);

/* Test hook (current device): D[128][N] = A[128][K] * B[N][K]^T through the 3xTF32 tcgen05 building block used by
 * the tensor-core Tucker iteration.  K in 8..64 (multiple of 8), N in 16..256 (multiple of 16).  Synchronous. */
int nlml_debug_tf32_gemm(const float* A_dev, const float* B_dev, int K, int N, float* D_dev);
/* mode 0: as above.  mode 1: the B tile is stored as the K-major image of its transpose and read as an MN-major operand
 * (the form that lets one shared-memory copy of a folded-Gram tile serve both GEMMs of the run-time-rank kernel).
 * mode 2 / 3: the FP16 hi/lo variant (kind::f16, K multiple of 16) with the A operand in shared / tensor memory. */
int nlml_debug_tf32_gemm_mode(const float* A_dev, const float* B_dev, int K, int N, float* D_dev, int mode);

#ifdef __cplusplus
}
#endif
#endif /* NLML_HPE_B200_H */
