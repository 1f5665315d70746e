/* hgru_b200.h -- C ABI of the B200-native hGRU-pose forward (libhgru_b200.so).
 *
 * The reference (krg-nandu/monkey-pose) is pure Python/TensorFlow and has no FFI; this header is
 * the drop-in boundary a maintainer binds (ctypes, see INTEGRATION.md) in place of the TF graph
 * nodes the two reference classes build.  Every entry point cites the reference interface it
 * replaces (paths relative to the reference checkout).
 *
 * Conventions
 *   - all tensors are dense row-major float32; activations NHWC, conv weights HWIO (TF layout);
 *   - `*_dev` pointers are CUDA device pointers, `*_host` pointers are host memory (pinned
 *     recommended); nothing here takes torch / framework types;
 *   - `stream` is a cudaStream_t passed as void* (0 = default stream); calls are asynchronous and
 *     stream-ordered unless stated otherwise;
 *   - every function returns 0 on success, non-zero on failure (HGRU_E_*); the message of the
 *     last failure on the calling thread is available from hgru_last_error(); nothing aborts;
 *   - one plan per GPU; a plan is not re-entrant (use it from one thread / stream at a time);
 *   - a plan's N is its capacity: the *_forward_batch entry points run any batch of 1 <= n <= N frames on it (the
 *     reference's placeholders have a run-time batch dimension), every tensor argument then has n frames, and the
 *     result equals that of a plan created for n frames, bit for bit.  The plain *_forward calls are the n = N case.
 *     An n outside [1, N] returns HGRU_E_INVALID before any CUDA call.
 */
#ifndef HGRU_B200_H_
#define HGRU_B200_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define HGRU_API __attribute__((visibility("default")))
#else
#define HGRU_API
#endif

#define HGRU_OK 0
#define HGRU_E_INVALID 1      /* bad shape / argument                                  */
#define HGRU_E_UNSUPPORTED 2  /* option the kernels do not implement                   */
#define HGRU_E_CUDA 3         /* CUDA runtime / driver error (see hgru_last_error)     */
#define HGRU_E_STATE 4        /* call order violation (e.g. forward before set_params) */

/* arithmetic of the horizontal convolutions (everything else is fp32 in every mode) */
#define HGRU_MODE_FP32 0 /* fp32 SIMT FFMA: the <= 1e-4 parity path                                */
#define HGRU_MODE_BF16 1 /* tcgen05 tensor cores, bf16 operands, fp32 accumulate + fp32 state      */
#define HGRU_MODE_BF16X3 2 /* tcgen05, bf16 hi/lo operand splits (3 products): fp32-class accuracy, S = 15    */
/* tcgen05, fp16 operands (11 significand bits, bf16: 8) at the bf16 mode's speed; otherwise the bf16 mode.  S = 15,
 * k <= 64.  Conversions saturate at +-65504 (never inf / NaN): an initial state beyond that is clamped in the first
 * timestep's gated operand. */
#define HGRU_MODE_FP16 3

typedef struct hgru_plan_s* hgru_plan_t;
typedef struct pose_plan_s* pose_plan_t;

HGRU_API const char* hgru_last_error(void);
HGRU_API int hgru_version(void);

/* ------------------------------------------------------------------------------------------
 * Recurrent layer: replaces hgru_module.ContextualCircuit (hgru_module.py:54-959) on the path
 * hgru_pose.py configures (aux dict hgru_pose.py:20-39: tanh, gru_gates, multiplicative_excitation,
 * gamma, adapation; 'alternate' integration).
 * ------------------------------------------------------------------------------------------ */

/* ContextualCircuit.__init__ (hgru_module.py:61-128): static shape [N,H,W,k] of X (:74),
 * S = SSF_ext = 2*floor(SSF/2)+1 (:94-97), T = timesteps.  Allocates all workspace. */
HGRU_API int hgru_plan_create(int N, int H, int W, int k, int S, int T, int mode, hgru_plan_t* out);
HGRU_API int hgru_plan_destroy(hgru_plan_t plan);

/* prepare_tensors (hgru_module.py:172-503): the variables of scope `contextual_circuit`.
 * p_r [S,S,k,k]; i_r, o_r [1,1,k,k]; i_b, o_b, beta, nu, gamma, kappa, omega, lateral_bias
 * [1,1,1,k]; rho [T].  Device pointers; copied/packed into plan-owned storage. */
HGRU_API int hgru_set_params(hgru_plan_t plan, const float* p_r_dev, const float* i_r_dev,
                    const float* i_b_dev, const float* o_r_dev, const float* o_b_dev,
                    const float* beta_dev, const float* nu_dev, const float* gamma_dev,
                    const float* kappa_dev, const float* omega_dev, const float* rho_dev,
                    const float* lateral_bias_dev, void* stream);

/* build() (hgru_module.py:872-959): T iterations of `full` (:825-857).
 * X, H2_init, H2_out: [N,H,W,k].  H2_init is the reference's O_0 (:884-887), explicit here.
 * H1_trace / H2_trace: NULL or [T,N,H,W,k] buffers receiving I / O after every timestep. */
HGRU_API int hgru_forward(hgru_plan_t plan, const float* X_dev, const float* H2_init_dev, float* H2_out_dev,
                 float* H1_trace_dev, float* H2_trace_dev, void* stream);
/* The same over n frames (1 <= n <= N): X, H2_init, H2_out [n,H,W,k], traces [T,n,H,W,k]. */
HGRU_API int hgru_forward_batch(hgru_plan_t plan, int n, const float* X_dev, const float* H2_init_dev,
                                float* H2_out_dev, float* H1_trace_dev, float* H2_trace_dev, void* stream);

HGRU_API size_t hgru_plan_workspace_bytes(hgru_plan_t plan);
/* number of kernels the last hgru_forward launched */
HGRU_API int hgru_plan_launch_count(hgru_plan_t plan);

/* ------------------------------------------------------------------------------------------
 * Pose model: replaces hgru_pose.model.build (hgru_pose.py:47-105), inference-mode batch norm.
 * ------------------------------------------------------------------------------------------ */

/* Variables of hgru_pose.model by their reference names (hgru_pose.py:165-194, tf.layers BN
 * scopes batch_normalization[_1.._4]); all device pointers. */
typedef struct pose_params_s {
  const float *conv_1_filters, *conv_1_biases; /* [3,3,1,C], [C]   hgru_pose.py:50  */
  const float *conv_2_filters, *conv_2_biases; /* [3,3,C,C], [C]   hgru_pose.py:61  */
  const float *conv_3_filters, *conv_3_biases; /* [3,3,C,C], [C]   hgru_pose.py:71  */
  const float *fc_1_weights, *fc_1_biases;     /* [HW*C,F], [F]    hgru_pose.py:91  */
  const float *fc_out_weights, *fc_out_biases; /* [F,O], [O]       hgru_pose.py:104 */
  /* batch_normalization, _1, _2, _3 (C channels each), _4 (F): gamma, beta, moving_mean,
   * moving_variance  (hgru_pose.py:52-60, 62-70, 72-80, 82-90, 95-103) */
  const float* bn[5][4];
  /* scope contextual_circuit (hgru_module.py:262-503), same order as hgru_set_params */
  const float *p_r, *i_r, *i_b, *o_r, *o_b, *beta, *nu, *gamma, *kappa, *omega, *rho, *lateral_bias;
} pose_params_t;

/* model.__init__ (hgru_pose.py:8-39) + the static shapes of build(): N frames of
 * [2*HW, 2*HW, 1] depth; C = stem / hidden channels (64 in the reference); S = SSF = 15;
 * T = timesteps = 8; F = fc_1 width (1024); O = output_shape (69). */
HGRU_API int pose_plan_create(int N, int HW, int C, int S, int T, int F, int O, int mode, pose_plan_t* out);
HGRU_API int pose_plan_destroy(pose_plan_t plan);
HGRU_API int pose_set_params(pose_plan_t plan, const pose_params_t* params, float bn_epsilon, void* stream);

/* model.build -> self.out_put (hgru_pose.py:47-105).  depth [N,2HW,2HW,1], H2_init [N,HW,HW,C]
 * (NULL = zeros, the reference's hidden_init='zeros'), out [N,O]. */
HGRU_API int pose_forward(pose_plan_t plan, const float* depth_dev, const float* H2_init_dev, float* out_dev,
                 void* stream);
/* Same through host buffers: H2D copy of depth, forward, D2H copy of out, stream-synchronised
 * on return.  H2_init stays a device pointer (it is state, not per-frame input). */
HGRU_API int pose_forward_host(pose_plan_t plan, const float* depth_host, const float* H2_init_dev,
                      float* out_host, void* stream);
/* pose_forward / pose_forward_host over n frames (1 <= n <= N): depth [n,2HW,2HW,1], H2_init [n,HW,HW,C], out [n,O];
 * only n frames are uploaded and read back.  No re-allocation and no re-packing of the parameters. */
HGRU_API int pose_forward_batch(pose_plan_t plan, int n, const float* depth_dev, const float* H2_init_dev,
                                float* out_dev, void* stream);
HGRU_API int pose_forward_host_batch(pose_plan_t plan, int n, const float* depth_host, const float* H2_init_dev,
                                     float* out_host, void* stream);

/* aux['hidden_init'] = 'identity' (hgru_module.py:876-878: O_0 = X, the hGRU's own input): when on, H2_init_dev
 * of the forward calls is ignored and the initial state is conv3 of the same forward.  Off by default. */
HGRU_API int pose_set_hidden_init(pose_plan_t plan, int identity);

/* Intermediate activations of the last pose_forward, by the reference's attribute names
 * ("pool1","conv2","conv3","hgru","fc1"; hgru_pose.py:50-105), copied into dst_dev in the
 * reference's layout ([n,HW,HW,C] / [n,F], n = the last forward's frames).  For parity tests. */
HGRU_API int pose_get_activation(pose_plan_t plan, const char* name, float* dst_dev, void* stream);

HGRU_API size_t pose_plan_workspace_bytes(pose_plan_t plan);
/* kernels the last pose_forward* launched */
HGRU_API int pose_plan_launch_count(pose_plan_t plan);
/* average device time (ms) of the horizontal-conv kernels in the last pose_forward/hgru_forward
 * when timing was enabled with hgru_enable_kernel_timing(plan-independent switch) */
HGRU_API int hgru_enable_kernel_timing(int on);
HGRU_API int pose_plan_kernel_times(pose_plan_t plan, float* hconv_ms_total, int* hconv_launches);
/* SM clock (GHz) the last horizontal-conv launch of the last timed forward actually ran at, measured inside the
 * kernel (clock64 cycles / %globaltimer nanoseconds of every CTA's MMA loop): mean and minimum over its CTAs, 0 when
 * timing was off.  nvidia-smi reports the nominal clock while these kernels run power-limited.  Synchronises. */
HGRU_API int pose_plan_sm_clock_ghz(pose_plan_t plan, float* ghz_mean, float* ghz_min);

/* ------------------------------------------------------------------------------------------
 * Stand-alone layers: the reference model's layer METHODS, for callers that compose the graph themselves the way
 * hgru_pose.model.build does (hgru_pose.py:47-105).  Exact fp32, unfused, any channel counts; pose_forward does not
 * go through these (it runs the fused tensor-core pipeline).  Dense fp32 NHWC activations, HWIO filters.
 *   layer_conv2d_forward      model.conv_layer (hgru_pose.py:139-154): relu?(conv2d(x, filters, stride 1, SAME) + biases)
 *   layer_max_pool2x2_forward model.max_pool (:134-137): 2x2, stride 2, SAME -> [N, ceil(H/2), ceil(W/2), C]
 *   layer_fc_forward          model.fc_layer (:156-163): x [M,K] @ weights [K,F] + biases
 *   layer_batch_norm_forward  tf.layers.batch_normalization(axis = last, momentum, epsilon, training) (:52-103) over
 *       x [rows, C].  training = 0: moving statistics.  training = 1: statistics of the batch (biased variance); when
 *       new_moving_mean / new_moving_var are given they receive moving * momentum + batch * (1 - momentum) (unbiased
 *       batch variance), the update the reference runs through UPDATE_OPS (train_cnn_networks_hgru.py:123-126);
 *       sums_ws = 2*C doubles of device workspace.  relu_first applies tf.nn.relu to x first (:92); dropout_keep < 1
 *       (training only) then applies tf.nn.dropout(x, keep) (:93-94) with a counter-based keep mask: element i is
 *       kept iff (splitmix64(seed ^ i * 0xD1B54A32D192ED03) >> 40) / 2^24 < keep, kept values scaled by 1 / keep.
 * ------------------------------------------------------------------------------------------ */
HGRU_API int layer_conv2d_forward(const float* x_dev, int N, int H, int W, int Cin, const float* filters_dev, int S,
                                  int Cout, const float* biases_dev, int relu, float* out_dev, void* stream);
/* The circuit's per-timestep building blocks as stand-alone exact-fp32 ops, for callers that compose `full()`
 * (hgru_module.py:825-857) themselves through ContextualCircuit.circuit_input / circuit_output / input_integration /
 * output_integration; hgru_forward never runs them (it runs the fused tensor-core pipeline).  Tensors [rows][k]
 * channels-last (rows = n*h*w); the 15x15 convolution between them is layer_conv2d_forward with lateral_bias as bias.
 *   circuit_gate_forward: gate = sigmoid(x *1x1 w + b) (:696-707, 729-740; w [k][k] in x out); gated (nullable) = x . gate
 *     (:709-711).
 *   circuit_input_integration_forward: I = tanh(xi X - (beta . O + nu) . P) (:795-804).
 *   circuit_output_integration_forward: O' = G . O + (1 - G) . tanh(kappa . (zeta I + gamma . P) + omega . (zeta I .
 *     gamma . P)) (:806-823), times *rho_dev when given (full()'s `O * rho[i0]`, :847-849). */
HGRU_API int circuit_gate_forward(const float* x_dev, size_t rows, int k, const float* w_dev, const float* b_dev,
                                  float* gate_dev, float* gated_dev, void* stream);
HGRU_API int circuit_input_integration_forward(const float* X_dev, const float* O_dev, const float* P_dev,
                                               const float* beta_dev, const float* nu_dev, float xi, size_t rows, int k,
                                               float* I_dev, void* stream);
HGRU_API int circuit_output_integration_forward(const float* I_dev, const float* P_dev, const float* O_dev,
                                                const float* G_dev, const float* gamma_dev, const float* kappa_dev,
                                                const float* omega_dev, float zeta, const float* rho_dev, size_t rows,
                                                int k, float* O_out_dev, void* stream);
HGRU_API int layer_max_pool2x2_forward(const float* x_dev, int N, int H, int W, int C, float* out_dev, void* stream);
/* The model's remaining pooling / normalisation helpers (hgru_pose.py:120-132; declared by the reference, not called
 * by its build()): tf.nn.max_pool / avg_pool with ksize = stride = ksize, SAME (max_pool_4: ksize 4; avg_pool: ksize 2,
 * average = 1; padding is left out of an average's count) -> out [N][ceil(H/k)][ceil(W/k)][C]; and `batchnorm` =
 * tf.nn.moments over axis 0 + tf.nn.batch_normalization without scale / offset: x [N][inner] -> (x - mean_n) *
 * rsqrt(var_n + epsilon) per inner index. */
HGRU_API int layer_pool_same_forward(const float* x_dev, int N, int H, int W, int C, int ksize, int average,
                                     float* out_dev, void* stream);
HGRU_API int layer_batchnorm_moments0_forward(const float* x_dev, int N, size_t inner, float epsilon, float* out_dev,
                                              void* stream);
HGRU_API int layer_fc_forward(const float* x_dev, int M, int K, const float* weights_dev, const float* biases_dev,
                              int F, float* out_dev, void* stream);
/* tf.image.resize_images(x, [OH, OW]) of the attention CNN (train_cnn_networks_hgru.py:442): TF 1.x bilinear,
 * align_corners = false, float32 without fused multiply-adds (bit-exact); x [N,H,W] -> out [N,OH,OW]. */
HGRU_API int layer_resize_bilinear_forward(const float* x_dev, int N, int H, int W, int OH, int OW, float* out_dev,
                                           void* stream);
HGRU_API int layer_batch_norm_forward(const float* x_dev, size_t rows, int C, const float* gamma_dev,
                                      const float* beta_dev, const float* moving_mean_dev,
                                      const float* moving_var_dev, float epsilon, int training, int relu_first,
                                      float dropout_keep, unsigned long long dropout_seed, float momentum,
                                      float* new_moving_mean_dev, float* new_moving_var_dev, double* sums_ws_dev,
                                      float* y_dev, void* stream);

/* ------------------------------------------------------------------------------------------
 * Crop stage (the step right before the pose network): replaces the per-frame host loop
 * prepare_data_test -> tfMonkeyDetector.cropArea3D (train_cnn_networks_hgru.py:61-74,
 * tf_monkeydetector.py:208-263, 292-365).  The window arithmetic (comToBounds, :193-206) stays on
 * the host and arrives as per-frame integers; the gather / z clamp / nearest resize / paste /
 * normalise runs on the device, bit-exact with the reference + OpenCV.
 *   frames [N,H,W] (device), multiplied by frame_scale (image_max_depth) as the caller does;
 *   iparams [N][8] = xstart, ystart, wb, hb, sz_w, sz_h, xs, ys;  zparams [N][2] = zstart, zend (fp32);
 *   out [N,dh,dw] = value / out_divisor, `background` where the resized crop does not reach.
 * ------------------------------------------------------------------------------------------ */
HGRU_API int crop_area3d_forward(const float* frames_dev, int N, int H, int W, float frame_scale,
                                 const int* iparams_dev, const float* zparams_dev, float background,
                                 double out_divisor, float* out_dev, int dh, int dw, void* stream);

/* Raw 16-bit depth frames (millimetres) -> float32 frames in [0, 1]: the pre-processing of the reference's real-data
 * loop (eval_model_on_real_data, train_cnn_networks_hgru.py:381-386: `im[im < 1000] = 10000; im[im > 3000] = 10000`)
 * + the division by image_max_depth (:359, :392), on the device: out[i] = (raw[i] < near || raw[i] > far ? fill :
 * raw[i]) / max_depth, quotient in double, rounded once to float32.  count = number of pixels. */
HGRU_API int depth_preprocess_forward(const unsigned short* raw_dev, size_t count, unsigned int near_mm,
                                      unsigned int far_mm, double fill, double max_depth, float* out_dev,
                                      void* stream);

/* The window arithmetic itself on the device: comToBounds (tf_monkeydetector.py:193-206) + the resize / paste integers
 * and the 3x3 joint transform of cropArea3D (:309-362) for a batch, in explicitly rounded IEEE double operations in the
 * reference's evaluation order (the integers equal the host's).  Centres of mass: com_in_dev [N][3] double (u, v, d mm)
 * when given, else attention outputs tr_dev [N][3] float32 times (s0, s1, s2) = (image height, width, max depth) as
 * prepare_data_test scales them (train_cnn_networks_hgru.py:66-68).  Outputs: coms [N][3] double, iparams [N][8] and
 * zparams [N][2] as crop_area3d_forward takes them, Ms [N][3][3] double, invalid [N] (1: the window misses the frame;
 * that frame's crop is all background).  (dw, dh) = destination size; cube in mm. */
HGRU_API int crop_windows_forward(const float* tr_dev, const double* com_in_dev, double s0, double s1, double s2,
                                  int N, int H, int W, int dw, int dh, double fx, double fy, double cube_x,
                                  double cube_y, double cube_z, double* coms_dev, int* iparams_dev,
                                  float* zparams_dev, double* Ms_dev, int* invalid_dev, void* stream);

/* tfMonkeyDetector.calculateCoM (tf_monkeydetector.py:73-90) for a batch on the device: pixels outside
 * [min_depth, max_depth] zeroed, (x, y) = centre of mass of the remaining mask, z = their mean depth.  The mean depth is a
 * float32 numpy.sum in the reference; it is reproduced in numpy's pairwise order, so coms equals the host's bit for bit.
 *   iparams_dev == zparams_dev == NULL: the image is each whole frame [H][W] times frame_scale -- what cropArea3D does
 *     when no centre of mass is given (:307-308).
 *   iparams_dev / zparams_dev as crop_windows_forward wrote them: the image is getCrop's z-clamped window (:208-244) and
 *     the result gets the `docom` refinement of cropArea3D (:316-326): an all-zero centre of mass takes the window's
 *     centre pixel as depth (300 if that is 0 too), then (xstart, ystart) is added.  Feed coms to crop_windows_forward
 *     again for the refined window.
 *   ws_dev: calculate_com_workspace_bytes(N, max_pixels) bytes; a window of more than max_pixels pixels gets a NaN
 *     centre of mass and overflow[n] = 1.  coms_dev [N][3] double (u, v, d). */
HGRU_API size_t calculate_com_workspace_bytes(int N, long long max_pixels);
HGRU_API int calculate_com_forward(const float* frames_dev, int N, int H, int W, float frame_scale, float min_depth,
                                   float max_depth, const int* iparams_dev, const float* zparams_dev,
                                   long long max_pixels, void* ws_dev, double* coms_dev, int* overflow_dev,
                                   void* stream);

/* ------------------------------------------------------------------------------------------
 * Post-processing (the step right after the pose network).
 * pose_postprocess_forward: out_put [N,3J] (normalised) -> xyz [N,J,3] = out*scale + uvdtoxyz(com),
 *   uvd [N,J,3] = xyztouvd(xyz): train_cnn_networks_hgru.py:293-296 + tfMonkeyDetector
 *   .getAbsoluteCoordinates (tf_monkeydetector.py:387-391).  com_uvd [N,3] float64 (u, v, d mm).
 * joint_error_forward: labels / results [N,J,3] (mm) -> result[0] = getMeanError_np,
 *   result[1] = getMaxError_np (pose_evaluation.py:10-23); workspace: N doubles + N floats.
 * ------------------------------------------------------------------------------------------ */
HGRU_API int pose_postprocess_forward(const float* out_put_dev, const double* com_uvd_dev, int N, int J,
                                      double fx, double fy, double ux, double uy, float scale,
                                      float* xyz_dev, float* uvd_dev, void* stream);
HGRU_API int joint_error_forward(const float* labels_dev, const float* results_dev, int N, int J,
                                 double* frame_mean_ws_dev, float* frame_max_ws_dev, double* result_dev,
                                 void* stream);

/* The rest of the reference's metric file on the device (pose_evaluation.py:10-88), in numpy's own float32
 * evaluation order (pairwise sums over contiguous axes, element-by-element sums over the others), so the values are
 * bit-identical to the host functions' on float32 inputs, not merely close.
 * joint_error_stats_forward: labels / results [N][J][3] float32 (mm) ->
 *   err [N][J]      per-joint Euclidean error sqrt(((l - r)^2).sum(axis=2)), the expression every metric starts from;
 *   frame_mean [N]  nanmean(err, axis=1) = getMeanErrors_N (:46-52), the statistic of getNumFramesWithinMeanDist (:72-78);
 *   frame_max [N]   nanmax(err, axis=1), the statistic of getNumFramesWithinMaxDist (:63-69);
 *   joint_mean [J]  nanmean(err[:, j]) = getJointMeanError(labels, results, j) (:81-88) for every joint;
 *   summary [2]     {nanmean(frame_mean) = getMeanError_np / getMeanError_train (:10-15, :30-36),
 *                    nanmax(err) = getMaxError_np / getMaxError (:18-23, :54-60)}.
 *   skip_nan = 1: numpy's nan* functions (NaN joints left out); 0: the TensorFlow variants (a NaN propagates).
 * joint_error_count_within_forward: *count = number of n with frame_stat[n] <= dist (:63-78).
 * axis1_error_mean_forward: getMean_np / getMeanError (:26-28, :38-44): a, b [N][M][C] (C = 1 for rank-2 inputs)
 *   -> rows_ws [N][C] = sqrt(((a - b)^2).sum(axis=1)), out [C] = (nan)mean over axis 0. */
HGRU_API int joint_error_stats_forward(const float* labels_dev, const float* results_dev, int N, int J, int skip_nan,
                                       float* err_dev, float* frame_mean_dev, float* frame_max_dev,
                                       float* joint_mean_dev, float* summary_dev, void* stream);
HGRU_API int joint_error_count_within_forward(const float* frame_stat_dev, int N, float dist, int* count_dev,
                                              void* stream);
HGRU_API int axis1_error_mean_forward(const float* a_dev, const float* b_dev, int N, int M, int C, int skip_nan,
                                      float* rows_ws_dev, float* out_dev, void* stream);

/* ------------------------------------------------------------------------------------------
 * Attention (centre-of-mass) CNN: the network right before the crop stage, reference
 * `attn_model_struct.build` (train_cnn_networks_hgru.py:422-525): bilinear resize to 128x128,
 * 5 x [conv (3,3,3,3,5) + relu -> max-pool -> batch-norm], fc -> relu -> batch-norm -> fc (O = 3 outputs:
 * u/height, v/width, d/max_depth of the centre of mass).  Inference mode (moving statistics).
 * widths = output channels of the five convolutions (reference: 64,128,256,512,1024; multiples of 8),
 * fc_hidden = 1024 in the reference.  Variables arrive under their TF names' meaning:
 *   conv_filters[i] = aconv_<i+1>_filters HWIO, conv_biases[i]; fc_1 = afc_1 [16*widths[4]][fc_hidden];
 *   fc_out = afc_out [fc_hidden][O]; bn[i] = batch_normalization[_i]/{gamma,beta,moving_mean,moving_variance},
 *   i = 0..4 after the pools, 5 after relu(afc_1).  All device pointers, fp32.
 * ------------------------------------------------------------------------------------------ */
typedef struct attn_plan_s* attn_plan_t;
typedef struct {
  const float* conv_filters[5];
  const float* conv_biases[5];
  const float* fc_1_weights;
  const float* fc_1_biases;
  const float* fc_out_weights;
  const float* fc_out_biases;
  const float* bn[6][4];
} attn_params_t;
HGRU_API int attn_plan_create(int N, int H, int W, const int* widths, int fc_hidden, int O, attn_plan_t* out);
/* The same with the arithmetic of the GEMM layers (aconv_2 .. aconv_5, afc_1; aconv_1, afc_out and everything between
 * the GEMMs are fp32 in both): HGRU_MODE_BF16X3 (bf16 hi/lo operand splits, three products per k-step, fp32-class
 * accuracy) is attn_plan_create's plan; HGRU_MODE_FP16 (fp16 operands, 11 significand bits, one product per k-step
 * at the bf16 rate, fp32 accumulate: <= 2.5e-3 relative on every activation).  fp16 conversions saturate at +-65504,
 * never inf / NaN.  Any other mode: HGRU_E_UNSUPPORTED. */
HGRU_API int attn_plan_create_mode(int N, int H, int W, const int* widths, int fc_hidden, int O, int mode,
                                   attn_plan_t* out);
HGRU_API int attn_plan_destroy(attn_plan_t plan);
HGRU_API int attn_set_params(attn_plan_t plan, const attn_params_t* params, float bn_epsilon, void* stream);
/* frames [N,H,W] fp32 (depth / image_max_depth, as the caller feeds the reference graph) -> out [N,O] */
HGRU_API int attn_forward(attn_plan_t plan, const float* frames_dev, float* out_dev, void* stream);
/* The same over n frames (1 <= n <= N): frames [n,H,W], out [n,O].  Each layer's K split is the one a plan created
 * for n frames takes, so the result depends on the batch only, not on the capacity. */
HGRU_API int attn_forward_batch(attn_plan_t plan, int n, const float* frames_dev, float* out_dev, void* stream);
/* name in {"resized","pool1",...,"pool5","fc1"}: dense fp32 NHWC copy of an intermediate tensor of the last
 * forward (its n frames) */
HGRU_API int attn_get_activation(attn_plan_t plan, const char* name, float* dst_dev, void* stream);
HGRU_API size_t attn_plan_workspace_bytes(attn_plan_t plan);
HGRU_API int attn_plan_launch_count(attn_plan_t plan);

#ifdef __cplusplus
}
#endif
#endif /* HGRU_B200_H_ */
