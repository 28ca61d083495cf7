/*
 * sparf_b200 -- C ABI of the B200-native SPARF ray-marching hot path.
 *
 * The reference (google-research/sparf) has NO FFI: its boundary for this path is the Python class
 * contract `Graph` / `NeRF` (source/models/renderer.py:28, source/models/frequency_nerf.py:72).  This
 * header is the C ABI we put UNDER that contract; each entry point names the reference code it
 * replaces.  Host-side mirror: sparf_b200/{renderer,frequency_nerf,camera}.py (ctypes, see
 * INTEGRATION.md for the binding a reference maintainer would add).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to fp32 (or int64 where stated) unless marked "host";
 *   - tensors are dense row-major; "R" = rays in the batch (B images x n rays flattened), "S" =
 *     samples per ray; per-sample tensors are [R,S] / [R,S,3];
 *   - all work is enqueued on `stream` (a cudaStream_t); nothing synchronises the device;
 *   - the caller owns every buffer incl. the workspace (sparf_workspace_bytes); no hidden allocation;
 *   - return value 0 = success, otherwise a SPARF_ERR_* code; sparf_last_error() gives the text
 *     (thread-local).  No exceptions cross the ABI.
 *   - gradient outputs of *_backward are ACCUMULATED (+=) into the given buffers so that several
 *     render passes of one step can share one flat gradient buffer (the caller zeroes it once).
 *
 * Process-level state (all of it): the thread-local error string; a launch counter (sparf_launch_count); per device,
 * lazily: the SM count, the kernels' shared-memory attributes, and up to three internal side streams + a few events on which
 * sparf_mlp_backward* runs its small CUDA-core reductions beside the weight-gradient kernel (fork after the dgrad
 * chain, join before the call returns control of `stream`: callers see ordinary stream order, and the pattern is
 * capturable into a CUDA graph).  A workspace must not be shared by calls running concurrently on different streams.
 */
#ifndef SPARF_B200_H_
#define SPARF_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPARF_B200_VERSION 100 /* 0.1.0 */
#define SPARF_MAX_TRUNK 12
#define SPARF_MAX_L 16

enum {
  SPARF_OK = 0,
  SPARF_ERR_INVALID = 1,     /* bad argument / unsupported configuration */
  SPARF_ERR_CUDA = 2,        /* a CUDA runtime call or kernel launch failed */
  SPARF_ERR_WORKSPACE = 3,   /* workspace too small */
  SPARF_ERR_UNSUPPORTED = 4  /* valid request that this build/engine cannot serve */
};

/* Which arithmetic evaluates the MLP GEMMs. */
enum {
  SPARF_ENGINE_AUTO = 0,
  SPARF_ENGINE_SIMT_FP32 = 1, /* CUDA-core FFMA, fp32 throughout (bit-level twin of the reference) */
  SPARF_ENGINE_TC_3X = 2, /* tcgen05: x*W = x_hi*W_hi + x_lo*W_hi + x_hi*W_lo on 16-bit halves (fp16 in the
                             forward, bf16 for gradients), fp32 TMEM accumulation: the parity engine */
  SPARF_ENGINE_TC_1X = 3, /* tcgen05, single 16-bit pass ("fast", NOT within the 1e-4 parity bound) */
  SPARF_ENGINE_TC_3X_W1 = 4 /* TC_3X forward and input / pose gradients (parity), but the wide layers' WEIGHT gradients
                               dW = G^T X in ONE bf16 pass over the hi halves of the saved images (and their bias gradients
                               as column sums of G_hi): the weight-gradient kernel reads half the bytes.  Non-default,
                               reduced precision (8-bit factors; the rounding errors average over the batch):
                               profiles/r02_engine_errors.md tabulates its error against fp64 */
};

typedef void* sparf_stream_t; /* cudaStream_t */

/*
 * View of one reference `NeRF` module (frequency_nerf.py:87-134): trunk `mlp_feat.{i}` and colour
 * head `mlp_rgb.{0,1}`; weights are the nn.Linear tensors themselves, [out,in] row-major fp32.
 *   trunk layer i: in = (i==0 ? E3 : width) + (i==skip_layer ? E3 : 0), out = width (+1 on the last:
 *                  row 0 = raw density, rows 1.. = features), E3 = 3 + 6*L_xyz
 *   head 0: in = width + Ev, out = head_width, Ev = 3 + 6*L_view;  head 1: in = head_width, out = 3
 * BARF coarse-to-fine (frequency_nerf.py:244-257): if use_c2f, the kernel reads the device scalar
 * `progress` (NeRF.progress) and applies w_j = (1-cos(pi*clamp((p-c2f_start)/c2f_range*L - j,0,1)))/2.
 */
typedef struct SparfMLP {
  int32_t n_trunk;    /* 8 */
  int32_t width;      /* 256 */
  int32_t head_width; /* 128 */
  int32_t skip_layer; /* 4; -1 = none */
  int32_t L_xyz;      /* 10 */
  int32_t L_view;     /* 4 */
  int32_t use_c2f;    /* opt.barf_c2f is not None */
  float c2f_start;    /* float(start) */
  float c2f_range;    /* float(end - start), the subtraction done in double like the reference's python floats */
  const float* progress; /* device scalar, may be NULL iff !use_c2f */
  const float* trunk_w[SPARF_MAX_TRUNK];
  const float* trunk_b[SPARF_MAX_TRUNK];
  const float* head_w[2];
  const float* head_b[2];
} SparfMLP;

/* Gradient destinations, same shapes as SparfMLP's tensors (param.grad storage). Accumulated. */
typedef struct SparfMLPGrad {
  float* trunk_w[SPARF_MAX_TRUNK];
  float* trunk_b[SPARF_MAX_TRUNK];
  float* head_w[2];
  float* head_b[2];
} SparfMLPGrad;

/* ---------------------------------------------------------------- misc */
int sparf_version(void);
const char* sparf_last_error(void);
/* number of CUDA kernels this library has launched so far in this process (bench.py: gpu_launches) */
uint64_t sparf_launch_count(void);
/* 1 if the library was built with the tcgen05 engine and the current device is sm_100 */
int sparf_engine_available(int engine);

/* ---------------------------------------------------------------- rays
 * camera.get_center_and_ray / get_center_and_ray_at_pixels (source/utils/camera.py:347-416), computed
 * only for the requested pixels (the reference builds the whole H*W grid and indexes it,
 * renderer.py:273-291).  pose_w2c [B,3,4], intr_inv [B,3,3] = K^-1 (host code inverts K).
 *   ray_idx: int64 [n] (shared, idx_per_image=0) or [B,n] (idx_per_image=1), pixel = (x+0.5,y+0.5),
 *            idx = y*W+x;   or pixels: fp32 [n,2] / [B,n,2] used as given (no +0.5).
 * Exactly one of ray_idx / pixels is non-NULL.  Outputs origins, dirs: [B*n,3].
 */
int sparf_raygen_forward(int32_t B, int32_t n, int32_t W, const float* pose_w2c, const float* intr_inv,
                         const int64_t* ray_idx, const float* pixels, int32_t per_image,
                         float* origins, float* dirs, sparf_stream_t stream);
/* d(origins), d(dirs) [B*n,3] -> d(pose_w2c) [B,3,4], accumulated (+=).  d_pixels (optional, float-pixel path only):
 * gradient w.r.t. the pixel locations, same shape as `pixels` -- written for per-image pixels [B,n,2], accumulated (+=,
 * caller zeroes) for a shared [n,2] list.  The reference's get_center_and_ray_at_pixels is differentiable in the pixels
 * and the depth-consistency loss relies on it (depth_cons_loss.py:247-283). */
int sparf_raygen_backward(int32_t B, int32_t n, int32_t W, const float* pose_w2c, const float* intr_inv,
                          const int64_t* ray_idx, const float* pixels, int32_t per_image,
                          const float* d_origins, const float* d_dirs, float* d_pose_w2c, float* d_pixels,
                          sparf_stream_t stream);

/* ---------------------------------------------------------------- depth samples
 * Graph.sample_depth (renderer.py:383-419) and sample_depth_diff_max_range_per_ray (:595-624).
 *   t[r,k] = ((u + k)/S) * range + near,  u = rand[r,k] (rand != NULL) or 0.5, or 1.0 when far_per_ray
 *   is given (then range = far_per_ray[r] - near);  inverse != 0 -> t = 1/(t + 1e-8).
 */
int sparf_sample_depth(int32_t R, int32_t S, float near, float range, int32_t inverse, const float* rand,
                       const float* far_per_ray, float* t, sparf_stream_t stream);

/* Graph.sample_depth_from_pdf + cat + sort (renderer.py:421-456, :334-336).
 *   weights [R,S], t_coarse [R,S], u [S_fine] = mid-points of the shared grid, bins = linspace(near,far,S+1)
 *   outputs t_fine [R,S_fine] (may be NULL) and t_all [R,S+S_fine] ascending. */
int sparf_sample_pdf_merge(int32_t R, int32_t S, int32_t S_fine, float near, float far, const float* weights,
                           const float* t_coarse, const float* u, float* t_fine, float* t_all,
                           sparf_stream_t stream);

/* ---------------------------------------------------------------- MLP
 * NeRF.forward_samples (frequency_nerf.py:260-281): x = o + t*d, positional encoding, trunk, softplus
 * density (+ noise[R,S] on the raw value when non-NULL), colour head, sigmoid.
 * Outputs sigma [R,S], rgb [R,S,3].
 * sparf_mlp_workspace_bytes: `backward` = 0 forward call, 1 sparf_mlp_backward (recompute), 2 sparf_mlp_backward_tape.
 */
size_t sparf_mlp_workspace_bytes(const SparfMLP* mlp, int32_t R, int32_t S, int32_t backward, int32_t engine);
int sparf_mlp_forward(const SparfMLP* mlp, int32_t engine, int32_t R, int32_t S, const float* origins,
                      const float* dirs, const float* t, const float* noise, float* sigma, float* rgb,
                      void* workspace, size_t workspace_bytes, sparf_stream_t stream);
/* Backward of the above (activations are recomputed, nothing is kept from the forward call).
 * d_sigma [R,S], d_rgb [R,S,3] -> parameter grads (+=) and, when non-NULL, d_origins/d_dirs [R,3] (+=). */
int sparf_mlp_backward(const SparfMLP* mlp, int32_t engine, int32_t R, int32_t S, const float* origins,
                       const float* dirs, const float* t, const float* noise, const float* d_sigma,
                       const float* d_rgb, const SparfMLPGrad* grad, float* d_origins, float* d_dirs,
                       void* workspace, size_t workspace_bytes, sparf_stream_t stream);

/* Tape variants (tcgen05 engine): the TRAINING forward additionally dumps, into a caller-held `tape`, the per-layer
 * operand images the backward needs, so that sparf_mlp_backward_tape skips the recompute.  The tape must stay
 * untouched between the two calls.  sparf_mlp_tape_bytes returns 0 when no tape is available for this call
 * (SIMT engine, unsupported shape, or a tape above 64 GB): use the recompute pair then.  Batches larger than one
 * backward chunk (1024 row tiles) keep ONE tape and walk it chunk by chunk in the backward.
 * Outputs and numerics of the forward are identical to sparf_mlp_forward. */
size_t sparf_mlp_tape_bytes(const SparfMLP* mlp, int32_t engine, int32_t R, int32_t S);
int sparf_mlp_forward_tape(const SparfMLP* mlp, int32_t engine, int32_t R, int32_t S, const float* origins,
                           const float* dirs, const float* t, const float* noise, float* sigma, float* rgb,
                           void* tape, size_t tape_bytes, void* workspace, size_t workspace_bytes,
                           sparf_stream_t stream);
int sparf_mlp_backward_tape(const SparfMLP* mlp, int32_t engine, int32_t R, int32_t S, const float* origins,
                            const float* dirs, const float* t, const float* sigma, const float* rgb,
                            const float* d_sigma, const float* d_rgb, const SparfMLPGrad* grad, float* d_origins,
                            float* d_dirs, void* tape, size_t tape_bytes, void* workspace, size_t workspace_bytes,
                            sparf_stream_t stream);

/* ---------------------------------------------------------------- compositing
 * NeRF.composite (frequency_nerf.py:283-343).  Outputs: rgb_map [R,3], depth/opacity/depth_var/rgb_var
 * [R], weights [R,S], all_cumulated [R] (= T at sample S-2).  white_bg: rgb += 1 - opacity.
 */
int sparf_composite_forward(int32_t R, int32_t S, const float* sigma, const float* rgb, const float* t,
                            const float* dirs, int32_t white_bg, float* rgb_map, float* depth,
                            float* opacity, float* depth_var, float* rgb_var, float* weights,
                            float* all_cumulated, sparf_stream_t stream);
/* Grads of (rgb_map, depth, opacity[, weights]) -> d_sigma [R,S], d_rgb [R,S,3] (written, not
 * accumulated) and d_dirs [R,3] (+=, through the ray length; may be NULL).  g_weights may be NULL. */
int sparf_composite_backward(int32_t R, int32_t S, const float* sigma, const float* rgb, const float* t,
                             const float* dirs, int32_t white_bg, const float* g_rgb_map,
                             const float* g_depth, const float* g_opacity, const float* g_weights,
                             float* d_sigma, float* d_rgb, float* d_dirs, sparf_stream_t stream);

/* ---------------------------------------------------------------- losses
 * 2*mean Huber(delta=0.5) of pred-target over n elements (base_losses.py:155-156): writes the scalar
 * loss (+=, pre-scaled by `scale`) and d_pred = scale * dLoss/dpred. */
int sparf_huber2_fwd_bwd(int64_t n, const float* pred, const float* target, float scale, float* loss,
                         float* d_pred, sparf_stream_t stream);

/* mip-NeRF-360 distortion regulariser of the renderer's (t, weights) [R,S] (regularization_losses.py:20-48 as called
 * from base_losses.py:166-172; default off in the reference's configs): loss += scale * mean over rays; d_w [R,S] and,
 * if not NULL, d_t [R,S] are WRITTEN with scale * dLoss/d.  O(S) per ray (prefix sums over the monotone mid-points)
 * instead of the reference's [S-1, S-1] matrix. */
/* ---------------------------------------------------------------- stand-alone positional encoding
 * FrequencyEmbedder.__call__ + the BARF mask of NeRF.positional_encoding (frequency_nerf.py:47-69, 229-258) as a tensor
 * op: x [n, channels] -> out [n, 2 * channels * L] (per channel L sines then L cosines, f_j = 2^j pi, times the c2f
 * weight when use_c2f).  The MLP entry points fuse this; it exists so that the mirrored methods work on their own.
 * Backward: d_out -> d_x [n, channels] (written). */
int sparf_posenc_forward(int64_t n, int32_t channels, int32_t L, const float* x, int32_t use_c2f, float c2f_start,
                         float c2f_range, const float* progress, float* out, sparf_stream_t stream);
int sparf_posenc_backward(int64_t n, int32_t channels, int32_t L, const float* x, int32_t use_c2f, float c2f_start,
                          float c2f_range, const float* progress, const float* d_out, float* d_x, sparf_stream_t stream);

int sparf_distortion_fwd_bwd(int32_t R, int32_t S, const float* t, const float* w, float scale, float* loss,
                             float* d_w, float* d_t, sparf_stream_t stream);

/* ---------------------------------------------------------------- parameter update (SURVEY.md 8f.1)
 * One optimiser group over FLAT fp32 buffers of n elements: non-finite-gradient check (a bad gradient skips the
 * update), clip_grad_norm_(max_norm; <= 0: none), torch.optim.Adam (betas, eps, no weight decay / amsgrad) with
 * lr = lr0 * gamma^(k-1) [* min(1, k / warmup_steps) if warmup_steps > 0] at iteration k = step[1] + 1 and bias
 * corrections of update t = step[0] + 1; then step[1] = k and, unless skipped, step[0] = t.  Replaces iter_based_trainer.py:128-147 (after_backward), nerf_trainer.py:181-204 (Adam +
 * ExponentialLR) and joint_pose_nerf_trainer.py:513-549 (update_parameters).  `step` (two int64) and `scratch`
 * (>= 4 doubles, zero before the first call) live in device memory: no host round trip, CUDA-graph capturable. */
int sparf_adam_step(int64_t n, float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t* step,
                    double* scratch, double lr0, double gamma, double warmup_steps, double beta1, double beta2,
                    double eps, double max_norm, sparf_stream_t stream);

/* ---------------------------------------------------------------- diagnostics
 * Minimal tcgen05 GEMM exercising every Blackwell primitive of the tensor-core engine (operand layout,
 * descriptors, bulk copy, TMEM): D[128,128] = bf16(A[128,K]) * bf16(B[128,K])^T, K in {64,...,256}.
 * `packed` is >= 128*K*2 bytes of scratch.  Used by tests/test_tc_engine.py. */
int sparf_tc_selftest(const float* A, const float* B, int32_t K, void* packed, float* D, sparf_stream_t stream);
/* Same GEMM with the A operand written to and read from tensor memory (tcgen05.st, tcgen05.mma with A in TMEM). */
int sparf_tc_selftest_ts(const float* A, const float* B, int32_t K, void* packed, float* D, sparf_stream_t stream);
/* Same for the weight-gradient shape: D[128,128] = G[rows,128]^T X[rows,128] through MN-major descriptors. */
int sparf_tc_selftest_tn(const float* G, const float* X, int32_t rows, float* D, sparf_stream_t stream);
/* probe: same with G in bf16 and X in fp16 (mixed operand formats in one kind::f16 instruction) */
int sparf_tc_selftest_tn_mixed(const float* G, const float* X, int32_t rows, float* D, sparf_stream_t stream);

/* Micro-benchmark of cp.async.bulk L2->shared throughput per SM vs copies in flight (tools/probe_bulkcopy.py). */
int sparf_tc_bulkcopy_probe(const void* src, uint32_t src_bytes, int32_t stages, uint32_t chunk, int32_t iters,
                            int32_t grid, long long* cycles, sparf_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* SPARF_B200_H_ */
