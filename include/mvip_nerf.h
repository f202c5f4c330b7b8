/*
 * mvip_nerf.h — C ABI of libmvip_nerf.so: the B200 (sm_100a) implementation of MVIP-NeRF's
 * volume-rendering hot path.
 *
 * The reference has no FFI on this path (it is Python calling torch ops); the only FFI precedent in
 * its tree is DS_NeRF/torchsearchsorted/src/cuda/searchsorted_cuda_wrapper.cpp:9-20 (caller
 * pre-allocates outputs, tensors must be CUDA + contiguous, library allocates nothing).  This header
 * keeps that contract and adds an explicit stream.  Each entry point names the reference code it
 * replaces (paths relative to the reference root).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the parameter is documented as "host array";
 *   - all buffers (inputs, outputs, stash, workspace) are owned by the caller; the library never
 *     allocates or frees device memory and never synchronises the stream;
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream);
 *   - return value: 0 = OK, negative = error (MVIP_E_*); mvip_last_error() gives a thread-local
 *     message.  There is no CPU fallback: without a CUDA device every compute call fails.
 *   - tensors are row-major and contiguous unless a stride parameter is given (strides in elements).
 */
#ifndef MVIP_NERF_H_
#define MVIP_NERF_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MVIP_ABI_VERSION 1

#define MVIP_OK 0
#define MVIP_E_INVALID (-1)     /* null / misaligned / out-of-range argument              */
#define MVIP_E_UNSUPPORTED (-2) /* shape outside what the kernels implement                */
#define MVIP_E_CUDA (-3)        /* CUDA runtime error (launch failure, no device, ...)     */

int mvip_abi_version(void);
const char* mvip_last_error(void);
/* compute capability of the current device as major*10+minor (e.g. 100), or <0 on error */
int mvip_device_arch(void);

/* ------------------------------------------------------------------------------------------------
 * Camera rays of a pinhole view, packed as the ray batch of the hot path.
 *   replaces DS_NeRF/run_nerf_helpers.py:249-260 (get_rays) + the batch assembly of render(), run.py:1171-1207
 *   c2w        [3,4] row-major camera-to-world pose (DEVICE pointer, 12 floats)
 *   c2w_static nullable [3,4]: if given, rays_o / rays_d come from this pose and only the view directions
 *              from c2w (the c2w_staticcam option, run.py:1180-1183)
 *   window     rows [i0, i0+h) x columns [j0, j0+w) of the H x W image (the `patch` option; whole image: 0,0,H,W)
 *   out        [h*w, 8 + 3*use_viewdirs]: o(0:3) d(3:6) near far [viewdir(8:11) = d_c2w / |d_c2w|]
 * Bit-exact against the reference's CPU result.
 */
int mvip_rays_from_pose(const float* c2w, const float* c2w_static, int H, int W, float focal, float near,
                        float far, int i0, int j0, int h, int w, int use_viewdirs, float* out, void* stream);
/* Same, with the NDC warp of DS_NeRF/run_nerf_helpers.py:283-300 (ndc_rays) applied to o / d when ndc != 0 (the view
 * directions stay those of the un-warped rays, run.py:1176-1190).  `focal` and `ndc_near` are doubles because the reference
 * forms -1/(W/(2 focal)) and 2*near as Python floats before they meet an fp32 tensor; render() passes ndc_near = 1. */
int mvip_rays_from_pose_ndc(const float* c2w, const float* c2w_static, int H, int W, double focal, float near,
                            float far, int i0, int j0, int h, int w, int use_viewdirs, int ndc, double ndc_near,
                            float* out, void* stream);
/* The `rays=` entry of render() (DS_NeRF/run.py:1176-1207): given rays_o / rays_d [n,3] (and optionally the directions the
 * view vectors are taken from, view_d [n,3], NULL = rays_d) -> the packed batch [n, 8 + 3*use_viewdirs] in one launch
 * (viewdir normalisation, optional ndc_rays, near / far columns, cat).  H, W, focal, ndc_near are read only when ndc != 0. */
int mvip_rays_pack(const float* rays_o, const float* rays_d, const float* view_d, int64_t n, float near, float far,
                   int use_viewdirs, int ndc, int H, int W, double focal, double ndc_near, float* out, void* stream);

/* Backward of the two entries above (autograd of the reference's fp32 formulas, in fp32): g_out [n, 8 + 3*use_viewdirs] is the
 * gradient of the packed batch; the near / far columns carry none.
 *   mvip_rays_pack_backward: -> g_rays_o, g_rays_d [n,3] (overwritten); g_view_d [n,3] when view_d is given (else the view
 *     vectors' gradient is added to g_rays_d).
 *   mvip_rays_from_pose_backward: -> g_c2w [3,4] (overwritten); with c2w_static (then g_c2w_static is required, and only then),
 *     g_c2w gets the view-direction part and g_c2w_static [3,4] the rays_o / rays_d part.  Bitwise reproducible: per-block partials in `workspace`
 *     (mvip_rays_from_pose_backward_workspace_bytes()) summed in a fixed order.  Two launches. */
int mvip_rays_pack_backward(const float* rays_o, const float* rays_d, const float* view_d, int64_t n, int use_viewdirs, int ndc,
                            int H, int W, double focal, double ndc_near, const float* g_out, float* g_rays_o, float* g_rays_d,
                            float* g_view_d, void* stream);
size_t mvip_rays_from_pose_backward_workspace_bytes(void);
int mvip_rays_from_pose_backward(const float* c2w, const float* c2w_static, int H, int W, double focal, int i0, int j0, int h,
                                 int w, int use_viewdirs, int ndc, double ndc_near, const float* g_out, float* g_c2w,
                                 float* g_c2w_static, void* workspace, void* stream);

/* Rays of a table of V poses at given pixels: the ray batch of a training step that mixes pixels from many views
 * (DS_NeRF/run.py:889-908 draws them from all views; here the poses stay differentiable).
 *   poses   [V,3,4] row-major camera-to-world poses
 *   pixels  int32 [n,3] = (view, row, col)
 *   out     [n, 8 + 3*use_viewdirs]: row k is bitwise equal to row row*W + col of mvip_rays_from_pose_ndc(poses[view], NULL, ...)
 *           over the whole H x W image.  An entry whose view, row or column is out of range gives a row of NaN and reads
 *           no pose.  No static camera.  One launch, no host synchronisation.
 * Backward: g_out [n, 8 + 3*use_viewdirs] -> g_poses [V,3,4] (overwritten; views no entry uses get 0, out-of-range entries add
 *   nothing).  Each view's 12 sums are taken in a fixed order that depends only on `pixels` (no atomics): bitwise reproducible.
 *   workspace: mvip_rays_from_poses_backward_workspace_bytes(n, V) bytes.  Two launches. */
int mvip_rays_from_poses(const float* poses, int V, const int* pixels, int64_t n, int H, int W, double focal, float near, float far,
                         int use_viewdirs, int ndc, double ndc_near, float* out, void* stream);
size_t mvip_rays_from_poses_backward_workspace_bytes(int64_t n, int V);
int mvip_rays_from_poses_backward(const float* poses, int V, const int* pixels, int64_t n, int H, int W, double focal,
                                  int use_viewdirs, int ndc, double ndc_near, const float* g_out, float* g_poses, void* workspace,
                                  void* stream);

/* ------------------------------------------------------------------------------------------------
 * Stratified sampling along rays.            replaces DS_NeRF/run.py:1759-1781 (render_rays)
 *   rays    [n_rays, ray_stride] fp32: o(0:3) d(3:6) near(6) far(7) ...
 *   t_vals  [n_samples]  the torch.linspace(0,1,n_samples) table, computed by the host
 *   t_rand  [n_rays, n_samples] uniform randoms (perturb > 0) or NULL (perturb == 0)
 *   z_out   [n_rays, n_samples]
 * Bit-exact against the reference's CPU result (every op rounded to fp32, no FMA contraction).
 */
int mvip_sample_coarse(const float* rays, int ray_stride, int64_t n_rays, const float* t_vals,
                       const float* t_rand, int n_samples, int lindisp, float* z_out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Inverse-CDF sampling.                      replaces DS_NeRF/run_nerf_helpers.py:304-347 (sample_pdf)
 *   bins    [n_rows, n_bins], weights [n_rows, n_bins-1]
 *   u       [n_rows, n_out] or, if u_is_row, one row [n_out] shared by every ray (det=True linspace)
 *   samples [n_rows, n_out];  inds [n_rows, n_out] int64 = searchsorted(cdf, u, right=True) (nullable);
 *   cdf     [n_rows, n_bins] (nullable).
 * cdf / inds / samples are bit-exact against torch CPU for 8 <= n_bins-1 <= 512.
 */
int mvip_sample_pdf(const float* bins, const float* weights, const float* u, int u_is_row,
                    int64_t n_rows, int n_bins, int n_out, float* samples, int64_t* inds, float* cdf,
                    void* stream);

/* ------------------------------------------------------------------------------------------------
 * Hierarchical sampling step of render_rays. replaces DS_NeRF/run.py:1809-1816 and :1836
 *   z_mid = .5*(z[1:]+z[:-1]); z_samples = sample_pdf(z_mid, weights[1:-1], n_out, u);
 *   z_merged = sort(cat(z_vals, z_samples)); z_std = std(z_samples, unbiased=False)
 *   z_vals, weights [n_rays, n_samples]; outputs z_samples [n_rays,n_out] (nullable),
 *   inds int64 [n_rays,n_out] (nullable), z_merged [n_rays, n_samples+n_out], z_std [n_rays] (nullable).
 */
int mvip_sample_fine(const float* z_vals, const float* weights, const float* u, int u_is_row,
                     int64_t n_rays, int n_samples, int n_out, float* z_samples, int64_t* inds,
                     float* z_merged, float* z_std, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Alpha compositing.                         replaces DS_NeRF/run_nerf_helpers.py:350-404 (raw2outputs)
 *   raw [n_rays, n_samples, 4], z_vals [n_rays, n_samples], rays_d [n_rays, rays_d_stride] (first 3 used)
 *   noise [n_rays, n_samples] already multiplied by raw_noise_std, or NULL
 *   outputs: rgb [n,3], disp [n], acc [n], weights [n,S], depth [n], alpha [n,S] (nullable)
 */
int mvip_composite_forward(const float* raw, const float* z_vals, const float* rays_d,
                           int rays_d_stride, const float* noise, int64_t n_rays, int n_samples,
                           int white_bkgd, float* rgb, float* disp, float* acc, float* weights,
                           float* depth, float* alpha, void* stream);

/* Hand-written backward of the above (what autograd computes for the reference function):
 *   upstream g_rgb [n,3], g_disp [n], g_acc [n], g_depth [n] (each nullable = zeros),
 *   g_weights [n,S] (nullable), g_alpha [n,S] (nullable);  d_raw [n,S,4] is overwritten.
 *   No gradient is produced for z_vals / rays_d (they carry none in the reference: run.py:1812). */
int mvip_composite_backward(const float* raw, const float* z_vals, const float* rays_d,
                            int rays_d_stride, const float* noise, int64_t n_rays, int n_samples,
                            int white_bkgd, int detach_weights, const float* g_rgb,
                            const float* g_disp, const float* g_acc, const float* g_depth,
                            const float* g_weights, const float* g_alpha, float* d_raw, void* stream);

/* The same with the photometric losses fused in (img2mse of run_nerf_helpers.py:15 as train() applies it to rgb / rgb0 /
 * disp, run.py:1000-1027).  n_samples must be 64 or 128.
 *   forward : also returns sq_out[0] = sum_rays sum_c (rgb_map - target_rgb)^2 and sq_out[1] = sum_rays (disp_map - target_disp)^2
 *             (either target may be NULL -> 0); bitwise reproducible.  `workspace`: mvip_composite_mse_workspace_bytes()
 *             bytes, zero-filled before its FIRST use (the kernel leaves it ready for the next call).
 *   backward: g_sq[2] = d loss / d sq_out, read from DEVICE memory; 2 g_sq (map - target) is added to g_rgb / g_disp
 *             (which may be NULL) inside the kernel, from the recomputed forward. */
size_t mvip_composite_mse_workspace_bytes(void);
int mvip_composite_forward_mse(const float* raw, const float* z_vals, const float* rays_d, int rays_d_stride,
                               const float* noise, int64_t n_rays, int n_samples, int white_bkgd, const float* target_rgb,
                               const float* target_disp, float* rgb, float* disp, float* acc, float* weights, float* depth,
                               float* alpha, float* sq_out, void* workspace, void* stream);
int mvip_composite_backward_mse(const float* raw, const float* z_vals, const float* rays_d, int rays_d_stride,
                                const float* noise, int64_t n_rays, int n_samples, int white_bkgd, int detach_weights,
                                const float* target_rgb, const float* target_disp, const float* g_sq, const float* g_rgb,
                                const float* g_disp, const float* g_acc, const float* g_depth, const float* g_weights,
                                const float* g_alpha, float* d_raw, void* stream);

/* mvip_composite_backward[_mse] that also differentiates the ray directions: d_rays_d [n,3] (overwritten) =
 * d|rays_d| * rays_d / |rays_d|, d|rays_d| = sum_s dalpha_s relu(sigma_s) dist_s exp(-relu(sigma_s) dist_s |rays_d|) (last dist
 * 1e10, as in the reference).  target_rgb / target_disp / g_sq as in mvip_composite_backward_mse, or all NULL for the plain form.
 * d_raw is bitwise equal to that of the entry without d_rays_d. */
int mvip_composite_backward_rays(const float* raw, const float* z_vals, const float* rays_d, int rays_d_stride,
                                 const float* noise, int64_t n_rays, int n_samples, int white_bkgd, int detach_weights,
                                 const float* target_rgb, const float* target_disp, const float* g_sq, const float* g_rgb,
                                 const float* g_disp, const float* g_acc, const float* g_depth, const float* g_weights,
                                 const float* g_alpha, float* d_raw, float* d_rays_d, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Depth -> least-squares plane normal.       replaces DS_NeRF/run.py:1909-1940
 *   (depth2xyz_torch + depth2normal_geo, zero-padded k x k window, normal NOT normalised)
 *   depth [H,W] -> normal [3,H,W].  workspace: mvip_normal_workspace_bytes(H,W) bytes.
 */
size_t mvip_normal_workspace_bytes(int H, int W);
int mvip_normal_forward(const float* depth, int H, int W, float fx, float fy, float cx, float cy,
                        int k, float* normal, void* workspace, void* stream);
int mvip_normal_backward(const float* depth, int H, int W, float fx, float fy, float cx, float cy,
                         int k, const float* g_normal, float* d_depth, void* workspace, void* stream);

/* Same least-squares normal on an arbitrary point map xyz [3,H,W] (the argument depth2normal_geo takes in the
 * reference, run.py:1924); backward returns d_xyz [3,H,W]. */
int mvip_normal_forward_xyz(const float* xyz, int H, int W, int k, float* normal, void* workspace, void* stream);
int mvip_normal_backward_xyz(const float* xyz, int H, int W, int k, const float* g_normal, float* d_xyz,
                             void* workspace, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Stand-alone positional encoding.           replaces DS_NeRF/run_nerf_helpers.py:22-52 (Embedder.embed)
 *   in [n, >=dims] with row stride in_stride -> out [n, dims*(1+2*num_freqs)]:
 *   [x, sin(x*2^0), cos(x*2^0), ..., sin(x*2^(L-1)), cos(x*2^(L-1))]  (log-sampled bands, include_input)
 */
int mvip_embed(const float* in, int64_t in_stride, int64_t n, int dims, int num_freqs, float* out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * One-launch Adam step over a list of fp32 tensors.   replaces optimizer.step() of the training loop
 *   (DS_NeRF/run.py:1003; torch.optim.Adam built at run.py:1536-1537; the decayed learning rate of
 *   run.py:1031-1039 is passed as `lr`).  torch.optim.Adam semantics with weight_decay = 0, amsgrad = False.
 *   params / grads / exp_avg / exp_avg_sq: HOST arrays of n_tensors device pointers; sizes: host array of
 *   element counts; step: 1-based step number of this update (bias correction).
 */
int mvip_adam_step(float* const* params, const float* const* grads, float* const* exp_avg,
                   float* const* exp_avg_sq, const int64_t* sizes, int n_tensors, float lr, float beta1,
                   float beta2, float eps, int64_t step, void* stream);
/* Same update with the learning rate (1 float) and the 1-based step number (1 int64) read from DEVICE memory at execution
 * time: the form a CUDA graph of the training step captures (both change between replays). */
int mvip_adam_step_dev(float* const* params, const float* const* grads, float* const* exp_avg,
                       float* const* exp_avg_sq, const int64_t* sizes, int n_tensors, const float* lr_dev, float beta1,
                       float beta2, float eps, const int64_t* step_dev, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Fused positional encoding + 8x256 NeRF MLP (use_viewdirs, skip at 4).
 *   replaces DS_NeRF/run.py:1108-1124 (run_network), run_nerf_helpers.py:22-52 (Embedder.embed) and
 *   :104-127 (NeRF.forward); backward = autograd of the same.
 *
 * Parameters are passed as a host array of MVIP_MLP_NUM_PARAMS device pointers in this order
 * (nn.Module names of run_nerf_helpers.py:86-100, fp32, [out,in] row-major):
 *   0..15  pts_linears.{0..7}.{weight,bias}   16,17 views_linears.0.{weight,bias}
 *   18,19  feature_linear.{weight,bias}       20,21 alpha_linear.{weight,bias}
 *   22,23  rgb_linear.{weight,bias}
 * mvip_mlp_pack_weights converts them to the bf16, pre-swizzled, TMA-friendly blob the kernels
 * stream (re-run after every optimizer step).
 */
#define MVIP_MLP_NUM_PARAMS 24
size_t mvip_mlp_packed_bytes(void);
int mvip_mlp_pack_weights(const float* const* params /* host array */, void* packed, void* stream);

/* Points are described either by rays + depths (pts = o + d*z, viewdir = rays[:, viewdir_offset:+3];
 * n_points = n_rays*n_samples) or, when rays == NULL, directly by pts/dirs rows with strides
 * (e.g. columns 0:3 and 63:66 of an already-embedded [P,90] tensor). */
typedef struct mvip_points {
  const float* rays;   int ray_stride;  int viewdir_offset;
  const float* z_vals; int64_t n_rays;  int n_samples;
  const float* pts;    int64_t pts_stride;
  const float* dirs;   int64_t dirs_stride;
  int64_t n_points;
} mvip_points;

/* stash: activations kept for the backward pass (NULL for inference); mvip_mlp_stash_bytes(n_points) bytes */
size_t mvip_mlp_stash_bytes(int64_t n_points);
int mvip_mlp_forward(const void* packed, const mvip_points* pts, float* raw /* [n_points,4] */,
                     void* stash, void* stream);

/* workspace for the backward: mvip_mlp_backward_workspace_bytes(n_points) bytes.
 * grads: host array of MVIP_MLP_NUM_PARAMS device pointers (same order/shapes as params), fp32;
 * accumulate != 0 adds into them, otherwise they are overwritten. */
size_t mvip_mlp_backward_workspace_bytes(int64_t n_points);
int mvip_mlp_backward(const void* packed, const float* d_raw /* [n_points,4] */, int64_t n_points,
                      const void* stash, void* workspace, float* const* grads /* host array */,
                      int accumulate, void* stream);

/* The same call split into its launches (bit 0: backward_fused_kernel = dgrad chain + all tensor-core weight gradients;
 * bit 1: kept for ABI compatibility, launches nothing; bit 2: head grads; bit 3: reduce) so a caller can bracket each
 * kernel with its own events; phases must run in order on the same workspace. */
int mvip_mlp_backward_phases(const void* packed, const float* d_raw, int64_t n_points, const void* stash,
                             void* workspace, float* const* grads, int accumulate, int phase_mask, void* stream);

/* Gradient with respect to the MLP's inputs, from the dZ images a completed mvip_mlp_backward left in `bwd_workspace` (same
 * stream, same packed weights, same points).  Points mode: d_points [n_points,6] = (d pts | d dirs).  Rays mode: d_points is a
 * [n_points,6] scratch and d_rays [n_rays, ray_stride] (overwritten, every column) receives d o = sum_s d pts, d d = sum_s z_s d pts
 * in columns 0:6 and d viewdir in viewdir_offset:+3 (fixed-order sums: bitwise reproducible).  z_vals get no gradient. */
int mvip_mlp_input_grad(const void* packed, const mvip_points* pts, const void* bwd_workspace, float* d_points, float* d_rays,
                        void* stream);

/* ------------------------------------------------------------------------------------------------
 * Self tests of the tcgen05 building blocks (descriptor / layout conventions), used by tests/.
 *   which: 0 = K-major A,B (forward / dgrad form)   1 = MN-major A,B (wgrad form)
 *   a [M=128,K] , b [N,K] fp32 row-major for which==0;  a [K,128], b [K,N] for which==1
 *   out [128, N] fp32 = A * B^T (bf16 inputs, fp32 accumulate).  K multiple of 64, N in {64,128,256}.
 */
/* Debug aid: cycle counters recorded by CTA 0 of the last mvip_mlp_forward launch (host array of 16 u64;
 * synchronises the device). */
int mvip_debug_profile(unsigned long long* out16);
/* event trace of a -DMVIP_TRACE build: out[3][1024][2] (code, SM clock), n_out[3]; MVIP_E_UNSUPPORTED otherwise */
int mvip_debug_trace(long long* out, int* n_out);
/* wgrad cycle counters of CTA 0: producer empty-wait / total, issuer full-wait / total, bias warps full-wait / total, flag wait */
int mvip_debug_wgrad_profile(unsigned long long* out8);
/* event stamps (SM clock) of one chain-epilogue warp of the fused backward, -DMVIP_TRACE_BWD builds: out[20][12]; MVIP_E_UNSUPPORTED otherwise */
int mvip_debug_bwd_trace(long long* out240);
/* hand-over lag of the dZ units in the last fused backward: out[80 CTA pairs][4] = sum / max of (pick-up - publication) in ns, units
 * consumed, units already published when asked for; synchronises the device */
int mvip_debug_bwd_lag(unsigned long long* out320);
/* byte offsets, inside the backward workspace, of the per-(tile, dZ unit) publication and pick-up time stamps (u32 %globaltimer_lo) */
int mvip_debug_bwd_stamp_offsets(int64_t n_points, size_t* pub, size_t* pick);
/* tuning aid of the fused backward: a chain holds a tile back for at most `cycles` while more than `units` dZ units (64 KB) are
 * published but not picked up (cycles = 0: never); gain > 0: the delay is (excess units) x gain cycles instead */
int mvip_debug_set_bwd_throttle(int units, int cycles, int gain);
/* tuning aid of the fused backward: SM cycles between the chain starts of consecutive CTA pairs (< 0: default) */
int mvip_debug_set_bwd_stagger(int cycles);

int mvip_selftest_umma(int which, const float* a, const float* b, int N, int K, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MVIP_NERF_H_ */
