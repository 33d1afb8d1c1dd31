/* trb.h — C ABI of libtrb_b200.so: B200 (sm_100a) kernels for the iterative
 * registration hot path of AgamChopra/TorchRegister.
 *
 * The reference has no FFI of its own (pure Python over torch ops); the entry
 * points below are what a binding for this path replaces, cited as file:line
 * relative to /root/reference/src/TorchRegister/.  INTEGRATION.md shows the
 * ctypes stub a reference maintainer would add.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer marked "dev" is a CUDA
 *     device pointer owned by the caller (torch allocations in our host code);
 *     the library borrows them for the duration of the enqueued work and never
 *     frees or retains them;
 *   - `stream` is a cudaStream_t passed as void*; every call is asynchronous on
 *     that stream and performs no host synchronisation;
 *   - return value 0 = ok, otherwise a negative trb error or a positive
 *     cudaError_t; trb_last_error() gives a message (thread local);
 *   - volumes are fp32, contiguous, [D][H][W] (3-D) or [H][W] (2-D, pass D=1);
 *     a batch of independent pairs is addressed with `pair_stride` (elements);
 *   - theta is row-major ndim x (ndim+1), row r <-> sampling coordinate r
 *     (0 = x/W axis, 1 = y/H, 2 = z/D) exactly as F.affine_grid consumes it.
 */
#ifndef TRB_H
#define TRB_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TRB_ABI_VERSION 1

/* error codes (negative; positive values are cudaError_t) */
#define TRB_OK 0
#define TRB_ERR_ARG (-1)
#define TRB_ERR_WORKSPACE (-2)
#define TRB_ERR_UNSUPPORTED (-3)

/* modes / optimisers */
#define TRB_MODE_RIGID 0   /* params = Regressor.reg (6 | 3 floats), utils.py:313-330 */
#define TRB_MODE_AFFINE 1  /* params = theta itself (12 | 6 floats), warpings.py:42-55 */
#define TRB_OPT_SGD 0      /* torch.optim.SGD(lr), warpings.py:58,131,192 */
#define TRB_OPT_ADAM 1     /* extension (north_star item 3); no reference counterpart */
#define TRB_FLAG_LARGE_ROTATION 1   /* trb_affine_optim_ex / trb_warp_affine_batch: see there */
#define TRB_FLAG_PAIR_VOLUME 2      /* with TRB_FLAG_LARGE_ROTATION: a pair volume is attached to the workspace (trb_affine_attach_pairs) */
#define TRB_FLAG_QUAD_VOLUME 4      /* with TRB_FLAG_LARGE_ROTATION: a quad volume is attached instead (trb_affine_build_quads) */
#define TRB_FLAG_NEAREST 8          /* trb_warp_affine_batch / trb_warp_flow_ex: nearest-neighbour sampling (label maps) */

/* Per-pair optimiser state: TRB_STATE_FLOATS fp32 values, device resident.
 *   [ 0..11] params        (rigid: 6|3 used, affine: 12|6 used)
 *   [12..23] theta         theta the NEXT epoch samples with (after the last epoch:
 *                          the reference's final_theta, warpings.py:105-109,171)
 *   [24..35] best_theta    pre-step theta of the lowest-loss epoch (warpings.py:85-93,151-159)
 *   [36]     best_loss     [37] last_loss
 *   [40..51] adam m        [52..63] adam v
 */
#define TRB_STATE_FLOATS 64
#define TRB_STATE_PARAMS 0
#define TRB_STATE_THETA 12
#define TRB_STATE_BEST_THETA 24
#define TRB_STATE_BEST_LOSS 36
#define TRB_STATE_LAST_LOSS 37
#define TRB_STATE_ADAM_M 40
#define TRB_STATE_ADAM_V 52

/* Moments produced by one pass over the voxels of a pair (fp64):
 *   [0..4]   sum t, sum w, sum t^2, sum w^2, sum t*w
 *   [5..16]  sum J        J[r][c] = d warped / d theta[r][c]
 *   [17..28] sum t*J      [29..40] sum w*J
 */
#define TRB_MOMENTS 41

int trb_abi_version(void);
const char *trb_last_error(void);
/* number of SMs of the current device (grid sizing); <0 on error */
int trb_sm_count(void);

/* Kernel selection for the 3-D rigid/affine epoch: 0 = automatic (persistent multi-epoch TMA-staged kernel whenever
 * the shape/alignment allows, direct-gather kernel otherwise), 1 = always the direct-gather kernel, 2 = the
 * one-launch-per-epoch TMA kernel instead of the persistent one.  Process-wide; meant for tests and A/B timing. */
int trb_set_kernel_path(int path);
/* What the last trb_affine_optim* call of this thread did about the persistent kernel (launched, or why not): diagnostics. */
const char *trb_affine_kernel_status(void);

/* ---- rigid / affine registration ---------------------------------------- */

/* Bytes of scratch (dev) needed by trb_affine_* for `n_pairs` pairs. */
size_t trb_affine_workspace_bytes(int n_pairs);

/* Pair volume for the large-rotation (gather) variant of the 3-D loops: P[pair][z][y][xr] = (v[xr-2], v[xr-1]), W + 3 records of
 * two floats per row, zeros outside — one 8-byte gather per (y, z) corner instead of two 4-byte ones (the gathers of a rotated
 * warp are bound by cache lines touched).  trb_affine_build_pairs fills it from the moving volumes ([n_pairs][D][H][W]
 * contiguous); trb_affine_attach_pairs records its address in the workspace that the trb_affine_* calls of this batch use
 * (NULL detaches).  Optional: without it the gather variant reads the moving volumes themselves.  The buffer must stay alive
 * and unchanged while attached. */
size_t trb_affine_pairs_bytes(int n_pairs, int D, int H, int W);
int trb_affine_build_pairs(const float *moving_dev, float *pairs_dev, int n_pairs, int D, int H, int W, void *stream);
/* Quad volume: Q[pair][z][yr][xr] = (v[y][x], v[y][x+1], v[y+1][x], v[y+1][x+1]) at (x, y) = (xr-2, yr-2), (H+3) x (W+3) records of four
 * floats per slice, zeros outside — one 16-byte gather per z plane of a cell (2 per voxel).  4x the moving volumes in memory: worth
 * it while it stays L2 resident.  Attached with trb_affine_attach_pairs like the pair volume; flag TRB_FLAG_QUAD_VOLUME. */
size_t trb_affine_quads_bytes(int n_pairs, int D, int H, int W);
int trb_affine_build_quads(const float *moving_dev, float *quads_dev, int n_pairs, int D, int H, int W, void *stream);
int trb_affine_attach_pairs(void *workspace_dev, size_t workspace_bytes, int n_pairs, const float *pairs_dev, void *stream);

/* Write start parameters from HOST memory into state[.][0..n_params) of n_pairs pairs (n_rows == 1: the same row for
 * every pair, else n_rows == n_pairs).  The values travel as kernel arguments: asynchronous, stream ordered, no pinned
 * memory and no host wait behind the work already queued on the stream.  Call trb_affine_init_state afterwards. */
int trb_affine_set_params(float *state_dev, int n_pairs, int n_params, const float *params_host, int n_rows, void *stream);

/* Fill state[.][12..23] (theta) from state[.][0..11] (params) and reset
 * best/adam slots.  Replaces Regressor()/Theta.forward at loop entry
 * (utils.py:287-330) and the identity bias of warpings.py:47-48,54-55. */
int trb_affine_init_state(int ndim, int mode, float *state_dev, int n_pairs, void *stream);

/* Enqueue `n_epochs` fused registration epochs for `n_pairs` independent pairs.
 * One epoch = one kernel launch that, per pair: builds the sampling coordinates
 * from theta on the fly, tri/bi-linearly samples `moving`, streams `target`,
 * accumulates the loss moments and d(loss)/d(theta), and — in the last block to
 * finish — forms loss = w_mse*MSE + w_ncc*100*(1-NCC), chains to the rigid
 * parameters, applies the optimiser step, tracks the best theta and logs the loss.
 * Replaces the loop bodies warpings.py:67-93 (affine) and :138-159 (rigid):
 * F.affine_grid + F.grid_sample (:24-25), MSELoss / NCCLoss (utils.py:197-205),
 * backward (:80,146) and SGD.step (:81,147).
 *
 *   xb,yb,zb   dev tables of the base coordinates per axis, linspace(-1,1,S)*(S-1)/S
 *              (lengths W,H,D; zb ignored for ndim==2)
 *   loss_log   dev [n_pairs][log_stride]; epoch e writes column epoch0+e
 *   epoch0     index of the first epoch enqueued (0 starts best tracking)
 */
int trb_affine_optim(int ndim, int mode,
                     const float *moving_dev, const float *target_dev, long long pair_stride, int n_pairs,
                     int D, int H, int W,
                     const float *xb_dev, const float *yb_dev, const float *zb_dev,
                     float *state_dev, float *loss_log_dev, int log_stride,
                     int epoch0, int n_epochs,
                     float w_mse, float w_ncc, float lr,
                     int optimiser, float beta1, float beta2, float adam_eps,
                     void *workspace_dev, size_t workspace_bytes, void *stream);

/* trb_affine_optim with option flags.  TRB_FLAG_LARGE_ROTATION selects, for 3-D shapes the persistent kernel accepts,
 * its large-rotation variant: the moving volume is gathered through L1 by 8x4-voxel warp patches instead of being staged
 * box by box with TMA — the right choice when theta rotates by more than a few degrees (e.g. the reference's own
 * Regressor start, torch.rand(6) rad, utils.py:317), where the source footprint of an output tile no longer fits the
 * staged box.  Same results either way (same arithmetic per voxel). */
int trb_affine_optim_ex(int ndim, int mode,
                        const float *moving_dev, const float *target_dev, long long pair_stride, int n_pairs,
                        int D, int H, int W,
                        const float *xb_dev, const float *yb_dev, const float *zb_dev,
                        float *state_dev, float *loss_log_dev, int log_stride,
                        int epoch0, int n_epochs,
                        float w_mse, float w_ncc, float lr,
                        int optimiser, float beta1, float beta2, float adam_eps, int flags,
                        void *workspace_dev, size_t workspace_bytes, void *stream);

/* Host-side helper for choosing that flag: 1 if the source footprint of a 32x16x8 output tile under `theta_host`
 * (12 floats, HOST memory, row-major 3x4) fits the box the TMA-staged kernels fetch, else 0. */
int trb_affine_tile_fits(int D, int H, int W, const float *theta_host);

/* One volume sharded into z-slabs over up to 8 GPUs of one box, fused form (replaces the trb_affine_moments ->
 * all-reduce -> trb_affine_apply triple): n_epochs launches of the epoch kernel on slices [s_begin, s_end); the last
 * CTA of every rank pushes its 41 partial moments into every rank's mailbox with peer stores over NVLink, waits for
 * the others' (bounded spin: a missing peer yields NaN losses, not a hang), adds them in rank order and runs the
 * epilogue, so every rank applies the identical update.  mailbox_ptrs[r] = rank r's mailbox (2*8*48+8 doubles, zeroed
 * once) as mapped into THIS process (CUDA IPC / symmetric memory; peer access enabled).  Every rank must make the
 * same calls with the same seq0 (>= 1, advance it by n_epochs per call).  3-D, shapes the TMA kernel accepts. */
int trb_affine_optim_peer(const float *moving_dev, const float *target_dev, int D, int H, int W, int s_begin, int s_end,
                          const float *xb_dev, const float *yb_dev, const float *zb_dev, int mode,
                          float *state_dev, float *loss_log_dev, int log_stride, int epoch0, int n_epochs,
                          float w_mse, float w_ncc, float lr, int optimiser, float beta1, float beta2, float adam_eps,
                          void *const *mailbox_ptrs, int rank, int world, unsigned long long seq0,
                          void *workspace_dev, size_t workspace_bytes, void *stream);

/* Sharded variant for one large volume split into z-slabs (2-D: y-slabs) across
 * GPUs: accumulate the TRB_MOMENTS fp64 moments of output slices [s_begin,s_end)
 * into moments_dev[n_pairs][TRB_MOMENTS] (overwritten), no update.  After the
 * caller has all-reduced the moments, trb_affine_apply performs the update that
 * trb_affine_optim fuses.  `n_total` = voxels of the WHOLE volume. */
int trb_affine_moments(int ndim,
                       const float *moving_dev, const float *target_dev, long long pair_stride, int n_pairs,
                       int D, int H, int W, int s_begin, int s_end,
                       const float *xb_dev, const float *yb_dev, const float *zb_dev,
                       const float *state_dev, double *moments_dev,
                       void *workspace_dev, size_t workspace_bytes, void *stream);

/* The same with option flags (TRB_FLAG_LARGE_ROTATION: gather variant, see trb_affine_optim_ex). */
int trb_affine_moments_ex(int ndim,
                          const float *moving_dev, const float *target_dev, long long pair_stride, int n_pairs,
                          int D, int H, int W, int s_begin, int s_end,
                          const float *xb_dev, const float *yb_dev, const float *zb_dev,
                          const float *state_dev, double *moments_dev, int flags,
                          void *workspace_dev, size_t workspace_bytes, void *stream);

/* extra_dev (optional, may be NULL): [n_pairs][13] fp64 = an additional loss term and its gradient w.r.t.
 * theta, evaluated outside (used for the NMI/KDE term, reference utils.py:224-259, until it is fused). */
int trb_affine_apply(int ndim, int mode, const double *moments_dev, int n_pairs,
                     int D, int H, int W,
                     float *state_dev, float *loss_log_dev, int log_stride, int epoch,
                     float w_mse, float w_ncc, float lr,
                     int optimiser, float beta1, float beta2, float adam_eps,
                     const double *extra_dev, void *stream);

/* Forward warp only: out[c] = grid_sample(moving[c], affine_grid(theta)) for
 * n_channels volumes sharing one theta (dev, 12|6 floats).
 * Replaces get_affine_warp (warpings.py:18-26) as used by Register.__call__
 * (torchregister.py:126-128). */
int trb_warp_affine(int ndim, const float *moving_dev, float *out_dev, int n_channels,
                    int D, int H, int W, const float *theta_dev,
                    const float *xb_dev, const float *yb_dev, const float *zb_dev, void *stream);

/* The same for a batch: n_pairs pairs of n_channels volumes each ([n_pairs][n_channels][D][H][W] contiguous), theta_dev
 * [n_pairs][12|6], ONE launch.  3-D shapes with W % 4 == 0, W >= 32, H >= 16 take the TMA-staged kernel (csrc/warp_tma.cu);
 * flags: TRB_FLAG_LARGE_ROTATION = theta is known to rotate by more than a few degrees (gather kernel instead);
 * TRB_FLAG_NEAREST = grid_sample(mode='nearest'): the source coordinate rounded half to even, zero outside the volume,
 * so only input values and 0 appear in out (label maps).  Same path selection with or without it.  The nearest kernels
 * need every spatial axis <= 2^22 = 4194304 voxels (TRB_ERR_UNSUPPORTED otherwise); the bilinear ones do not. */
int trb_warp_affine_batch(int ndim, const float *moving_dev, float *out_dev, int n_pairs, int n_channels,
                          int D, int H, int W, const float *theta_dev,
                          const float *xb_dev, const float *yb_dev, const float *zb_dev, int flags, void *stream);

/* Vector-Jacobian product of the affine warp with respect to theta:
 * dtheta[12|6] (fp64, dev) = sum_v gout_v * d warped_v / d theta.
 * (autograd of warpings.py:24-25 for callers that differentiate get_affine_warp.) */
int trb_warp_affine_vjp(int ndim, const float *moving_dev, const float *gout_dev,
                        int D, int H, int W, const float *theta_dev,
                        const float *xb_dev, const float *yb_dev, const float *zb_dev,
                        double *dtheta_dev, void *workspace_dev, size_t workspace_bytes, void *stream);

int trb_warp_affine_vjp_ex(int ndim, const float *moving_dev, const float *gout_dev,
                           int D, int H, int W, const float *theta_dev,
                           const float *xb_dev, const float *yb_dev, const float *zb_dev,
                           double *dtheta_dev, int flags, void *workspace_dev, size_t workspace_bytes, void *stream);

/* ---- flow field ----------------------------------------------------------- */
/* flow layout [ndim][D][H][W] fp32 in voxel units, channel i displaces spatial
 * axis i (0 = D (3-D) or H (2-D)), the SpatialTransformer convention utils.py:350-365.
 * The calls below that sample a volume (every one but trb_flow_jacobian) need every spatial axis >= 2,
 * D*H*W < 2^31 (TRB_ERR_ARG otherwise) and every axis <= 2^22 = 4194304 voxels: their kernels take floor and rint with
 * a 1.5*2^23 add, which indexes exactly only up to there (TRB_ERR_UNSUPPORTED otherwise). */

size_t trb_flow_workspace_bytes(void);

/* warped[c] = SpatialTransformer(src[c], flow); replaces utils.py:350-365 as used by
 * flow_register.deform (warpings.py:238-242) and Register.__call__ (torchregister.py:124-125). */
int trb_warp_flow(int ndim, const float *src_dev, const float *flow_dev, float *out_dev, int n_channels,
                  int D, int H, int W, void *stream);

/* The same with option flags: TRB_FLAG_NEAREST = grid_sample(mode='nearest', align_corners=True) on the reference's
 * grid, bit for bit (label maps); 0 = trb_warp_flow. */
int trb_warp_flow_ex(int ndim, const float *src_dev, const float *flow_dev, float *out_dev, int n_channels,
                     int D, int H, int W, int flags, void *stream);

/* Jacobian determinant of phi(p) = p + u(p), u = flow_dev in voxel units (the layout above).  J_ij = delta_ij + du_i/dp_j
 * with numpy.gradient's differences (central inside, one-sided at both ends; every spatial axis >= 2, else TRB_ERR_ARG),
 * formed in fp64 with the 3x3 (2x2) determinant.  det_out_dev (nullable): the field as fp32 [D][H][W].
 * stats_out_dev (dev, TRB_JAC_NSTATS doubles): n det <= 0, n non-finite det, min det, max det, sum det, sum det^2,
 * sum L, sum L^2 with L = log(clamp(det, 1e-9, 1e9)); all but the non-finite count are over finite det only.  Sums in a
 * fixed order: the same bits on every run.  workspace: trb_flow_workspace_bytes() (its ticket must be zero, as for the
 * flow calls; the call leaves it so). */
#define TRB_JAC_NSTATS 8
int trb_flow_jacobian(int ndim, const float *flow_dev, int D, int H, int W, float *det_out_dev, double *stats_out_dev,
                      void *workspace_dev, size_t workspace_bytes, void *stream);

/* Transform algebra (csrc/transform.cu).  A flow u stands for phi_u(p) = p + u(p); trb_warp_flow samples at phi_u(p).
 * trb_warp_affine samples at T(q) = M q + c, theta's map in voxel units (affine_grid(align_corners=False) un-normalised by
 * grid_sample): with S_r the size along sampling coordinate r (0 = x/W, 1 = y/H, 2 = z/D),
 *   M_rc = theta_rc S_r / S_c,   c_r = S_r/2 (theta_r,ndim + 1 - sum_c theta_rc (1 - 1/S_c)) - 1/2.
 * The composed field w of "first, then second" satisfies warp_flow(m, w) = warp_flow(warp(m, first), second) up to the
 * interpolation of the intermediate volume that it avoids.  first~ is the (bi|tri)linear interpolant of a flow with border
 * padding: each coordinate clamped to [0, S-1] (grid_sample(padding_mode='border', align_corners=True) on voxel positions).
 * N == 1, no gradients; the shape rules of the flow calls above (TRB_ERR_ARG, TRB_ERR_UNSUPPORTED).  An output that
 * overlaps an input is refused (TRB_ERR_ARG).  A non-finite sample position p + u(p) gives NaN in every channel of its
 * voxel; a NaN among the corners of a cell that is read propagates to that channel. */

/* w = T_theta(p + u(p)) - p, evaluated as u + (M - I) q + c with q = p + u (fp32 per voxel; M - I and c formed in fp64 from
 * theta_dev, ndim*(ndim+1) floats in device memory, read by the kernel: no host synchronisation).  Exact: T is affine.
 * flow_dev NULL: u = 0 (the affine's own displacement, T(p) - p).  out_dev: [ndim][D][H][W]. */
int trb_compose_affine_flow(int ndim, const float *theta_dev, const float *flow_dev, int D, int H, int W,
                            float *out_dev, void *stream);
/* w = u(p) + first~(p + u(p)), u = second_dev; all three [ndim][D][H][W]. */
int trb_compose_flows(int ndim, const float *first_dev, const float *second_dev, int D, int H, int W,
                      float *out_dev, void *stream);
/* Inverse: v = the fixed point of v(p) = -u~(p + v(p)), so that phi_u(phi_v(p)) = p, iterated per voxel: v_0 = -u(p);
 * iteration k evaluates r_k = |v_k + u~(p + v_k)|_inf and stops when r_k <= tol or k = max_iter - 1, else
 * v_{k+1} = -u~(p + v_k).  The v_k whose residual was evaluated is written to inv_out_dev, so each voxel's residual is the
 * one counted below.  The iteration converges where u~ is a contraction (Lipschitz constant < 1 in the inf-norm: a mild,
 * fold-free flow); the call does not require it and reports what did not converge.  A voxel that meets a non-finite
 * position or residual stops there with NaN in every channel.  max_iter in [1, 1000], tol (voxels) finite and > 0
 * (TRB_ERR_ARG otherwise).  stats_out_dev (dev, TRB_INV_NSTATS doubles): n not converged (finite, r > tol), n non-finite,
 * max r over the finite voxels (0 if none), sum over all voxels of the residual evaluations made (iterations started).
 * Counts and sums in a fixed order: the same bits on every run.  workspace: trb_flow_workspace_bytes() (its ticket must
 * be zero, as for the flow calls; the call leaves it so). */
#define TRB_INV_NSTATS 4
int trb_invert_flow(int ndim, const float *flow_dev, int D, int H, int W, int max_iter, float tol,
                    float *inv_out_dev, double *stats_out_dev, void *workspace_dev, size_t workspace_bytes, void *stream);

/* dflow = J^T gout for the warp above (autograd of utils.py:365 w.r.t. flow);
 * used when the caller supplies its own criterion (torchregister.py:71-73). */
int trb_warp_flow_vjp(int ndim, const float *src_dev, const float *flow_dev, const float *gout_dev,
                      float *dflow_dev, int D, int H, int W, void *stream);

/* Fused warp + similarity + gradient: loss = w_mse*MSE + w_ncc*100*(1-NCC) of
 * (target, warp(moving, flow)) and dflow = d loss / d flow; optionally also the
 * warped volume.  Replaces utils.py:350-365 + warpings.py:213-215 (forward of the
 * similarity and the backward down to the flow).  loss_dev: 1 float. */
int trb_flow_loss_grad(int ndim, const float *moving_dev, const float *target_dev, const float *flow_dev,
                       int D, int H, int W, float w_mse, float w_ncc,
                       float *loss_dev, float *dflow_dev, float *warped_dev_or_null,
                       void *workspace_dev, size_t workspace_bytes, void *stream);

/* U-Net head fused with the node (SURVEY.md 8 f-3): replaces  y = padNd(y, x); flow = out(y); warp; similarity  of
 * Attention_UNet.forward / flow_register.optimize (utils.py:553-557, warpings.py:211-215) and their backward.
 * feat_dev: the decoder output [C][fd][fh][fw] (C <= 8, un-padded); w_dev [ndim][C], b_dev [ndim]: the 1x1 `out`
 * convolution (device memory: the module's parameters as they are).  forward: writes flow_out_dev [ndim][D][H][W] (= Register.theta) and *loss_dev, leaves the loss
 * coefficients in the workspace; backward (same workspace, after forward): dfeat_dev [C][fd][fh][fw] = d loss / d feat,
 * dwb_dev[ndim*C + ndim] = d loss / d W, d loss / d b.  d loss / d flow is never written.  Both calls refuse C > 8
 * (TRB_ERR_UNSUPPORTED) and a feature map larger than the volume on some axis (TRB_ERR_ARG). */
int trb_flow_head_forward(int ndim, const float *moving_dev, const float *target_dev, const float *feat_dev, int C,
                          int fd, int fh, int fw, const float *w_dev, const float *b_dev, int D, int H, int W,
                          float w_mse, float w_ncc, float *loss_dev, float *flow_out_dev,
                          void *workspace_dev, size_t workspace_bytes, void *stream);
int trb_flow_head_backward(int ndim, const float *moving_dev, const float *target_dev, const float *flow_dev,
                           const float *feat_dev, int C, int fd, int fh, int fw, const float *w_dev, int D, int H, int W,
                           float *dfeat_dev, float *dwb_dev, void *workspace_dev, size_t workspace_bytes, void *stream);

/* ---- EXTENSION: direct per-voxel flow optimisation (north_star items 2b/3) ---------------------
 * No counterpart in the reference (it optimises U-Net weights, warpings.py:178-233, and has no smoothness
 * term).  One epoch = trb_flow_direct_stats -> [all-reduce of the 6 moments when sharded] ->
 * trb_flow_direct_update.  loss = w_mse*MSE + w_ncc*100*(1-NCC) + lambda * smooth,
 * smooth = mean over axes of mean((forward difference of every flow channel)^2).
 * Slab form (one volume sharded over GPUs by z): target/flow/adam arrays hold slices [z_off, z_off+Ds),
 * `moving` is the whole volume, halo_lo/halo_hi are the neighbouring ranks' flow slices z_off-1 and
 * z_off+Ds ([ndim][H][W]; NULL at the volume boundary).  A single GPU passes z_off=0, Ds=D, no halos.
 * Every spatial axis must be <= 2^22 = 4194304 voxels, as for the flow calls above (TRB_ERR_UNSUPPORTED otherwise).
 * moments6: sum t, sum w, sum t^2, sum w^2, sum t*w, smooth (fp64, overwritten by stats). */
size_t trb_flow_direct_workspace_bytes(void);

int trb_flow_direct_stats(int ndim, const float *moving_dev, const float *target_slab_dev, const float *flow_slab_dev,
                          const float *halo_lo_dev, const float *halo_hi_dev, int D, int H, int W, int z_off, int Ds,
                          float smooth_lambda, double *moments6_dev, void *workspace_dev, size_t workspace_bytes,
                          void *stream);

/* flow_out = optimiser(flow_in, d loss / d flow); out of place (the smoothness stencil reads neighbours).
 * optimiser TRB_OPT_SGD or TRB_OPT_ADAM (torch.optim.Adam semantics; adam_m/v slab-shaped, step_index 1-based).
 * loss_log_dev[epoch] receives the loss of flow_in (may be NULL). */
int trb_flow_direct_update(int ndim, const float *moving_dev, const float *target_slab_dev,
                           const float *flow_in_slab_dev, float *flow_out_slab_dev,
                           const float *halo_lo_dev, const float *halo_hi_dev, int D, int H, int W, int z_off, int Ds,
                           const double *moments6_dev, float w_mse, float w_ncc, float smooth_lambda, float lr,
                           int optimiser, float beta1, float beta2, float adam_eps, int step_index,
                           float *adam_m_dev, float *adam_v_dev, float *loss_log_dev, int epoch, void *stream);

/* Fused 3-D epoch: ONE streaming pass per epoch (32 B/voxel SGD, 80 B/voxel Adam) instead of stats + update.
 * Needs 3*Ds*H*W < 2^31.  moments6_dev is read and then overwritten:
 *   in : [0..4] similarity sums of flow_in over the WHOLE volume (only used when w_ncc != 0: run
 *        trb_flow_direct_stats with lambda 0 once before the first epoch, all-reduced when sharded);
 *   out: [0..4] this slab's similarity sums of flow_out (w_ncc != 0) or of flow_in (w_ncc == 0), [5] this slab's
 *        smoothness sum of flow_in.  Sharded callers all-reduce the 6 values between epochs.
 * loss_log_dev[epoch-1] is completed by the call for `epoch` when complete_prev != 0 (= the previous call was a
 * fused step with the same weights and no trb_flow_direct_finish in between), the last one by
 * trb_flow_direct_finish (epochs_done = number of epochs done).  workspace as trb_flow_direct_workspace_bytes(), the same one for every call. */
int trb_flow_direct_step(const float *moving_dev, const float *target_slab_dev,
                         const float *flow_in_slab_dev, float *flow_out_slab_dev,
                         const float *halo_lo_dev, const float *halo_hi_dev, int D, int H, int W, int z_off, int Ds,
                         double *moments6_dev, float w_mse, float w_ncc, float smooth_lambda, float lr,
                         int optimiser, float beta1, float beta2, float adam_eps, int step_index,
                         float *adam_m_dev, float *adam_v_dev, float *loss_log_dev, int epoch, int complete_prev,
                         void *workspace_dev, size_t workspace_bytes, void *stream);

/* trb_flow_direct_step for ONE volume sharded into z-slabs over up to 8 GPUs of one box, with no NCCL call in the epoch:
 * halo_lo/halo_hi point INTO the neighbour ranks' flow buffers (their last / first slice, mapped into this process;
 * channel stride = the neighbour's Ds*H*W elements), and the last CTA all-reduces the 6 sums through the peer mailboxes
 * of trb_affine_optim_peer, so moments6_dev holds the GLOBAL sums when the kernel ends.  That exchange also orders the
 * epochs: a rank's flow buffer is only read by its neighbours after it is complete and only overwritten after they have
 * read it (ping-pong buffers, every rank in the same phase).  seq >= 1, +1 per call, identical on every rank. */
int trb_flow_direct_step_peer(const float *moving_dev, const float *target_slab_dev,
                              const float *flow_in_slab_dev, float *flow_out_slab_dev,
                              const float *halo_lo_dev, long long halo_lo_channel_stride,
                              const float *halo_hi_dev, long long halo_hi_channel_stride,
                              int D, int H, int W, int z_off, int Ds,
                              double *moments6_dev, float w_mse, float w_ncc, float smooth_lambda, float lr,
                              int optimiser, float beta1, float beta2, float adam_eps, int step_index,
                              float *adam_m_dev, float *adam_v_dev, float *loss_log_dev, int epoch, int complete_prev,
                              void *const *mailbox_ptrs, int rank, int world, unsigned long long seq,
                              void *workspace_dev, size_t workspace_bytes, void *stream);

/* A/B switch for the smoothness variants of trb_flow_direct_step: 0 (default) = TMA-staged tiles, 1 = register-staged. */
void trb_flow_direct_set_path(int no_tma);

int trb_flow_direct_finish(const double *moments6_dev, int D, int H, int W, float w_mse, float w_ncc,
                           float smooth_lambda, float *loss_log_dev, int epochs_done,
                           void *workspace_dev, size_t workspace_bytes, void *stream);

/* The update pass of the direct-flow epoch driven by local NCC (single GPU, whole volume): one epoch is
 * trb_flow_direct_stats -> trb_warp_flow (J) -> trb_lncc_forward -> trb_lncc_backward (resid = dL/dJ, its pointwise
 * MSE / NCC terms from moments6) -> this call.  It recomputes the sample gradient G at flow_in and applies
 * resid * G + lambda * (smoothness stencil) with SGD or Adam, as trb_flow_direct_update; flow_out must not overlap
 * flow_in or resid (TRB_ERR_ARG).  loss_log_dev[epoch] (nullable) receives the loss of flow_in:
 * w_mse*MSE + w_ncc*100*(1-NCC) (from moments6_dev) + w_lncc * lncc_stats_dev[1] + lambda * moments6_dev[5].
 * Shape rules of trb_flow_direct_update with z_off = 0, Ds = D. */
int trb_flow_direct_update_lncc(int ndim, const float *moving_dev, const float *flow_in_dev, float *flow_out_dev,
                                const float *resid_dev, int D, int H, int W, const double *moments6_dev,
                                const double *lncc_stats_dev, float w_mse, float w_ncc, float w_lncc,
                                float smooth_lambda, float lr, int optimiser, float beta1, float beta2,
                                float adam_eps, int step_index, float *adam_m_dev, float *adam_v_dev,
                                float *loss_log_dev, int epoch, void *stream);

/* ---- local normalised cross-correlation (csrc/lncc.cu) ------------------------------------------------------
 * VoxelMorph's windowed NCC with the sign turned so that the loss is >= 0.  target I and warped J: fp32
 * [N][D][H][W] (2-D: D ignored), N pairs that never share a window; win odd in [3, 15] (TRB_ERR_UNSUPPORTED
 * otherwise); n = win^ndim; S_X the box sum of X over the window with zero padding (out-of-volume positions count
 * as zeros, n stays fixed):
 *   A = S_IJ - S_I S_J / n,  B = S_II - S_I^2 / n,  C = S_JJ - S_J^2 / n,  cc = A^2 / (B C + eps),
 *   loss = 1 - (sum of cc over every voxel of every pair) / (N D H W).
 * Shape rules: every axis >= 1, D*H*W < 2^31 (TRB_ERR_ARG) and every axis <= 2^22 (TRB_ERR_UNSUPPORTED).  An
 * output that overlaps an input is refused (TRB_ERR_ARG).  Every sum is formed in a fixed order: the same bits on
 * every run. */
size_t trb_lncc_workspace_bytes(void);

/* coef_dev: 3 N D H W floats, written as alpha, beta, gamma planes ([3][N][D][H][W]) with den = B C + eps,
 * gamma = 2 A / den, beta = -A^2 B / den^2, alpha = -gamma S_I / n - 2 beta S_J / n (the derivatives of cc w.r.t.
 * S_J, S_JJ, S_IJ).  stats_dev (dev, 2 doubles): sum of cc, loss.  eps finite and > 0.  workspace:
 * trb_lncc_workspace_bytes() (its ticket must be zero, e.g. a zeroed buffer; the call leaves it so). */
int trb_lncc_forward(int ndim, const float *target_dev, const float *warped_dev, int N, int D, int H, int W, int win,
                     float eps, float *coef_dev, double *stats_dev, void *workspace_dev, size_t workspace_bytes,
                     void *stream);

/* grad_dev (N D H W floats) = scale * dloss/dJ = -(scale / (N D H W)) (box(alpha) + 2 J box(beta) + I box(gamma)),
 * from the coef_dev of trb_lncc_forward on the same I, J and win.  With moments6_dev (N == 1 only; the layout of
 * trb_flow_direct_stats), it adds the pointwise gradient of w_mse*MSE + w_ncc*100*(1-NCC): cw J + ct I + c0. */
int trb_lncc_backward(int ndim, const float *target_dev, const float *warped_dev, const float *coef_dev, int N, int D,
                      int H, int W, int win, float scale, const double *moments6_dev, float w_mse, float w_ncc,
                      float *grad_dev, void *stream);

/* ---- Edge3D pre-filter (SURVEY.md 8 f-4) --------------------------------------------------------------
 * Replaces utils.py:130-183 (Edge3D.__call__ with a pad that works): reflect padding, the nine 3x3x3 Sobel-type
 * cross-correlations of get_sobel_kernel3D (utils.py:82-127; passed as weights_host[9][27], HOST memory, (x,y,z) order),
 * gradient magnitude (1/C) sqrt(sum_s (sum_c (corr_s + eps))^2 + eps), min-max normalisation over the whole batch
 * (utils.py:262-267) and the band threshold lo < e < hi -> {0,1}.  out_dev [B][X][Y][Z] fp32; minmax_dev: 2 x u32 scratch;
 * norm_out_dev (optional): the normalised magnitude before thresholding. */
int trb_edge3d(const float *img_dev, float *out_dev, int B, int C, int X, int Y, int Z, const float *weights_host,
               float thresh_lo, float thresh_hi, unsigned *minmax_dev, float *norm_out_dev, void *stream);

/* ---- NMI/KDE term of the reference's default loss (SURVEY.md 8 f-1) -----------------------------------
 * Replaces utils.py:18-79 (K_gauss, PDF_xis, get_pdf, NMI) + utils.py:224-259 (NMILoss.forward with its default
 * bins=256, patch_size=100) and autograd's backward down to the warped volume, for ONE pair [1,1,(D,)H,W]:
 * nearest resample to 200^n, 2^n chunks of 100^n values, 256-bin Gaussian KDE (bandwidth h) of target, warped
 * and their concatenation over swapped/detached ranges, loss = alpha * mean_k |NMI_k - 1|.
 * trb_nmi_prepare: once per target (resample + the target's own marginal, cached in the workspace).
 * trb_nmi_loss_grad: per epoch; *loss_dev = weight*loss (fp64), gout_dev[D][H][W] = weight * d loss / d warped
 * (NULL: forward only).  Chain gout to theta with trb_warp_affine_vjp or to a flow with trb_warp_flow_vjp. */
size_t trb_nmi_workspace_bytes(int ndim, int D, int H, int W);
int trb_nmi_prepare(int ndim, const float *target_dev, int D, int H, int W, float bandwidth,
                    void *workspace_dev, size_t workspace_bytes, void *stream);
int trb_nmi_loss_grad(int ndim, const float *warped_dev, int D, int H, int W, float bandwidth, float alpha,
                      float weight, double *loss_dev, float *gout_dev, void *workspace_dev,
                      size_t workspace_bytes, void *stream);

/* Same term in SOURCE-voxel space (2-D and 3-D, batched over pairs; csrc/nmi_src.cu): no resampled arrays, one pass over the warped
 * volumes for 12 Hermite moments per chunk about a fixed centre, one pass writing d term / d warped.  Valid when all values
 * of target and warped volumes lie in [lo, hi] with hi - lo <= 0.6 * bandwidth (TRB_ERR_UNSUPPORTED otherwise; the loss is
 * NaN if a value leaves the bounds).  volumes: [n_pairs] x D*H*W, pair_stride floats apart.
 * trb_nmi_src_prepare: once per batch of targets.  trb_nmi_src_loss_grad: loss_dev[pair*loss_stride] = weight*loss (fp64),
 * gout_dev (same layout as warped_dev; NULL: forward only) = weight * d loss / d warped. */
size_t trb_nmi_src_workspace_bytes(int ndim, int n_pairs, int D, int H, int W);
int trb_nmi_src_prepare(int ndim, const float *target_dev, long long pair_stride, int n_pairs, int D, int H, int W,
                        float bandwidth, float lo, float hi, void *workspace_dev, size_t workspace_bytes, void *stream);
int trb_nmi_src_loss_grad(int ndim, const float *warped_dev, long long pair_stride, int n_pairs, int D, int H, int W,
                          float bandwidth, float alpha, float weight, float lo, float hi, double *loss_dev, int loss_stride,
                          float *gout_dev, void *workspace_dev, size_t workspace_bytes, void *stream);

/* The rigid / affine loop with the reference's DEFAULT criterions [MSE, NCC, NMI] (warpings.py:36-40,60-93,123-159),
 * n_epochs epochs enqueued by one call (no host work per epoch): MSE/NCC moments -> warp with the current theta -> NMI
 * term (source-space form above; trb_nmi_src_prepare must have run on nmi_workspace_dev with these targets and bounds)
 * -> its d/dtheta by a second moments pass -> fused update and bookkeeping as trb_affine_apply.  moving/target:
 * [n_pairs][(D)][H][W] contiguous (ndim == 2: D is ignored); warped_scratch_dev / gout_scratch_dev: same size; workspace_dev as trb_affine_moments. */
int trb_affine_optim_nmi(int ndim, int mode, const float *moving_dev, const float *target_dev, int n_pairs, int D, int H, int W,
                         const float *xb_dev, const float *yb_dev, const float *zb_dev, float *state_dev,
                         float *loss_log_dev, int log_stride, int epoch0, int n_epochs, float w_mse, float w_ncc,
                         float w_nmi, float lr, int optimiser, float beta1, float beta2, float adam_eps, int flags,
                         float bandwidth, float alpha, float lo, float hi, float *warped_scratch_dev,
                         float *gout_scratch_dev, void *nmi_workspace_dev, size_t nmi_workspace_bytes,
                         void *workspace_dev, size_t workspace_bytes, void *stream);

/* ---- InstanceNorm of the flow U-Net (SURVEY.md 8 f-3; csrc/instnorm.cu) --------------------------------
 * Replaces nn.InstanceNorm3d / nn.InstanceNorm2d (affine=False, no running statistics) of Attention_UNet
 * (utils.py:368-520) and autograd's backward, optionally fused with the ReLU in front of it (relu != 0:
 * y = IN(max(x, 0))).  x, y, dy, dx: [n_inst][S] contiguous (n_inst = N*C instances of S spatial elements);
 * stats_dev [n_inst][2] = (mean, rstd) written by forward and read by backward; coef_dev [n_inst][2] scratch. */
size_t trb_instnorm_workspace_bytes(int n_inst, long long S);
/* gate_dev (optional, [S], shared by the instances = channels of ONE sample, no ReLU): y_c = IN(x_c * gate) — the attention gate's
 * `bnorm(x * w)` (utils.py:403-405) without the product tensor; backward then also returns dgate_dev [S] = sum_c dv_c x_c. */
int trb_instnorm_forward(const float *x_dev, const float *gate_dev, float *y_dev, int n_inst, long long S, float eps, int relu,
                         float *stats_dev, void *workspace_dev, size_t workspace_bytes, void *stream);
int trb_instnorm_backward(const float *x_dev, const float *gate_dev, const float *dy_dev, float *dx_dev, float *dgate_dev,
                          int n_inst, long long S, int relu, const float *stats_dev, float *coef_dev, void *workspace_dev,
                          size_t workspace_bytes, void *stream);

/* ---- thin 3x3x3 convolutions of the flow U-Net (SURVEY.md 8 f-3; csrc/thinconv.cu) -----------------------
 * Replaces nn.Conv3d(kernel_size=3) (stride 1, no padding; any C_in, C_out <= 4 and the pairs 8->4, 4->8, 8->8: the two finest
 * levels of Attention_UNet at the reference's n = 32, utils.py:409-520) and autograd's backward.  x [n][CI][D][H][W] -> y [n][CO][D-2][H-2][W-2];
 * w [CO][CI][3][3][3], b [CO] or NULL, all device fp32.  backward: gx_dev and/or gw_dev (+ gb_dev) may be NULL to skip
 * that gradient; the weight gradient handles one sample per call.  Weights travel through constant memory on `stream`:
 * calls on different streams of one device must not overlap. */
size_t trb_thinconv3_workspace_bytes(int CI, int CO);
int trb_thinconv3_forward(const float *x_dev, const float *w_dev, const float *b_dev, float *y_dev, int n_batch, int CI,
                          int CO, int D, int H, int W, void *stream);
int trb_thinconv3_backward(const float *x_dev, const float *w_dev, const float *gy_dev, float *gx_dev, float *gw_dev,
                           float *gb_dev, int n_batch, int CI, int CO, int D, int H, int W, void *workspace_dev,
                           size_t workspace_bytes, void *stream);

/* 1x1x1 convolutions with <= 4 channels each way (attention gates, utils.py:368-406): y[co][o] = b[co] + sum_ci w[co][ci] x[ci][o*stride];
 * x [CI][D][H][W] (2-D: D = 1), y [CO][OD][OH][OW] with O* = (I* - 1) / stride + 1; one sample per call; NULL gradients are skipped. */
size_t trb_pointconv_workspace_bytes(int CI, int CO);
int trb_pointconv_forward(const float *x_dev, const float *w_dev, const float *b_dev, float *y_dev, int CI, int CO, int D,
                          int H, int W, int stride, void *stream);
int trb_pointconv_backward(const float *x_dev, const float *w_dev, const float *gy_dev, float *gx_dev, float *gw_dev,
                           float *gb_dev, int CI, int CO, int D, int H, int W, int stride, void *workspace_dev,
                           size_t workspace_bytes, void *stream);

/* 2x2x2 stride-2 transposed convolutions with <= 4 channels each way (the U-Net's last up-sampling, utils.py:409-520):
 * y[co][2z+a][2y+b][2x+c] = b[co] + sum_ci w[ci][co][a][b][c] x[ci][z][y][x]; x [CI][D][H][W] -> y [CO][2D][2H][2W], w in
 * nn.ConvTranspose3d's layout [CI][CO][2][2][2]; one sample per call; NULL gradients are skipped. */
size_t trb_upconv2_workspace_bytes(int CI, int CO);
int trb_upconv2_forward(const float *x_dev, const float *w_dev, const float *b_dev, float *y_dev, int CI, int CO, int D, int H,
                        int W, void *stream);
int trb_upconv2_backward(const float *x_dev, const float *w_dev, const float *gy_dev, float *gx_dev, float *gw_dev, float *gb_dev,
                         int CI, int CO, int D, int H, int W, void *workspace_dev, size_t workspace_bytes, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* TRB_H */
