/* libsqloss -- C ABI of the B200-native superquadric (SQ) inside-outside losses.
 *
 * Drop-in boundary for the loss hot path of timoblak/sq-recovery.  The reference has no FFI of its own (it is
 * pure Python on torch ops); each entry point below replaces the body of one reference method, and the Python
 * classes in sq_recovery_b200/classes.py (same names and signatures as torch/classes.py) are the binding a
 * maintainer would add -- see INTEGRATION.md.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the parameter name ends in _host;
 *   - the caller owns all buffers; the library keeps no state between calls except inside an sq_ctx;
 *   - launches are asynchronous on `stream` (a cudaStream_t); nothing here synchronises, except the *_host calls;
 *   - return value: 0 on success, otherwise a cudaError_t value (sq_error_string() describes it);
 *   - parameter rows are [a1 a2 a3 | e1 e2 | t1 t2 t3 | qx qy qz qw] (torch/train.py:89), dtype SQ_F32 or SQ_F64;
 *     gradients are written in the same dtype as the parameters they belong to;
 *   - a grid is (n, step, z0): coordinate(i) = i*step, except coordinate(0) = z0.  That covers every grid the
 *     reference builds: ExplicitLoss arange(0,1+1/R,1/R) with 0 -> 1e-4 (torch/classes.py:122-126),
 *     ImplicitLoss linspace(0,1,R) with 0 -> 1e-4 (:218-221), IoUAccuracy linspace(0,1,R) (:389).
 */
#ifndef SQLOSS_H
#define SQLOSS_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* sq_stream_t;           /* cudaStream_t */
enum { SQ_F32 = 0, SQ_F64 = 1, SQ_U8 = 2 };   /* SQ_U8: 8-bit depth images of the host-buffer calls, 8-bit voxels */

/* Library / device introspection. */
const char* sq_version(void);
const char* sq_error_string(int err);
int sq_device_sm_count(int device, int* sm_count);

/* Measurement hook: the next column kernel (the dominant kernel of sq_implicit_loss / sq_explicit_loss /
 * sq_iou_counts) launched by the calling thread is bracketed by cudaEventRecord(ev_before) / (ev_after) on its
 * stream.  One-shot; pass cudaEvent_t handles created with timing enabled.  bench.py uses it for the roofline. */
void sq_profile_events(void* ev_before, void* ev_after);

/* Bytes of device scratch a call with this batch size and grid size needs (same for all entry points).
 *
 * Scratch contract: the first 256 bytes of a scratch buffer are a control block (work-queue counters of the
 * persistent kernels) that must be ZERO when a call starts.  Call sq_scratch_init() once after allocating the buffer
 * (or zero it yourself); every entry point leaves the block zero again when its kernels have finished, so one buffer
 * can be reused by any sequence of stream-ordered calls, with any batch / grid sizes it is large enough for, without
 * a memset on the per-call path.  A buffer must not be used by two streams at once.  After a call that returned an
 * error, call sq_scratch_init() again.
 */
size_t sq_scratch_bytes(int batch, int n);
int sq_scratch_init(void* scratch, size_t scratch_bytes, sq_stream_t stream);

/* ImplicitLoss.__call__ + depth_projection (torch/classes.py:232-295), forward and backward in one pass.
 *   pred        [batch,12] parameters (pred_dtype)
 *   target      depth images, fp32; pixel (row, col) of the render_size x render_size NEAREST-resized image of
 *               sample b is target[b*target_stride_b + row_off[row] + col_off[col]]  (F.interpolate, :286);
 *               NULL = no loss (depth_out only)
 *   tau, sharpness  ImplicitLoss(tau, sigmoid_sharpness) (:208)
 *   loss_out    [1]  fp64: mean_b mean_pix |target - depth|            (may be NULL)
 *   per_sample  [batch] fp64: mean_pix |target - depth| per sample     (may be NULL)
 *   grad_pred   [batch,12] d loss_out / d pred (pred_dtype)            (NULL = forward only)
 *   depth_out   [batch,n,n] fp32 rendered depth, image orientation (:279) (may be NULL)
 */
int sq_implicit_loss(const void* pred, int pred_dtype, int batch, int n, double step, double z0,
                     const float* target, long long target_stride_b, const int* row_off, const int* col_off,
                     float tau, float sharpness,
                     double* loss_out, double* per_sample, void* grad_pred, float* depth_out,
                     void* scratch, size_t scratch_bytes, sq_stream_t stream);

/* The same with the network heads fused in (SURVEY 8f-3): rows of raw_heads are the raw outputs of the four linear
 * heads [size(3) | shape(2) | position(3) | rotation(4)]; the kernel applies sigmoid to the first eight and L2
 * normalisation to the quaternion (torch/models.py:28,52,75,98), the torch.cat of torch/train.py:89 and the clamp, and
 * returns d loss / d raw_heads in grad_raw -- replacing the ~14 small elementwise launches around the loss per step.
 */
int sq_implicit_loss_heads(const void* raw_heads, int dtype, int batch, int n, double step, double z0,
                           const float* target, long long target_stride_b, const int* row_off, const int* col_off,
                           float tau, float sharpness,
                           double* loss_out, double* per_sample, void* grad_raw, float* depth_out,
                           void* scratch, size_t scratch_bytes, sq_stream_t stream);

/* Vector-Jacobian product of ImplicitLoss.depth_projection (torch/classes.py:232-282):
 *   grad_depth  [batch,n,n] fp32, contiguous, image orientation (the layout of depth_out)
 *   grad_pred   [batch,12] (pred_dtype) = sum_pix grad_depth[b,pix] * d depth[b,pix] / d pred[b]
 *               (clamp masks as in the loss; quaternion not normalised)
 * Same scratch contract as the other entry points; asynchronous on `stream`.  Self-contained: it reads nothing an earlier
 * call left in the scratch buffer (it renders the columns again), so any calls may run between the forward and this one.
 * For the MAE objective the fused sq_implicit_loss is cheaper: it needs one walk of the grid, this path two.
 */
int sq_depth_projection_vjp(const void* pred, int pred_dtype, int batch, int n, double step, double z0,
                            float tau, float sharpness, const float* grad_depth, void* grad_pred,
                            void* scratch, size_t scratch_bytes, sq_stream_t stream);

/* Jacobian of ImplicitLoss.depth_projection (torch/classes.py:232-282), one row per pixel:
 *   jac        [batch,n,n,12] fp32, image orientation: jac[b,r,c,j] = d depth[b,r,c] / d pred[b,j]
 *              (clamp masks as in the loss; quaternion not normalised).  fp32 for fp32 and fp64 pred alike: each entry
 *              is an fp32 sum, and fp64 storage would double the call's largest buffer (48 bytes per pixel).
 *   depth_out  [batch,n,n] fp32 render of the same walk (may be NULL)
 * Weight cut of one sample (as sq_depth_projection_vjp): row (b,r,c) is that call's result for a one-hot grad_depth on
 * pixel (b,r,c).  Scratch: sq_scratch_bytes(batch, n), usual control-block contract.  Asynchronous, self-contained,
 * capturable; its column kernel is timed by sq_profile_events.  NULL pred or jac: cudaErrorInvalidValue. */
int sq_depth_projection_jacobian(const void* pred, int pred_dtype, int batch, int n, double step, double z0,
                                 float tau, float sharpness, float* depth_out, float* jac,
                                 void* scratch, size_t scratch_bytes, sq_stream_t stream);

/* ExplicitLoss.__call__ (torch/classes.py:138-201): mean_b( mult * mean_pts (o_true - o_pred)^2 ),
 * o = sigmoid(sharpness (1 - F)); the reference uses sharpness 5, mult 100 (:187, :198).
 *   grad_pred   [batch,12] d loss / d pred (params_dtype)              (NULL = forward only)
 */
int sq_explicit_loss(const void* true_params, const void* pred, int params_dtype, int batch,
                     int n, double step, double z0, float sharpness, float mult,
                     double* loss_out, double* per_sample, void* grad_pred,
                     void* scratch, size_t scratch_bytes, sq_stream_t stream);

/* IoUAccuracy.__call__ (torch/classes.py:394-447): voxel counts of (F_true<=1 & F_pred<=1) and (.. | ..) per
 * sample, no clamping, no zero fix-up.  inter/uni: [batch] int64.  The ratios are formed by the caller.
 */
int sq_iou_counts(const void* true_params, const void* pred, int params_dtype, int batch,
                  int n, double step, double z0, long long* inter, long long* uni,
                  void* scratch, size_t scratch_bytes, sq_stream_t stream);

/* LeastSquares.__call__ (torch/classes.py:318-371): points are the pixels > 0 of the nearest-resized depth image,
 * (col/R, 1 - row/R, depth); loss = mean_b sum_pts (sqrt(a1 a2 a3) (F - 1))^2.  Target addressing as above.
 */
int sq_least_squares(const void* pred, int pred_dtype, int batch, int render_size,
                     const float* target, long long target_stride_b, const int* row_off, const int* col_off,
                     double* loss_out, double* per_sample, void* grad_pred,
                     void* scratch, size_t scratch_bytes, sq_stream_t stream);

/* LeastSquares.energy_function (torch/classes.py:318-356) on an explicit point list -- the stored-point-cloud variant.
 *   points      compacted structure of arrays, fp32: row 0 = x, row 1 = y, row 2 = z of the points of ALL samples back
 *               to back; rows are `stride` floats apart; stride is a multiple of 4 and >= the total point count rounded
 *               up to a multiple of 4, and `points` is 16-byte aligned (the kernel reads four points per 16-byte load)
 *   offsets     [batch+1] int64: sample b owns points [offsets[b], offsets[b+1])
 *   max_points  the largest offsets[b+1] - offsets[b] (host value: it sizes the launch)
 *   per_sample  [batch] fp64 energies sum_pts (sqrt(a1 a2 a3) (F - 1))^2      (may be NULL)
 *   loss_out    [1] fp64 their mean over the batch (:371)                      (may be NULL)
 *   grad_pred   [batch,12] d per_sample[b] / d pred[b]                         (NULL = forward only)
 * Scratch: sq_points_scratch_bytes(batch, max_points).
 */
size_t sq_points_scratch_bytes(int batch, long long max_points);
int sq_least_squares_points(const void* pred, int pred_dtype, int batch, const float* points, long long stride,
                            const long long* offsets, long long max_points,
                            double* loss_out, double* per_sample, void* grad_pred,
                            void* scratch, size_t scratch_bytes, sq_stream_t stream);

/* Gauss-Newton normal equations of LeastSquares: per sample b, with residuals r_i = sqrt(a1 a2 a3) (F(x_i) - 1) over the
 * sample's points and J_b their Jacobian (rows dr_i / dpred[b]), and no 1 / batch factor:
 *   per_sample  [batch] fp64 E_b = sum_i r_i^2                 (the bits of sq_least_squares_points' / sq_least_squares' per_sample)
 *   grad_pred   [batch,12] dE_b / dpred[b] = 2 J_b^T r_b (pred_dtype; the bits of sq_least_squares_points' grad_pred)
 *   jtj         [batch,12,12] fp64 J_b^T J_b, row-major, exactly symmetric
 * J carries the clamp masks as the gradient does (a clamped-out parameter has an exactly zero row and column of jtj), the
 * quaternion is not normalised, and a point whose F >= 1e18 adds nothing to jtj (as it adds nothing to the gradient).
 * Points and their addressing are those of sq_least_squares (the image call) and sq_least_squares_points (the list call).
 * A NULL per_sample, grad_pred or jtj returns cudaErrorInvalidValue.  Scratch: sq_normal_scratch_bytes(batch, max_points),
 * with max_points = render_size * render_size for the image call; the control-block contract is that of
 * sq_scratch_bytes.  Asynchronous on `stream`, self-contained, and capturable into a CUDA graph.
 */
size_t sq_normal_scratch_bytes(int batch, long long max_points);
int sq_least_squares_normal(const void* pred, int pred_dtype, int batch, int render_size,
                            const float* target, long long target_stride_b, const int* row_off, const int* col_off,
                            double* per_sample, void* grad_pred, double* jtj,
                            void* scratch, size_t scratch_bytes, sq_stream_t stream);
int sq_least_squares_points_normal(const void* pred, int pred_dtype, int batch, const float* points, long long stride,
                                   const long long* offsets, long long max_points,
                                   double* per_sample, void* grad_pred, double* jtj,
                                   void* scratch, size_t scratch_bytes, sq_stream_t stream);

/* ExplicitLoss.occupancy / IoUAccuracy.ins_outs (torch/classes.py:138-189, 394-426): the full field [batch,n,n,n]
 * (index order [x][y][z], fp32).  mode 0: F without clamp/fix-up (ins_outs); mode 1: sigmoid(sharpness (1-F))
 * with clamp and fix-up (occupancy).  A convenience for callers that want the grid itself.
 */
int sq_field(const void* params, int params_dtype, int batch, int n, double step, double z0,
             int mode, float sharpness, float* out, void* scratch, size_t scratch_bytes, sq_stream_t stream);

/* Vector-Jacobian product of ExplicitLoss.occupancy / sq_field mode 1 (torch/classes.py:138-189):
 *   grad_field  [batch,n,n,n] fp32, contiguous, index order [x][y][z] (the layout sq_field writes)
 *   grad_params [batch,12] (params_dtype) = sum_vox grad_field[b,vox] * d occ[b,vox] / d params[b]
 *               (clamp masks and zero fix-up as in the loss; quaternion not normalised)
 * Same scratch contract as the other entry points; asynchronous on `stream`.  Self-contained: it reads nothing an earlier
 * call left in the scratch buffer, so any calls may run between the forward and this one.  Voxels whose weight
 * o (1 - o) is below 2^-36 are dropped (DESIGN.md 2).  For the MSE against the occupancy of known parameters the fused
 * sq_explicit_loss is cheaper: it needs neither the field nor its gradient in memory.
 */
int sq_occupancy_vjp(const void* params, int params_dtype, int batch, int n, double step, double z0,
                     float sharpness, const float* grad_field, void* grad_params,
                     void* scratch, size_t scratch_bytes, sq_stream_t stream);

/* ExplicitLoss's MSE of the occupancy field against voxel data (torch/classes.py:138-189), forward and backward in one
 * walk, with no field in memory:
 *   loss = mean_b mult * mean_vox (v - o_pred)^2,  o = sigmoid(sharpness (1 - F)), clamp and zero fix-up as in the loss,
 *   v = voxel_scale * voxels[b][x][y][z]   (voxels: [batch,n,n,n] contiguous, index order [x][y][z], SQ_F32 or SQ_U8)
 *   loss_out    [1] fp64 (may be NULL);  per_sample [batch] fp64 mult * mean_vox (v - o_pred)^2 (may be NULL)
 *   grad_pred   [batch,12] d loss_out / d pred (params_dtype)          (NULL = forward only; the loss bits are the same)
 * Same scratch contract as the other entry points; asynchronous on `stream`; self-contained.  Every voxel is read once
 * and every one counts: where the predicted occupancy is below the cut, the term is v^2.  The walk and the backward cut
 * are those of sq_occupancy_vjp (o (1 - o) < 2^-36: the difference v - o can be large and of one sign over the whole soft
 * shell).  A NULL voxels or pred, or another voxel_dtype, returns cudaErrorInvalidValue.
 */
int sq_voxel_loss(const void* voxels, int voxel_dtype, float voxel_scale,
                  const void* pred, int params_dtype, int batch, int n, double step, double z0,
                  float sharpness, float mult, double* loss_out, double* per_sample, void* grad_pred,
                  void* scratch, size_t scratch_bytes, sq_stream_t stream);

/* ---- host-buffer entry points (what a non-torch caller binds; H2D/D2H copies happen inside) -------------------
 * An sq_ctx owns a stream, device buffers and pinned staging buffers on one device; buffers grow on demand and are
 * reused across calls.  The *_host calls return after the results are in the caller's host memory.
 */
typedef struct sq_ctx sq_ctx;
int sq_ctx_create(int device, sq_ctx** out);
void sq_ctx_destroy(sq_ctx* ctx);

/* ImplicitLoss on host data: pred_host [batch,12] fp32, images_host [batch,H,W] fp32 (nearest-resized to
 * render_size inside, like F.interpolate), grad_host [batch,12] fp32 or NULL, loss_host [1] fp64. */
int sq_implicit_loss_host(sq_ctx* ctx, const float* pred_host, int batch, int render_size,
                          const float* images_host, int height, int width, float tau, float sharpness,
                          double* loss_host, float* grad_host);

/* The same in two halves, on one of the context's SQ_HOST_SLOTS slots (0 ... SQ_HOST_SLOTS-1), so that a caller can keep
 * several batches in flight: while one slot's kernels run, the next slots' images cross PCIe (three in flight keep the
 * bus busy all the time on BASELINE config 2).
 *   submit  enqueues the copies and kernels of one ImplicitLoss call on the slot's stream and returns at once.
 *           images_host [batch,H,W] of image_dtype SQ_F32, or SQ_U8 for 8-bit depth images -- the reference's data are
 *           8-bit BMPs divided by 255 (torch/test.py:29-30, torch/classes.py:82-88); every sampled pixel is multiplied by
 *           image_scale (1/255 for such images, 1 for fp32 depth in [0,1]).  Of pinned (or registered) images only the
 *           sampled rows cross the bus: as one strided copy-engine transfer when H and W are multiples of render_size,
 *           else read in place by a kernel; pageable images are copied whole.  pred_host is copied before submit returns;
 *           images_host must stay valid and unchanged until the matching wait.  cudaErrorNotReady if the slot still
 *           holds a result.
 *   wait    blocks until that call has finished and copies loss (and the gradient if it was asked for) out.
 */
#define SQ_HOST_SLOTS 8
int sq_implicit_loss_host_submit(sq_ctx* ctx, int slot, const float* pred_host, int batch, int render_size,
                                 const void* images_host, int image_dtype, int height, int width, float image_scale,
                                 float tau, float sharpness, int want_grad);
int sq_implicit_loss_host_wait(sq_ctx* ctx, int slot, double* loss_host, float* grad_host);

/* ExplicitLoss on host data: parameters [batch,12] fp32, grid of ExplicitLoss(render_size). */
int sq_explicit_loss_host(sq_ctx* ctx, const float* true_host, const float* pred_host, int batch, int render_size,
                          double* loss_host, float* grad_host);

/* IoUAccuracy on host data: per-sample counts [batch] int64. */
int sq_iou_counts_host(sq_ctx* ctx, const float* true_host, const float* pred_host, int batch, int render_size,
                       long long* inter_host, long long* uni_host);

#ifdef __cplusplus
}
#endif
#endif /* SQLOSS_H */
