/*
 * sdfrender.h -- C ABI of libsdfrender.so, the B200 (sm_100a) differentiable depth
 * renderer for discretised signed distance fields.
 *
 * This is the drop-in boundary for the one hot path of roym899/sdfest: it replaces the
 * pybind11 module `sdf_renderer_cpp` that the reference JIT-builds from
 *   sdfest/differentiable_renderer/csrc/sdf_renderer.cpp      (forward :42-61, backward :63-86,
 *                                                              module def :88-91)
 *   sdfest/differentiable_renderer/csrc/sdf_renderer_cuda.cu  (launchers :472-556, kernels :241-468)
 * and is bound from Python with ctypes (sdfest_b200/_lib.py; INTEGRATION.md shows the stub a
 * reference maintainer would add to sdf_renderer.py:21-28, 311, 347).
 *
 * Conventions (identical to the reference unless stated)
 *   - every pointer is a DEVICE pointer to contiguous float32 (int32 where stated) memory on
 *     the CURRENT CUDA device; the library never allocates, frees, or synchronises; all work is
 *     enqueued on `stream` (a cudaStream_t passed as void*, NULL = legacy default stream) and is
 *     CUDA-graph capturable.  (The reference allocates its outputs with ATen and launches on the
 *     legacy default stream: sdf_renderer_cuda.cu:484, 495, 525-528, 536.)
 *   - sdf: `resolution`^3 grid(s), index order x,y,z with z contiguous (sdf_renderer_cuda.cu:13,
 *     226-238).  Any resolution >= 2 (the reference kernels hard-code 64: :225-230, 327, 347).
 *     Hypothesis b reads the grid at sdf + b*sdf_stride (elements); sdf_stride = 0 shares one grid.
 *     sdf_layout = SDFR_LAYOUT_DENSE is that layout; SDFR_LAYOUT_SKEWED is the pitched copy made by
 *     sdfr_skew_grids (same fp32 values, element (x,y,z) at x*pitch_x + y*pitch_y + z), which
 *     removes the L1 bank conflicts of the 8-corner gathers (DESIGN.md section 4).  Gradient
 *     grids are always dense.
 *   - position [batch,3], orientation [batch,4] (x,y,z,w; must be unit length -- not normalised,
 *     sdf_renderer_cuda.cu:95-98 is never instantiated), inv_scale [batch]: pose of the grid in the
 *     OpenGL camera frame (camera looks down -z, y up; image row 0 is the top row).
 *   - cx, cy, fx, fy: pinhole parameters in the pixel-centre-0.5 convention
 *     (Camera.get_pinhole_camera_parameters(0.5), sdf_renderer.py:116-133, 310).
 *     NOTE the argument order cx, cy, fx, fy of the reference binding (sdf_renderer.cpp:48-51).
 *   - depth [batch,height,width]: 0 = no surface, else positive z-distance; the kernels write
 *     every element (no pre-zeroing needed; the reference relies on torch::zeros, :484).
 *   - gradients are ACCUMULATED (+=) into the output buffers; pass SDFR_ZERO_GRADS to have the
 *     library clear the requested ones first (cudaMemsetAsync on `stream`).  Buffers whose flag is
 *     not set may be NULL and are never touched (the reference always computes all four,
 *     sdf_renderer.py:346-357).
 *
 * Return value: 0 on success; negative = argument error (SDFR_E_*); positive = cudaError_t
 * reported by the launch.  sdfr_last_error() returns a thread-local description.
 */
#ifndef SDFRENDER_H_
#define SDFRENDER_H_

#ifdef __cplusplus
extern "C" {
#endif

#define SDFR_ABI_VERSION 12

#define SDFR_E_NULL (-1)  /* a required pointer is NULL */
#define SDFR_E_SHAPE (-2) /* resolution < 2, negative sizes, image too large */
#define SDFR_E_FLAGS (-3) /* unknown flag bits */

/* sdf_layout */
#define SDFR_LAYOUT_DENSE 0
#define SDFR_LAYOUT_SKEWED 1

/* flags of the backward entry points */
#define SDFR_GRAD_SDF 0x01u
#define SDFR_GRAD_POSITION 0x02u
#define SDFR_GRAD_ORIENTATION 0x04u
#define SDFR_GRAD_INV_SCALE 0x08u
#define SDFR_GRAD_ALL 0x0fu
/* SDF-gradient corner weights: default = the list the reference CUDA kernel uses
 * (sdf_renderer_cuda.cu:373-388, a permutation of the trilinear weights -- SURVEY.md Q2);
 * with this flag = the true trilinear weights of the reference CPU renderer
 * (simple_renderer.py:399-408). */
#define SDFR_SDF_GRAD_EXACT 0x10u
#define SDFR_ZERO_GRADS 0x20u /* clear the requested gradient buffers before accumulating */
/* sdfr_point_loss_fused only: loss_sum[b] += upstream[b] * sum_m |.| instead of the raw sum, so that
 * hypotheses of different object instances (clouds of different sizes, padded to n_points with points
 * outside the volume) carry their own pc_weight / n_points_b into the loss as well as the gradients */
#define SDFR_LOSS_WEIGHTED 0x40u

/* flags of sdfr_hypothesis_step */
#define SDFR_STEP_CLEAR_INPUTS 0x100u /* zero the sums / gradient inputs after consuming them */
#define SDFR_STEP_NO_UPDATE 0x200u    /* only derive unit_orientation / inv_scale / loss */
/* sdfr_track_best with SDFR_STEP_CLEAR_INPUTS: zero n_inlier only (n_valid depends on the observation
 * alone and was counted once) */
#define SDFR_TRACK_KEEP_VALID 0x400u

int sdfr_abi_version(void);
const char* sdfr_last_error(void);
/* "sm_100a;..." -- what the library was compiled for */
const char* sdfr_build_info(void);
/* upper bound on sphere-tracing steps per ray (the reference has none, SURVEY.md Q5) */
int sdfr_max_steps(void);

/*
 * Skewed layout: pitches (elements) and the number of elements one skewed grid occupies.
 * Any of the output pointers may be NULL.
 */
int sdfr_skewed_pitches(int resolution, int* pitch_y, int* pitch_x, long long* elems);

/*
 * Copy `batch` dense grids (sdf + b*sdf_stride) into skewed grids (skewed + b*skewed_stride,
 * skewed_stride >= elems of sdfr_skewed_pitches).  One streaming pass, ~2*4*R^3 bytes per grid.
 */
int sdfr_skew_grids(const float* sdf, int resolution, long long sdf_stride, int batch,
                    float* skewed, long long skewed_stride, void* stream);

/*
 * Cell bounds of a grid: the first / last CELL index per axis (cell i spans voxels i and i+1) whose
 * smallest corner value is below `tau`, the largest value the interpolated field can have where the
 * march of any hypothesis using the grid can still terminate (sdf_renderer_cuda.cu:286: dist <
 * threshold * t, so trilinear < threshold * t / scale <= tau).  lo > hi: no such cell.
 */
typedef struct sdfr_cell_bounds {
  int lo[3];
  int hi[3];
  float tau;
  int pad;
} sdfr_cell_bounds;

/*
 * Empty-space bounds for the render entry points (their optional `bounds` argument).  The reference
 * marches every ray that enters the grid's [-1,1]^3 box (sdf_renderer_cuda.cu:272-293); most of
 * them cross only space where the field stays above the hit threshold and end with depth 0.  This
 * pass finds, per grid, the box of cells where a hit is possible at all; the render kernels then write 0
 * for rays that miss that box (plus one cell of margin) without marching them, and march all other
 * rays from the reference's own box entry -- identical samples, identical depth, identical gradients.
 * One entry per grid: bounds[b] for grid sdf + b*sdf_stride, a single entry (valid for all `batch`
 * hypotheses) when sdf_stride == 0.  position / inv_scale / threshold are those of the render that
 * will use the bounds (tau depends on them); an entry is ignored by a render whose own tau is larger.
 * Cost: one streaming read of the grids.
 */
int sdfr_grid_bounds(const float* sdf, int resolution, long long sdf_stride, int sdf_layout,
                     const float* position, const float* inv_scale, int batch, float threshold,
                     sdfr_cell_bounds* bounds, void* stream);

/*
 * The same bounds for grids that do not change between renders (fixed shapes, pose-only optimisation):
 * sdfr_grid_slab_minima reads the grids ONCE and keeps, per grid and axis, the smallest voxel value of
 * every slab -- minima [n_grids, 3, resolution] (x, y, z), pose independent; sdfr_bounds_from_minima
 * then derives the cell bounds of the current poses from 3 * resolution comparisons per grid (the box of
 * the cells below tau is the bounding box of the voxels below tau, low side moved down by one cell).
 * n_grids = batch (bounds[b] for hypothesis b) or 1 (one shared grid, one entry, tau = max over the
 * batch).  Results are identical to sdfr_grid_bounds.
 */
int sdfr_grid_slab_minima(const float* sdf, int resolution, long long sdf_stride, int sdf_layout,
                          int n_grids, float* minima, void* stream);
int sdfr_bounds_from_minima(const float* minima, int resolution, int n_grids, const float* position,
                            const float* inv_scale, int batch, float threshold,
                            sdfr_cell_bounds* bounds, void* stream);

/*
 * sdfr_skew_grids and sdfr_grid_bounds in ONE read of the dense grids: writes the skewed copies and
 * their cell bounds (for renders that read the skewed copies).  With sdf_stride == 0 one shared grid is
 * copied once and gets one bounds entry valid for all `batch` hypotheses.
 */
int sdfr_skew_grids_bounds(const float* sdf, int resolution, long long sdf_stride, int batch,
                           float* skewed, long long skewed_stride, const float* position,
                           const float* inv_scale, float threshold, sdfr_cell_bounds* bounds,
                           void* stream);

/*
 * Forward: replaces sdf_renderer_cpp.forward (sdf_renderer.cpp:42-61 ->
 * sdf_renderer_cuda.cu:472-510 -> forward kernel :241-298), batched over `batch` hypotheses.
 */
int sdfr_forward(const float* sdf, int resolution, long long sdf_stride, int sdf_layout, const float* position,
                 const float* orientation, const float* inv_scale, int batch, int width,
                 int height, float cx, float cy, float fx, float fy, float threshold,
                 float* depth, const sdfr_cell_bounds* bounds, void* stream);

/*
 * Same as sdfr_forward, additionally accumulating work counters into stats[4] (device,
 * unsigned long long, caller-zeroed): [0] trilinear samples, [1] pixels whose ray enters the
 * box, [2] hit pixels, [3] rays stopped by the step cap.  Used for the roofline's S and Hh.
 */
int sdfr_forward_stats(const float* sdf, int resolution, long long sdf_stride, int sdf_layout,
                       const float* position, const float* orientation, const float* inv_scale,
                       int batch, int width, int height, float cx, float cy, float fx, float fy,
                       float threshold, float* depth, unsigned long long* stats,
                       const sdfr_cell_bounds* bounds, void* stream);

/*
 * Backward: replaces sdf_renderer_cpp.backward (sdf_renderer.cpp:63-86 ->
 * sdf_renderer_cuda.cu:512-556 -> backward kernel :300-468), batched.
 * grad_depth, depth: [batch,height,width].  grad_sdf: hypothesis b accumulates into
 * grad_sdf + b*grad_sdf_stride (0 = all hypotheses into one grid).  grad_position [batch,3],
 * grad_orientation [batch,4] (x,y,z,w), grad_inv_scale [batch].  `bounds` (optional) must be bounds
 * that were valid for the forward that produced `depth`; they only shrink the image region scanned.
 */
int sdfr_backward(const float* grad_depth, const float* depth, const float* sdf, int resolution,
                  long long sdf_stride, int sdf_layout, const float* position, const float* orientation,
                  const float* inv_scale, int batch, int width, int height, float cx, float cy,
                  float fx, float fy, float* grad_sdf, long long grad_sdf_stride,
                  float* grad_position, float* grad_orientation, float* grad_inv_scale,
                  unsigned flags, const sdfr_cell_bounds* bounds, void* stream);

/*
 * Fused render-and-compare, forward: renders `batch` hypotheses and compares each with an
 * observed depth map using the masked L1 of the reference pipeline
 * (estimation/simple_setup.py:125-131):  overlap = (obs > 0) & (est > 0),
 *   loss_sum[b] += sum_overlap |est - obs|,  n_overlap[b] += |overlap|   (both caller-zeroed
 * unless SDFR_ZERO_GRADS is in `flags`), so that loss_depth[b] = loss_sum[b] / n_overlap[b].
 * depth_obs: hypothesis b compares with depth_obs + b*obs_stride (0 = one shared map).
 */
int sdfr_compare_forward(const float* sdf, int resolution, long long sdf_stride, int sdf_layout,
                         const float* position, const float* orientation,
                         const float* inv_scale, int batch, int width, int height, float cx,
                         float cy, float fx, float fy, float threshold, const float* depth_obs,
                         long long obs_stride, float* depth, float* loss_sum, float* n_overlap,
                         unsigned flags, const sdfr_cell_bounds* bounds, void* stream);

/*
 * Fused render-and-compare, backward: gradient of  sum_b upstream[b] * loss_sum[b]/n_overlap[b]
 * without materialising grad_depth:  g(pixel) = upstream[b] * sign(est - obs) / n_overlap[b] on
 * overlap pixels (sign(0) = 0, as torch.abs), 0 elsewhere.  upstream may be NULL (= 1 for all b).
 * Hypotheses with n_overlap[b] == 0 contribute nothing.
 */
int sdfr_compare_backward(const float* depth, const float* depth_obs, long long obs_stride,
                          const float* n_overlap, const float* upstream, const float* sdf,
                          int resolution, long long sdf_stride, int sdf_layout, const float* position,
                          const float* orientation, const float* inv_scale, int batch,
                          int width, int height, float cx, float cy, float fx, float fy,
                          float* grad_sdf, long long grad_sdf_stride, float* grad_position,
                          float* grad_orientation, float* grad_inv_scale, unsigned flags,
                          const sdfr_cell_bounds* bounds, void* stream);

/*
 * Fused render-and-compare with the backward folded into the SAME traversal (one kernel): as
 * sdfr_compare_forward, plus UNNORMALISED gradients of  sum_overlap |est - obs|  accumulated into
 * the requested buffers while each ray is still live in registers.  The per-hypothesis factor
 * upstream[b] / n_overlap[b] is only known once every pixel is done; all gradients are linear in
 * it, so it is applied afterwards by sdfr_scale_grads (or by the caller, e.g. folded into an
 * optimizer step).  With SDFR_GRAD_SDF each hypothesis needs its own grad grid
 * (grad_sdf_stride != 0 unless batch == 1).  SDFR_ZERO_GRADS also clears loss_sum / n_overlap.
 */
int sdfr_compare_fused(const float* sdf, int resolution, long long sdf_stride, int sdf_layout,
                       const float* position, const float* orientation, const float* inv_scale,
                       int batch, int width, int height, float cx, float cy, float fx, float fy,
                       float threshold, const float* depth_obs, long long obs_stride,
                       float* depth, float* loss_sum, float* n_overlap, float* grad_sdf,
                       long long grad_sdf_stride, float* grad_position, float* grad_orientation,
                       float* grad_inv_scale, unsigned flags, const sdfr_cell_bounds* bounds,
                       void* stream);

/* In place:  grad[b] *= (upstream ? upstream[b] : 1) / n_overlap[b]  (0 where n_overlap == 0)
 * for the buffers selected by `flags`.  bounds (optional): the empty-space bounds that the render which
 * produced the gradients USED (bounds[b * bounds_stride]; bounds_stride 1 = one entry per hypothesis, 0 = the
 * single entry of a shared grid): the SDF gradient can only be non-zero at the voxels of cells inside them,
 * so only those are visited.  Pass NULL when the render ran without bounds. */
int sdfr_scale_grads(const float* n_overlap, const float* upstream, int resolution, int batch,
                     float* grad_sdf, long long grad_sdf_stride, float* grad_position,
                     float* grad_orientation, float* grad_inv_scale, unsigned flags,
                     const sdfr_cell_bounds* bounds, long long bounds_stride, void* stream);

/*
 * Multi-object frame: `n_objects` posed grids rendered into ONE depth map, per-pixel minimum
 * positive depth; winner [height,width] int32 receives the index of the object that produced
 * the pixel (-1 = none; ties go to the lowest index).  No counterpart in the reference (it
 * renders one object per call); semantics are those of oracle.composite_min_depth.
 */
int sdfr_forward_composite(const float* sdf, int resolution, long long sdf_stride, int sdf_layout,
                           const float* position, const float* orientation,
                           const float* inv_scale, int n_objects, int width, int height,
                           float cx, float cy, float fx, float fy, float threshold, float* depth,
                           int* winner, const sdfr_cell_bounds* bounds, void* stream);

/* Backward of sdfr_forward_composite: every pixel back-propagates to its winner. */
int sdfr_backward_composite(const float* grad_depth, const float* depth, const int* winner,
                            const float* sdf, int resolution, long long sdf_stride, int sdf_layout,
                            const float* position, const float* orientation,
                            const float* inv_scale, int n_objects, int width, int height,
                            float cx, float cy, float fx, float fy, float* grad_sdf,
                            long long grad_sdf_stride, float* grad_position,
                            float* grad_orientation, float* grad_inv_scale, unsigned flags,
                            void* stream);

/*
 * Point-cloud loss of the render-and-compare loop, batched: replaces the caller-side torch helper
 * estimation/losses.py:32-135 (pc_loss) as used by estimation/simple_setup.py:134-144
 * (loss_pc = mean |pc_loss|).  points [n_points,3] in the camera frame (hypothesis b reads
 * points + b*points_stride; 0 = one shared cloud); orientation is NOT required to be unit length
 * (normalised inside, with the gradient of the normalisation, losses.py:56); `scale` (not its
 * inverse) as in the reference.  Forward:  loss_sum[b] += sum_m |SDF_b(x_m) * scale_b|  with 0
 * for points outside the grid.  Backward: gradients of  sum_b upstream[b]*loss_sum[b]  (upstream
 * NULL = 1) accumulated into grad_sdf (dense, true trilinear weights), grad_position,
 * grad_orientation and grad_scale (selected by SDFR_GRAD_INV_SCALE).  SDFR_ZERO_GRADS as above.
 */
int sdfr_point_loss_forward(const float* points, long long points_stride, int n_points,
                            const float* sdf, int resolution, long long sdf_stride, int sdf_layout,
                            const float* position, const float* orientation, const float* scale,
                            int batch, float* loss_sum, unsigned flags, void* stream);

int sdfr_point_loss_backward(const float* points, long long points_stride, int n_points,
                             const float* sdf, int resolution, long long sdf_stride,
                             int sdf_layout, const float* position, const float* orientation,
                             const float* scale, int batch, const float* upstream,
                             float* grad_sdf, long long grad_sdf_stride, float* grad_position,
                             float* grad_orientation, float* grad_scale, unsigned flags,
                             void* stream);

/*
 * sdfr_point_loss_forward and _backward in ONE traversal: valid whenever `upstream` does not depend
 * on this call's loss_sum -- in the loop it is the constant pc_weight / n_points
 * (estimation/simple_setup.py:447-452).  loss_sum as in _forward (times upstream[b] with
 * SDFR_LOSS_WEIGHTED), gradients as in _backward; SDFR_ZERO_GRADS clears loss_sum and the requested
 * gradient buffers first.
 */
int sdfr_point_loss_fused(const float* points, long long points_stride, int n_points,
                          const float* sdf, int resolution, long long sdf_stride, int sdf_layout,
                          const float* position, const float* orientation, const float* scale,
                          int batch, const float* upstream, float* loss_sum, float* grad_sdf,
                          long long grad_sdf_stride, float* grad_position, float* grad_orientation,
                          float* grad_scale, unsigned flags, void* stream);

/*
 * The optimiser side of one render-and-compare iteration for `batch` hypotheses, one kernel:
 * replaces torch.optim.Adam over the four parameter groups of estimation/simple_setup.py:400-406
 * (learning rates lr[4] = position, orientation, scale, latent; HOST array), the chain rule through
 * norm_orientation = orientation/|orientation| (:411) and 1/scale (:431), the weighted loss (:447-452)
 * and the renormalisation orientation /= |orientation| (:462).  Per hypothesis b:
 *   coef     = n_overlap[b] > 0 ? depth_weight / n_overlap[b] : 0
 *   g_pos    = coef * gr_position + g2_position
 *   g_unit_q = coef * gr_orientation + g2_orientation;  g_orient = (g_unit_q - q (q.g_unit_q)) / |orientation|
 *   g_scale  = -coef * gr_inv_scale / scale^2 + g2_scale;  g_latent as given
 *   Adam with bias correction (torch/optim/adam.py, no weight decay, no amsgrad), state
 *   exp_avg / exp_avg_sq [batch, 8 + latent_size] (position 0-2, orientation 3-6, scale 7, latent
 *   8..) and step [batch] (int32), all caller-zeroed before the first call;
 *   then orientation is renormalised in place and, if given,
 *   unit_orientation = orientation/|orientation|, inv_scale = 1/scale  (the next iteration's
 *   renderer inputs), loss = depth_weight * loss_sum/n_overlap (NaN without overlap: the reference's
 *   mean over an empty selection, simple_setup.py:131 -- the gradients are 0 there, not NaN) +
 *   point_weight * point_sum + loss_extra.
 * g_orientation_raw (optional) is added to the orientation gradient AFTER the chain rule, i.e. it is a
 * gradient w.r.t. the un-normalised orientation: the point-constraint loss of simple_setup.py:164-175.
 * gr_* are the RAW gradients of sdfr_compare_fused (w.r.t. the unit quaternion and inv_scale);
 * g2_* an already weighted second set (sdfr_point_loss_fused: w.r.t. the quaternion it was given --
 * the unit one -- and scale).  Any gradient pointer may be NULL (= 0); latent / g_latent NULL or
 * latent_size 0 = no latent group (latent_size <= 64).  With SDFR_STEP_CLEAR_INPUTS the kernel zeroes
 * loss_sum, n_overlap, point_sum and every gradient input after reading them (the next
 * iteration's kernels then accumulate without memsets); with SDFR_STEP_NO_UPDATE parameters and
 * state are left untouched and only unit_orientation / inv_scale / loss are written.
 */
int sdfr_hypothesis_step(float* position, float* orientation, float* scale, float* latent,
                         int latent_size, int batch, float* loss_sum, float* n_overlap,
                         float* gr_position, float* gr_orientation, float* gr_inv_scale,
                         float depth_weight, float* point_sum, float point_weight,
                         float* g2_position, float* g2_orientation, float* g2_scale,
                         float* g_latent, float* g_orientation_raw, float* loss_extra, float* exp_avg,
                         float* exp_avg_sq, int* step, const float* lr, float beta1, float beta2,
                         float eps, float* unit_orientation, float* inv_scale, float* loss,
                         unsigned flags, void* stream);

/*
 * Several camera views of one object (estimation/simple_setup.py:420-446): the pose lives in the world
 * frame and is moved into each of n_views camera frames,
 *   position_c[v,b]    = R(conj(cam_orientation[v])) (position[b] - cam_position[v])
 *   orientation_c[v,b] = conj(cam_orientation[v]) (x) unit_orientation[b]      (scalar-last, unit)
 *   inv_scale_c[v,b]   = inv_scale[b]
 * (initialization/quaternion_utils.py:12-66); outputs [n_views, batch, ...] so that view v is one
 * batched render of `batch` hypotheses at position_c + v*batch*3 etc.
 */
int sdfr_view_poses(const float* position, const float* unit_orientation, const float* inv_scale,
                    const float* cam_position, const float* cam_orientation, int n_views, int batch,
                    float* position_c, float* orientation_c, float* inv_scale_c, void* stream);

/*
 * Adjoint of sdfr_view_poses plus the loss of the view loop: per hypothesis, summed over the views,
 *   g_position    = sum_v R(cam_orientation[v]) (gr_position[v] + g2_position[v])
 *   g_orientation = sum_v cam_orientation[v] (x) (gr_orientation[v] + g2_orientation[v])   (w.r.t. the
 *                   world-frame UNIT quaternion)
 *   g_scale       = sum_v g2_scale[v] - gr_inv_scale[v] / scale^2
 *   loss         += sum_v depth_weight * loss_sum[v]/n_overlap[v] (NaN without overlap) + point_sum[v]
 * gr_* = gradients of the (already weighted and normalised) depth loss of each view w.r.t. its
 * camera-frame pose (sdfr_compare_backward with upstream = depth_weight), g2_* / point_sum = the weighted
 * point loss of each view (sdfr_point_loss_fused with SDFR_LOSS_WEIGHTED); all [n_views, batch, ...],
 * any may be NULL.  The outputs feed sdfr_hypothesis_step as its g2_* inputs (and `loss` as its
 * loss_extra).  SDFR_STEP_CLEAR_INPUTS zeroes the per-view inputs after reading them.
 */
int sdfr_views_pull_back(const float* cam_orientation, const float* scale, int n_views, int batch,
                         float* gr_position, float* gr_orientation, float* gr_inv_scale,
                         float* g2_position, float* g2_orientation, float* g2_scale, float* loss_sum,
                         float* n_overlap, float depth_weight, float* point_sum, float* g_position,
                         float* g_orientation, float* g_scale, float* loss, unsigned flags,
                         void* stream);

/*
 * Point constraint of the loop (estimation/simple_setup.py:164-175 -> estimation/losses.py:138-153):
 *   loss[b] += weight * | q_b (x) (source,0) (x) conj(q_b) - target |,   q_b = orientation[b] as stored,
 * NOT normalised (quaternion_utils.py:37-54 does not normalise either), and its gradient w.r.t. that
 * un-normalised quaternion accumulated into g_orientation_raw [batch,4] -- the two optional inputs of
 * sdfr_hypothesis_step.  source / target: HOST float[3].  Either output may be NULL.
 */
int sdfr_point_constraint(const float* orientation, int batch, const float* source, const float* target,
                          float weight, float* g_orientation_raw, float* loss, void* stream);

/*
 * Result selection of the loop, batched and without the reference's host synchronisation
 * (estimation/simple_setup.py:177-211, called every iteration at :463).
 * sdfr_inlier_count:  n_inlier[b] += #{pixels: |obs - est| / obs < rel_threshold}  (IEEE division: a
 *   pixel with obs == 0 gives inf or nan and is never an inlier, as in the torch expression :183-184),
 *   n_valid[b] += #{obs != 0} (:186).  depth [batch, height*width] = the estimate (e.g. the image
 *   sdfr_compare_fused wrote); hypothesis b is compared with depth_obs + b*obs_stride (0 = one shared
 *   observation).  SDFR_ZERO_GRADS clears both counters first.
 * sdfr_track_best:  ratio[b] = n_inlier[b] / n_valid[b] (:187; 0/0 = nan); where best_iteration[b] < 0
 *   (nothing kept yet, the reference's `is None`) or ratio[b] > best_ratio[b] (:205), best_ratio,
 *   best_iteration (= step[b], the counter sdfr_hypothesis_step maintains; 0 if NULL) and the snapshots
 *   best_position / best_orientation / best_scale / best_latent are overwritten with the current
 *   parameters.  NOTE: the reference stores REFERENCES to the live parameter tensors (:207-210), which
 *   the in-place optimiser keeps mutating, so its "best" estimate always equals the last iterate; this
 *   entry point keeps the copy the code evidently intends.  ratio / latent / best_latent may be NULL.
 *   SDFR_STEP_CLEAR_INPUTS zeroes n_inlier / n_valid after reading them (n_inlier only with
 *   SDFR_TRACK_KEEP_VALID).
 * sdfr_compare_fused_inliers:  sdfr_compare_fused that also counts the inliers in the same traversal
 *   (no extra pass over the images): n_inlier[b] += #{overlap pixels (est > 0, obs > 0):
 *   |obs - est| / obs < rel_threshold}.  Equal to sdfr_inlier_count's n_inlier whenever the observed
 *   depth is non-negative and rel_threshold <= 1 (a pixel the estimate misses has relative error
 *   exactly 1 and a pixel without observation is never an inlier; larger thresholds are rejected with
 *   SDFR_E_SHAPE).  n_valid = #{obs != 0} depends on the observation only: count it once with
 *   sdfr_inlier_count.  SDFR_ZERO_GRADS also clears n_inlier.
 */
int sdfr_inlier_count(const float* depth, const float* depth_obs, long long obs_stride, int batch,
                      int width, int height, float rel_threshold, float* n_inlier, float* n_valid,
                      unsigned flags, void* stream);

int sdfr_compare_fused_inliers(const float* sdf, int resolution, long long sdf_stride, int sdf_layout,
                               const float* position, const float* orientation,
                               const float* inv_scale, int batch, int width, int height, float cx,
                               float cy, float fx, float fy, float threshold, const float* depth_obs,
                               long long obs_stride, float* depth, float* loss_sum, float* n_overlap,
                               float rel_threshold, float* n_inlier, float* grad_sdf,
                               long long grad_sdf_stride, float* grad_position,
                               float* grad_orientation, float* grad_inv_scale, unsigned flags,
                               const sdfr_cell_bounds* bounds, void* stream);

int sdfr_track_best(float* n_inlier, float* n_valid, const float* position, const float* orientation,
                    const float* scale, const float* latent, int latent_size, int batch,
                    const int* step, float* ratio, float* best_ratio, int* best_iteration,
                    float* best_position, float* best_orientation, float* best_scale,
                    float* best_latent, unsigned flags, void* stream);

/*
 * Decoder tail (SURVEY.md section 8f rank 2): the last two operators of the reference SDF decoder,
 *   interpolate(x -> (R,R,R), mode="trilinear", align_corners=False)   sdfest/vae/sdf_vae.py:235-244
 *   Conv3d(channels -> 1, kernel_size=1), no ReLU                       sdfest/vae/sdf_vae.py:245-247
 * as ONE pass that never materialises the channels x R^3 intermediate and writes the grid in the
 * layout the renderer reads (dense or skewed; sdf_stride >= elements of one grid in that layout).
 * x [batch, channels, in_size^3]; weight [channels] (the conv weight (1,C,1,1,1) flattened); bias
 * [1] or NULL; base: an optional dense [R,R,R] grid added to every hypothesis' output (residual
 * decoding around a fixed shape; NULL for the reference decoder).  channels <= 16; in_size,
 * resolution <= 128.  Interpolation indices and weights
 * are ATen's (upsample_trilinear3d, align_corners = false); the channel contraction is done before
 * the interpolation (both are linear), so results agree with torch to fp32 rounding.
 */
int sdfr_decoder_tail_forward(const float* x, int channels, int in_size, const float* weight,
                              const float* bias, const float* base, int batch, int resolution,
                              float* sdf, long long sdf_stride, int sdf_layout, void* stream);

/*
 * sdfr_decoder_tail_forward that also produces the empty-space bounds of the grids it writes (one entry per
 * hypothesis, identical to sdfr_grid_bounds on the written grids for the given poses and threshold): the
 * values are compared with the hit-threshold bound as they are stored, so the loop needs no separate read of
 * the grids.
 */
int sdfr_decoder_tail_forward_bounds(const float* x, int channels, int in_size, const float* weight,
                                     const float* bias, const float* base, int batch, int resolution,
                                     float* sdf, long long sdf_stride, int sdf_layout,
                                     const float* position, const float* inv_scale, float threshold,
                                     sdfr_cell_bounds* bounds, void* stream);

/*
 * Adjoint of sdfr_decoder_tail_forward w.r.t. x (the decoder is frozen in the estimation loop,
 * simple_setup.py:65: no weight / bias gradients):  grad_x[b] = (written, not accumulated)
 *   weight[c] * W^T ( coef[b] * grad_sdf[b] + grad_sdf_extra[b] ),
 * coef[b] = (upstream ? upstream[b] : 1) / n_overlap[b] (0 where n_overlap[b] == 0) when n_overlap
 * is given -- the normalisation sdfr_compare_fused defers -- else upstream[b] (or 1).  Both
 * gradient grids are dense; grad_sdf_extra may be NULL.
 */
int sdfr_decoder_tail_backward(const float* grad_sdf, long long grad_sdf_stride,
                               const float* n_overlap, const float* upstream,
                               const float* grad_sdf_extra, long long extra_stride,
                               const float* weight, int channels, int in_size, int batch,
                               int resolution, float* grad_x, void* stream);

/*
 * Decoder trunk stages (sdfest/vae/sdf_vae.py:225-247: per stage `interpolate(..., "trilinear",
 * align_corners=False)` to the stage's in_size, Conv3d, optional ReLU).  Every decoder the reference
 * ships (vae/configs/*.yaml, initialization/configs/vae_models/*.yaml) uses 3x3x3 "valid"
 * convolutions between 4..32 channels.  All tensors contiguous NCDHW fp32.
 *
 * sdfr_upsample3d_forward:  y[n] = trilinear resize of x[n] (in_size^3 -> out_size^3) for n_volumes
 *   volumes (batch*channels); ATen's align_corners = false indices / weights.  _backward: its adjoint
 *   (grad_x written, not accumulated).  Sizes <= 128.
 * sdfr_conv3d_forward:  y [batch, out_channels, (in_size-2)^3] = conv3d(x, weight [Co,Ci,3,3,3]) + bias
 *   (NULL = none), ReLU if `relu`.  out_channels in {4, 8, 16, 32}.
 * sdfr_conv3d_backward_data:  grad_x [batch, in_channels, in_size^3] = transposed convolution of
 *   grad_y * (y > 0)  (y = the forward's output, the ReLU mask; NULL = no ReLU) with weight;
 *   in_channels in {4, 8, 16, 32}.  The decoder is frozen in the estimation loop
 *   (simple_setup.py:65): there is no weight gradient.
 */
int sdfr_upsample3d_forward(const float* x, int n_volumes, int in_size, int out_size, float* y,
                            void* stream);
int sdfr_upsample3d_backward(const float* grad_y, int n_volumes, int in_size, int out_size,
                             float* grad_x, void* stream);
int sdfr_conv3d_forward(const float* x, int batch, int in_channels, int in_size, const float* weight,
                        const float* bias, int out_channels, int kernel_size, int relu, float* y,
                        void* stream);
int sdfr_conv3d_backward_data(const float* grad_y, const float* y, int batch, int in_channels,
                              int in_size, const float* weight, int out_channels, int kernel_size,
                              float* grad_x, void* stream);

/*
 * Observed point clouds of K object instances, without a host synchronisation (the reference builds one
 * cloud per detection with torch.nonzero: initialization/pointset_utils.py:34-89).
 * Pixel p of instance k is selected where its masked depth is non-zero:
 *   masked = depth[k*depth_stride + p], 0 where mask[k*H*W + p] == 0, 0 where masked > far_field
 * (depth_stride = 0 shares one depth image; mask: bytes 0/1 such as a torch.bool tensor, NULL = no mask;
 * far_field = +inf for none).  Selected pixels become points in row-major pixel order (the order of
 * torch.nonzero), in the OpenGL camera frame:
 *   ((col - cx) * z / fx, -(row - cy) * z / fy, -z),  z = masked depth,
 * with cx, cy, fx, fy in the pixel-centre-0 convention (Camera.get_pinhole_camera_parameters(0.0)); the
 * division is a multiplication by the fp32 reciprocal, as torch computes it on CUDA, so the values equal
 * losses.depth_to_pointcloud's on the same device bit for bit.
 * Outputs: masked_depth [K,H,W] (NULL skips it); points [K,capacity,3], rows [count, capacity) set to
 * 1e6 (losses.PAD_COORDINATE: outside every SDF volume); counts [K] int64, the TRUE number of selected
 * pixels even when it exceeds capacity (only the first `capacity` points are written).  points may be
 * NULL with capacity 0: counts (and masked_depth) only.  scratch: device memory of the size
 * sdfr_depth_to_points_scratch reports.  At most 2^30 pixels per image.
 */
int sdfr_depth_to_points_scratch(int n_instances, int width, int height, long long* bytes);
int sdfr_depth_to_points(const float* depth, long long depth_stride, const unsigned char* mask,
                         int n_instances, int width, int height, float far_field, float fx, float fy,
                         float cx, float cy, float* masked_depth, float* points, int capacity,
                         long long* counts, void* scratch, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SDFRENDER_H_ */
