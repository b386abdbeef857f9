/*
 * dfusion.h -- C ABI of the B200-native DynamicFusion hot path (libdfusion.so).
 *
 * The reference (mihaibujanca/dynamicfusion) has no FFI layer; its seam is the internal launcher layer
 * `kfusion::device::*` declared in kfusion/src/internal.hpp:105-147, called by the host classes
 * cuda::TsdfVolume / cuda::ProjectiveICP / imgproc free functions / WarpField / KinFu.  Every entry point
 * below replaces one of those launchers (cited per function) and is what the C++ mirror classes in
 * include/kfusion/ (and the ctypes binding in dynamicfusion_b200/capi.py) bind.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - 2-D images are (ptr, pitch in BYTES, cols, rows), as kfusion::cuda::PtrStepSz (kernel_containers.hpp:37-63);
 *   - float4 maps hold (x, y, z, w) per pixel: kfusion::Point / Normal (types.hpp:31-42);
 *   - `stream` is a cudaStream_t passed as void* (0 = default stream); calls are asynchronous unless stated;
 *   - return value: 0 on success, otherwise a cudaError_t value (df_error_string() describes it).  The C++
 *     mirror turns a non-zero status into the reference's behaviour (print "KinFu2 error: ..." and exit,
 *     device_memory.cpp:7-11).
 * No torch / C++ types cross this boundary.
 */
#ifndef DFUSION_H
#define DFUSION_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* device::TsdfVolume POD (internal.hpp:29-49).  data: one u32 per voxel, low 16 bits = fp16 TSDF, high 16 bits =
 * u16 weight (ushort2{x,y}); linear index x + y*dims[0] + z*dims[0]*dims[1] (device.hpp:17-27). */
typedef struct df_volume {
    uint32_t *data;
    int dims[3];
    float voxel_size[3];
    float trunc_dist;
    int max_weight;
} df_volume;

/* device::Aff3f (internal.hpp:26-27): R row-major, then t */
typedef struct df_aff3f { float R[9]; float t[3]; } df_aff3f;
/* kfusion::Intr (types.hpp:20-27) */
typedef struct df_intr { float fx, fy, cx, cy; } df_intr;

const char *df_error_string(int status);
int df_version(void);

/* ------------------------------------------------------------------ TSDF volume ---------------------------------------------------------- */
/* device::clear_volume (internal.hpp:105, tsdf_volume.cu:15-41) */
int df_clear_volume(df_volume vol, void *stream);

/* device::compute_dists (internal.hpp:121, imgproc.cu:259-294): u16 mm depth -> fp16 metric ray length */
int df_compute_dists(const uint16_t *depth, size_t depth_pitch, int cols, int rows, df_intr intr,
                     uint16_t *dists, size_t dists_pitch, void *stream);

/* device::integrate (internal.hpp:106, tsdf_volume.cu:51-112,141-161).  vol2cam = camera_pose^-1 * volume_pose
 * (tsdf_volume.cpp:112).  If n_updated (device, u64) is non-NULL the number of voxels written is ADDED to it. */
int df_integrate(df_volume vol, const uint16_t *dists, size_t dists_pitch, int cols, int rows,
                 df_aff3f vol2cam, df_intr intr, unsigned long long *n_updated, void *stream);

/* Activity map (optional accelerator for df_extract_cloud_tracked): one byte per DF_ACTIVITY_VOXELS consecutive voxels of the
 * volume array, non-zero iff an integration stored a voxel with W != 0 && F != 1 there since the map was last zeroed.  Only such
 * voxels can emit a zero crossing (tsdf_volume.cu:548-633), so extraction may skip every other stretch of the volume and still
 * return exactly the full scan's points.  The caller zeroes the map whenever it clears the volume and must route EVERY
 * integration of that volume through df_integrate_tracked. */
#define DF_ACTIVITY_VOXELS 1024
/* Second part of the same allocation (behind the per-stretch bytes, see df_volume_activity_bytes): a BRICK table, one byte per
 * DF_BRICK x DF_BRICK x DF_BRICK block of voxels (brick (bx, by, bz) at ((bz * nby) + by) * nbx + bx, n* = ceil(dims / DF_BRICK)), non-zero iff an
 * integration stored a voxel with F < 0 there since the map was last zeroed.  The ray-cast's march only ever acts on a sample pair that
 * contains a negative value (tsdf_volume.cu:311-336: (-,+) stops the ray, (+,-) is the surface), so df_raycast_points_tracked replays the
 * march's float chain without fetching from bricks that hold no negative voxel and returns exactly the dense march's maps.  The volume
 * itself stays the reference's dense array (TsdfVolume::data()/swap() are part of its API): sparse traversal, not sparse storage. */
#define DF_BRICK 8
size_t df_volume_activity_bytes(df_volume vol);
/* workspace (optional, device memory, df_integrate_workspace_bytes(cols, rows) bytes): per-tile maximum ray length of the frame,
 * used to skip the parts of the volume that lie behind the observed surface; NULL = allocated stream-ordered per call. */
size_t df_integrate_workspace_bytes(int cols, int rows);
int df_integrate_launch_count(df_volume vol);   /* kernels one integrate call launches for this volume (bookkeeping for gpu_launches) */
int df_integrate_last_kernel(void);             /* diagnostic: which integrate kernel the last call of this process launched (5 = packed-arithmetic kernel, 3 / 4 = scalar culling kernels, 0 = plain) */
int df_integrate_selftest(unsigned long long *mismatch_dev4, void *stream);   /* test hook: the packed integrate kernel's division / square-root sequences against the '/' operator and sqrtf() on this device; 4 mismatch counters (all 0 on a conforming device) */
int df_integrate_tracked(df_volume vol, const uint16_t *dists, size_t dists_pitch, int cols, int rows,
                         df_aff3f vol2cam, df_intr intr, unsigned long long *n_updated, unsigned char *activity, void *workspace,
                         void *stream);

/* device::raycast, points variant (internal.hpp:113-114, tsdf_volume.cu:341-405,459-474).
 * cam2vol = volume_pose^-1 * camera_pose, Rinv = cam2vol.R^-1 (tsdf_volume.cpp:157-174). */
int df_raycast_points(df_volume vol, df_aff3f cam2vol, const float *Rinv_host9, df_intr intr, int cols, int rows,
                      float step_factor, float delta_factor,
                      float *points, size_t points_pitch, float *normals, size_t normals_pitch, void *stream);

/* same maps, bit for bit; the march skips the bricks that hold no negative voxel (activity: the volume's activity map, maintained by
 * df_integrate_tracked / df_integrate_warped -- NULL falls back to df_raycast_points) */
int df_raycast_points_tracked(df_volume vol, df_aff3f cam2vol, const float *Rinv_host9, df_intr intr, int cols, int rows,
                              float step_factor, float delta_factor, float *points, size_t points_pitch, float *normals, size_t normals_pitch,
                              const unsigned char *activity, void *stream);

/* Measurement variant of df_raycast_points (bench.py's ray-cast roofline; never on the frame path): the same kernel instantiated with
 * counters.  touched: df_raycast_touched_bytes(vol) bytes, zeroed by the caller, one bit per voxel the launch reads (its popcount is U of
 * SURVEY.md 8d: algorithmic bytes = 4*U + 32*cols*rows); stats (device, 2 x u64, zeroed by the caller): [0] rays that produced a vertex,
 * [1] march samples fetched after the entry sample. */
size_t df_raycast_touched_bytes(df_volume vol);
int df_raycast_points_stats(df_volume vol, df_aff3f cam2vol, const float *Rinv_host9, df_intr intr, int cols, int rows,
                            float step_factor, float delta_factor, float *points, size_t points_pitch,
                            float *normals, size_t normals_pitch, unsigned int *touched, unsigned long long *stats, void *stream);

/* the counting instantiation of df_raycast_points_tracked (activity != NULL: [1] counts the march samples EXAMINED; only those in
 * negative bricks are fetched and appear in `touched`) */
int df_raycast_points_stats_tracked(df_volume vol, df_aff3f cam2vol, const float *Rinv_host9, df_intr intr, int cols, int rows,
                                    float step_factor, float delta_factor, float *points, size_t points_pitch,
                                    float *normals, size_t normals_pitch, unsigned int *touched, unsigned long long *stats,
                                    const unsigned char *activity, void *stream);

/* device::project_and_remove (internal.hpp:108-109, tsdf_volume.cu:114-137,164-177): `dists` is sampled as fp16 and
 * the pixels the vertices land on are zeroed; vertices become (u*Dp, v*Dp, Dp, 0) or NaN when off-image.
 * Deterministic (the reference races the scatter with the sampling): samples always see the original image.
 * workspace: df_project_workspace_bytes(cols, rows) bytes, zero on entry, returned zeroed. */
size_t df_project_workspace_bytes(int cols, int rows);
int df_project_and_remove(uint16_t *dists, size_t dists_pitch, int cols, int rows, df_intr intr,
                          float *points, size_t points_pitch, int pcols, int prows, void *workspace, void *stream);

/* device::extractCloud (internal.hpp:138, tsdf_volume.cu:486-710,799-815).  Deterministic: points are emitted in
 * ascending (z, y, x) voxel order, +x,+y,+z edge within a voxel.  `workspace` needs df_extract_workspace_bytes();
 * the point count (clamped to capacity) is written to *count (device, int32) -- no host sync. */
size_t df_extract_workspace_bytes(df_volume vol);
int df_extract_cloud(df_volume vol, df_aff3f pose, float *out_points, int capacity, int *count,
                     void *workspace, void *stream);
/* same, skipping the stretches of the volume whose activity byte is zero (activity == NULL: full scan) */
int df_extract_cloud_tracked(df_volume vol, df_aff3f pose, float *out_points, int capacity, int *count, void *workspace,
                             const unsigned char *activity, void *stream);

/* device::extractNormals (internal.hpp:139, tsdf_volume.cu:714-795,817-831).  n_points may be given on the host
 * (count_dev == NULL) or read from device memory (count_dev != NULL, upper bound n_points). */
int df_extract_normals(df_volume vol, const float *points, int n_points, const int *count_dev, df_aff3f pose,
                       const float *Rinv_host9, float delta_factor, float *out_normals, void *stream);

/* Triangle mesh of the volume's zero level set (marching cubes; not in the reference, whose next steps ask for a .ply / .obj export,
 * Report.md:57).  Definition -- in the volume's own conventions, so that it agrees with the cloud:
 *   a voxel is ACTIVE iff W != 0 && F != 1 (as for the cloud); a corner is INSIDE iff F < 0 (-0 is not inside);
 *   cell (x, y, z), x < Dx-1, y < Dy-1, z < Dz-1, has the 8 corners (x+i, y+j, z+k); it is MESHED iff all 8 are active and its inside
 *   mask is neither 0 nor 255;
 *   one VERTEX per voxel edge (v, axis) (axis 0/1/2 = +x/+y/+z) whose endpoints differ in the inside test and which borders at least one
 *   meshed cell; its edge key is 3*v + axis (v = linear voxel index; fits in 32 bits up to 1024^3 voxels); vertices come out in
 *   ascending key order; the position is the cloud's interpolation of that edge, posed by `pose` -- the same device code, so a vertex on an
 *   edge the cloud also emits (strict sign change, both endpoints active) is bit-identical to that cloud point;
 *   TRIANGLES (int32[3] indices into the vertices): every meshed cell in ascending cell index emits the triangles of its case in the order
 *   of the generated table (csrc/mc_table.h, tools/gen_mc_table.py), counter-clockwise seen from the outside (F > 0), so the face normal
 *   points along the TSDF gradient as df_extract_normals does.  Each cube face is decided from its own four signs (an ambiguous face
 *   separates its inside corners), so neighbouring cells agree and the mesh has no cracks.
 * Deterministic (no atomics decide order or content).  Every crossing edge's lower endpoint and every meshed cell's min corner is active,
 * so the activity map (as df_extract_cloud_tracked; NULL = full scan) returns exactly the full scan's mesh.  Vertices are found by binary
 * search of their keys -- no per-voxel index array.
 * counts_dev (device, 2 x int32): [0] vertices, [1] triangles -- the TRUE totals, never clamped.  Vertices beyond vcap and triangles
 * beyond tcap are not written; if the vertices overflow, no triangle is written (their indices would be unresolvable).
 * workspace: df_extract_mesh_workspace_bytes() bytes. */
size_t df_extract_mesh_workspace_bytes(df_volume vol);
int df_extract_mesh(df_volume vol, df_aff3f pose, const unsigned char *activity,
                    float *vertices /* float4, w = 0 */, uint32_t *edge_keys, int vcap,
                    int32_t *triangles /* [tcap][3] */, int tcap, int *counts_dev, void *workspace, void *stream);

/* ------------------------------------------------------------------ image processing ----------------------------------------------------- */
/* device::bilateralFilter (internal.hpp:125, imgproc.cu:11-57) */
int df_bilateral(const uint16_t *src, size_t src_pitch, int cols, int rows, uint16_t *dst, size_t dst_pitch,
                 int kernel_size, float sigma_spatial, float sigma_depth, void *stream);
/* device::truncateDepth (internal.hpp:124, imgproc.cu:66-85) */
int df_truncate_depth(uint16_t *depth, size_t pitch, int cols, int rows, float max_dist, void *stream);
/* device::depthPyr (internal.hpp:126, imgproc.cu:94-136): dst is (src_cols/2, src_rows/2) */
int df_pyr_down(const uint16_t *src, size_t src_pitch, int src_cols, int src_rows, uint16_t *dst, size_t dst_pitch,
                float sigma_depth, void *stream);
/* device::computePointNormals (internal.hpp:132, imgproc.cu:210-250) */
int df_points_normals(df_intr intr, const uint16_t *depth, size_t depth_pitch, int cols, int rows,
                      float *points, size_t points_pitch, float *normals, size_t normals_pitch, void *stream);
/* device::resizePointsNormals (internal.hpp:129, imgproc.cu:368-414): dst is (src_cols/2, src_rows/2) */
int df_resize_points_normals(const float *vsrc, size_t vsrc_pitch, const float *nsrc, size_t nsrc_pitch,
                             int src_cols, int src_rows, float *vdst, size_t vdst_pitch, float *ndst, size_t ndst_pitch,
                             void *stream);

/* device::renderImage points variant / renderTangentColors (internal.hpp:134-136, imgproc.cu:484-583): display only, BGRA out */
int df_render_image(const float *points, size_t points_pitch, const float *normals, size_t normals_pitch, int cols, int rows,
                    const float *light_pose_host3, void *image_bgra, size_t image_pitch, void *stream);
int df_render_tangent_colors(const float *normals, size_t normals_pitch, int cols, int rows, void *image_bgra, size_t image_pitch,
                             void *stream);

/* The reference's USE_DEPTH-path image operations (cuda/imgproc.hpp:15,21,23,31; imgproc.cu:145-200,277-303,307-366,420-537).  The
 * default build of the reference does not take this path; they exist so that every function of its public header is served. */
int df_render_image_depth(const uint16_t *depth, size_t depth_pitch, const float *normals, size_t normals_pitch, int cols, int rows,
                          df_intr intr, const float *light_pose_host3, void *image_bgra, size_t image_pitch, void *stream);
int df_normals_mask_depth(df_intr intr, uint16_t *depth, size_t depth_pitch, int cols, int rows, float *normals, size_t normals_pitch, void *stream);
int df_cloud_to_depth(const float *cloud, size_t cloud_pitch, int cols, int rows, uint16_t *depth, size_t depth_pitch, void *stream);
int df_resize_depth_normals(const uint16_t *dsrc, size_t dsrc_pitch, const float *nsrc, size_t nsrc_pitch, int src_cols, int src_rows,
                            uint16_t *ddst, size_t ddst_pitch, float *ndst, size_t ndst_pitch, void *stream);

/* ------------------------------------------------------------------ projective ICP -------------------------------------------------------- */
/* ComputeIcpHelper::operator() points variant (internal.hpp:67-102, proj_icp.cu:80-108,350-394,448-467): one
 * data-association + 27-term reduction pass at one pyramid level.  scratch: 16-byte aligned device buffer of
 * DF_ICP_SCRATCH_DOUBLES doubles; on completion scratch[0..26] hold the 27 sums, order (i, j>=i) for i = 0..5, j = 0..6 (the rest holds the
 * per-block partials, summed in a fixed order: results are run-to-run deterministic).  intr_level are the level's
 * intrinsics (setLevelIntr, projective_icp.cpp:17-23). */
#define DF_ICP_SCRATCH_DOUBLES (32 + 27 * 1024)
int df_icp_accumulate(const float *vcurr, size_t vcurr_pitch, const float *ncurr, size_t ncurr_pitch,
                      const float *vprev, size_t vprev_pitch, const float *nprev, size_t nprev_pitch,
                      int cols, int rows, df_intr intr_level, df_aff3f T, float dist2_thres, float min_cosine,
                      double *scratch, void *stream);

/* ProjectiveICP::estimateTransform, points variant (projective_icp.hpp:39, projective_icp.cpp:169-213) executed
 * entirely on the device: per iteration the association/reduction kernel, then the 6x6 solve + Rodrigues update in a
 * one-thread tail (replaces StreamHelper::get + cv::solve + 19 host round trips).  Arrays of `levels` entries, index 0 =
 * finest.  T_dev (device, 12 floats: R row-major + t) receives curr->prev; ok_dev (device int) is 0 when the
 * reference would have returned false (|det| < 1e-15 or NaN). */
int df_icp_estimate(const float *const *vcurr, const float *const *ncurr, const float *const *vprev, const float *const *nprev,
                    const int *cols, const int *rows, const size_t *pitch, int levels, const int *iters,
                    df_intr intr, float dist_thres, float angle_thres, float *T_dev, int *ok_dev, double *scratch,
                    void *stream);

/* The reference's compile-time USE_DEPTH alternative (internal.hpp:6; ComputeIcpHelper::find_coresp proj_icp.cu:47-78,
 * ComputeIcpHelper::operator()(const Depth&, ...) proj_icp.cu:396-418): the current depth map (u16 millimetres) is
 * re-projected per pixel, the previous depth map is point-sampled at the projection and re-projected at the fractional
 * coordinates; normal maps as above.  Same scratch / sums layout as df_icp_accumulate. */
int df_icp_accumulate_depth(const unsigned short *dcurr, size_t dcurr_pitch, const float *ncurr, size_t ncurr_pitch,
                            const unsigned short *dprev, size_t dprev_pitch, const float *nprev, size_t nprev_pitch,
                            int cols, int rows, df_intr intr_level, df_aff3f T, float dist2_thres, float min_cosine,
                            double *scratch, void *stream);

/* ProjectiveICP::estimateTransform, depth-pyramid overload (projective_icp.hpp:38, projective_icp.cpp:126-167), device
 * resident like df_icp_estimate. */
int df_icp_estimate_depth(const unsigned short *const *dcurr, const float *const *ncurr, const unsigned short *const *dprev,
                          const float *const *nprev, const int *cols, const int *rows, const size_t *depth_pitch,
                          const size_t *normals_pitch, int levels, const int *iters, df_intr intr, float dist_thres,
                          float angle_thres, float *T_dev, int *ok_dev, double *scratch, void *stream);

/* ------------------------------------------------------------------ warp field ------------------------------------------------------------ */
/* deformation_node (warp_field.hpp:35-40) as 12 floats: vertex[3], rotation quat (w,x,y,z), dual/translation quat
 * (w,x,y,z) = 0.5*t*r (dual_quaternion.hpp:59-63), weight. */
#define DF_NODE_STRIDE 12
#define DF_KNN 8                          /* KNN_NEIGHBOURS, warp_field.hpp:10 */

/* WarpField::KNN (warp_field.hpp:66, warp_field.cpp:247-251) for N queries: exact 8-NN, ascending squared distance,
 * ties -> lower node index; idx = -1 / d2 = FLT_MAX for NaN queries or when M < 8.  qstride in floats. */
int df_knn8(const float *nodes, int M, const void *node_grid, const float *queries, int N, int qstride, int32_t *idx, float *d2,
            void *stream);

/* WarpField::buildKDTree (warp_field.hpp:84, warp_field.cpp:275-282): uniform grid over the node vertices that replaces the
 * nanoflann index.  Optional everywhere (`node_grid` = NULL -> exhaustive shared-memory scan); results are identical either
 * way (candidates ranked by (distance, index)).  Build once per node set: vertices do not move after WarpField::init. */
size_t df_node_grid_bytes(int M);
int df_build_node_grid(const float *nodes, int M, void *node_grid, void *stream);

/* Extending the warp field (SURVEY.md 8f(3); Report.md "4. Extending the warp field - stubbed out functionality"): nodes are appended for
 * the points of the extracted canonical cloud that the field does not support.  A point is unsupported when its nearest node (of the M
 * nodes present on entry) is farther than `radius`; every step-th unsupported point, in cloud order (the subsampling rule of
 * WarpField::init, warp_field.cpp:49-60), becomes a node as init makes them (identity DualQuaternion(), weight 3, :68-80), appended to
 * `nodes` (capacity max_nodes) until it is full.  cloud: float[capacity][stride], count_dev (optional, device) = valid points;
 * M_out_dev (device int) receives the new node count -- rebuild the node grid (df_build_node_grid) when it differs from M.
 * workspace: df_extend_field_workspace_bytes(capacity) bytes. */
size_t df_extend_field_workspace_bytes(int capacity);
int df_extend_field(float *nodes, int M, int max_nodes, const void *node_grid, const float *cloud, int capacity, const int *count_dev,
                    int stride, float radius, int step, int *M_out_dev, void *workspace, void *stream);

/* WarpField::warp (warp_field.hpp:62, warp_field.cpp:180-195): k-NN + weights + DQB + transform of points and
 * normals in place (stride in floats, 3 or 4).  flags: bit0 = reference normal cursor (advance only on valid points),
 * bit1 = rotate normals only (extension).  idx_out / w_out (optional, N*8) receive the neighbours and weights. */
#define DF_WARP_REF_NORMAL_INDEX 1
#define DF_WARP_NORMAL_ROTATE_ONLY 2
#define DF_WARP_REUSE_KNN 4        /* idx_out / w_out are INPUTS: neighbours + weights of these points from an earlier pass */
/* flags bits 8..23: the points are an image of that many columns (N = cols * rows, cols % 32 == 0, rows % 8 == 0): a warp then takes an
 * 8 x 4 pixel patch, whose queries share one short candidate list in the 8-NN search.  Results do not depend on it. */
#define DF_WARP_IMAGE_COLS(c) (((c) & 0xffff) << 8)
int df_warp(const float *nodes, int M, const void *node_grid, float *points, float *normals, int N, int stride, df_aff3f warp_to_live,
            int flags, int32_t *idx_out, float *w_out, void *stream);

/* Per-voxel warped integration (SURVEY.md 8f(1)): the update TsdfVolume::surface_fusion (tsdf_volume.hpp:76-79,
 * tsdf_volume.cpp:228-254) was written towards and left commented out (:248-251) -- DynamicFusion eq. 4-5.  For every voxel:
 *   x_c = vol2world * (x*vs, y*vs, z*vs);  x_t = world2cam * DQB(8-NN of x_c).transform(x_c)   (WarpField::warp, warp_field.cpp:180-251)
 *   rho = depth_mm(floor v, floor u) * 0.001 - x_t.z                                            (TsdfVolume::psdf, tsdf_volume.cpp:266-292)
 *   if rho > -trunc:  tsdf = min(1, rho/trunc);  w = clamp(rint(weight_scale * mean node distance), 1, max_weight)  (TsdfVolume::weighting,
 *   :300-306; weight_scale <= 0 -> w = 1);  F' = (F*W + tsdf*w)/(W + w);  W' = min(W + w, max_weight).
 * depth: the frame's u16 millimetre image (not the ray lengths df_integrate takes); nodes / node_grid: the warp field (node_grid is
 * required).  counters (optional, device, 2 x u64): [0] += voxels written, [1] += voxels warped (k-NN + blend evaluated).
 * activity: as df_integrate_tracked.  workspace (optional, device): df_integrate_warped_workspace_bytes(cols, rows, M) bytes
 * (M = the largest node count it will be used with). */
size_t df_integrate_warped_workspace_bytes(int cols, int rows, int M);
int df_integrate_warped_launch_count(void);
int df_integrate_warped(df_volume vol, const uint16_t *depth, size_t depth_pitch, int cols, int rows, df_aff3f vol2world,
                        df_aff3f world2cam, df_intr intr, const float *nodes, int M, const void *node_grid, float weight_scale,
                        unsigned long long *counters, unsigned char *activity, void *workspace, void *stream);

/* WarpFieldOptimiser::optimiseWarpData (warp_field_optimiser.hpp:14-17) -> CombinedSolver (CombinedSolver.h:25-110)
 * -> Opt LM/PCG on kfusion/solvers/dynamicfusion.t: translation-only data term solved on the device; node
 * translations are updated in place (encodeTranslation, CombinedSolver.h:189-197).
 * params: nonlinear (LM) iterations, linear (PCG) iterations; stats_dev (device, 8 doubles): initial cost, final cost,
 * LM iterations run, valid rows, PCG iterations run, row-overflow flag, [6] non-zeros of the normal matrix, [7] diagnostics (>= 0: solved
 * by the one-exchange cluster kernel, value = halo columns exchanged per PCG step; < 0: by its fallback; fraction .5: matrix assembled from tile records).  If a node's row of the normal matrix couples to more columns
 * than the kernels store (512), the flag is raised and the solve leaves the node translations UNCHANGED (0 LM iterations) rather than
 * solving a truncated, asymmetric system; callers must look at stats[5] (the frame loop reports it through df_kinfu_get_info[11] and on
 * stderr, the C++ mirror prints an error).  workspace from df_solve_workspace_bytes(M, N).
 * Rows with a NaN in canon or live are skipped (the reference zero-fills them with stale k-NN scratch). */
size_t df_solve_workspace_bytes(int M, int N);
/* after df_solve_data_term: the per-vertex neighbour indices (N*8, -1 for skipped rows) and weights (N*8) it computed for
 * `canon`, inside `workspace` -- valid until the workspace is reused; lets the following warp of the same vertices skip its
 * k-NN pass (DF_WARP_REUSE_KNN) */
int df_solve_knn_buffers(void *workspace, int M, int N, int32_t **idx, float **w);
#define DF_SOLVE_REF_GRAPH_QUIRK 1
/* flags bits 8..23: the vertices are an image of that many columns (N = cols * rows, row-major, cols % 16 == 0, rows % 8 == 0): lets the
 * assembly of the normal matrix work tile by tile (16 x 8 pixels share a dozen nodes) instead of entry by entry.  Same result up to the
 * order of the double sums; 0 (a flat vertex list) always takes the per-entry path. */
#define DF_SOLVE_IMAGE_COLS(c) (((c) & 0xffff) << 8)
int df_solve_data_term(float *nodes, int M, const void *node_grid, const float *canon, const float *live, int N, int stride,
                       int nonlinear_iters, int linear_iters, int flags, double *stats_dev, void *workspace, void *stream);

/* SURVEY.md 8f(2), OPT-IN beside df_solve_data_term: the robust data term over 6-DoF node increments plus the regularisation term -- the
 * energy the reference defines piecewise and never assembles (6-wide parameter blocks optimisation.hpp:108-110,141-143; tukeyPenalty :84-88,
 * dynamicfusion.t:43-51; huberPenalty optimisation.hpp:134-138, dynamicfusion.t:34-40; empty DynamicFusionRegEnergy :125-132 /
 * WarpField::energy_reg warp_field.cpp:168-172; KinFu::edges_ kinfu.hpp:95).  PARITY UNPINNED (no reference code evaluates it); restated in
 * oracle/orc_reg.c, solved in csrc/regsolve.cu:
 *   E = sum_v sum_c rho_T(live_v - warp(canon_v))_c  +  reg_lambda sum_(i,j) max(weight_i, weight_j) sum_c rho_H(T_i(g_j) - T_j(g_j))_c
 * warp = WarpField::DQB + transform over the 8 nearest nodes; T_k(p) = rotate(q_k, p) + t_k; j runs over the reg_k (<= 7) nearest other nodes
 * of node i; rho_T' = tukeyPenalty(., tukey_c) (DF_F2_TUKEY, else squared loss); rho_H = huberPenalty(., huber_delta) (DF_F2_HUBER, else
 * squared loss).  Unknowns per node: (omega, tau), q <- exp(omega) q, t <- t + tau (DF_F2_TWIST; without it omega = 0: translation-only).
 * Gauss-Newton / IRLS, gn_iters steps, each solved by block-Jacobi PCG (at most lin_iters steps) with Levenberg damping lm_mu * diag(H).
 * Nodes are updated in place (rotation + dual part).  stats_dev (device, 16 doubles): [0] energy before, [1] energy after, [2] GN steps,
 * [3] valid vertices, [4] data energy after, [5] regularisation energy after, [6] edge slots, [7] PCG steps in total, [8 + i] energy before
 * GN step i (i < 8).  workspace: df_solve_f2_workspace_bytes(M, N, reg_k). */
typedef struct df_f2_params {
    double reg_lambda, tukey_c, huber_delta, lm_mu;   /* 0 = no regulariser, 0.01, 1e-4 (the reference's defaults for c and delta), 1e-4 */
    int gn_iters, reg_k, flags, lin_iters;
} df_f2_params;
#define DF_F2_TWIST 1
#define DF_F2_TUKEY 2
#define DF_F2_HUBER 4
size_t df_solve_f2_workspace_bytes(int M, int N, int reg_k);
int df_solve_f2(float *nodes, int M, const void *node_grid, const float *canon, const float *live, int N, int stride,
                const df_f2_params *params, double *stats_dev, void *workspace, void *stream);

/* ------------------------------------------------------------------ per-frame pipeline ----------------------------------------------------- */
/* kfusion::KinFuParams (kinfu.hpp:15-47) as a POD, plus the solver settings KinFu::KinFu hard-codes (kinfu.cpp:114-120)
 * and the knobs of the GPU-resident warp field. */
typedef struct df_kinfu_params {
    int cols, rows;
    df_intr intr;
    int volume_dims[3];
    float volume_size[3];
    df_aff3f volume_pose;
    float bilateral_sigma_depth, bilateral_sigma_spatial;
    int bilateral_kernel_size;
    float icp_truncate_depth_dist, icp_dist_thres, icp_angle_thres;
    int icp_iter_num[4];
    float tsdf_min_camera_movement, tsdf_trunc_dist;
    int tsdf_max_weight;
    float raycast_step_factor, gradient_delta_factor;
    float light_pose[3];
    int solver_nonlinear_iters, solver_linear_iters;   /* 5, 100 (kinfu.cpp:116-117) */
    int max_nodes;        /* cap on warp nodes; node_step grows to respect it */
    int node_step;        /* every node_step-th extracted point becomes a node: 50 (warp_field.cpp:49) */
    int cloud_capacity;   /* extracted-cloud buffer, points: 256^3 in the reference (tsdf_volume.cpp:184) */
    int flags;            /* DF_KINFU_* */
    float fusion_weight_scale;   /* DF_KINFU_WARPED_INTEGRATE: weight_scale of df_integrate_warped (0 = every sample weighs 1) */
    float extend_radius;         /* DF_KINFU_EXTEND_FIELD: support radius of df_extend_field in metres (<= 0: 0.03) */
} df_kinfu_params;

#define DF_KINFU_RIGID_ONLY 1      /* skip warp + solve (plain KinFu loop: config 1) */
#define DF_KINFU_STAGE_TIMING 2    /* record CUDA events per stage (df_kinfu_get_stage_ms) */
#define DF_KINFU_REF_GRAPH_QUIRK 4 /* forward DF_SOLVE_REF_GRAPH_QUIRK to the solve */
#define DF_KINFU_WARPED_INTEGRATE 8 /* SURVEY 8f(1): the fusion step of KinFu::dynamicfusion integrates the frame through the warp field, voxel by
                                      voxel (df_integrate_warped), instead of project_and_remove + the rigid integrate the reference falls back to
                                      (tsdf_volume.cpp:234-238).  Also switched on by the environment variable DF_KINFU_WARPED_INTEGRATE=1, so that an
                                      unchanged apps/demo.cpp can run it; DF_FUSION_WEIGHT_SCALE sets fusion_weight_scale the same way. */

#define DF_KINFU_F2_SOLVE 32       /* SURVEY 8f(2): the frame's warp solve is df_solve_f2 (robust 6-DoF data term + regulariser) instead of the reference's
                                      translation-only data term; parameters from df_kinfu_set_f2_params (defaults: lambda 5, reg_k 4, twist + Tukey(0.05) + Huber(1e-4),
                                      2 GN x 30 PCG steps).  Environment: DF_KINFU_F2_SOLVE=1. */
#define DF_KINFU_USE_DEPTH 64       /* the reference's compile-time USE_DEPTH frame loop (internal.hpp:6; kinfu.cpp:237-238,253-255,271,293-295): normals from the depth
                                      pyramid with masking (df_normals_mask_depth), ICP on depth pyramids (df_icp_estimate_depth), the model ray-cast stored as a depth map
                                      (df_cloud_to_depth) and halved by df_resize_depth_normals.  Environment: DF_KINFU_USE_DEPTH=1. */
#define DF_KINFU_EXTEND_FIELD 16    /* SURVEY 8f(3): after every extraction the warp field is extended (df_extend_field, radius = extend_radius, step = node_step,
                                      up to max_nodes) and the node grid rebuilt; costs one 4-byte read-back per frame.  Environment: DF_KINFU_EXTEND_FIELD=1,
                                      DF_EXTEND_RADIUS. */

/* which = 0: KinFuParams::default_params_dynamicfusion (kinfu.cpp:14-49); 1: default_params (kinfu.cpp:55-89) */
void df_kinfu_default_params(df_kinfu_params *p, int which);
/* KinFu::KinFu (kinfu.cpp:95-125): allocates volume, pyramids, ICP and warp/solver state on the current device */
void *df_kinfu_create(const df_kinfu_params *p);
void df_kinfu_destroy(void *kinfu);
int df_kinfu_set_stream(void *kinfu, void *stream);
/* KinFu::reset (kinfu.cpp:196-207) */
int df_kinfu_reset(void *kinfu);
/* KinFu::operator()(depth) (kinfu.cpp:221-305).  Returns 1 = frame fused and ray-cast image available, 0 = first frame or
 * tracking reset (the reference's `false`), < 0 = -(cudaError).  _host: depth is a HOST u16 image (any pitch), copied to
 * the device inside the call (the path apps/demo.cpp takes: imread -> upload -> operator()); _device: depth already in HBM. */
int df_kinfu_process_host(void *kinfu, const uint16_t *depth_host, size_t pitch);
int df_kinfu_process_device(void *kinfu, const uint16_t *depth_dev, size_t pitch);
/* Multi-device host entry (config 5: independent sequences batched across the GPUs of one box).  A KinFu object belongs to the CUDA device
 * that was current when it was created (cudaSetDevice(i) before df_kinfu_create) and every df_kinfu_* call switches to it.  This call
 * advances n objects by one frame each CONCURRENTLY -- one host thread per object, because a frame contains one host synchronisation --
 * and returns 0 or the most negative status; results[i] = what df_kinfu_process_host returns for object i. */
int df_kinfu_batch_process_host(void *const *kinfus, const uint16_t *const *depth_host, const size_t *pitch, int n, int *results);
/* KinFu::dynamicfusion(depth, live_frame, current_normals) (kinfu.hpp:87, kinfu.cpp:344-400) on caller-provided device buffers,
 * at the latest pose: raycast -> warp -> solve -> warp -> project/remove -> integrate -> extract.  depth is modified in place. */
int df_kinfu_dynamicfusion(void *kinfu, uint16_t *depth_dev, size_t depth_pitch, const float *live_points_dev, size_t live_pitch);
/* The surface extraction of a frame (compute_points / compute_normals, kinfu.cpp:398-399) runs on an auxiliary stream of the object and
 * overlaps the frame's last ray-cast and the next frame's pre-processing + ICP: nothing later in the loop reads the cloud, and the volume it
 * reads is not written before the next integrate (which waits for it).  Every accessor of the cloud (df_kinfu_get_info, _read_buffer,
 * _get_buffer(9|10), _state_digest) waits for it; df_kinfu_join makes the object's MAIN stream wait for it without a host synchronisation
 * (what a caller timing frames with events on that stream wants).  DF_KINFU_OVERLAP_EXTRACT=0 (environment) keeps everything on one stream. */
int df_kinfu_join(void *kinfu);
/* KinFu::getCameraPose(time) (kinfu.cpp:213-218): 12 floats, R row-major then t; time < 0 = latest */
int df_kinfu_get_pose(void *kinfu, int time, float *pose12_host);
/* info[0] frame counter, [1] warp nodes M, [2] extracted cloud points, [3] poses stored, [4] last ICP ok,
 * [5] kernels launched in the last frame, [6] resets so far, [7] solver LM iterations (last frame),
 * [8] voxels written by the last integrate (DF_KINFU_STAGE_TIMING only), [9] solver PCG iterations (last frame),
 * [10] voxels carried through the warp field by the last df_integrate_warped (DF_KINFU_WARPED_INTEGRATE + STAGE_TIMING),
 * [11] frames whose warp solve was skipped because a normal-matrix row overflowed (df_solve_data_term: stats[5]); also reported on stderr */
int df_kinfu_get_info(void *kinfu, long long *info_host, int n);
/* device buffers of the current state: 0 volume(u32), 1 dists, 2 curr depth L0, 3 curr points L0, 4 curr normals L0,
 * 5 prev points L0, 6 prev normals L0, 7 canonical (after 2nd warp), 8 canonical normals, 9 extracted cloud,
 * 10 extracted normals, 11 nodes, 12 canonical_visible, 13 solver stats (8 doubles), 14 activity map (bytes) */
int df_kinfu_get_buffer(void *kinfu, int which, void **ptr, size_t *pitch, int *cols, int *rows);
/* synchronous device-to-host copy of one of those buffers (diagnostics / tests), at most `bytes` bytes */
int df_kinfu_read_buffer(void *kinfu, int which, void *dst_host, size_t bytes);
/* Lock-step parity hook (tests; never used by the frame loop's callers): one-shot replacements for the NEXT df_kinfu_process_* call.
 * Each non-NULL argument replaces the corresponding intermediate result of that frame, so that everything downstream can be compared
 * with a CPU run of the same frame BIT FOR BIT instead of statistically:
 *   bilateral_depth_host  cols x rows u16: used instead of this frame's bilateral filter output (CUDA expf vs glibc expf: +-1 LSB);
 *   pose12_host           absolute camera pose of the frame (R row-major, t): used instead of poses.back() * ICP(affine); ICP is skipped;
 *   nodes_host            M x DF_NODE_STRIDE floats: the node table after the data-term solve (ignored unless M equals the loop's node count).
 * NULL = compute as usual. */
int df_kinfu_set_overrides(void *kinfu, const uint16_t *bilateral_depth_host, size_t pitch, const float *pose12_host, const float *nodes_host, int M);
/* parameters of the DF_KINFU_F2_SOLVE variant of the frame loop */
int df_kinfu_set_f2_params(void *kinfu, const df_f2_params *params);
/* digest of the current state (multi-GPU correctness record, SURVEY 8e: ranks exchange it and rank 0 compares every rank's with a
 * single-GPU run of the same sequence): out4_host[0] order-independent 64-bit checksum of the packed volume, [1] the same over the node
 * table, [2] extracted cloud points, [3] FNV-style hash of every camera pose so far (bit patterns).  Synchronous. */
int df_kinfu_state_digest(void *kinfu, unsigned long long *out4_host);
/* per-stage milliseconds of the last frame (DF_KINFU_STAGE_TIMING): preprocess, icp, raycast_canonical, warp1, solve,
 * warp2, project_remove, integrate, extract, raycast_prev; returns the number written */
int df_kinfu_get_stage_ms(void *kinfu, float *ms_host, int n);

/* The frame loop's current model as a mesh (df_extract_mesh of its volume at the volume pose, through its activity map), on the object's
 * stream, ordered after its last integrate.  Synchronous; counts_host[2] as df_extract_mesh's counts.  normals (optional, float4):
 * df_extract_normals at the vertices.  DF_MESH_LIVE: vertices (and normals, rotation only) are carried through the current warp field by
 * df_warp with warp_to_live = identity, as the loop warps its canonical points -- a vertex whose normal is NaN (within two voxels of the
 * volume's border) stays where it is, as df_warp leaves such points; an object without warp nodes (rigid-only, or before the field exists)
 * returns cudaErrorInvalidValue.  Runs on demand, never inside df_kinfu_process_*: the object's state (volume, cloud, nodes, poses, the
 * pending extraction on its auxiliary stream) is left exactly as it was.  The workspace is allocated on first use, not at create. */
#define DF_MESH_LIVE 1
int df_kinfu_extract_mesh(void *kinfu, int flags, float *vertices, float *normals, uint32_t *edge_keys, int vcap,
                          int32_t *triangles, int tcap, int *counts_host);

#ifdef __cplusplus
}
#endif
#endif /* DFUSION_H */
