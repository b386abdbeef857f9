// pipeline.cu -- the per-frame DynamicFusion loop, device-resident, behind the C ABI (df_kinfu_*).
// Mirrors kfusion::KinFu (kfusion/include/kfusion/kinfu.hpp:49-97, kfusion/src/kinfu.cpp): same stage order, buffer swaps,
// first-frame special case and pose chaining.  What changes is where the data lives: the reference's
// KinFu::dynamicfusion (kinfu.cpp:344-400) downloads three 4.9 MB maps, runs ~1 M CPU k-NN queries, re-uploads, and
// syncs ~25 times a frame; here the frame touches the host exactly once (ICP status + 12-float pose, needed for the
// return value) and everything else is stream-ordered kernels on one stream.
#include "df_common.cuh"
#include "../../include/df_hostmath.h"
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include <chrono>
#include <thread>

using namespace dfb;

namespace {

constexpr int MAX_LEVELS = 4;      // ProjectiveICP::MAX_PYRAMID_LEVELS, projective_icp.hpp:12
constexpr int NSTAGES = 10;

struct Img { void *ptr = nullptr; size_t pitch = 0; int cols = 0, rows = 0; };

struct KinFu {
    df_kinfu_params p;
    int device = 0;                       // the CUDA device the object was created on; every entry point switches to it
    cudaStream_t stream = 0;
    int levels = 0;                       // icp used levels
    float trunc_dist = 0.f;
    float voxel_size[3];
    uint32_t *volume = nullptr;
    Img depth_in, dists;
    Img cur_depth[MAX_LEVELS], cur_pts[MAX_LEVELS], cur_nrm[MAX_LEVELS], prev_pts[MAX_LEVELS], prev_nrm[MAX_LEVELS];
    Img prev_depth[MAX_LEVELS];           // DF_KINFU_USE_DEPTH only: the model's depth pyramid (prev_.depth_pyr)
    Img canon, canon_nrm, canon_visible;
    float *cloud = nullptr, *cloud_nrm = nullptr; int *cloud_count = nullptr;
    float *nodes = nullptr; int M = 0; void *node_grid = nullptr;
    float *icp_T = nullptr; int *icp_ok = nullptr; double *icp_scratch = nullptr;
    void *solve_ws = nullptr; size_t solve_ws_bytes = 0; double *solve_stats = nullptr;
    double *f2_stats = nullptr;
    void *extract_ws = nullptr; void *project_ws = nullptr;
    void *integrate_ws = nullptr;
    void *extend_ws = nullptr; int *M_dev = nullptr;   // df_extend_field workspace / new node count (DF_KINFU_EXTEND_FIELD)
    void *fusion_ws = nullptr;             // df_integrate_warped workspace (DF_KINFU_WARPED_INTEGRATE)
    void *mesh_ws = nullptr; size_t mesh_ws_bytes = 0;   // df_kinfu_extract_mesh: workspace, counts, scratch normals (allocated on first use)
    unsigned char *activity = nullptr; size_t activity_bytes = 0;   // dfusion.h DF_ACTIVITY_VOXELS: which stretches of the volume hold surface
    float *pinned = nullptr;             // 16 floats: T(12) + ok
    std::vector<float> poses;            // 12 floats per pose
    int frame_counter = 0, resets = 0, last_ok = 1, launches = 0;
    // df_kinfu_set_overrides (lock-step parity hook): one-shot replacements for the NEXT frame
    std::vector<uint16_t> ov_depth; bool has_ov_depth = false;       // bilateral-filtered depth, dense cols x rows
    float ov_pose[12]; bool has_ov_pose = false;                     // absolute camera pose of the frame
    std::vector<float> ov_nodes; bool has_ov_nodes = false;          // node table after the solve
    df_f2_params f2; void *f2_ws = nullptr;      // DF_KINFU_F2_SOLVE (SURVEY 8f(2))
    bool raycast_bricks = true;          // DF_RAYCAST_BRICKS=0: dense march (A/B)
    long long solve_overflows = 0;       // frames whose solve was skipped because a normal-matrix row overflowed (solve.cu ROWCAP); info[11]
    long long last_cloud = -1;
    double host_us[4] = {0, 0, 0, 0}; long long host_frames = 0;   // DF_KINFU_HOSTPROF: launch A, ICP wait, launch B, total
    unsigned long long *n_upd = nullptr;   // voxels written by the last integrate (filled when DF_KINFU_STAGE_TIMING)
    // Extraction runs on a second stream: nothing later in the frame loop reads the extracted cloud (the reference recomputes it every
    // frame for its host copies, kinfu.cpp:398-399), it only READS the volume, and the volume is not written again before the next
    // frame's integrate -- so it overlaps the ray-cast and the next frame's pre-processing + ICP (0.3 ms of mostly launch latency).
    cudaStream_t aux = nullptr;           // extraction stream (non-blocking, lowest priority: the main stream's kernels are placed first)
    cudaEvent_t ev_volume_ready = nullptr, ev_extract_done = nullptr, ev_before_lm = nullptr;
    bool extract_deferred = false;        // frame t's extraction has not been launched yet: it starts when frame t+1's LM/PCG kernel does
                                          // (one 16-SM cluster for ~1 ms, 132 SMs idle), or as soon as anybody needs the cloud or the volume
    bool extract_pending = false;         // an extraction is in flight on `aux`
    bool overlap_extract = true;          // DF_KINFU_OVERLAP_EXTRACT=0: everything on one stream
    cudaEvent_t ev[NSTAGES + 1];
    float stage_ms[NSTAGES];
    int stage_mark[NSTAGES + 1];
};

#define CK(call)                                      \
    do {                                              \
        cudaError_t e__ = (call);                     \
        if (e__ != cudaSuccess) return -(int)e__;     \
    } while (0)
#define CKD(call)                                     \
    do {                                              \
        int s__ = (call);                             \
        if (s__ != 0) return -s__;                    \
    } while (0)

int alloc_img(Img &im, int rows, int cols, size_t elem)
{
    im.cols = cols; im.rows = rows; im.pitch = (size_t)cols * elem;     // dense rows (pitch is still carried everywhere)
    return (int)cudaMalloc(&im.ptr, im.pitch * rows);
}

df_volume vol_of(const KinFu &k)
{
    df_volume v;
    v.data = k.volume;
    for (int i = 0; i < 3; ++i) { v.dims[i] = k.p.volume_dims[i]; v.voxel_size[i] = k.voxel_size[i]; }
    v.trunc_dist = k.trunc_dist; v.max_weight = k.p.tsdf_max_weight;
    return v;
}

df_aff3f to_aff(const float *a12) { df_aff3f a; memcpy(a.R, a12, 36); memcpy(a.t, a12 + 9, 12); return a; }

// canonical[i] = inverse_pose * cloud[i]: cv::Affine3f * Vec3f, m0*x + m1*y + m2*z + m3 left to right (kinfu.cpp:356-362);
// NaN pixels stay NaN.  Also writes the `canonical_visible` copy (kinfu.cpp:383).
__global__ void __launch_bounds__(256) to_canonical_kernel(const float4 *src, Aff inv_pose, float4 *dst, float4 *dst_copy, int n)
{
    DF_PDL_ENTRY();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 v = src[i];
    float4 o;
    o.x = inv_pose.r0.x * v.x + inv_pose.r0.y * v.y + inv_pose.r0.z * v.z + inv_pose.t.x;
    o.y = inv_pose.r1.x * v.x + inv_pose.r1.y * v.y + inv_pose.r1.z * v.z + inv_pose.t.y;
    o.z = inv_pose.r2.x * v.x + inv_pose.r2.y * v.y + inv_pose.r2.z * v.z + inv_pose.t.z;
    o.w = v.w;
    dst[i] = o;
    dst_copy[i] = o;
}

// WarpField::init (warp_field.cpp:41-62): every `step`-th extracted point becomes a node with the identity
// DualQuaternion() (rotation (1,0,0,0), dual part (1,0,0,0)) and weight 3 * voxel_size with voxel_size forced to 1.
__global__ void __launch_bounds__(256) init_nodes_kernel(const float4 *cloud, int step, int M, float *nodes)
{
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= M) return;
    const float4 p = cloud[(size_t)m * step];
    float *n = nodes + (size_t)m * DF_NODE_STRIDE;
    n[0] = p.x; n[1] = p.y; n[2] = p.z;
    n[3] = 1.f; n[4] = 0.f; n[5] = 0.f; n[6] = 0.f;
    n[7] = 1.f; n[8] = 0.f; n[9] = 0.f; n[10] = 0.f;
    n[11] = 3.f;
}

// order-independent 64-bit checksum of a u32 array: sum over i of mix(i, a[i]) (splitmix64 finaliser); one u64 atomicAdd per block
__global__ void __launch_bounds__(256) digest_kernel(const uint32_t *__restrict__ a, size_t n, unsigned long long *out)
{
    unsigned long long acc = 0ull;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        unsigned long long z = ((unsigned long long)a[i] << 32) ^ (unsigned long long)i;
        z += 0x9e3779b97f4a7c15ull;
        z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
        z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
        acc += z ^ (z >> 31);
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(out, acc);
}

df_volume vol_of(const KinFu &k);

// the extraction itself (compute_points + compute_normals, tsdf_volume.cpp:313-325) on stream `es`
int run_extract(KinFu &k, cudaStream_t es)
{
    const df_kinfu_params &p = k.p;
    float vol_pose[12], Rinv_vol[9];
    memcpy(vol_pose, p.volume_pose.R, 36); memcpy(vol_pose + 9, p.volume_pose.t, 12);
    dfh_mat3_inv(vol_pose, Rinv_vol);
    const df_volume vol = vol_of(k);
    int st = df_extract_cloud_tracked(vol, p.volume_pose, k.cloud, p.cloud_capacity, k.cloud_count, k.extract_ws, k.activity, es);
    if (st) return st;
    k.last_cloud = -1;
    return df_extract_normals(vol, k.cloud, p.cloud_capacity, k.cloud_count, p.volume_pose, Rinv_vol, p.gradient_delta_factor, k.cloud_nrm, es);
}

// start the deferred extraction on the auxiliary stream once `after` (an event of the main stream) has happened
int launch_deferred_extract(KinFu &k, cudaEvent_t after)
{
    if (!k.extract_deferred) return 0;
    k.extract_deferred = false;
    if (cudaStreamWaitEvent(k.aux, after, 0) != cudaSuccess) return (int)cudaGetLastError();
    if (int st = run_extract(k, k.aux)) return st;
    if (cudaEventRecord(k.ev_extract_done, k.aux) != cudaSuccess) return (int)cudaGetLastError();
    k.extract_pending = true;
    return 0;
}

// the main stream may not write the volume / activity map / cloud buffers while an extraction is still owed or in flight
int wait_extract_on_main(KinFu &k)
{
    if (k.extract_deferred) {
        if (cudaEventRecord(k.ev_volume_ready, k.stream) != cudaSuccess) return (int)cudaGetLastError();
        if (int st = launch_deferred_extract(k, k.ev_volume_ready)) return st;
    }
    if (!k.extract_pending) return 0;
    k.extract_pending = false;
    return (int)cudaStreamWaitEvent(k.stream, k.ev_extract_done, 0);
}
// host-side readers of the cloud (count, buffers, digest) make sure the extraction has been launched and wait for it
void sync_extract(KinFu &k)
{
    if (!k.aux) return;
    if (k.extract_deferred) {
        cudaEventRecord(k.ev_volume_ready, k.stream);
        launch_deferred_extract(k, k.ev_volume_ready);
    }
    cudaStreamSynchronize(k.aux);
}

void mark(KinFu &k, int stage)
{
    if (k.p.flags & DF_KINFU_STAGE_TIMING) cudaEventRecord(k.ev[stage], k.stream);
    k.stage_mark[stage] = 1;
}

int do_reset(KinFu &k)
{
    if (k.frame_counter) { printf("Reset\n"); ++k.resets; }          // kinfu.cpp:198-199
    k.frame_counter = 0;
    k.M = 0;                                                         // warp_->clear(), kinfu.cpp:206: the next first frame re-initialises the field
    k.poses.clear();
    k.poses.resize(12);
    dfh_aff_identity(k.poses.data());
    if (int w = wait_extract_on_main(k)) return w;
    if (k.activity && cudaMemsetAsync(k.activity, 0, k.activity_bytes, k.stream) != cudaSuccess) return (int)cudaGetLastError();
    return df_clear_volume(vol_of(k), k.stream);
}

// A normal-matrix row that does not fit (solve.cu: more than ROWCAP coupled columns) makes the solve leave the warp field unchanged for
// that frame and raise stats[5]; the flag is copied to pinned memory after every solve and reported here, loudly, at the next sync.
void note_solve_overflow(KinFu &k)
{
    double f;
    memcpy(&f, k.pinned + 14, sizeof f);
    if (f != 0.0) {
        ++k.solve_overflows;
        fprintf(stderr, "df_kinfu: warp solve skipped for one frame: a normal-matrix row exceeded the row capacity (df_kinfu_get_info[11] = %lld)\n", k.solve_overflows);
        f = 0.0;
        memcpy(k.pinned + 14, &f, sizeof f);
    }
}

static inline double now_us() { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

int process(KinFu &k, const uint16_t *depth_dev, size_t depth_pitch, bool only_df = false)
{
    const double t_begin = now_us();
    double t_sync0 = t_begin, t_sync1 = t_begin;
    const df_kinfu_params &p = k.p;
    cudaStream_t s = k.stream;
    const int LEVELS = k.levels;
    k.launches = 0;
    memset(k.stage_mark, 0, sizeof k.stage_mark);
    mark(k, 0);

    if (!only_df) {
    // ---- pre-processing, kinfu.cpp:226-242 -----------------------------------------------------------------------
    CKD(df_compute_dists(depth_dev, depth_pitch, p.cols, p.rows, p.intr, (uint16_t *)k.dists.ptr, k.dists.pitch, s));
    if (k.has_ov_depth) {              // lock-step parity hook: the caller's bilateral image instead of this frame's (expf differs by 1 LSB between CUDA and glibc)
        CK(cudaMemcpy2DAsync(k.cur_depth[0].ptr, k.cur_depth[0].pitch, k.ov_depth.data(), (size_t)p.cols * 2, (size_t)p.cols * 2, p.rows, cudaMemcpyHostToDevice, s));
        CK(cudaStreamSynchronize(s));  // the host vector may be replaced right after the call
        k.has_ov_depth = false;
        ++k.launches;
    } else {
        CKD(df_bilateral(depth_dev, depth_pitch, p.cols, p.rows, (uint16_t *)k.cur_depth[0].ptr, k.cur_depth[0].pitch,
                         p.bilateral_kernel_size, p.bilateral_sigma_spatial, p.bilateral_sigma_depth, s));
        k.launches += 2;
    }
    if (p.icp_truncate_depth_dist > 0) {
        CKD(df_truncate_depth((uint16_t *)k.cur_depth[0].ptr, k.cur_depth[0].pitch, p.cols, p.rows, p.icp_truncate_depth_dist, s));
        ++k.launches;
    }
    for (int i = 1; i < LEVELS; ++i) {
        CKD(df_pyr_down((const uint16_t *)k.cur_depth[i - 1].ptr, k.cur_depth[i - 1].pitch, k.cur_depth[i - 1].cols, k.cur_depth[i - 1].rows,
                        (uint16_t *)k.cur_depth[i].ptr, k.cur_depth[i].pitch, p.bilateral_sigma_depth, s));
        ++k.launches;
    }
    const bool use_depth = (p.flags & DF_KINFU_USE_DEPTH) != 0;
    for (int i = 0; i < LEVELS; ++i) {
        const int div = 1 << i;                                       // Intr::operator()(level), precomp.cpp:10-14
        const df_intr li = {p.intr.fx / div, p.intr.fy / div, p.intr.cx / div, p.intr.cy / div};
        if (use_depth) {
            // the reference's compile-time USE_DEPTH loop (internal.hpp:6, kinfu.cpp:237-238): normals from the depth map, depth masked
            // where the normal is invalid; the vertex pyramid is not built.  KinFu::dynamicfusion is still handed curr_.points_pyr[0]
            // (kinfu.cpp:284-287), which that build never writes; here it receives what the variable is meant to hold: the vertex map of
            // the level-0 depth (computed before the masking, normals to a scratch map) -- documented divergence, DESIGN 5.
            if (i == 0) {
                CKD(df_points_normals(li, (const uint16_t *)k.cur_depth[0].ptr, k.cur_depth[0].pitch, k.cur_depth[0].cols, k.cur_depth[0].rows,
                                      (float *)k.cur_pts[0].ptr, k.cur_pts[0].pitch, (float *)k.canon_nrm.ptr, k.canon_nrm.pitch, s));
                ++k.launches;
            }
            CKD(df_normals_mask_depth(li, (uint16_t *)k.cur_depth[i].ptr, k.cur_depth[i].pitch, k.cur_depth[i].cols, k.cur_depth[i].rows,
                                      (float *)k.cur_nrm[i].ptr, k.cur_nrm[i].pitch, s));
        } else
        CKD(df_points_normals(li, (const uint16_t *)k.cur_depth[i].ptr, k.cur_depth[i].pitch, k.cur_depth[i].cols, k.cur_depth[i].rows,
                              (float *)k.cur_pts[i].ptr, k.cur_pts[i].pitch, (float *)k.cur_nrm[i].ptr, k.cur_nrm[i].pitch, s));
        ++k.launches;
    }
    mark(k, 1);
    }

    const df_volume vol = vol_of(k);
    float vol_pose[12];
    memcpy(vol_pose, p.volume_pose.R, 36); memcpy(vol_pose + 9, p.volume_pose.t, 12);
    float Rinv_vol[9];
    dfh_mat3_inv(vol_pose, Rinv_vol);

    auto integrate_with = [&](const Img &dists, const float *cam_pose) -> int {
        float inv[12], vol2cam[12];
        dfh_aff_inv(cam_pose, inv);
        dfh_aff_mul(inv, vol_pose, vol2cam);                           // camera_pose.inv() * pose_, tsdf_volume.cpp:112
        k.launches += df_integrate_launch_count(vol);
        unsigned long long *counter = (p.flags & DF_KINFU_STAGE_TIMING) ? k.n_upd : nullptr;
        if (counter) cudaMemsetAsync(counter, 0, 8, s);
        if (int w = wait_extract_on_main(k)) return w;                 // write-after-read: the previous frame's extraction reads this volume
        return df_integrate_tracked(vol, (const uint16_t *)dists.ptr, dists.pitch, p.cols, p.rows, to_aff(vol2cam), p.intr, counter, k.activity, k.integrate_ws, s);
    };
    auto raycast_to = [&](const float *cam_pose, Img &pts, Img &nrm) -> int {
        float inv[12], cam2vol[12], Rinv[9];
        dfh_aff_inv(vol_pose, inv);
        dfh_aff_mul(inv, cam_pose, cam2vol);                           // pose_.inv() * camera_pose, tsdf_volume.cpp:162
        dfh_mat3_inv(cam2vol, Rinv);
        ++k.launches;
        // the loop's own volume is only ever integrated through the activity map, so the march may skip the bricks without negative voxels
        return df_raycast_points_tracked(vol, to_aff(cam2vol), Rinv, p.intr, p.cols, p.rows, p.raycast_step_factor, p.gradient_delta_factor,
                                         (float *)pts.ptr, pts.pitch, (float *)nrm.ptr, nrm.pitch, k.raycast_bricks ? k.activity : nullptr, s);
    };
    auto extract = [&](bool needed_now) -> int {                       // compute_points + compute_normals, tsdf_volume.cpp:313-325
        // needed_now: the caller reads the cloud right after (first frame: node initialisation; field extension): stay on the main stream
        k.launches += 5;                                               // count, 2 scans, emit + the normals kernel
        const bool overlap = k.overlap_extract && !needed_now && !(p.flags & DF_KINFU_STAGE_TIMING);
        if (int w = wait_extract_on_main(k)) return w;                 // an older extraction may still own the cloud buffers
        if (!overlap) return run_extract(k, s);
        k.extract_deferred = true;                                     // launched when the next frame's LM/PCG kernel starts, or on demand
        k.last_cloud = -1;
        return 0;
    };

    auto extend = [&]() -> int {                                       // SURVEY 8f(3) / Report.md step 4, DF_KINFU_EXTEND_FIELD
        if (!(p.flags & DF_KINFU_EXTEND_FIELD) || k.M <= 0) return 0;
        const int maxM = p.max_nodes > 0 ? p.max_nodes : (p.cloud_capacity + 49) / 50;
        if (k.M >= maxM) return 0;
        int st = df_extend_field(k.nodes, k.M, maxM, k.node_grid, k.cloud, p.cloud_capacity, k.cloud_count, 4,
                                 p.extend_radius > 0 ? p.extend_radius : 0.03f, p.node_step > 0 ? p.node_step : 50, k.M_dev, k.extend_ws, s);
        if (st) return st;
        k.launches += 3;
        int Mn = k.M;
        if (cudaMemcpyAsync(&Mn, k.M_dev, sizeof(int), cudaMemcpyDeviceToHost, s) != cudaSuccess) return (int)cudaGetLastError();
        if (cudaStreamSynchronize(s) != cudaSuccess) return (int)cudaGetLastError();
        if (Mn != k.M) {
            k.M = Mn;
            st = df_build_node_grid(k.nodes, k.M, k.node_grid, s);     // buildKDTree() after the node set changed
            ++k.launches;
        }
        return st;
    };

    // ---- first frame, kinfu.cpp:245-264 ----------------------------------------------------------------------------
    if (!only_df && k.frame_counter == 0) {
        CKD(integrate_with(k.dists, &k.poses[k.poses.size() - 12]));
        CKD(extract(true));
        if (!(p.flags & DF_KINFU_RIGID_ONLY)) {
            int count = 0;
            CK(cudaMemcpyAsync(&count, k.cloud_count, sizeof(int), cudaMemcpyDeviceToHost, s));
            CK(cudaStreamSynchronize(s));
            k.last_cloud = count;
            int step = p.node_step > 0 ? p.node_step : 50;
            int M = (count + step - 1) / step;
            if (p.max_nodes > 0 && M > p.max_nodes) { step = (count + p.max_nodes - 1) / p.max_nodes; M = (count + step - 1) / step; }
            k.M = M;
            if (M > 0) {
                init_nodes_kernel<<<div_up(M, 256), 256, 0, s>>>((const float4 *)k.cloud, step, M, k.nodes);
                CKD(df_build_node_grid(k.nodes, M, k.node_grid, s));       // buildKDTree(), warp_field.cpp:61
                k.launches += 2;
            }
        }
        for (int i = 0; i < MAX_LEVELS; ++i) {                          // kinfu.cpp:253-261
            if (p.flags & DF_KINFU_USE_DEPTH) std::swap(k.cur_depth[i], k.prev_depth[i]);
            else std::swap(k.cur_pts[i], k.prev_pts[i]);
            std::swap(k.cur_nrm[i], k.prev_nrm[i]);
        }
        ++k.frame_counter;
        return 0;
    }

    // ---- ICP, kinfu.cpp:268-278 (device-resident; one host read of {ok, T}) -----------------------------------------
    const bool pose_given = !only_df && k.has_ov_pose;               // lock-step parity hook: the caller's pose instead of this frame's ICP
    if (pose_given) { k.last_ok = 1; CK(cudaStreamSynchronize(s)); note_solve_overflow(k); }
    if (!only_df && !pose_given) {
        const float *vc[MAX_LEVELS], *nc[MAX_LEVELS], *vp[MAX_LEVELS], *np[MAX_LEVELS];
        int cols[MAX_LEVELS], rows[MAX_LEVELS]; size_t pitch[MAX_LEVELS];
        for (int i = 0; i < LEVELS; ++i) {
            vc[i] = (const float *)k.cur_pts[i].ptr; nc[i] = (const float *)k.cur_nrm[i].ptr;
            vp[i] = (const float *)k.prev_pts[i].ptr; np[i] = (const float *)k.prev_nrm[i].ptr;
            cols[i] = k.cur_pts[i].cols; rows[i] = k.cur_pts[i].rows; pitch[i] = k.cur_pts[i].pitch;
        }
        if (p.flags & DF_KINFU_USE_DEPTH) {                            // estimateTransform(depth pyramids), kinfu.cpp:271
            const unsigned short *dc[MAX_LEVELS], *dp[MAX_LEVELS];
            size_t dpitch[MAX_LEVELS], npitch[MAX_LEVELS];
            for (int i = 0; i < LEVELS; ++i) {
                dc[i] = (const unsigned short *)k.cur_depth[i].ptr; dp[i] = (const unsigned short *)k.prev_depth[i].ptr;
                dpitch[i] = k.cur_depth[i].pitch; npitch[i] = k.cur_nrm[i].pitch;
            }
            CKD(df_icp_estimate_depth(dc, nc, dp, np, cols, rows, dpitch, npitch, LEVELS, p.icp_iter_num, p.intr, p.icp_dist_thres, p.icp_angle_thres,
                                      k.icp_T, k.icp_ok, k.icp_scratch, s));
        } else
        CKD(df_icp_estimate(vc, nc, vp, np, cols, rows, pitch, LEVELS, p.icp_iter_num, p.intr, p.icp_dist_thres, p.icp_angle_thres,
                            k.icp_T, k.icp_ok, k.icp_scratch, s));
        for (int i = 0; i < LEVELS; ++i) k.launches += 2 * p.icp_iter_num[i];
        ++k.launches;
        CK(cudaMemcpyAsync(k.pinned, k.icp_T, 12 * sizeof(float), cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(k.pinned + 12, k.icp_ok, sizeof(int), cudaMemcpyDeviceToHost, s));
        t_sync0 = now_us();
        CK(cudaStreamSynchronize(s));
        t_sync1 = now_us();
        int ok;
        memcpy(&ok, k.pinned + 12, sizeof(int));
        k.last_ok = ok;
        note_solve_overflow(k);                                       // the previous frame's solve flag arrived with this sync
        if (!ok) { CKD(do_reset(k)); return 0; }                      // kinfu.cpp:276-277
    }
    mark(k, 2);
    if (pose_given) {
        k.poses.insert(k.poses.end(), k.ov_pose, k.ov_pose + 12);
        k.has_ov_pose = false;
    } else if (!only_df) {
        float pose[12];
        dfh_aff_mul(&k.poses[k.poses.size() - 12], k.pinned, pose);   // poses_.back() * affine, kinfu.cpp:280
        k.poses.insert(k.poses.end(), pose, pose + 12);
    }
    const float *cam_pose = &k.poses[k.poses.size() - 12];
    const int npix = p.cols * p.rows;

    if (!(p.flags & DF_KINFU_RIGID_ONLY) && k.M >= 8) {
        // ---- KinFu::dynamicfusion, kinfu.cpp:344-400 ------------------------------------------------------------------
        CKD(raycast_to(cam_pose, k.canon_visible, k.canon_nrm));       // tsdf().raycast(camera_pose, ...), :351 (camera frame)
        float inv_pose[12];
        dfh_aff_inv(cam_pose, inv_pose);
        launch_pdl(to_canonical_kernel, dim3(div_up(npix, 256)), dim3(256), 0, s, (const float4 *)k.canon_visible.ptr, make_aff(to_aff(inv_pose)),
                                                               (float4 *)k.canon.ptr, (float4 *)k.canon_visible.ptr, npix);
        ++k.launches;
        mark(k, 3);
        df_aff3f ident; float id12[12]; dfh_aff_identity(id12); ident = to_aff(id12);    // warp_to_live_ stays identity (never set)
        CKD(df_warp(k.nodes, k.M, k.node_grid, (float *)k.canon.ptr, (float *)k.canon_nrm.ptr, npix, 4, ident, DF_WARP_IMAGE_COLS(p.cols), nullptr, nullptr, s));   // :385
        ++k.launches;
        mark(k, 4);
        const bool f2_solve = (p.flags & DF_KINFU_F2_SOLVE) != 0;
        if (f2_solve) {
            // SURVEY 8f(2): robust 6-DoF data term + regulariser instead of the reference's translation-only data term (opt-in)
            CKD(df_solve_f2(k.nodes, k.M, k.node_grid, (const float *)k.canon.ptr, (const float *)k.cur_pts[0].ptr, npix, 4, &k.f2, k.f2_stats, k.f2_ws, s));
            k.launches += 6 + (k.f2.gn_iters + 1) * 4 + k.f2.gn_iters * (3 + 3 * k.f2.lin_iters);
        } else {
        CKD(solve_data_term_ev(k.nodes, k.M, k.node_grid, (const float *)k.canon.ptr, (const float *)k.cur_pts[0].ptr, npix, 4,
                               p.solver_nonlinear_iters, p.solver_linear_iters,
                               ((p.flags & DF_KINFU_REF_GRAPH_QUIRK) ? DF_SOLVE_REF_GRAPH_QUIRK : 0) | DF_SOLVE_IMAGE_COLS(p.cols), k.solve_stats, k.solve_ws, s,
                               k.ev_before_lm));   // :387
        k.launches += 9;                                               // prepare, blockscan, scan, tiles, rows (tiles), fill + rows (fallback), lm v6, lm v5 (fallback)
        CKD(launch_deferred_extract(k, k.ev_before_lm));               // the previous frame's extraction rides on the 132 SMs the solve leaves idle
        }
        // row-overflow flag of this solve (stats[5]): lands in pinned memory, looked at after the next stream synchronisation
        CK(cudaMemcpyAsync(k.pinned + 14, k.solve_stats + 5, sizeof(double), cudaMemcpyDeviceToHost, s));
        if (k.has_ov_nodes) {          // lock-step parity hook: the caller's solved node table (CPU and GPU PCG round differently in the last bits)
            if (k.ov_nodes.size() == (size_t)k.M * DF_NODE_STRIDE) {
                CK(cudaMemcpyAsync(k.nodes, k.ov_nodes.data(), k.ov_nodes.size() * 4, cudaMemcpyHostToDevice, s));
                CK(cudaStreamSynchronize(s));
            }
            k.has_ov_nodes = false;
        }
        mark(k, 5);
        if (f2_solve) {
            CKD(df_warp(k.nodes, k.M, k.node_grid, (float *)k.canon.ptr, (float *)k.canon_nrm.ptr, npix, 4, ident, 0, nullptr, nullptr, s));
        } else {
            // second warp (:389) queries exactly the vertices the solve just built its graph for (CombinedSolver.h:66-84):
            // re-use those neighbours + weights instead of a third k-NN pass
            int32_t *knn_idx; float *knn_w;
            CKD(df_solve_knn_buffers(k.solve_ws, k.M, npix, &knn_idx, &knn_w));
            CKD(df_warp(k.nodes, k.M, k.node_grid, (float *)k.canon.ptr, (float *)k.canon_nrm.ptr, npix, 4, ident, DF_WARP_REUSE_KNN, knn_idx, knn_w, s));
        }
        ++k.launches;
        mark(k, 6);
        if (p.flags & DF_KINFU_WARPED_INTEGRATE) {
            // SURVEY 8f(1): the update surface_fusion was written towards (tsdf_volume.cpp:240-252) -- every voxel is carried through
            // the field solved above and fused against the (bilateral-filtered) frame; no pixel is removed, no rigid integrate.
            mark(k, 7);
            unsigned long long *counter = (p.flags & DF_KINFU_STAGE_TIMING) ? k.n_upd : nullptr;
            if (counter) cudaMemsetAsync(counter, 0, 16, s);
            CKD(df_integrate_warped(vol, (const uint16_t *)k.cur_depth[0].ptr, k.cur_depth[0].pitch, p.cols, p.rows, p.volume_pose, to_aff(inv_pose),
                                    p.intr, k.nodes, k.M, k.node_grid, p.fusion_weight_scale, counter, k.activity, k.fusion_ws, s));
            k.launches += df_integrate_warped_launch_count();
            mark(k, 8);
            CKD(extract((p.flags & DF_KINFU_EXTEND_FIELD) != 0));
            CKD(extend());
            mark(k, 9);
        } else {
        // surface_fusion (tsdf_volume.cpp:228-255): psdf projects the warped vertices into the (bilateral-filtered) depth,
        // zeroes the pixels they explain, then the ordinary rigid integrate runs on what is left.
        CKD(df_project_and_remove((uint16_t *)k.cur_depth[0].ptr, k.cur_depth[0].pitch, p.cols, p.rows, p.intr,
                                  (float *)k.canon.ptr, k.canon.pitch, p.cols, p.rows, k.project_ws, s));
        k.launches += 2;
        CKD(df_compute_dists((const uint16_t *)k.cur_depth[0].ptr, k.cur_depth[0].pitch, p.cols, p.rows, p.intr,
                             (uint16_t *)k.dists.ptr, k.dists.pitch, s));
        ++k.launches;
        mark(k, 7);                                                    // stage "integrate" brackets the integrate kernel alone
        CKD(integrate_with(k.dists, cam_pose));
        mark(k, 8);
        CKD(extract((p.flags & DF_KINFU_EXTEND_FIELD) != 0));          // compute_points / compute_normals, :398-399
        CKD(extend());
        mark(k, 9);
        }
    } else {
        // plain KinFu (Nerei) loop: integrate the frame rigidly
        mark(k, 3); mark(k, 4); mark(k, 5); mark(k, 6); mark(k, 7);
        CKD(integrate_with(k.dists, cam_pose));
        mark(k, 8); mark(k, 9);
    }

    if (only_df) return 1;
    // ---- ray-cast for the next frame's ICP, kinfu.cpp:297-301 --------------------------------------------------------
    CKD(raycast_to(cam_pose, k.prev_pts[0], k.prev_nrm[0]));
    if (p.flags & DF_KINFU_USE_DEPTH) {
        // TsdfVolume::raycast(pose, intr, Depth&, Normals&) (tsdf_volume.cu:273-339,441-456) = the same march storing ushort(vertex.z * 1000),
        // then resizeDepthNormals per level (kinfu.cpp:293-295)
        CKD(df_cloud_to_depth((const float *)k.prev_pts[0].ptr, k.prev_pts[0].pitch, p.cols, p.rows, (uint16_t *)k.prev_depth[0].ptr, k.prev_depth[0].pitch, s));
        ++k.launches;
        for (int i = 1; i < LEVELS; ++i) {
            CKD(df_resize_depth_normals((const uint16_t *)k.prev_depth[i - 1].ptr, k.prev_depth[i - 1].pitch, (const float *)k.prev_nrm[i - 1].ptr,
                                        k.prev_nrm[i - 1].pitch, k.prev_depth[i - 1].cols, k.prev_depth[i - 1].rows,
                                        (uint16_t *)k.prev_depth[i].ptr, k.prev_depth[i].pitch, (float *)k.prev_nrm[i].ptr, k.prev_nrm[i].pitch, s));
            ++k.launches;
        }
    } else
    for (int i = 1; i < LEVELS; ++i) {
        CKD(df_resize_points_normals((const float *)k.prev_pts[i - 1].ptr, k.prev_pts[i - 1].pitch, (const float *)k.prev_nrm[i - 1].ptr,
                                     k.prev_nrm[i - 1].pitch, k.prev_pts[i - 1].cols, k.prev_pts[i - 1].rows,
                                     (float *)k.prev_pts[i].ptr, k.prev_pts[i].pitch, (float *)k.prev_nrm[i].ptr, k.prev_nrm[i].pitch, s));
        ++k.launches;
    }
    mark(k, 10);
    ++k.frame_counter;
    {
        const double t_end = now_us();
        k.host_us[0] += t_sync0 - t_begin; k.host_us[1] += t_sync1 - t_sync0; k.host_us[2] += t_end - t_sync1; k.host_us[3] += t_end - t_begin;
        ++k.host_frames;
    }
    return 1;
}

}  // namespace

extern "C" void df_kinfu_default_params(df_kinfu_params *p, int which)
{
    memset(p, 0, sizeof *p);
    p->cols = 640; p->rows = 480;
    const int iters[4] = {10, 5, 4, 0};
    memcpy(p->icp_iter_num, iters, sizeof iters);
    float pose[12];
    dfh_aff_identity(pose);
    if (which == 0) {          // default_params_dynamicfusion, kinfu.cpp:14-49
        p->intr = df_intr{570.342f, 570.342f, 320.f, 240.f};
        for (int i = 0; i < 3; ++i) { p->volume_dims[i] = 256; p->volume_size[i] = 1.f; }
    } else {                   // default_params, kinfu.cpp:55-89
        p->intr = df_intr{525.f, 525.f, 640 / 2 - 0.5f, 480 / 2 - 0.5f};
        for (int i = 0; i < 3; ++i) { p->volume_dims[i] = 512; p->volume_size[i] = 3.f; }
    }
    pose[9] = -p->volume_size[0] / 2; pose[10] = -p->volume_size[1] / 2; pose[11] = 0.5f;
    memcpy(p->volume_pose.R, pose, 36); memcpy(p->volume_pose.t, pose + 9, 12);
    p->bilateral_sigma_depth = 0.04f; p->bilateral_sigma_spatial = 4.5f; p->bilateral_kernel_size = 7;
    p->icp_truncate_depth_dist = 0.f; p->icp_dist_thres = 0.1f; p->icp_angle_thres = 30.f * 0.017453293f;
    p->tsdf_min_camera_movement = 0.f; p->tsdf_trunc_dist = 0.04f; p->tsdf_max_weight = 64;
    p->raycast_step_factor = 0.75f; p->gradient_delta_factor = 0.5f;
    p->solver_nonlinear_iters = 5; p->solver_linear_iters = 100;     // kinfu.cpp:116-117
    p->max_nodes = 4096; p->node_step = 50; p->cloud_capacity = 256 * 256 * 256 / 4;
    p->flags = 0;
}

extern "C" void df_kinfu_destroy(void *kinfu);

extern "C" void *df_kinfu_create(const df_kinfu_params *pp)
{
    if (pp->volume_dims[0] % 32 != 0) {                               // CV_Assert, kinfu.cpp:97
        fprintf(stderr, "df_kinfu_create: volume_dims[0] %% 32 != 0\n");
        return nullptr;
    }
    KinFu *k = new KinFu();
    k->p = *pp;
    cudaGetDevice(&k->device);
    {
        const char *e = getenv("DF_KINFU_WARPED_INTEGRATE");
        if (e && atoi(e) != 0) k->p.flags |= DF_KINFU_WARPED_INTEGRATE;
        const char *x = getenv("DF_KINFU_EXTEND_FIELD");
        if (x && atoi(x) != 0) k->p.flags |= DF_KINFU_EXTEND_FIELD;
        const char *xr = getenv("DF_EXTEND_RADIUS");
        if (xr) k->p.extend_radius = (float)atof(xr);
        const char *ud = getenv("DF_KINFU_USE_DEPTH");
        if (ud && atoi(ud) != 0) k->p.flags |= DF_KINFU_USE_DEPTH;
        const char *f2e = getenv("DF_KINFU_F2_SOLVE");
        if (f2e && atoi(f2e) != 0) k->p.flags |= DF_KINFU_F2_SOLVE;
        const char *rb = getenv("DF_RAYCAST_BRICKS");
        if (rb && atoi(rb) == 0) k->raycast_bricks = false;
        const char *w = getenv("DF_FUSION_WEIGHT_SCALE");
        if (w) k->p.fusion_weight_scale = (float)atof(w);
    }
    const df_kinfu_params &p = k->p;
    int i = MAX_LEVELS - 1;                                           // getUsedLevelsNum, projective_icp.cpp:110-115
    for (; i >= 0 && !p.icp_iter_num[i]; --i) {}
    k->levels = i + 1;
    float vmax = 0.f;
    for (int d = 0; d < 3; ++d) { k->voxel_size[d] = p.volume_size[d] / p.volume_dims[d]; vmax = vmax > k->voxel_size[d] ? vmax : k->voxel_size[d]; }
    k->trunc_dist = p.tsdf_trunc_dist > 2.1f * vmax ? p.tsdf_trunc_dist : 2.1f * vmax;   // setTruncDist, tsdf_volume.cpp:68-73
    const size_t nvox = (size_t)p.volume_dims[0] * p.volume_dims[1] * p.volume_dims[2];
    bool ok = cudaMalloc(&k->volume, nvox * 4) == cudaSuccess;
    ok = ok && alloc_img(k->depth_in, p.rows, p.cols, 2) == 0 && alloc_img(k->dists, p.rows, p.cols, 2) == 0;
    int cols = p.cols, rows = p.rows;
    for (int l = 0; l < MAX_LEVELS && ok; ++l) {                      // allocate_buffers, kinfu.cpp:151-194
        ok = ok && alloc_img(k->cur_depth[l], rows, cols, 2) == 0 && alloc_img(k->cur_pts[l], rows, cols, 16) == 0 &&
             alloc_img(k->cur_nrm[l], rows, cols, 16) == 0 && alloc_img(k->prev_pts[l], rows, cols, 16) == 0 &&
             alloc_img(k->prev_nrm[l], rows, cols, 16) == 0 && alloc_img(k->prev_depth[l], rows, cols, 2) == 0;
        cols /= 2; rows /= 2;
    }
    ok = ok && alloc_img(k->canon, p.rows, p.cols, 16) == 0 && alloc_img(k->canon_nrm, p.rows, p.cols, 16) == 0 &&
         alloc_img(k->canon_visible, p.rows, p.cols, 16) == 0;
    ok = ok && cudaMalloc(&k->cloud, (size_t)p.cloud_capacity * 16) == cudaSuccess && cudaMalloc(&k->cloud_nrm, (size_t)p.cloud_capacity * 16) == cudaSuccess;
    ok = ok && cudaMalloc(&k->cloud_count, 64) == cudaSuccess;
    const int maxM = p.max_nodes > 0 ? p.max_nodes : (p.cloud_capacity + 49) / 50;
    ok = ok && cudaMalloc(&k->nodes, (size_t)maxM * DF_NODE_STRIDE * 4) == cudaSuccess && cudaMalloc(&k->node_grid, df_node_grid_bytes(maxM)) == cudaSuccess;
    ok = ok && cudaMalloc(&k->icp_T, 64) == cudaSuccess && cudaMalloc(&k->icp_ok, 64) == cudaSuccess &&
         cudaMalloc(&k->icp_scratch, (size_t)DF_ICP_SCRATCH_DOUBLES * 8) == cudaSuccess;
    k->solve_ws_bytes = df_solve_workspace_bytes(maxM, p.cols * p.rows);
    ok = ok && cudaMalloc(&k->solve_ws, k->solve_ws_bytes) == cudaSuccess && cudaMalloc(&k->solve_stats, 64) == cudaSuccess;
    k->f2 = df_f2_params{5.0, 0.05, 1e-4, 1e-4, 2, 4, DF_F2_TWIST | DF_F2_TUKEY | DF_F2_HUBER, 30};
    if (p.flags & DF_KINFU_F2_SOLVE)
        ok = ok && cudaMalloc(&k->f2_ws, df_solve_f2_workspace_bytes(maxM, p.cols * p.rows, 7)) == cudaSuccess && cudaMalloc(&k->f2_stats, 16 * 8) == cudaSuccess;
    df_volume v = vol_of(*k);
    ok = ok && cudaMalloc(&k->extract_ws, df_extract_workspace_bytes(v)) == cudaSuccess;
    ok = ok && cudaMalloc(&k->integrate_ws, df_integrate_workspace_bytes(p.cols, p.rows)) == cudaSuccess;
    ok = ok && cudaMalloc(&k->extend_ws, df_extend_field_workspace_bytes(p.cloud_capacity)) == cudaSuccess && cudaMalloc((void **)&k->M_dev, 64) == cudaSuccess;
    ok = ok && cudaMalloc(&k->fusion_ws, df_integrate_warped_workspace_bytes(p.cols, p.rows, maxM)) == cudaSuccess;
    k->activity_bytes = df_volume_activity_bytes(v);
    ok = ok && cudaMalloc(&k->activity, k->activity_bytes) == cudaSuccess && cudaMemset(k->activity, 0, k->activity_bytes) == cudaSuccess;
    ok = ok && cudaMalloc(&k->project_ws, df_project_workspace_bytes(p.cols, p.rows)) == cudaSuccess;
    ok = ok && cudaMemset(k->project_ws, 0, df_project_workspace_bytes(p.cols, p.rows)) == cudaSuccess;
    ok = ok && cudaMemset(k->solve_stats, 0, 64) == cudaSuccess && cudaMemset(k->cloud_count, 0, 64) == cudaSuccess;
    ok = ok && cudaMallocHost(&k->pinned, 64) == cudaSuccess && (memset(k->pinned, 0, 64), true) && cudaMalloc(&k->n_upd, 64) == cudaSuccess && cudaMemset(k->n_upd, 0, 64) == cudaSuccess;
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);              // lo = numerically greatest = lowest priority
    ok = ok && cudaStreamCreateWithPriority(&k->aux, cudaStreamNonBlocking, prio_lo) == cudaSuccess &&
         cudaEventCreateWithFlags(&k->ev_before_lm, cudaEventDisableTiming) == cudaSuccess &&
         cudaEventCreateWithFlags(&k->ev_volume_ready, cudaEventDisableTiming) == cudaSuccess &&
         cudaEventCreateWithFlags(&k->ev_extract_done, cudaEventDisableTiming) == cudaSuccess;
    { const char *oe = getenv("DF_KINFU_OVERLAP_EXTRACT"); if (oe && atoi(oe) == 0) k->overlap_extract = false; }
    for (int e = 0; e <= NSTAGES; ++e) k->ev[e] = nullptr;
    for (int e = 0; e <= NSTAGES && ok; ++e) ok = cudaEventCreate(&k->ev[e]) == cudaSuccess;
    if (!ok) {
        fprintf(stderr, "df_kinfu_create: CUDA allocation failed: %s\n", cudaGetErrorString(cudaGetLastError()));
        df_kinfu_destroy(k);                                          // frees whatever was allocated (cudaFree(nullptr) is a no-op)
        return nullptr;
    }
    memset(k->stage_ms, 0, sizeof k->stage_ms);
    do_reset(*k);
    cudaStreamSynchronize(k->stream);
    return k;
}

extern "C" void df_kinfu_destroy(void *h)
{
    KinFu *k = (KinFu *)h;
    if (!k) return;
    cudaSetDevice(k->device);
    if (getenv("DF_KINFU_HOSTPROF") && k->host_frames)
        fprintf(stderr, "[df_kinfu host profile] frames %lld: launch-A %.1f us, ICP wait %.1f us, launch-B %.1f us, total %.1f us per frame\n", k->host_frames,
                k->host_us[0] / k->host_frames, k->host_us[1] / k->host_frames, k->host_us[2] / k->host_frames, k->host_us[3] / k->host_frames);
    cudaStreamSynchronize(k->stream);
    if (k->aux) { cudaStreamSynchronize(k->aux); cudaStreamDestroy(k->aux); }
    if (k->ev_volume_ready) cudaEventDestroy(k->ev_volume_ready);
    if (k->ev_before_lm) cudaEventDestroy(k->ev_before_lm);
    if (k->ev_extract_done) cudaEventDestroy(k->ev_extract_done);
    cudaFree(k->volume); cudaFree(k->depth_in.ptr); cudaFree(k->dists.ptr);
    for (int l = 0; l < MAX_LEVELS; ++l) { cudaFree(k->cur_depth[l].ptr); cudaFree(k->cur_pts[l].ptr); cudaFree(k->cur_nrm[l].ptr); cudaFree(k->prev_pts[l].ptr); cudaFree(k->prev_nrm[l].ptr); cudaFree(k->prev_depth[l].ptr); }
    cudaFree(k->canon.ptr); cudaFree(k->canon_nrm.ptr); cudaFree(k->canon_visible.ptr);
    cudaFree(k->cloud); cudaFree(k->cloud_nrm); cudaFree(k->cloud_count); cudaFree(k->nodes); cudaFree(k->node_grid);
    cudaFree(k->icp_T); cudaFree(k->icp_ok); cudaFree(k->icp_scratch); cudaFree(k->solve_ws); cudaFree(k->solve_stats);
    cudaFree(k->f2_ws); cudaFree(k->f2_stats);
    cudaFree(k->extract_ws); cudaFree(k->project_ws); cudaFree(k->activity); cudaFree(k->integrate_ws); cudaFree(k->fusion_ws); cudaFree(k->mesh_ws); cudaFree(k->extend_ws); cudaFree(k->M_dev); cudaFreeHost(k->pinned); cudaFree(k->n_upd);
    for (int e = 0; e <= NSTAGES; ++e) if (k->ev[e]) cudaEventDestroy(k->ev[e]);
    delete k;
}

extern "C" int df_kinfu_set_stream(void *h, void *stream) { ((KinFu *)h)->stream = (cudaStream_t)stream; return 0; }
extern "C" int df_kinfu_reset(void *h) { KinFu *k = (KinFu *)h; int s = do_reset(*k); return s ? -s : 0; }

static void finish_timing(KinFu &k)
{
    if (!(k.p.flags & DF_KINFU_STAGE_TIMING)) return;
    cudaStreamSynchronize(k.stream);
    int prev = 0;
    for (int s = 1; s <= NSTAGES; ++s) {
        k.stage_ms[s - 1] = 0.f;
        if (!k.stage_mark[s]) continue;
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, k.ev[prev], k.ev[s]) == cudaSuccess) k.stage_ms[s - 1] = ms;
        prev = s;
    }
}

// Multi-device host entry (SURVEY 8e: the path shards by SEQUENCE): n independent KinFu objects -- typically one per GPU, created after
// cudaSetDevice(i) -- advance by one frame each, concurrently: one host thread per object (a frame has one host synchronisation, the ICP
// status, so a sequential loop would serialise the devices).  results[i] receives what df_kinfu_process_host returns for object i.
extern "C" int df_kinfu_batch_process_host(void *const *kinfus, const uint16_t *const *depth_host, const size_t *pitch, int n, int *results)
{
    if (n <= 0) return 0;
    std::vector<std::thread> th;
    th.reserve((size_t)n);
    for (int i = 1; i < n; ++i)
        th.emplace_back([=] { results[i] = df_kinfu_process_host(kinfus[i], depth_host[i], pitch[i]); });
    results[0] = df_kinfu_process_host(kinfus[0], depth_host[0], pitch[0]);
    for (auto &t : th) t.join();
    int worst = 0;
    for (int i = 0; i < n; ++i) if (results[i] < worst) worst = results[i];
    return worst;                                                    // 0, or the first negative status (-cudaError) of any object
}

extern "C" int df_kinfu_process_device(void *h, const uint16_t *depth_dev, size_t pitch)
{
    KinFu *k = (KinFu *)h;
    cudaSetDevice(k->device);
    const int r = process(*k, depth_dev, pitch);
    finish_timing(*k);
    return r;
}

// KinFu::dynamicfusion(depth, live_frame, current_normals) (kinfu.hpp:87, kinfu.cpp:344-400) as a stand-alone call on
// caller-provided device buffers (depth is modified in place by the project-and-remove step, like the reference)
extern "C" int df_kinfu_dynamicfusion(void *h, uint16_t *depth_dev, size_t depth_pitch, const float *live_points_dev, size_t live_pitch)
{
    KinFu *k = (KinFu *)h;
    if (k->poses.size() < 12) return 0;
    const Img saved_depth = k->cur_depth[0], saved_pts = k->cur_pts[0];
    k->cur_depth[0].ptr = depth_dev; k->cur_depth[0].pitch = depth_pitch;
    k->cur_pts[0].ptr = (void *)live_points_dev; k->cur_pts[0].pitch = live_pitch;
    const int r = process(*k, nullptr, 0, true);
    k->cur_depth[0] = saved_depth; k->cur_pts[0] = saved_pts;
    return r;
}

extern "C" int df_kinfu_process_host(void *h, const uint16_t *depth_host, size_t pitch)
{
    KinFu *k = (KinFu *)h;
    cudaSetDevice(k->device);                                         // per host thread: lets one process drive one object per GPU
    // depth_device_.upload(depth.data, depth.step, rows, cols), apps/demo.cpp:89
    cudaError_t e = cudaMemcpy2DAsync(k->depth_in.ptr, k->depth_in.pitch, depth_host, pitch, (size_t)k->p.cols * 2, k->p.rows,
                                      cudaMemcpyHostToDevice, k->stream);
    if (e != cudaSuccess) return -(int)e;
    const int r = process(*k, (const uint16_t *)k->depth_in.ptr, k->depth_in.pitch);
    if (r < 0) return r;
    e = cudaStreamSynchronize(k->stream);        // the caller owns the result when the call returns (renderImage / getCameraPose next)
    if (e == cudaSuccess) note_solve_overflow(*k);
    finish_timing(*k);
    return e == cudaSuccess ? r : -(int)e;
}

extern "C" int df_kinfu_get_pose(void *h, int time, float *pose12)
{
    KinFu *k = (KinFu *)h;
    const int n = (int)(k->poses.size() / 12);
    if (time > n || time < 0) time = n - 1;                            // kinfu.cpp:213-218
    if (time >= n) time = n - 1;
    memcpy(pose12, &k->poses[(size_t)time * 12], 48);
    return 0;
}

extern "C" int df_kinfu_get_info(void *h, long long *info, int n)
{
    KinFu *k = (KinFu *)h;
    sync_extract(*k);
    if (k->last_cloud < 0) {
        int c = 0;
        cudaMemcpyAsync(&c, k->cloud_count, sizeof(int), cudaMemcpyDeviceToHost, k->stream);
        cudaStreamSynchronize(k->stream);
        k->last_cloud = c;
    }
    double st[8] = {0};
    cudaMemcpyAsync(st, k->solve_stats, sizeof st, cudaMemcpyDeviceToHost, k->stream);
    cudaStreamSynchronize(k->stream);
    unsigned long long nu2[2] = {0, 0};
    cudaMemcpyAsync(nu2, k->n_upd, 16, cudaMemcpyDeviceToHost, k->stream);
    cudaStreamSynchronize(k->stream);
    const unsigned long long nu = nu2[0];
    note_solve_overflow(*k);
    const long long vals[12] = {k->frame_counter, k->M, k->last_cloud, (long long)(k->poses.size() / 12), k->last_ok, k->launches, k->resets,
                                (long long)st[2], (long long)nu, (long long)st[4], (long long)nu2[1], k->solve_overflows};
    for (int i = 0; i < n && i < 12; ++i) info[i] = vals[i];
    return 0;
}

// stream-ordered join: the object's main stream waits for the extraction in flight on its auxiliary stream (no host synchronisation)
extern "C" int df_kinfu_join(void *h)
{
    KinFu *k = (KinFu *)h;
    return wait_extract_on_main(*k);
}

extern "C" int df_kinfu_get_buffer(void *h, int which, void **ptr, size_t *pitch, int *cols, int *rows)
{
    KinFu *k = (KinFu *)h;
    if (which == 9 || which == 10) sync_extract(*k);               // the caller is about to use the cloud on a stream of its own
    Img im;
    switch (which) {
        case 0: im.ptr = k->volume; im.pitch = (size_t)k->p.volume_dims[0] * 4; im.cols = k->p.volume_dims[0]; im.rows = k->p.volume_dims[1] * k->p.volume_dims[2]; break;
        case 1: im = k->dists; break;
        case 2: im = k->cur_depth[0]; break;
        case 3: im = k->cur_pts[0]; break;
        case 4: im = k->cur_nrm[0]; break;
        case 5: im = k->prev_pts[0]; break;
        case 6: im = k->prev_nrm[0]; break;
        case 7: im = k->canon; break;
        case 8: im = k->canon_nrm; break;
        case 9: im.ptr = k->cloud; im.pitch = 16; im.cols = 1; im.rows = k->p.cloud_capacity; break;
        case 10: im.ptr = k->cloud_nrm; im.pitch = 16; im.cols = 1; im.rows = k->p.cloud_capacity; break;
        case 11: im.ptr = k->nodes; im.pitch = DF_NODE_STRIDE * 4; im.cols = 1; im.rows = k->M; break;
        case 12: im = k->canon_visible; break;
        case 13: im.ptr = k->solve_stats; im.pitch = 64; im.cols = 8; im.rows = 1; break;
        case 15: im.ptr = k->f2_stats; im.pitch = 128; im.cols = 16; im.rows = 1; break;
        case 14: im.ptr = k->activity; im.pitch = k->activity_bytes; im.cols = (int)k->activity_bytes; im.rows = 1; break;
        default: return (int)cudaErrorInvalidValue;
    }
    *ptr = im.ptr; *pitch = im.pitch; *cols = im.cols; *rows = im.rows;
    return 0;
}

extern "C" int df_kinfu_read_buffer(void *h, int which, void *dst_host, size_t bytes)
{
    KinFu *k = (KinFu *)h;
    void *ptr; size_t pitch; int cols, rows;
    const int st = df_kinfu_get_buffer(h, which, &ptr, &pitch, &cols, &rows);
    if (st) return st;
    const size_t have = pitch * (size_t)rows;
    sync_extract(*k);
    cudaError_t e = cudaStreamSynchronize(k->stream);
    if (e != cudaSuccess) return (int)e;
    e = cudaMemcpy(dst_host, ptr, bytes < have ? bytes : have, cudaMemcpyDeviceToHost);
    return (int)e;
}

extern "C" int df_kinfu_set_overrides(void *h, const uint16_t *bilateral_depth_host, size_t pitch, const float *pose12_host, const float *nodes_host, int M)
{
    KinFu *k = (KinFu *)h;
    k->has_ov_depth = bilateral_depth_host != nullptr;
    if (bilateral_depth_host) {
        k->ov_depth.resize((size_t)k->p.cols * k->p.rows);
        for (int y = 0; y < k->p.rows; ++y) memcpy(&k->ov_depth[(size_t)y * k->p.cols], (const char *)bilateral_depth_host + (size_t)y * pitch, (size_t)k->p.cols * 2);
    }
    k->has_ov_pose = pose12_host != nullptr;
    if (pose12_host) memcpy(k->ov_pose, pose12_host, 48);
    k->has_ov_nodes = nodes_host != nullptr && M > 0;
    if (k->has_ov_nodes) k->ov_nodes.assign(nodes_host, nodes_host + (size_t)M * DF_NODE_STRIDE);
    return 0;
}

extern "C" int df_kinfu_set_f2_params(void *h, const df_f2_params *prm)
{
    KinFu *k = (KinFu *)h;
    if (!prm) return (int)cudaErrorInvalidValue;
    k->f2 = *prm;
    if (k->f2.reg_k > 7) k->f2.reg_k = 7;
    return 0;
}

extern "C" int df_kinfu_state_digest(void *h, unsigned long long *out4_host)
{
    KinFu *k = (KinFu *)h;
    sync_extract(*k);
    unsigned long long *d = nullptr;
    if (cudaMalloc((void **)&d, 32) != cudaSuccess) return (int)cudaGetLastError();
    cudaMemsetAsync(d, 0, 32, k->stream);
    const size_t nvox = (size_t)k->p.volume_dims[0] * k->p.volume_dims[1] * k->p.volume_dims[2];
    digest_kernel<<<148 * 8, 256, 0, k->stream>>>(k->volume, nvox, d);
    if (k->M > 0) digest_kernel<<<8, 256, 0, k->stream>>>((const uint32_t *)k->nodes, (size_t)k->M * DF_NODE_STRIDE, d + 1);
    cudaMemcpyAsync(d + 2, k->cloud_count, sizeof(int), cudaMemcpyDeviceToDevice, k->stream);
    cudaError_t e = cudaMemcpyAsync(out4_host, d, 32, cudaMemcpyDeviceToHost, k->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(k->stream);
    cudaFree(d);
    if (e != cudaSuccess) return (int)e;
    unsigned long long ph = 0x243f6a8885a308d3ull;                      // camera poses so far, bit pattern by bit pattern
    for (float f : k->poses) { uint32_t u; memcpy(&u, &f, 4); ph = (ph ^ u) * 0x100000001b3ull; }
    out4_host[3] = ph;
    return 0;
}

extern "C" int df_kinfu_get_stage_ms(void *h, float *ms, int n)
{
    KinFu *k = (KinFu *)h;
    const int m = n < NSTAGES ? n : NSTAGES;
    for (int i = 0; i < m; ++i) ms[i] = k->stage_ms[i];
    return m;
}

// Mesh of the current model, on demand.  It only reads the volume and the activity map, on the main stream after the last integrate; it
// neither launches nor waits for the deferred extraction (which only reads the volume as well) and writes nothing the loop owns.
extern "C" int df_kinfu_extract_mesh(void *h, int flags, float *vertices, float *normals, uint32_t *edge_keys, int vcap,
                                     int32_t *triangles, int tcap, int *counts_host)
{
    KinFu *k = (KinFu *)h;
    if (!k || !counts_host || vcap < 0 || tcap < 0) return (int)cudaErrorInvalidValue;
    const bool live = (flags & DF_MESH_LIVE) != 0;
    if (live && ((k->p.flags & DF_KINFU_RIGID_ONLY) || k->M < 8)) return (int)cudaErrorInvalidValue;   // no field the loop would warp with
    cudaSetDevice(k->device);
    cudaStream_t s = k->stream;
    const df_volume vol = vol_of(*k);
    const size_t ws_bytes = df_extract_mesh_workspace_bytes(vol);
    const bool scratch_normals = live && !normals;     // the warp needs normals: a vertex with a NaN normal is left in place
    const size_t need = ws_bytes + 256 + (scratch_normals ? (size_t)vcap * 16 : 0);
    if (need > k->mesh_ws_bytes) {
        cudaFree(k->mesh_ws);
        k->mesh_ws = nullptr; k->mesh_ws_bytes = 0;
        if (cudaMalloc(&k->mesh_ws, need) != cudaSuccess) return (int)cudaGetLastError();
        k->mesh_ws_bytes = need;
    }
    int *counts_dev = (int *)((char *)k->mesh_ws + ws_bytes);
    float *nrm = scratch_normals ? (float *)((char *)k->mesh_ws + ws_bytes + 256) : normals;
    const df_kinfu_params &p = k->p;
    if (int st = df_extract_mesh(vol, p.volume_pose, k->activity, vertices, edge_keys, vcap, triangles, tcap, counts_dev, k->mesh_ws, s)) return st;
    if (nrm) {
        float vol_pose[12], Rinv_vol[9];
        memcpy(vol_pose, p.volume_pose.R, 36); memcpy(vol_pose + 9, p.volume_pose.t, 12);
        dfh_mat3_inv(vol_pose, Rinv_vol);
        if (int st = df_extract_normals(vol, vertices, vcap, counts_dev, p.volume_pose, Rinv_vol, p.gradient_delta_factor, nrm, s)) return st;
    }
    int counts[2] = {0, 0};
    if (cudaMemcpyAsync(counts, counts_dev, sizeof counts, cudaMemcpyDeviceToHost, s) != cudaSuccess || cudaStreamSynchronize(s) != cudaSuccess)
        return (int)cudaGetLastError();
    counts_host[0] = counts[0]; counts_host[1] = counts[1];
    if (live) {
        const int n = counts[0] < vcap ? counts[0] : vcap;
        float id12[12];
        dfh_aff_identity(id12);
        if (int st = df_warp(k->nodes, k->M, k->node_grid, vertices, nrm, n, 4, to_aff(id12), DF_WARP_NORMAL_ROTATE_ONLY, nullptr, nullptr, s)) return st;
        if (cudaStreamSynchronize(s) != cudaSuccess) return (int)cudaGetLastError();
    }
    return 0;
}
