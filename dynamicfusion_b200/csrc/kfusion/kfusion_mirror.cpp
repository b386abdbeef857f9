// kfusion_mirror.cpp -- host-side C++ mirror of the reference's public classes (include/kfusion/*.hpp) over the C ABI of
// libdfusion.so.  Same names, argument meaning and error behaviour as kfusion/src/{device_memory,imgproc,projective_icp,
// tsdf_volume,warp_field,warp_field_optimiser,kinfu,precomp}.cpp of the reference; the compute is never here -- every
// method forwards to a df_* entry point (hand-written sm_100a kernels).  Builds into libkfusion.so.
#include <kfusion/kinfu.hpp>
#include <kfusion/cuda/imgproc.hpp>
#include <dfusion.h>
#include <df_hostmath.h>
#include <cuda_runtime.h>
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <iostream>

using namespace kfusion;
using namespace kfusion::cuda;

// ------------------------------------------------------------------------------------------------------------------
// error(): device_memory.cpp:7-11 -- print and exit(0)
void kfusion::cuda::error(const char *error_string, const char *file, const int line, const char * /*func*/)
{
    std::cout << "KinFu2 error: " << error_string << "\t" << file << ":" << line << std::endl;
    exit(0);
}
#define cudaSafeCall(expr)                                                                         \
    do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) kfusion::cuda::error(cudaGetErrorString(e__), __FILE__, __LINE__); } while (0)
#define dfSafeCall(expr)                                                                           \
    do { int s__ = (expr); if (s__ != 0) kfusion::cuda::error(df_error_string(s__ < 0 ? -s__ : s__), __FILE__, __LINE__); } while (0)

// ------------------------------------------------------------------------------------------------------------------
// DeviceMemory / DeviceMemory2D: device_memory.cpp:34-252
static inline int xadd(int *addr, int delta) { return __sync_fetch_and_add(addr, delta); }

DeviceMemory::DeviceMemory() : data_(0), sizeBytes_(0), refcount_(0) {}
DeviceMemory::DeviceMemory(void *ptr_arg, size_t sizeBytes_arg) : data_(ptr_arg), sizeBytes_(sizeBytes_arg), refcount_(0) {}
DeviceMemory::DeviceMemory(size_t sizeBytes_arg) : data_(0), sizeBytes_(0), refcount_(0) { create(sizeBytes_arg); }
DeviceMemory::~DeviceMemory() { release(); }
DeviceMemory::DeviceMemory(const DeviceMemory& o) : data_(o.data_), sizeBytes_(o.sizeBytes_), refcount_(o.refcount_) { if (refcount_) xadd(refcount_, 1); }
DeviceMemory& DeviceMemory::operator=(const DeviceMemory& o)
{
    if (this != &o) {
        if (o.refcount_) xadd(o.refcount_, 1);
        release();
        data_ = o.data_; sizeBytes_ = o.sizeBytes_; refcount_ = o.refcount_;
    }
    return *this;
}
void DeviceMemory::create(size_t sizeBytes_arg)
{
    if (sizeBytes_arg == sizeBytes_) return;
    if (sizeBytes_arg > 0) {
        if (data_) release();
        sizeBytes_ = sizeBytes_arg;
        cudaSafeCall(cudaMalloc(&data_, sizeBytes_));
        refcount_ = new int;
        *refcount_ = 1;
    }
}
void DeviceMemory::copyTo(DeviceMemory& other) const
{
    if (empty()) other.release();
    else { other.create(sizeBytes_); cudaSafeCall(cudaMemcpy(other.data_, data_, sizeBytes_, cudaMemcpyDeviceToDevice)); }
}
void DeviceMemory::release()
{
    if (refcount_ && xadd(refcount_, -1) == 1) { delete refcount_; cudaSafeCall(cudaFree(data_)); }
    data_ = 0; sizeBytes_ = 0; refcount_ = 0;
}
void DeviceMemory::upload(const void *host_ptr_arg, size_t sizeBytes_arg)
{ create(sizeBytes_arg); cudaSafeCall(cudaMemcpy(data_, host_ptr_arg, sizeBytes_, cudaMemcpyHostToDevice)); }
void DeviceMemory::download(void *host_ptr_arg) const { cudaSafeCall(cudaMemcpy(host_ptr_arg, data_, sizeBytes_, cudaMemcpyDeviceToHost)); }
void DeviceMemory::swap(DeviceMemory& o) { std::swap(data_, o.data_); std::swap(sizeBytes_, o.sizeBytes_); std::swap(refcount_, o.refcount_); }
bool DeviceMemory::empty() const { return !data_; }
size_t DeviceMemory::sizeBytes() const { return sizeBytes_; }

DeviceMemory2D::DeviceMemory2D() : data_(0), step_(0), colsBytes_(0), rows_(0), refcount_(0) {}
DeviceMemory2D::DeviceMemory2D(int rows_arg, int colsBytes_arg) : data_(0), step_(0), colsBytes_(0), rows_(0), refcount_(0) { create(rows_arg, colsBytes_arg); }
DeviceMemory2D::DeviceMemory2D(int rows_arg, int colsBytes_arg, void *data_arg, size_t step_arg)
    : data_(data_arg), step_(step_arg), colsBytes_(colsBytes_arg), rows_(rows_arg), refcount_(0) {}
DeviceMemory2D::~DeviceMemory2D() { release(); }
DeviceMemory2D::DeviceMemory2D(const DeviceMemory2D& o) : data_(o.data_), step_(o.step_), colsBytes_(o.colsBytes_), rows_(o.rows_), refcount_(o.refcount_)
{ if (refcount_) xadd(refcount_, 1); }
DeviceMemory2D& DeviceMemory2D::operator=(const DeviceMemory2D& o)
{
    if (this != &o) {
        if (o.refcount_) xadd(o.refcount_, 1);
        release();
        colsBytes_ = o.colsBytes_; rows_ = o.rows_; data_ = o.data_; step_ = o.step_; refcount_ = o.refcount_;
    }
    return *this;
}
void DeviceMemory2D::create(int rows_arg, int colsBytes_arg)
{
    if (colsBytes_ == colsBytes_arg && rows_ == rows_arg) return;
    if (rows_arg > 0 && colsBytes_arg > 0) {
        if (data_) release();
        colsBytes_ = colsBytes_arg; rows_ = rows_arg;
        cudaSafeCall(cudaMallocPitch((void **)&data_, &step_, colsBytes_, rows_));
        refcount_ = new int;
        *refcount_ = 1;
    }
}
void DeviceMemory2D::release()
{
    if (refcount_ && xadd(refcount_, -1) == 1) { delete refcount_; cudaSafeCall(cudaFree(data_)); }
    colsBytes_ = 0; rows_ = 0; data_ = 0; step_ = 0; refcount_ = 0;
}
void DeviceMemory2D::copyTo(DeviceMemory2D& other) const
{
    if (empty()) other.release();
    else { other.create(rows_, colsBytes_); cudaSafeCall(cudaMemcpy2D(other.data_, other.step_, data_, step_, colsBytes_, rows_, cudaMemcpyDeviceToDevice)); }
}
void DeviceMemory2D::upload(const void *host_ptr_arg, size_t host_step_arg, int rows_arg, int colsBytes_arg)
{ create(rows_arg, colsBytes_arg); cudaSafeCall(cudaMemcpy2D(data_, step_, host_ptr_arg, host_step_arg, colsBytes_, rows_, cudaMemcpyHostToDevice)); }
void DeviceMemory2D::download(void *host_ptr_arg, size_t host_step_arg) const
{ cudaSafeCall(cudaMemcpy2D(host_ptr_arg, host_step_arg, data_, step_, colsBytes_, rows_, cudaMemcpyDeviceToHost)); }
void DeviceMemory2D::swap(DeviceMemory2D& o)
{ std::swap(data_, o.data_); std::swap(step_, o.step_); std::swap(colsBytes_, o.colsBytes_); std::swap(rows_, o.rows_); std::swap(refcount_, o.refcount_); }
bool DeviceMemory2D::empty() const { return !data_; }
int DeviceMemory2D::colsBytes() const { return colsBytes_; }
int DeviceMemory2D::rows() const { return rows_; }
size_t DeviceMemory2D::step() const { return step_; }

// ------------------------------------------------------------------------------------------------------------------
// Intr, timers: precomp.cpp:7-21
Intr::Intr() {}
Intr::Intr(float fx_, float fy_, float cx_, float cy_) : fx(fx_), fy(fy_), cx(cx_), cy(cy_) {}
Intr Intr::operator()(int level_index) const { int div = 1 << level_index; return Intr(fx / div, fy / div, cx / div, cy / div); }
std::ostream& kfusion::operator<<(std::ostream& os, const Intr& intr)
{ return os << "([f = " << intr.fx << ", " << intr.fy << "] [cp = " << intr.cx << ", " << intr.cy << "])"; }

static double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
ScopeTime::ScopeTime(const char *name_) : name(name_), start(now_ms()) {}
ScopeTime::~ScopeTime() { std::cout << "Time(" << name << ") = " << (now_ms() - start) << "ms" << std::endl; }
SampledScopeTime::SampledScopeTime(double& time_ms) : time_ms_(time_ms), start(now_ms()) {}
double SampledScopeTime::getTime() { return now_ms() - start; }
SampledScopeTime::~SampledScopeTime()
{
    static int i_ = 0;
    time_ms_ += getTime();
    if (i_ % EACH == 0 && i_) { std::cout << "Average frame time = " << time_ms_ / EACH << "ms ( " << 1000.f * EACH / time_ms_ << "fps )" << std::endl; time_ms_ = 0.0; }
    ++i_;
}

static inline df_intr to_df(const Intr& i) { df_intr r = {i.fx, i.fy, i.cx, i.cy}; return r; }
static inline df_aff3f to_df(const Affine3f& a)
{
    df_aff3f r;
    for (int i = 0; i < 3; ++i) { for (int j = 0; j < 3; ++j) r.R[i * 3 + j] = a.matrix(i, j); r.t[i] = a.matrix(i, 3); }
    return r;
}
static inline Affine3f from12(const float *p)
{
    Affine3f a;
    for (int i = 0; i < 3; ++i) { for (int j = 0; j < 3; ++j) a.matrix(i, j) = p[i * 3 + j]; a.matrix(i, 3) = p[9 + i]; }
    return a;
}
static inline void to12(const Affine3f& a, float *p) { df_aff3f d = to_df(a); for (int i = 0; i < 9; ++i) p[i] = d.R[i]; for (int i = 0; i < 3; ++i) p[9 + i] = d.t[i]; }

// ------------------------------------------------------------------------------------------------------------------
// imgproc free functions: imgproc.cpp:10-201
void kfusion::cuda::waitAllDefaultStream() { cudaSafeCall(cudaDeviceSynchronize()); }
void kfusion::cuda::depthBilateralFilter(const Depth& in, Depth& out, int kernel_size, float sigma_spatial, float sigma_depth)
{
    out.create(in.rows(), in.cols());
    dfSafeCall(df_bilateral(in.ptr(), in.step(), in.cols(), in.rows(), out.ptr(), out.step(), kernel_size, sigma_spatial, sigma_depth, 0));
}
void kfusion::cuda::depthTruncation(Depth& depth, float threshold) { dfSafeCall(df_truncate_depth(depth.ptr(), depth.step(), depth.cols(), depth.rows(), threshold, 0)); }
void kfusion::cuda::depthBuildPyramid(const Depth& depth, Depth& pyramid, float sigma_depth)
{
    pyramid.create(depth.rows() / 2, depth.cols() / 2);
    dfSafeCall(df_pyr_down(depth.ptr(), depth.step(), depth.cols(), depth.rows(), pyramid.ptr(), pyramid.step(), sigma_depth, 0));
}
void kfusion::cuda::computePointNormals(const Intr& intr, const Depth& depth, Cloud& points, Normals& normals)
{
    points.create(depth.rows(), depth.cols());
    normals.create(depth.rows(), depth.cols());
    dfSafeCall(df_points_normals(to_df(intr), depth.ptr(), depth.step(), depth.cols(), depth.rows(), (float *)points.ptr(), points.step(),
                                 (float *)normals.ptr(), normals.step(), 0));
}
void kfusion::cuda::computeDists(const Depth& depth, Dists& dists, const Intr& intr)
{
    dists.create(depth.rows(), depth.cols());
    dfSafeCall(df_compute_dists(depth.ptr(), depth.step(), depth.cols(), depth.rows(), to_df(intr), dists.ptr(), dists.step(), 0));
}
void kfusion::cuda::resizePointsNormals(const Cloud& points, const Normals& normals, Cloud& points_out, Normals& normals_out)
{
    points_out.create(points.rows() / 2, points.cols() / 2);
    normals_out.create(normals.rows() / 2, normals.cols() / 2);
    dfSafeCall(df_resize_points_normals((const float *)points.ptr(), points.step(), (const float *)normals.ptr(), normals.step(), points.cols(), points.rows(),
                                        (float *)points_out.ptr(), points_out.step(), (float *)normals_out.ptr(), normals_out.step(), 0));
}
void kfusion::cuda::renderImage(const Cloud& points, const Normals& normals, const Intr& /*intr*/, const Vec3f& light_pose, Image& image)
{
    image.create(points.rows(), points.cols());
    dfSafeCall(df_render_image((const float *)points.ptr(), points.step(), (const float *)normals.ptr(), normals.step(), points.cols(), points.rows(),
                               light_pose.val, image.ptr(), image.step(), 0));
    waitAllDefaultStream();
}
void kfusion::cuda::renderTangentColors(const Normals& normals, Image& image)
{
    image.create(normals.rows(), normals.cols());
    dfSafeCall(df_render_tangent_colors((const float *)normals.ptr(), normals.step(), normals.cols(), normals.rows(), image.ptr(), image.step(), 0));
    waitAllDefaultStream();
}
// USE_DEPTH-path entry points of the reference (internal.hpp:6 leaves USE_DEPTH undefined, so its own frame loop never calls them);
// host wrappers as imgproc.cpp:52-60,98-103,112-121,152-164
void kfusion::cuda::computeNormalsAndMaskDepth(const Intr& intr, Depth& depth, Normals& normals)
{
    normals.create(depth.rows(), depth.cols());
    dfSafeCall(df_normals_mask_depth(to_df(intr), depth.ptr(), depth.step(), depth.cols(), depth.rows(), (float *)normals.ptr(), normals.step(), 0));
}
void kfusion::cuda::cloudToDepth(const Cloud& cloud, Depth& depth)
{
    depth.create(cloud.rows(), cloud.cols());
    dfSafeCall(df_cloud_to_depth((const float *)cloud.ptr(), cloud.step(), cloud.cols(), cloud.rows(), depth.ptr(), depth.step(), 0));
}
void kfusion::cuda::resizeDepthNormals(const Depth& depth, const Normals& normals, Depth& depth_out, Normals& normals_out)
{
    depth_out.create(depth.rows() / 2, depth.cols() / 2);
    normals_out.create(normals.rows() / 2, normals.cols() / 2);
    dfSafeCall(df_resize_depth_normals(depth.ptr(), depth.step(), (const float *)normals.ptr(), normals.step(), depth.cols(), depth.rows(),
                                       depth_out.ptr(), depth_out.step(), (float *)normals_out.ptr(), normals_out.step(), 0));
}
void kfusion::cuda::renderImage(const Depth& depth, const Normals& normals, const Intr& intr, const Vec3f& light_pose, Image& image)
{
    image.create(depth.rows(), depth.cols());
    dfSafeCall(df_render_image_depth(depth.ptr(), depth.step(), (const float *)normals.ptr(), normals.step(), depth.cols(), depth.rows(), to_df(intr),
                                     light_pose.val, image.ptr(), image.step(), 0));
    waitAllDefaultStream();
}

// ------------------------------------------------------------------------------------------------------------------
// ProjectiveICP: projective_icp.cpp:68-213
struct ProjectiveICP::StreamHelper
{
    float *T_dev; int *ok_dev; double *scratch; float *pinned;
    StreamHelper()
    {
        cudaSafeCall(cudaMalloc(&T_dev, 64)); cudaSafeCall(cudaMalloc(&ok_dev, 64));
        cudaSafeCall(cudaMalloc(&scratch, (size_t)DF_ICP_SCRATCH_DOUBLES * 8)); cudaSafeCall(cudaMallocHost(&pinned, 64));
    }
    ~StreamHelper() { cudaFree(T_dev); cudaFree(ok_dev); cudaFree(scratch); cudaFreeHost(pinned); }
};
ProjectiveICP::ProjectiveICP() : angle_thres_(deg2rad(20.f)), dist_thres_(0.1f)
{
    const int iters[] = {10, 5, 4, 0};
    setIterationsNum(std::vector<int>(iters, iters + 4));
    shelp_ = cv::Ptr<StreamHelper>(new StreamHelper());
}
ProjectiveICP::~ProjectiveICP() {}
float ProjectiveICP::getDistThreshold() const { return dist_thres_; }
void ProjectiveICP::setDistThreshold(float distance) { dist_thres_ = distance; }
float ProjectiveICP::getAngleThreshold() const { return angle_thres_; }
void ProjectiveICP::setAngleThreshold(float angle) { angle_thres_ = angle; }
void ProjectiveICP::setIterationsNum(const std::vector<int>& iters)
{
    if (iters.size() >= MAX_PYRAMID_LEVELS) iters_.assign(iters.begin(), iters.begin() + MAX_PYRAMID_LEVELS);
    else { iters_ = std::vector<int>(MAX_PYRAMID_LEVELS, 0); std::copy(iters.begin(), iters.end(), iters_.begin()); }
}
int ProjectiveICP::getUsedLevelsNum() const
{
    int i = MAX_PYRAMID_LEVELS - 1;
    for (; i >= 0 && !iters_[i]; --i) {}
    return i + 1;
}
bool ProjectiveICP::estimateTransform(Affine3f&, const Intr&, const Frame&, const Frame&) { CV_Assert(!"Not implemented"); return false; }
bool ProjectiveICP::estimateTransform(Affine3f& affine, const Intr& intr, const DepthPyr& dcurr, const NormalsPyr ncurr, const DepthPyr dprev, const NormalsPyr nprev)
{
    // the reference's compile-time USE_DEPTH alternative (projective_icp.cpp:126-167); always available here
    const int LEVELS = getUsedLevelsNum();
    const unsigned short *dc[MAX_PYRAMID_LEVELS], *dp[MAX_PYRAMID_LEVELS];
    const float *nc[MAX_PYRAMID_LEVELS], *np[MAX_PYRAMID_LEVELS];
    int cols[MAX_PYRAMID_LEVELS], rows[MAX_PYRAMID_LEVELS]; size_t dpitch[MAX_PYRAMID_LEVELS], npitch[MAX_PYRAMID_LEVELS];
    for (int i = 0; i < LEVELS; ++i) {
        dc[i] = (const unsigned short *)dcurr[i].ptr(); dp[i] = (const unsigned short *)dprev[i].ptr();
        nc[i] = (const float *)ncurr[i].ptr(); np[i] = (const float *)nprev[i].ptr();
        cols[i] = dcurr[i].cols(); rows[i] = dcurr[i].rows(); dpitch[i] = dcurr[i].step(); npitch[i] = ncurr[i].step();
        CV_Assert(dprev[i].step() == dpitch[i] && nprev[i].step() == npitch[i]);
    }
    StreamHelper& sh = *shelp_;
    dfSafeCall(df_icp_estimate_depth(dc, nc, dp, np, cols, rows, dpitch, npitch, LEVELS, &iters_[0], to_df(intr), dist_thres_, angle_thres_, sh.T_dev, sh.ok_dev, sh.scratch, 0));
    cudaSafeCall(cudaMemcpy(sh.pinned, sh.T_dev, 48, cudaMemcpyDeviceToHost));
    cudaSafeCall(cudaMemcpy(sh.pinned + 12, sh.ok_dev, 4, cudaMemcpyDeviceToHost));
    int ok; memcpy(&ok, sh.pinned + 12, 4);
    if (!ok) return false;
    affine = from12(sh.pinned);
    return true;
}
bool ProjectiveICP::estimateTransform(Affine3f& affine, const Intr& intr, const PointsPyr& vcurr, const NormalsPyr ncurr, const PointsPyr vprev, const NormalsPyr nprev)
{
    const int LEVELS = getUsedLevelsNum();
    const float *vc[MAX_PYRAMID_LEVELS], *nc[MAX_PYRAMID_LEVELS], *vp[MAX_PYRAMID_LEVELS], *np[MAX_PYRAMID_LEVELS];
    int cols[MAX_PYRAMID_LEVELS], rows[MAX_PYRAMID_LEVELS]; size_t pitch[MAX_PYRAMID_LEVELS];
    for (int i = 0; i < LEVELS; ++i) {
        vc[i] = (const float *)vcurr[i].ptr(); nc[i] = (const float *)ncurr[i].ptr(); vp[i] = (const float *)vprev[i].ptr(); np[i] = (const float *)nprev[i].ptr();
        cols[i] = vcurr[i].cols(); rows[i] = vcurr[i].rows(); pitch[i] = vcurr[i].step();
        CV_Assert(ncurr[i].step() == pitch[i] && vprev[i].step() == pitch[i] && nprev[i].step() == pitch[i]);
    }
    StreamHelper& sh = *shelp_;
    dfSafeCall(df_icp_estimate(vc, nc, vp, np, cols, rows, pitch, LEVELS, &iters_[0], to_df(intr), dist_thres_, angle_thres_, sh.T_dev, sh.ok_dev, sh.scratch, 0));
    cudaSafeCall(cudaMemcpy(sh.pinned, sh.T_dev, 48, cudaMemcpyDeviceToHost));
    cudaSafeCall(cudaMemcpy(sh.pinned + 12, sh.ok_dev, 4, cudaMemcpyDeviceToHost));
    int ok; memcpy(&ok, sh.pinned + 12, 4);
    if (!ok) return false;
    affine = from12(sh.pinned);
    return true;
}

// ------------------------------------------------------------------------------------------------------------------
// TsdfVolume: tsdf_volume.cpp
static df_volume vol_of(const DeviceMemory& data, const Vec3i& dims, const Vec3f& vsz, float trunc, float max_weight)
{
    df_volume v;
    v.data = (uint32_t *)data.ptr<uint32_t>();
    for (int i = 0; i < 3; ++i) { v.dims[i] = dims[i]; v.voxel_size[i] = vsz[i]; }
    v.trunc_dist = trunc; v.max_weight = (int)max_weight;
    return v;
}
TsdfVolume::TsdfVolume(const Vec3i& dims)
    : data_(), cloud_buffer_(0), cloud_(0), normal_buffer_(0), cloud_host_(0), normal_host_(0), trunc_dist_(0.03f), max_weight_(128), dims_(dims),
      size_(Vec3f::all(3.f)), pose_(Affine3f::Identity()), gradient_delta_factor_(0.75f), raycast_step_factor_(0.75f)
{ create(dims_); }
TsdfVolume::~TsdfVolume() { delete cloud_host_; delete cloud_buffer_; delete cloud_; delete normal_host_; delete normal_buffer_; }
void TsdfVolume::create(const Vec3i& dims)
{
    dims_ = dims;
    int voxels_number = dims_[0] * dims_[1] * dims_[2];
    data_.create((size_t)voxels_number * sizeof(int));
    setTruncDist(trunc_dist_);
    clear();
}
Vec3i TsdfVolume::getDims() const { return dims_; }
Vec3f TsdfVolume::getVoxelSize() const { return Vec3f(size_[0] / dims_[0], size_[1] / dims_[1], size_[2] / dims_[2]); }
const CudaData TsdfVolume::data() const { return data_; }
CudaData TsdfVolume::data() { return data_; }
Vec3f TsdfVolume::getSize() const { return size_; }
void TsdfVolume::setSize(const Vec3f& size) { size_ = size; setTruncDist(trunc_dist_); }
float TsdfVolume::getTruncDist() const { return trunc_dist_; }
void TsdfVolume::setTruncDist(float distance)
{
    Vec3f vsz = getVoxelSize();
    float max_coeff = std::max<float>(std::max<float>(vsz[0], vsz[1]), vsz[2]);
    trunc_dist_ = std::max(distance, 2.1f * max_coeff);
}
// KinFu's view: the frame loop extracted cloud + normals on the device (buffers 9 / 10); the reference's per-frame downloads
// (compute_points / compute_normals, kinfu.cpp:249-250,398-399) happen here, on first use after a frame
void TsdfVolume::refresh_host_clouds() const
{
    if (!pipeline_ || !host_clouds_stale_) return;
    host_clouds_stale_ = false;
    long long info[3];
    df_kinfu_get_info(pipeline_, info, 3);
    const int n = (int)info[2];
    *cloud_host_ = cv::Mat(1, n, CV_32FC4);
    *normal_host_ = cv::Mat(1, n, CV_32FC4);
    if (n > 0) {
        dfSafeCall(df_kinfu_read_buffer(pipeline_, 9, cloud_host_->ptr<Point>(), (size_t)n * sizeof(Point)));
        dfSafeCall(df_kinfu_read_buffer(pipeline_, 10, normal_host_->ptr<Normal>(), (size_t)n * sizeof(Normal)));
    }
}
cv::Mat TsdfVolume::get_cloud_host() const { refresh_host_clouds(); return *cloud_host_; }
cv::Mat TsdfVolume::get_normal_host() const { refresh_host_clouds(); return *normal_host_; }
cv::Mat* TsdfVolume::get_cloud_host_ptr() const { refresh_host_clouds(); return cloud_host_; }
cv::Mat* TsdfVolume::get_normal_host_ptr() const { refresh_host_clouds(); return normal_host_; }
int TsdfVolume::getMaxWeight() const { return (int)max_weight_; }
void TsdfVolume::setMaxWeight(int weight) { max_weight_ = (float)weight; }
Affine3f TsdfVolume::getPose() const { return pose_; }
void TsdfVolume::setPose(const Affine3f& pose) { pose_ = pose; }
float TsdfVolume::getRaycastStepFactor() const { return raycast_step_factor_; }
void TsdfVolume::setRaycastStepFactor(float factor) { raycast_step_factor_ = factor; }
float TsdfVolume::getGradientDeltaFactor() const { return gradient_delta_factor_; }
void TsdfVolume::setGradientDeltaFactor(float factor) { gradient_delta_factor_ = factor; }
Vec3i TsdfVolume::getGridOrigin() const { return Vec3i(0, 0, 0); }      // declared but never defined by the reference
void TsdfVolume::setGridOrigin(const Vec3i&) {}
void TsdfVolume::swap(CudaData& data) { data_.swap(data); }
void TsdfVolume::applyAffine(const Affine3f& affine) { pose_ = affine * pose_; }
void TsdfVolume::clear()
{
    delete cloud_buffer_; delete cloud_; delete normal_buffer_; delete cloud_host_; delete normal_host_;    // the reference leaks these on every clear()
    cloud_buffer_ = new cuda::DeviceArray<Point>();
    cloud_ = new cuda::DeviceArray<Point>();
    normal_buffer_ = new cuda::DeviceArray<Normal>();
    cloud_host_ = new cv::Mat();
    normal_host_ = new cv::Mat();
    dfSafeCall(df_clear_volume(vol_of(data_, dims_, getVoxelSize(), trunc_dist_, max_weight_), 0));
}
void TsdfVolume::integrate(const Dists& dists, const Affine3f& camera_pose, const Intr& intr)
{
    Affine3f vol2cam = camera_pose.inv() * pose_;
    // activity_ != 0: this is KinFu's view of the frame loop's volume, whose extraction trusts the activity map (dfusion.h)
    dfSafeCall(df_integrate_tracked(vol_of(data_, dims_, getVoxelSize(), trunc_dist_, max_weight_), dists.ptr(), dists.step(), dists.cols(), dists.rows(),
                                    to_df(vol2cam), to_df(intr), 0, activity_, 0, 0));
    cudaSafeCall(cudaDeviceSynchronize());                                // the reference's launcher synchronises (tsdf_volume.cu:160)
}
// depth variant (tsdf_volume.cu:273-339,441-456): the same march; on a hit the reference stores static_cast<ushort>(vertex.z * 1000) of the
// camera-frame vertex and 0 elsewhere -- i.e. the points variant followed by cloud_to_depth's conversion (NaN -> 0)
void TsdfVolume::raycast(const Affine3f& camera_pose, const Intr& intr, Depth& depth, Normals& normals)
{
    Cloud points;
    points.create(depth.rows(), depth.cols());
    raycast(camera_pose, intr, points, normals);
    dfSafeCall(df_cloud_to_depth((const float *)points.ptr(), points.step(), points.cols(), points.rows(), depth.ptr(), depth.step(), 0));
    cudaSafeCall(cudaDeviceSynchronize());
}
void TsdfVolume::raycast(const Affine3f& camera_pose, const Intr& intr, Cloud& points, Normals& normals)
{
    Affine3f cam2vol = pose_.inv() * camera_pose;
    Mat3f Rinv = cam2vol.rotation().inv(cv::DECOMP_SVD);
    dfSafeCall(df_raycast_points(vol_of(data_, dims_, getVoxelSize(), trunc_dist_, max_weight_), to_df(cam2vol), Rinv.val, to_df(intr), points.cols(), points.rows(),
                                 raycast_step_factor_, gradient_delta_factor_, (float *)points.ptr(), points.step(), (float *)normals.ptr(), normals.step(), 0));
}
DeviceArray<Point> TsdfVolume::fetchCloud(DeviceArray<Point>& cloud_buffer) const
{
    enum { DEFAULT_CLOUD_BUFFER_SIZE = 256 * 256 * 256 };
    if (cloud_buffer.empty()) cloud_buffer.create(DEFAULT_CLOUD_BUFFER_SIZE);
    const df_volume v = vol_of(data_, dims_, getVoxelSize(), trunc_dist_, max_weight_);
    workspace_.create(df_extract_workspace_bytes(v));
    count_.create(64);
    dfSafeCall(df_extract_cloud(v, to_df(pose_), (float *)cloud_buffer.ptr(), (int)cloud_buffer.size(), count_.ptr<int>(), workspace_.ptr<void>(), 0));
    int size = 0;
    cudaSafeCall(cudaMemcpy(&size, count_.ptr<int>(), sizeof(int), cudaMemcpyDeviceToHost));      // cudaMemcpyFromSymbol in the reference (:813)
    return DeviceArray<Point>((Point *)cloud_buffer.ptr(), (size_t)size);
}
void TsdfVolume::fetchNormals(const DeviceArray<Point>& cloud, DeviceArray<Normal>& normals) const
{
    normals.create(cloud.size());
    if (cloud.size() == 0) return;
    Mat3f Rinv = pose_.rotation().inv(cv::DECOMP_SVD);
    dfSafeCall(df_extract_normals(vol_of(data_, dims_, getVoxelSize(), trunc_dist_, max_weight_), (const float *)cloud.ptr(), (int)cloud.size(), 0, to_df(pose_),
                                  Rinv.val, gradient_delta_factor_, (float *)normals.ptr(), 0));
    cudaSafeCall(cudaDeviceSynchronize());
}
void TsdfVolume::fetchMesh(DeviceArray<Point>& vertices, DeviceArray<Normal>& normals, DeviceArray<int>& triangles) const
{
    const df_volume v = vol_of(data_, dims_, getVoxelSize(), trunc_dist_, max_weight_);
    DeviceMemory ws(df_extract_mesh_workspace_bytes(v)), counts(64), keys;
    for (;;) {     // the counts are the true totals: a second call with the arrays resized to them fits exactly
        keys.create(std::max<size_t>(vertices.size(), 1) * sizeof(uint32_t));
        dfSafeCall(df_extract_mesh(v, to_df(pose_), activity_, (float *)vertices.ptr(), keys.ptr<uint32_t>(), (int)vertices.size(), triangles.ptr(),
                                   (int)(triangles.size() / 3), counts.ptr<int>(), ws.ptr<void>(), 0));
        int c[2];
        cudaSafeCall(cudaMemcpy(c, counts.ptr<int>(), sizeof c, cudaMemcpyDeviceToHost));
        if ((size_t)c[0] == vertices.size() && (size_t)c[1] * 3 == triangles.size()) break;
        if (c[0]) vertices.create(c[0]); else vertices.release();
        if (c[1]) triangles.create((size_t)c[1] * 3); else triangles.release();
    }
    fetchNormals(vertices, normals);
}
void TsdfVolume::compute_points()
{
    *cloud_ = fetchCloud(*cloud_buffer_);
    *cloud_host_ = cv::Mat(1, (int)cloud_->size(), CV_32FC4);
    if (cloud_->size()) cloud_->download(cloud_host_->ptr<Point>());
}
void TsdfVolume::compute_normals()
{
    fetchNormals(*cloud_, *normal_buffer_);
    *normal_host_ = cv::Mat(1, (int)cloud_->size(), CV_32FC4);
    if (cloud_->size()) normal_buffer_->download(normal_host_->ptr<Normal>());
}
float TsdfVolume::weighting(const std::vector<float>& dist_sqr, int k) const
{
    float distances = 0;
    for (size_t i = 0; i < dist_sqr.size(); ++i) distances += std::sqrt(dist_sqr[i]);
    return distances / k;
}
std::vector<float> TsdfVolume::psdf(const std::vector<Vec3f>& warped, Dists& dists, const Intr& intr)
{
    std::vector<Point> pts(warped.size());
    for (size_t i = 0; i < warped.size(); ++i) { pts[i].x = warped[i][0]; pts[i].y = warped[i][1]; pts[i].z = warped[i][2]; pts[i].data[3] = 0.f; }
    Cloud points;
    points.upload(pts, dists.cols());
    DeviceMemory ws(df_project_workspace_bytes(dists.cols(), dists.rows()));
    cudaSafeCall(cudaMemset(ws.ptr<void>(), 0, ws.sizeBytes()));
    dfSafeCall(df_project_and_remove(dists.ptr(), dists.step(), dists.cols(), dists.rows(), to_df(intr), (float *)points.ptr(), points.step(), points.cols(), points.rows(),
                                     ws.ptr<void>(), 0));
    int cols;
    points.download(pts, cols);
    Mat3f K = Mat3f(intr.fx, 0, intr.cx, 0, intr.fy, intr.cy, 0, 0, 1).inv();
    std::vector<float> distances(warped.size());
    for (size_t i = 0; i < warped.size(); ++i) distances[i] = (K * Vec3f(pts[i].x, pts[i].y, pts[i].z))[2] - warped[i][2];
    return distances;
}
void TsdfVolume::surface_fusion(const WarpField&, std::vector<Vec3f> warped, std::vector<Vec3f> /*canonical*/, cuda::Depth& depth,
                                const Affine3f& camera_pose, const Intr& intr)
{
    std::vector<float> ro = psdf(warped, depth, intr);
    (void)ro;                       // the reference's per-point k-NN loop computes weights it never uses (tsdf_volume.cpp:241-254)
    cuda::Dists dists;
    cuda::computeDists(depth, dists, intr);
    integrate(dists, camera_pose, intr);
}

void TsdfVolume::integrate(const Depth& depth, const WarpField& warp_field, const Affine3f& camera_pose, const Intr& intr, float weight_scale)
{
    warp_field.uploadNodes();
    const Affine3f world2cam = camera_pose.inv() * warp_field.getWarpToLive();       // WarpField::warp applies warp_to_live_ last (warp_field.cpp:191)
    dfSafeCall(df_integrate_warped(vol_of(data_, dims_, getVoxelSize(), trunc_dist_, max_weight_), depth.ptr(), depth.step(), depth.cols(), depth.rows(),
                                   to_df(pose_), to_df(world2cam), to_df(intr), warp_field.deviceNodes(), warp_field.deviceNodeCount(), warp_field.deviceGrid(),
                                   weight_scale, 0, activity_, 0, 0));
    cudaSafeCall(cudaDeviceSynchronize());                                           // as device::integrate does (tsdf_volume.cu:160)
}

// ------------------------------------------------------------------------------------------------------------------
// WarpField: warp_field.cpp
struct WarpField::Impl
{
    mutable float *nodes_dev = 0; mutable void *grid_dev = 0; mutable int M = 0; mutable int cap = 0;
    mutable bool owns = true;
    mutable std::vector<float> host12;
    mutable std::vector<float> out_dist_sqr_;
    mutable std::vector<size_t> ret_index_;
    ~Impl() { if (owns) { cudaFree(nodes_dev); cudaFree(grid_dev); } }
};
WarpField::WarpField() : nodes_(new std::vector<deformation_node>()), impl_(new Impl()), warp_to_live_(Affine3f())
{
    impl_->ret_index_ = std::vector<size_t>(KNN_NEIGHBOURS);
    impl_->out_dist_sqr_ = std::vector<float>(KNN_NEIGHBOURS);
}
WarpField::~WarpField() { delete nodes_; delete impl_; }
static void node_to12(const deformation_node& n, float *o)
{
    // the dual part is private to DualQuaternion: reconstruct it from the public accessors (0.5 * (0,t) * r, dual_quaternion.hpp:82-85)
    utils::Quaternion<float> r = n.transform.getRotation();
    float tx, ty, tz; n.transform.getTranslation(tx, ty, tz);
    utils::Quaternion<float> d = 0.5 * utils::Quaternion<float>(0, tx, ty, tz) * r;
    o[0] = n.vertex[0]; o[1] = n.vertex[1]; o[2] = n.vertex[2];
    o[3] = r.w_; o[4] = r.x_; o[5] = r.y_; o[6] = r.z_;
    o[7] = d.w_; o[8] = d.x_; o[9] = d.y_; o[10] = d.z_;
    o[11] = n.weight;
}
void WarpField::init(const cv::Mat& first_frame)
{
    // every 50th point of the 1 x P extracted cloud becomes a node (warp_field.cpp:41-62); only the filled nodes are kept here
    nodes_->clear();
    const int step = 50;
    for (int i = 0; i < first_frame.rows; i += step)
        for (int j = 0; j < first_frame.cols; j += step) {
            const Point& p = first_frame.at<Point>(i, j);
            if (!std::isnan(p.x)) {
                deformation_node n;
                n.transform = utils::DualQuaternion<float>();
                n.vertex = Vec3f(p.x, p.y, p.z);
                n.weight = 3 * 1.f;                                   // voxel_size forced to 1 (warp_field.cpp:48)
                nodes_->push_back(n);
            }
        }
    buildKDTree();
}
void WarpField::init(const std::vector<Vec3f>& first_frame)
{
    nodes_->clear();
    nodes_->resize(first_frame.size());
    for (size_t i = 0; i < first_frame.size(); ++i)
        if (!std::isnan(first_frame[i][0])) {
            nodes_->at(i).transform = utils::DualQuaternion<float>();
            nodes_->at(i).vertex = first_frame[i];
            nodes_->at(i).weight = 3 * 1.f;
        }
    buildKDTree();
}
void WarpField::energy(const cuda::Cloud &frame, const cuda::Normals &normals, const Affine3f&, const cuda::TsdfVolume&,
                       const std::vector<std::pair<utils::DualQuaternion<float>, utils::DualQuaternion<float>>>&)
{ CV_Assert(normals.cols() == frame.cols()); CV_Assert(normals.rows() == frame.rows()); }
void WarpField::energy_reg(const std::vector<std::pair<utils::DualQuaternion<float>, utils::DualQuaternion<float>>>&) {}
void WarpField::energy_data(const std::vector<Vec3f> &canonical_vertices, const std::vector<Vec3f> &canonical_normals,
                            const std::vector<Vec3f> &live_vertices, const std::vector<Vec3f> &live_normals)
{
    // the reference solves the same translation-only data term with Ceres here (warp_field.cpp:117-163); this build has one solver
    CombinedSolverParameters p; p.numIter = 1; p.nonLinearIter = 15; p.linearIter = 250; p.earlyOut = true;
    CombinedSolver s(this, p);
    s.initializeProblemInstance(canonical_vertices, canonical_normals, live_vertices, live_normals);
    s.solveAll();
}
void WarpField::uploadNodes() const
{
    Impl& I = *impl_;
    if (!I.owns) return;                                                      // KinFu's table is authoritative
    const int M = (int)nodes_->size();
    std::vector<float> h((size_t)M * DF_NODE_STRIDE);
    for (int i = 0; i < M; ++i) node_to12(nodes_->at(i), &h[(size_t)i * DF_NODE_STRIDE]);
    bool vertices_changed = (M != I.M) || I.host12.size() != h.size();
    if (!vertices_changed)
        for (int i = 0; i < M && !vertices_changed; ++i)
            for (int c = 0; c < 3; ++c) vertices_changed |= h[(size_t)i * DF_NODE_STRIDE + c] != I.host12[(size_t)i * DF_NODE_STRIDE + c];
    if (M > I.cap) {
        cudaFree(I.nodes_dev); cudaFree(I.grid_dev);
        I.cap = M;
        cudaSafeCall(cudaMalloc(&I.nodes_dev, (size_t)I.cap * DF_NODE_STRIDE * 4));
        cudaSafeCall(cudaMalloc(&I.grid_dev, df_node_grid_bytes(I.cap)));
        vertices_changed = true;
    }
    I.M = M;
    if (M == 0) return;
    if (h != I.host12) cudaSafeCall(cudaMemcpy(I.nodes_dev, &h[0], h.size() * 4, cudaMemcpyHostToDevice));
    if (vertices_changed) dfSafeCall(df_build_node_grid(I.nodes_dev, M, I.grid_dev, 0));
    I.host12.swap(h);
}
void WarpField::downloadTranslations()
{
    Impl& I = *impl_;
    const int M = I.M;
    if (M == 0) return;
    std::vector<float> h((size_t)M * DF_NODE_STRIDE);
    cudaSafeCall(cudaMemcpy(&h[0], I.nodes_dev, h.size() * 4, cudaMemcpyDeviceToHost));
    if ((int)nodes_->size() != M) {                                           // adopted table (KinFu): rebuild the host view
        nodes_->assign(M, deformation_node());
        for (int i = 0; i < M; ++i) {
            const float *n = &h[(size_t)i * DF_NODE_STRIDE];
            nodes_->at(i).vertex = Vec3f(n[0], n[1], n[2]);
            nodes_->at(i).weight = n[11];
        }
    }
    for (int i = 0; i < M; ++i) {
        const float *n = &h[(size_t)i * DF_NODE_STRIDE];
        // translation = 2 * dual * conj(rotation) with a unit rotation; set through the public API like CombinedSolver.h:189-197
        utils::Quaternion<float> rot(n[3], n[4], n[5], n[6]);
        utils::Quaternion<float> t = 2 * utils::Quaternion<float>(n[7], n[8], n[9], n[10]) * rot.conjugate();
        nodes_->at(i).transform.encodeTranslation(t.x_, t.y_, t.z_);
    }
    I.host12.swap(h);
}
float *WarpField::deviceNodes() const { return impl_->nodes_dev; }
void *WarpField::deviceGrid() const { return impl_->grid_dev; }
int WarpField::deviceNodeCount() const { return impl_->M; }
void WarpField::adoptDeviceNodes(float *nodes_dev, void *grid_dev, int M)
{
    Impl& I = *impl_;
    if (I.owns) { cudaFree(I.nodes_dev); cudaFree(I.grid_dev); }
    I.owns = false; I.nodes_dev = nodes_dev; I.grid_dev = grid_dev; I.M = M; I.cap = M; I.host12.clear();
}
void WarpField::warp(std::vector<Vec3f>& points, std::vector<Vec3f>& normals) const
{
    uploadNodes();
    const int N = (int)points.size();
    if (N == 0 || impl_->M == 0) return;
    CV_Assert(normals.size() >= points.size());
    DeviceMemory p((size_t)N * 12), n((size_t)N * 12);
    cudaSafeCall(cudaMemcpy(p.ptr<void>(), &points[0], (size_t)N * 12, cudaMemcpyHostToDevice));
    cudaSafeCall(cudaMemcpy(n.ptr<void>(), &normals[0], (size_t)N * 12, cudaMemcpyHostToDevice));
    dfSafeCall(df_warp(impl_->nodes_dev, impl_->M, impl_->grid_dev, p.ptr<float>(), n.ptr<float>(), N, 3, to_df(warp_to_live_), 0, 0, 0, 0));
    cudaSafeCall(cudaMemcpy(&points[0], p.ptr<void>(), (size_t)N * 12, cudaMemcpyDeviceToHost));
    cudaSafeCall(cudaMemcpy(&normals[0], n.ptr<void>(), (size_t)N * 12, cudaMemcpyDeviceToHost));
}
void WarpField::KNN(Vec3f point) const
{
    uploadNodes();
    DeviceMemory q(12), idx(32), d2(32);
    cudaSafeCall(cudaMemcpy(q.ptr<void>(), point.val, 12, cudaMemcpyHostToDevice));
    dfSafeCall(df_knn8(impl_->nodes_dev, impl_->M, impl_->grid_dev, q.ptr<float>(), 1, 3, idx.ptr<int32_t>(), d2.ptr<float>(), 0));
    int32_t hi[8];
    cudaSafeCall(cudaMemcpy(hi, idx.ptr<void>(), 32, cudaMemcpyDeviceToHost));
    cudaSafeCall(cudaMemcpy(&impl_->out_dist_sqr_[0], d2.ptr<void>(), 32, cudaMemcpyDeviceToHost));
    for (int i = 0; i < KNN_NEIGHBOURS; ++i) impl_->ret_index_[i] = hi[i] < 0 ? 0 : (size_t)hi[i];
}
float WarpField::weighting(float squared_dist, float weight) const { return (float)exp(-squared_dist / (2 * weight * weight)); }
void WarpField::getWeightsAndUpdateKNN(const Vec3f& vertex, float weights[KNN_NEIGHBOURS]) const
{
    KNN(vertex);
    for (size_t i = 0; i < KNN_NEIGHBOURS; i++) weights[i] = weighting(impl_->out_dist_sqr_[i], nodes_->at(impl_->ret_index_[i]).weight);
}
utils::DualQuaternion<float> WarpField::DQB(const Vec3f& vertex) const
{
    float weights[KNN_NEIGHBOURS];
    getWeightsAndUpdateKNN(vertex, weights);
    utils::Quaternion<float> translation_sum(0, 0, 0, 0), rotation_sum(0, 0, 0, 0);
    for (size_t i = 0; i < KNN_NEIGHBOURS; i++) {
        translation_sum += weights[i] * nodes_->at(impl_->ret_index_[i]).transform.getTranslation();
        rotation_sum += weights[i] * nodes_->at(impl_->ret_index_[i]).transform.getRotation();
    }
    rotation_sum.normalize();
    return utils::DualQuaternion<float>(translation_sum, rotation_sum);
}
const std::vector<deformation_node>* WarpField::getNodes() const { return nodes_; }
std::vector<deformation_node>* WarpField::getNodes() { return nodes_; }
void WarpField::buildKDTree() { uploadNodes(); }
const cv::Mat WarpField::getNodesAsMat() const
{
    if (!impl_->owns) const_cast<WarpField *>(this)->downloadTranslations();
    cv::Mat matrix(1, (int)nodes_->size(), CV_32FC3);
    for (size_t i = 0; i < nodes_->size(); i++) {
        nodes_->at(i).transform.getTranslation(matrix.at<cv::Vec3f>((int)i));
        matrix.at<cv::Vec3f>((int)i) += nodes_->at(i).vertex;
    }
    return matrix;
}
int WarpField::extend(const cv::Mat& cloud, float radius, int step, int max_nodes)
{
    uploadNodes();
    Impl& I = *impl_;
    const int M = I.M, P = cloud.cols * cloud.rows;
    if (M <= 0 || P <= 0 || max_nodes <= M || !I.owns) return M;       // (KinFu's own table is extended by DF_KINFU_EXTEND_FIELD)
    DeviceMemory table((size_t)max_nodes * DF_NODE_STRIDE * 4), pts((size_t)P * 16), ws(df_extend_field_workspace_bytes(P)), m_out(64);
    cudaSafeCall(cudaMemcpy(table.ptr<void>(), I.nodes_dev, (size_t)M * DF_NODE_STRIDE * 4, cudaMemcpyDeviceToDevice));
    cudaSafeCall(cudaMemcpy(pts.ptr<void>(), cloud.ptr<float>(), (size_t)P * 16, cudaMemcpyHostToDevice));
    dfSafeCall(df_extend_field(table.ptr<float>(), M, max_nodes, I.grid_dev, pts.ptr<float>(), P, 0, 4, radius, step, m_out.ptr<int>(), ws.ptr<void>(), 0));
    int Mn = M;
    cudaSafeCall(cudaMemcpy(&Mn, m_out.ptr<void>(), sizeof(int), cudaMemcpyDeviceToHost));
    if (Mn > M) {
        std::vector<float> added((size_t)(Mn - M) * DF_NODE_STRIDE);
        cudaSafeCall(cudaMemcpy(&added[0], table.ptr<float>() + (size_t)M * DF_NODE_STRIDE, added.size() * 4, cudaMemcpyDeviceToHost));
        for (int i = 0; i < Mn - M; ++i) {
            deformation_node n;
            n.transform = utils::DualQuaternion<float>();
            n.vertex = Vec3f(added[(size_t)i * DF_NODE_STRIDE], added[(size_t)i * DF_NODE_STRIDE + 1], added[(size_t)i * DF_NODE_STRIDE + 2]);
            n.weight = added[(size_t)i * DF_NODE_STRIDE + 11];
            nodes_->push_back(n);
        }
        buildKDTree();
    }
    return Mn;
}
void WarpField::clear()
{
    // the reference's clear() is an empty stub (warp_field.cpp:298-301); here it really drops the field, so that a tracking-loss
    // reset cannot leave a stale field behind (KinFu::reset calls it, kinfu.cpp:206)
    nodes_->clear();
    Impl& I = *impl_;
    if (I.owns) { cudaFree(I.nodes_dev); cudaFree(I.grid_dev); }
    I.nodes_dev = 0; I.grid_dev = 0; I.M = 0; I.cap = 0; I.owns = true;
    I.host12.clear();
}
void WarpField::setWarpToLive(const Affine3f &pose) { warp_to_live_ = pose; }
std::vector<float>* WarpField::getDistSquared() const { return &impl_->out_dist_sqr_; }
std::vector<size_t>* WarpField::getRetIndex() const { return &impl_->ret_index_; }

// ------------------------------------------------------------------------------------------------------------------
// CombinedSolver / WarpFieldOptimiser: CombinedSolver.h, warp_field_optimiser.cpp
struct CombinedSolver::Impl
{
    std::vector<cv::Vec3f> canon, live;
    DeviceMemory ws, stats;
};
CombinedSolver::CombinedSolver(kfusion::WarpField *warpField, CombinedSolverParameters params)
    : m_warp(warpField), m_combinedSolverParameters(params), impl_(new Impl()) {}
CombinedSolver::~CombinedSolver() { delete impl_; }
void CombinedSolver::initializeProblemInstance(const std::vector<cv::Vec3f> &canonical_vertices, const std::vector<cv::Vec3f> &,
                                               const std::vector<cv::Vec3f> &live_vertices, const std::vector<cv::Vec3f> &)
{ impl_->canon = canonical_vertices; impl_->live = live_vertices; }
void CombinedSolver::solveAll()
{
    m_warp->uploadNodes();
    const int N = (int)impl_->canon.size(), M = m_warp->deviceNodeCount();
    if (N == 0 || M == 0) return;
    DeviceMemory c((size_t)N * 12), l((size_t)N * 12);
    cudaSafeCall(cudaMemcpy(c.ptr<void>(), &impl_->canon[0], (size_t)N * 12, cudaMemcpyHostToDevice));
    cudaSafeCall(cudaMemcpy(l.ptr<void>(), &impl_->live[0], (size_t)N * 12, cudaMemcpyHostToDevice));
    impl_->ws.create(df_solve_workspace_bytes(M, N));
    impl_->stats.create(64);
    // CombinedSolverBase::solveAll (deps/Opt/examples/shared/CombinedSolverBase.h:98-119): numIter passes, one when earlyOut
    const unsigned passes = m_combinedSolverParameters.earlyOut ? 1u : std::max(1u, m_combinedSolverParameters.numIter);
    for (unsigned it = 0; it < passes; ++it)
        dfSafeCall(df_solve_data_term(m_warp->deviceNodes(), M, m_warp->deviceGrid(), c.ptr<float>(), l.ptr<float>(), N, 3,
                                      (int)m_combinedSolverParameters.nonLinearIter, (int)m_combinedSolverParameters.linearIter, 0,
                                      impl_->stats.ptr<double>(), impl_->ws.ptr<void>(), 0));
    double st[8];
    cudaSafeCall(cudaMemcpy(st, impl_->stats.ptr<void>(), 64, cudaMemcpyDeviceToHost));
    last_cost_ = st[1];
    if (st[5] != 0.0)
        std::cerr << "CombinedSolver: a normal-matrix row exceeded the row capacity of df_solve_data_term; the warp field was left unchanged" << std::endl;
    m_warp->downloadTranslations();                                           // copyResultToCPUFromFloat3, CombinedSolver.h:189-197
}
WarpFieldOptimiser::WarpFieldOptimiser(WarpField *warp, CombinedSolver *solver) : warp_(warp), solver_(solver) {}
WarpFieldOptimiser::WarpFieldOptimiser(WarpField *warp, CombinedSolverParameters params) : warp_(warp) { solver_ = new CombinedSolver(warp, params); }
void WarpFieldOptimiser::optimiseWarpData(const std::vector<Vec3f> &canonical_vertices, const std::vector<Vec3f> &canonical_normals,
                                          const std::vector<Vec3f> &live_vertices, const std::vector<Vec3f> &live_normals)
{
    solver_->initializeProblemInstance(canonical_vertices, canonical_normals, live_vertices, live_normals);
    solver_->solveAll();
}

// ------------------------------------------------------------------------------------------------------------------
// KinFuParams / KinFu: kinfu.cpp
static KinFuParams params_from(const df_kinfu_params& d)
{
    KinFuParams p;
    p.cols = d.cols; p.rows = d.rows;
    p.intr = Intr(d.intr.fx, d.intr.fy, d.intr.cx, d.intr.cy);
    p.volume_dims = Vec3i(d.volume_dims[0], d.volume_dims[1], d.volume_dims[2]);
    p.volume_size = Vec3f(d.volume_size[0], d.volume_size[1], d.volume_size[2]);
    float a[12]; for (int i = 0; i < 9; ++i) a[i] = d.volume_pose.R[i]; for (int i = 0; i < 3; ++i) a[9 + i] = d.volume_pose.t[i];
    p.volume_pose = from12(a);
    p.bilateral_sigma_depth = d.bilateral_sigma_depth; p.bilateral_sigma_spatial = d.bilateral_sigma_spatial; p.bilateral_kernel_size = d.bilateral_kernel_size;
    p.icp_truncate_depth_dist = d.icp_truncate_depth_dist; p.icp_dist_thres = d.icp_dist_thres; p.icp_angle_thres = d.icp_angle_thres;
    p.icp_iter_num.assign(d.icp_iter_num, d.icp_iter_num + 4);
    p.tsdf_min_camera_movement = d.tsdf_min_camera_movement; p.tsdf_trunc_dist = d.tsdf_trunc_dist; p.tsdf_max_weight = d.tsdf_max_weight;
    p.raycast_step_factor = d.raycast_step_factor; p.gradient_delta_factor = d.gradient_delta_factor;
    p.light_pose = Vec3f(d.light_pose[0], d.light_pose[1], d.light_pose[2]);
    return p;
}
static df_kinfu_params params_to(const KinFuParams& p)
{
    df_kinfu_params d;
    df_kinfu_default_params(&d, 0);
    d.cols = p.cols; d.rows = p.rows; d.intr = to_df(p.intr);
    for (int i = 0; i < 3; ++i) { d.volume_dims[i] = p.volume_dims[i]; d.volume_size[i] = p.volume_size[i]; d.light_pose[i] = p.light_pose[i]; }
    d.volume_pose = to_df(p.volume_pose);
    d.bilateral_sigma_depth = p.bilateral_sigma_depth; d.bilateral_sigma_spatial = p.bilateral_sigma_spatial; d.bilateral_kernel_size = p.bilateral_kernel_size;
    d.icp_truncate_depth_dist = p.icp_truncate_depth_dist; d.icp_dist_thres = p.icp_dist_thres; d.icp_angle_thres = p.icp_angle_thres;
    for (int i = 0; i < 4; ++i) d.icp_iter_num[i] = i < (int)p.icp_iter_num.size() ? p.icp_iter_num[i] : 0;
    d.tsdf_min_camera_movement = p.tsdf_min_camera_movement; d.tsdf_trunc_dist = p.tsdf_trunc_dist; d.tsdf_max_weight = p.tsdf_max_weight;
    d.raycast_step_factor = p.raycast_step_factor; d.gradient_delta_factor = p.gradient_delta_factor;
    d.flags |= p.dfusion_flags & (DF_KINFU_WARPED_INTEGRATE | DF_KINFU_EXTEND_FIELD);
    d.fusion_weight_scale = p.fusion_weight_scale; d.extend_radius = p.extend_radius;
    return d;
}
KinFuParams KinFuParams::default_params_dynamicfusion() { df_kinfu_params d; df_kinfu_default_params(&d, 0); return params_from(d); }
KinFuParams KinFuParams::default_params() { df_kinfu_params d; df_kinfu_default_params(&d, 1); return params_from(d); }

static void *buffer_of(void *h, int which, size_t *pitch = 0, int *cols = 0, int *rows = 0)
{
    void *ptr; size_t pi; int c, r;
    dfSafeCall(df_kinfu_get_buffer(h, which, &ptr, &pi, &c, &r));
    if (pitch) *pitch = pi; if (cols) *cols = c; if (rows) *rows = r;
    return ptr;
}

KinFu::KinFu(const KinFuParams& params) : frame_counter_(0), params_(params), handle_(0)
{
    CV_Assert(params.volume_dims[0] % 32 == 0);
    df_kinfu_params d = params_to(params_);
    handle_ = df_kinfu_create(&d);
    if (!handle_) kfusion::cuda::error("df_kinfu_create failed", __FILE__, __LINE__);
    // component views over the pipeline's device state, so tsdf() / icp() / getWarp() behave like the reference's members
    volume_ = cv::Ptr<cuda::TsdfVolume>(new cuda::TsdfVolume(Vec3i(32, 32, 32)));
    {   // re-point the view at the pipeline's volume (non-owning DeviceMemory, device_memory.cpp:49); create() with the real
        // dims is then a no-op allocation-wise because the byte size already matches (device_memory.cpp:73-76)
        CudaData view(buffer_of(handle_, 0), (size_t)params_.volume_dims[0] * params_.volume_dims[1] * params_.volume_dims[2] * 4);
        volume_->swap(view);
        volume_->create(params_.volume_dims);
    }
    volume_->setTruncDist(params_.tsdf_trunc_dist);
    volume_->setMaxWeight(params_.tsdf_max_weight);
    volume_->setSize(params_.volume_size);
    volume_->setPose(params_.volume_pose);
    volume_->setRaycastStepFactor(params_.raycast_step_factor);
    volume_->setGradientDeltaFactor(params_.gradient_delta_factor);
    volume_->activity_ = (unsigned char *)buffer_of(handle_, 14);      // the view's integrations stay visible to the loop's extraction
    volume_->pipeline_ = handle_;
    warp_ = cv::Ptr<WarpField>(new WarpField());
    icp_ = cv::Ptr<cuda::ProjectiveICP>(new cuda::ProjectiveICP());
    icp_->setDistThreshold(params_.icp_dist_thres);
    icp_->setAngleThreshold(params_.icp_angle_thres);
    icp_->setIterationsNum(params_.icp_iter_num);
    CombinedSolverParameters solverParameters;                          // kinfu.cpp:114-120
    solverParameters.numIter = 5; solverParameters.nonLinearIter = 5; solverParameters.linearIter = 100;
    solverParameters.useOpt = false; solverParameters.useOptLM = true; solverParameters.earlyOut = true;
    optimiser_ = new WarpFieldOptimiser(warp_, solverParameters);
    allocate_buffers();
    poses_.clear();
    poses_.push_back(Affine3f::Identity());
}
KinFu::~KinFu() { df_kinfu_destroy(handle_); }
const KinFuParams& KinFu::params() const { return params_; }
KinFuParams& KinFu::params() { return params_; }
const cuda::TsdfVolume& KinFu::tsdf() const { return *volume_; }
cuda::TsdfVolume& KinFu::tsdf() { return *volume_; }
const cuda::ProjectiveICP& KinFu::icp() const { return *icp_; }
cuda::ProjectiveICP& KinFu::icp() { return *icp_; }
const WarpField& KinFu::getWarp() const { return *warp_; }
WarpField& KinFu::getWarp() { return *warp_; }
void KinFu::allocate_buffers()
{
    depths_.create(params_.rows, params_.cols);
    normals_.create(params_.rows, params_.cols);
    points_.create(params_.rows, params_.cols);
}
void KinFu::reset()
{
    if (frame_counter_) std::cout << "Reset" << std::endl;
    frame_counter_ = 0;
    poses_.clear();
    poses_.reserve(30000);
    poses_.push_back(Affine3f::Identity());
    dfSafeCall(df_kinfu_reset(handle_));
    warp_->clear();
}
Affine3f KinFu::getCameraPose(int time) const
{
    if (time > (int)poses_.size() || time < 0) time = (int)poses_.size() - 1;
    float p[12];
    df_kinfu_get_pose(handle_, time, p);
    return from12(p);
}
bool KinFu::operator()(const cuda::Depth& depth, const cuda::Image& /*image*/)
{
    const int r = df_kinfu_process_device(handle_, depth.ptr(), depth.step());
    if (r < 0) kfusion::cuda::error(df_error_string(-r), __FILE__, __LINE__);
    df_kinfu_join(handle_);                                             // the C++ API keeps the reference's contract: the frame's extraction is done on return
    cudaSafeCall(cudaDeviceSynchronize());                              // waitAllDefaultStream(), kinfu.cpp:301
    long long info[10];
    df_kinfu_get_info(handle_, info, 10);
    frame_counter_ = (int)info[0];
    // the pose chain only grows by one per frame (or restarts after a reset): copy what is new
    const size_t have = (size_t)info[3] >= poses_.size() && info[6] == resets_seen_ ? poses_.size() : 0;
    resets_seen_ = info[6];
    poses_.resize((size_t)info[3]);
    for (size_t i = have ? have - 1 : 0; i < poses_.size(); ++i) { float p[12]; df_kinfu_get_pose(handle_, (int)i, p); poses_[i] = from12(p); }
    volume_->host_clouds_stale_ = true;                                // get_cloud_host() / get_normal_host() fetch the frame's extraction on demand
    if (info[1] == 0 && warp_->deviceNodeCount() != 0) warp_->clear();  // the loop dropped its field (tracking-loss reset)
    if (info[1] > 0 && warp_->deviceNodeCount() != (int)info[1]) {       // nodes were (re)initialised on the device: adopt them
        size_t pitch; int cols, rows;
        float *nodes = (float *)buffer_of(handle_, 11, &pitch, &cols, &rows);
        warp_->adoptDeviceNodes(nodes, 0, (int)info[1]);
    }
    return r == 1;
}
void KinFu::getMesh(cv::Mat& vertices, cv::Mat& normals, cv::Mat& triangles, bool live) const
{
    int vcap = std::max(params_.volume_dims[0] * params_.volume_dims[1] * 4, 1024), tcap = 2 * vcap, c[2] = {0, 0};
    for (;;) {     // the counts are the true totals: one more call with buffers of that size fits
        DeviceMemory v((size_t)vcap * 16), n((size_t)vcap * 16), keys((size_t)vcap * 4), t((size_t)tcap * 12);
        const int st = df_kinfu_extract_mesh(handle_, live ? DF_MESH_LIVE : 0, v.ptr<float>(), n.ptr<float>(), keys.ptr<uint32_t>(), vcap,
                                             t.ptr<int32_t>(), tcap, c);
        if (st) kfusion::cuda::error(df_error_string(st), __FILE__, __LINE__);
        if (c[0] <= vcap && c[1] <= tcap) {
            vertices.create(1, c[0], CV_32FC4); normals.create(1, c[0], CV_32FC4); triangles.create(c[1], 1, CV_32SC3);
            if (c[0]) {
                cudaSafeCall(cudaMemcpy(vertices.ptr<float>(), v.ptr<float>(), (size_t)c[0] * 16, cudaMemcpyDeviceToHost));
                cudaSafeCall(cudaMemcpy(normals.ptr<float>(), n.ptr<float>(), (size_t)c[0] * 16, cudaMemcpyDeviceToHost));
            }
            if (c[1]) cudaSafeCall(cudaMemcpy(triangles.ptr<int>(), t.ptr<int32_t>(), (size_t)c[1] * 12, cudaMemcpyDeviceToHost));
            return;
        }
        vcap = std::max(vcap, c[0]); tcap = std::max(tcap, c[1]);
    }
}
void KinFu::dynamicfusion(cuda::Depth& depth, cuda::Cloud live_frame, cuda::Normals /*current_normals*/)
{
    const int r = df_kinfu_dynamicfusion(handle_, depth.ptr(), depth.step(), (const float *)live_frame.ptr(), live_frame.step());
    if (r < 0) kfusion::cuda::error(df_error_string(-r), __FILE__, __LINE__);
}
void KinFu::renderImage(cuda::Image& image, int flag)
{
    const KinFuParams& p = params_;
    image.create(p.rows, flag != 3 ? p.cols : p.cols * 2);
    size_t pp, np; int c, r;
    const float *pts = (const float *)buffer_of(handle_, 5, &pp, &c, &r);
    const float *nrm = (const float *)buffer_of(handle_, 6, &np, &c, &r);
    if (flag < 1 || flag > 3) {
        dfSafeCall(df_render_image(pts, pp, nrm, np, p.cols, p.rows, p.light_pose.val, image.ptr(), image.step(), 0));
    } else if (flag == 2) {
        dfSafeCall(df_render_tangent_colors(nrm, np, p.cols, p.rows, image.ptr(), image.step(), 0));
    } else {
        dfSafeCall(df_render_image(pts, pp, nrm, np, p.cols, p.rows, p.light_pose.val, image.ptr(), image.step(), 0));
        dfSafeCall(df_render_tangent_colors(nrm, np, p.cols, p.rows, image.ptr() + p.cols, image.step(), 0));
    }
    cudaSafeCall(cudaDeviceSynchronize());
}
void KinFu::renderImage(cuda::Image& image, const Affine3f& pose, int flag)
{
    const KinFuParams& p = params_;
    image.create(p.rows, flag != 3 ? p.cols : p.cols * 2);
    depths_.create(p.rows, p.cols); normals_.create(p.rows, p.cols); points_.create(p.rows, p.cols);
    // ray-cast the pipeline's volume from the requested pose
    df_kinfu_params d = params_to(params_);
    df_volume v;
    v.data = (uint32_t *)buffer_of(handle_, 0);
    float vmax = 0.f;
    for (int i = 0; i < 3; ++i) { v.dims[i] = d.volume_dims[i]; v.voxel_size[i] = d.volume_size[i] / d.volume_dims[i]; vmax = std::max(vmax, v.voxel_size[i]); }
    v.trunc_dist = std::max(d.tsdf_trunc_dist, 2.1f * vmax); v.max_weight = d.tsdf_max_weight;
    Affine3f cam2vol = p.volume_pose.inv() * pose;
    Mat3f Rinv = cam2vol.rotation().inv(cv::DECOMP_SVD);
    dfSafeCall(df_raycast_points(v, to_df(cam2vol), Rinv.val, to_df(p.intr), p.cols, p.rows, p.raycast_step_factor, p.gradient_delta_factor,
                                 (float *)points_.ptr(), points_.step(), (float *)normals_.ptr(), normals_.step(), 0));
    if (flag < 1 || flag > 3) cuda::renderImage(points_, normals_, p.intr, p.light_pose, image);
    else if (flag == 2) cuda::renderTangentColors(normals_, image);
    else {
        dfSafeCall(df_render_image((const float *)points_.ptr(), points_.step(), (const float *)normals_.ptr(), normals_.step(), p.cols, p.rows, p.light_pose.val,
                                   image.ptr(), image.step(), 0));
        dfSafeCall(df_render_tangent_colors((const float *)normals_.ptr(), normals_.step(), p.cols, p.rows, image.ptr() + p.cols, image.step(), 0));
        cudaSafeCall(cudaDeviceSynchronize());
    }
}
