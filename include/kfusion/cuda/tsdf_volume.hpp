#pragma once
// Dense TSDF volume; same interface as the reference's kfusion/cuda/tsdf_volume.hpp:11-100.
#include <kfusion/types.hpp>
#include <dual_quaternion.hpp>

namespace kfusion
{
    class WarpField;
    class KinFu;
    namespace cuda
    {
        class KF_EXPORTS TsdfVolume
        {
        public:
            TsdfVolume(const cv::Vec3i& dims);
            virtual ~TsdfVolume();

            void create(const Vec3i& dims);
            Vec3i getDims() const;
            Vec3f getVoxelSize() const;
            const CudaData data() const;
            CudaData data();
            cv::Mat get_cloud_host() const;
            cv::Mat get_normal_host() const;
            cv::Mat* get_cloud_host_ptr() const;
            cv::Mat* get_normal_host_ptr() const;
            Vec3f getSize() const;
            void setSize(const Vec3f& size);
            float getTruncDist() const;
            void setTruncDist(float distance);
            int getMaxWeight() const;
            void setMaxWeight(int weight);
            Affine3f getPose() const;
            void setPose(const Affine3f& pose);
            float getRaycastStepFactor() const;
            void setRaycastStepFactor(float factor);
            float getGradientDeltaFactor() const;
            void setGradientDeltaFactor(float factor);
            Vec3i getGridOrigin() const;
            void setGridOrigin(const Vec3i& origin);

            std::vector<float> psdf(const std::vector<Vec3f>& warped, Dists& depth_img, const Intr& intr);
            float weighting(const std::vector<float>& dist_sqr, int k) const;
            void surface_fusion(const WarpField& warp_field, std::vector<Vec3f> warped, std::vector<Vec3f> canonical,
                                cuda::Depth &depth, const Affine3f& camera_pose, const Intr& intr);

            virtual void clear();
            virtual void applyAffine(const Affine3f& affine);
            virtual void integrate(const Dists& dists, const Affine3f& camera_pose, const Intr& intr);
            // not in the reference: the per-voxel warped fusion surface_fusion() was written towards and left commented out
            // (tsdf_volume.cpp:240-252; SURVEY 8f(1)) -> df_integrate_warped.  depth = the u16 millimetre frame.
            virtual void integrate(const Depth& depth, const WarpField& warp_field, const Affine3f& camera_pose, const Intr& intr, float weight_scale = 0.f);
            virtual void raycast(const Affine3f& camera_pose, const Intr& intr, Depth& depth, Normals& normals);   // USE_DEPTH path: aborts
            virtual void raycast(const Affine3f& camera_pose, const Intr& intr, Cloud& points, Normals& normals);

            void swap(CudaData& data);
            DeviceArray<Point> fetchCloud(DeviceArray<Point>& cloud_buffer) const;
            void fetchNormals(const DeviceArray<Point>& cloud, DeviceArray<Normal>& normals) const;
            // not in the reference: the triangle mesh of the zero level set (dfusion.h df_extract_mesh, marching cubes) at the volume pose; the
            // arrays are resized to the mesh (triangles: 3 vertex indices each), normals as fetchNormals computes them at the vertices
            void fetchMesh(DeviceArray<Point>& vertices, DeviceArray<Normal>& normals, DeviceArray<int>& triangles) const;
            void compute_points();
            void compute_normals();

        private:
            CudaData data_;
            cuda::DeviceArray<Point> *cloud_buffer_;
            cuda::DeviceArray<Point> *cloud_;
            cuda::DeviceArray<Normal> *normal_buffer_;
            cv::Mat *cloud_host_;
            cv::Mat *normal_host_;
            float trunc_dist_;
            float max_weight_;
            Vec3i dims_;
            Vec3f size_;
            Affine3f pose_;
            float gradient_delta_factor_;
            float raycast_step_factor_;
            struct Entry { float tsdf_value; float tsdf_weight; };
            std::vector<Entry> tsdf_entries_;
            mutable DeviceMemory workspace_;          // extraction / projection scratch (not in the reference)
            mutable DeviceMemory count_;
            // When this object is KinFu's view over the frame loop's volume (KinFu::tsdf()): the loop's activity map (every integration
            // of that volume must be tracked, dfusion.h) and the loop's extracted cloud / normals, copied to the host clouds on demand
            // (the reference fills them every frame, kinfu.cpp:249-250,398-399).
            friend class ::kfusion::KinFu;
            unsigned char *activity_ = 0;
            void *pipeline_ = 0;
            mutable bool host_clouds_stale_ = false;
            void refresh_host_clouds() const;
        };
    }
}
