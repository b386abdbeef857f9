#pragma once
// kfusion::KinFuParams / kfusion::KinFu -- same interface as the reference's kfusion/kinfu.hpp:15-97, so apps/demo.cpp's use of
// it (default_params_dynamicfusion, KinFu::Ptr, operator()(depth), renderImage, getCameraPose, getWarp().getNodesAsMat())
// compiles unchanged.  The per-frame loop runs device-resident behind df_kinfu_* (include/dfusion.h).
#include <kfusion/types.hpp>
#include <vector>
#include <string>
#include <dual_quaternion.hpp>
#include <quaternion.hpp>
#include <kfusion/cuda/projective_icp.hpp>
#include <kfusion/cuda/tsdf_volume.hpp>
#include <kfusion/warp_field.hpp>
#include "warp_field_optimiser.hpp"

namespace kfusion
{
    struct KF_EXPORTS KinFuParams
    {
        static KinFuParams default_params();
        static KinFuParams default_params_dynamicfusion();

        int cols;  //pixels
        int rows;  //pixels
        Intr intr;  //Camera parameters
        Vec3i volume_dims; //number of voxels
        Vec3f volume_size; //meters
        Affine3f volume_pose; //meters, inital pose
        float bilateral_sigma_depth;   //meters
        float bilateral_sigma_spatial;   //pixels
        int   bilateral_kernel_size;   //pixels
        float icp_truncate_depth_dist; //meters
        float icp_dist_thres;          //meters
        float icp_angle_thres;         //radians
        std::vector<int> icp_iter_num; //iterations for level index 0,1,..,3
        float tsdf_min_camera_movement; //meters, integrate only if exceedes
        float tsdf_trunc_dist;             //meters;
        int tsdf_max_weight;               //frames
        float raycast_step_factor;   // in voxel sizes
        float gradient_delta_factor; // in voxel sizes
        Vec3f light_pose; //meters

        // not in the reference: opt-in extensions of the fusion step (SURVEY 8f), forwarded to df_kinfu_params; the defaults keep the
        // reference's behaviour.  (The same switches exist as environment variables for an unchanged apps/demo.cpp, dfusion.h.)
        int dfusion_flags = 0;             // DF_KINFU_WARPED_INTEGRATE (8) | DF_KINFU_EXTEND_FIELD (16)
        float fusion_weight_scale = 0.f;   // df_integrate_warped's weight quantisation (0: every sample weighs 1)
        float extend_radius = 0.f;         // df_extend_field's support radius in metres (0: 0.03)
    };

    class KF_EXPORTS KinFu
    {
    public:
        typedef cv::Ptr<KinFu> Ptr;

        KinFu(const KinFuParams& params);
        ~KinFu();

        const KinFuParams& params() const;
        KinFuParams& params();
        const cuda::TsdfVolume& tsdf() const;
        cuda::TsdfVolume& tsdf();
        const cuda::ProjectiveICP& icp() const;
        cuda::ProjectiveICP& icp();
        const WarpField& getWarp() const;
        WarpField& getWarp();

        void reset();
        bool operator()(const cuda::Depth& depth, const cuda::Image& image = cuda::Image());
        void renderImage(cuda::Image& image, int flags = 0);
        void dynamicfusion(cuda::Depth& depth, cuda::Cloud live_frame, cuda::Normals current_normals);
        void renderImage(cuda::Image& image, const Affine3f& pose, int flags = 0);
        Affine3f getCameraPose (int time = -1) const;
        // not in the reference: the current model as a host mesh (df_kinfu_extract_mesh) -- vertices / normals 1 x N CV_32FC4, triangles
        // M x 1 CV_32SC3; live = true carries it through the warp field into the live frame.  kfusion::writePly(path, vertices, normals,
        // triangles) exports it.
        void getMesh(cv::Mat& vertices, cv::Mat& normals, cv::Mat& triangles, bool live = false) const;
    private:
        void allocate_buffers();

        int frame_counter_;
        KinFuParams params_;
        std::vector<Affine3f> poses_;
        cuda::Dists dists_;
        cuda::Frame curr_, prev_, first_;
        cuda::Cloud points_;
        cuda::Normals normals_;
        cuda::Depth depths_;
        cv::Ptr<cuda::TsdfVolume> volume_;
        cv::Ptr<cuda::ProjectiveICP> icp_;
        cv::Ptr<WarpField> warp_;
        std::vector<std::pair<utils::DualQuaternion<float>, utils::DualQuaternion<float>>> edges_;
        cv::Ptr<WarpFieldOptimiser> optimiser_;
        void *handle_;          // df_kinfu_* pipeline object (not in the reference)
        long long resets_seen_ = 0;   // tracking-loss resets already mirrored into poses_
    };
}
