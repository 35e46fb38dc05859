// Drop-in adapters: LocUtils::MatchingInterface implementations backed by liblocreg.so (include/locreg.h).
//
//   LocUtils::CudaIcpRegistration(IcpOptions)   replaces LocUtils::IcpRegistration
//       (LocUtils/include/LocUtils/model/matching/3d/icp/icp_registration.hpp:41-142)
//   LocUtils::CudaNdtRegistration(NdtOptions)   replaces LocUtils::NdtRegistration (DIRECT_NDT and INCREMENTAL_NDT)
//       (LocUtils/include/LocUtils/model/matching/3d/ndt/ndt_registration.hpp:69-135)
//
// Same constructors, same virtual methods, same always-true bool results (icp_registration.cpp:243,
// ndt_registration.cpp:260), so the callers - Loc (LocUtils/src/slam/3d/loc.cpp:41,55), Lio (lio.cpp:30,40),
// LoamRegistration (loam_registration.cpp:56,66) - change one make_shared<> line each (INTEGRATION.md).
//
// Header-only and generic over the host types so that it can be compiled both
//   * inside LocUtils (PCL / Sophus / Eigen present):   #include "LocUtils/model/matching/3d/matching_interface.h"
//     BEFORE this header; the adapters then derive from the real LocUtils::MatchingInterface, and
//   * in this repo's container, where those libraries do not exist: tests/cpp/adapter_standin.cpp defines
//     stand-in CloudPtr / SE3 / Mat6d / Vec6d types with the same members the adapter touches and
//     LOCREG_ADAPTER_STANDIN, and checks that the marshalling compiles and links against liblocreg.so.
// What the adapter needs from the host types (all true for PCL 1.8 / Sophus / Eigen):
//   cloud->points.data(), cloud->points.size(), sizeof(PointType) == point stride, x/y/z the first three floats
//   (pcl::PointXYZI: 32 B stride, point_types.h:18); cloud->width/height/is_dense; cloud.reset(new PointCloudType);
//   SE3::data() -> 7 doubles [qx qy qz qw tx ty tz] (Sophus::SE3d; eigen_types.h:66); Mat6d/Vec6d::data() column-major.
#pragma once
#include <memory>
#include <stdexcept>
#include <string>
#include <utility>

#include "locreg.h"

namespace LocUtils {

namespace locreg_detail {
inline void check(int rc, const char* what) {
    // The reference's methods cannot report errors (bool, always true).  A CUDA failure is not an algorithmic outcome,
    // so it is raised instead of being swallowed: there is no CPU path to fall back to.
    if (rc != LOCREG_OK) throw std::runtime_error(std::string(what) + ": " + locreg_last_error());
}
// Pose algebra on Sophus::SE3d's memory layout [qx qy qz qw tx ty tz] (the trackers below stay independent of the
// host's SE3 type; inside LocUtils `a * b` and `a.inverse()` do the same).
inline void quat_rotate(const double* q, const double* v, double* out) {
    const double tx = 2.0 * (q[1] * v[2] - q[2] * v[1]), ty = 2.0 * (q[2] * v[0] - q[0] * v[2]), tz = 2.0 * (q[0] * v[1] - q[1] * v[0]);
    out[0] = v[0] + q[3] * tx + (q[1] * tz - q[2] * ty);
    out[1] = v[1] + q[3] * ty + (q[2] * tx - q[0] * tz);
    out[2] = v[2] + q[3] * tz + (q[0] * ty - q[1] * tx);
}
inline void se3_mul(const double* a, const double* b, double* out) {  // out = a * b (out may not alias a or b)
    const double qx = a[3] * b[0] + a[0] * b[3] + a[1] * b[2] - a[2] * b[1], qy = a[3] * b[1] - a[0] * b[2] + a[1] * b[3] + a[2] * b[0],
                 qz = a[3] * b[2] + a[0] * b[1] - a[1] * b[0] + a[2] * b[3], qw = a[3] * b[3] - a[0] * b[0] - a[1] * b[1] - a[2] * b[2];
    double n = qx * qx + qy * qy + qz * qz + qw * qw;
    n = n > 0.0 ? 1.0 / __builtin_sqrt(n) : 1.0;
    out[0] = qx * n; out[1] = qy * n; out[2] = qz * n; out[3] = qw * n;
    double r[3];
    quat_rotate(a, b + 4, r);
    out[4] = a[4] + r[0]; out[5] = a[5] + r[1]; out[6] = a[6] + r[2];
}
inline void se3_inv(const double* a, double* out) {
    const double qi[4] = {-a[0], -a[1], -a[2], a[3]};
    double r[3];
    quat_rotate(qi, a + 4, r);
    out[0] = qi[0]; out[1] = qi[1]; out[2] = qi[2]; out[3] = qi[3];
    out[4] = -r[0]; out[5] = -r[1]; out[6] = -r[2];
}
inline double se3_rotation_angle(const double* a) {  // |log(R)|
    return 2.0 * __builtin_atan2(__builtin_sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]), __builtin_fabs(a[3]));
}
// predict = result * last^-1 * result: the constant-velocity model of Loc::Update (loc.cpp:232) and
// Lio::AlignWithLocalMap (lio.cpp:464)
template <class SE3T>
inline void predict_next(const SE3T& result, const SE3T& last, SE3T& predict) {
    double inv[7], tmp[7], out[7];
    se3_inv(last.data(), inv);
    se3_mul(result.data(), inv, tmp);
    se3_mul(tmp, result.data(), out);
    for (int i = 0; i < 7; ++i) predict.data()[i] = out[i];
}
template <class Cloud>
inline const float* cloud_xyz(const Cloud& c) {
    return c.points.empty() ? nullptr : reinterpret_cast<const float*>(c.points.data());
}
}  // namespace locreg_detail

class CudaRegistrationBase : public MatchingInterface {
   public:
    ~CudaRegistrationBase() override { locreg_destroy(handle_); }
    CudaRegistrationBase(const CudaRegistrationBase&) = delete;
    CudaRegistrationBase& operator=(const CudaRegistrationBase&) = delete;

    // MatchingInterface::SetInputTarget (matching_interface.h:18): deep copy + index build, on the device.
    bool SetInputTarget(const CloudPtr& input_target) override {
        locreg_detail::check(locreg_set_target(handle_, locreg_detail::cloud_xyz(*input_target), input_target->points.size(),
                                               sizeof(PointType)),
                             "locreg_set_target");
        return true;
    }

    // MatchingInterface::CaculateMatrixHAndB (matching_interface.h:23-29; sole caller loam_registration.cpp:56,66).
    bool CaculateMatrixHAndB(const CloudPtr& input_source, const SE3& predict_pose, Mat6d& H, Vec6d& B) override {
        locreg_result res{};
        locreg_detail::check(locreg_compute_hb(handle_, locreg_detail::cloud_xyz(*input_source), input_source->points.size(),
                                               sizeof(PointType), predict_pose.data(), H.data(), B.data(), &res),
                             "locreg_compute_hb");
        last_result_ = res;
        return res.degenerate == 0;  // icp_registration.cpp:100-102,204-212: false when too few points / det(H) == 0
    }

    // MatchingInterface::ScanMatch (matching_interface.h:30-36).  result_cloud_ptr is overwritten with the
    // transformed input (pcl::transformPointCloud, icp_registration.cpp:241); result_pose is IN/OUT exactly as in
    // the reference: direct NDT's det(H) == 0 early return leaves it untouched (ndt_registration.cpp:435-436).
    bool ScanMatch(const CloudPtr& input_source, const SE3& predict_pose, CloudPtr& result_cloud_ptr, SE3& result_pose) override {
        const size_t n = input_source->points.size();
        if (!result_cloud_ptr) result_cloud_ptr.reset(new PointCloudType);
        if (result_cloud_ptr.get() != input_source.get()) {
            result_cloud_ptr->header = input_source->header;
            result_cloud_ptr->is_dense = input_source->is_dense;
            result_cloud_ptr->width = input_source->width;
            result_cloud_ptr->height = input_source->height;
            result_cloud_ptr->points.resize(n);
        }
        locreg_result res{};
        locreg_detail::check(
            locreg_align(handle_, locreg_detail::cloud_xyz(*input_source), n, sizeof(PointType), predict_pose.data(), result_pose.data(),
                         n ? reinterpret_cast<float*>(result_cloud_ptr->points.data()) : nullptr, &res),
            "locreg_align");
        last_result_ = res;
        return true;  // icp_registration.cpp:243, ndt_registration.cpp:260
    }

    float GetFitnessScore() override { return 0.0f; }  // icp_registration.cpp:246-250, ndt_registration.cpp:466-471

    // ---- the callers' map state, kept on the device (no counterpart in MatchingInterface; INTEGRATION.md section 3) ----
    // Loc::InitGlobalMap (loc.cpp:268-283): the global map is uploaded once.
    void SetGlobalMap(const CloudPtr& global_map) {
        locreg_detail::check(locreg_set_global_map(handle_, locreg_detail::cloud_xyz(*global_map), global_map->points.size(),
                                                   sizeof(PointType)),
                             "locreg_set_global_map");
    }
    // Loc::ResetLocalMap (loc.cpp:187-206): BoxFilter::SetOrigin + Filter + SetInputTarget; returns the local map's size.
    size_t ResetLocalMap(float x, float y, float z, const float (&half_size)[3]) {
        const float origin[3] = {x, y, z};
        size_t n_local = 0;
        locreg_detail::check(locreg_reset_local_map(handle_, origin, half_size, &n_local), "locreg_reset_local_map");
        return n_local;
    }
    // The key-frame block of Lio::AddCloud (lio.cpp:277-307): transformPointCloud(scan, pose), slide the window of
    // num_kfs_in_local_map scans, voxel-filter the local map (leaf <= 0: NoFilter), SetInputTarget.
    size_t AddKeyFrame(const CloudPtr& scan, const SE3& pose, int num_kfs_in_local_map, float leaf) {
        size_t n_local = 0;
        locreg_detail::check(locreg_local_map_add_keyframe(handle_, locreg_detail::cloud_xyz(*scan), scan->points.size(), sizeof(PointType),
                                                           pose.data(), num_kfs_in_local_map, leaf, &n_local),
                             "locreg_local_map_add_keyframe");
        return n_local;
    }

    // what the reference logs or drops: iterations, effective points, convergence, degeneracy
    const locreg_result& LastResult() const { return last_result_; }
    locreg_handle* Handle() const { return handle_; }

   protected:
    explicit CudaRegistrationBase(const locreg_options& opt, int device) {
        locreg_detail::check(locreg_create(&opt, device, &handle_), "locreg_create");
    }
    locreg_handle* handle_ = nullptr;
    locreg_result last_result_{};
};

class CudaIcpRegistration : public CudaRegistrationBase {
   public:
    explicit CudaIcpRegistration(IcpOptions options, int device = 0) : CudaRegistrationBase(Convert(options), device), options_(options) {}

   private:
    static locreg_options Convert(const IcpOptions& o) {
        locreg_options c{};
        int method = LOCREG_ICP_P2P;
        switch (o.method_) {
            case IcpMethod::P2P: method = LOCREG_ICP_P2P; break;
            case IcpMethod::P2LINE: method = LOCREG_ICP_P2LINE; break;
            case IcpMethod::P2PLANE: method = LOCREG_ICP_P2PLANE; break;
            case IcpMethod::PCLICP: throw std::runtime_error("PCLICP is a passthrough to pcl::IterativeClosestPoint: keep IcpRegistration for it");
        }
        locreg_default_options(&c, method);
        c.max_iteration = o.max_iteration_;
        c.max_nn_distance = o.max_nn_distance_;
        c.max_plane_distance = o.max_plane_distance_;
        c.max_line_distance = o.max_line_distance_;
        c.min_effective_pts = o.min_effective_pts_;
        c.eps = o.eps_;
        c.use_ann = o.use_ann ? 1 : 0;  // accepted, ignored: the search is exact (DESIGN.md, deviation Q1)
        // !use_initial_translation_: Align* start from target_center_ - source_center_, which is zero - neither centre is
        // ever computed (icp_registration.cpp:22-26,261-264,272-276)
        c.zero_initial_translation = o.use_initial_translation_ ? 0 : 1;
        return c;
    }
    IcpOptions options_;
};

class CudaNdtRegistration : public CudaRegistrationBase {
   public:
    explicit CudaNdtRegistration(NdtOptions options, int device = 0) : CudaRegistrationBase(Convert(options), device), options_(options) {}

   private:
    static locreg_options Convert(const NdtOptions& o) {
        if (o.method_ == NdtMethod::PCL_NDT) throw std::runtime_error("PCL_NDT is an unimplemented stub in the reference");
        locreg_options c{};
        locreg_default_options(&c, o.method_ == NdtMethod::INCREMENTAL_NDT ? LOCREG_NDT_INCREMENTAL : LOCREG_NDT_DIRECT);
        c.ndt_capacity = static_cast<int32_t>(o.capacity_);
        c.max_iteration = o.max_iteration_;
        c.voxel_size = o.voxel_size_;  // inv_voxel_size_ is recomputed, as in ndt_registration.cpp:25
        c.min_effective_pts = o.min_effective_pts_;
        c.min_pts_in_voxel = o.min_pts_in_voxel_;
        c.eps = o.eps_;
        c.res_outlier_th = o.res_outlier_th_;
        c.nearby_type = o.nearby_type_ == NdtNearbyType::NEARBY6 ? LOCREG_NEARBY6 : LOCREG_NEARBY_CENTER;
        c.zero_initial_translation = o.remove_centroid_ ? 1 : 0;  // AlignNdt only (ndt_registration.cpp:380-384)
        return c;
    }
    NdtOptions options_;
};

// LoamRegistration::ScanMatch's loop (loam_registration.cpp:38-99, SURVEY.md 3.3) on the device: a P2Plane
// CudaIcpRegistration for the surf cloud and a P2Line one for the edge cloud, each with its own options and gates; one
// Align call runs every Gauss-Newton trip (both halves' H and B summed, one step) with no host round trip in between
// (locreg_align_loam).  max_iteration and eps are the LOAM loop's (LoamOption), not either half's.  It does not implement
// MatchingInterface's two-cloud overloads: the names here say which cloud is which.
class CudaLoamMatcher {
   public:
    CudaLoamMatcher(IcpOptions surf_options, IcpOptions edge_options, int max_iteration = 10, double eps = 1e-2, int device = 0)
        : surf_(Checked(surf_options, IcpMethod::P2PLANE, "surf"), device),
          edge_(Checked(edge_options, IcpMethod::P2LINE, "edge"), device),
          max_iteration_(max_iteration), eps_(eps) {}

    void SetTargets(const CloudPtr& surf_map, const CloudPtr& edge_map) {
        surf_.SetInputTarget(surf_map);
        edge_.SetInputTarget(edge_map);
    }
    // result_pose is always written.  LastResults()[0] / [1]: the loop's trips, updates and convergence, and the surf /
    // edge half's last evaluation.
    void Align(const CloudPtr& surf, const CloudPtr& edge, const SE3& predict_pose, SE3& result_pose) {
        locreg_detail::check(locreg_align_loam(surf_.Handle(), edge_.Handle(), locreg_detail::cloud_xyz(*surf), surf->points.size(),
                                               locreg_detail::cloud_xyz(*edge), edge->points.size(), sizeof(PointType),
                                               predict_pose.data(), max_iteration_, eps_, result_pose.data(), last_results_),
                             "locreg_align_loam");
    }
    const locreg_result* LastResults() const { return last_results_; }
    CudaIcpRegistration& Surf() { return surf_; }
    CudaIcpRegistration& Edge() { return edge_; }

   private:
    static IcpOptions Checked(IcpOptions o, IcpMethod want, const char* half) {
        if (o.method_ != want) throw std::runtime_error(std::string("CudaLoamMatcher: the ") + half + " half needs " +
                                                        (want == IcpMethod::P2PLANE ? "P2PLANE" : "P2LINE") + " options");
        return o;
    }
    CudaIcpRegistration surf_, edge_;
    int max_iteration_;
    double eps_;
    locreg_result last_results_[2] = {};
};

// ---- the two callers' loops around ScanMatch, with the map state on the device ------------------------------------
// Loc::Update without the ROS / ESKF parts (loc.cpp:208-246): ScanMatch from the constant-velocity prediction, and a new
// local map (crop of the device-resident global map) whenever the pose comes within `margin` of the box edge.
class CudaLocTracker {
   public:
    CudaLocTracker(std::shared_ptr<CudaRegistrationBase> reg, const CloudPtr& global_map, const SE3& init_pose, float half_size = 150.0f,
                   double margin = 50.0)
        : reg_(std::move(reg)), half_{half_size, half_size, half_size}, margin_(margin), last_(init_pose), predict_(init_pose) {
        reg_->SetGlobalMap(global_map);
        Reset(init_pose);
    }
    // returns the registered pose; result_cloud as in ScanMatch
    SE3 Update(const CloudPtr& scan, CloudPtr& result_cloud) {
        SE3 result = predict_;
        reg_->ScanMatch(scan, predict_, result_cloud, result);
        locreg_detail::predict_next(result, last_, predict_);
        last_ = result;
        const double* t = result.data() + 4;
        for (int i = 0; i < 3; ++i) {  // loc.cpp:235-246
            const double lo = -half_[i] + origin_[i], hi = half_[i] + origin_[i];
            if (__builtin_fabs(t[i] - lo) > margin_ && __builtin_fabs(t[i] - hi) > margin_) continue;
            Reset(result);
            break;
        }
        return result;
    }
    size_t LocalMapSize() const { return n_local_; }
    int Resets() const { return resets_; }
    const SE3& Predict() const { return predict_; }

   private:
    void Reset(const SE3& pose) {
        for (int i = 0; i < 3; ++i) origin_[i] = static_cast<float>(pose.data()[4 + i]);
        n_local_ = reg_->ResetLocalMap(origin_[0], origin_[1], origin_[2], half_);
        ++resets_;
    }
    std::shared_ptr<CudaRegistrationBase> reg_;
    float half_[3], origin_[3] = {0, 0, 0};
    double margin_;
    SE3 last_, predict_;
    size_t n_local_ = 0;
    int resets_ = 0;
};

// Lio::AddCloud / AlignWithLocalMap without the ROS / ESKF / file parts (lio.cpp:238-307, 445-470, 616-623).
class CudaLioTracker {
   public:
    explicit CudaLioTracker(std::shared_ptr<CudaRegistrationBase> reg, int num_kfs_in_local_map = 10, double kf_distance = 1.0,
                            double kf_angle_deg = 10.0, float local_map_leaf = 0.5f)
        : reg_(std::move(reg)), max_kfs_(num_kfs_in_local_map), kf_distance_(kf_distance),
          kf_angle_(kf_angle_deg * 3.14159265358979323846 / 180.0), leaf_(local_map_leaf) {
        locreg_detail::check(locreg_local_map_clear(reg_->Handle()), "locreg_local_map_clear");
    }
    // scan: the raw scan (what a key frame stores, :279); filtered: cur_scan_filter_ptr_'s output (what is matched, and
    // what the FIRST key frame stores, :236,:244), free of NaN points (Lio runs RemoveNanPoint first, :452).  Returns the
    // pose; *is_keyframe tells whether the local map moved on.
    SE3 AddCloud(const CloudPtr& scan, const CloudPtr& filtered, bool* is_keyframe = nullptr) {
        if (keyframes_ == 0) {
            n_local_ = reg_->AddKeyFrame(filtered, last_kf_pose_, max_kfs_, leaf_);
            keyframes_ = 1;
            if (is_keyframe) *is_keyframe = true;
            return last_kf_pose_;
        }
        SE3 result = predict_;
        CloudPtr aligned;
        reg_->ScanMatch(filtered, predict_, aligned, result);
        locreg_detail::predict_next(result, last_pose_, predict_);
        last_pose_ = result;
        double inv[7], delta[7];
        locreg_detail::se3_inv(last_kf_pose_.data(), inv);
        locreg_detail::se3_mul(inv, result.data(), delta);
        const double dist = __builtin_sqrt(delta[4] * delta[4] + delta[5] * delta[5] + delta[6] * delta[6]);
        const bool kf = dist > kf_distance_ || locreg_detail::se3_rotation_angle(delta) > kf_angle_;
        if (kf) {
            last_kf_pose_ = result;
            n_local_ = reg_->AddKeyFrame(scan, result, max_kfs_, leaf_);
            ++keyframes_;
        }
        if (is_keyframe) *is_keyframe = kf;
        return result;
    }
    size_t LocalMapSize() const { return n_local_; }
    int KeyFrames() const { return keyframes_; }

   private:
    std::shared_ptr<CudaRegistrationBase> reg_;
    int max_kfs_;
    double kf_distance_, kf_angle_;
    float leaf_;
    SE3 last_kf_pose_, last_pose_, predict_;  // identity: the function statics of AlignWithLocalMap start there too
    size_t n_local_ = 0;
    int keyframes_ = 0;
};

}  // namespace LocUtils
