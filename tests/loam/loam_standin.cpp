// TEST-ONLY: compiles CudaLoamMatcher (include/locreg_adapter.hpp) against adapter_standin.cpp's stand-ins for the PCL /
// Sophus / Eigen types and drives it the way LoamRegistration::ScanMatch would: SetTargets(surf map, edge map), then
// one Align(surf, edge, predict, result) per scan.  Exit code 0: ran on a GPU and recovered the pose; 3: no CUDA device
// (the adapter threw, as designed: no CPU fallback); anything else: failure.
#define main adapter_standin_main  // reuse the stand-in types and the adapter include, not that program's main
#include "../cpp/adapter_standin.cpp"
#undef main

// surf: the plane z = 0; edge: two vertical poles.  Neither constrains all six degrees of freedom alone.
static void make_scene(CloudPtr& plane, CloudPtr& poles) {
    plane = std::make_shared<PointCloudType>();
    poles = std::make_shared<PointCloudType>();
    for (int i = -40; i <= 40; ++i)
        for (int j = -40; j <= 40; ++j) plane->points.push_back(PointType{0.1f * i, 0.1f * j, 0, 0, 1, 0, 0, 0});
    for (int k = 0; k <= 60; ++k) {
        const float z = 0.05f * k;
        poles->points.push_back(PointType{1.5f, 0.5f, z, 0, 2, 0, 0, 0});
        poles->points.push_back(PointType{-1.0f, -2.0f, z, 0, 2, 0, 0, 0});
    }
    plane->width = static_cast<uint32_t>(plane->points.size());
    poles->width = static_cast<uint32_t>(poles->points.size());
}

int main() {
    IcpOptions so, eo;
    so.method_ = IcpMethod::P2PLANE;
    eo.method_ = IcpMethod::P2LINE;
    std::unique_ptr<CudaLoamMatcher> loam;
    try {
        loam.reset(new CudaLoamMatcher(so, eo, 10, 1e-6));
    } catch (const std::exception& e) {
        std::printf("loam: %s\n", e.what());
        return std::strstr(e.what(), "no CUDA device") ? 3 : 1;
    }
    CloudPtr plane, poles;
    make_scene(plane, poles);
    loam->SetTargets(plane, poles);
    // the sensor moved by (0.03, -0.02, 0.025): the scans see the scene shifted the other way
    auto surf = std::make_shared<PointCloudType>(*plane);
    auto edge = std::make_shared<PointCloudType>(*poles);
    for (auto* c : {surf.get(), edge.get()})
        for (PointType& p : c->points) { p.x -= 0.03f; p.y += 0.02f; p.z -= 0.025f; }
    SE3 predict, result;
    loam->Align(surf, edge, predict, result);
    const double* t = result.data() + 4;
    std::printf("loam: t = (%.5f %.5f %.5f), %d trips\n", t[0], t[1], t[2], loam->LastResults()[0].iters);
    if (std::fabs(t[0] - 0.03) > 1e-3 || std::fabs(t[1] + 0.02) > 1e-3 || std::fabs(t[2] - 0.025) > 1e-3) return 1;
    if (loam->LastResults()[0].n_inlier <= 0 || loam->LastResults()[1].n_inlier <= 0) return 1;
    return 0;
}
