// TEST-ONLY: LoamRegistration::ScanMatch's loop (loam_registration.cpp:38-99, SURVEY.md 3.3) restated over the CPU
// oracle's entry points (oracle/oracle.h): per trip oracle_icp_compute_hb on the surf (P2Plane) and the edge (P2Line)
// oracle, H = Hs + He and B = Bs + Be whatever the halves' bools say, the oracle's 6x6 inverse (la.hpp: lu6, what
// oracle_icp_align inverts with), dx = H^-1 B, oracle_pose_update, |dx| < eps.  A trip with det(H) == 0 makes no update
// (the reference would step by Eigen's inf / NaN inverse; DESIGN.md section 7).  The checker for locreg_align_loam.
#include <cstring>

#include "../../oracle/la.hpp"
#include "../../oracle/oracle.h"

using oracle::Mat6;
using oracle::Vec6;

extern "C" int oracle_loam_align(oracle_icp* surf, oracle_icp* edge, const float* surf_xyz, size_t n_surf, const float* edge_xyz,
                                 size_t n_edge, size_t stride, const double* pose_in, int32_t max_iteration, double eps,
                                 double* pose_out, oracle_result* res2) {
    double pose[7];
    std::memcpy(pose, pose_in, sizeof(pose));
    oracle_result loop{}, half[2] = {};
    loop.pose_written = 1;
    for (int it = 0; it < max_iteration; ++it) {
        double Hs[36], Bs[6], He[36], Be[6];
        const int ok_s = oracle_icp_compute_hb(surf, surf_xyz, n_surf, stride, pose, Hs, Bs, &half[0], nullptr, nullptr);
        const int ok_e = oracle_icp_compute_hb(edge, edge_xyz, n_edge, stride, pose, He, Be, &half[1], nullptr, nullptr);
        half[0].degenerate = ok_s ? 0 : 1;
        half[1].degenerate = ok_e ? 0 : 1;
        Mat6 H;
        Vec6 B;
        for (int i = 0; i < 36; ++i) H.a[i] = Hs[i] + He[i];
        for (int i = 0; i < 6; ++i) B.v[i] = Bs[i] + Be[i];
        loop.iters = it + 1;
        Mat6 Hinv;
        const double det = oracle::lu6(H, &Hinv);
        if (det == 0.0 || det != det) continue;
        const Vec6 dx = oracle::mul(Hinv, B);
        oracle_pose_update(pose, dx.v);
        loop.updates++;
        if (dx.norm() < eps) { loop.converged = 1; break; }
    }
    std::memcpy(pose_out, pose, sizeof(pose));
    for (int i = 0; res2 && i < 2; ++i) {
        res2[i] = half[i];
        res2[i].iters = loop.iters;
        res2[i].updates = loop.updates;
        res2[i].converged = loop.converged;
        res2[i].pose_written = 1;
    }
    return 0;
}
