/* locreg — C ABI of the B200-native scan-to-map registration hot path.
 *
 * Drop-in boundary for maotian123/loc_lib's LocUtils::MatchingInterface
 * (LocUtils/include/LocUtils/model/matching/3d/matching_interface.h:13-54) as implemented by
 * IcpRegistration (icp_registration.hpp:41-142 / icp_registration.cpp) and NdtRegistration
 * (ndt_registration.hpp:69-135 / ndt_registration.cpp).  A header-only C++ adapter that derives from
 * MatchingInterface and forwards to these entry points is in include/locreg_adapter.hpp; the reference
 * side binding is shown in INTEGRATION.md.
 *
 * Conventions
 *   clouds   : pointer to the first float of the first point + point count + stride in bytes between
 *              points (32 for pcl::PointXYZI, LocUtils point_types.h:18; 16 for float4; >= 12).  x,y,z are
 *              the first three floats of a point.
 *   poses    : 7 doubles [qx qy qz qw tx ty tz] = Sophus::SE3d::data() (LocUtils eigen_types.h:66).
 *   H, B     : 6x6 column-major (Eigen default) and 6x1 doubles, rotation block first, as the reference's
 *              Mat6d / Vec6d (matching_interface.h:23-26).
 *   return   : 0 on success, negative LOCREG_E_* on failure; locreg_last_error() describes the last failure
 *              of the calling thread.  Algorithmic outcomes (too few points, singular H, ...) are NOT
 *              errors: like the reference's always-true bool they are reported in locreg_result.
 *   threading: one handle = one CUDA stream; a handle is not thread-safe, distinct handles are independent
 *              (the reference's classes are not re-entrant either: mutable source_/target_ members).
 *   there is no CPU fallback: every entry point that computes fails with LOCREG_E_CUDA without a B200.
 */
#ifndef LOCREG_H
#define LOCREG_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define LOCREG_OK 0
#define LOCREG_E_ARG (-1)         /* invalid argument */
#define LOCREG_E_CUDA (-2)        /* CUDA runtime error (no device, out of memory, launch failure) */
#define LOCREG_E_STATE (-3)       /* call order (e.g. align before set_target) */
#define LOCREG_E_UNSUPPORTED (-4) /* not built (PCLICP), or NCCL is not available for the multi-GPU entry points */

/* IcpMethod (icp_registration.hpp:15-20) and NdtMethod (ndt_registration.hpp:21-26) in one enum */
enum locreg_method {
    LOCREG_ICP_P2P = 0,
    LOCREG_ICP_P2LINE = 1,
    LOCREG_ICP_P2PLANE = 2,
    LOCREG_NDT_DIRECT = 3,
    LOCREG_NDT_INCREMENTAL = 4 /* NdtMethod::INCREMENTAL_NDT: locreg_set_target ADDS a cloud to an LRU voxel cache */
};
/* NdtNearbyType (ndt_registration.hpp:16-20) */
enum locreg_nearby { LOCREG_NEARBY_CENTER = 0, LOCREG_NEARBY6 = 1 };
/* how the Gauss-Newton loop is kept on the device */
enum locreg_loop { LOCREG_LOOP_PERSISTENT = 0, /* the whole Gauss-Newton loop of one ScanMatch in ONE cooperative kernel
                                                  (grid barrier per iteration): k_align_persist (NDT), k_icp_persist (ICP) */
                   LOCREG_LOOP_GRAPH = 1 /* per-iteration kernels (search, stage 2, fit, normal equations, solve) queued back
                                            to back on the stream for all iterations with no host round trip; stop flags in
                                            device memory make the kernels of a finished scan exit at once.  (The name is
                                            historical: the launches are plain stream launches, not a captured CUDA graph;
                                            batches and relocalisation always run this way.) */ };

/* POD mirror of IcpOptions (icp_registration.hpp:22-39) + NdtOptions (ndt_registration.hpp:27-42). */
typedef struct locreg_options {
    int32_t method;               /* enum locreg_method */
    int32_t max_iteration;        /* max_iteration_ = 20 */
    int32_t min_effective_pts;    /* min_effective_pts_ = 10 */
    int32_t use_ann;              /* IcpOptions::use_ann: accepted and ignored — the search is always exact (deviation Q1) */
    double eps;                   /* eps_ = 1e-2 */
    double max_nn_distance;       /* max_nn_distance_ = 1.0 (compared with a squared distance, quirk Q6) */
    double max_plane_distance;    /* max_plane_distance_ = 0.1 */
    double max_line_distance;     /* max_line_distance_ = 0.5 (P2LINE: residual gate and FitLine's eps) */
    double voxel_size;            /* NdtOptions::voxel_size_ = 1.0 (inv_voxel_size_ is always recomputed, ndt_registration.cpp:25) */
    double res_outlier_th;        /* res_outlier_th_ = 20.0 */
    int32_t min_pts_in_voxel;     /* min_pts_in_voxel_ = 3 */
    int32_t nearby_type;          /* enum locreg_nearby, default NEARBY6 */
    /* GPU-side knobs (no reference counterpart) */
    double knn_cell_size;         /* voxel-hash cell edge in metres for ICP k-NN; <= 0: 0.5 */
    int32_t loop_mode;            /* enum locreg_loop: how ONE ScanMatch keeps its loop on the device (batches always run
                                     the per-iteration pipeline: there is enough work per launch) */
    int32_t knn_lists;            /* 1 (default): build per-cell 3x3x3 neighbourhood lists (27x point storage) for the fast k-NN path */
    int32_t ndt_capacity;         /* NdtOptions::capacity_ = 100000: voxels the incremental NDT cache holds (LRU) */
    int32_t zero_initial_translation; /* 1 = IcpOptions::use_initial_translation_ == false or NdtOptions::remove_centroid_
                                         == true: Align* replaces the translation of the initial pose by target_center_ -
                                         source_center_ (icp_registration.cpp:272-276,311-314,352-355; ndt_registration.cpp:
                                         380-384), and both centres are never computed (the code that would is commented
                                         out, icp_registration.cpp:22-26,261-264), so the translation starts from ZERO.
                                         AlignIncNdt and CaculateMatrixHAndB do not look at the flag. */
} locreg_options;

/* Outcome of one registration (what the reference logs or silently drops, SURVEY.md §5). */
typedef struct locreg_result {
    int32_t iters;        /* Gauss-Newton loop trips executed */
    int32_t updates;      /* trips whose H/B evaluation succeeded and moved the pose */
    int32_t converged;    /* 1 if ||dx|| < eps ended the loop */
    int32_t degenerate;   /* 1 if the LAST evaluation failed (effective_num < min_effective_pts or det(H) == 0) */
    int64_t n_effective;  /* effective_num of the last evaluation */
    int64_t n_inlier;     /* residuals that entered H/B in the last evaluation */
    double sum_sq_res;    /* sum of squared gated residuals of the last evaluation */
    int32_t pose_written; /* 0 only on direct NDT's det(H)==0 early return, which leaves pose_out untouched (quirk Q11) */
    int32_t pad_;
} locreg_result;

typedef struct locreg_handle locreg_handle;

/* Fills *opt with the reference's defaults for `method`. */
int locreg_default_options(locreg_options* opt, int32_t method);

/* IcpRegistration(IcpOptions) / NdtRegistration(NdtOptions) constructors (icp_registration.hpp:59, ndt_registration.cpp:20). */
int locreg_create(const locreg_options* opt, int32_t device, locreg_handle** out);
int locreg_destroy(locreg_handle* h);
/* Use the caller's CUDA stream (a cudaStream_t) for all work of this handle; NULL = the handle's own stream. */
int locreg_set_stream(locreg_handle* h, void* cuda_stream);

/* MatchingInterface::SetInputTarget (matching_interface.h:18; icp_registration.cpp:9-29, ndt_registration.cpp:65-148).
 * Deep-copies the cloud to the device and builds the voxel-hash map (ICP) or the NDT voxel grid.  Incremental NDT:
 * the cloud is ADDED to the LRU voxel cache (SetIncNdtTargetCloud, ndt_registration.cpp:150-183). */
int locreg_set_target(locreg_handle* h, const float* xyz, size_t n, size_t stride_bytes);
/* Same, cloud already in device memory (stride as above). */
int locreg_set_target_device(locreg_handle* h, const float* d_xyz, size_t n, size_t stride_bytes);

/* MatchingInterface::ScanMatch (matching_interface.h:30-33; icp_registration.cpp:216-244, ndt_registration.cpp:238-261).
 * pose_out is IN/OUT: on direct NDT's det(H)==0 early return it is left as the caller passed it.  out_xyz (may be
 * NULL) receives pcl::transformPointCloud(src, pose_out) with the same stride; bytes 12.. of each point are copied. */
int locreg_align(locreg_handle* h, const float* src, size_t n, size_t stride_bytes, const double* pose_in,
                 double* pose_out, float* out_xyz, locreg_result* res);

/* MatchingInterface::CaculateMatrixHAndB (matching_interface.h:23-26; icp_registration.cpp:31-55).
 * Returns 1/0 in res->degenerate's complement like the reference's bool; NDT's reference body is empty (quirk Q12),
 * here it returns the loop-body accumulation of AlignNdt (ndt_registration.cpp:399-433). */
int locreg_compute_hb(locreg_handle* h, const float* src, size_t n, size_t stride_bytes, const double* pose,
                      double* H36, double* B6, locreg_result* res);

/* LoamRegistration::ScanMatch's loop (loam_registration.cpp:38-99, SURVEY 3.3) on the device, with no host round trip
 * between iterations.  Per trip, at the current pose: the surf cloud's H/B on the `surf` handle (LOCREG_ICP_P2PLANE)
 * and the edge cloud's on the `edge` handle (LOCREG_ICP_P2LINE), each with its own handle's gates, exactly as
 * locreg_compute_hb computes them; H = Hs + He, B = Bs + Be (the halves' degenerate flags do not gate the sum);
 * dx = H^-1 B; R <- R Exp(dx[0:3]), t <- t + dx[3:6]; stop when |dx| < eps or after max_iteration trips.  A trip with
 * det(H) == 0 makes no update.  The loop starts from pose_in as given (zero_initial_translation does not apply); the
 * handles' own max_iteration / eps are not used.  The two halves of a trip run concurrently on the two handles'
 * streams (serially when both were given the same stream with locreg_set_stream).  Clouds share one stride; either may
 * be empty (that half contributes zeros).  pose_out is always written.  res2 (may be NULL) has 2 entries, [0] surf and
 * [1] edge: iters / updates / converged / pose_written are the loop's (equal in both), degenerate / n_effective /
 * n_inlier / sum_sq_res that half's last evaluation, as locreg_compute_hb reports it at that pose.
 * locreg_last_timing(surf) reports the call's kernels.  Both handles need a target (LOCREG_E_STATE). */
int locreg_align_loam(locreg_handle* surf, locreg_handle* edge, const float* surf_xyz, size_t n_surf, const float* edge_xyz,
                      size_t n_edge, size_t stride_bytes, const double* pose_in, int32_t max_iteration, double eps,
                      double* pose_out, locreg_result* res2);
/* S independent locreg_align_loam calls against the current surf and edge targets, in one device-resident loop: every
 * trip evaluates all S scans' surf halves on the surf handle and their edge halves on the edge handle, then one warp
 * per scan solves.  Scan s is surf points [surf_offsets[s], surf_offsets[s+1]) of surf_xyz and edge points
 * [edge_offsets[s], edge_offsets[s+1]) of edge_xyz (offsets relative to their cloud pointer; both clouds share one
 * stride; any half may be empty).  poses_in / poses_out are S*7 doubles; poses_out is always written.  results (may
 * be NULL) has 2*S entries: [2s] and [2s+1] are scan s's res2 of locreg_align_loam.  Each scan's pose and results are
 * bit-identical to a locreg_align_loam call on that scan alone; a scan that stops early does not affect the others.
 * Arguments are checked before any device work (LOCREG_E_ARG: handles as in locreg_align_loam, offsets negative or
 * decreasing, stride or pointers, S >= 2^31; LOCREG_E_STATE: a handle without a target).  S == 0 does nothing.
 * locreg_last_timing(surf) reports the call's kernels. */
int locreg_align_loam_batch(locreg_handle* surf, locreg_handle* edge, const float* surf_xyz, const int64_t* surf_offsets,
                            const float* edge_xyz, const int64_t* edge_offsets, size_t stride_bytes, const double* poses_in,
                            size_t S, int32_t max_iteration, double eps, double* poses_out, locreg_result* results);
/* locreg_align_loam_batch over all ranks of the SURF handle's communicator (the edge handle's is not used; none, or a
 * one-rank communicator: it IS locreg_align_loam_batch, with the same launches and no NCCL call).  The batch has
 * S_global scans; this rank owns the block [lo, hi) = locreg_shard_range(S_global, rank, world) and passes ONLY that
 * block, as in locreg_align_batch_sharded: surf_offsets / edge_offsets (S_local + 1 entries each, relative to their
 * cloud pointer) and poses_in (S_local * 7) with S_local = hi - lo.  EVERY rank passes the same S_global,
 * max_iteration and eps.  A rank may own no scan (S_global < world): it runs no registration but joins the exchange,
 * and may pass NULL offsets and poses_in.  No collective on the data path; at the end, on surf's stream, each block's
 * poses, loop results and half records (200 bytes per scan) reach every rank with one grouped ncclBroadcast per rank
 * block (an all-gather with ragged counts).  poses_out (S_global * 7, always written) and results (2 * S_global
 * entries or NULL, [2s] surf and [2s+1] edge as in locreg_align_loam_batch) are complete on every rank and bit for bit
 * what locreg_align_loam_batch returns on one GPU for the whole batch.  Arguments are checked before any device work
 * and any collective (LOCREG_E_ARG: handles as in locreg_align_loam, S_global >= 2^31, S_local not this rank's block,
 * this block's offsets negative or decreasing, stride or pointers, a null poses_out; LOCREG_E_STATE: a handle
 * without a target).  S_global == 0 does nothing.  locreg_last_timing(surf) covers the kernels and the exchange. */
int locreg_align_loam_batch_sharded(locreg_handle* surf, locreg_handle* edge, const float* surf_xyz,
                                    const int64_t* surf_offsets, const float* edge_xyz, const int64_t* edge_offsets,
                                    size_t stride_bytes, const double* poses_in, size_t S_local, size_t S_global,
                                    int32_t max_iteration, double eps, double* poses_out, locreg_result* results);

/* Parity probe for SearchPointInterface::FindNearstPoints (search_point_interface.h:9-24; kdtree.cpp:272-283):
 * exact k-NN (k = 1 or 5) under the total order (float32 dis2, index); idx is nq*k, -1 padded. ICP handles only.
 * Runs the production search: stage 1 per thread, then the queued rest per warp (small probes, like one scan) or per
 * thread (large probes, like a batch). */
int locreg_knn(locreg_handle* h, const float* queries, size_t nq, size_t stride_bytes, int32_t k, int32_t* idx);

/* Parity probe: per-point gate code (0 skipped, 1 plane fit failed, 2 residual gated out, 3 inlier; NDT: number
 * of gated-in voxels) and, for ICP, neighbour indices (n*k, may be NULL) at `pose`. */
int locreg_debug_points(locreg_handle* h, const float* src, size_t n, size_t stride_bytes, const double* pose,
                        uint8_t* gate, int32_t* nn);

/* Batch offline mapping (BASELINE config 4): S independent ScanMatch calls against the current target.
 * Scan s is points [offsets[s], offsets[s+1]) of `srcs`; poses_in/poses_out are S*7 doubles (poses_out is IN/OUT as
 * in locreg_align); results is S entries or NULL.
 * Pass `srcs` in page-locked memory (cudaHostAlloc / cudaHostRegister) when the batch is large (>= 16 scans and >= 1 M
 * points): the batch is then cut into chunks of whole scans whose host-to-device copies hide behind the registration of
 * the chunks before them, each chunk on its own stream (782 against 830 M points/s with the scans already on the
 * device; pageable memory: one staged copy up front, ~610 M).  The poses do not depend on the chunking. */
int locreg_align_batch(locreg_handle* h, const float* srcs, const int64_t* offsets, size_t stride_bytes,
                       const double* poses_in, size_t S, double* poses_out, locreg_result* results);
/* Same with every buffer already on the device: d_srcs is float4 (stride 16). */
int locreg_align_batch_device(locreg_handle* h, const float* d_srcs, const int64_t* d_offsets, const double* d_poses_in,
                              size_t S, size_t total_points, double* d_poses_out, locreg_result* d_results);

/* Global relocalisation (BASELINE config 5): n_hyp ScanMatch calls of ONE scan from different initial poses.
 * score = sum_sq_res / n_inlier at the final pose (+inf when the last evaluation is degenerate or has no inlier);
 * best = argmin with lowest index winning ties.  scores / poses_out may be NULL.  The cross-GPU argmin is one
 * min-allreduce of locreg_pack_score(score, global index) (see loc_lib_b200/dist.py). */
int locreg_relocalise(locreg_handle* h, const float* src, size_t n, size_t stride_bytes, const double* poses_in,
                      size_t n_hyp, double* best_pose, int64_t* best_idx, double* best_score, double* scores,
                      double* poses_out);
/* (float32 score bits << 32) | index: unsigned order = (score, index) order for score >= 0. */
uint64_t locreg_pack_score(double score, uint32_t index);

/* Staged global relocalisation: locreg_relocalise in n_rounds rounds, with the hypotheses that score worst dropped
 * between rounds, so that far-off hypotheses do not pay for every trip.  It is the chain
 *     alive = [0, n_hyp) (ascending original index); pose[i] = poses_in[i]
 *     for r in 0 .. n_rounds-1:
 *         every alive i runs locreg_relocalise's loop and score pass from pose[i] with trips[r] trips (the handle's eps
 *         and gates; zero_initial_translation applies in round 0 only; later rounds start from the pose exactly as the
 *         previous round left it) -> pose[i], score[i] (score as in locreg_relocalise)
 *         if r < n_rounds-1: alive = the min(keep[r], |alive|) alive i with the smallest locreg_pack_score(score[i], i)
 *     best = argmin over the last round's alive of locreg_pack_score(score[i], i) (lowest index on ties)
 * Each round is a fresh loop: only the pose is carried over, no search state, so round r of hypothesis i is bit for
 * bit what locreg_relocalise returns from that pose on a handle whose max_iteration is trips[r].  The handle's own
 * max_iteration is not used, and its options are unchanged afterwards; trips[r] == 0 is a score-only round.  The
 * cut ranks each hypothesis by its own score, so it does not depend on how hypotheses are grouped on the device.
 * Every handle type locreg_relocalise accepts works (ICP and both NDT methods).  All rounds are queued back to back
 * (the survivors are selected and gathered on the device) and the call synchronises once.
 *   trips      n_rounds entries >= 0
 *   keep       n_rounds - 1 entries >= 1 (may be NULL when n_rounds == 1)
 *   scores / poses_out / rounds_out (n_hyp, n_hyp * 7, n_hyp; each may be NULL): every hypothesis's score and pose of
 *              the last round it ran, and how many rounds it ran (1 .. n_rounds)
 *   best_pose  poses_out[best_idx] bit for bit; best_score its score
 * locreg_last_timing covers the kernels of all rounds.  Arguments are checked before any device work: LOCREG_E_ARG
 * for bad cloud arguments (as locreg_relocalise), a null poses_in, n_hyp == 0 or n_hyp >= 2^31, n_rounds outside
 * [1, 32], a null trips or trips[r] < 0, a null keep with n_rounds > 1, keep[r] < 1; LOCREG_E_STATE without a target. */
int locreg_relocalise_staged(locreg_handle* h, const float* src, size_t n, size_t stride_bytes, const double* poses_in,
                             size_t n_hyp, const int32_t* trips, const int64_t* keep, int32_t n_rounds, double* best_pose,
                             int64_t* best_idx, double* best_score, double* scores, double* poses_out, int32_t* rounds_out);

/* ---- multi-GPU (SURVEY.md 8e): one process (or thread) per GPU, one handle each, NCCL inside this library -----------
 * The two workloads that shard keep a replica of the map per GPU and need ONE exchange step each; it runs on the
 * handle's stream right behind the kernels, so nothing returns to the host in between.  NCCL is bound at run time
 * (dlopen of libnccl.so.2: the copy already in the process - e.g. torch's - or the system's), so single-GPU users
 * need no NCCL at all; without it these entry points fail with LOCREG_E_UNSUPPORTED.
 *   locreg_comm_unique_id   ncclGetUniqueId: call on ONE rank, hand the 128 bytes to every rank (MPI, a file, a socket,
 *                           torch.distributed ...)
 *   locreg_comm_init        ncclCommInitRank for this handle's device; collective over all `world` ranks
 *   locreg_comm_destroy     ncclCommDestroy (also done by locreg_destroy)
 *   locreg_shard_range      the block partition [lo, hi) of n items rank `rank` owns (remainder to the first ranks) */
#define LOCREG_UNIQUE_ID_BYTES 128
int locreg_comm_unique_id(unsigned char* id128);
int locreg_comm_init(locreg_handle* h, const unsigned char* id128, int32_t rank, int32_t world);
int locreg_comm_destroy(locreg_handle* h);
int locreg_comm_info(locreg_handle* h, int32_t* rank, int32_t* world, int32_t* nccl_version);
int locreg_shard_range(size_t n, int32_t rank, int32_t world, size_t* lo, size_t* hi);

/* Global relocalisation over all ranks of the handle's communicator (BASELINE config 5).  EVERY rank passes the same
 * scan and the same n_hyp hypotheses; rank r registers hypotheses r, r + world, ... (neighbouring hypotheses cost
 * alike, far-off ones several times more: a strided deal balances the ranks), reduces its scores to one packed key
 * (locreg_pack_score) on the device, and then, on the handle's stream:
 *     ncclAllReduce(key, ncclUint64, ncclMin, count 1)       the argmin, lowest global index winning ties
 *     ncclBroadcast(8 doubles: pose + score, root = winner's owner)
 * best_pose / best_idx (GLOBAL hypothesis index) / best_score are identical on every rank.  A handle without a
 * communicator behaves as world = 1 (no NCCL call). */
int locreg_relocalise_sharded(locreg_handle* h, const float* src, size_t n, size_t stride_bytes, const double* poses_in,
                              size_t n_hyp, double* best_pose, int64_t* best_idx, double* best_score);

/* locreg_relocalise_staged over all ranks of the handle's communicator (none, or a one-rank communicator: it IS
 * locreg_relocalise_staged).  EVERY rank passes the same scan, the same n_hyp hypotheses and the same schedule.  In
 * round r the m alive hypotheses (positions 0 .. m-1 in ascending original index, the same list on every rank) are
 * dealt by position: rank q runs positions q, q + world, ... (round 0 is locreg_relocalise_sharded's deal; after every
 * cut the survivors are dealt afresh, so the ranks stay balanced to one hypothesis).  Then, on the handle's stream,
 *     ncclAllGather(ceil(m / world) records of 8 doubles: pose + score, in place)
 * gives every rank the whole round, and every rank makes the same cut (and at the end picks the same winner) on the
 * device.  Every output - best_pose, best_idx, best_score, scores, poses_out, rounds_out (each may be NULL) - is bit
 * for bit what locreg_relocalise_staged returns on one GPU with the same arguments, on every rank.  Each round moves
 * m * 64 bytes through the all-gather; a rank with no hypothesis in a round runs no registration but joins the
 * collective.  Argument checks and error codes are those of locreg_relocalise_staged; the handle's options are
 * unchanged afterwards; locreg_last_timing covers all rounds and their collectives. */
int locreg_relocalise_staged_sharded(locreg_handle* h, const float* src, size_t n, size_t stride_bytes,
                                     const double* poses_in, size_t n_hyp, const int32_t* trips, const int64_t* keep,
                                     int32_t n_rounds, double* best_pose, int64_t* best_idx, double* best_score,
                                     double* scores, double* poses_out, int32_t* rounds_out);

/* LOAM global relocalisation: n_hyp locreg_align_loam calls of ONE surf / edge scan from different initial poses, in
 * one device-resident loop (hypotheses run in waves that bound the per-point scratch; the waves do not change results).
 *   loop     hypothesis i runs the LOAM loop of locreg_align_loam from poses_in[i] (7 doubles) as given, with the same
 *            max_iteration / eps, the same singular-H rule and each half's own gates; zero_initial_translation does
 *            not apply.
 *   score    after the loop both halves are evaluated once more at the final pose; score = (sum_sq_res_surf +
 *            sum_sq_res_edge) / (n_inlier_surf + n_inlier_edge) from that pass: the plain sum of what the two halves
 *            report, unweighted.  +inf when det(H_surf + H_edge) == 0 there or neither half has an inlier; the halves'
 *            own degenerate flags do not gate it.
 *   best     the argmin of locreg_pack_score(score, index), lowest index winning ties; index 0 when every score is
 *            +inf.  best_pose is poses_out[best] bit for bit.
 * scores (n_hyp) and poses_out (n_hyp * 7) may be NULL.  Clouds share one stride; either may be empty (that half
 * contributes zeros).  locreg_last_timing(surf) reports the call's kernels.  Arguments are checked before any device
 * work: LOCREG_E_ARG for the handles as in locreg_align_loam, bad cloud arguments, a null poses_in, n_hyp == 0 or
 * n_hyp >= 2^31; LOCREG_E_STATE for a handle without a target. */
int locreg_relocalise_loam(locreg_handle* surf, locreg_handle* edge, const float* surf_xyz, size_t n_surf,
                           const float* edge_xyz, size_t n_edge, size_t stride_bytes, const double* poses_in, size_t n_hyp,
                           int32_t max_iteration, double eps, double* best_pose, int64_t* best_idx, double* best_score,
                           double* scores, double* poses_out);
/* locreg_relocalise_loam over all ranks of the SURF handle's communicator (the edge handle's is not used; none: world
 * = 1).  Every rank passes the same clouds and all n_hyp hypotheses and registers hypotheses rank, rank + world, ...;
 * then, on surf's stream, one ncclAllReduce(MIN) of the packed key and the owner's ncclBroadcast of pose + score, as in
 * locreg_relocalise_sharded.  best_* are identical on every rank.  locreg_last_timing(surf) covers the kernels and the
 * collectives.  Argument errors as in locreg_relocalise_loam. */
int locreg_relocalise_loam_sharded(locreg_handle* surf, locreg_handle* edge, const float* surf_xyz, size_t n_surf,
                                   const float* edge_xyz, size_t n_edge, size_t stride_bytes, const double* poses_in,
                                   size_t n_hyp, int32_t max_iteration, double eps, double* best_pose, int64_t* best_idx,
                                   double* best_score);

/* Staged LOAM relocalisation: locreg_relocalise_staged's rounds over locreg_relocalise_loam's loop and score.  Round r
 * runs locreg_relocalise_loam over the hypotheses still alive, with max_iteration = trips[r] and the caller's eps, from
 * the poses the previous round left (round 0: poses_in); after it only the min(keep[r], alive) hypotheses with the
 * smallest locreg_pack_score(score, original index) go on, in ascending original index.  The winner is the smallest key
 * of the last round.  Poses are used as given in every round: the LOAM loop ignores zero_initial_translation.
 * Each round is a fresh loop: only the pose is carried over, so round r of hypothesis i is bit for bit what
 * locreg_relocalise_loam returns from that pose with max_iteration = trips[r].  The score is locreg_relocalise_loam's;
 * trips[r] == 0 is a score-only round.  Neither handle's options are used for the schedule or changed.  All rounds are
 * queued back to back on surf's stream (edge's stream joins it every round) and the call synchronises once.
 *   trips      n_rounds entries >= 0
 *   keep       n_rounds - 1 entries >= 1 (may be NULL when n_rounds == 1)
 *   scores / poses_out / rounds_out (n_hyp, n_hyp * 7, n_hyp; each may be NULL): every hypothesis's score and pose of
 *              the last round it ran, and how many rounds it ran (1 .. n_rounds)
 *   best_pose  poses_out[best_idx] bit for bit; best_score its score
 * locreg_last_timing(surf) covers the kernels of all rounds.  Arguments are checked before any device work: LOCREG_E_ARG
 * for the handles and clouds as in locreg_relocalise_loam, a null poses_in, n_hyp == 0 or n_hyp >= 2^31, and the
 * schedule as in locreg_relocalise_staged (n_rounds outside [1, 32], a null trips or trips[r] < 0, a null keep with
 * n_rounds > 1, keep[r] < 1); LOCREG_E_STATE for a handle without a target. */
int locreg_relocalise_loam_staged(locreg_handle* surf, locreg_handle* edge, const float* surf_xyz, size_t n_surf,
                                  const float* edge_xyz, size_t n_edge, size_t stride_bytes, const double* poses_in,
                                  size_t n_hyp, const int32_t* trips, const int64_t* keep, int32_t n_rounds, double eps,
                                  double* best_pose, int64_t* best_idx, double* best_score, double* scores,
                                  double* poses_out, int32_t* rounds_out);
/* locreg_relocalise_loam_staged over all ranks of the SURF handle's communicator (the edge handle's is not used; none,
 * or a one-rank communicator: it IS locreg_relocalise_loam_staged, with the same launches).  Every rank passes the same
 * clouds, hypotheses and schedule.  Each round's alive hypotheses are dealt by position and exchanged with one in-place
 * ncclAllGather of pose + score on surf's stream, as in locreg_relocalise_staged_sharded.  Every output is bit for bit
 * what locreg_relocalise_loam_staged returns on one GPU, on every rank.  Argument errors as in
 * locreg_relocalise_loam_staged; locreg_last_timing(surf) covers all rounds and their collectives. */
int locreg_relocalise_loam_staged_sharded(locreg_handle* surf, locreg_handle* edge, const float* surf_xyz, size_t n_surf,
                                          const float* edge_xyz, size_t n_edge, size_t stride_bytes,
                                          const double* poses_in, size_t n_hyp, const int32_t* trips, const int64_t* keep,
                                          int32_t n_rounds, double eps, double* best_pose, int64_t* best_idx,
                                          double* best_score, double* scores, double* poses_out, int32_t* rounds_out);

/* Batch offline mapping over all ranks (BASELINE config 4).  The batch has S_global scans; this rank owns the block
 * [lo, hi) = locreg_shard_range(S_global, rank, world) and passes ONLY that block: srcs / offsets (S_local + 1
 * entries, relative to srcs) / poses_in (S_local * 7) with S_local = hi - lo.  No collective on the data path; at the
 * end the poses (and results) of all blocks are exchanged on the handle's stream with one grouped
 * ncclBroadcast per rank (an all-gather with ragged counts), so poses_out (S_global * 7, IN/OUT as in locreg_align)
 * and results (S_global entries or NULL) are complete on every rank. */
int locreg_align_batch_sharded(locreg_handle* h, const float* srcs, const int64_t* offsets, size_t stride_bytes,
                               const double* poses_in, size_t S_local, size_t S_global, double* poses_out,
                               locreg_result* results);

/* pcl::transformPointCloud (icp_registration.cpp:241) on its own. */
int locreg_transform_cloud(locreg_handle* h, const float* src, size_t n, size_t stride_bytes, const double* pose,
                           float* out_xyz);

/* Cloud pre-filters the reference runs right before SetInputTarget / ScanMatch (CloudFilterInterface:
 * LocUtils/src/model/cloud_filter/{voxel_filter,box_filter}.cpp; RemoveNanPoint, point_cloud_utils.h:13-20), on the
 * device.  out_xyz has room for n points of the same stride; *n_out receives the number written.
 *   remove_nan : pcl::removeNaNFromPointCloud - points with finite x, y, z, order kept
 *   crop_box   : pcl::CropBox(min, max), identity transform - finite points with min <= p <= max per axis, order kept
 *   voxel_grid : pcl::VoxelGrid(leaf, leaf, leaf), all fields - per occupied voxel the float32 mean of every float
 *                word of its points (summed in point order), voxels in ascending PCL voxel index; when extent / leaf
 *                would overflow PCL's int voxel index (> 2^31 - 1 voxels) the cloud is returned unfiltered, as PCL does */
int locreg_filter_remove_nan(locreg_handle* h, const float* xyz, size_t n, size_t stride_bytes, float* out_xyz, size_t* n_out);
int locreg_filter_crop_box(locreg_handle* h, const float* xyz, size_t n, size_t stride_bytes, const float* min3,
                           const float* max3, float* out_xyz, size_t* n_out);
int locreg_filter_voxel_grid(locreg_handle* h, const float* xyz, size_t n, size_t stride_bytes, float leaf_size,
                             float* out_xyz, size_t* n_out);
/* pcl::removeNaNFromPointCloud / pcl::VoxelGrid of every scan of a batch; scan s = points [offsets[s], offsets[s+1])
 * of xyz (offsets relative to xyz, non-decreasing).  out_xyz has room for offsets[S] - offsets[0] points of the same
 * stride; out_offsets (S + 1, relative to out_xyz, out_offsets[0] = 0) receives the filtered batch's offsets.  Segment s
 * is byte for byte locreg_filter_remove_nan / locreg_filter_voxel_grid of scan s alone (empty scans, scans without a
 * finite point and scans whose grid would overflow PCL's int index included).  One pass over the whole batch: the
 * launches do not depend on S, and the call synchronises twice (voxel grid: once after the per-scan bounding boxes,
 * once at the end; NaN removal: once).  The voxel grid's per-scan bitmaps are processed in waves of at most
 * LOCREG_FILTER_WAVE_MIB MiB (default 1 GiB, less when free memory is short); the waves do not change results.
 * Arguments are checked before any device work: LOCREG_E_ARG for a null offsets / out_offsets, a null out_xyz with
 * points in the batch, decreasing or negative offsets, bad cloud arguments, S >= 2^31, leaf_size <= 0.
 * locreg_last_timing covers the filter kernels. */
int locreg_filter_remove_nan_batch(locreg_handle* h, const float* xyz, const int64_t* offsets, size_t S,
                                   size_t stride_bytes, float* out_xyz, int64_t* out_offsets);
int locreg_filter_voxel_grid_batch(locreg_handle* h, const float* xyz, const int64_t* offsets, size_t S,
                                   size_t stride_bytes, float leaf_size, float* out_xyz, int64_t* out_offsets);

/* Loc::Update's front end and ScanMatch for every scan of a batch: scan s is RemoveNanPoint then VoxelFilter(leaf_size)
 * (the order of loc.cpp:217-218; lio.cpp's order gives the same cloud), then registered exactly as locreg_align_batch
 * registers it.  The filtered clouds never leave the device.  poses_in / poses_out / results as in locreg_align_batch;
 * n_filtered (S entries or NULL) receives each filtered scan's size.  Poses and results are bit for bit those of
 * locreg_align_batch on the concatenation of locreg_filter_voxel_grid(locreg_filter_remove_nan(scan s)).  Every handle
 * type locreg_align_batch accepts works.  The raw batch goes to the device in one copy (not in chunks).  Arguments are
 * checked before any device work as in locreg_align_batch, plus LOCREG_E_ARG for leaf_size <= 0; a failing call
 * writes nothing.  locreg_last_timing covers the filter and the registration kernels. */
int locreg_align_batch_filtered(locreg_handle* h, const float* srcs, const int64_t* offsets, size_t stride_bytes,
                                const double* poses_in, size_t S, float leaf_size, double* poses_out,
                                locreg_result* results, int64_t* n_filtered);

/* Caller state kept on the device (Loc, LocUtils/src/slam/3d/loc.cpp): the global map is uploaded once
 * (Loc::InitGlobalMap, loc.cpp:268-283); locreg_reset_local_map is Loc::ResetLocalMap (loc.cpp:187-206) -
 * BoxFilter::SetOrigin(origin) + Filter (crop to origin +- half_size) + SetInputTarget(local map) - with the crop and
 * the index build both on the device; *n_local (may be NULL) receives the size of the local map. */
int locreg_set_global_map(locreg_handle* h, const float* xyz, size_t n, size_t stride_bytes);
int locreg_reset_local_map(locreg_handle* h, const float* origin3, const float* half_size3, size_t* n_local);

/* Lio's sliding local map of key frames (Lio::AddCloud, LocUtils/src/slam/3d/lio.cpp:238-307), kept on the device.
 * locreg_local_map_add_keyframe: key_frame = pcl::transformPointCloud(scan, pose.matrix()) - the Matrix4d is passed
 * without a cast (:243,:278), so PCL evaluates in double and casts once to float; ScanMatch's result cloud is the one
 * that uses the float32 matrix - joins the window (:281).  If the window then holds more than max_keyframes scans the oldest is dropped and the local map is
 * rebuilt as the concatenation of the scans left (:283-292); otherwise the key frame is appended to the local map as it
 * stands, i.e. to the OUTPUT of the previous filter pass (:294-297).  The local map is voxel-grid filtered in place with
 * leaf size `leaf` (local_map_filter_ptr_->Filter, :299; leaf <= 0: NoFilter) and becomes the registration target
 * (:307) - for LOCREG_NDT_INCREMENTAL the key frame alone is added to the voxel cache (:301-303).  Nothing but the scan
 * crosses PCIe.  *n_local (may be NULL) receives the size of the local map.  The call is transactional: when a step
 * fails (out of memory) the window and the local
 * map are left as they were.
 * locreg_local_map_get copies the local map to the host (parity probe / PCD dump); locreg_local_map_clear forgets it. */
int locreg_local_map_add_keyframe(locreg_handle* h, const float* scan_xyz, size_t n, size_t stride_bytes, const double* pose7,
                                  int32_t max_keyframes, float leaf, size_t* n_local);
int locreg_local_map_get(locreg_handle* h, float* out_xyz, size_t capacity_points, size_t* n_local, size_t* stride_bytes);
int locreg_local_map_clear(locreg_handle* h);

/* NDT parity probe: voxel count and, sorted by (kx,ky,kz), keys (nv*3), mu (nv*3), info (nv*9 row-major), npts (nv). */
int locreg_ndt_num_voxels(locreg_handle* h, size_t* nv);
int locreg_ndt_get_voxels(locreg_handle* h, int32_t* keys, double* mu, double* info, int32_t* npts);

/* Device time in milliseconds of the last align / align_batch / relocalise / set_target call's kernels
 * (CUDA events on the handle's stream), and how many kernels that call launched. */
int locreg_last_timing(locreg_handle* h, double* kernel_ms, int64_t* launches);
/* Size of the search index the last locreg_set_target* built (diagnostics / bench): bytes of device memory over all
 * levels, points indexed, neighbourhood lists (ICP; 0 for NDT) or voxels (NDT).  Any pointer may be NULL. */
int locreg_index_info(locreg_handle* h, size_t* bytes, size_t* points, size_t* lists_or_voxels);

/* Per-kernel-class device timing for the ICP pipeline (0 neighbour search stage 1, 1 fit + reduce, 2 solve,
 * 3 neighbour search stage 2): returns and clears the milliseconds / launch counts (4 entries each) accumulated
 * since the last call, then switches the instrumentation (a CUDA event pair around every launch) on or off.
 * Off by default; meant for bench.py's roofline pass. */
int locreg_profile(locreg_handle* h, int32_t enable, double* ms4, int64_t* launches4);

const char* locreg_last_error(void);
const char* locreg_version(void);

#ifdef __cplusplus
}
#endif
#endif
