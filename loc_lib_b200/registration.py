"""Host-side mirror of the reference's registration interface over the C ABI.

Same names, argument meaning and return behaviour as LocUtils::MatchingInterface
(LocUtils/include/LocUtils/model/matching/3d/matching_interface.h:13-54) and its two implementations
IcpRegistration (icp_registration.hpp:41-142) and NdtRegistration (ndt_registration.hpp:69-135):
    SetInputTarget(cloud) -> bool
    ScanMatch(cloud, predict_pose) -> (True, result_cloud, result_pose)      # ScanMatch always returns true
    CaculateMatrixHAndB(cloud, predict_pose) -> (bool, H, B)
    GetFitnessScore() -> 0.0                                                  # always 0 in the reference
Clouds are (n, >=3) float32 numpy arrays (row stride = point stride, e.g. (n, 8) for pcl::PointXYZI's 32 B);
poses are 7 doubles [qx qy qz qw tx ty tz] (Sophus::SE3d::data()).  All computation happens in the CUDA
kernels behind liblocreg.so; there is no CPU path.
"""
import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _lib
from ._lib import (ICP_P2P, ICP_P2LINE, ICP_P2PLANE, NDT_DIRECT, NDT_INCREMENTAL, NEARBY6, NEARBY_CENTER,  # noqa: F401
                   LOOP_PERSISTENT, LOOP_GRAPH)


class IcpMethod:  # icp_registration.hpp:15-20
    P2P, P2LINE, P2PLANE, PCLICP = 0, 1, 2, 3


class NdtNearbyType:  # ndt_registration.hpp:16-20
    CENTER, NEARBY6 = 0, 1


class NdtMethod:  # ndt_registration.hpp:21-26
    PCL_NDT, DIRECT_NDT, INCREMENTAL_NDT = 0, 1, 2


@dataclass
class IcpOptions:  # icp_registration.hpp:22-39
    max_iteration_: int = 20
    max_nn_distance_: float = 1.0
    max_plane_distance_: float = 0.1
    max_line_distance_: float = 0.5
    min_effective_pts_: int = 10
    eps_: float = 1e-2
    euc_fitness_eps_: float = 0.36
    use_initial_translation_: bool = True
    use_ann: bool = False
    method_: int = IcpMethod.P2P
    # GPU-side knobs
    knn_cell_size: float = 0.5
    knn_lists: bool = True
    loop_mode: int = LOOP_PERSISTENT


@dataclass
class NdtOptions:  # ndt_registration.hpp:27-42
    max_iteration_: int = 20
    voxel_size_: float = 1.0
    inv_voxel_size_: float = 1.0  # ignored: recomputed from voxel_size_ (ndt_registration.cpp:25)
    min_effective_pts_: int = 10
    min_pts_in_voxel_: int = 3
    max_pts_in_voxel_: int = 50
    eps_: float = 1e-2
    res_outlier_th_: float = 20.0
    remove_centroid_: bool = False
    capacity_: int = 100000
    nearby_type_: int = NdtNearbyType.NEARBY6
    method_: int = NdtMethod.DIRECT_NDT
    loop_mode: int = LOOP_PERSISTENT


def _cloud(a):
    """(array, point count, point stride in bytes) of an (n, >= 3) float32 cloud; anything that is not a C-contiguous
    float32 matrix (other dtypes, sliced views) is copied first, so that the row stride is always shape[1] * 4 and an
    output array made with empty_like has the same layout."""
    a = np.asarray(a)
    if a.dtype != np.float32 or a.ndim != 2 or a.shape[1] < 3 or not a.flags.c_contiguous:
        a = np.ascontiguousarray(a, np.float32)
        assert a.ndim == 2 and a.shape[1] >= 3, "cloud must be (n, >=3) float32"
    return a, a.shape[0], a.shape[1] * 4


def _pose(p):
    p = np.ascontiguousarray(p, np.float64)
    assert p.shape == (7,), "pose must be 7 doubles [qx qy qz qw tx ty tz]"
    return p


def _schedule(trips, keep):
    """(trips int32, keep int64) of a staged relocalisation; keep has len(trips) - 1 entries."""
    trips = np.ascontiguousarray(trips, np.int32).reshape(-1)
    keep = np.ascontiguousarray([] if keep is None else keep, np.int64).reshape(-1)
    if keep.shape[0] != max(trips.shape[0] - 1, 0):
        raise ValueError("keep must have len(trips) - 1 entries")
    return trips, keep


class _Registration:
    """Common C-ABI plumbing; subclasses only build the options."""

    def __init__(self, copt, device=0):
        self._h = C.c_void_p()
        self._opt = copt
        _lib.check(_lib.lib().locreg_create(C.byref(copt), device, C.byref(self._h)))
        self.last_result = None

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            _lib.lib().locreg_destroy(self._h)
            self._h = None

    __del__ = close

    def set_stream(self, cuda_stream):
        _lib.check(_lib.lib().locreg_set_stream(self._h, C.c_void_p(cuda_stream)))

    # ---- MatchingInterface ----
    def SetInputTarget(self, cloud):
        a, n, s = _cloud(cloud)
        _lib.check(_lib.lib().locreg_set_target(self._h, a.ctypes.data, n, s))
        return True

    def SetInputTargetDevice(self, dev_ptr, n, stride):
        _lib.check(_lib.lib().locreg_set_target_device(self._h, C.c_void_p(dev_ptr), n, stride))
        return True

    def ScanMatch(self, cloud, predict_pose, result_pose_init=None, want_cloud=True):
        a, n, s = _cloud(cloud)
        pin = _pose(predict_pose)
        pout = np.array([0, 0, 0, 1, 0, 0, 0], np.float64) if result_pose_init is None else \
            _pose(result_pose_init).copy()
        out = np.empty_like(a) if want_cloud else None
        res = _lib.Result()
        _lib.check(_lib.lib().locreg_align(self._h, a.ctypes.data, n, s, pin.ctypes.data, pout.ctypes.data,
                                           out.ctypes.data if want_cloud else None, C.byref(res)))
        self.last_result = res.as_dict()
        return True, out, pout

    def CaculateMatrixHAndB(self, cloud, predict_pose):
        a, n, s = _cloud(cloud)
        pin = _pose(predict_pose)
        H = np.zeros(36)
        B = np.zeros(6)
        res = _lib.Result()
        _lib.check(_lib.lib().locreg_compute_hb(self._h, a.ctypes.data, n, s, pin.ctypes.data, H.ctypes.data,
                                                B.ctypes.data, C.byref(res)))
        self.last_result = res.as_dict()
        return res.degenerate == 0, H.reshape(6, 6).T.copy(), B

    def GetFitnessScore(self):
        return 0.0  # icp_registration.cpp:246-250 / ndt_registration.cpp:466-471

    # ---- batch / relocalisation (new capabilities, BASELINE configs 4 and 5) ----
    def ScanMatchBatch(self, clouds, offsets, predict_poses, result_poses_init=None):
        a, n, s = _cloud(clouds)
        offsets = np.ascontiguousarray(offsets, np.int64)
        S = offsets.shape[0] - 1
        pin = np.ascontiguousarray(predict_poses, np.float64).reshape(S, 7)
        pout = pin.copy() if result_poses_init is None else np.ascontiguousarray(result_poses_init, np.float64).copy()
        res = (_lib.Result * S)()
        _lib.check(_lib.lib().locreg_align_batch(self._h, a.ctypes.data, offsets.ctypes.data, s, pin.ctypes.data, S,
                                                 pout.ctypes.data, res))
        return pout, [r.as_dict() for r in res]

    def Relocalise(self, cloud, hypotheses, want_all=False):
        a, n, s = _cloud(cloud)
        hyp = np.ascontiguousarray(hypotheses, np.float64).reshape(-1, 7)
        nh = hyp.shape[0]
        best_pose = np.zeros(7)
        best_idx = C.c_int64(-1)
        best_score = C.c_double(np.inf)
        scores = np.zeros(nh) if want_all else None
        poses = np.zeros((nh, 7)) if want_all else None
        _lib.check(_lib.lib().locreg_relocalise(self._h, a.ctypes.data, n, s, hyp.ctypes.data, nh,
                                                best_pose.ctypes.data, C.byref(best_idx), C.byref(best_score),
                                                scores.ctypes.data if want_all else None,
                                                poses.ctypes.data if want_all else None))
        return best_pose, int(best_idx.value), float(best_score.value), scores, poses

    def RelocaliseStaged(self, cloud, hypotheses, trips, keep, want_all=False):
        """Relocalise in len(trips) rounds of trips[r] Gauss-Newton trips, keeping the keep[r] best-scoring hypotheses
        after round r (keep has len(trips) - 1 entries; see locreg_relocalise_staged).  Returns (best_pose, best_idx,
        best_score, scores, poses, rounds): with want_all, every hypothesis's score and pose of the last round it ran and
        how many rounds it ran; otherwise the last three are None."""
        return self._relocalise_staged("locreg_relocalise_staged", cloud, hypotheses, trips, keep, want_all)

    def _relocalise_staged(self, symbol, cloud, hypotheses, trips, keep, want_all):
        a, n, s = _cloud(cloud)
        hyp = np.ascontiguousarray(hypotheses, np.float64).reshape(-1, 7)
        nh = hyp.shape[0]
        trips, keep = _schedule(trips, keep)
        best_pose = np.zeros(7)
        best_idx = C.c_int64(-1)
        best_score = C.c_double(np.inf)
        scores = np.zeros(nh) if want_all else None
        poses = np.zeros((nh, 7)) if want_all else None
        rounds = np.zeros(nh, np.int32) if want_all else None
        _lib.check(getattr(_lib.lib(), symbol)(self._h, a.ctypes.data, n, s, hyp.ctypes.data, nh, trips.ctypes.data,
                      keep.ctypes.data if keep.size else None, trips.shape[0],
                      best_pose.ctypes.data, C.byref(best_idx), C.byref(best_score),
                      scores.ctypes.data if want_all else None,
                      poses.ctypes.data if want_all else None,
                      rounds.ctypes.data if want_all else None))
        return best_pose, int(best_idx.value), float(best_score.value), scores, poses, rounds

    # ---- multi-GPU: NCCL inside liblocreg.so (one process per GPU; see loc_lib_b200/dist.py for the torchrun plumbing) ----
    @staticmethod
    def CommUniqueId():
        """ncclGetUniqueId: 128 bytes to be created on ONE rank and handed to all of them."""
        buf = (C.c_ubyte * 128)()
        _lib.check(_lib.lib().locreg_comm_unique_id(buf))
        return bytes(buf)

    def CommInit(self, unique_id, rank, world):
        buf = (C.c_ubyte * 128).from_buffer_copy(bytes(unique_id))
        _lib.check(_lib.lib().locreg_comm_init(self._h, buf, int(rank), int(world)))

    def CommDestroy(self):
        _lib.check(_lib.lib().locreg_comm_destroy(self._h))

    def CommInfo(self):
        r, w, v = C.c_int32(), C.c_int32(), C.c_int32()
        _lib.check(_lib.lib().locreg_comm_info(self._h, C.byref(r), C.byref(w), C.byref(v)))
        return r.value, w.value, v.value

    def RelocaliseSharded(self, cloud, hypotheses):
        """All ranks pass the same scan and hypotheses; the argmin is one ncclAllReduce(MIN) on the handle's stream.
        Returns (best_pose, best GLOBAL index, best_score), identical on every rank."""
        a, n, s = _cloud(cloud)
        hyp = np.ascontiguousarray(hypotheses, np.float64).reshape(-1, 7)
        best_pose = np.zeros(7)
        best_idx = C.c_int64(-1)
        best_score = C.c_double(np.inf)
        _lib.check(_lib.lib().locreg_relocalise_sharded(self._h, a.ctypes.data, n, s, hyp.ctypes.data, hyp.shape[0],
                                                        best_pose.ctypes.data, C.byref(best_idx), C.byref(best_score)))
        return best_pose, int(best_idx.value), float(best_score.value)

    def RelocaliseStagedSharded(self, cloud, hypotheses, trips, keep, want_all=False):
        """RelocaliseStaged over all ranks of the handle's communicator (locreg_relocalise_staged_sharded): every rank
        passes the same scan, hypotheses and schedule; each round's alive hypotheses are dealt over the ranks and
        their results all-gathered on the handle's stream.  Returns the same 6-tuple as RelocaliseStaged, bit for bit
        what one GPU returns, on every rank."""
        return self._relocalise_staged("locreg_relocalise_staged_sharded", cloud, hypotheses, trips, keep, want_all)

    def ScanMatchBatchSharded(self, clouds, offsets, predict_poses, S_global):
        """This rank's block of a batch of S_global scans (block partition: shard_range); returns the poses and results
        of ALL scans, exchanged over NCCL on the handle's stream."""
        a, n, s = _cloud(clouds)
        offsets = np.ascontiguousarray(offsets, np.int64)
        S = offsets.shape[0] - 1
        pin = np.ascontiguousarray(predict_poses, np.float64).reshape(S, 7)
        rank, world, _ = self.CommInfo()
        lo = C.c_size_t()
        hi = C.c_size_t()
        _lib.check(_lib.lib().locreg_shard_range(S_global, rank, world, C.byref(lo), C.byref(hi)))
        pout = np.zeros((S_global, 7))
        pout[lo.value:hi.value] = pin
        res = (_lib.Result * S_global)()
        _lib.check(_lib.lib().locreg_align_batch_sharded(self._h, a.ctypes.data, offsets.ctypes.data, s, pin.ctypes.data, S,
                                                         S_global, pout.ctypes.data, res))
        return pout, [r.as_dict() for r in res]

    # ---- parity probes ----
    def Knn(self, queries, k):
        a, n, s = _cloud(queries)
        out = np.empty((n, k), np.int32)
        _lib.check(_lib.lib().locreg_knn(self._h, a.ctypes.data, n, s, k, out.ctypes.data))
        return out

    def DebugPoints(self, cloud, pose, k):
        a, n, s = _cloud(cloud)
        gate = np.zeros(n, np.uint8)
        nn = np.full((n, k), -1, np.int32) if k else None
        _lib.check(_lib.lib().locreg_debug_points(self._h, a.ctypes.data, n, s, _pose(pose).ctypes.data,
                                                  gate.ctypes.data, nn.ctypes.data if k else None))
        return gate, nn

    def TransformCloud(self, cloud, pose):
        a, n, s = _cloud(cloud)
        out = np.empty_like(a)
        _lib.check(_lib.lib().locreg_transform_cloud(self._h, a.ctypes.data, n, s, _pose(pose).ctypes.data,
                                                     out.ctypes.data))
        return out

    # ---- cloud pre-filters (CloudFilterInterface / RemoveNanPoint of the reference), on the device ----
    def _filter(self, fn, cloud, *args):
        a, n, s = _cloud(cloud)
        out = np.empty_like(a)
        n_out = C.c_size_t(0)
        _lib.check(fn(self._h, a.ctypes.data, n, s, *args, out.ctypes.data, C.byref(n_out)))
        return out[:n_out.value]

    def RemoveNanPoint(self, cloud):
        """pcl::removeNaNFromPointCloud (point_cloud_utils.h:13-20)."""
        return self._filter(_lib.lib().locreg_filter_remove_nan, cloud)

    def BoxFilter(self, cloud, min3, max3):
        """BoxFilter::Filter = pcl::CropBox(min, max) (box_filter.cpp:24-32)."""
        lo = np.ascontiguousarray(min3, np.float32)
        hi = np.ascontiguousarray(max3, np.float32)
        return self._filter(_lib.lib().locreg_filter_crop_box, cloud, lo.ctypes.data, hi.ctypes.data)

    def VoxelFilter(self, cloud, voxel_size):
        """VoxelFilter::Filter = pcl::VoxelGrid with a cubic leaf (voxel_filter.cpp:10-26)."""
        return self._filter(_lib.lib().locreg_filter_voxel_grid, cloud, C.c_float(voxel_size))

    # ---- Loc's map state on the device (loc.cpp:187-206, 268-283) ----
    def SetGlobalMap(self, cloud):
        a, n, s = _cloud(cloud)
        _lib.check(_lib.lib().locreg_set_global_map(self._h, a.ctypes.data, n, s))

    def ResetLocalMap(self, x, y, z, half_size=(150.0, 150.0, 150.0)):
        """Loc::ResetLocalMap: crop the global map to (x, y, z) +- half_size and make it the target; returns its size."""
        o = np.ascontiguousarray([x, y, z], np.float32)
        hs = np.ascontiguousarray(half_size, np.float32)
        n_local = C.c_size_t(0)
        _lib.check(_lib.lib().locreg_reset_local_map(self._h, o.ctypes.data, hs.ctypes.data, C.byref(n_local)))
        return n_local.value

    def AddKeyFrame(self, scan, pose, max_keyframes=10, leaf=0.5):
        """Lio::AddCloud's local-map update (lio.cpp:277-307) on the device: transform the key-frame scan by `pose`,
        slide the window of `max_keyframes` scans, voxel-filter the local map with `leaf` (<= 0: no filter) and make it
        the target (incremental NDT: add the key frame to the voxel cache).  Returns the size of the local map."""
        a, n, s = _cloud(scan)
        p = np.ascontiguousarray(pose, np.float64)
        n_local = C.c_size_t(0)
        _lib.check(_lib.lib().locreg_local_map_add_keyframe(self._h, a.ctypes.data, n, s, p.ctypes.data, int(max_keyframes),
                                                            float(leaf), C.byref(n_local)))
        return n_local.value

    def GetLocalMap(self):
        """The current sliding local map, copied to the host: (n, stride / 4) float32."""
        n, stride = C.c_size_t(0), C.c_size_t(0)
        _lib.check(_lib.lib().locreg_local_map_get(self._h, None, 0, C.byref(n), C.byref(stride)))
        out = np.empty((n.value, max(stride.value // 4, 3)), np.float32)
        if n.value:
            _lib.check(_lib.lib().locreg_local_map_get(self._h, out.ctypes.data, n.value, C.byref(n), C.byref(stride)))
        return out

    def ClearLocalMap(self):
        _lib.check(_lib.lib().locreg_local_map_clear(self._h))

    def profile(self, enable):
        """Returns ({'search','fit','solve','rings'} -> (ms, launches)) accumulated so far, then switches instrumentation."""
        ms = np.zeros(4)
        ln = np.zeros(4, np.int64)
        _lib.check(_lib.lib().locreg_profile(self._h, int(enable), ms.ctypes.data, ln.ctypes.data))
        return {k: (float(ms[i]), int(ln[i])) for i, k in enumerate(("search", "fit", "solve", "rings"))}

    def ScanMatchBatchDevice(self, d_srcs, d_offsets, d_poses_in, S, total_points, d_poses_out, d_results=0):
        """Batch ScanMatch with every buffer already in device memory (raw device pointers; clouds are float4)."""
        _lib.check(_lib.lib().locreg_align_batch_device(self._h, C.c_void_p(d_srcs), C.c_void_p(d_offsets),
                                                        C.c_void_p(d_poses_in), S, total_points,
                                                        C.c_void_p(d_poses_out), C.c_void_p(d_results)))

    def index_info(self):
        """(bytes of device memory, points indexed, neighbourhood lists or voxels) of the current target's search index."""
        b, p, l = C.c_size_t(0), C.c_size_t(0), C.c_size_t(0)
        _lib.check(_lib.lib().locreg_index_info(self._h, C.byref(b), C.byref(p), C.byref(l)))
        return b.value, p.value, l.value

    def last_timing(self):
        ms = C.c_double()
        launches = C.c_int64()
        _lib.lib().locreg_last_timing(self._h, C.byref(ms), C.byref(launches))
        return ms.value, launches.value


class IcpRegistration(_Registration):
    """IcpRegistration(IcpOptions) (icp_registration.hpp:59-82)."""

    def __init__(self, options=None, device=0):
        options = options or IcpOptions()
        if options.method_ == IcpMethod.PCLICP:
            raise _lib.LocregError("PCLICP is a passthrough to pcl::IterativeClosestPoint and is out of scope")
        o = _lib.Options()
        _lib.lib().locreg_default_options(C.byref(o), options.method_)
        o.max_iteration = options.max_iteration_
        o.max_nn_distance = options.max_nn_distance_
        o.max_plane_distance = options.max_plane_distance_
        o.max_line_distance = options.max_line_distance_
        o.min_effective_pts = options.min_effective_pts_
        o.eps = options.eps_
        o.use_ann = int(options.use_ann)
        o.knn_cell_size = options.knn_cell_size
        o.knn_lists = int(options.knn_lists)
        o.loop_mode = options.loop_mode
        # Align* start from target_center_ - source_center_ = 0 when the flag is cleared (icp_registration.cpp:272-276)
        o.zero_initial_translation = 0 if options.use_initial_translation_ else 1
        self.options_ = options
        super().__init__(o, device)


class LoamRegistration:
    """LoamRegistration::ScanMatch (loam_registration.cpp:38-99, SURVEY.md 3.3) over two IcpRegistration handles: a
    P2Plane one for the surf cloud and a P2Line one for the edge cloud, each with its own options and gates.  Every
    Gauss-Newton trip sums the two halves' H and B and takes one step; the whole loop stays on the device
    (locreg_align_loam).  max_iteration and eps belong to the LOAM loop (LoamOption), not to either half."""

    def __init__(self, surf_options=None, edge_options=None, max_iteration=10, eps=1e-2, device=0):
        surf_options = surf_options or IcpOptions(method_=IcpMethod.P2PLANE)
        edge_options = edge_options or IcpOptions(method_=IcpMethod.P2LINE)
        if surf_options.method_ != IcpMethod.P2PLANE or edge_options.method_ != IcpMethod.P2LINE:
            raise _lib.LocregError("LoamRegistration needs P2PLANE options for the surf half and P2LINE options for the edge half")
        self.surf = IcpRegistration(surf_options, device)
        self.edge = IcpRegistration(edge_options, device)
        self.max_iteration = int(max_iteration)
        self.eps = float(eps)
        self.last_result = None

    def SetInputTarget(self, surf_map, edge_map):
        self.surf.SetInputTarget(surf_map)
        self.edge.SetInputTarget(edge_map)
        return True

    def ScanMatch(self, surf_cloud, edge_cloud, predict_pose):
        """Returns (pose, (res_surf, res_edge)): iters / updates / converged are the loop's, the counts and the degenerate
        flag each half's last evaluation."""
        a, n_s, s_s, b, n_e = self._clouds(surf_cloud, edge_cloud)
        pin = _pose(predict_pose)
        pout = pin.copy()
        res = (_lib.Result * 2)()
        _lib.check(_lib.lib().locreg_align_loam(self.surf._h, self.edge._h, a.ctypes.data, n_s, b.ctypes.data, n_e, s_s,
                                                pin.ctypes.data, self.max_iteration, self.eps, pout.ctypes.data, res))
        self.last_result = (res[0].as_dict(), res[1].as_dict())
        return pout, self.last_result

    def ScanMatchBatch(self, surf_clouds, surf_offsets, edge_clouds, edge_offsets, predict_poses):
        """S independent ScanMatch calls in one device-resident loop (locreg_align_loam_batch).  Scan s is
        surf_clouds[surf_offsets[s]:surf_offsets[s + 1]] and edge_clouds[edge_offsets[s]:edge_offsets[s + 1]].
        Returns (poses (S, 7), [(res_surf, res_edge)] * S), each scan's exactly what its ScanMatch call returns."""
        a, _, s_s, b, _ = self._clouds(surf_clouds, edge_clouds)
        so = np.ascontiguousarray(surf_offsets, np.int64)
        eo = np.ascontiguousarray(edge_offsets, np.int64)
        S = so.shape[0] - 1
        if S < 0 or eo.shape != so.shape:
            raise _lib.LocregError("surf_offsets and edge_offsets need S + 1 entries each")
        pin = np.ascontiguousarray(predict_poses, np.float64).reshape(S, 7)
        pout = pin.copy()
        res = (_lib.Result * (2 * S))()
        _lib.check(_lib.lib().locreg_align_loam_batch(self.surf._h, self.edge._h, a.ctypes.data, so.ctypes.data, b.ctypes.data,
                                                      eo.ctypes.data, s_s, pin.ctypes.data, S, self.max_iteration, self.eps,
                                                      pout.ctypes.data, res))
        return pout, [(res[2 * s].as_dict(), res[2 * s + 1].as_dict()) for s in range(S)]

    def Relocalise(self, surf_cloud, edge_cloud, hypotheses, want_all=False):
        """Global relocalisation of one surf / edge scan (locreg_relocalise_loam): every hypothesis runs the ScanMatch
        loop, then both halves are scored once more at its final pose, score = (sum_sq_res_surf + sum_sq_res_edge) /
        (n_inlier_surf + n_inlier_edge), +inf when the summed H is singular or no half has an inlier.  Returns
        (best_pose, best_idx, best_score, scores, poses) as IcpRegistration.Relocalise; scores (n,) and poses (n, 7)
        only with want_all."""
        a, n_s, s_s, b, n_e = self._clouds(surf_cloud, edge_cloud)
        hyp = np.ascontiguousarray(hypotheses, np.float64).reshape(-1, 7)
        nh = hyp.shape[0]
        best_pose = np.zeros(7)
        best_idx = C.c_int64(-1)
        best_score = C.c_double(np.inf)
        scores = np.zeros(nh) if want_all else None
        poses = np.zeros((nh, 7)) if want_all else None
        _lib.check(_lib.lib().locreg_relocalise_loam(self.surf._h, self.edge._h, a.ctypes.data, n_s, b.ctypes.data, n_e, s_s,
                                                     hyp.ctypes.data, nh, self.max_iteration, self.eps, best_pose.ctypes.data,
                                                     C.byref(best_idx), C.byref(best_score),
                                                     scores.ctypes.data if want_all else None,
                                                     poses.ctypes.data if want_all else None))
        return best_pose, int(best_idx.value), float(best_score.value), scores, poses

    def RelocaliseSharded(self, surf_cloud, edge_cloud, hypotheses):
        """Relocalise over the ranks of the surf handle's communicator (CommInit): every rank passes the same clouds and
        hypotheses.  Returns (best_pose, best GLOBAL index, best_score), identical on every rank."""
        a, n_s, s_s, b, n_e = self._clouds(surf_cloud, edge_cloud)
        hyp = np.ascontiguousarray(hypotheses, np.float64).reshape(-1, 7)
        best_pose = np.zeros(7)
        best_idx = C.c_int64(-1)
        best_score = C.c_double(np.inf)
        _lib.check(_lib.lib().locreg_relocalise_loam_sharded(self.surf._h, self.edge._h, a.ctypes.data, n_s, b.ctypes.data, n_e,
                                                             s_s, hyp.ctypes.data, hyp.shape[0], self.max_iteration, self.eps,
                                                             best_pose.ctypes.data, C.byref(best_idx), C.byref(best_score)))
        return best_pose, int(best_idx.value), float(best_score.value)

    def RelocaliseStaged(self, surf_cloud, edge_cloud, hypotheses, trips, keep, want_all=False):
        """Relocalise in len(trips) rounds of trips[r] LOAM trips (eps: self.eps), keeping the keep[r] best-scoring
        hypotheses after round r (locreg_relocalise_loam_staged; self.max_iteration is not used).  Returns (best_pose,
        best_idx, best_score, scores, poses, rounds) as IcpRegistration.RelocaliseStaged."""
        return self._relocalise_staged("locreg_relocalise_loam_staged", surf_cloud, edge_cloud, hypotheses, trips, keep,
                                       want_all)

    def RelocaliseStagedSharded(self, surf_cloud, edge_cloud, hypotheses, trips, keep, want_all=False):
        """RelocaliseStaged over all ranks of the surf handle's communicator (locreg_relocalise_loam_staged_sharded):
        every rank passes the same clouds, hypotheses and schedule.  Returns the same 6-tuple as RelocaliseStaged, bit
        for bit what one GPU returns, on every rank."""
        return self._relocalise_staged("locreg_relocalise_loam_staged_sharded", surf_cloud, edge_cloud, hypotheses, trips,
                                       keep, want_all)

    def _relocalise_staged(self, symbol, surf_cloud, edge_cloud, hypotheses, trips, keep, want_all):
        a, n_s, s_s, b, n_e = self._clouds(surf_cloud, edge_cloud)
        hyp = np.ascontiguousarray(hypotheses, np.float64).reshape(-1, 7)
        nh = hyp.shape[0]
        trips, keep = _schedule(trips, keep)
        best_pose = np.zeros(7)
        best_idx = C.c_int64(-1)
        best_score = C.c_double(np.inf)
        scores = np.zeros(nh) if want_all else None
        poses = np.zeros((nh, 7)) if want_all else None
        rounds = np.zeros(nh, np.int32) if want_all else None
        _lib.check(getattr(_lib.lib(), symbol)(self.surf._h, self.edge._h, a.ctypes.data, n_s, b.ctypes.data, n_e, s_s,
                      hyp.ctypes.data, nh, trips.ctypes.data, keep.ctypes.data if keep.size else None, trips.shape[0],
                      self.eps, best_pose.ctypes.data, C.byref(best_idx), C.byref(best_score),
                      scores.ctypes.data if want_all else None,
                      poses.ctypes.data if want_all else None,
                      rounds.ctypes.data if want_all else None))
        return best_pose, int(best_idx.value), float(best_score.value), scores, poses, rounds

    # the communicator of the sharded relocalisation is the surf handle's (loc_lib_b200.dist.comm_init works unchanged)
    CommUniqueId = staticmethod(_Registration.CommUniqueId)

    def CommInit(self, unique_id, rank, world):
        self.surf.CommInit(unique_id, rank, world)

    def CommInfo(self):
        return self.surf.CommInfo()

    def CommDestroy(self):
        self.surf.CommDestroy()

    @staticmethod
    def _clouds(surf_cloud, edge_cloud):
        a, n_s, s_s = _cloud(surf_cloud)
        b, n_e, s_e = _cloud(edge_cloud)
        if s_e != s_s:  # the C ABI takes one stride for both clouds
            b = np.ascontiguousarray(np.pad(b[:, :3], ((0, 0), (0, s_s // 4 - 3))), np.float32)
        return a, n_s, s_s, b, n_e

    def last_timing(self):
        return self.surf.last_timing()

    def close(self):
        self.surf.close()
        self.edge.close()


class NdtRegistration(_Registration):
    """NdtRegistration(NdtOptions) (ndt_registration.cpp:20-28): DIRECT_NDT, or INCREMENTAL_NDT where every
    SetInputTarget ADDS its cloud to an LRU cache of capacity_ voxels (ndt_registration.cpp:150-183)."""

    def __init__(self, options=None, device=0):
        options = options or NdtOptions()
        if options.method_ == NdtMethod.PCL_NDT:
            raise _lib.LocregError("PCL_NDT is an unimplemented stub in the reference (ndt_registration.cpp:69-70)")
        o = _lib.Options()
        _lib.lib().locreg_default_options(C.byref(o), NDT_INCREMENTAL if options.method_ == NdtMethod.INCREMENTAL_NDT else NDT_DIRECT)
        o.ndt_capacity = int(options.capacity_)
        o.max_iteration = options.max_iteration_
        o.voxel_size = options.voxel_size_
        o.min_effective_pts = options.min_effective_pts_
        o.min_pts_in_voxel = options.min_pts_in_voxel_
        o.eps = options.eps_
        o.res_outlier_th = options.res_outlier_th_
        o.nearby_type = options.nearby_type_
        o.loop_mode = options.loop_mode
        o.zero_initial_translation = 1 if options.remove_centroid_ else 0  # ndt_registration.cpp:380-384 (AlignNdt only)
        self.options_ = options
        super().__init__(o, device)

    def Voxels(self):
        nv = C.c_size_t()
        _lib.check(_lib.lib().locreg_ndt_num_voxels(self._h, C.byref(nv)))
        nv = nv.value
        keys = np.zeros((nv, 3), np.int32)
        mu = np.zeros((nv, 3))
        info = np.zeros((nv, 3, 3))
        npts = np.zeros(nv, np.int32)
        _lib.check(_lib.lib().locreg_ndt_get_voxels(self._h, keys.ctypes.data, mu.ctypes.data, info.ctypes.data,
                                                    npts.ctypes.data))
        return keys, mu, info, npts


# ---- the slice of Loc (LocUtils/src/slam/3d/loc.cpp) that decides what the registration is called with ----------------
def _q_mul(a, b):
    ax, ay, az, aw = a
    bx, by, bz, bw = b
    return np.array([aw * bx + ax * bw + ay * bz - az * by, aw * by - ax * bz + ay * bw + az * bx,
                     aw * bz + ax * by - ay * bx + az * bw, aw * bw - ax * bx - ay * by - az * bz])


def _q_rot(q, v):
    x, y, z, w = q
    u = np.array([x, y, z])
    t = 2.0 * np.cross(u, v)
    return v + w * t + np.cross(u, t)


def se3_mul(a, b):
    """Sophus SE3d product of two [qx qy qz qw tx ty tz] poses."""
    q = _q_mul(a[:4], b[:4])
    return np.concatenate([q / np.linalg.norm(q), a[4:] + _q_rot(a[:4], b[4:])])


def se3_inv(a):
    qi = np.array([-a[0], -a[1], -a[2], a[3]])
    return np.concatenate([qi, -_q_rot(qi, a[4:])])


def se3_log_angle(a):
    """|log(R)| of a pose's rotation, radians."""
    q = np.asarray(a[:4], np.float64)
    return 2.0 * np.arctan2(np.linalg.norm(q[:3]), abs(q[3]))


class LioTracker:
    """Lio::AddCloud / AlignWithLocalMap without the ROS / ESKF / file parts (lio.cpp:238-307, 445-470, 616-623): the
    first scan becomes the local map at the initial pose; every later scan is matched against the local map from the
    constant-velocity prediction predict = result * last^-1 * result (starting from identity, like the function's
    statics), and becomes a key frame - transformed, pushed into the sliding window of `num_kfs_in_local_map` scans,
    local map re-filtered and re-indexed, all on the device - when it moved more than kf_distance metres or
    kf_angle_deg degrees from the last key frame."""

    def __init__(self, registration, init_pose=None, num_kfs_in_local_map=10, kf_distance=1.0, kf_angle_deg=10.0,
                 local_map_leaf=0.5):
        self.reg = registration
        self.max_kfs, self.kf_distance, self.kf_angle = num_kfs_in_local_map, kf_distance, np.deg2rad(kf_angle_deg)
        self.leaf = local_map_leaf
        ident = np.array([0, 0, 0, 1, 0, 0, 0], np.float64)
        self.last_kf_pose = ident.copy() if init_pose is None else np.asarray(init_pose, np.float64).copy()
        self.last_pose, self.predict = ident.copy(), ident.copy()
        self.keyframes = 0
        self.n_local = 0
        self.reg.ClearLocalMap()

    def IsKeyframe(self, pose):
        delta = se3_mul(se3_inv(self.last_kf_pose), pose)
        return np.linalg.norm(delta[4:]) > self.kf_distance or se3_log_angle(delta) > self.kf_angle

    def AddCloud(self, scan, filtered_scan=None):
        """scan: the raw scan (what a key frame stores, lio.cpp:279); filtered_scan: cur_scan_filter_ptr_'s output (what
        is matched, and what the FIRST key frame stores, :236,:244); defaults to scan.  Returns (pose, is_keyframe)."""
        src = scan if filtered_scan is None else filtered_scan
        if self.keyframes == 0:
            self.n_local = self.reg.AddKeyFrame(src, self.last_kf_pose, self.max_kfs, self.leaf)
            self.keyframes = 1
            return self.last_kf_pose.copy(), True
        _, _, result = self.reg.ScanMatch(self.reg.RemoveNanPoint(src), self.predict, want_cloud=False)
        self.predict = se3_mul(se3_mul(result, se3_inv(self.last_pose)), result)
        self.last_pose = result
        if not self.IsKeyframe(result):
            return result, False
        self.last_kf_pose = result.copy()
        self.n_local = self.reg.AddKeyFrame(scan, result, self.max_kfs, self.leaf)
        self.keyframes += 1
        return result, True


class LocTracker:
    """Loc::Update without the ROS / ESKF parts (loc.cpp:208-246): ScanMatch from the constant-velocity prediction
    predict = result * last^-1 * result (:232), and a new 150 m local map (ResetLocalMap, on the device) whenever the
    pose comes within 50 m of the box edge on any axis (:235-246)."""

    def __init__(self, registration, global_map, init_pose, half_size=(150.0, 150.0, 150.0), margin=50.0):
        self.reg, self.half, self.margin = registration, np.asarray(half_size, np.float32), margin
        self.reg.SetGlobalMap(global_map)
        self.last_pose = np.asarray(init_pose, np.float64).copy()
        self.predict = self.last_pose.copy()
        self.resets = 0
        self._reset(self.last_pose[4:])

    def _reset(self, t):
        self.origin = np.asarray(t, np.float32)
        self.n_local = self.reg.ResetLocalMap(*self.origin, half_size=self.half)
        self.edge = np.stack([-self.half + self.origin, self.half + self.origin], 1)  # per axis [lo, hi]
        self.resets += 1

    def Update(self, scan):
        _, cloud, result = self.reg.ScanMatch(scan, self.predict)
        self.predict = se3_mul(se3_mul(result, se3_inv(self.last_pose)), result)
        self.last_pose = result
        t = result[4:]
        for i in range(3):
            if abs(t[i] - self.edge[i, 0]) > self.margin and abs(t[i] - self.edge[i, 1]) > self.margin:
                continue
            self._reset(t)
            break
        return result, cloud
