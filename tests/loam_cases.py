"""Shared pieces of the LOAM tests (TEST INFRASTRUCTURE): the LOAM loop over the CPU oracle (tests/loam/oracle_loam.cpp),
the host loop LoamRegistration runs today over two CaculateMatrixHAndB handles, and a scene neither half solves alone."""
import ctypes as C
import os

import numpy as np

import oracle_py as O

_SO = os.path.join(os.path.dirname(os.path.abspath(__file__)), "loam", "_build", "liboracle_loam.so")
_LIB = None


def _lib():
    global _LIB
    if _LIB is None:
        O.lib()  # liboracle.so first: liboracle_loam.so links against it
        L = C.CDLL(_SO)
        vp, sz = C.c_void_p, C.c_size_t
        L.oracle_loam_align.argtypes = [vp, vp, vp, sz, vp, sz, sz, vp, C.c_int32, C.c_double, vp, vp]
        _LIB = L
    return _LIB


def xyz(cloud):
    return np.ascontiguousarray(np.asarray(cloud, np.float32)[:, :3])


def oracle_loam_align(surf, edge, surf_cloud, edge_cloud, pose, max_iteration, eps):
    """surf / edge: OracleIcp (P2Plane / P2Line).  Returns (pose, (res_surf, res_edge)) as locreg_align_loam does."""
    a, b = xyz(surf_cloud), xyz(edge_cloud)
    pin = np.ascontiguousarray(pose, np.float64)
    pout = np.zeros(7)
    res = (O.Result * 2)()
    _lib().oracle_loam_align(surf._h, edge._h, a.ctypes.data, a.shape[0], b.ctypes.data, b.shape[0], 12, pin.ctypes.data,
                             int(max_iteration), float(eps), pout.ctypes.data, res)
    return pout, (res[0].as_dict(), res[1].as_dict())


def quat_mul(a, b):
    ax, ay, az, aw = a
    bx, by, bz, bw = b
    return np.array([aw * bx + ax * bw + ay * bz - az * by, aw * by + ay * bw + az * bx - ax * bz,
                     aw * bz + az * bw + ax * by - ay * bx, aw * bw - ax * bx - ay * by - az * bz])


def pose_update(pose, dx):
    """R <- R * Exp(dx[0:3]) (Sophus SO3::exp, unit quaternion), t <- t + dx[3:6]."""
    w = np.asarray(dx[:3], float)
    th = float(np.linalg.norm(w))
    if th < 1e-10:
        imag, real = 0.5 - th * th / 48.0, 1.0 - th * th / 8.0
    else:
        imag, real = np.sin(0.5 * th) / th, np.cos(0.5 * th)
    q = quat_mul(pose[:4], np.array([imag * w[0], imag * w[1], imag * w[2], real]))
    out = np.array(pose, float)
    out[:4] = q / np.linalg.norm(q)
    out[4:] += dx[3:]
    return out


def host_loop(surf, edge, surf_cloud, edge_cloud, pose, max_iteration, eps, timings=None):
    """What LoamRegistration::ScanMatch does today over two IcpRegistration handles (one CaculateMatrixHAndB per half
    per trip, the sum solved on the host).  Returns (pose, {'iters', 'updates', 'converged'}); timings (a list, optional)
    receives each call's last_timing()."""
    pose = np.array(pose, float)
    r = {"iters": 0, "updates": 0, "converged": 0}
    for it in range(max_iteration):
        _, Hs, Bs = surf.CaculateMatrixHAndB(surf_cloud, pose)
        if timings is not None:
            timings.append(surf.last_timing())
        _, He, Be = edge.CaculateMatrixHAndB(edge_cloud, pose)
        if timings is not None:
            timings.append(edge.last_timing())
        H, B = Hs + He, Bs + Be
        r["iters"] = it + 1
        if np.linalg.det(H) == 0:
            continue
        dx = np.linalg.solve(H, B)
        pose = pose_update(pose, dx)
        r["updates"] += 1
        if np.linalg.norm(dx) < eps:
            r["converged"] = 1
            break
    return pose, r


def pose_from_rpy_t(rpy, t):
    q = np.array([0.0, 0.0, 0.0, 1.0])
    for axis, ang in zip(range(3), rpy):
        e = np.zeros(4)
        e[axis] = np.sin(0.5 * ang)
        e[3] = np.cos(0.5 * ang)
        q = quat_mul(q, e)
    return np.concatenate([q, t])


def transform(pose, pts):
    x, y, z, w = pose[:4]
    R = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                  [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                  [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])
    return (np.asarray(pts, float) @ R.T + pose[4:]).astype(np.float32)


def inverse(pose):
    qi = np.array([-pose[0], -pose[1], -pose[2], pose[3]])
    t = transform(np.concatenate([qi, [0, 0, 0]]), pose[4:][None])[0].astype(float)
    return np.concatenate([qi, -t])


class KatScene:
    """Surf map: the plane z = 0 (constrains tz, roll, pitch).  Edge map: two vertical poles at different (x, y)
    (constrain tx, ty, yaw, roll, pitch, but never tz).  Sources: the maps seen from the pose `truth`."""

    def __init__(self):
        g = np.arange(-40, 41) * 0.1
        gx, gy = np.meshgrid(g, g, indexing="ij")
        self.surf_map = np.stack([gx.ravel(), gy.ravel(), np.zeros(gx.size)], 1).astype(np.float32)
        z = np.arange(0, 151) * 0.02
        self.edge_map = np.concatenate([np.stack([np.full_like(z, 1.5), np.full_like(z, 0.5), z], 1),
                                        np.stack([np.full_like(z, -1.0), np.full_like(z, -2.0), z], 1)]).astype(np.float32)
        self.truth = pose_from_rpy_t([0.01, -0.015, 0.02], [0.05, -0.03, 0.04])
        inv = inverse(self.truth)
        inner = np.all(np.abs(self.surf_map[:, :2]) < 3.5, axis=1)  # away from the plane's border
        self.surf = transform(inv, self.surf_map[inner][::3])
        tall = (self.edge_map[:, 2] > 0.2) & (self.edge_map[:, 2] < 2.8)  # away from the poles' ends
        self.edge = transform(inv, self.edge_map[tall][::2])
        self.init = np.array([0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0])


def rot_diff(a, b):
    """Rotation angle [rad] between two 7-double poses, accurate for tiny angles (unlike an arccos of a dot product)."""
    qa = np.array([-a[0], -a[1], -a[2], a[3]], float)
    d = quat_mul(qa, np.asarray(b[:4], float))
    return 2.0 * float(np.arcsin(min(1.0, np.linalg.norm(d[:3]))))
