"""ORACLE — TEST INFRASTRUCTURE ONLY.

ctypes front-end of oracle/pointops_ref.c (the CPU restatement of the reference's CUDA point
operators).  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs may import this; sceneverse_b200/ never does.

`RefExt` exposes the nine function names of the reference's pybind module
(/root/reference/modules/third_party/pointnet2/_ext_src/src/bindings.cpp:6-19) on CPU torch
tensors, so that the unmodified reference Python layers can run on CPU with
`pointnet2_utils._ext = RefExt()` (SURVEY.md §8c).
"""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "pointops_ref.c")
_OUT = os.path.join(_HERE, "_build", "libsvref.so")
_lib = None


def build(force=False):
    """gcc -O2 -ffp-contract=off -fopenmp; returns the .so path.  It goes to oracle/_build, or to a fresh temporary
    directory when that cannot be written (a read-only checkout)."""
    global _OUT
    if force or not os.path.exists(_OUT) or os.path.getmtime(_OUT) < os.path.getmtime(_SRC):
        try:
            os.makedirs(os.path.dirname(_OUT), exist_ok=True)
        except OSError:
            pass
        if not os.access(os.path.dirname(_OUT), os.W_OK):
            _OUT = os.path.join(tempfile.mkdtemp(prefix="svref-"), "libsvref.so")
        tmp = _OUT + ".%d.tmp" % os.getpid()
        subprocess.check_call(
            ["gcc", "-O2", "-ffp-contract=off", "-fopenmp", "-shared", "-fPIC", "-o", tmp, _SRC, "-lm"])
        os.replace(tmp, _OUT)
    return _OUT


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
        _lib.svref_opt_n_threads.restype = ctypes.c_int
    return _lib


def _f(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    return a, a.ctypes.data_as(ctypes.c_void_p)


def _i(a):
    a = np.ascontiguousarray(a, dtype=np.int32)
    return a, a.ctypes.data_as(ctypes.c_void_p)


def opt_n_threads(n):
    return int(lib().svref_opt_n_threads(ctypes.c_int(int(n))))


# ---------------------------------------------------------------- numpy API
def furthest_point_sampling(xyz, m):
    xyz, p = _f(xyz)
    B, N, _ = xyz.shape
    out = np.zeros((B, m), np.int32)
    lib().svref_furthest_point_sampling(p, B, N, int(m), out.ctypes.data_as(ctypes.c_void_p))
    return out


def gather_points(points, idx):
    points, pp = _f(points)
    idx, ip = _i(idx)
    B, C, N = points.shape
    M = idx.shape[1]
    out = np.zeros((B, C, M), np.float32)
    lib().svref_gather_points(pp, ip, B, C, N, M, out.ctypes.data_as(ctypes.c_void_p))
    return out


def gather_points_grad(grad_out, idx, n):
    grad_out, gp = _f(grad_out)
    idx, ip = _i(idx)
    B, C, M = grad_out.shape
    out = np.zeros((B, C, n), np.float32)
    lib().svref_gather_points_grad(gp, ip, B, C, int(n), M, out.ctypes.data_as(ctypes.c_void_p))
    return out


def ball_query(new_xyz, xyz, radius, nsample):
    new_xyz, qp = _f(new_xyz)
    xyz, pp = _f(xyz)
    B, M, _ = new_xyz.shape
    N = xyz.shape[1]
    out = np.zeros((B, M, nsample), np.int32)
    lib().svref_ball_query(qp, pp, B, N, M, ctypes.c_float(radius), int(nsample),
                           out.ctypes.data_as(ctypes.c_void_p))
    return out


def group_points(points, idx):
    points, pp = _f(points)
    idx, ip = _i(idx)
    B, C, N = points.shape
    _, NP, NS = idx.shape
    out = np.zeros((B, C, NP, NS), np.float32)
    lib().svref_group_points(pp, ip, B, C, N, NP, NS, out.ctypes.data_as(ctypes.c_void_p))
    return out


def group_points_grad(grad_out, idx, n):
    grad_out, gp = _f(grad_out)
    idx, ip = _i(idx)
    B, C, NP, NS = grad_out.shape
    out = np.zeros((B, C, n), np.float32)
    lib().svref_group_points_grad(gp, ip, B, C, int(n), NP, NS, out.ctypes.data_as(ctypes.c_void_p))
    return out


def three_nn(unknown, known):
    unknown, up = _f(unknown)
    known, kp = _f(known)
    B, n, _ = unknown.shape
    m = known.shape[1]
    d = np.zeros((B, n, 3), np.float32)
    i = np.zeros((B, n, 3), np.int32)
    with np.errstate(over="ignore"):
        lib().svref_three_nn(up, kp, B, n, m, d.ctypes.data_as(ctypes.c_void_p),
                             i.ctypes.data_as(ctypes.c_void_p))
    return d, i


def three_interpolate(points, idx, weight):
    points, pp = _f(points)
    idx, ip = _i(idx)
    weight, wp = _f(weight)
    B, c, m = points.shape
    n = idx.shape[1]
    out = np.zeros((B, c, n), np.float32)
    lib().svref_three_interpolate(pp, ip, wp, B, c, m, n, out.ctypes.data_as(ctypes.c_void_p))
    return out


def three_interpolate_grad(grad_out, idx, weight, m):
    grad_out, gp = _f(grad_out)
    idx, ip = _i(idx)
    weight, wp = _f(weight)
    B, c, n = grad_out.shape
    out = np.zeros((B, c, m), np.float32)
    lib().svref_three_interpolate_grad(gp, ip, wp, B, c, n, int(m), out.ctypes.data_as(ctypes.c_void_p))
    return out


# ---------------------------------------------------------------- torch `_ext` look-alike
class RefExt:
    """CPU stand-in for `pointnet2._ext` (bindings.cpp:6-19) backed by the C restatement."""

    @staticmethod
    def _t(a):
        import torch
        return torch.from_numpy(a)

    def furthest_point_sampling(self, points, nsamples):
        return self._t(furthest_point_sampling(points.detach().cpu().numpy(), nsamples))

    def gather_points(self, points, idx):
        return self._t(gather_points(points.detach().cpu().numpy(), idx.cpu().numpy()))

    def gather_points_grad(self, grad_out, idx, n):
        return self._t(gather_points_grad(grad_out.detach().cpu().numpy(), idx.cpu().numpy(), n))

    def ball_query(self, new_xyz, xyz, radius, nsample):
        return self._t(ball_query(new_xyz.detach().cpu().numpy(), xyz.detach().cpu().numpy(), radius, nsample))

    def group_points(self, points, idx):
        return self._t(group_points(points.detach().cpu().numpy(), idx.cpu().numpy()))

    def group_points_grad(self, grad_out, idx, n):
        return self._t(group_points_grad(grad_out.detach().cpu().numpy(), idx.cpu().numpy(), n))

    def three_nn(self, unknowns, knows):
        d, i = three_nn(unknowns.detach().cpu().numpy(), knows.detach().cpu().numpy())
        return [self._t(d), self._t(i)]

    def three_interpolate(self, points, idx, weight):
        return self._t(three_interpolate(points.detach().cpu().numpy(), idx.cpu().numpy(), weight.detach().cpu().numpy()))

    def three_interpolate_grad(self, grad_out, idx, weight, m):
        return self._t(three_interpolate_grad(grad_out.detach().cpu().numpy(), idx.cpu().numpy(),
                                              weight.detach().cpu().numpy(), m))
