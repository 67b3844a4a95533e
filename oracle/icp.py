"""CPU oracle bindings for K6, point-to-point ICP loop verification (TEST INFRASTRUCTURE): ctypes over ``orc_icp_align``
of ``oracle/ilsm_oracle_icp.cpp``, built into ``oracle/_build/libilsm_oracle.so`` with the rest of the oracle."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _f32, _p, _stride, lib


class IcpOpts(C.Structure):
    """= ilsm_icp_opts; the defaults are PCL 1.10's."""
    _fields_ = [("max_correspondence_distance", C.c_double), ("max_iterations", C.c_int32), ("pad", C.c_int32),
                ("transformation_epsilon", C.c_double), ("transformation_rotation_epsilon", C.c_double),
                ("euclidean_fitness_epsilon", C.c_double), ("fitness_max_range", C.c_double)]

    def __init__(self, **kw):
        fmax = np.finfo(np.float64).max
        super().__init__(max_correspondence_distance=float(np.sqrt(fmax)), max_iterations=10, transformation_epsilon=0.0,
                         transformation_rotation_epsilon=0.0, euclidean_fitness_epsilon=-fmax, fitness_max_range=fmax)
        for k, v in kw.items():
            setattr(self, k, v)


class IcpResult(C.Structure):
    """= ilsm_icp_result"""
    _fields_ = [("q_xyzw", C.c_double * 4), ("t", C.c_double * 3), ("fitness", C.c_double), ("mse", C.c_double),
                ("iterations", C.c_int32), ("state", C.c_int32), ("converged", C.c_int32), ("n_correspondences", C.c_int32)]

    @property
    def q(self):
        return np.array(self.q_xyzw[:], np.float64)

    @property
    def tv(self):
        return np.array(self.t[:], np.float64)


def icp_align(target, source, q=(0.0, 0.0, 0.0, 1.0), t=(0.0, 0.0, 0.0), **opts):
    """pcl::IterativeClosestPoint<PointXYZI, PointXYZI>::align(out, guess) + getFitnessScore() restated (see the header of
    ilsm_oracle_icp.cpp), single-threaded.  opts: IcpOpts fields.  Returns IcpResult."""
    tg, sr = _f32(target), _f32(source)
    g = np.ascontiguousarray(np.concatenate([np.asarray(q, np.float64), np.asarray(t, np.float64)]))
    o = IcpOpts(**opts)
    r = IcpResult()
    lib().orc_icp_align(_p(tg), len(tg), _stride(tg), _p(sr), len(sr), _stride(sr), _p(g), C.byref(o), C.byref(r))
    return r
