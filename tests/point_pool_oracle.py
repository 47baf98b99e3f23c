"""The tracker's point pool restated on the CPU (tests/point_pool_oracle.c) around the oracle's unchanged sequence step.

The C file is compiled with the oracle's sources and flags (oracle/Makefile: -std=c99 -O2 -ffp-contract=off) into a
temporary directory, so the checked tree is never written to."""
import atexit
import ctypes as C
import functools
import os
import shutil
import subprocess
import tempfile
import types

import numpy as np

from oracle.pyoracle import OracleSeq, StepStats, _p, c_dp, c_ip, c_u8p

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE = os.path.join(os.path.dirname(HERE), "oracle")


@functools.lru_cache(maxsize=None)
def library():
    out = tempfile.mkdtemp(prefix="svo_point_pool_")
    atexit.register(shutil.rmtree, out, True)
    so = os.path.join(out, "libsvo_point_pool.so")
    subprocess.check_call([os.environ.get("CC", "gcc"), "-std=c99", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-o", so,
                           os.path.join(HERE, "point_pool_oracle.c"), os.path.join(ORACLE, "svo_oracle.c"),
                           os.path.join(ORACLE, "svo_oracle_map.c"), "-lm", "-lpthread"])
    L = C.CDLL(so)
    V = C.c_void_p
    L.pp_attach.restype = V
    L.pp_attach.argtypes = [V, C.c_int]
    L.pp_destroy.argtypes = [V]
    L.pp_step.argtypes = [V, c_u8p, c_dp, c_dp, C.POINTER(StepStats), c_dp, c_ip]
    L.pp_add_keyframe.argtypes = [V, C.c_float, C.c_float]
    L.pp_get_points.argtypes = [V, V, c_dp, c_ip, c_ip, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    return L


class PoolSeq(OracleSeq):
    """OracleSeq with an optional point pool of `capacity` slots (None: the oracle's sequence exactly as it is)."""

    def __init__(self, cam, n_levels, max_level, min_level, n_pyr_levels_cfg, conv_thresh, depth_mean, depth_min, reseed, capacity=None):
        super().__init__(types.SimpleNamespace(lib=library()), cam, n_levels, max_level, min_level, n_pyr_levels_cfg, conv_thresh,
                         depth_mean, depth_min, reseed)
        self.capacity, self.pool = capacity, None

    def set_keyframe(self, img, T_kf_w, kf_px, kf_level, pt_world, seed_px, seed_level):
        n = len(kf_level)
        P = n if self.capacity is None else max(n, self.capacity)
        pad = lambda a, shape, t: np.concatenate([np.asarray(a, t).reshape((n,) + shape), np.zeros((P - n,) + shape, t)])
        super().set_keyframe(img, T_kf_w, pad(kf_px, (2,), np.float64), pad(kf_level, (), np.int32), pad(pt_world, (3,), np.float64),
                             seed_px, seed_level)
        if self.capacity is not None:
            self.pool = C.c_void_p(self.lib.pp_attach(self.h, n))
            L, pool = self.lib, self.pool
            self._step = lambda h, *a: L.pp_step(pool, *a)

    def add_keyframe(self, depth_mean, depth_min):
        if self.pool is None:
            return super().add_keyframe(depth_mean, depth_min)
        n = int(self.lib.pp_add_keyframe(self.pool, float(depth_mean), float(depth_min)))
        self.S = self.num_slots()
        return n

    def points(self):
        """(pos[P,3], type[P], n_obs[P], created, dropped) of the point slots; type SVO_POINT_*"""
        P = self.N
        pos = np.zeros((max(P, 1), 3)); ty = np.zeros(max(P, 1), np.int32); no = np.zeros(max(P, 1), np.int32)
        cr, dr = C.c_int(0), C.c_int(0)
        self.lib.pp_get_points(self.h, self.pool, _p(pos, c_dp), _p(ty, c_ip), _p(no, c_ip), C.byref(cr), C.byref(dr))
        return pos[:P], ty[:P], no[:P], cr.value, dr.value

    def close(self):
        if self.pool is not None:
            self.lib.pp_destroy(self.pool)
            self.pool = None
        super().close()

