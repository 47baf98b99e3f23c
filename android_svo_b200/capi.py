"""ctypes bindings of libsvob200.so (include/svob200.h) — the thin Python layer tests and bench.py
drive the CUDA path through.  There is no fallback of any kind: if the shared library is missing
or no CUDA device is usable, importing / creating a context raises.
"""
import ctypes as C
import os
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# SVOB200_LIB: alternative build of the same library (A/B experiments); default is the in-tree build
LIB_PATH = os.environ.get("SVOB200_LIB") or os.path.join(HERE, "lib", "libsvob200.so")
MAX_LEVELS = 8
MEM_HOST, MEM_DEVICE = 0, 1
ROUND_TRUNC, ROUND_SSE2 = 0, 1
SEED_BEHIND, SEED_NOT_IN_FRAME, SEED_NO_MATCH, SEED_UPDATED, SEED_CONVERGED, SEED_NAN_ERASED, SEED_TOO_OLD = 1, 2, 3, 4, 5, 6, 7

c_u8p = C.POINTER(C.c_uint8)
c_dp = C.POINTER(C.c_double)
c_fp = C.POINTER(C.c_float)
c_ip = C.POINTER(C.c_int)


class Camera(C.Structure):
    _fields_ = [("width", C.c_int), ("height", C.c_int), ("fx", C.c_double), ("fy", C.c_double),
                ("cx", C.c_double), ("cy", C.c_double)]

    @staticmethod
    def make(w, h, fx, fy, cx, cy):
        return Camera(int(w), int(h), float(fx), float(fy), float(cx), float(cy))


class AlignOpts(C.Structure):
    _fields_ = [("max_level", C.c_int), ("min_level", C.c_int), ("n_iter", C.c_int), ("eps", C.c_double)]


class MatcherOpts(C.Structure):
    _fields_ = [("align_1d", C.c_int), ("align_max_iter", C.c_int), ("max_epi_search_steps", C.c_int),
                ("subpix_refinement", C.c_int), ("epi_search_edgelet_filtering", C.c_int),
                ("epi_search_edgelet_max_angle", C.c_double), ("max_search_level", C.c_int)]


# numpy dtypes with C layout (align=True reproduces the struct padding)
corner_dt = np.dtype([("x", "i4"), ("y", "i4"), ("level", "i4"), ("score", "f4")], align=True)
align_result_dt = np.dtype([("T_cur_ref", "f8", 7), ("H", "f8", 36), ("Jres", "f8", 6), ("x", "f8", 6), ("chi2", "f8"),
                            ("n_meas", "i4"), ("iters", "i4", MAX_LEVELS), ("stop", "i4"), ("n_exact_chi2", "i4"), ("n_factorisations", "i4")], align=True)
feature_ref_dt = np.dtype([("ref_frame_id", "i8"), ("ref_image", "i4"), ("cur_image", "i4"), ("level", "i4"), ("type", "i4"),
                           ("px", "f8", 2), ("f", "f8", 3), ("grad", "f8", 2), ("T_cur_ref", "f8", 7)], align=True)
match_result_dt = np.dtype([("success", "i4"), ("search_level", "i4"), ("px_cur", "f8", 2), ("A_cur_ref", "f8", 4),
                            ("h_inv", "f8"), ("patch_with_border", "u1", 100), ("patch", "u1", 64)], align=True)
epi_result_dt = np.dtype([("success", "i4"), ("search_level", "i4"), ("reject", "i4"), ("zmssd_best", "i4"), ("n_evals", "i4"),
                          ("n_steps", "i4"), ("depth", "f8"), ("px_cur", "f8", 2), ("epi_length", "f8"), ("A_cur_ref", "f8", 4),
                          ("h_inv", "f8"), ("epi_dir", "f8", 2), ("px_cur_valid", "i4"), ("patch_with_border", "u1", 100),
                          ("patch", "u1", 64)], align=True)
seed_dt = np.dtype([("a", "f4"), ("b", "f4"), ("mu", "f4"), ("z_range", "f4"), ("sigma2", "f4")], align=True)
step_stats_dt = np.dtype([("T_cur_w", "f8", 7), ("chi2", "f8"), ("n_tracked", "i4"), ("n_matched", "i4"), ("n_seeds_updated", "i4"),
                          ("n_seeds_converged", "i4"), ("n_seeds_failed", "i4"), ("n_seeds_skipped", "i4"), ("align_iters", "i4"),
                          ("n_exact_chi2", "i4"), ("n_reproj_trials", "i4"), ("n_pose_obs", "i4")], align=True)
seed_obs_dt = np.dtype([("status", "i4"), ("search_level", "i4"), ("zmssd_best", "i4"), ("n_evals", "i4"), ("z", "f8"),
                        ("px_cur", "f8", 2), ("epi_length", "f8")], align=True)

map_point_dt = np.dtype([("pos", "f8", 3), ("type", "i4"), ("obs_begin", "i4"), ("obs_end", "i4"), ("reserved", "i4")], align=True)
reproj_result_dt = np.dtype([("status", "i4"), ("cell", "i4"), ("obs", "i4"), ("search_level", "i4"), ("px", "f8", 2),
                             ("A_cur_ref", "f8", 4)], align=True)
reproj_stats_dt = np.dtype([("n_matches", "i4"), ("n_trials", "i4"), ("n_in_frame", "i4"), ("n_cells", "i4")], align=True)
pose_opt_result_dt = np.dtype([("A", "f8", 36), ("chi2", "f8"), ("estimated_scale", "f8"), ("error_init", "f8"), ("error_final", "f8"),
                               ("iters", "i4"), ("num_obs", "i4"), ("rolled_back", "i4"), ("reserved", "i4")], align=True)
POINT_DELETED, POINT_CANDIDATE, POINT_UNKNOWN, POINT_GOOD = 0, 1, 2, 3
REPROJ_NOT_IN_FRAME, REPROJ_UNTRIED, REPROJ_DELETED, REPROJ_FAILED, REPROJ_MATCHED = 0, 1, 2, 3, 4


class PoseOptOpts(C.Structure):
    _fields_ = [("reproj_thresh", C.c_double), ("n_iter", C.c_int), ("eps", C.c_double), ("tukey_b", C.c_float)]


_lib = None


def load_library():
    """Load libsvob200.so; raise loudly if it is not there (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("libsvob200.so is missing (%s): run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "or android_svo_b200/build.sh — there is no CPU fallback" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    L.svob200_last_error.restype = C.c_char_p
    L.svob200_ctx_stream.restype = C.c_void_p
    L.svob200_ctx_launch_count.restype = C.c_longlong
    L.svob200_tracker_device_bytes.restype = C.c_longlong
    V = C.c_void_p
    L.svob200_ctx_create.argtypes = [C.c_int, C.POINTER(V)]
    for name in ("svob200_ctx_destroy", "svob200_ctx_sync", "svob200_ctx_timer_start"):
        getattr(L, name).argtypes = [V]
    L.svob200_last_error.argtypes = [V]
    L.svob200_ctx_stream.argtypes = [V]
    L.svob200_ctx_launch_count.argtypes = [V]
    L.svob200_ctx_timer_stop_ms.argtypes = [V, c_fp]
    L.svob200_frame_create.argtypes = [V, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int]
    L.svob200_frame_upload.argtypes = [V, C.c_int64, V, C.c_int, c_ip, C.c_int]
    L.svob200_frame_bind.argtypes = [V, C.c_int64, V, C.c_int, c_ip]
    L.svob200_frame_slot.argtypes = [V, C.c_int64]
    L.svob200_frame_download.argtypes = [V, C.c_int64, C.c_int, C.c_int, V, C.c_int]
    L.svob200_frame_release.argtypes = [V, C.c_int64]
    L.svob200_frame_info.argtypes = [V, C.c_int64, c_ip, c_ip, c_ip, c_ip]
    L.svob200_half_sample.argtypes = [V, V, C.c_int, C.c_int, C.c_int, V, C.c_int, C.c_int]
    L.svob200_fast_detect.argtypes = [V, C.c_int64, C.c_int, C.c_int, C.c_double, V, V, V, C.c_int]
    L.svob200_fast_corners.argtypes = [V, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, V, V, V]
    L.svob200_sparse_align.argtypes = [V, C.c_int64, C.c_int64, C.POINTER(Camera), C.c_int, V, V, V, V, V, C.POINTER(AlignOpts), V, C.c_int]
    L.svob200_align_patches.argtypes = [V, C.c_int64, C.c_int, C.c_int, V, V, V, V, C.c_int, V, V, V, C.c_int]
    L.svob200_matcher_opts_default.argtypes = [C.POINTER(MatcherOpts), C.c_int]
    L.svob200_match_direct.argtypes = [V, C.c_int64, C.POINTER(Camera), C.c_int, V, V, V, C.POINTER(MatcherOpts), V, C.c_int]
    L.svob200_epipolar_match.argtypes = [V, C.c_int64, C.POINTER(Camera), C.c_int, V, V, C.POINTER(MatcherOpts), V, C.c_int]
    L.svob200_seeds_update.argtypes = [V, C.c_int64, C.POINTER(Camera), C.c_int, V, V, V, C.POINTER(MatcherOpts), C.c_double, V, V, C.c_int]
    L.svob200_update_seed.argtypes = [V, C.c_int, V, V, V]
    L.svob200_compute_tau.argtypes = [V, C.c_int, V, V, V, C.c_double, V]
    L.svob200_debug_chi2_chain.argtypes = [V, C.c_int, C.c_int, V, V, V, V, V]
    L.svob200_features_prepare.argtypes = [V, C.POINTER(Camera), C.c_int, V, V, V, C.c_int, V, V, V, C.c_int]
    L.svob200_compose_poses.argtypes = [V, C.c_int, V, V, V, C.c_int]
    L.svob200_reproject_prepare.argtypes = [V, C.POINTER(Camera), C.c_int, V, V, V, C.c_int, V, V, V, C.c_int]
    L.svob200_tracker_create.argtypes = [V, C.POINTER(Camera), C.c_int, C.c_int, C.POINTER(AlignOpts), C.POINTER(MatcherOpts), C.c_double,
                                         C.c_float, C.c_float, C.c_int, C.POINTER(V)]
    L.svob200_tracker_destroy.argtypes = [V]
    L.svob200_tracker_set_keyframe.argtypes = [V, V, C.c_int, V, V, V, V, V, V, V, V]
    L.svob200_tracker_set_last.argtypes = [V, V, C.c_int, C.c_int]
    L.svob200_tracker_set_seed_pool.argtypes = [V, C.c_int, C.c_int, C.c_int, C.c_int]
    L.svob200_tracker_set_detector.argtypes = [V, C.c_int, C.c_int, C.c_double]
    L.svob200_tracker_add_keyframe.argtypes = [V, V, V, V, V]
    L.svob200_tracker_add_keyframes.argtypes = [V, V, V, V, V, V, C.c_int]
    L.svob200_tracker_scene_depth.argtypes = [V, V, V, V, C.c_int]
    L.svob200_tracker_get_seed_refs.argtypes = [V, V, V, V, V, V]
    L.svob200_tracker_num_seed_slots.argtypes = [V]
    L.svob200_tracker_set_point_pool.argtypes = [V, C.c_int]
    L.svob200_tracker_num_point_slots.argtypes = [V]
    L.svob200_tracker_device_bytes.argtypes = [V]
    L.svob200_tracker_get_points.argtypes = [V, V, V, V, V, V]
    L.svob200_tracker_step.argtypes = [V, V, C.c_int, V, V, V, V, V, C.c_int]
    L.svob200_tracker_get_seeds.argtypes = [V, V]
    L.svob200_tracker_enable_profiling.argtypes = [V, C.c_int]
    L.svob200_tracker_stage_ms.argtypes = [V, c_fp, C.c_int]
    L.svob200_tracker_stage_name.restype = C.c_char_p
    L.svob200_tracker_stage_name.argtypes = [C.c_int]
    L.svob200_tracker_get_seed_obs.argtypes = [V, V]
    L.svob200_tracker_debug_align.argtypes = [V, V]
    L.svob200_tracker_set_chain.argtypes = [V, C.c_int, C.c_int, C.c_int]
    L.svob200_dev_alloc.argtypes = [V, C.c_size_t, C.POINTER(V)]
    L.svob200_dev_free.argtypes = [V, V]
    L.svob200_dev_upload.argtypes = [V, V, V, C.c_size_t]
    L.svob200_dev_download.argtypes = [V, V, V, C.c_size_t]
    L.svob200_host_alloc_pinned.argtypes = [V, C.c_size_t, C.POINTER(V)]
    L.svob200_host_free_pinned.argtypes = [V, V]
    L.svob200_frame_upload_level.argtypes = [V, C.c_int64, C.c_int, C.c_int, V, C.c_int]
    L.svob200_shi_tomasi.argtypes = [V, V, C.c_int, C.c_int, C.c_int, C.c_int, V, V]
    L.svob200_warp_matrix_affine.argtypes = [V, C.POINTER(Camera), C.c_int, V, V, V, V, V, V, C.c_int]
    L.svob200_warp_affine.argtypes = [V, V, C.c_int, C.c_int, C.c_int, V, V, C.c_int, C.c_int, C.c_int, V]
    L.svob200_depth_from_triangulation.argtypes = [V, C.c_int, V, V, V, V, V]
    L.svob200_synth_render.argtypes = [V, V, C.c_int, C.c_double, C.c_double, C.POINTER(Camera), C.c_int, V, V]
    L.svob200_frame_upload_yuv420.argtypes = [V, C.c_int64, V, C.c_int, V, V, C.c_int, C.c_int, C.c_size_t, C.c_size_t, c_ip, C.c_int]
    L.svob200_reproject_map.argtypes = [V, C.c_int64, C.POINTER(Camera), C.c_int, V, V, C.c_int, V, C.c_int, V, V, C.c_int, C.c_int,
                                        C.POINTER(MatcherOpts), V, V, V, C.c_int]
    L.svob200_pose_opt_opts_default.argtypes = [C.POINTER(PoseOptOpts)]
    L.svob200_pose_optimize.argtypes = [V, C.POINTER(Camera), C.c_int, V, V, V, V, C.POINTER(PoseOptOpts), V, V, V, C.c_int]
    L.svob200_points_optimize.argtypes = [V, C.c_int, V, V, V, C.c_int, C.c_double, V, V, C.c_int]
    L.svob200_seeds_initialize.argtypes = [V, C.c_int64, C.c_int, C.c_int, C.c_double, V, V, V, V, V, V, V, C.c_int]
    _lib = L
    return L


EXPORTED_SYMBOLS = [
    "svob200_ctx_create", "svob200_ctx_destroy", "svob200_last_error", "svob200_ctx_sync", "svob200_ctx_stream",
    "svob200_ctx_launch_count", "svob200_abi_sizes", "svob200_ctx_timer_start", "svob200_ctx_timer_stop_ms", "svob200_round_mode_x86",
    "svob200_frame_create", "svob200_frame_upload", "svob200_frame_bind", "svob200_frame_slot", "svob200_frame_download",
    "svob200_frame_release", "svob200_frame_info", "svob200_half_sample", "svob200_fast_detect", "svob200_fast_corners",
    "svob200_sparse_align", "svob200_align_patches", "svob200_matcher_opts_default", "svob200_match_direct",
    "svob200_epipolar_match", "svob200_seeds_update", "svob200_update_seed", "svob200_compute_tau", "svob200_dev_alloc",
    "svob200_dev_free", "svob200_dev_upload", "svob200_dev_download", "svob200_host_alloc_pinned", "svob200_host_free_pinned",
    "svob200_synth_render", "svob200_features_prepare", "svob200_compose_poses", "svob200_reproject_prepare",
    "svob200_tracker_create", "svob200_tracker_destroy", "svob200_tracker_set_keyframe", "svob200_tracker_set_last",
    "svob200_tracker_step", "svob200_tracker_get_seeds", "svob200_tracker_launches_per_step",
    "svob200_tracker_enable_profiling", "svob200_tracker_stage_ms", "svob200_tracker_get_seed_obs",
    "svob200_tracker_num_stages", "svob200_tracker_stage_name",
    "svob200_frame_upload_level", "svob200_shi_tomasi", "svob200_warp_matrix_affine", "svob200_warp_affine",
    "svob200_depth_from_triangulation", "svob200_debug_chi2_chain",
    "svob200_frame_upload_yuv420", "svob200_reproject_map", "svob200_pose_opt_opts_default", "svob200_pose_optimize",
    "svob200_points_optimize", "svob200_seeds_initialize", "svob200_tracker_debug_align", "svob200_tracker_set_chain",
    "svob200_tracker_set_seed_pool", "svob200_tracker_set_detector", "svob200_tracker_add_keyframe", "svob200_tracker_get_seed_refs",
    "svob200_tracker_num_seed_slots", "svob200_tracker_set_point_pool", "svob200_tracker_num_point_slots", "svob200_tracker_get_points",
    "svob200_tracker_add_keyframes", "svob200_tracker_scene_depth", "svob200_tracker_device_bytes",
]


def _ptr(a):
    """host numpy array, int device address, or None -> void*"""
    if a is None:
        return None
    if isinstance(a, (int, np.integer)):
        return C.c_void_p(int(a))
    return C.c_void_p(a.ctypes.data)


class Svob200Error(RuntimeError):
    pass


class Context:
    """One CUDA stream + device-resident frame store on one GPU."""

    def __init__(self, device=0):
        self.L = load_library()
        h = C.c_void_p()
        rc = self.L.svob200_ctx_create(int(device), C.byref(h))
        if rc != 0 or not h:
            raise Svob200Error("svob200_ctx_create(device=%d) failed with %d: no usable CUDA device — "
                               "this library has no CPU fallback" % (device, rc))
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.L.svob200_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc < 0:
            raise Svob200Error("svob200 error %d: %s" % (rc, self.L.svob200_last_error(self.h).decode()))
        return rc

    # ---- context
    def sync(self):
        self._ck(self.L.svob200_ctx_sync(self.h))

    def launch_count(self):
        return int(self.L.svob200_ctx_launch_count(self.h))

    def timer_start(self):
        self._ck(self.L.svob200_ctx_timer_start(self.h))

    def timer_stop_ms(self):
        ms = C.c_float(0)
        self._ck(self.L.svob200_ctx_timer_stop_ms(self.h, C.byref(ms)))
        return ms.value

    # ---- frames
    def frame_create(self, fid, batch, w, h, n_levels):
        self._ck(self.L.svob200_frame_create(self.h, fid, batch, w, h, n_levels))

    def frame_upload(self, fid, gray, stride=None, round_modes=None, mem=MEM_HOST):
        if mem == MEM_HOST:
            gray = np.ascontiguousarray(gray, dtype=np.uint8)
            stride = gray.shape[-1] if stride is None else stride
        modes = np.ascontiguousarray(round_modes, dtype=np.int32) if round_modes is not None else None
        self._ck(self.L.svob200_frame_upload(self.h, fid, _ptr(gray), int(stride), modes.ctypes.data_as(c_ip) if modes is not None else None, mem))

    def frame_bind(self, fid, dev_ptr, stride, round_modes=None):
        modes = np.ascontiguousarray(round_modes, dtype=np.int32) if round_modes is not None else None
        self._ck(self.L.svob200_frame_bind(self.h, fid, _ptr(dev_ptr), int(stride), modes.ctypes.data_as(c_ip) if modes is not None else None))

    def frame_slot(self, fid):
        return self._ck(self.L.svob200_frame_slot(self.h, fid))

    def frame_info(self, fid):
        b, w, h, n = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        self._ck(self.L.svob200_frame_info(self.h, fid, C.byref(b), C.byref(w), C.byref(h), C.byref(n)))
        return b.value, w.value, h.value, n.value

    def frame_download(self, fid, image, level):
        _, w, h, _ = self.frame_info(fid)
        lw, lh = w >> level, h >> level
        out = np.zeros((lh, lw), np.uint8)
        self._ck(self.L.svob200_frame_download(self.h, fid, image, level, _ptr(out), lw))
        return out

    def frame_release(self, fid):
        self._ck(self.L.svob200_frame_release(self.h, fid))

    def half_sample(self, img, mode):
        img = np.ascontiguousarray(img, dtype=np.uint8)
        h, w = img.shape
        out = np.zeros((h // 2, w // 2), np.uint8)
        self._ck(self.L.svob200_half_sample(self.h, _ptr(img), w, h, w, _ptr(out), w // 2, int(mode)))
        return out

    # ---- FAST
    def fast_detect(self, fid, n_detect_levels, cell, thr, occupancy=None):
        batch, w, h, _ = self.frame_info(fid)
        n_cells = -(-w // cell) * -(-h // cell)
        cells = np.zeros((batch, n_cells), corner_dt)
        counts = np.zeros(batch, np.int32)
        occ = np.ascontiguousarray(occupancy, dtype=np.uint8) if occupancy is not None else None
        self._ck(self.L.svob200_fast_detect(self.h, fid, n_detect_levels, cell, float(thr), _ptr(occ), _ptr(cells), _ptr(counts), MEM_HOST))
        return cells, counts

    def fast_corners(self, fid, image, level, thr=10, nonmax=True):
        _, w, h, _ = self.frame_info(fid)
        cap = (w >> level) * (h >> level)
        xs, ys, sc = np.zeros(cap, np.int32), np.zeros(cap, np.int32), np.zeros(cap, np.int32)
        n = self._ck(self.L.svob200_fast_corners(self.h, fid, image, level, int(thr), int(nonmax), cap, _ptr(xs), _ptr(ys), _ptr(sc)))
        return xs[:n].copy(), ys[:n].copy(), sc[:n].copy()

    # ---- sparse align
    def sparse_align(self, ref_fid, cur_fid, cam, offsets, px, xyz_ref, has_point, T_cur_ref, max_level, min_level, n_iter=30, eps=1e-6):
        offsets = np.ascontiguousarray(offsets, dtype=np.int32)
        batch = len(offsets) - 1
        px = np.ascontiguousarray(px, dtype=np.float64)
        xyz_ref = np.ascontiguousarray(xyz_ref, dtype=np.float64)
        has_point = np.ascontiguousarray(has_point, dtype=np.uint8)
        T = np.ascontiguousarray(T_cur_ref, dtype=np.float64)
        opts = AlignOpts(max_level, min_level, n_iter, eps)
        res = np.zeros(batch, align_result_dt)
        self._ck(self.L.svob200_sparse_align(self.h, ref_fid, cur_fid, C.byref(cam), batch, _ptr(offsets), _ptr(px), _ptr(xyz_ref),
                                             _ptr(has_point), _ptr(T), C.byref(opts), _ptr(res), MEM_HOST))
        return res

    # ---- feature alignment
    def align_patches(self, fid, level, image, pwb, patch, n_iter, px, dirv=None):
        image = np.ascontiguousarray(image, dtype=np.int32)
        n = len(image)
        pwb = np.ascontiguousarray(pwb, dtype=np.uint8)
        patch = np.ascontiguousarray(patch, dtype=np.uint8)
        px = np.ascontiguousarray(px, dtype=np.float64).copy()
        conv = np.zeros(n, np.int32)
        h_inv = np.zeros(n, np.float64)
        d = np.ascontiguousarray(dirv, dtype=np.float32) if dirv is not None else None
        self._ck(self.L.svob200_align_patches(self.h, fid, level, n, _ptr(image), _ptr(pwb), _ptr(patch), _ptr(d), n_iter,
                                              _ptr(px), _ptr(conv), _ptr(h_inv), MEM_HOST))
        return conv, px.reshape(n, 2), h_inv

    # ---- callers either side of the hot path (SURVEY §8f)
    def frame_upload_yuv420(self, fid, y, u, v, y_stride, uv_stride, uv_pixel_stride, y_image_stride=0, uv_image_stride=0,
                            round_modes=None, mem=MEM_HOST):
        """y/u/v: host uint8 arrays (u, v may be overlapping views of one interleaved buffer) or device addresses"""
        modes = np.ascontiguousarray(round_modes, dtype=np.int32) if round_modes is not None else None
        self._ck(self.L.svob200_frame_upload_yuv420(self.h, fid, _ptr(y), int(y_stride), _ptr(u), _ptr(v), int(uv_stride), int(uv_pixel_stride),
                                                    int(y_image_stride), int(uv_image_stride),
                                                    modes.ctypes.data_as(c_ip) if modes is not None else None, mem))

    def reproject_map(self, cur_fid, cam, T_cur_w, point_offsets, points, obs, T_obs_w, cell, max_fts, opts):
        T_cur_w = np.ascontiguousarray(T_cur_w, dtype=np.float64).reshape(-1, 7)
        batch = len(T_cur_w)
        off = np.ascontiguousarray(point_offsets, dtype=np.int32)
        points = np.ascontiguousarray(points, dtype=map_point_dt)
        obs = np.ascontiguousarray(obs, dtype=feature_ref_dt)
        T_obs_w = np.ascontiguousarray(T_obs_w, dtype=np.float64)
        n_cells = -(-cam.width // cell) * -(-cam.height // cell)
        res = np.zeros(len(points), reproj_result_dt)
        winner = np.zeros((batch, n_cells), np.int32)
        stats = np.zeros(batch, reproj_stats_dt)
        self._ck(self.L.svob200_reproject_map(self.h, cur_fid, C.byref(cam), batch, _ptr(T_cur_w), _ptr(off), len(points), _ptr(points),
                                              len(obs), _ptr(obs), _ptr(T_obs_w), int(cell), int(max_fts), C.byref(opts), _ptr(res),
                                              _ptr(winner), _ptr(stats), MEM_HOST))
        return res, winner, stats

    def pose_opt_opts(self, **kw):
        o = PoseOptOpts()
        self.L.svob200_pose_opt_opts_default(C.byref(o))
        for k, v in kw.items():
            setattr(o, k, v)
        return o

    def pose_optimize(self, cam, ftr_offsets, f, level, pos, T_f_w, opts=None):
        off = np.ascontiguousarray(ftr_offsets, dtype=np.int32)
        batch = len(off) - 1
        f = np.ascontiguousarray(f, dtype=np.float64); pos = np.ascontiguousarray(pos, dtype=np.float64)
        level = np.ascontiguousarray(level, dtype=np.int32)
        T = np.ascontiguousarray(T_f_w, dtype=np.float64).reshape(batch, 7).copy()
        res = np.zeros(batch, pose_opt_result_dt)
        outl = np.zeros(max(len(level), 1), np.uint8)
        opts = opts or self.pose_opt_opts()
        self._ck(self.L.svob200_pose_optimize(self.h, C.byref(cam), batch, _ptr(off), _ptr(f), _ptr(level), _ptr(pos), C.byref(opts), _ptr(T),
                                              _ptr(res), _ptr(outl), MEM_HOST))
        return T, res, outl[:len(level)]

    def points_optimize(self, obs_offsets, T_f_w, f, pos, n_iter=20, eps=1e-10):
        off = np.ascontiguousarray(obs_offsets, dtype=np.int32)
        n = len(off) - 1
        T = np.ascontiguousarray(T_f_w, dtype=np.float64); f = np.ascontiguousarray(f, dtype=np.float64)
        p = np.ascontiguousarray(pos, dtype=np.float64).reshape(n, 3).copy()
        it = np.zeros(n, np.int32)
        self._ck(self.L.svob200_points_optimize(self.h, n, _ptr(off), _ptr(T), _ptr(f), int(n_iter), float(eps), _ptr(p), _ptr(it), MEM_HOST))
        return p, it

    def seeds_initialize(self, fid, n_detect_levels, cell, thr, existing_offsets, existing_px, depth_mean, depth_min):
        batch, w, h, _ = self.frame_info(fid)
        n_cells = -(-w // cell) * -(-h // cell)
        off = np.ascontiguousarray(existing_offsets, dtype=np.int32)
        epx = np.ascontiguousarray(existing_px, dtype=np.float64)
        dm = np.ascontiguousarray(depth_mean, dtype=np.float32); dn = np.ascontiguousarray(depth_min, dtype=np.float32)
        corners = np.zeros((batch, n_cells), corner_dt)
        seeds = np.zeros((batch, n_cells), seed_dt)
        counts = np.zeros(batch, np.int32)
        self._ck(self.L.svob200_seeds_initialize(self.h, fid, int(n_detect_levels), int(cell), float(thr), _ptr(off), _ptr(epx), _ptr(dm), _ptr(dn),
                                                 _ptr(corners), _ptr(seeds), _ptr(counts), MEM_HOST))
        return corners, seeds, counts

    # ---- matcher
    def matcher_opts(self, n_pyr_levels, **kw):
        o = MatcherOpts()
        self.L.svob200_matcher_opts_default(C.byref(o), int(n_pyr_levels))
        for k, v in kw.items():
            setattr(o, k, v)
        return o

    def match_direct(self, cur_fid, cam, ftrs, depth_ref, px_cur_in, opts):
        n = len(ftrs)
        res = np.zeros(n, match_result_dt)
        d = np.ascontiguousarray(depth_ref, dtype=np.float64)
        p = np.ascontiguousarray(px_cur_in, dtype=np.float64)
        self._ck(self.L.svob200_match_direct(self.h, cur_fid, C.byref(cam), n, _ptr(ftrs), _ptr(d), _ptr(p), C.byref(opts), _ptr(res), MEM_HOST))
        return res

    def epipolar_match(self, cur_fid, cam, ftrs, d, opts):
        n = len(ftrs)
        res = np.zeros(n, epi_result_dt)
        d = np.ascontiguousarray(d, dtype=np.float64)
        self._ck(self.L.svob200_epipolar_match(self.h, cur_fid, C.byref(cam), n, _ptr(ftrs), _ptr(d), C.byref(opts), _ptr(res), MEM_HOST))
        return res

    # ---- depth filter
    def seeds_update(self, cur_fid, cam, ftrs, T_ref_w, T_cur_w, opts, conv_thresh, seeds):
        n = len(ftrs)
        obs = np.zeros(n, seed_obs_dt)
        seeds = np.ascontiguousarray(seeds, dtype=seed_dt).copy()
        Tr = np.ascontiguousarray(T_ref_w, dtype=np.float64)
        Tc = np.ascontiguousarray(T_cur_w, dtype=np.float64)
        self._ck(self.L.svob200_seeds_update(self.h, cur_fid, C.byref(cam), n, _ptr(ftrs), _ptr(Tr), _ptr(Tc), C.byref(opts),
                                             float(conv_thresh), _ptr(seeds), _ptr(obs), MEM_HOST))
        return seeds, obs

    def update_seed(self, x, tau2, seeds):
        x = np.ascontiguousarray(x, dtype=np.float32)
        tau2 = np.ascontiguousarray(tau2, dtype=np.float32)
        seeds = np.ascontiguousarray(seeds, dtype=seed_dt).copy()
        self._ck(self.L.svob200_update_seed(self.h, len(x), _ptr(x), _ptr(tau2), _ptr(seeds)))
        return seeds

    def debug_chi2_chain(self, res, visible, contrib, block=256):
        """The device replays of the reference's sequential float chi2 chain: [(sum, count)] for serial, parallel (latency mode),
        parallel (128-thread batch kernel, one staging buffer), parallel (256/512-thread batch kernels, double-buffered)."""
        res = np.ascontiguousarray(res, dtype=np.float32).reshape(-1, 16)
        vis = np.ascontiguousarray(visible, dtype=np.uint8)
        con = np.ascontiguousarray(contrib, dtype=np.uint8)
        sums = np.zeros(4, np.float32)
        cnts = np.zeros(4, np.int32)
        self._ck(self.L.svob200_debug_chi2_chain(self.h, int(block), len(res), _ptr(res), _ptr(vis), _ptr(con), _ptr(sums), _ptr(cnts)))
        return [(sums[i], int(cnts[i])) for i in range(4)]

    def compute_tau(self, T_ref_cur, f, z, ang):
        T = np.ascontiguousarray(T_ref_cur, dtype=np.float64)
        f = np.ascontiguousarray(f, dtype=np.float64)
        z = np.ascontiguousarray(z, dtype=np.float64)
        out = np.zeros(len(z))
        self._ck(self.L.svob200_compute_tau(self.h, len(z), _ptr(T), _ptr(f), _ptr(z), float(ang), _ptr(out)))
        return out

    # ---- raw device helpers
    def dev_alloc(self, nbytes):
        p = C.c_void_p()
        self._ck(self.L.svob200_dev_alloc(self.h, nbytes, C.byref(p)))
        return p.value

    def dev_free(self, dptr):
        self._ck(self.L.svob200_dev_free(self.h, C.c_void_p(dptr)))

    def dev_upload(self, dptr, arr):
        arr = np.ascontiguousarray(arr)
        self._ck(self.L.svob200_dev_upload(self.h, C.c_void_p(dptr), _ptr(arr), arr.nbytes))

    def dev_download(self, arr, dptr):
        self._ck(self.L.svob200_dev_download(self.h, _ptr(arr), C.c_void_p(dptr), arr.nbytes))

    def synth_render(self, dev_tex, tex_size, ppm, plane_z, cam, poses, dev_out):
        poses = np.ascontiguousarray(poses, dtype=np.float64).reshape(-1, 7)
        self._ck(self.L.svob200_synth_render(self.h, C.c_void_p(dev_tex), tex_size, float(ppm), float(plane_z), C.byref(cam),
                                             len(poses), _ptr(poses), C.c_void_p(dev_out)))


def abi_sizes():
    """(C sizeof, numpy/ctypes sizeof) pairs for every struct crossing the ABI."""
    L = load_library()
    buf = (C.c_int * 32)()
    n = L.svob200_abi_sizes(buf, 32)
    mine = [C.sizeof(Camera), corner_dt.itemsize, C.sizeof(AlignOpts), align_result_dt.itemsize, C.sizeof(MatcherOpts),
            feature_ref_dt.itemsize, match_result_dt.itemsize, epi_result_dt.itemsize, seed_dt.itemsize, seed_obs_dt.itemsize,
            step_stats_dt.itemsize, map_point_dt.itemsize, reproj_result_dt.itemsize, reproj_stats_dt.itemsize,
            pose_opt_result_dt.itemsize, C.sizeof(PoseOptOpts)]
    return list(buf[:n]), mine


def make_feature_refs(n):
    return np.zeros(n, feature_ref_dt)


class Tracker:
    """svob200_tracker: one front-end step per call over a batch of independent sequences."""

    def __init__(self, ctx, cam, batch, n_levels, max_level, min_level, n_pyr_levels_cfg, conv_thresh=100.0, depth_mean=2.4,
                 depth_min=1.2, reseed=1, n_iter=30, eps=1e-6):
        self.ctx, self.L, self.batch = ctx, ctx.L, batch
        self.cam = cam
        ao = AlignOpts(max_level, min_level, n_iter, eps)
        mo = ctx.matcher_opts(n_pyr_levels_cfg)
        h = C.c_void_p()
        ctx._ck(self.L.svob200_tracker_create(ctx.h, C.byref(cam), batch, n_levels, C.byref(ao), C.byref(mo), float(conv_thresh),
                                              depth_mean, depth_min, int(reseed), C.byref(h)))
        self.h = h
        self.N = self.S = 0

    def set_keyframe(self, imgs, T_kf_w, ftr_offsets, kf_px, kf_level, pt_world, seed_offsets, seed_px, seed_level):
        imgs = np.ascontiguousarray(imgs, dtype=np.uint8)
        a = lambda x, t: np.ascontiguousarray(x, dtype=t)
        fo, so = a(ftr_offsets, np.int32), a(seed_offsets, np.int32)
        self.N, self.S = int(fo[-1]), int(so[-1])
        args = [a(T_kf_w, np.float64), fo, a(kf_px, np.float64), a(kf_level, np.int32), a(pt_world, np.float64), so,
                a(seed_px, np.float64), a(seed_level, np.int32)]
        self.ctx._ck(self.L.svob200_tracker_set_keyframe(self.h, _ptr(imgs), imgs.shape[-1], *[_ptr(x) for x in args]))
        self.S = int(self.L.svob200_tracker_num_seed_slots(self.h))          # pool slots (>= the seeds given)
        self.N = int(self.L.svob200_tracker_num_point_slots(self.h))         # point slots (>= the map points given)

    @property
    def P(self):
        """point slots: the length of every per-map-feature array of a step"""
        return self.N

    # ---- keyframe insertion inside the tracker
    def set_seed_pool(self, capacity_per_sequence, max_keyframes=4, max_n_kfs=3, reseed=3):
        self.ctx._ck(self.L.svob200_tracker_set_seed_pool(self.h, int(capacity_per_sequence), int(max_keyframes), int(max_n_kfs), int(reseed)))

    def set_point_pool(self, capacity_per_sequence):
        """converged seeds become map points (svob200_tracker_set_point_pool): call before set_keyframe"""
        self.ctx._ck(self.L.svob200_tracker_set_point_pool(self.h, int(capacity_per_sequence)))

    def points(self):
        """(pos[P,3], type[P], n_obs[P], created[batch], dropped[batch]) of the point slots; type SVOB200_POINT_*"""
        P = self.N
        pos = np.zeros((max(P, 1), 3)); ty = np.zeros(max(P, 1), np.int32); no = np.zeros(max(P, 1), np.int32)
        cr = np.zeros(self.batch, np.int32); dr = np.zeros(self.batch, np.int32)
        self.ctx._ck(self.L.svob200_tracker_get_points(self.h, _ptr(pos), _ptr(ty), _ptr(no), _ptr(cr), _ptr(dr)))
        return pos[:P], ty[:P], no[:P], cr, dr

    def device_bytes(self):
        """bytes of device memory the tracker's own arrays hold now (svob200_tracker_device_bytes; frames not included)"""
        return int(self.L.svob200_tracker_device_bytes(self.h))

    def set_detector(self, cell, levels, thr):
        self.ctx._ck(self.L.svob200_tracker_set_detector(self.h, int(cell), int(levels), float(thr)))

    def add_keyframe(self, depth_mean, depth_min):
        """the frame of the most recent step becomes a keyframe: returns (new seeds, dropped corners) per sequence"""
        dm = np.ascontiguousarray(np.broadcast_to(np.asarray(depth_mean, np.float32), (self.batch,)))
        dn = np.ascontiguousarray(np.broadcast_to(np.asarray(depth_min, np.float32), (self.batch,)))
        n_new = np.zeros(self.batch, np.int32); n_drop = np.zeros(self.batch, np.int32)
        self.ctx._ck(self.L.svob200_tracker_add_keyframe(self.h, _ptr(dm), _ptr(dn), _ptr(n_new), _ptr(n_drop)))
        return n_new, n_drop

    def add_keyframes(self, which, depth_mean, depth_min):
        """the frame of the most recent step becomes a keyframe of the sequences with which[b] != 0 (None: every sequence), each
        in its own ring: returns (new seeds, dropped corners) per sequence, 0 for the sequences not selected and -1 for a
        selected sequence that has used up its 65,534 keyframes"""
        w = None if which is None else np.ascontiguousarray(np.broadcast_to(np.asarray(which) != 0, (self.batch,)), dtype=np.uint8)
        dm = np.ascontiguousarray(np.broadcast_to(np.asarray(depth_mean, np.float32), (self.batch,)))
        dn = np.ascontiguousarray(np.broadcast_to(np.asarray(depth_min, np.float32), (self.batch,)))
        n_new = np.zeros(self.batch, np.int32); n_drop = np.zeros(self.batch, np.int32)
        self.ctx._ck(self.L.svob200_tracker_add_keyframes(self.h, _ptr(w), _ptr(dm), _ptr(dn), _ptr(n_new), _ptr(n_drop), MEM_HOST))
        return n_new, n_drop

    def add_keyframes_raw(self, which_ptr, depth_mean_ptr, depth_min_ptr, n_new_ptr=0, n_dropped_ptr=0, mem=MEM_DEVICE):
        """Pointer-level add_keyframes (device addresses by default: ordered on the context's stream, no synchronisation);
        0 for which_ptr = every sequence, 0 for an output = not wanted."""
        V = lambda p: C.c_void_p(p) if p else None
        self.ctx._ck(self.L.svob200_tracker_add_keyframes(self.h, V(which_ptr), V(depth_mean_ptr), V(depth_min_ptr), V(n_new_ptr), V(n_dropped_ptr), int(mem)))

    def scene_depth(self, depth_mean=None, depth_min=None):
        """frame_utils::getSceneDepth of the most recent step's frame per sequence: (depth_mean, depth_min, n_points); a sequence
        without a matched point keeps the value of the arrays passed in (default NaN)"""
        dm = np.array(np.broadcast_to(np.nan if depth_mean is None else np.asarray(depth_mean, np.float32), (self.batch,)), np.float32)
        dn = np.array(np.broadcast_to(np.nan if depth_min is None else np.asarray(depth_min, np.float32), (self.batch,)), np.float32)
        n = np.zeros(self.batch, np.int32)
        self.ctx._ck(self.L.svob200_tracker_scene_depth(self.h, _ptr(dm), _ptr(dn), _ptr(n), MEM_HOST))
        return dm, dn, n

    def scene_depth_raw(self, depth_mean_ptr, depth_min_ptr, n_points_ptr=0, mem=MEM_DEVICE):
        """Pointer-level scene_depth (device addresses by default: ordered on the context's stream, no synchronisation)"""
        self.ctx._ck(self.L.svob200_tracker_scene_depth(self.h, C.c_void_p(depth_mean_ptr), C.c_void_p(depth_min_ptr),
                                                         C.c_void_p(n_points_ptr) if n_points_ptr else None, int(mem)))

    def seed_refs(self):
        """(px[S,2], level, kf, batch_id, state) of every pool slot; state 0 = alive"""
        S = self.S
        px = np.zeros((max(S, 1), 2)); lv = np.zeros(max(S, 1), np.int32); kf = np.zeros(max(S, 1), np.int32)
        bt = np.zeros(max(S, 1), np.int32); st = np.zeros(max(S, 1), np.int32)
        self.ctx._ck(self.L.svob200_tracker_get_seed_refs(self.h, _ptr(px), _ptr(lv), _ptr(kf), _ptr(bt), _ptr(st)))
        return px[:S], lv[:S], kf[:S], bt[:S], st[:S]

    def set_last(self, imgs, mem=MEM_HOST, stride=None):
        if mem == MEM_HOST:
            imgs = np.ascontiguousarray(imgs, dtype=np.uint8)
            stride = imgs.shape[-1]
        self.ctx._ck(self.L.svob200_tracker_set_last(self.h, _ptr(imgs), int(stride), mem))

    def set_chain(self, cell_size=30, max_fts=120, pose_opt=1):
        """reprojector grid rules + pose optimiser between alignment and the depth filter (svob200_tracker_set_chain)"""
        self.ctx._ck(self.L.svob200_tracker_set_chain(self.h, int(cell_size), int(max_fts), int(pose_opt)))

    def step(self, cur_imgs, T_last_w, last_px, want_px=False):
        """Host-memory step: returns per-sequence stats (and refined pixels / success flags)."""
        cur_imgs = np.ascontiguousarray(cur_imgs, dtype=np.uint8)
        T = np.ascontiguousarray(T_last_w, dtype=np.float64)
        lp = np.ascontiguousarray(last_px, dtype=np.float64)
        stats = np.zeros(self.batch, step_stats_dt)
        px = np.zeros((self.N, 2)) if want_px else None
        ok = np.zeros(self.N, np.int32) if want_px else None
        self.ctx._ck(self.L.svob200_tracker_step(self.h, _ptr(cur_imgs), cur_imgs.shape[-1], _ptr(T), _ptr(lp), _ptr(stats),
                                                 _ptr(px), _ptr(ok), MEM_HOST))
        return (stats, px, ok) if want_px else stats

    def step_device(self, cur_imgs, T_last_w, last_px, want_px=False):
        """The same step with EVERY argument resident in device memory (SVOB200_MEM_DEVICE): level 0 of the current
        frame aliases the caller's device buffer, nothing is staged, the whole batch runs on the
        context's stream (a CUDA graph with forked branches for small batches, the depth filter on its own stream for larger
        ones).  This is the path bench.py's `value` times.  The images go through a ring of three device buffers (the aliased
        frame must stay valid through the next two steps)."""
        cur_imgs = np.ascontiguousarray(cur_imgs, dtype=np.uint8)
        T = np.ascontiguousarray(T_last_w, dtype=np.float64)
        lp = np.ascontiguousarray(last_px, dtype=np.float64)
        ctx = self.ctx
        if getattr(self, "_dev", None) is None:
            self._dev = dict(ring=[ctx.dev_alloc(cur_imgs.nbytes) for _ in range(3)], k=0, T=ctx.dev_alloc(T.nbytes), lp=ctx.dev_alloc(max(lp.nbytes, 8)),
                             stats=ctx.dev_alloc(self.batch * step_stats_dt.itemsize), px=ctx.dev_alloc(max(self.N, 1) * 16),
                             ok=ctx.dev_alloc(max(self.N, 1) * 4))
        d = self._dev
        img = d["ring"][d["k"] % 3]
        d["k"] += 1
        ctx.dev_upload(img, cur_imgs); ctx.dev_upload(d["T"], T); ctx.dev_upload(d["lp"], lp)
        V = C.c_void_p
        ctx._ck(self.L.svob200_tracker_step(self.h, V(img), cur_imgs.shape[-1], V(d["T"]), V(d["lp"]), V(d["stats"]),
                                            V(d["px"]) if want_px else None, V(d["ok"]) if want_px else None, MEM_DEVICE))
        ctx.sync()
        stats = np.zeros(self.batch, step_stats_dt)
        ctx.dev_download(stats, d["stats"])
        if not want_px:
            return stats
        px = np.zeros((self.N, 2)); ok = np.zeros(self.N, np.int32)
        if self.N:
            ctx.dev_download(px, d["px"]); ctx.dev_download(ok, d["ok"])
        return stats, px, ok

    def set_last_device(self, imgs):
        """last frame from a device buffer (svob200_tracker_set_last with SVOB200_MEM_DEVICE)"""
        imgs = np.ascontiguousarray(imgs, dtype=np.uint8)
        d = self.ctx.dev_alloc(imgs.nbytes)
        self.ctx.dev_upload(d, imgs)
        self.ctx._ck(self.L.svob200_tracker_set_last(self.h, C.c_void_p(d), imgs.shape[-1], MEM_DEVICE))
        self.ctx.sync()
        self.ctx.dev_free(d)

    def step_raw(self, cur_ptr, stride, T_ptr, px_ptr, stats_ptr, mem):
        """Pointer-level step (pinned host or device addresses), no allocation on the Python side."""
        rc = self.L.svob200_tracker_step(self.h, C.c_void_p(cur_ptr), int(stride), C.c_void_p(T_ptr), C.c_void_p(px_ptr),
                                         C.c_void_p(stats_ptr) if stats_ptr else None, None, None, mem)
        if rc < 0:
            self.ctx._ck(rc)

    def seeds(self):
        out = np.zeros(max(self.S, 1), seed_dt)
        self.ctx._ck(self.L.svob200_tracker_get_seeds(self.h, _ptr(out)))
        return out[:self.S]

    def seed_obs(self):
        out = np.zeros(max(self.S, 1), seed_obs_dt)
        self.ctx._ck(self.L.svob200_tracker_get_seed_obs(self.h, _ptr(out)))
        return out[:self.S]

    def enable_profiling(self, on=True):
        self.ctx._ck(self.L.svob200_tracker_enable_profiling(self.h, int(on)))

    def stage_ms(self):
        """CUDA-event duration of every stage (kernel) of the most recent step, by name."""
        n = self.L.svob200_tracker_num_stages()
        ms = (C.c_float * n)()
        self.ctx._ck(self.L.svob200_tracker_stage_ms(self.h, ms, n))
        return {self.L.svob200_tracker_stage_name(i).decode(): float(ms[i]) for i in range(n)}

    def close(self):
        if getattr(self, "h", None):
            self.L.svob200_tracker_destroy(self.h)          # synchronises the stream first
            self.h = None
            d = getattr(self, "_dev", None)
            if d is not None:
                for p in d["ring"] + [d[k] for k in ("T", "lp", "stats", "px", "ok")]:
                    self.ctx.dev_free(p)
                self._dev = None
