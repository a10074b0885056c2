"""ctypes binding of libhafgpu.so (include/hafgpu.h).  Thin: every call goes straight to the C ABI.

There is no CPU fallback anywhere in this package: if libhafgpu.so is missing or no sm_100 device is
visible, construction raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build

HAF_SVM_TENSOR_GUARD = 0
HAF_SVM_FP64_EXACT = 1
HAF_SVM_FP32_GUARD = 2
CHUNK_RECORD = 10   # ints per chunk of haf_debug_chunk_copy_waits (HAF_CHUNK_RECORD)


class HafError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libhafgpu error %d: %s" % (code, msg))
        self.code = code


class haf_config(C.Structure):
    _fields_ = [("features_path", C.c_char_p), ("range_path", C.c_char_p), ("model_path", C.c_char_p),
                ("nr_features_without_shaf", C.c_int), ("grid", C.c_int), ("roll_step_deg", C.c_int),
                ("roll_max_deg", C.c_int), ("device", C.c_int), ("emulate_text_roundtrip", C.c_int),
                ("svm_mode", C.c_int), ("guard_rel", C.c_float), ("reserved", C.c_int * 4), ("n_devices", C.c_int),
                ("devices", C.POINTER(C.c_int))]


class haf_request(C.Structure):
    _fields_ = [("center", C.c_double * 3), ("area_len_x", C.c_float), ("area_len_y", C.c_float),
                ("approach", C.c_double * 3), ("gripper_opening_width", C.c_int), ("return_only_best", C.c_int),
                ("graspval_top", C.c_int), ("roll_limit", C.c_int), ("roll_begin", C.c_int), ("svm_with_probability", C.c_int)]


class haf_best(C.Structure):
    _fields_ = [("row", C.c_int), ("col", C.c_int), ("roll", C.c_int), ("tilt", C.c_int), ("approach_idx", C.c_int),
                ("topval", C.c_int), ("eval", C.c_int), ("roll_rad", C.c_float), ("M", C.c_float * 16),
                ("rolls_done", C.c_int), ("n_windows_scored", C.c_int), ("n_guard", C.c_int), ("reserved", C.c_int)]

    def astuple(self):
        return (self.row, self.col, self.roll, self.tilt, self.topval)


class haf_grasp(C.Structure):
    """GraspOutput (msg/GraspOutput.msg) of one grasp plus the cell and roll it was built from (include/hafgpu.h)."""
    _fields_ = [("eval", C.c_int), ("roll", C.c_float), ("graspPoint1", C.c_double * 3), ("graspPoint2", C.c_double * 3),
                ("averagedGraspPoint", C.c_double * 3), ("approachVector", C.c_double * 3), ("row", C.c_int), ("col", C.c_int),
                ("roll_index", C.c_int), ("reserved", C.c_int)]

    def as_array(self) -> np.ndarray:
        """the 13 doubles gp1 xyz, gp2 xyz, averaged xyz, approach xyz, roll (rad) -- the oracle's transform_gp_in_wcs order"""
        return np.array(list(self.graspPoint1) + list(self.graspPoint2) + list(self.averagedGraspPoint) +
                        list(self.approachVector) + [self.roll], np.float64)


class haf_rank_params(C.Structure):
    """parameters of haf_search_batch_candidates (include/hafgpu.h)"""
    _fields_ = [("k", C.c_int), ("per_unit", C.c_int), ("min_distance", C.c_double), ("reserved", C.c_int * 4)]


class haf_candidate(C.Structure):
    """one ranked grasp candidate: the full haf_grasp, the graspseval value of its cell and its request within the cloud"""
    _fields_ = [("grasp", haf_grasp), ("score", C.c_float), ("request", C.c_int)]


HAF_DEPTH_U16 = 1   # 16UC1 / mono16, 0 = no return
HAF_DEPTH_F32 = 2   # 32FC1 metres, non-finite = no return


class haf_depth_image(C.Structure):
    """one depth image of haf_depth_to_xyz_batch (include/hafgpu.h): size, encoding, row step, intrinsics, scale and pose"""
    _fields_ = [("width", C.c_int), ("height", C.c_int), ("encoding", C.c_int), ("has_pose", C.c_int), ("step", C.c_longlong),
                ("fx", C.c_double), ("fy", C.c_double), ("cx", C.c_double), ("cy", C.c_double), ("depth_scale", C.c_float),
                ("camera_to_base", C.c_float * 16), ("reserved", C.c_int * 3)]


class haf_info(C.Structure):
    _fields_ = [("n_features", C.c_int), ("n_dims", C.c_int), ("n_sv", C.c_int), ("n_rolls", C.c_int), ("grid", C.c_int),
                ("label0", C.c_int), ("label1", C.c_int), ("sm_count", C.c_int), ("gamma", C.c_double),
                ("rho", C.c_double), ("reserved", C.c_int * 4)]


class haf_timing(C.Structure):
    _fields_ = [("ms_total", C.c_float), ("ms_bin", C.c_float), ("ms_integral", C.c_float), ("ms_mask", C.c_float),
                ("ms_features", C.c_float), ("ms_svm", C.c_float), ("ms_guard", C.c_float), ("ms_score", C.c_float),
                ("n_points", C.c_longlong), ("n_units", C.c_longlong), ("n_windows", C.c_longlong),
                ("n_guard", C.c_longlong), ("launches", C.c_longlong), ("n_chunks", C.c_longlong),
                ("n_exact", C.c_longlong), ("n_audit", C.c_longlong), ("audit_max_rel", C.c_float), ("tc_passes", C.c_int),
                ("escalations", C.c_int), ("graph_replays", C.c_int), ("n_clamped", C.c_longlong)]


EXPORTS = ["haf_create", "haf_destroy", "haf_last_error", "haf_get_info", "haf_set_stream", "haf_set_profiling",
           "haf_get_timing", "haf_launch_count", "haf_set_debug", "haf_search", "haf_search_batch", "haf_search_batch_packed",
           "haf_search_grasps", "haf_search_batch_packed_grasps", "haf_search_batch_requests", "haf_search_batch_candidates", "haf_debug_unit_params", "haf_debug_chunk_copy_waits", "haf_debug_heights", "haf_build_transform", "haf_build_transform_wcs", "haf_best_key", "haf_pack_best_records", "haf_debug_window_count", "haf_debug_windows", "haf_debug_features",
           "haf_debug_decisions", "haf_debug_tensor_inputs", "haf_debug_integral", "haf_debug_cell_indices", "haf_debug_text_roundtrip", "haf_debug_tc_probe",
           "haf_version", "haf_pcd_decode", "haf_search_pcd", "haf_pointcloud2_to_xyz", "haf_debug_pcd_xyz",
           "haf_pcd_decode_batch", "haf_search_batch_pcd", "haf_pointcloud2_batch_to_xyz", "haf_depth_to_xyz_batch", "haf_search_batch_depth", "haf_svm_create", "haf_svm_create_config", "haf_svm_destroy", "haf_svm_predict", "haf_svm_predict_probability", "haf_svm_check_probability_model", "haf_scale_minmax", "haf_scale_apply"]

_lib = None


def load_library(build_if_missing: bool = True) -> C.CDLL:
    """Loads (building first if the .so is absent or stale and nvcc is here) libhafgpu.so.  Raises if impossible."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    if build_if_missing and _build.needs_build():
        try:
            _build.build_lib()
        except Exception as exc:  # no nvcc on this box: use the prebuilt file if there is one
            if not os.path.exists(path):
                raise RuntimeError("libhafgpu.so is not built and cannot be built here: %s" % exc)
    if not os.path.exists(path):
        raise RuntimeError("libhafgpu.so missing at %s (run __graft_entry__.build())" % path)
    L = C.CDLL(path)
    vp, ci, cs = C.c_void_p, C.c_int, C.c_size_t
    L.haf_create.argtypes = [C.POINTER(vp), C.POINTER(haf_config)]
    L.haf_destroy.argtypes = [vp]
    L.haf_destroy.restype = None
    L.haf_last_error.argtypes = [vp]
    L.haf_last_error.restype = C.c_char_p
    L.haf_get_info.argtypes = [vp, C.POINTER(haf_info)]
    L.haf_set_stream.argtypes = [vp, vp]
    L.haf_set_profiling.argtypes = [vp, ci]
    L.haf_set_debug.argtypes = [vp, ci]
    L.haf_get_timing.argtypes = [vp, C.POINTER(haf_timing)]
    L.haf_launch_count.argtypes = [vp]
    L.haf_launch_count.restype = C.c_longlong
    L.haf_search.argtypes = [vp, vp, cs, cs, C.POINTER(haf_request), ci, C.POINTER(haf_best), C.POINTER(haf_best), vp, vp, vp, vp]
    L.haf_search_batch.argtypes = [vp, C.POINTER(vp), C.POINTER(cs), ci, C.POINTER(haf_request), C.POINTER(haf_best)]
    L.haf_search_batch_packed.argtypes = [vp, vp, C.POINTER(cs), ci, C.POINTER(haf_request), C.POINTER(haf_best)]
    L.haf_search_grasps.argtypes = [vp, vp, cs, cs, C.POINTER(haf_request), ci, C.POINTER(haf_best), C.POINTER(haf_best), vp, vp, vp, vp,
                                    C.POINTER(haf_grasp), C.POINTER(haf_grasp), C.POINTER(haf_grasp)]
    L.haf_search_batch_packed_grasps.argtypes = [vp, vp, C.POINTER(cs), ci, C.POINTER(haf_request), C.POINTER(haf_best),
                                                 C.POINTER(haf_grasp), C.POINTER(haf_grasp)]
    L.haf_search_batch_requests.argtypes = [vp, vp, C.POINTER(cs), ci, C.POINTER(haf_request), C.POINTER(ci), C.POINTER(haf_best),
                                            C.POINTER(haf_best), vp, C.POINTER(haf_grasp), C.POINTER(haf_grasp), C.POINTER(haf_grasp)]
    L.haf_search_batch_candidates.argtypes = [vp, vp, C.POINTER(cs), ci, C.POINTER(haf_request), C.POINTER(ci), C.POINTER(haf_rank_params),
                                              C.POINTER(haf_best), C.POINTER(haf_grasp), C.POINTER(haf_candidate), vp]
    L.haf_debug_unit_params.argtypes = [vp, vp, vp, vp, ci]
    L.haf_debug_chunk_copy_waits.argtypes = [vp, vp, ci]
    L.haf_debug_heights.argtypes = [vp, vp, cs]
    L.haf_build_transform.argtypes = [C.POINTER(haf_request), ci, ci, C.POINTER(C.c_float)]
    L.haf_build_transform_wcs.argtypes = [C.POINTER(haf_request), ci, ci, C.POINTER(C.c_float)]
    L.haf_best_key.argtypes = [ci, C.c_uint32]
    L.haf_best_key.restype = C.c_uint64
    L.haf_pack_best_records.argtypes = [vp, ci, vp]
    L.haf_debug_window_count.argtypes = [vp]
    L.haf_debug_windows.argtypes = [vp, vp, ci]
    L.haf_debug_features.argtypes = [vp, vp, vp, ci]
    L.haf_debug_decisions.argtypes = [vp, vp, vp, vp, ci]
    L.haf_debug_tensor_inputs.argtypes = [vp, vp, ci]
    L.haf_debug_integral.argtypes = [vp, vp, cs]
    L.haf_debug_cell_indices.argtypes = [vp, vp, cs, cs, C.POINTER(haf_request), ci, vp]
    L.haf_debug_text_roundtrip.argtypes = [vp, vp, ci, vp, vp, ci, vp]
    L.haf_debug_tc_probe.argtypes = [vp, vp, ci]
    L.haf_version.restype = C.c_char_p
    L.haf_pcd_decode.argtypes = [vp, vp, cs, C.POINTER(vp), C.POINTER(cs)]
    L.haf_search_pcd.argtypes = [vp, vp, cs, C.POINTER(haf_request), ci, C.POINTER(haf_best), C.POINTER(haf_best), vp, vp, vp, vp]
    L.haf_pointcloud2_to_xyz.argtypes = [vp, vp, cs, cs, ci, ci, ci, C.POINTER(vp)]
    L.haf_debug_pcd_xyz.argtypes = [vp, vp, cs]
    L.haf_pcd_decode_batch.argtypes = [vp, vp, C.POINTER(cs), ci, C.POINTER(vp), C.POINTER(cs)]
    L.haf_search_batch_pcd.argtypes = [vp, vp, C.POINTER(cs), ci, C.POINTER(haf_request), C.POINTER(ci), C.POINTER(haf_best),
                                       C.POINTER(haf_best), vp, C.POINTER(haf_grasp), C.POINTER(haf_grasp), C.POINTER(haf_grasp)]
    L.haf_pointcloud2_batch_to_xyz.argtypes = [vp, vp, C.POINTER(cs), ci, C.POINTER(ci), C.POINTER(vp), C.POINTER(cs)]
    L.haf_depth_to_xyz_batch.argtypes = [vp, vp, C.POINTER(cs), ci, C.POINTER(haf_depth_image), C.POINTER(vp), C.POINTER(cs)]
    L.haf_search_batch_depth.argtypes = [vp, vp, C.POINTER(cs), ci, C.POINTER(haf_depth_image), C.POINTER(haf_request), C.POINTER(ci),
                                         C.POINTER(haf_best), C.POINTER(haf_best), vp, C.POINTER(haf_grasp), C.POINTER(haf_grasp), C.POINTER(haf_grasp)]
    L.haf_svm_create.argtypes = [C.POINTER(vp), C.c_char_p, ci, ci, ci, C.c_float]
    L.haf_svm_create_config.argtypes = [C.POINTER(vp), C.POINTER(haf_config), ci]
    L.haf_svm_destroy.argtypes = [vp]
    L.haf_svm_destroy.restype = None
    L.haf_svm_predict.argtypes = [vp, vp, vp, vp, ci, vp, vp]
    L.haf_svm_predict_probability.argtypes = [vp, vp, vp, vp, ci, vp, vp]
    L.haf_svm_check_probability_model.argtypes = [vp]
    L.haf_scale_minmax.argtypes = [ci, vp, vp, vp, ci, ci, vp, vp]
    L.haf_scale_apply.argtypes = [ci, vp, vp, vp, ci, ci, vp, vp, C.c_double, C.c_double, vp]
    _lib = L
    return L


def make_request(center=(0.0, 0.0, 0.0), area=(32.0, 44.0), approach=(0.0, 0.0, 1.0), width=1, return_only_best=0,
                 graspval_top=119, roll_limit=0, roll_begin=0, svm_with_probability=0) -> haf_request:
    """GraspInput defaults of the reference client (client.cpp:79-118; area = size + 14, client.cpp:183-184)."""
    rq = haf_request()
    rq.center[:] = center
    rq.area_len_x, rq.area_len_y = area
    rq.approach[:] = approach
    rq.gripper_opening_width = width
    rq.return_only_best = return_only_best
    rq.graspval_top = graspval_top
    rq.roll_limit = roll_limit
    rq.roll_begin = roll_begin
    rq.svm_with_probability = svm_with_probability
    return rq


def make_requests(n=None, centers=(0.0, 0.0, 0.0), approaches=(0.0, 0.0, 1.0), areas=(32.0, 44.0), widths=1, return_only_best=0,
                  graspval_top=119, roll_limit=0, roll_begin=0, svm_with_probability=0):
    """Vectorised ``make_request``: a ctypes array of n haf_request.  Every argument is one value (broadcast) or one per request:
    centers / approaches [n, 3], areas [n, 2], the int fields [n].  n defaults to the longest per-request argument."""
    vec = dict(centers=np.asarray(centers, np.float64), approaches=np.asarray(approaches, np.float64), areas=np.asarray(areas, np.float32))
    ints = dict(gripper_opening_width=widths, return_only_best=return_only_best, graspval_top=graspval_top, roll_limit=roll_limit,
                roll_begin=roll_begin, svm_with_probability=svm_with_probability)
    ints = {k: np.asarray(v, np.int32) for k, v in ints.items()}
    if n is None:
        n = max([len(v) for v in vec.values() if v.ndim == 2] + [len(v) for v in ints.values() if v.ndim == 1] + [1])
    arr = (haf_request * n)()
    rec = np.frombuffer(arr, np.dtype({"names": [f[0] for f in haf_request._fields_],
                                       "formats": [(np.float64, 3), np.float32, np.float32, (np.float64, 3)] + [np.int32] * 6,
                                       "offsets": [getattr(haf_request, f[0]).offset for f in haf_request._fields_],
                                       "itemsize": C.sizeof(haf_request)}))
    rec["center"] = np.broadcast_to(vec["centers"], (n, 3))
    areas = np.broadcast_to(vec["areas"], (n, 2))
    rec["area_len_x"], rec["area_len_y"] = areas[:, 0], areas[:, 1]
    rec["approach"] = np.broadcast_to(vec["approaches"], (n, 3))
    for k, v in ints.items():
        rec[k] = np.broadcast_to(v, (n,))
    return arr


def _ptr(a):
    """host numpy array, torch tensor (host or cuda) or raw int address -> void*"""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(C.c_void_p)
    if hasattr(a, "data_ptr"):
        return C.c_void_p(a.data_ptr())
    return C.c_void_p(int(a))


def _set_svm_knobs(cfg, svm_mode, guard_rel, tc_variant, tc_passes, audit_every, guard_tier2, guard_kernel, sv_table_global):
    """the decision-value switches of a haf_config, shared by GraspSearch and SvmPredictor"""
    cfg.svm_mode = svm_mode
    cfg.guard_rel = guard_rel
    # tc_variant: 0 auto (X-resident CTA pair where eligible), 1 single CTA, 2 streaming CTA pair; tc_passes: 0 = calibrated
    # per model, 1-3 forced; audit_every: None = library default (every 4096th window), 0 = no sample, n = every n-th window
    cfg.reserved[0] = tc_variant | (tc_passes << 4)
    if audit_every is not None:
        cfg.reserved[0] |= 0x100 if audit_every == 0 else (int(audit_every) << 16)
    # guard_tier2: 0 on, 1 off, 2 on + escalate everything (tests); guard_kernel: 0 auto, 1 FP64 tensor cores (DMMA), 2 DFMA
    cfg.reserved[2] = guard_tier2 | (guard_kernel << 2)
    cfg.reserved[3] = sv_table_global   # 1: SV table read from global memory (the > 4096-SV path)


class GraspSearch:
    """One context = one GPU.  Mirrors the reference's per-goal flow: construct once with the three files the
    action server is configured with (server.cpp:218-225), then ``search`` per goal."""

    def __init__(self, features_path, range_path, model_path, grid=56, roll_step_deg=15, roll_max_deg=190,
                 nr_features_without_shaf=302, device=0, emulate_text_roundtrip=True, svm_mode=HAF_SVM_TENSOR_GUARD,
                 guard_rel=0.0, tc_variant=0, guard_tier2=0, sv_table_global=0, tc_passes=0, audit_every=None, bin_variant=0,
                 devices=None, guard_kernel=0, use_graph=False):
        self.L = load_library()
        cfg = haf_config()
        self._keep = [features_path.encode(), range_path.encode(), model_path.encode()]
        cfg.features_path, cfg.range_path, cfg.model_path = self._keep
        cfg.nr_features_without_shaf = nr_features_without_shaf
        cfg.grid, cfg.roll_step_deg, cfg.roll_max_deg = grid, roll_step_deg, roll_max_deg
        cfg.device = device
        cfg.emulate_text_roundtrip = 1 if emulate_text_roundtrip else -1   # 0 would also mean "on" (zeroed config = reference-exact)
        _set_svm_knobs(cfg, svm_mode, guard_rel, tc_variant, tc_passes, audit_every, guard_tier2, guard_kernel, sv_table_global)
        # bin_variant: 0 auto, 1 point-parallel binning only, 2 whole-cloud kernel with scalar loads; bit 4: CUDA graph capture / replay
        cfg.reserved[1] = bin_variant | (16 if use_graph else 0)
        if devices is not None and len(devices) > 1:   # one context driving several GPUs (haf_config.n_devices / devices)
            self._devs = (C.c_int * len(devices))(*devices)
            cfg.n_devices, cfg.devices = len(devices), self._devs
            cfg.device = devices[0]
        self.h = C.c_void_p()
        rc = self.L.haf_create(C.byref(self.h), C.byref(cfg))
        if rc != 0:
            raise HafError(rc, (self.L.haf_last_error(None) or b"").decode())
        self.info = haf_info()
        self.L.haf_get_info(self.h, C.byref(self.info))
        self.G, self.R, self.F, self.D = self.info.grid, self.info.n_rolls, self.info.n_features, self.info.n_dims

    def close(self):
        if getattr(self, "h", None):
            self.L.haf_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc < 0:
            raise HafError(rc, (self.L.haf_last_error(self.h) or b"").decode())
        return rc

    def set_stream(self, cuda_stream_handle: int):
        self._check(self.L.haf_set_stream(self.h, C.c_void_p(cuda_stream_handle)))

    def set_profiling(self, on: bool):
        self._check(self.L.haf_set_profiling(self.h, int(on)))

    def set_debug(self, keep_batch_state: bool):
        """batch calls keep their per-window state for the debug_* accessors (single-pass batches only)"""
        self._check(self.L.haf_set_debug(self.h, int(keep_batch_state)))

    def timing(self) -> haf_timing:
        t = haf_timing()
        self._check(self.L.haf_get_timing(self.h, C.byref(t)))
        return t

    def launch_count(self) -> int:
        return int(self.L.haf_launch_count(self.h))

    def search(self, xyz, requests=None, n_points=None, stride_bytes=None, outputs=True):
        """xyz: numpy float32 [n,3] (host), or a torch CUDA tensor [n,3]/[n,4] (device pointer).  Returns a dict."""
        xyz, reqs, nreq, n, stride, best, per, out = self._search_args(xyz, requests, n_points, stride_bytes, outputs)
        self._check(self.L.haf_search(self.h, _ptr(xyz), n, stride, reqs, nreq, C.byref(best), per,
                                      _ptr(out.get("graspseval")), _ptr(out.get("mask")), _ptr(out.get("heights")),
                                      _ptr(out["per_roll_top"])))
        out["best"] = best
        out["best_per_request"] = list(per)
        return out

    def search_grasps(self, xyz, requests=None, per_roll=False, outputs=False, n_points=None, stride_bytes=None):
        """``search`` plus the grasp poses computed on the device (haf_search_grasps): the dict also carries ``grasp`` (haf_grasp
        of ``best``), ``grasp_per_request`` (list) and, with per_roll, ``grasp_per_roll`` ([n_requests][R] lists; only the
        evaluated rolls are written).  per_roll may also be a ctypes array of n_requests * R haf_grasp records to fill in place."""
        xyz, reqs, nreq, n, stride, best, per, out = self._search_args(xyz, requests, n_points, stride_bytes, outputs)
        grasp = haf_grasp()
        gper = (haf_grasp * nreq)()
        groll = None
        if per_roll is not False and per_roll is not None:
            groll = per_roll if not isinstance(per_roll, bool) else (haf_grasp * (nreq * self.R))()
            if len(groll) != nreq * self.R:
                raise ValueError("per_roll needs n_requests * R = %d records" % (nreq * self.R))
        self._check(self.L.haf_search_grasps(self.h, _ptr(xyz), n, stride, reqs, nreq, C.byref(best), per,
                                             _ptr(out.get("graspseval")), _ptr(out.get("mask")), _ptr(out.get("heights")),
                                             _ptr(out["per_roll_top"]), C.byref(grasp), gper, groll))
        out["best"] = best
        out["best_per_request"] = list(per)
        out["grasp"] = grasp
        out["grasp_per_request"] = list(gper)
        if groll is not None:
            out["grasp_per_roll"] = [list(groll[a * self.R:(a + 1) * self.R]) for a in range(nreq)]
        return out

    def _search_args(self, xyz, requests, n_points, stride_bytes, outputs):
        if requests is None:
            requests = [make_request()]
        if isinstance(requests, haf_request):
            requests = [requests]
        nreq = len(requests)
        reqs = (haf_request * nreq)(*requests)
        if isinstance(xyz, np.ndarray):
            xyz = np.ascontiguousarray(xyz, np.float32)
            n = len(xyz) if n_points is None else n_points
            stride = xyz.strides[0] if stride_bytes is None else stride_bytes
        else:
            n = xyz.shape[0] if n_points is None else n_points
            stride = xyz.stride(0) * 4 if stride_bytes is None else stride_bytes
        best = haf_best()
        per = (haf_best * nreq)()
        out = {}
        G, R = self.G, self.R
        if outputs:
            out["graspseval"] = np.zeros((nreq, R, G, G), np.float32)
            out["mask"] = np.zeros((nreq, R, G, G), np.uint8)
            out["heights"] = np.zeros((nreq, R, G, G), np.float32)
        out["per_roll_top"] = np.full((nreq, R, 3), -1, np.int32)
        return xyz, reqs, nreq, n, stride, best, per, out

    def search_batch_packed(self, xyz_all, point_offsets, request=None):
        """xyz_all: packed float32 [N,3] host array or CUDA tensor; point_offsets: n_clouds+1 ints."""
        rq = request or make_request()
        off = (C.c_size_t * len(point_offsets))(*[int(o) for o in point_offsets])
        n_clouds = len(point_offsets) - 1
        best = (haf_best * n_clouds)()
        if isinstance(xyz_all, np.ndarray):
            xyz_all = np.ascontiguousarray(xyz_all, np.float32)
        self._check(self.L.haf_search_batch_packed(self.h, _ptr(xyz_all), off, n_clouds, C.byref(rq), best))
        return best

    def search_batch_packed_grasps(self, xyz_all, point_offsets, request=None, per_roll=False):
        """``search_batch_packed`` plus one grasp pose per cloud (haf_search_batch_packed_grasps).  Returns a dict: ``best``
        (haf_best array), ``grasp`` (haf_grasp array, one per cloud) and, with per_roll, ``grasp_per_roll`` (haf_grasp array
        [n_clouds * R], evaluated rolls only; per_roll may also be such an array to fill in place)."""
        rq = request or make_request()
        off = (C.c_size_t * len(point_offsets))(*[int(o) for o in point_offsets])
        n_clouds = len(point_offsets) - 1
        best = (haf_best * n_clouds)()
        grasp = (haf_grasp * n_clouds)()
        groll = None
        if per_roll is not False and per_roll is not None:
            groll = per_roll if not isinstance(per_roll, bool) else (haf_grasp * (n_clouds * self.R))()
            if len(groll) != n_clouds * self.R:
                raise ValueError("per_roll needs n_clouds * R = %d records" % (n_clouds * self.R))
        if isinstance(xyz_all, np.ndarray):
            xyz_all = np.ascontiguousarray(xyz_all, np.float32)
        self._check(self.L.haf_search_batch_packed_grasps(self.h, _ptr(xyz_all), off, n_clouds, C.byref(rq), best, grasp, groll))
        out = {"best": best, "grasp": grasp}
        if groll is not None:
            out["grasp_per_roll"] = groll
        return out

    def search_batch_requests(self, xyz_all, point_offsets, requests, request_offsets=None, grasps=True, per_roll=False,
                              per_roll_top=False):
        """Each cloud with its own requests (haf_search_batch_requests): cloud c is searched with
        requests[request_offsets[c]:request_offsets[c + 1]] (None: one request per cloud).  requests: a haf_request array (see
        ``make_requests``) or a list.  Returns a dict like ``search_batch_packed_grasps``: ``best`` and, with grasps, ``grasp`` per
        cloud, plus ``best_per_request``, with grasps ``grasp_per_request``, with per_roll ``grasp_per_roll`` (haf_grasp array
        [n_requests * R], evaluated rolls only) and with per_roll_top ``per_roll_top`` (int32 [n_requests, R, 3])."""
        if not isinstance(requests, C.Array):
            requests = (haf_request * len(requests))(*requests)
        n_clouds = len(point_offsets) - 1
        nreq = len(requests)
        off = (C.c_size_t * len(point_offsets))(*[int(o) for o in point_offsets])
        roff = None if request_offsets is None else (C.c_int * len(request_offsets))(*[int(o) for o in request_offsets])
        best, bpr = (haf_best * n_clouds)(), (haf_best * nreq)()
        grasp = (haf_grasp * n_clouds)() if grasps else None
        gpr = (haf_grasp * nreq)() if grasps else None
        groll = (haf_grasp * (nreq * self.R))() if grasps and per_roll else None
        top = np.full((nreq, self.R, 3), -1, np.int32) if per_roll_top else None
        if isinstance(xyz_all, np.ndarray):
            xyz_all = np.ascontiguousarray(xyz_all, np.float32)
        self._check(self.L.haf_search_batch_requests(self.h, _ptr(xyz_all), off, n_clouds, requests, roff, best, bpr, _ptr(top),
                                                     grasp, gpr, groll))
        out = {"best": best, "best_per_request": bpr}
        if grasps:
            out["grasp"], out["grasp_per_request"] = grasp, gpr
        if groll is not None:
            out["grasp_per_roll"] = groll
        if top is not None:
            out["per_roll_top"] = top
        return out

    def search_batch_candidates(self, xyz_all, point_offsets, requests, request_offsets=None, k=16, per_unit=0, min_distance=0.0,
                                rank_params=None):
        """The k best distinct grasps of every cloud (haf_search_batch_candidates), inputs as ``search_batch_requests``.  Returns a
        dict: ``best`` and ``grasp`` per cloud, ``candidates`` (haf_candidate array [n_clouds * k], cloud c at [c * k, c * k +
        n_candidates[c])) and ``n_candidates`` (int32 [n_clouds]).  rank_params: a haf_rank_params to pass as it is (overrides k,
        per_unit and min_distance)."""
        if not isinstance(requests, C.Array):
            requests = (haf_request * len(requests))(*requests)
        rp = rank_params
        if rp is None:
            rp = haf_rank_params()
            rp.k, rp.per_unit, rp.min_distance = int(k), int(per_unit), float(min_distance)
        n_clouds = len(point_offsets) - 1
        off = (C.c_size_t * len(point_offsets))(*[int(o) for o in point_offsets])
        roff = None if request_offsets is None else (C.c_int * len(request_offsets))(*[int(o) for o in request_offsets])
        best, grasp = (haf_best * n_clouds)(), (haf_grasp * n_clouds)()
        cand = (haf_candidate * (n_clouds * max(int(rp.k), 1)))()
        ncand = np.zeros(n_clouds, np.int32)
        if isinstance(xyz_all, np.ndarray):
            xyz_all = np.ascontiguousarray(xyz_all, np.float32)
        self._check(self.L.haf_search_batch_candidates(self.h, _ptr(xyz_all), off, n_clouds, requests, roff, C.byref(rp), best, grasp,
                                                       cand, _ptr(ncand)))
        return {"best": best, "grasp": grasp, "candidates": cand, "n_candidates": ncand}

    def search_candidates(self, xyz, requests=None, k=16, per_unit=0, min_distance=0.0):
        """``search_batch_candidates`` for one cloud (packed float32 [n, 3], host array or CUDA tensor) and its requests."""
        if requests is None:
            requests = [make_request()]
        if isinstance(requests, haf_request):
            requests = [requests]
        return self.search_batch_candidates(xyz, [0, len(xyz)], requests, [0, len(requests)], k=k, per_unit=per_unit,
                                            min_distance=min_distance)

    def debug_unit_params(self, n_units, poses=True):
        """unit parameters of the last search (haf_debug_unit_params): (M [U, 16], mask [U, 10], Minv [U, 16] or None)"""
        M, mask = np.zeros((n_units, 16), np.float32), np.zeros((n_units, 10), np.float32)
        Minv = np.zeros((n_units, 16), np.float32) if poses else None
        U = self._check(self.L.haf_debug_unit_params(self.h, _ptr(M), _ptr(mask), _ptr(Minv), n_units))
        return M[:U], mask[:U], (Minv[:U] if poses else None)

    def debug_chunk_copy_waits(self):
        """chunks of the last search (haf_debug_chunk_copy_waits): int32 [n, 10] = first cloud, end cloud, stream set, copy piece
        waited for (-1: device input), end cloud of that piece, binning kernel (0 point-parallel, 1 whole-cloud with 16-byte loads,
        2 whole-cloud with scalar loads), unit groups, units per group, slices (whole-cloud kernel; 0 otherwise), integral image
        (0 one kernel, 1 row + column passes)"""
        t = self.timing()
        out = np.zeros((max(int(t.n_chunks), 1), CHUNK_RECORD), np.int32)
        n = self._check(self.L.haf_debug_chunk_copy_waits(self.h, _ptr(out), len(out)))
        return out[:n]

    def pack_best_records(self, best, out):
        """haf_best array of a batch -> int32 [n, 8] records (topval, row, col, roll, tilt, approach_idx, n_windows, rolls_done)
        written by the library into `out` (numpy array or pinned torch tensor)"""
        self._check(self.L.haf_pack_best_records(best, len(best), _ptr(out)))
        return out

    def search_batch(self, clouds, request=None):
        """clouds: list of float32 [n_i,3] host arrays or CUDA tensors."""
        rq = request or make_request()
        n_clouds = len(clouds)
        keep = [np.ascontiguousarray(c, np.float32) if isinstance(c, np.ndarray) else c for c in clouds]
        ptrs = (C.c_void_p * n_clouds)(*[_ptr(c) for c in keep])
        npts = (C.c_size_t * n_clouds)(*[int(c.shape[0]) for c in keep])
        best = (haf_best * n_clouds)()
        self._check(self.L.haf_search_batch(self.h, ptrs, npts, n_clouds, C.byref(rq), best))
        return best

    # ---- parity / inspection -----------------------------------------------------------
    # ---- PCD / PointCloud2 ingest on the device (SURVEY 8f-2) ----
    def pcd_decode(self, file_bytes: bytes):
        """the bytes of a .pcd file -> (device pointer of packed xyz, n_points); the buffer belongs to the context"""
        buf = np.frombuffer(file_bytes, np.uint8)
        d = C.c_void_p()
        n = C.c_size_t()
        self._check(self.L.haf_pcd_decode(self.h, _ptr(buf), len(buf), C.byref(d), C.byref(n)))
        return (d.value or 0), n.value

    def pcd_decode_to_host(self, file_bytes: bytes) -> np.ndarray:
        """decode on the device, then copy the packed xyz back (parity tests)"""
        _, n = self.pcd_decode(file_bytes)
        return self.debug_pcd_xyz(n)

    def debug_pcd_xyz(self, n_points: int) -> np.ndarray:
        out = np.zeros((n_points, 3), np.float32)
        if n_points:
            self._check(self.L.haf_debug_pcd_xyz(self.h, _ptr(out), n_points))
        return out

    def pointcloud2_to_xyz(self, data, n_points, point_step, off_x=0, off_y=4, off_z=8):
        d = C.c_void_p()
        self._check(self.L.haf_pointcloud2_to_xyz(self.h, _ptr(data), n_points, point_step, off_x, off_y, off_z, C.byref(d)))
        return d.value or 0

    def search_pcd(self, file_bytes: bytes, requests=None):
        """haf_search_pcd: decode on the device + search; returns the same dict as search (no per-roll grids)"""
        buf = np.frombuffer(file_bytes, np.uint8)
        reqs = requests or [make_request()]
        arr = (haf_request * len(reqs))(*reqs)
        best = haf_best()
        per = (haf_best * len(reqs))()
        top = np.zeros((len(reqs), self.R, 3), np.int32)
        self._check(self.L.haf_search_pcd(self.h, _ptr(buf), len(buf), arr, len(reqs), C.byref(best), per, None, None, None, _ptr(top)))
        return {"best": best, "best_per_request": list(per), "per_roll_top": top}

    # ---- batches of PCD files / PointCloud2 buffers: one decode for all clouds ----
    @staticmethod
    def _pcd_batch(files):
        """files: a list of bytes-like objects (concatenated here once), or (data, file_offsets) with data a contiguous uint8
        numpy array or host torch tensor (pinned or not) that already holds the files back to back"""
        if isinstance(files, tuple):
            data, offs = files
            offs = [int(o) for o in offs]
            if isinstance(data, np.ndarray):
                data = np.ascontiguousarray(data, np.uint8)
        else:
            lens = [len(memoryview(f).cast("B")) for f in files]
            offs = [0] + list(np.cumsum(lens, dtype=np.int64).tolist())
            data = np.frombuffer(b"".join(files), np.uint8) if files else np.zeros(0, np.uint8)
        return data, (C.c_size_t * len(offs))(*offs), len(offs) - 1

    def pcd_decode_batch(self, files):
        """PCD files -> (device pointer of the packed xyz of every cloud, point_offsets int64 [n_files + 1]) (haf_pcd_decode_batch);
        the buffer belongs to the context.  files: see _pcd_batch."""
        data, off, n = self._pcd_batch(files)
        d = C.c_void_p()
        po = (C.c_size_t * (n + 1))()
        self._check(self.L.haf_pcd_decode_batch(self.h, _ptr(data), off, n, C.byref(d), po))
        return (d.value or 0), np.array(po[:], np.int64)

    def pcd_decode_batch_to_host(self, files):
        """decode a batch on the device, then copy it back: a list of float32 [n_i, 3] arrays"""
        _, po = self.pcd_decode_batch(files)
        xyz = self.debug_pcd_xyz(int(po[-1]))
        return [xyz[po[f]:po[f + 1]] for f in range(len(po) - 1)]

    def search_batch_pcd(self, files, requests=None, request_offsets=None, grasps=True, per_roll=False, per_roll_top=False):
        """haf_search_batch_pcd: decode every file on the device, then ``search_batch_requests`` on the clouds.  requests=None:
        ``make_request()`` for every file.  Returns the dict of ``search_batch_requests`` plus ``point_offsets``."""
        data, off, n = self._pcd_batch(files)
        if requests is None:
            requests = make_requests(n)
        elif not isinstance(requests, C.Array):
            requests = (haf_request * len(requests))(*requests)
        nreq = len(requests)
        roff = None if request_offsets is None else (C.c_int * len(request_offsets))(*[int(o) for o in request_offsets])
        best, bpr = (haf_best * n)(), (haf_best * nreq)()
        grasp = (haf_grasp * n)() if grasps else None
        gpr = (haf_grasp * nreq)() if grasps else None
        groll = (haf_grasp * (nreq * self.R))() if grasps and per_roll else None
        top = np.full((nreq, self.R, 3), -1, np.int32) if per_roll_top else None
        self._check(self.L.haf_search_batch_pcd(self.h, _ptr(data), off, n, requests, roff, best, bpr, _ptr(top), grasp, gpr, groll))
        out = {"best": best, "best_per_request": bpr}
        if grasps:
            out["grasp"], out["grasp_per_request"] = grasp, gpr
        if groll is not None:
            out["grasp_per_roll"] = groll
        if top is not None:
            out["per_roll_top"] = top
        out["point_offsets"] = self._pcd_point_offsets(data, off, n)
        return out

    @staticmethod
    def _pcd_point_offsets(data, off, n):
        """cumulative POINTS of the headers (what the decode reports as point_offsets)"""
        from . import pcd
        raw = data.numpy() if hasattr(data, "numpy") else data
        po = [0]
        for f in range(n):
            po.append(po[-1] + pcd.header_points(raw[off[f]:off[f + 1]]))
        return np.array(po, np.int64)

    def pointcloud2_batch_to_xyz(self, data, byte_offsets, layouts):
        """haf_pointcloud2_batch_to_xyz: data (host array or CUDA tensor) holds the clouds' records back to back, cloud c =
        bytes [byte_offsets[c], byte_offsets[c + 1]); layouts [n_clouds][4] = (point_step, off_x, off_y, off_z).  Returns
        (device pointer of the packed xyz, point_offsets int64 [n_clouds + 1])."""
        n = len(byte_offsets) - 1
        off = (C.c_size_t * (n + 1))(*[int(o) for o in byte_offsets])
        lay = np.ascontiguousarray(np.asarray(layouts, np.int32).reshape(n, 4))
        d = C.c_void_p()
        po = (C.c_size_t * (n + 1))()
        self._check(self.L.haf_pointcloud2_batch_to_xyz(self.h, _ptr(data), off, n, lay.ctypes.data_as(C.POINTER(C.c_int)), C.byref(d), po))
        return (d.value or 0), np.array(po[:], np.int64)

    # ---- batches of depth images: back-projection and the camera -> base transform on the device ----
    @staticmethod
    def _depth_batch(images, intrinsics, poses, depth_scale):
        """(data, byte_offsets, haf_depth_image array, n) of a batch.  images: a list of 2-D uint16 / float32 numpy arrays (row
        stride may exceed the row: the step keeps it), one (N, H, W) numpy array or torch tensor (host, pinned or not, or CUDA; made
        contiguous), or (data, byte_offsets, records) passed as they are.  intrinsics: (fx, fy, cx, cy) or one per image; poses:
        None, one 4x4 camera -> base matrix or one per image (None entries: no pose); depth_scale: one value or one per image."""
        if isinstance(images, tuple):
            data, offs, recs = images
            if not isinstance(recs, C.Array):
                recs = (haf_depth_image * len(recs))(*recs)
            return data, (C.c_size_t * len(offs))(*[int(o) for o in offs]), recs, len(recs)
        if isinstance(images, list):
            n = len(images)
            shapes, encs, steps, bufs = [], [], [], []
            for im in images:
                if im.ndim != 2 or im.dtype not in (np.uint16, np.float32):
                    raise ValueError("a depth image is a 2-D uint16 or float32 array")
                h, w = im.shape
                isz = im.itemsize
                step = im.strides[0] if (im.strides[1] == isz and im.strides[0] >= w * isz) else w * isz
                rows = np.zeros((h, step), np.uint8)
                if h and w:
                    rows[:, :w * isz] = np.ascontiguousarray(im).astype(im.dtype.newbyteorder("<"), copy=False).view(np.uint8).reshape(h, w * isz)
                shapes.append((h, w)); encs.append(HAF_DEPTH_U16 if im.dtype == np.uint16 else HAF_DEPTH_F32); steps.append(step)
                bufs.append(rows.reshape(-1))
            data = np.concatenate(bufs) if bufs else np.zeros(0, np.uint8)
            offs = [0] + np.cumsum([len(b) for b in bufs], dtype=np.int64).tolist()
        else:
            if len(images.shape) != 3:
                raise ValueError("a stack of depth images is (N, H, W)")
            n, h, w = (int(v) for v in images.shape)
            if isinstance(images, np.ndarray):
                if images.dtype not in (np.uint16, np.float32):
                    raise ValueError("depth images are uint16 or float32")
                images = np.ascontiguousarray(images)
                isz, u16 = images.itemsize, images.dtype == np.uint16
            else:
                import torch
                if images.dtype not in (torch.uint16, torch.float32, torch.int16):
                    raise ValueError("depth images are uint16 or float32")
                images = images.contiguous()
                isz, u16 = images.element_size(), images.dtype != torch.float32
            data, row = images, w * isz
            shapes, encs, steps = [(h, w)] * n, [HAF_DEPTH_U16 if u16 else HAF_DEPTH_F32] * n, [row] * n
            offs = [k * h * row for k in range(n + 1)]
        recs = (haf_depth_image * n)()
        names = [f[0] for f in haf_depth_image._fields_]
        rec = np.frombuffer(recs, np.dtype({"names": names,
                                            "formats": [np.int32] * 4 + [np.int64] + [np.float64] * 4 + [np.float32, (np.float32, 16), (np.int32, 3)],
                                            "offsets": [getattr(haf_depth_image, f).offset for f in names],
                                            "itemsize": C.sizeof(haf_depth_image)}))
        if n:
            rec["height"], rec["width"] = np.asarray(shapes, np.int32).reshape(n, 2).T
            rec["encoding"], rec["step"] = encs, steps
            K = np.broadcast_to(np.asarray(intrinsics, np.float64), (n, 4))
            rec["fx"], rec["fy"], rec["cx"], rec["cy"] = K.T
            rec["depth_scale"] = np.broadcast_to(np.asarray(depth_scale, np.float32), (n,))
            if poses is not None and not isinstance(poses, (list, tuple)) and np.asarray(poses).ndim == 2:
                rec["has_pose"], rec["camera_to_base"] = 1, np.asarray(poses, np.float32).reshape(16)
            elif poses is not None:
                for i, m in enumerate(poses):
                    if m is not None:
                        rec["has_pose"][i], rec["camera_to_base"][i] = 1, np.asarray(m, np.float32).reshape(16)
        return data, (C.c_size_t * len(offs))(*[int(o) for o in offs]), recs, n

    def depth_to_xyz_batch(self, images, intrinsics=None, poses=None, depth_scale=0.0):
        """haf_depth_to_xyz_batch: depth images (see _depth_batch) -> (device pointer of the packed xyz of every cloud, point_offsets
        int64 [n_images + 1]); image i gives width x height points in row-major pixel order, invalid pixels as NaN points.  The buffer
        belongs to the context (valid until the next ingest call)."""
        data, off, recs, n = self._depth_batch(images, intrinsics, poses, depth_scale)
        d = C.c_void_p()
        po = (C.c_size_t * (n + 1))()
        self._check(self.L.haf_depth_to_xyz_batch(self.h, _ptr(data), off, n, recs, C.byref(d), po))
        return (d.value or 0), np.array(po[:], np.int64)

    def depth_to_xyz_batch_to_host(self, images, intrinsics=None, poses=None, depth_scale=0.0):
        """back-project on the device, then copy back: a list of float32 [width * height, 3] arrays"""
        _, po = self.depth_to_xyz_batch(images, intrinsics, poses, depth_scale)
        xyz = self.debug_pcd_xyz(int(po[-1]))
        return [xyz[po[i]:po[i + 1]] for i in range(len(po) - 1)]

    def search_batch_depth(self, images, intrinsics=None, poses=None, depth_scale=0.0, requests=None, request_offsets=None, grasps=True,
                           per_roll=False, per_roll_top=False):
        """haf_search_batch_depth: back-project every image on the device, then ``search_batch_requests`` on the clouds.
        requests=None: ``make_request()`` for every image.  Returns the dict of ``search_batch_pcd``."""
        data, off, recs, n = self._depth_batch(images, intrinsics, poses, depth_scale)
        if requests is None:
            requests = make_requests(n)
        elif not isinstance(requests, C.Array):
            requests = (haf_request * len(requests))(*requests)
        nreq = len(requests)
        roff = None if request_offsets is None else (C.c_int * len(request_offsets))(*[int(o) for o in request_offsets])
        best, bpr = (haf_best * n)(), (haf_best * nreq)()
        grasp = (haf_grasp * n)() if grasps else None
        gpr = (haf_grasp * nreq)() if grasps else None
        groll = (haf_grasp * (nreq * self.R))() if grasps and per_roll else None
        top = np.full((nreq, self.R, 3), -1, np.int32) if per_roll_top else None
        self._check(self.L.haf_search_batch_depth(self.h, _ptr(data), off, n, recs, requests, roff, best, bpr, _ptr(top), grasp, gpr, groll))
        out = {"best": best, "best_per_request": bpr}
        if grasps:
            out["grasp"], out["grasp_per_request"] = grasp, gpr
        if groll is not None:
            out["grasp_per_roll"] = groll
        if top is not None:
            out["per_roll_top"] = top
        out["point_offsets"] = np.cumsum([0] + [recs[i].width * recs[i].height for i in range(n)]).astype(np.int64)
        return out

    def debug_windows(self):
        W = self._check(self.L.haf_debug_window_count(self.h))
        a = np.zeros((max(W, 1), 2), np.int32)
        self._check(self.L.haf_debug_windows(self.h, _ptr(a), W))
        return a[:W]

    def debug_features(self, raw=True, scaled=True):
        W = self._check(self.L.haf_debug_window_count(self.h))
        r = np.zeros((max(W, 1), self.F), np.float32) if raw else None
        s = np.zeros((max(W, 1), self.D), np.float64) if scaled else None
        self._check(self.L.haf_debug_features(self.h, _ptr(r), _ptr(s), W))
        return (r[:W] if raw else None), (s[:W] if scaled else None)

    def debug_tensor_inputs(self):
        W = self._check(self.L.haf_debug_window_count(self.h))
        x = np.zeros((max(W, 1), self.D), np.float32)
        self._check(self.L.haf_debug_tensor_inputs(self.h, _ptr(x), W))
        return x[:W]

    def debug_decisions(self):
        W = self._check(self.L.haf_debug_window_count(self.h))
        d = np.zeros(max(W, 1), np.float64)
        lab = np.zeros(max(W, 1), np.int32)
        g = np.zeros(max(W, 1), np.uint8)
        self._check(self.L.haf_debug_decisions(self.h, _ptr(d), _ptr(lab), _ptr(g), W))
        return d[:W], lab[:W], g[:W]

    def debug_heights(self, n_units):
        """decoded height grids [n_units, G, G] of the last search (haf_debug_heights); only active units are defined"""
        a = np.zeros((n_units, self.G, self.G), np.float32)
        self._check(self.L.haf_debug_heights(self.h, _ptr(a), a.size))
        return a

    def debug_integral(self, n_units):
        a = np.zeros((n_units, self.G + 1, self.G + 1), np.float32)
        self._check(self.L.haf_debug_integral(self.h, _ptr(a), a.size))
        return a

    def debug_cell_indices(self, xyz, request, roll):
        xyz = np.ascontiguousarray(xyz, np.float32)
        out = np.zeros(len(xyz), np.int32)
        self._check(self.L.haf_debug_cell_indices(self.h, _ptr(xyz), len(xyz), xyz.strides[0], C.byref(request), roll, _ptr(out)))
        return out

    def debug_tc_probe(self, n_ctas=148):
        out = np.zeros((n_ctas, 16), np.uint64)
        self._check(self.L.haf_debug_tc_probe(self.h, _ptr(out), n_ctas))
        return out

    def debug_text_roundtrip(self, in4=None, in6=None):
        in4 = np.ascontiguousarray(in4 if in4 is not None else np.zeros(0), np.float32)
        in6 = np.ascontiguousarray(in6 if in6 is not None else np.zeros(0), np.float64)
        o4, o6 = np.zeros(len(in4), np.float64), np.zeros(len(in6), np.float64)
        self._check(self.L.haf_debug_text_roundtrip(self.h, _ptr(in4), len(in4), _ptr(o4), _ptr(in6), len(in6), _ptr(o6)))
        return o4, o6


def build_transform(request: haf_request, roll: int, roll_step_deg: int = 15) -> np.ndarray:
    L = load_library()
    M = (C.c_float * 16)()
    L.haf_build_transform(C.byref(request), roll, roll_step_deg, M)
    return np.array(M, np.float32)


# ---- libsvm front ends (include/hafgpu.h, SURVEY 8f-3) ---------------------------------------------------------
def _csr(rows_or_dense):
    """dense [n][D] array (zeros = absent) or (row_ptr, index, value) -> CSR arrays with libsvm's 1-based indices"""
    if isinstance(rows_or_dense, tuple):
        rp, idx, val = rows_or_dense
        return (np.ascontiguousarray(rp, np.int64), np.ascontiguousarray(idx, np.int32), np.ascontiguousarray(val, np.float64))
    x = np.asarray(rows_or_dense, np.float64)
    nz = x != 0
    rp = np.zeros(len(x) + 1, np.int64)
    rp[1:] = np.cumsum(nz.sum(1))
    r, c = np.nonzero(nz)
    return rp, (c + 1).astype(np.int32), np.ascontiguousarray(x[r, c])


class SvmPredictor:
    """svm_predict on the GPU for a libsvm text model (C-SVC, RBF, two classes): what svm-predict-b200 binds."""

    def __init__(self, model_path, device=0, svm_mode=HAF_SVM_TENSOR_GUARD, min_dims=0, guard_rel=0.0, tc_variant=0, tc_passes=0,
                 sv_table_global=0, guard_tier2=0, guard_kernel=0, audit_every=None):
        """the keyword arguments after min_dims mean what they mean for GraspSearch"""
        self.L = load_library()
        self.h = C.c_void_p()
        cfg = haf_config()
        self._model = model_path.encode()
        cfg.model_path = self._model
        cfg.device = device
        _set_svm_knobs(cfg, svm_mode, guard_rel, tc_variant, tc_passes, audit_every, guard_tier2, guard_kernel, sv_table_global)
        rc = self.L.haf_svm_create_config(C.byref(self.h), C.byref(cfg), min_dims)
        if rc != 0:
            raise HafError(rc, (self.L.haf_last_error(None) or b"").decode())
        self.info = haf_info()
        self.L.haf_get_info(self.h, C.byref(self.info))

    def predict(self, rows, want_dec=True):
        """(labels [n], decision values [n] or None); afterwards info.reserved[2] / [3] name the contraction kernel that ran
        and its support-vector split"""
        rp, idx, val = _csr(rows)
        n = len(rp) - 1
        labels = np.zeros(max(n, 1), np.float64)
        dec = np.zeros(max(n, 1), np.float64) if want_dec else None
        rc = self.L.haf_svm_predict(self.h, _ptr(rp), _ptr(idx), _ptr(val), n, _ptr(labels), _ptr(dec))
        if rc != 0:
            raise HafError(rc, (self.L.haf_last_error(self.h) or b"").decode())
        self.L.haf_get_info(self.h, C.byref(self.info))
        return labels[:n], (dec[:n] if want_dec else None)

    def check_probability_model(self):
        return bool(self.L.haf_svm_check_probability_model(self.h))

    def predict_probability(self, rows):
        """svm-predict -b 1: (labels [n], prob_estimates [n][2] in the order of the model's labels)"""
        rp, idx, val = _csr(rows)
        n = len(rp) - 1
        labels = np.zeros(max(n, 1), np.float64)
        probs = np.zeros((max(n, 1), 2), np.float64)
        rc = self.L.haf_svm_predict_probability(self.h, _ptr(rp), _ptr(idx), _ptr(val), n, _ptr(labels), _ptr(probs))
        if rc != 0:
            raise HafError(rc, (self.L.haf_last_error(self.h) or b"").decode())
        self.L.haf_get_info(self.h, C.byref(self.info))
        return labels[:n], probs[:n]

    def timing(self):
        t = haf_timing()
        self.L.haf_get_timing(self.h, C.byref(t))
        return t

    def close(self):
        if self.h:
            self.L.haf_svm_destroy(self.h)
            self.h = C.c_void_p()


def scale_minmax(rows, max_index, fmin=None, fmax=None, device=0):
    """svm-scale pass 2 on the device; returns (fmin, fmax) arrays of max_index + 1 entries (entry 0 unused)."""
    L = load_library()
    rp, idx, val = _csr(rows)
    fmin = np.full(max_index + 1, np.finfo(np.float64).max) if fmin is None else np.ascontiguousarray(fmin, np.float64)
    fmax = np.full(max_index + 1, -np.finfo(np.float64).max) if fmax is None else np.ascontiguousarray(fmax, np.float64)
    rc = L.haf_scale_minmax(device, _ptr(rp), _ptr(idx), _ptr(val), len(rp) - 1, max_index, _ptr(fmin), _ptr(fmax))
    if rc != 0:
        raise HafError(rc, (L.haf_last_error(None) or b"").decode())
    return fmin, fmax


def scale_apply(rows, max_index, fmin, fmax, lower=-1.0, upper=1.0, device=0):
    """svm-scale pass 3 on the device: dense [n][max_index] scaled values (0 = not printed)."""
    L = load_library()
    rp, idx, val = _csr(rows)
    out = np.zeros((len(rp) - 1, max_index), np.float64)
    rc = L.haf_scale_apply(device, _ptr(rp), _ptr(idx), _ptr(val), len(rp) - 1, max_index, _ptr(np.ascontiguousarray(fmin, np.float64)),
                           _ptr(np.ascontiguousarray(fmax, np.float64)), lower, upper, _ptr(out))
    if rc != 0:
        raise HafError(rc, (L.haf_last_error(None) or b"").decode())
    return out
