"""_capi.py -- ctypes binding of libadas_b200.so (the C ABI declared in include/adas_b200.h).

The product path has no CPU fallback: if the shared library is missing or there is no sm_100
device, the calls raise.  Errors returned by the library become Python `Exception`s, mirroring
the reference's error style (coreEngine.py:12-14,20,26).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libadas_b200.so")

_lib = None

# every symbol include/adas_b200.h declares (checked by tests/test_capi_symbols.py)
SYMBOLS = [
    "adas_last_error", "adas_version", "adas_launch_count", "adas_engine_create", "adas_engine_destroy",
    "adas_engine_model_kind", "adas_engine_meta", "adas_engine_input_shape", "adas_engine_num_outputs", "adas_engine_output_shape",
    "adas_engine_infer", "adas_engine_infer_dev", "adas_yolo_detect", "adas_yolo_postprocess", "adas_yolo_preprocess",
    "adas_ufld_detect", "adas_ufld_postprocess", "adas_ufld_v1_postprocess", "adas_lane_geometry", "adas_ufld_lane_geometry", "adas_warp_perspective", "adas_engine_warp_perspective", "adas_ufld_preprocess", "adas_iou_cost", "adas_lap", "adas_associate",
    "adas_engine_stream", "adas_engine_num_buffers", "adas_engine_buffer_info", "adas_engine_write_buffer", "adas_engine_read_buffer",
    "adas_engine_run", "adas_engine_event_record", "adas_event_elapsed_ms", "adas_engine_time_ops", "adas_engine_num_steps", "adas_engine_time_step", "adas_engine_step_tiles", "adas_detect_pair",
    "adas_comm_unique_id", "adas_comm_create", "adas_comm_destroy", "adas_comm_all_gather", "adas_comm_sync", "adas_comm_read", "adas_comm_info",
    "adas_tracker_create", "adas_tracker_destroy", "adas_tracker_reset", "adas_tracker_update", "adas_tracker_update_batch", "adas_tracker_get", "adas_tracker_count", "adas_tracker_stats",
]


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise Exception(
                f"libadas_b200.so not built ({LIB_PATH}); run `python -c 'import __graft_entry__ as g; g.build()'`. "
                "There is no CPU fallback for the B200 path.")
        _lib = C.CDLL(LIB_PATH)
        _lib.adas_last_error.restype = C.c_char_p
        _lib.adas_launch_count.restype = C.c_int64
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        raise Exception(lib().adas_last_error().decode("utf-8", "replace"))


def launch_count() -> int:
    return int(lib().adas_launch_count())


def _p(a: np.ndarray, typ):
    return a.ctypes.data_as(C.POINTER(typ))


def as_c(a, dtype) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=dtype)


class TrackRec(C.Structure):
    _fields_ = [("track_id", C.c_int32), ("state", C.c_int32), ("is_activated", C.c_int32), ("class_id", C.c_int32),
                ("start_frame", C.c_int32), ("frame_id", C.c_int32), ("tracklet_len", C.c_int32), ("pad", C.c_int32),
                ("score", C.c_double), ("tlwh", C.c_double * 4), ("mean", C.c_double * 8), ("det_tlbr", C.c_double * 4), ("traj_frame", C.c_int32), ("pad2", C.c_int32)]


TRACK_DTYPE = np.dtype([("track_id", "<i4"), ("state", "<i4"), ("is_activated", "<i4"), ("class_id", "<i4"), ("start_frame", "<i4"),
                        ("frame_id", "<i4"), ("tracklet_len", "<i4"), ("pad", "<i4"), ("score", "<f8"), ("tlwh", "<f8", (4,)), ("mean", "<f8", (8,)), ("det_tlbr", "<f8", (4,)), ("traj_frame", "<i4"), ("pad2", "<i4")])
assert TRACK_DTYPE.itemsize == C.sizeof(TrackRec)


class NativeTracker:
    """Owns one adas_tracker handle (native ByteTrack; association stages on the device)."""
    MAX_OUT = 1024

    def __init__(self, device=0, track_thresh=0.5, track_buffer=30, match_thresh=0.8, frame_rate=30):
        self._h = C.c_void_p()
        check(lib().adas_tracker_create(int(device), C.c_double(track_thresh), int(track_buffer), C.c_double(match_thresh), int(frame_rate),
                                        C.byref(self._h)))
        self._out = np.zeros(self.MAX_OUT, TRACK_DTYPE)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            lib().adas_tracker_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self):
        check(lib().adas_tracker_reset(self._h))

    def update(self, boxes_xyxy, scores, class_ids) -> np.ndarray:
        b = as_c(np.asarray(boxes_xyxy, np.float64).reshape(-1, 4), np.float64)
        s = as_c(scores, np.float64)
        c = as_c(class_ids, np.int32)
        n = C.c_int()
        check(lib().adas_tracker_update(self._h, int(b.shape[0]), _p(b, C.c_double), _p(s, C.c_double), _p(c, C.c_int32), self.MAX_OUT,
                                        self._out.ctypes.data_as(C.c_void_p), C.byref(n)))
        return self._out[:min(n.value, self.MAX_OUT)].copy()

    def stats(self):
        """{frames, total_ms, wait_ms, launches} of update_batch since creation (wait_ms = launch -> result of the association kernel)."""
        o = (C.c_double * 4)()
        check(lib().adas_tracker_stats(self._h, o))
        return {"frames": int(o[0]), "total_ms": float(o[1]), "wait_ms": float(o[2]), "launches": int(o[3])}

    def update_batch(self, counts, boxes_xyxy, scores, class_ids, max_out: int = 256):
        """All frames of a step in one library call -> list (per frame) of TRACK_DTYPE record arrays."""
        cnt = as_c(counts, np.int32)
        nf = int(cnt.shape[0])
        b = as_c(np.asarray(boxes_xyxy, np.float64).reshape(-1, 4), np.float64)
        s = as_c(scores, np.float64)
        c = as_c(class_ids, np.int32)
        out = np.zeros((nf, max_out), TRACK_DTYPE)
        n_out = np.zeros(nf, np.int32)
        check(lib().adas_tracker_update_batch(self._h, nf, _p(cnt, C.c_int32), _p(b, C.c_double), _p(s, C.c_double), _p(c, C.c_int32), int(max_out),
                                              out.ctypes.data_as(C.c_void_p), _p(n_out, C.c_int32)))
        if int(n_out.max(initial=0)) > max_out:          # rare: more live tracks than the caller-sized output rows; redo nothing, tell the caller
            raise Exception(f"adas_tracker_update_batch: {int(n_out.max())} tracks exceed max_out {max_out}")
        return [out[f, :int(n_out[f])] for f in range(nf)]

    def get(self, which: int) -> np.ndarray:
        n = C.c_int()
        check(lib().adas_tracker_get(self._h, which, self.MAX_OUT, self._out.ctypes.data_as(C.c_void_p), C.byref(n)))
        return self._out[:min(n.value, self.MAX_OUT)].copy()

    @staticmethod
    def count() -> int:
        return int(lib().adas_tracker_count())


class Engine:
    """Owns one adas_engine handle (one plan on one device with one private stream)."""

    def __init__(self, plan_path: str, device: int = 0, max_batch: int = 1, conv_impl: int = 0):
        self._h = C.c_void_p()
        check(lib().adas_engine_create(plan_path.encode(), int(device), int(max_batch), int(conv_impl), C.byref(self._h)))
        self.device, self.max_batch = device, max_batch
        k = C.c_int()
        check(lib().adas_engine_model_kind(self._h, C.byref(k)))
        self.model_kind = k.value
        self.meta = []
        for i in range(16):
            check(lib().adas_engine_meta(self._h, i, C.byref(k)))
            self.meta.append(int(k.value))
        s = (C.c_int64 * 4)()
        check(lib().adas_engine_input_shape(self._h, s))
        self.input_shape = [int(v) for v in s]
        n = C.c_int()
        check(lib().adas_engine_num_outputs(self._h, C.byref(n)))
        self.output_shapes = []
        for i in range(n.value):
            r = C.c_int()
            check(lib().adas_engine_output_shape(self._h, i, s, C.byref(r)))
            self.output_shapes.append([int(v) for v in s][: r.value])

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h:
            lib().adas_engine_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- test hooks -------------------------------------------------------------------------
    def buffer_info(self, idx: int):
        info = (C.c_int64 * 5)()
        check(lib().adas_engine_buffer_info(self._h, idx, info))
        return dict(rows_per_img=int(info[0]), C=int(info[1]), dtype=np.float32 if info[2] == 1 else np.float16, H=int(info[3]), W=int(info[4]))

    def write_buffer(self, idx: int, arr: np.ndarray) -> None:
        arr = np.ascontiguousarray(arr)
        check(lib().adas_engine_write_buffer(self._h, idx, arr.ctypes.data_as(C.c_void_p), C.c_int64(arr.nbytes)))

    def read_buffer(self, idx: int, batch: int) -> np.ndarray:
        bi = self.buffer_info(idx)
        out = np.empty((batch * bi["rows_per_img"], bi["C"]), bi["dtype"])
        check(lib().adas_engine_read_buffer(self._h, idx, out.ctypes.data_as(C.c_void_p), C.c_int64(out.nbytes)))
        return out

    def run(self, batch: int) -> None:
        check(lib().adas_engine_run(self._h, batch))

    # ---- timing hooks ------------------------------------------------------------------------
    def event_record(self, slot: int) -> None:
        check(lib().adas_engine_event_record(self._h, slot))

    def elapsed_ms(self, slot_a: int, other: "Engine", slot_b: int) -> float:
        ms = C.c_float()
        check(lib().adas_event_elapsed_ms(self._h, slot_a, other._h, slot_b, C.byref(ms)))
        return float(ms.value)

    def time_ops(self, batch: int, type_mask: int, iters: int):
        ms, n = C.c_float(), C.c_int()
        check(lib().adas_engine_time_ops(self._h, batch, C.c_uint(type_mask), iters, C.byref(ms), C.byref(n)))
        return float(ms.value), int(n.value)

    def num_steps(self, batch: int) -> int:
        n = C.c_int()
        check(lib().adas_engine_num_steps(self._h, batch, C.byref(n)))
        return int(n.value)

    def time_step(self, batch: int, step: int, iters: int):
        """(ms per launch, plan op type, description) of one launch of the plan replayed alone."""
        ms, t = C.c_float(), C.c_int()
        buf = C.create_string_buffer(256)
        check(lib().adas_engine_time_step(self._h, batch, step, iters, C.byref(ms), C.byref(t), buf, 256))
        return float(ms.value), int(t.value), buf.value.decode()

    def step_tiles(self, batch: int, step: int):
        """([(BN, MT), ...], chosen): the tiles the tcgen05 GEMM of launch `step` could have run with at `batch`, in cost-model order,
        and the index of the one it runs.  ([], -1) for a step that is not a tcgen05 GEMM."""
        bn, mt = (C.c_int * 16)(), (C.c_int * 16)()
        n, chosen = C.c_int(), C.c_int()
        check(lib().adas_engine_step_tiles(self._h, batch, step, 16, bn, mt, C.byref(n), C.byref(chosen)))
        assert n.value <= 16
        return [(int(bn[i]), int(mt[i])) for i in range(n.value)], int(chosen.value)

    # engine_inference: fp32 NCHW host -> list of fp32 host arrays
    def infer(self, x: np.ndarray):
        x = as_c(x, np.float32)
        batch = int(x.shape[0])
        outs = [np.empty([batch] + s[1:], np.float32) for s in self.output_shapes]
        arr = (C.POINTER(C.c_float) * len(outs))(*[_p(o, C.c_float) for o in outs])
        check(lib().adas_engine_infer(self._h, _p(x, C.c_float), batch, arr))
        return outs

    def infer_dev(self, x_ptr: int, batch: int, out_ptrs):
        arr = (C.POINTER(C.c_float) * len(out_ptrs))(*[C.cast(C.c_void_p(p), C.POINTER(C.c_float)) for p in out_ptrs])
        check(lib().adas_engine_infer_dev(self._h, C.cast(C.c_void_p(x_ptr), C.POINTER(C.c_float)), batch, arr))

    def yolo_detect(self, frames, box_score: float, nms_iou: float, max_det: int = 1024, on_device: bool = False, shape=None):
        """frames: uint8 [B,H,W,3] numpy (host) or (device pointer, (B,H,W)) when on_device."""
        if on_device:
            ptr, (B, H, W) = frames, shape
            fptr = C.cast(C.c_void_p(ptr), C.POINTER(C.c_uint8))
        else:
            frames = as_c(frames, np.uint8)
            B, H, W = frames.shape[:3]
            fptr = _p(frames, C.c_uint8)
        boxes = np.empty((B, max_det, 4), np.float32)
        scores = np.empty((B, max_det), np.float32)
        cls = np.empty((B, max_det), np.int32)
        idx = np.empty((B, max_det), np.int32)
        counts = np.empty((B,), np.int32)
        ncand = np.empty((B,), np.int32)
        check(lib().adas_yolo_detect(self._h, fptr, 1 if on_device else 0, B, H, W, C.c_double(box_score), C.c_double(nms_iou), max_det,
                                     _p(boxes, C.c_float), _p(scores, C.c_float), _p(cls, C.c_int32), _p(idx, C.c_int32),
                                     _p(counts, C.c_int32), _p(ncand, C.c_int32)))
        return boxes, scores, cls, idx, counts, ncand

    def _ufld_max_pts(self) -> int:
        """points per lane the lane decode can emit: max(row anchors, column anchors) for v2, rows for v1 (model kind 4)"""
        return self.output_shapes[0][2] if self.model_kind == 4 else max(self.output_shapes[0][2], self.output_shapes[1][2])

    def warp_perspective(self, batch: int, M, dsize) -> np.ndarray:
        """bird view (cv2.warpPerspective, INTER_LINEAR) of the frames of the LAST detect call on this engine, from the device copy."""
        Mb = as_c(np.broadcast_to(np.asarray(M, np.float64).reshape(-1, 3, 3), (batch, 3, 3)), np.float64)
        out = np.empty((batch, dsize[1], dsize[0], 3), np.uint8)
        check(lib().adas_engine_warp_perspective(self._h, batch, _p(Mb, C.c_double), dsize[1], dsize[0], _p(out, C.c_uint8)))
        return out

    def lane_geometry(self, batch: int, img_wh, adjust_lanes: bool = False, M=None, bird_wh=(1280, 720)):
        """lane polygon / polyfit resampling / bird-view points / curvature + offset of the frames of the LAST ufld_detect (or
        detect_pair) on this engine, computed from the lane points still resident on the device."""
        mp = self._ufld_max_pts()
        cap, area, bird, out = _lane_geom_outputs(batch, mp, img_wh[1], adjust_lanes)
        Mb = None
        if M is not None:
            Mb = as_c(np.broadcast_to(np.asarray(M, np.float64).reshape(-1, 3, 3), (batch, 3, 3)), np.float64)
        check(lib().adas_ufld_lane_geometry(self._h, batch, img_wh[0], img_wh[1], 1 if adjust_lanes else 0, _p(Mb, C.c_double) if Mb is not None else None,
                                            bird_wh[0], bird_wh[1], _p(area, C.c_int32), cap, _p(bird, C.c_int32), out.ctypes.data_as(C.c_void_p)))
        return _lane_geom_result(area, bird, out, Mb is not None)

    def ufld_detect(self, frames, on_device: bool = False, shape=None, want_coords: bool = False):
        if on_device:
            ptr, (B, H, W) = frames, shape
            fptr = C.cast(C.c_void_p(ptr), C.POINTER(C.c_uint8))
        else:
            frames = as_c(frames, np.uint8)
            B, H, W = frames.shape[:3]
            fptr = _p(frames, C.c_uint8)
        mp = self._ufld_max_pts()
        pts = np.empty((B, 4, mp, 2), np.int32)
        npts = np.empty((B, 4), np.int32)
        status = np.empty((B, 4), np.uint8)
        coords = np.empty((B, 4, mp), np.float64) if want_coords else None
        check(lib().adas_ufld_detect(self._h, fptr, 1 if on_device else 0, B, H, W, _p(pts, C.c_int32), _p(npts, C.c_int32),
                                     _p(status, C.c_uint8), _p(coords, C.c_double) if want_coords else None))
        return pts, npts, status, coords


def detect_pair(yolo: "Engine", ufld: "Engine", frames, box_score: float, nms_iou: float, max_det: int = 1024, on_device: bool = False, shape=None):
    """One library call: YOLO detect then UFLD lane detect on the same frames -> (yolo tuple, ufld tuple)."""
    if on_device:
        ptr, (B, H, W) = frames, shape
        fptr = C.cast(C.c_void_p(ptr), C.POINTER(C.c_uint8))
    else:
        frames = as_c(frames, np.uint8)
        B, H, W = frames.shape[:3]
        fptr = _p(frames, C.c_uint8)
    boxes = np.empty((B, max_det, 4), np.float32)
    scores = np.empty((B, max_det), np.float32)
    cls = np.empty((B, max_det), np.int32)
    idx = np.empty((B, max_det), np.int32)
    counts = np.empty((B,), np.int32)
    ncand = np.empty((B,), np.int32)
    mp = ufld._ufld_max_pts()
    pts = np.empty((B, 4, mp, 2), np.int32)
    npts = np.empty((B, 4), np.int32)
    status = np.empty((B, 4), np.uint8)
    check(lib().adas_detect_pair(yolo._h, ufld._h, fptr, 1 if on_device else 0, B, H, W, C.c_double(box_score), C.c_double(nms_iou), max_det,
                                 _p(boxes, C.c_float), _p(scores, C.c_float), _p(cls, C.c_int32), _p(idx, C.c_int32), _p(counts, C.c_int32),
                                 _p(ncand, C.c_int32), _p(pts, C.c_int32), _p(npts, C.c_int32), _p(status, C.c_uint8)))
    return (boxes, scores, cls, idx, counts, ncand), (pts, npts, status, None)


def yolo_postprocess(raw: np.ndarray, model_kind: int, n_classes: int, in_hw, src_hw, box_score: float, nms_iou: float,
                     max_det: int = 1024, device: int = 0):
    raw = as_c(raw, np.float32)
    B = raw.shape[0]
    A = raw.shape[2] if model_kind == 0 else raw.shape[1]
    boxes = np.empty((B, max_det, 4), np.float32)
    scores = np.empty((B, max_det), np.float32)
    cls = np.empty((B, max_det), np.int32)
    idx = np.empty((B, max_det), np.int32)
    counts = np.empty((B,), np.int32)
    ncand = np.empty((B,), np.int32)
    check(lib().adas_yolo_postprocess(device, _p(raw, C.c_float), model_kind, B, A, n_classes, in_hw[0], in_hw[1], src_hw[0], src_hw[1],
                                      C.c_double(box_score), C.c_double(nms_iou), max_det, _p(boxes, C.c_float), _p(scores, C.c_float),
                                      _p(cls, C.c_int32), _p(idx, C.c_int32), _p(counts, C.c_int32), _p(ncand, C.c_int32)))
    return boxes, scores, cls, idx, counts, ncand


def yolo_preprocess(frames: np.ndarray, in_hw, device: int = 0) -> np.ndarray:
    frames = as_c(frames, np.uint8)
    B, H, W = frames.shape[:3]
    blob = np.empty((B, 3, in_hw[0], in_hw[1]), np.float32)
    check(lib().adas_yolo_preprocess(device, _p(frames, C.c_uint8), B, H, W, in_hw[0], in_hw[1], _p(blob, C.c_float)))
    return blob


def ufld_preprocess(frames: np.ndarray, in_hw, crop_ratio: float, device: int = 0) -> np.ndarray:
    frames = as_c(frames, np.uint8)
    B, H, W = frames.shape[:3]
    blob = np.empty((B, 3, in_hw[0], in_hw[1]), np.float32)
    check(lib().adas_ufld_preprocess(device, _p(frames, C.c_uint8), B, H, W, in_hw[0], in_hw[1], C.c_double(crop_ratio), _p(blob, C.c_float)))
    return blob


def ufld_postprocess(heads: np.ndarray, dims, img_wh, row_anchor, col_anchor, device: int = 0, want_coords: bool = True):
    heads = as_c(heads, np.float32)
    B = heads.shape[0]
    ngr, ncr, ngc, ncc, nl = dims
    mp = max(ncr, ncc)
    pts = np.empty((B, 4, mp, 2), np.int32)
    npts = np.empty((B, 4), np.int32)
    status = np.empty((B, 4), np.uint8)
    coords = np.empty((B, 4, mp), np.float64)
    ra, ca = as_c(row_anchor, np.float64), as_c(col_anchor, np.float64)
    check(lib().adas_ufld_postprocess(device, _p(heads, C.c_float), B, ngr, ncr, ngc, ncc, nl, img_wh[0], img_wh[1], _p(ra, C.c_double),
                                      _p(ca, C.c_double), _p(pts, C.c_int32), _p(npts, C.c_int32), _p(status, C.c_uint8),
                                      _p(coords, C.c_double)))
    return pts, npts, status, coords


LANE_GEOM_DTYPE = np.dtype([("area_status", "<i4"), ("n_area", "<i4"), ("n_bird", "<i4", (4,)), ("direction", "<i4"), ("pad", "<i4"),
                            ("curvature", "<f8"), ("offset", "<f8")])
assert LANE_GEOM_DTYPE.itemsize == 48          # struct adas_lane_geom (include/adas_b200.h)


def _lane_geom_outputs(B, mp, img_h, adjust):
    cap = max(2 * mp, 2 * img_h if adjust else 0)
    return cap, np.zeros((B, cap, 2), np.int32), np.zeros((B, 4, mp, 2), np.int32), np.zeros(B, LANE_GEOM_DTYPE)


def _lane_geom_result(area, bird, out, have_M):
    """list per frame of dict(area_status, area [n,2], bird [4 arrays] or None, direction 'L'/'F'/'R'/None, curvature, offset)"""
    res = []
    for b in range(out.shape[0]):
        o = out[b]
        d = {-1: "L", 0: "F", 1: "R"}.get(int(o["direction"]))
        res.append({"area_status": bool(o["area_status"]), "area": area[b, :int(o["n_area"])].copy(),
                    "bird": [bird[b, l, :int(o["n_bird"][l])].copy() for l in range(4)] if have_M else None,
                    "direction": d, "curvature": float(o["curvature"]) if d is not None else None,
                    "offset": float(o["offset"]) if d is not None else None})
    return res


def warp_perspective(frames: np.ndarray, M, dsize, device: int = 0) -> np.ndarray:
    """cv2.warpPerspective(frame, M, dsize, flags=cv2.INTER_LINEAR) for uint8 [B,H,W,3] frames on the device, bit-exact.
    M: one 3x3 matrix for all frames or [B,3,3]; dsize = (width, height) as in cv2."""
    frames = as_c(frames, np.uint8)
    B, H, W = frames.shape[:3]
    Mb = as_c(np.broadcast_to(np.asarray(M, np.float64).reshape(-1, 3, 3), (B, 3, 3)), np.float64)
    out = np.empty((B, dsize[1], dsize[0], 3), np.uint8)
    check(lib().adas_warp_perspective(device, _p(frames, C.c_uint8), B, H, W, _p(Mb, C.c_double), dsize[1], dsize[0], _p(out, C.c_uint8)))
    return out


def lane_geometry(pts, npts, status, img_wh, adjust_lanes: bool = False, M=None, bird_wh=(1280, 720), device: int = 0):
    """Rows K + 8f-1 on the device from host arrays shaped like ufld_detect's outputs (see adas_lane_geometry in include/adas_b200.h).
    M: one 3x3 matrix for all frames or [B,3,3]."""
    pts, npts, status = as_c(pts, np.int32), as_c(npts, np.int32), as_c(status, np.uint8)
    B, _, mp, _ = pts.shape
    cap, area, bird, out = _lane_geom_outputs(B, mp, img_wh[1], adjust_lanes)
    Mb = None
    if M is not None:
        Mb = as_c(np.broadcast_to(np.asarray(M, np.float64).reshape(-1, 3, 3), (B, 3, 3)), np.float64)
    check(lib().adas_lane_geometry(device, _p(pts, C.c_int32), _p(npts, C.c_int32), _p(status, C.c_uint8), B, mp, img_wh[0], img_wh[1],
                                   1 if adjust_lanes else 0, _p(Mb, C.c_double) if Mb is not None else None, bird_wh[0], bird_wh[1],
                                   _p(area, C.c_int32), cap, _p(bird, C.c_int32), out.ctypes.data_as(C.c_void_p)))
    return _lane_geom_result(area, bird, out, Mb is not None)


def ufld_v1_postprocess(head: np.ndarray, griding_num: int, rows: int, in_wh, cfg_wh, img_wh, row_anchor, device: int = 0):
    """UFLD v1 decode of head tensors [B, griding_num+1, rows, 4] (see adas_ufld_v1_postprocess)."""
    head = as_c(head, np.float32)
    B = head.shape[0]
    pts = np.empty((B, 4, rows, 2), np.int32)
    npts = np.empty((B, 4), np.int32)
    status = np.empty((B, 4), np.uint8)
    coords = np.empty((B, 4, rows), np.float64)
    ra = as_c(row_anchor, np.float64)
    check(lib().adas_ufld_v1_postprocess(device, _p(head, C.c_float), B, griding_num, rows, in_wh[0], in_wh[1], cfg_wh[0], cfg_wh[1], img_wh[0], img_wh[1],
                                         _p(ra, C.c_double), _p(pts, C.c_int32), _p(npts, C.c_int32), _p(status, C.c_uint8), _p(coords, C.c_double)))
    return pts, npts, status, coords


def iou_cost(a_list, b_list, scores_list=None, device: int = 0):
    """Batched 1 - IoU (optionally fused with detection scores). Lists of [T_i,4] / [D_i,4] float64 tlbr arrays."""
    P = len(a_list)
    a_off = np.zeros(P + 1, np.int32)
    b_off = np.zeros(P + 1, np.int32)
    c_off = np.zeros(P + 1, np.int64)
    for i in range(P):
        a_off[i + 1] = a_off[i] + len(a_list[i])
        b_off[i + 1] = b_off[i] + len(b_list[i])
        c_off[i + 1] = c_off[i] + len(a_list[i]) * len(b_list[i])
    a = as_c(np.concatenate([np.asarray(x, np.float64).reshape(-1, 4) for x in a_list]) if P else np.zeros((0, 4)), np.float64)
    b = as_c(np.concatenate([np.asarray(x, np.float64).reshape(-1, 4) for x in b_list]) if P else np.zeros((0, 4)), np.float64)
    fuse = scores_list is not None
    sc = as_c(np.concatenate([np.asarray(s, np.float64).ravel() for s in scores_list]) if fuse else np.zeros(1), np.float64)
    cost = np.empty(int(c_off[-1]), np.float64)
    if cost.size:
        check(lib().adas_iou_cost(device, P, _p(a, C.c_double), _p(a_off, C.c_int32), _p(b, C.c_double), _p(b_off, C.c_int32),
                                  _p(sc, C.c_double), 1 if fuse else 0, _p(cost, C.c_double), _p(c_off, C.c_int64)))
    return [cost[c_off[i]:c_off[i + 1]].reshape(len(a_list[i]), len(b_list[i])) for i in range(P)]


def lap(cost_list, thresh_list, device: int = 0):
    """Batched exact assignment with lap.lapjv(extend_cost=True, cost_limit=thresh) semantics -> [(x_i, y_i)]."""
    P = len(cost_list)
    T = np.array([c.shape[0] for c in cost_list], np.int32)
    D = np.array([c.shape[1] for c in cost_list], np.int32)
    c_off = np.zeros(P + 1, np.int64)
    x_off = np.zeros(P + 1, np.int32)
    y_off = np.zeros(P + 1, np.int32)
    for i in range(P):
        c_off[i + 1] = c_off[i] + int(T[i]) * int(D[i])
        x_off[i + 1] = x_off[i] + T[i]
        y_off[i + 1] = y_off[i] + D[i]
    cost = as_c(np.concatenate([np.asarray(c, np.float64).ravel() for c in cost_list]) if P else np.zeros(0), np.float64)
    th = as_c(thresh_list, np.float64)
    x = np.full(max(int(x_off[-1]), 1), -1, np.int32)
    y = np.full(max(int(y_off[-1]), 1), -1, np.int32)
    check(lib().adas_lap(device, P, _p(cost, C.c_double), _p(c_off, C.c_int64), _p(T, C.c_int32), _p(D, C.c_int32), _p(th, C.c_double),
                         _p(x, C.c_int32), _p(x_off, C.c_int32), _p(y, C.c_int32), _p(y_off, C.c_int32)))
    return [(x[x_off[i]:x_off[i + 1]].copy(), y[y_off[i]:y_off[i + 1]].copy()) for i in range(P)]


def associate(a_tlbr, b_tlbr, det_scores, thresh: float, device: int = 0, want_cost: bool = False):
    """One ByteTrack association stage on the device: cost = 1 - IoU (optionally fused with scores) + exact assignment."""
    a = as_c(np.asarray(a_tlbr, np.float64).reshape(-1, 4), np.float64)
    b = as_c(np.asarray(b_tlbr, np.float64).reshape(-1, 4), np.float64)
    T, D = a.shape[0], b.shape[0]
    x = np.full(max(T, 1), -1, np.int32)
    y = np.full(max(D, 1), -1, np.int32)
    fuse = det_scores is not None
    sc = as_c(det_scores if fuse else np.zeros(1), np.float64)
    cost = np.empty((T, D), np.float64) if want_cost else None
    check(lib().adas_associate(device, T, D, _p(a, C.c_double), _p(b, C.c_double), _p(sc, C.c_double), 1 if fuse else 0, C.c_double(thresh),
                               _p(x, C.c_int32), _p(y, C.c_int32), _p(cost, C.c_double) if want_cost else None))
    return x[:T], y[:D], cost


class Comm:
    """NCCL gather of fixed-size per-batch record blocks, driven from C on a private stream (include/adas_b200.h, adas_comm_*)."""

    def __init__(self, device: int, rank: int, world: int, unique_id: bytes, bytes_per_rank: int):
        self._h = C.c_void_p()
        idb = (C.c_uint8 * 128).from_buffer_copy(unique_id)
        check(lib().adas_comm_create(int(device), int(rank), int(world), idb, C.c_int64(bytes_per_rank), C.byref(self._h)))
        self.world, self.bytes = world, bytes_per_rank

    @staticmethod
    def unique_id() -> bytes:
        idb = (C.c_uint8 * 128)()
        check(lib().adas_comm_unique_id(idb))
        return bytes(idb)

    def all_gather(self, rec: np.ndarray) -> None:
        assert rec.nbytes == self.bytes and rec.flags["C_CONTIGUOUS"]
        check(lib().adas_comm_all_gather(self._h, rec.ctypes.data_as(C.c_void_p)))

    def sync(self) -> None:
        check(lib().adas_comm_sync(self._h))

    def read(self, dtype=np.float32) -> np.ndarray:
        out = np.empty(self.world * self.bytes // np.dtype(dtype).itemsize, dtype)
        check(lib().adas_comm_read(self._h, out.ctypes.data_as(C.c_void_p)))
        return out.reshape(self.world, -1)

    def info(self):
        n, g = C.c_int(), C.c_int64()
        check(lib().adas_comm_info(self._h, C.byref(n), C.byref(g)))
        return int(n.value), int(g.value)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            lib().adas_comm_destroy(self._h)
            self._h = C.c_void_p()
