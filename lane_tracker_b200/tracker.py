"""Host-side mirror of the reference's ``LaneTracker`` (lane_tracker.py:85-1209).

``LaneTracker``         drop-in for the reference class: same constructor, same methods, NumPy in /
                        NumPy out, one stream.  Every method runs on the GPU through the C ABI.
``BatchedLaneTracker``  the throughput interface: S independent streams per call on device-resident
                        ``torch`` tensors, per-stream tracking state held in device memory.

PyTorch is used for device memory, pinned staging buffers and CUDA streams only.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import LT_MAX_LEVELS, check, lt_config, lt_params, lt_result, lt_state

RESULT_DTYPE = np.dtype(lt_result)

_FILTER_TYPES = {"bilateral": 0, "neighborhood": 1}

# layouts of the input frames of the hot path (lt_set_frame_format)
FRAME_RGB, FRAME_NV12 = 0, 1
_FRAME_FORMATS = {"rgb": FRAME_RGB, "nv12": FRAME_NV12}

# keyword defaults of the reference methods (SURVEY.md B.2)
PROCESS_DEFAULTS = dict(
    ksize_r=15, C_r=8, ksize_b=35, C_b=5, filter_type="bilateral", mask_noise=False, noise_thresh=140,
    ksize_noise=65, C_noise=10, window_width=30, window_height=40, search_range=20, mu=0.1,
    no_success_limit=8, start_slice=0.25, ignore_sides=360, ignore_bottom=30, bandwidth=25, partial=1.0,
    n_tries=2)


def _filter_code(filter_type):
    if filter_type not in _FILTER_TYPES:
        # same exception type and message as lane_tracker.py:219-220
        raise ValueError("Unexpected filter mode. Expected modes are 'bilateral' or 'neighborhood'.")
    return _FILTER_TYPES[filter_type]


def make_params(**kw):
    p = dict(PROCESS_DEFAULTS)
    unknown = set(kw) - set(p)
    if unknown:
        raise TypeError("process() got unexpected keyword arguments %s" % sorted(unknown))
    p.update(kw)
    out = lt_params()
    out.filter_type = _filter_code(p.pop("filter_type"))
    out.mask_noise = int(bool(p.pop("mask_noise")))
    for k, v in p.items():
        setattr(out, k, float(v) if k in ("mu", "start_slice", "partial") else int(v))
    return out


def _float64_mean(v):
    """np.average of a short list in NumPy's float64 summation order (pairwise unrolled by 8 from 8 elements on)."""
    if len(v) == 8:
        return (((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]))) / 8.0
    acc = v[0]
    for x in v[1:]:
        acc = acc + x
    return acc / len(v)


def bilateral_adaptive_threshold(img, ksize=30, C=0, mode='floor', true_value=255, false_value=0, device=None):
    """Drop-in for the reference's module-level ``bilateral_adaptive_threshold`` (lane_tracker.py:14-83): cross-shaped
    adaptive threshold of a single-channel uint8 image, computed on the GPU.  NumPy in, NumPy out."""
    if mode not in ('floor', 'ceil'):
        raise ValueError("Unexpected mode value. Expected value is 'floor' or 'ceil'.")     # lane_tracker.py:71
    if not torch.cuda.is_available():
        raise _lib.LaneTrackerError("lane_tracker_b200 needs a CUDA device; there is no CPU path")
    lib = _lib.load()
    a = np.ascontiguousarray(img)
    if a.ndim != 2 or a.dtype != np.uint8:
        raise ValueError("img must be a single-channel uint8 image")
    dev = torch.device("cuda", torch.cuda.current_device() if device is None else device)
    with torch.cuda.device(dev):
        d = torch.from_numpy(a).to(dev)
        out = torch.empty_like(d)
        check(lib.lt_bilateral_adaptive_threshold(_ptr(d), int(a.shape[1]), int(a.shape[0]), int(a.shape[1]), _ptr(out),
                                                  int(a.shape[1]), int(ksize), int(C), 0 if mode == 'floor' else 1,
                                                  int(true_value), int(false_value), _stream_ptr(dev)))
        return out.cpu().numpy()


def _calibration(cam_matrix, dist_coeffs, warp_matrices, mpp_conversion):
    """The calibration arguments of the constructor and of ``set_camera`` -> lt_camera (checked)."""
    c = _lib.lt_camera()
    c.cam_matrix[:] = [float(v) for v in np.asarray(cam_matrix, dtype=np.float64).reshape(9)]
    d = np.asarray(dist_coeffs, dtype=np.float64).ravel()
    if d.size > 5 and np.any(d[5:] != 0):
        raise ValueError("only the 5-coefficient distortion model (k1,k2,p1,p2,k3) is supported")
    c.dist_coeffs[:] = [float(v) for v in np.concatenate([d[:5], np.zeros(max(0, 5 - d.size))])]
    c.M[:] = [float(v) for v in np.asarray(warp_matrices[0], dtype=np.float64).reshape(9)]
    c.Minv[:] = [float(v) for v in np.asarray(warp_matrices[1], dtype=np.float64).reshape(9)]
    c.mppv, c.mpph = float(mpp_conversion[0]), float(mpp_conversion[1])
    return c


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _stream_ptr(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class BatchedLaneTracker:
    """S independent lane trackers advanced by one frame each per ``process`` call."""

    def __init__(self, n_streams, img_size, warped_size, cam_matrix, dist_coeffs, warp_matrices,
                 mpp_conversion, n_fail=8, n_reset=4, n_average=2, print_frame_count=False, device=None):
        self._h = None
        if not torch.cuda.is_available():
            raise _lib.LaneTrackerError("lane_tracker_b200 needs a CUDA device; there is no CPU path")
        self.lib = _lib.load()
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else
                                   (device if isinstance(device, int) else torch.device(device).index or 0))
        self.n_streams = int(n_streams)
        self.img_size = tuple(int(v) for v in img_size)
        self.warped_size = tuple(int(v) for v in warped_size)
        self.n_fail, self.n_reset, self.n_average = int(n_fail), int(n_reset), int(n_average)
        cfg = lt_config()
        cfg.img_w, cfg.img_h = self.img_size
        cfg.bv_w, cfg.bv_h = self.warped_size
        cal = _calibration(cam_matrix, dist_coeffs, warp_matrices, mpp_conversion)
        for name, _ in _lib.lt_camera._fields_:
            setattr(cfg, name, getattr(cal, name))
        cfg.n_fail, cfg.n_reset, cfg.n_average = self.n_fail, self.n_reset, self.n_average
        cfg.print_frame_count = int(bool(print_frame_count))
        cfg.max_streams = self.n_streams
        cfg.device = self.device.index
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            check(self.lib.lt_create(C.byref(cfg), C.byref(h)))
        self._h = h
        self._format_set = FRAME_RGB           # what the handle was last set to (lt_set_frame_format)
        S = self.n_streams
        self._results_dev = torch.zeros(S * RESULT_DTYPE.itemsize, dtype=torch.uint8, device=self.device)
        self._results_host = torch.zeros(S * RESULT_DTYPE.itemsize, dtype=torch.uint8).pin_memory()
        from .text import TextSprites
        self.text_enabled = False
        self.text_rows = (0, 0)
        if TextSprites.available():
            self.set_text(True)
        geo = np.zeros(9, dtype=np.int32)
        check(self.lib.lt_debug_read(self._h, 10, 0, geo.ctypes.data_as(C.c_void_p), geo.nbytes))
        self.geometry = dict(roi_rows=(int(geo[0]), int(geo[1])), overlay_rows=(int(geo[2]), int(geo[3])),
                             plane_width=int(geo[4]), mask_words=int(geo[5]), pixel_capacity=int(geo[6]),
                             source_rows=(int(geo[7]), int(geo[8])))
        self.camera_rows = {}                  # camera -> its rows (lt_debug_read 13), see ``set_camera``
        self._read_camera_rows(0)
        self.camera_epoch = 0                  # bumped by set_camera (GraphedProcess refuses to replay across it)

    def _read_camera_rows(self, k):
        v = np.zeros(6, dtype=np.int32)
        check(self.lib.lt_debug_read(self._h, 13, int(k), v.ctypes.data_as(C.c_void_p), v.nbytes))
        self.camera_rows[int(k)] = dict(roi_rows=(int(v[0]), int(v[1])), overlay_rows=(int(v[2]), int(v[3])),
                                        source_rows=(int(v[4]), int(v[5])))

    def rows_any_camera(self):
        """(source rows, overlay rows) over camera 0 and every camera set: the frame rows the tracker may read, and
        those the lane overlay may change, whichever cameras a batch uses (half-open; overlay (0, 0) if none)."""
        src = [r["source_rows"] for r in self.camera_rows.values()]
        ov = [r["overlay_rows"] for r in self.camera_rows.values() if r["overlay_rows"][1] > r["overlay_rows"][0]]
        return ((min(a for a, _ in src), max(b for _, b in src)),
                (min(a for a, _ in ov), max(b for _, b in ov)) if ov else (0, 0))

    def set_camera(self, k, cam_matrix, dist_coeffs, warp_matrices, mpp_conversion):
        """Set camera k (1 <= k < LT_MAX_CAMERAS) for the ``cameras=`` argument of the process calls: a calibration in
        the constructor's forms (camera 0 is the constructor's and cannot change).  Image and bird's-eye sizes stay
        the handle's.  Synchronises the device.  A stream whose camera was re-mounted keeps its tracking state: flag
        its first frame from the new mounting in ``starts=`` to start it afresh.  A ``GraphedProcess`` captured with
        cameras before this call can no longer replay."""
        cal = _calibration(cam_matrix, dist_coeffs, warp_matrices, mpp_conversion)
        with torch.cuda.device(self.device):
            check(self.lib.lt_set_camera(self._h, int(k), C.byref(cal)))
        self._read_camera_rows(k)
        # a graph holds pointers to the camera tables and the camera undistort buffer, which this call may replace
        self.camera_epoch += 1

    # -- lifetime -----------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self.lib.lt_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self, ids=None):
        """Re-zero the state of the streams ``ids`` (None: all) synchronously, outside every CUDA stream: only with no
        work of this tracker in flight.  ``reset_async`` and ``starts=`` are ordered with the batches."""
        if ids is None:
            check(self.lib.lt_reset(self._h, None, 0))
        else:
            arr = (C.c_int32 * len(ids))(*[int(i) for i in ids])
            check(self.lib.lt_reset(self._h, arr, len(ids)))

    def reset_async(self, ids=None):
        """Enqueue on the current CUDA stream what ``reset(ids)`` writes (None: every stream): the next frame of each
        stream is processed as by a freshly reset stream.  Capturable in a CUDA graph."""
        arr = None if ids is None else self._check_ids(ids, len(ids))
        with torch.cuda.device(self.device):
            check(self.lib.lt_reset_async(self._h, arr, 0 if ids is None else len(ids), _stream_ptr(self.device)))

    @property
    def record_bytes(self):
        """Size of one stream's state record (``export_states`` / ``import_states``)."""
        return int(check(self.lib.lt_state_record_bytes(self._h)))

    def export_states(self, ids, out=None):
        """The state records of streams ``ids`` (distinct) -> CUDA uint8 tensor [n, record_bytes] (``out`` if given),
        gathered on the current CUDA stream: tracking state, averaged polylines and cached lane polygon, everything a
        later frame of the stream reads (layout: include/lane_tracker_b200.h).  Capturable in a CUDA graph."""
        h_ids = self._check_ids(ids, len(ids))
        n, rb = len(ids), self.record_bytes
        if out is None:
            out = torch.empty((n, rb), dtype=torch.uint8, device=self.device)
        self._check_records(out, n, "out")
        with torch.cuda.device(self.device):
            check(self.lib.lt_export_states(self._h, h_ids, n, _ptr(out), _stream_ptr(self.device)))
        return out

    def import_states(self, ids, records, check=True):
        """Write the state records ``records`` [n, record_bytes] (from ``export_states`` of this or another tracker of
        the same bird's-eye size, n_average, n_fail and n_reset, moved to this tracker's device) into slots ``ids``, on
        the current CUDA stream.  Each record is checked on the device first; a refused one is not applied and its
        slot keeps its state.  -> int32 CUDA tensor [n] of status codes (LT_RECORD_OK, LT_RECORD_BAD_HEADER,
        LT_RECORD_BAD_STATE).  check=True synchronises the current stream and raises ValueError naming the first
        refused position."""
        do_check = check
        h_ids = self._check_ids(ids, len(ids))
        n = len(ids)
        self._check_records(records, n, "records")
        status = torch.empty(n, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.lt_import_states(self._h, h_ids, n, _ptr(records), _ptr(status),
                                                 _stream_ptr(self.device)))
        if do_check:
            got = status.cpu().numpy()        # synchronises the current stream
            bad = np.flatnonzero(got != _lib.LT_RECORD_OK)
            if bad.size:
                i = int(bad[0])
                why = {_lib.LT_RECORD_BAD_HEADER: "its header does not match this tracker (magic, ABI version, state "
                                                  "size, bird's-eye size, n_average, n_fail or n_reset)",
                       _lib.LT_RECORD_BAD_STATE: "its state is inconsistent (ring_len, radii_len, polyline lengths, "
                                                 "polygon rows or box out of range)"}.get(int(got[i]), "code %d" % got[i])
                raise ValueError("state record at position %d (stream %d) refused: %s" % (i, int(ids[i]), why))
        return status

    def _check_records(self, t, n, name):
        rb = self.record_bytes
        if not (isinstance(t, torch.Tensor) and t.dtype == torch.uint8 and t.device == self.device and
                t.is_contiguous() and tuple(t.shape) == (n, rb)):
            raise ValueError("%s must be a contiguous uint8 tensor [%d, %d] on %s" % (name, n, rb, self.device))
        if t.data_ptr() % 16:
            raise ValueError("%s must start at a 16-byte aligned address" % name)

    def set_validity(self, **kw):
        """Override the acceptance windows of check_validity (lane_tracker.py:588-593, 617); no arguments restores
        the shipped constants.  Keys: min/max_dist_y1..y3, tangent_thresh (see lane_tracker_b200.presets)."""
        if not kw:
            check(self.lib.lt_set_validity(self._h, None))
            return
        v = _lib.lt_validity()
        check(self.lib.lt_get_validity(self._h, C.byref(v)))
        for k, val in kw.items():
            if not hasattr(v, k):
                raise TypeError("unknown validity option %r" % k)
            setattr(v, k, float(val))
        check(self.lib.lt_set_validity(self._h, C.byref(v)))

    def set_profile(self, k, params=None, validity=None, **kw):
        """Store parameter profile k (0 <= k < LT_MAX_PROFILES) for the ``profiles=`` argument of the process calls:
        ``params`` (default: ``make_params(**kw)``) and the check_validity windows ``validity``, a dict with the keys of
        ``set_validity`` (missing keys and None: the shipped windows).  A batch uses the profiles as they stood when its
        front half was enqueued, so this may be called with work in flight.

            bt.set_profile(1, validity=presets.DEMO_1["validity"], **presets.DEMO_1["process"])
        """
        p = params if params is not None else make_params(**kw)
        if params is not None and kw:
            raise ValueError("pass either params or keyword options, not both")
        v = None
        if validity is not None:
            from .presets import SHIPPED_VALIDITY
            v = _lib.lt_validity(**{key: float(val) for key, val in SHIPPED_VALIDITY.items()})
            for key, val in validity.items():
                if not hasattr(v, key):
                    raise TypeError("unknown validity option %r" % key)
                setattr(v, key, float(val))
        check(self.lib.lt_set_profile(self._h, int(k), C.byref(p), C.byref(v) if v is not None else None))

    def set_text(self, enable=True):
        """Install (or remove) the glyph sprites of the reference's putText overlays (lane_tracker.py:653-659, 668-672)."""
        from .text import TextSprites
        if not enable:
            check(self.lib.lt_set_text_sprites(self._h, None, 0, None, 0, None, None, None, 0, None, 0))
            self.text_enabled = False
            self.text_rows = (0, 0)
            return
        sp = TextSprites.load()
        vp = lambda a: a.ctypes.data_as(C.c_void_p)
        check(self.lib.lt_set_text_sprites(self._h, vp(sp.tables), int(sp.tables.shape[0]), vp(sp.char_start),
                                           int(len(sp.advance)), vp(sp.dy), vp(sp.dx), vp(sp.lut), int(len(sp.dy)),
                                           vp(sp.advance), sp.first_char))
        self.text_enabled = True
        self.text_rows = (max(0, 35 + int(sp.dy.min())), min(self.img_size[1], 105 + int(sp.dy.max()) + 1))

    def set_remap_mode(self, mode="exact"):
        """'exact': two-stage undistort + warp, bit-exact with OpenCV (default).  'fused': single resample from the
        raw frame (not bit-exact; mask IoU >= 0.6 per frame, >= 0.8 mean on the bundled frames)."""
        codes = {"exact": 0, "fused": 1}
        if mode not in codes:
            raise ValueError("remap mode must be 'exact' or 'fused'")
        check(self.lib.lt_set_remap_mode(self._h, codes[mode]))

    def copy_rows(self, dst, src, row0, row1, to_device):
        """Copy frame rows [row0, row1) of a batch of full frames between pinned host and device tensors on the
        current stream (strided 2-D copy, no staging).  NV12 batches ([n, H * 3 / 2, W]) move luma rows [row0, row1)
        and the chroma rows that cover them."""
        n = int(src.shape[0])
        self._use_format(FRAME_NV12 if src.dim() == 3 else FRAME_RGB)
        check(self.lib.lt_memcpy_rows(self._h, _ptr(dst), _ptr(src), n, int(row0), int(row1), int(bool(to_device)),
                                      _stream_ptr(self.device)))

    @property
    def sm_count(self):
        return self._launch_geometry()[2]

    def morph_bands(self):
        """(row bands of the 55x55 job, of the 29x29 job) in the last ellipse-morphology launch."""
        g = self._launch_geometry()
        return int(g[0]), int(g[1])

    def _launch_geometry(self):
        g = np.zeros(3, dtype=np.int32)
        check(self.lib.lt_debug_read(self._h, 11, 0, g.ctypes.data_as(C.c_void_p), g.nbytes))
        return g

    def set_capture(self, enable=True):
        check(self.lib.lt_set_capture(self._h, int(bool(enable))))

    def set_pixel_capacity(self, capacity):
        """Entries per stream and side of the captured pixel lists (default: enough for bandwidth <= 32)."""
        check(self.lib.lt_set_pixel_capacity(self._h, int(capacity)))
        self.geometry["pixel_capacity"] = int(capacity)

    def profile_begin(self, max_calls):
        """Arm in-stream CUDA-event timing of every stage of the next `max_calls` process() calls."""
        check(self.lib.lt_profile_begin(self._h, int(max_calls)))

    def profile_select(self, stages=None):
        """Mark only the boundaries of the named stages (None: all).  Name the boundary before a stage too."""
        mask = 0
        if stages:
            names = {self.lib.lt_stage_name(i).decode(): i for i in range(_lib.LT_NSTAGES)}
            for st in stages:
                mask |= 1 << names[st]
        check(self.lib.lt_profile_select(self._h, mask))

    def profile_read(self):
        """-> ({stage name: total ms}, calls); synchronises."""
        ms = (C.c_double * _lib.LT_NSTAGES)()
        calls = C.c_int32(0)
        check(self.lib.lt_profile_read(self._h, ms, C.byref(calls)))
        return {self.lib.lt_stage_name(i).decode(): float(ms[i]) for i in range(1, _lib.LT_NSTAGES)}, calls.value

    # -- hot path -----------------------------------------------------------
    def _frame_format(self, frames):
        """-> (n, format) of an input batch: uint8 [n, H, W, 3] is RGB, uint8 [n, H * 3 / 2, W] is NV12."""
        w, h = self.img_size
        if not (isinstance(frames, torch.Tensor) and frames.dtype == torch.uint8):
            raise ValueError("frames must be a uint8 tensor")
        if frames.dim() == 4 and tuple(frames.shape[1:]) == (h, w, 3):
            fmt = FRAME_RGB
        elif frames.dim() == 3 and tuple(frames.shape[1:]) == (h * 3 // 2, w) and h % 2 == 0:
            fmt = FRAME_NV12
        else:
            raise ValueError("frames must be RGB [n, %d, %d, 3] or NV12 [n, %d, %d], got %s"
                             % (h, w, h * 3 // 2, w, list(frames.shape)))
        if not (frames.is_cuda and frames.is_contiguous()):
            raise ValueError("frames must be a contiguous CUDA tensor")
        if frames.data_ptr() % 4:
            raise ValueError("frames must start at a 4-byte aligned address (the kernels access frames as 32-bit words)")
        if frames.shape[0] < 1 or frames.shape[0] > self.n_streams:
            raise ValueError("got %d frames for %d streams" % (frames.shape[0], self.n_streams))
        return int(frames.shape[0]), fmt

    def _use_format(self, fmt):
        if fmt != self._format_set:
            check(self.lib.lt_set_frame_format(self._h, int(fmt)))
            self._format_set = fmt

    def _input(self, frames):
        """Check an input batch of RGB or NV12 frames and set the handle's frame format to it; -> n."""
        n, fmt = self._frame_format(frames)
        self._use_format(fmt)
        return n

    def _check_frames(self, frames):
        """Check an input batch of RGB frames (the stage calls take no NV12); -> n."""
        n, fmt = self._frame_format(frames)
        if fmt != FRAME_RGB:
            w, h = self.img_size
            raise ValueError("frames must be RGB [n, %d, %d, 3] here, got NV12 frames" % (h, w))
        return n

    def _check_ids(self, ids, n, repeats=False):
        """Stream ids of a batch of n frames -> ctypes int32 array (None: None).  Any int sequence, NumPy array or CPU
        tensor of n distinct ids in [0, n_streams); frame i belongs to stream ids[i].  repeats=True (a sequence batch):
        ids may repeat."""
        if ids is None:
            return None
        if isinstance(ids, torch.Tensor):
            if ids.is_cuda:
                raise ValueError("ids must be host data (a sequence, a NumPy array or a CPU tensor), not a CUDA tensor")
            ids = ids.numpy()
        a = np.asarray(ids)
        if a.ndim != 1 or (a.size and a.dtype.kind not in "iu"):
            raise ValueError("ids must be a 1-D sequence of integers")
        if a.size != n:
            raise ValueError("got %d stream ids for %d frames" % (a.size, n))
        bad = a[(a < 0) | (a >= self.n_streams)]
        if bad.size:
            raise ValueError("stream id %d outside [0, %d)" % (int(bad[0]), self.n_streams))
        u, counts = np.unique(a, return_counts=True)
        if not repeats and (counts > 1).any():
            raise ValueError("stream id %d appears more than once in the batch" % int(u[counts > 1][0]))
        return (C.c_int32 * n)(*[int(v) for v in a])

    def _check_profiles(self, profiles, n):
        """Profile indices of a batch of n frames -> ctypes int32 array (None: None).  Any int sequence, NumPy array or
        CPU tensor of n indices in [0, LT_MAX_PROFILES); frame i uses profile profiles[i] (see ``set_profile``)."""
        if profiles is None:
            return None
        if isinstance(profiles, torch.Tensor):
            if profiles.is_cuda:
                raise ValueError("profiles must be host data (a sequence, a NumPy array or a CPU tensor), not a CUDA tensor")
            profiles = profiles.numpy()
        a = np.asarray(profiles)
        if a.ndim != 1 or (a.size and a.dtype.kind not in "iu"):
            raise ValueError("profiles must be a 1-D sequence of integers")
        if a.size != n:
            raise ValueError("got %d profile indices for %d frames" % (a.size, n))
        bad = np.flatnonzero((a < 0) | (a >= _lib.LT_MAX_PROFILES))
        if bad.size:
            raise ValueError("profile %d at batch position %d outside [0, %d)"
                             % (int(a[bad[0]]), int(bad[0]), _lib.LT_MAX_PROFILES))
        return (C.c_int32 * n)(*[int(v) for v in a])

    def _check_cameras(self, cameras, n):
        """Camera indices of a batch of n frames -> ctypes int32 array (None: None).  Any int sequence, NumPy array or
        CPU tensor of n indices in [0, LT_MAX_CAMERAS); frame i was filmed by camera cameras[i] (see ``set_camera``)."""
        if cameras is None:
            return None
        if isinstance(cameras, torch.Tensor):
            if cameras.is_cuda:
                raise ValueError("cameras must be host data (a sequence, a NumPy array or a CPU tensor), not a CUDA tensor")
            cameras = cameras.numpy()
        a = np.asarray(cameras)
        if a.ndim != 1 or (a.size and a.dtype.kind not in "iu"):
            raise ValueError("cameras must be a 1-D sequence of integers")
        if a.size != n:
            raise ValueError("got %d camera indices for %d frames" % (a.size, n))
        bad = np.flatnonzero((a < 0) | (a >= _lib.LT_MAX_CAMERAS))
        if bad.size:
            raise ValueError("camera %d at batch position %d outside [0, %d)"
                             % (int(a[bad[0]]), int(bad[0]), _lib.LT_MAX_CAMERAS))
        unset = [i for i, k in enumerate(a) if int(k) not in self.camera_rows]
        if unset:
            raise ValueError("camera %d at batch position %d is unset" % (int(a[unset[0]]), unset[0]))
        return (C.c_int32 * n)(*[int(v) for v in a])

    @staticmethod
    def _check_sequence(sequence, ids, profiles, cameras):
        if not sequence:
            return
        if ids is None:
            raise ValueError("sequence=True needs ids: the stream of every frame")
        if profiles is not None or cameras is not None:
            raise ValueError("sequence=True takes neither profiles nor cameras")

    @staticmethod
    def _check_starts(starts, ids, n, sequence):
        """``starts`` of a batch of n frames -> the stream ids to start (None: no starts).  One bool per batch position:
        position i starts a new video on its stream (ids[i], or i without ids).  In a sequence batch a start may only
        be at a stream's first position in the batch."""
        if starts is None:
            return None
        if isinstance(starts, torch.Tensor):
            if starts.is_cuda:
                raise ValueError("starts must be host data (a sequence, a NumPy array or a CPU tensor), not a CUDA tensor")
            starts = starts.numpy()
        if isinstance(starts, np.ndarray) and starts.ndim != 1:
            raise ValueError("starts must be a 1-D sequence of bools")
        a = list(starts)
        if len(a) != n:
            raise ValueError("got %d starts for %d frames" % (len(a), n))
        for i, v in enumerate(a):
            if not isinstance(v, (bool, np.bool_)):
                raise ValueError("starts[%d] is %r: starts must be bools" % (i, v))
        sids = [int(ids[i]) if ids is not None else i for i in range(n)]
        if sequence:
            first = {}
            for i, s in enumerate(sids):
                first.setdefault(s, i)
            for i, v in enumerate(a):
                if v and first[sids[i]] != i:
                    raise ValueError("starts[%d]: stream %d starts a new video after its frame at position %d of this "
                                     "sequence batch; a start must be a stream's first position: split the batch there"
                                     % (i, sids[i], first[sids[i]]))
        flagged = [s for s, v in zip(sids, a) if v]
        return flagged or None

    @staticmethod
    def _no_params_with_profiles(profiles, params, kw):
        if profiles is not None and (params is not None or kw):
            raise ValueError("profiles= selects the parameters of every frame: pass it without params or keyword options")

    def _check_out(self, out, frames):
        """out: RGB [n, H, W, 3] for RGB and NV12 frames alike."""
        if out is None:
            return
        w, h = self.img_size
        if (tuple(out.shape) != (int(frames.shape[0]), h, w, 3) or out.dtype != torch.uint8 or not out.is_cuda or
                not out.is_contiguous()):
            raise ValueError("out must be a contiguous CUDA uint8 tensor [n, %d, %d, 3] for n frames" % (h, w))
        if out.data_ptr() % 4:
            raise ValueError("out must start at a 4-byte aligned address (the kernels access frames as 32-bit words)")

    def process_async(self, frames, out=None, params=None, results_dev=None, ids=None, profiles=None, cameras=None,
                      sequence=False, starts=None, **kw):
        """Enqueue one frame per stream on the current CUDA stream; returns the number of frames.

        frames: uint8 CUDA tensor [n, H, W, 3] (RGB) or [n, H * 3 / 2, W] (NV12: the luma plane, then interleaved
        U, V rows, as video decoders deliver it; same results as RGB frames converted by ``nv12_to_rgb``).
        out: RGB [n, H, W, 3] or None (fits-only mode); for NV12 frames it is a separate buffer.
        results_dev: optional uint8 CUDA buffer of n * RESULT_DTYPE.itemsize bytes (default: internal).
        ids: None -- frame i belongs to stream i; else n distinct stream ids in [0, n_streams), any order (int
        sequence, NumPy array or CPU tensor): frame i belongs to stream ids[i], and the streams not listed keep their
        state.  out and the result records stay in batch order.
        profiles: None -- every frame uses ``params`` (or ``make_params(**kw)``); else n profile indices (any int
        sequence, NumPy array or CPU tensor; see ``set_profile``): frame i uses profile profiles[i], and ``params`` /
        keyword options may not be given.
        cameras: None -- every frame comes from camera 0 (the constructor's calibration); else n camera indices (see
        ``set_camera``): frame i was filmed by camera cameras[i].  A caller with one camera per stream passes
        camera_of[ids].
        sequence: True -- ids may repeat: the frames of one stream are consecutive frames of that stream, in batch
        order, and the results equal feeding them one at a time (``ids`` required; no ``profiles`` or ``cameras``).
        One video, 64 frames per call::

            for chunk, out in chunks:          # [<= n_streams, H, W, 3] consecutive frames of stream 0
                tracker.process_async(chunk, out, ids=[0] * len(chunk), sequence=True)

        starts: None, or one bool per frame: frame i is the first frame of a new video on its stream (ids[i], or i
        without ids) and is processed as by a freshly reset stream (``reset_async`` of the flagged streams, enqueued
        right before the back half).  In a sequence batch only a stream's first position may start.  Refused before
        anything is enqueued: a wrong length or an entry that is not a bool.  The reset is enqueued after every check
        made here and before the library call; a batch the library itself then refuses (LaneTrackerError: an unset
        profile, parameters out of range, a back half whose profiles or cameras differ from its front half's) has
        already reset its flagged streams, which start their new videos with the next frames they are given."""
        return self._process_call(frames, out, None, params, results_dev, ids, kw, profiles, cameras, sequence, starts)

    def process_front_async(self, frames, buffer_set, params=None, profiles=None, cameras=None, **kw):
        """First half of ``process_async`` (undistort, warp, first-attempt filter) into intermediate buffer set
        0 or 1, on the current CUDA stream.  Stateless.  See ``DevicePipeline``.  RGB or NV12 frames.  With
        ``profiles`` or ``cameras``, the back half of this buffer set must be given the same indices."""
        n = self._input(frames)
        self._no_params_with_profiles(profiles, params, kw)
        h_prof = self._check_profiles(profiles, n)
        h_cam = self._check_cameras(cameras, n)
        if h_cam is not None:
            p = None if h_prof is not None else (params if params is not None else make_params(**kw))
            check(self.lib.lt_process_front_cameras(self._h, _ptr(frames), h_cam, n, C.byref(p) if p is not None else None,
                                                    h_prof, int(buffer_set), _stream_ptr(self.device)))
            return n
        if h_prof is not None:
            check(self.lib.lt_process_front_profiles(self._h, _ptr(frames), h_prof, n, int(buffer_set),
                                                     _stream_ptr(self.device)))
            return n
        p = params if params is not None else make_params(**kw)
        check(self.lib.lt_process_front(self._h, _ptr(frames), n, C.byref(p), int(buffer_set), _stream_ptr(self.device)))
        return n

    def process_back_async(self, frames, out, buffer_set, params=None, results_dev=None, ids=None, profiles=None,
                           cameras=None, sequence=False, starts=None, **kw):
        """Second half of ``process_async`` (searches, second attempt, state machine, overlay) from intermediate
        buffer set 0 or 1, on the current CUDA stream.  Advances the per-stream state of the streams in ``ids``
        (None: streams 0..n-1), as ``process_async``.  RGB or NV12 frames, as given to the front half.  ``profiles``,
        ``cameras``: those the front half of this buffer set was given.  ``sequence``, ``starts``: as
        ``process_async`` (the front half takes no ids; a start only touches the state the back half reads)."""
        return self._process_call(frames, out, buffer_set, params, results_dev, ids, kw, profiles, cameras, sequence,
                                  starts)

    def _process_call(self, frames, out, buffer_set, params, results_dev, ids, kw, profiles=None, cameras=None,
                      sequence=False, starts=None):
        """Checks and C call of ``process_async`` (buffer_set None: both halves) or ``process_back_async``; -> n."""
        n = self._input(frames)
        self._check_out(out, frames)
        self._check_sequence(sequence, ids, profiles, cameras)
        h_ids = self._check_ids(ids, n, repeats=sequence)
        self._no_params_with_profiles(profiles, params, kw)
        h_prof = self._check_profiles(profiles, n)
        h_cam = self._check_cameras(cameras, n)
        started = self._check_starts(starts, ids, n, sequence)
        res = self._results_dev if results_dev is None else results_dev
        if res.numel() < n * RESULT_DTYPE.itemsize or not res.is_cuda:
            raise ValueError("results buffer too small")
        if started is not None:
            # the new videos begin right before the back half that reads their first frames, on its stream
            self.reset_async(started)
        if h_cam is not None:
            p = None if h_prof is not None else (params if params is not None else make_params(**kw))
            pp = C.byref(p) if p is not None else None
            if buffer_set is None:
                check(self.lib.lt_process_cameras(self._h, _ptr(frames), _ptr(out), h_ids, h_cam, n, pp, h_prof,
                                                  _ptr(res), _stream_ptr(self.device)))
            else:
                check(self.lib.lt_process_back_cameras(self._h, _ptr(frames), _ptr(out), h_ids, h_cam, n, pp, h_prof,
                                                       int(buffer_set), _ptr(res), _stream_ptr(self.device)))
            return n
        if h_prof is not None:
            if buffer_set is None:
                check(self.lib.lt_process_profiles(self._h, _ptr(frames), _ptr(out), h_ids, h_prof, n, _ptr(res),
                                                   _stream_ptr(self.device)))
            else:
                check(self.lib.lt_process_back_profiles(self._h, _ptr(frames), _ptr(out), h_ids, h_prof, n,
                                                        int(buffer_set), _ptr(res), _stream_ptr(self.device)))
            return n
        p = params if params is not None else make_params(**kw)
        if buffer_set is None:
            plain, streams, set_arg = self.lib.lt_process, self.lib.lt_process_streams, ()
            if sequence:
                streams = self.lib.lt_process_sequence
        else:
            plain, streams, set_arg = self.lib.lt_process_back, self.lib.lt_process_back_streams, (int(buffer_set),)
            if sequence:
                streams = self.lib.lt_process_back_sequence
        fn, ids_arg = (plain, ()) if h_ids is None else (streams, (h_ids,))
        check(fn(self._h, _ptr(frames), _ptr(out), *ids_arg, n, C.byref(p), *set_arg, _ptr(res),
                 _stream_ptr(self.device)))
        return n

    def fetch_results(self, n=None, results_dev=None):
        """Copy the first n result records of ``results_dev`` (default: the internal buffer ``process_async`` fills
        when given none) to pinned host memory and return them as a structured array (synchronises)."""
        n = self.n_streams if n is None else n
        res = self._results_dev if results_dev is None else results_dev
        nbytes = n * RESULT_DTYPE.itemsize
        self._results_host[:nbytes].copy_(res[:nbytes], non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        return self._results_host[:nbytes].numpy().view(RESULT_DTYPE).copy()

    def process(self, frames, out=None, params=None, ids=None, profiles=None, cameras=None, sequence=False, starts=None,
                **kw):
        """``process_async`` followed by ``fetch_results``: the n result records, in batch order.  With ``ids``, frame
        i advances stream ids[i] and the other streams keep their state; with ``profiles``, frame i uses parameter
        profile profiles[i] (``set_profile``); with ``cameras``, frame i comes from camera cameras[i] (``set_camera``);
        with ``sequence=True``, ids may repeat and a stream's frames are its consecutive frames, in batch order; with
        ``starts``, the flagged frames begin new videos on their streams."""
        n = self.process_async(frames, out, params, ids=ids, profiles=profiles, cameras=cameras, sequence=sequence,
                               starts=starts, **kw)
        return self.fetch_results(n)

    # -- stage methods (device tensors) ---------------------------------------
    def remap(self, frames, want_bv=True):
        """Undistort + warp of RGB or NV12 frames -> bird's-eye RGB [n, bv_h, bv_w, 3] (None without want_bv)."""
        n = self._input(frames)
        bw, bh = self.warped_size
        bv = torch.empty((n, bh, bw, 3), dtype=torch.uint8, device=self.device) if want_bv else None
        check(self.lib.lt_remap(self._h, _ptr(frames), _ptr(bv), n, _stream_ptr(self.device)))
        return bv

    def filter_lane_points(self, bv, filter_type="bilateral", ksize_r=25, C_r=8, ksize_b=35, C_b=5,
                           mask_noise=False, ksize_noise=65, C_noise=10, noise_thresh=135):
        """bv: uint8 CUDA [n, bh, bw, 3] or None (reuse the planes of the last remap)."""
        bw, bh = self.warped_size
        n = self.n_streams if bv is None else int(bv.shape[0])
        if bv is not None and not (bv.is_cuda and bv.dtype == torch.uint8 and bv.is_contiguous() and
                                   tuple(bv.shape[1:]) == (bh, bw, 3)):
            raise ValueError("bv must be a contiguous CUDA uint8 tensor [n, %d, %d, 3]" % (bh, bw))
        mask = torch.empty((n, bh, bw), dtype=torch.uint8, device=self.device)
        check(self.lib.lt_filter_lane_points(self._h, _ptr(bv), _ptr(mask), n, _filter_code(filter_type),
                                             int(ksize_r), int(C_r), int(ksize_b), int(C_b), int(bool(mask_noise)),
                                             int(ksize_noise), int(C_noise), int(noise_thresh),
                                             _stream_ptr(self.device)))
        return mask

    def _decode_pixels(self, pixels, counts, n):
        pix = pixels.cpu().numpy().view(np.uint32)
        cnt = counts.cpu().numpy().reshape(n, 2)
        out = []
        for s in range(n):
            sides = []
            for side in range(2):
                k = int(cnt[s, side])
                if k > pix.shape[2]:
                    raise _lib.LaneTrackerError("pixel capacity exceeded: %d > %d" % (k, pix.shape[2]))
                v = pix[s, side, :k]
                sides.append(((v >> 16).astype(np.int64), (v & 0xFFFF).astype(np.int64) - 32768))
            out.append(sides)
        return out, cnt

    def sliding_window_search(self, mask, window_width, window_height, search_range, mu, no_success_limit,
                              start_slice=0.25, ignore_sides=360, ignore_bottom=30, partial=1, capacity=None):
        n = int(mask.shape[0])
        capacity = capacity or self.geometry["pixel_capacity"]
        pixels = torch.empty((n, 2, capacity), dtype=torch.int32, device=self.device)
        counts = torch.zeros((n, 2), dtype=torch.int32, device=self.device)
        cents = torch.zeros((n, 2, LT_MAX_LEVELS), dtype=torch.int32, device=self.device)
        ncents = torch.zeros((n, 2), dtype=torch.int32, device=self.device)
        det = torch.zeros((n,), dtype=torch.int32, device=self.device)
        check(self.lib.lt_sliding_window_search(
            self._h, _ptr(mask), n, int(window_width), int(window_height), int(search_range), float(mu),
            int(no_success_limit), float(start_slice), int(ignore_sides), int(ignore_bottom), float(partial),
            _ptr(pixels), capacity, _ptr(counts), _ptr(cents), _ptr(ncents), _ptr(det), _stream_ptr(self.device)))
        px, _ = self._decode_pixels(pixels, counts, n)
        c = cents.cpu().numpy()
        nc = ncents.cpu().numpy()
        cent_lists = [[list(map(int, c[s, side, :nc[s, side]])) for side in range(2)] for s in range(n)]
        return px, cent_lists, det.cpu().numpy().astype(bool)

    def band_search(self, mask, coeffs, bandwidth, ignore_bottom=30, partial=1, capacity=None):
        n = int(mask.shape[0])
        capacity = capacity or self.geometry["pixel_capacity"]
        cf = torch.as_tensor(np.asarray(coeffs, dtype=np.float64).reshape(n, 2, 3)).to(self.device)
        pixels = torch.empty((n, 2, capacity), dtype=torch.int32, device=self.device)
        counts = torch.zeros((n, 2), dtype=torch.int32, device=self.device)
        det = torch.zeros((n,), dtype=torch.int32, device=self.device)
        check(self.lib.lt_band_search(self._h, _ptr(mask), n, _ptr(cf), int(bandwidth), int(ignore_bottom),
                                      float(partial), _ptr(pixels), capacity, _ptr(counts), _ptr(det),
                                      _stream_ptr(self.device)))
        px, _ = self._decode_pixels(pixels, counts, n)
        return px, det.cpu().numpy().astype(bool)

    def fit_poly(self, pixel_sets):
        """pixel_sets: per stream [(ly, lx), (ry, rx)] integer arrays -> float64 [n, 2, 3]."""
        n = len(pixel_sets)
        cap = max(1, max(len(side[0]) for ps in pixel_sets for side in ps))
        buf = np.zeros((n, 2, cap), dtype=np.uint32)
        cnt = np.zeros((n, 2), dtype=np.int32)
        for s, ps in enumerate(pixel_sets):
            for side, (ys, xs) in enumerate(ps):
                ys = np.asarray(ys, dtype=np.int64)
                xs = np.asarray(xs, dtype=np.int64)
                buf[s, side, :len(ys)] = ((ys << 16) | (xs + 32768)).astype(np.uint32)
                cnt[s, side] = len(ys)
        d_buf = torch.as_tensor(buf.view(np.int32)).to(self.device)
        d_cnt = torch.as_tensor(cnt).to(self.device)
        fits = torch.zeros((n, 2, 3), dtype=torch.float64, device=self.device)
        check(self.lib.lt_fit_poly(self._h, _ptr(d_buf), cap, _ptr(d_cnt), n, _ptr(fits), _stream_ptr(self.device)))
        return fits.cpu().numpy()

    def check_validity(self, fits):
        f = torch.as_tensor(np.asarray(fits, dtype=np.float64).reshape(-1, 2, 3)).to(self.device)
        n = int(f.shape[0])
        valid = torch.zeros((n,), dtype=torch.int32, device=self.device)
        diffs = torch.zeros((n, 3), dtype=torch.float64, device=self.device)
        check(self.lib.lt_check_validity(self._h, _ptr(f), n, _ptr(valid), _ptr(diffs), _stream_ptr(self.device)))
        return valid.cpu().numpy().astype(bool), diffs.cpu().numpy()

    def get_poly_points(self, fits, partial=1.0):
        f = torch.as_tensor(np.asarray(fits, dtype=np.float64).reshape(-1, 2, 3)).to(self.device)
        n = int(f.shape[0])
        bh = self.warped_size[1]
        xs = torch.zeros((n, 2, bh), dtype=torch.int32, device=self.device)
        cnt = torch.zeros((n, 2), dtype=torch.int32, device=self.device)
        check(self.lib.lt_get_poly_points(self._h, _ptr(f), n, float(partial), _ptr(xs), _ptr(cnt),
                                          _stream_ptr(self.device)))
        return xs, cnt

    def draw_lane(self, frames, xs, counts):
        n = self._check_frames(frames)
        out = torch.empty_like(frames)
        check(self.lib.lt_draw_lane(self._h, _ptr(frames), _ptr(out), n, _ptr(xs), _ptr(counts),
                                    _stream_ptr(self.device)))
        return out

    def lane_metrics(self, fits, xs=None, counts=None):
        """Curve radii [n, 2] (int64, metres) and eccentricity [n] (metres) of get_curve_radius / get_eccentricity
        (lane_tracker.py:530-559) from pixel-space fits [n, 2, 3] and the polylines of ``get_poly_points``."""
        f = torch.as_tensor(np.asarray(fits, dtype=np.float64).reshape(-1, 2, 3)).to(self.device)
        n = int(f.shape[0])
        radii = torch.zeros((n, 2), dtype=torch.int64, device=self.device)
        ecc = torch.zeros((n,), dtype=torch.float64, device=self.device) if xs is not None else None
        check(self.lib.lt_lane_metrics(self._h, _ptr(f), _ptr(xs), _ptr(counts), n, _ptr(radii), _ptr(ecc),
                                       _stream_ptr(self.device)))
        return radii.cpu().numpy(), (ecc.cpu().numpy() if ecc is not None else None)

    def draw_text(self, frames, kinds, radii=None, eccentricities=None, counters=None):
        """The putText overlays of draw_lane (kind 0) / print_failure (kind 1) in place on device frames
        (lane_tracker.py:653-659, 668-672)."""
        n = self._check_frames(frames)
        k = (C.c_int32 * n)(*[int(v) for v in kinds])
        r = (C.c_int64 * n)(*[int(v) for v in (radii if radii is not None else [0] * n)])
        e = (C.c_double * n)(*[float(v) for v in (eccentricities if eccentricities is not None else [0.0] * n)])
        c = (C.c_int32 * n)(*[int(v) for v in (counters if counters is not None else [0] * n)])
        check(self.lib.lt_draw_text(self._h, _ptr(frames), n, k, r, e, c, _stream_ptr(self.device)))
        return frames

    # -- debug views ---------------------------------------------------------
    def warp_frame(self, frames):
        """``cv2.warpPerspective(img, M, warped_size)`` of raw frames (lane_tracker.py:1035) -> [n, bv_h, bv_w, 3]."""
        n = self._check_frames(frames)
        bw, bh = self.warped_size
        out = torch.empty((n, bh, bw, 3), dtype=torch.uint8, device=self.device)
        check(self.lib.lt_warp_frame(self._h, _ptr(frames), n, _ptr(out), _stream_ptr(self.device)))
        return out

    def visualize_search(self, mask, mode, left, right, new_fits, rects=None, band_fits=None, bandwidth=0, partial=1.0):
        """One search visualisation (lane_tracker.py:689-771).  mask: uint8 [bv_h, bv_w] tensor on the device;
        left / right: (y, x) integer arrays; new_fits / band_fits: [2][3]; rects: int32 [n][5] (mode 'sws')."""
        bw, bh = self.warped_size
        if tuple(mask.shape) != (bh, bw) or mask.dtype != torch.uint8 or not mask.is_contiguous():
            raise ValueError("mask must be a contiguous uint8 [%d, %d] tensor" % (bh, bw))
        v = _lib.lt_vis()
        v.mode = {"sws": 0, "bs": 1}[mode]
        packed = []
        for ys, xs in (left, right):
            ys = np.asarray(ys, dtype=np.int64)
            xs = np.asarray(xs, dtype=np.int64)
            buf = ((ys << 16) | (xs + 32768)).astype(np.uint32)
            packed.append(torch.as_tensor(buf.view(np.int32)).to(self.device) if len(buf) else None)
        v.n_left, v.n_right = len(left[0]), len(right[0])
        r = np.ascontiguousarray(rects if rects is not None else np.zeros((0, 5)), dtype=np.int32).reshape(-1, 5)
        v.n_rects, v.bandwidth, v.partial = len(r), int(bandwidth), float(partial)
        nf = np.asarray(new_fits, dtype=np.float64).reshape(2, 3)
        bf = np.asarray(band_fits if band_fits is not None else np.zeros((2, 3)), dtype=np.float64).reshape(2, 3)
        for j in range(3):
            v.left_fit[j], v.right_fit[j] = nf[0, j], nf[1, j]
            v.band_left[j], v.band_right[j] = bf[0, j], bf[1, j]
        out = torch.empty((bh, bw, 3), dtype=torch.uint8, device=self.device)
        check(self.lib.lt_visualize_search(self._h, C.byref(v), _ptr(mask), _ptr(packed[0]), _ptr(packed[1]),
                                           r.ctypes.data_as(C.c_void_p), _ptr(out), _stream_ptr(self.device)))
        return out

    def nv12_to_rgb(self, nv12, out=None):
        """Decoder output -> the RGB frames ``process`` consumes: ``cv2.cvtColor(f, cv2.COLOR_YUV2RGB_NV12)`` of every
        frame of a uint8 device tensor [n, H * 3 / 2, W] (luma plane, then interleaved U, V rows), bit-exact.  The
        reference receives RGB frames from moviepy / ffmpeg (process_video.py:42-44); a hardware decoder delivers NV12."""
        if nv12.dim() != 3 or nv12.dtype != torch.uint8 or not nv12.is_contiguous() or nv12.shape[1] % 3:
            raise ValueError("nv12_to_rgb: expected a contiguous uint8 tensor [n, H * 3 / 2, W]")
        n, h, w = int(nv12.shape[0]), int(nv12.shape[1]) * 2 // 3, int(nv12.shape[2])
        if out is None:
            out = torch.empty((n, h, w, 3), dtype=torch.uint8, device=nv12.device)
        if tuple(out.shape) != (n, h, w, 3) or not out.is_contiguous():
            raise ValueError("nv12_to_rgb: bad destination layout")
        check(self.lib.lt_nv12_to_rgb(_ptr(nv12), _ptr(out), n, w, h, _stream_ptr(self.device)))
        return out

    def resize_linear(self, src, dsize, out=None):
        """``cv2.resize(src, dsize)`` (utils.py:88) of a uint8 [h, w] or [h, w, 3] device tensor; ``out`` may be a
        view into a larger canvas (rows strided, pixels contiguous)."""
        dw, dh = int(dsize[0]), int(dsize[1])
        cn = 1 if src.dim() == 2 else int(src.shape[2])
        if out is None:
            out = torch.empty((dh, dw) if src.dim() == 2 else (dh, dw, cn), dtype=torch.uint8, device=src.device)
        if src.stride(-1) != 1 or out.stride(-1) != 1 or tuple(out.shape[:2]) != (dh, dw):
            raise ValueError("resize_linear: bad source / destination layout")
        check(self.lib.lt_resize_linear(_ptr(src), int(src.shape[1]), int(src.shape[0]), cn, int(src.stride(0)),
                                        _ptr(out), dw, dh, int(out.stride(0)), _stream_ptr(self.device)))
        return out

    # -- state / debug -------------------------------------------------------
    def get_state(self, stream_id=0):
        st = lt_state()
        bh = self.warped_size[1]
        lx = np.zeros(bh, dtype=np.int32)
        rx = np.zeros(bh, dtype=np.int32)
        check(self.lib.lt_get_state(self._h, int(stream_id), C.byref(st), lx.ctypes.data_as(C.c_void_p),
                                    rx.ctypes.data_as(C.c_void_p)))
        return st, lx[:st.n_left_avg].copy(), rx[:st.n_right_avg].copy()

    def set_state(self, stream_id, st, left_avg_x=None, right_avg_x=None):
        bh = self.warped_size[1]
        lx = np.zeros(bh, dtype=np.int32)
        rx = np.zeros(bh, dtype=np.int32)
        if left_avg_x is not None:
            lx[:len(left_avg_x)] = left_avg_x
        if right_avg_x is not None:
            rx[:len(right_avg_x)] = right_avg_x
        check(self.lib.lt_set_state(self._h, int(stream_id), C.byref(st), lx.ctypes.data_as(C.c_void_p),
                                    rx.ctypes.data_as(C.c_void_p)))

    def read_capture(self, stream_id, attempt):
        """Ordered pixel sets [(ly, lx), (ry, rx)] and centroid lists of one attempt of the last process()."""
        cap = self.geometry["pixel_capacity"]
        sides, cents = [], []
        for side in range(2):
            buf = np.zeros(cap, dtype=np.uint32)
            cnt = C.c_int32(0)
            cbuf = np.zeros(LT_MAX_LEVELS, dtype=np.int32)
            ncent = C.c_int32(0)
            check(self.lib.lt_read_capture(self._h, int(stream_id), int(attempt), side,
                                           buf.ctypes.data_as(C.c_void_p), cap, C.byref(cnt),
                                           cbuf.ctypes.data_as(C.c_void_p), C.byref(ncent)))
            if cnt.value > cap:
                raise _lib.LaneTrackerError("pixel capacity exceeded")
            v = buf[:cnt.value]
            sides.append(((v >> 16).astype(np.int64), (v & 0xFFFF).astype(np.int64) - 32768))
            cents.append([int(c) for c in cbuf[:ncent.value]])
        return sides, cents

    _DEBUG = dict(undistort_map=0, bv_map=1, overlay_map=2, r_plane=3, b_plane=4, r_tophat=5, b_tophat=6,
                  mask=7, merged=8, lane_rows=9, draw_lane_rows=12)

    def debug_read(self, what, stream_id=0):
        code = self._DEBUG[what]
        w, h = self.img_size
        bw, bh = self.warped_size
        if code in (0, 2):
            out = np.zeros((h, w, 2), dtype=np.int32)
        elif code == 1:
            out = np.zeros((bh, bw, 2), dtype=np.int32)
        elif code in (9, 12):
            out = np.zeros((bh, 2), dtype=np.int32)
        else:
            out = np.zeros((bh, bw), dtype=np.uint8)
        check(self.lib.lt_debug_read(self._h, code, int(stream_id), out.ctypes.data_as(C.c_void_p), out.nbytes))
        return out


class GraphedProcess:
    """``process_async`` of a fixed batch shape captured once into a CUDA graph and replayed per frame: the chain
    of ~20 small launches costs one launch.  Pays off for few streams (one stream: 0.25 -> 0.21 ms per frame);
    ``lt_process`` only enqueues kernels (and forks/joins its side stream with events), so it is capturable.

        g = GraphedProcess(tracker, n_streams)          # static device buffers g.frames / g.out
        g.frames.copy_(batch, non_blocking=True); g.replay(); results = g.fetch_results()

    With ``profiles`` (n profile indices, see ``BatchedLaneTracker.set_profile``) frame i uses profile profiles[i].
    The graph holds the profile indices and the profile table as they stood at capture time: a later ``set_profile``
    does not reach it (capture a new ``GraphedProcess`` instead).  With ``cameras`` (n camera indices, see
    ``BatchedLaneTracker.set_camera``) frame i comes from camera cameras[i]; the graph then holds the camera tables and
    buffers of capture time, and ``replay`` raises RuntimeError after a later ``set_camera``.
    """

    def __init__(self, tracker, n=None, overlay=True, params=None, frame_format="rgb", profiles=None, cameras=None):
        """frame_format 'nv12': ``self.frames`` is NV12 [n, H * 3 / 2, W]; ``self.out`` stays RGB."""
        if frame_format not in _FRAME_FORMATS:
            raise ValueError("frame_format must be 'rgb' or 'nv12'")
        BatchedLaneTracker._no_params_with_profiles(profiles, params, {})
        self.t = tracker
        n = tracker.n_streams if n is None else int(n)
        dev = tracker.device
        w, h = tracker.img_size
        self.n = n
        shape = (n, h * 3 // 2, w) if frame_format == "nv12" else (n, h, w, 3)
        self.frames = torch.zeros(shape, dtype=torch.uint8, device=dev)
        self.out = torch.empty((n, h, w, 3), dtype=torch.uint8, device=dev) if overlay else None
        self.results_dev = torch.zeros(n * RESULT_DTYPE.itemsize, dtype=torch.uint8, device=dev)
        self.params = params if params is not None or profiles is not None else make_params()
        self.profiles = None if profiles is None else np.array(profiles, dtype=np.int64)
        tracker._check_profiles(self.profiles, n)
        self.cameras = None if cameras is None else np.array(cameras, dtype=np.int64)
        tracker._check_cameras(self.cameras, n)
        self.camera_epoch = tracker.camera_epoch
        # first-use initialisation (module load, shared-memory attributes) cannot happen inside a capture: run the
        # chain once for real on a side stream, with the state records of its streams exported before and imported
        # after it on that stream
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            saved = tracker.export_states(range(n))
            tracker.process_async(self.frames, self.out, params=self.params, results_dev=self.results_dev,
                                  profiles=self.profiles, cameras=self.cameras)
            tracker.import_states(range(n), saved, check=False)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, stream=side):
            tracker.process_async(self.frames, self.out, params=self.params, results_dev=self.results_dev,
                                  profiles=self.profiles, cameras=self.cameras)
        torch.cuda.current_stream(dev).wait_stream(side)

    def replay(self):
        """Enqueue one frame per stream (read from ``self.frames``) on the current stream."""
        if self.cameras is not None and self.t.camera_epoch != self.camera_epoch:
            raise RuntimeError("set_camera ran after this graph was captured with cameras: the graph holds the camera "
                               "tables and buffers it replaced; capture a new GraphedProcess")
        self.graph.replay()

    def fetch_results(self):
        return self.t.fetch_results(self.n, self.results_dev)


class DevicePipeline:
    """Two batches in flight on the device: the stateless front half of batch k+1 (undistort, warp, filter) runs on
    one CUDA stream while the stateful back half of batch k (searches, state machine, overlay) runs on another.
    The back half is a chain of small kernels (one CTA per stream) that leaves most SMs idle; the front half of the
    next batch fills them.  Results are those of sequential ``process`` calls: back halves execute in submission
    order on one stream, and a buffer set is reused only after the back half that read it has finished.

        pipe = DevicePipeline(tracker)
        for frames, out in batches:            # CUDA tensors; produced on the current stream
            done = pipe.submit(frames, out)    # torch.cuda.Event: out / results of this batch are complete
        pipe.join()                            # the current stream waits for everything submitted

    ``submit(frames, out, ids=...)`` advances the listed streams only (see ``BatchedLaneTracker.process_async``);
    results stay in batch order.  ``frames`` may be RGB or NV12 (``out`` is RGB either way), batch by batch.
    ``submit(..., profiles=...)`` gives frame i parameter profile profiles[i] (``BatchedLaneTracker.set_profile``)
    instead of the pipeline's ``params``; ``submit(..., cameras=...)`` says that frame i comes from camera cameras[i]
    (``BatchedLaneTracker.set_camera``).  ``submit(frames, out, ids=..., sequence=True)`` lets ids repeat: the frames
    of one stream are its consecutive frames, in batch order.  One video, 64 frames per batch::

        for chunk, out in chunks:              # consecutive frames of one video, up to n_streams per chunk
            pipe.submit(chunk, out, ids=[0] * len(chunk), sequence=True)

    ``submit(..., starts=...)`` flags the frames that begin a new video on their stream (see
    ``BatchedLaneTracker.process_async``): the start is enqueued on the back stream, after every back half submitted
    before and before this batch's, so the pipeline need not be drained.  ``export_states`` / ``import_states`` move
    state records on the back stream in the same order.
    """

    def __init__(self, tracker, params=None):
        self.t = tracker
        self.params = params if params is not None else make_params()
        dev = tracker.device
        self.s_front = torch.cuda.Stream(dev)
        self.s_back = torch.cuda.Stream(dev)
        self._k = 0
        self._back_done = [None, None]          # per buffer set: event of the last back half that used it
        self._last = None
        self.results_dev = [torch.zeros(tracker.n_streams * RESULT_DTYPE.itemsize, dtype=torch.uint8, device=dev)
                            for _ in range(2)]

    def submit(self, frames, out=None, ids=None, profiles=None, cameras=None, sequence=False, starts=None):
        dev = self.t.device
        n = self.t._frame_format(frames)[0]
        self.t._check_sequence(sequence, ids, profiles, cameras)
        self.t._check_ids(ids, n, repeats=sequence)    # refuse bad frames / ids / profiles / cameras before anything is enqueued
        self.t._check_profiles(profiles, n)
        self.t._check_cameras(cameras, n)
        self.t._check_starts(starts, ids, n, sequence)
        params = self.params if profiles is None else None
        k, bs = self._k, self._k & 1
        ready = torch.cuda.Event()
        ready.record(torch.cuda.current_stream(dev))            # frames (and out) belong to the caller until here
        with torch.cuda.stream(self.s_front):
            self.s_front.wait_event(ready)
            if self._back_done[bs] is not None:
                self.s_front.wait_event(self._back_done[bs])    # set `bs` is free again
            self.t.process_front_async(frames, bs, params=params, profiles=profiles, cameras=cameras)
            front_done = torch.cuda.Event()
            front_done.record(self.s_front)
        with torch.cuda.stream(self.s_back):
            self.s_back.wait_event(front_done)
            self.s_back.wait_event(ready)
            self.t.process_back_async(frames, out, bs, params=params, results_dev=self.results_dev[bs], ids=ids,
                                      profiles=profiles, cameras=cameras, sequence=sequence, starts=starts)
            done = torch.cuda.Event()
            done.record(self.s_back)
        self._back_done[bs] = done
        self._last = done
        self._k = k + 1
        return done

    def export_states(self, ids):
        """State records of streams ``ids`` as they stand after every batch submitted so far (and before any submitted
        later), gathered on the back stream -> (uint8 CUDA tensor [n, record_bytes], torch.cuda.Event after which it
        is complete)."""
        return _on_stream(self.t, self.s_back, lambda: self.t.export_states(ids))

    def import_states(self, ids, records):
        """Write state records into slots ``ids`` on the back stream, after every batch submitted so far and before any
        submitted later.  ``records`` are read after the work enqueued so far on the current stream.  -> (int32 CUDA
        status tensor [n], see ``BatchedLaneTracker.import_states``; torch.cuda.Event after which it is complete)."""
        return _on_stream(self.t, self.s_back, lambda: self.t.import_states(ids, records, check=False), records)

    def last_results_dev(self):
        """Device buffer holding the lt_result records of the most recently submitted batch."""
        return self.results_dev[(self._k - 1) & 1]

    def join(self):
        if self._last is not None:
            torch.cuda.current_stream(self.t.device).wait_event(self._last)

    def fetch_results(self, n=None):
        """Results of the most recently submitted batch as a structured array (synchronises)."""
        self.join()
        return self.t.fetch_results(n, self.last_results_dev())


def _on_stream(tracker, stream, fn, reads=None):
    """Run ``fn`` (a state-record call of ``tracker``) on a pipeline's back stream, after the work enqueued so far on
    the current stream (``reads``, a tensor it reads, is kept alive for that stream) -> (fn's tensor, its event)."""
    dev = tracker.device
    ready = torch.cuda.Event()
    ready.record(torch.cuda.current_stream(dev))
    with torch.cuda.stream(stream):
        stream.wait_event(ready)
        if reads is not None:
            reads.record_stream(stream)
        t = fn()
        done = torch.cuda.Event()
        done.record(stream)
    return t, done


def _rows_minus(rows, covered):
    """Row range `rows` minus the range `covered` (both half-open): up to two non-empty segments."""
    (ta, tb), (a, b) = rows, covered
    if tb <= ta:
        return []
    if b <= a:
        return [(ta, tb)]
    return [seg for seg in ((ta, min(tb, a)), (max(ta, b), tb)) if seg[1] > seg[0]]


class HostPipeline:
    """Host-to-host streaming through a ``BatchedLaneTracker``: pinned host frames in, annotated frames and
    result records out, with the H2D copy of batch k+1, the kernels of batch k and the D2H copy of batch k-1
    overlapped on three CUDA streams (`depth` buffer sets in flight).  Batches are processed in submission
    order, so per-stream tracking state evolves exactly as with sequential ``process`` calls.

        pipe = HostPipeline(tracker)
        for batch in batches:                 # pinned uint8 [n, H, W, 3]
            pipe.submit(batch)
            for out, results in pipe.ready(): ...   # finished batches, oldest first
        for out, results in pipe.drain(): ...

    ``submit(batch, ids=...)`` advances the listed streams only (see ``BatchedLaneTracker.process_async``); the
    frames and records of a finished batch are in batch order.  ``submit(batch, profiles=...)`` gives frame i
    parameter profile profiles[i] (``BatchedLaneTracker.set_profile``) instead of the pipeline's ``params``, and
    ``submit(batch, cameras=...)`` says that frame i comes from camera cameras[i] (``BatchedLaneTracker.set_camera``).
    ``submit(batch, ids=..., sequence=True)`` lets ids repeat: the frames of one stream are its consecutive frames, in
    batch order (``pipe.submit(chunk, ids=[0] * len(chunk), sequence=True)`` for one video).  ``submit(batch,
    starts=...)`` flags the frames that begin a new video on their stream, and ``export_states`` / ``import_states``
    move state records, all in submission order on the stream of the back halves (see ``DevicePipeline``).
    """

    def __init__(self, tracker, depth=3, overlay=True, params=None, inplace=False, frame_format="rgb"):
        """inplace=True: annotate the caller's pinned frames in place.  Only the frame rows the tracker reads
        (geometry['source_rows'] + overlay rows) go host->device and only the rows the overlay can change
        (geometry['overlay_rows']) come back, written into the submitted tensor; every other row of the frame is
        already identical to the annotated frame, so the host ends up with the same image as overlay mode while
        about a third of the bytes cross PCIe.

        frame_format='nv12': submitted batches are pinned NV12 [n, H * 3 / 2, W], as video decoders deliver them.
        With overlay=True whole NV12 frames go host->device and whole annotated RGB frames come back; with
        overlay=False only the rows the tracker reads (geometry['source_rows']) and the chroma rows that cover them
        go host->device.  inplace is RGB only (an RGB annotation cannot be written into NV12 frames)."""
        if frame_format not in _FRAME_FORMATS:
            raise ValueError("frame_format must be 'rgb' or 'nv12'")
        self.t = tracker
        self.depth = int(depth)
        self.overlay = overlay
        self.inplace = bool(inplace)
        self.nv12 = frame_format == "nv12"
        if self.inplace and not overlay:
            raise ValueError('inplace needs overlay=True')
        if self.inplace and self.nv12:
            raise ValueError("inplace annotation needs RGB frames: NV12 frames are annotated into separate RGB frames")
        self.rows_text = tracker.text_rows if tracker.text_enabled else (0, 0)   # putText rows: read and rewritten
        self.params = params if params is not None else make_params()
        dev = tracker.device
        w, h = tracker.img_size
        S = tracker.n_streams
        # H2D, front half (stateless kernels), back half (searches, state, overlay), D2H: four streams, so that the
        # front half of batch k+1 also fills the SMs the small back-half kernels of batch k leave idle
        self.s_in, self.s_front, self.s_run, self.s_out = (torch.cuda.Stream(dev) for _ in range(4))
        self._k = 0
        self._set_free = [None, None]   # per intermediate buffer set: event of the last back half that read it
        self.slots = []
        for _ in range(self.depth):
            self.slots.append(dict(
                d_in=torch.empty((S, h * 3 // 2, w) if self.nv12 else (S, h, w, 3), dtype=torch.uint8, device=dev),
                d_out=torch.empty((S, h, w, 3), dtype=torch.uint8, device=dev) if (overlay and not inplace) else None,
                d_res=torch.zeros(S * RESULT_DTYPE.itemsize, dtype=torch.uint8, device=dev),
                h_out=torch.empty((S, h, w, 3), dtype=torch.uint8).pin_memory() if (overlay and not inplace) else None,
                h_res=torch.zeros(S * RESULT_DTYPE.itemsize, dtype=torch.uint8).pin_memory(),
                e_in=torch.cuda.Event(), e_run=torch.cuda.Event(), e_out=torch.cuda.Event(), n=0, busy=False))
        self.head = 0          # next slot to submit into
        self.tail = 0          # oldest slot in flight
        self.inflight = 0

    @property
    def rows_in(self):
        """Frame rows the partial host->device transfers move: over camera 0 and every camera set, so that any batch
        is covered (set_camera may run between submissions)."""
        src, ov = self.t.rows_any_camera()
        if self.nv12:       # the fused variant refuses NV12: the undistort reads exactly the source rows
            return src
        h_img = self.t.img_size[1]     # +-2 rows of slack: the fused remap variant samples the raw frame directly
        return max(0, min(src[0], ov[0]) - 2), min(h_img, max(src[1], ov[1]) + 2)

    @property
    def rows_out(self):
        """Frame rows the lane overlay can change, over camera 0 and every camera set: what inplace mode copies back."""
        return self.t.rows_any_camera()[1]

    def submit(self, host_frames, ids=None, profiles=None, cameras=None, sequence=False, starts=None):
        if self.inflight == self.depth:
            raise RuntimeError("pipeline full: collect a finished batch first")
        if not (host_frames.dtype == torch.uint8 and host_frames.is_pinned() and host_frames.is_contiguous()):
            raise ValueError("host_frames must be a contiguous pinned uint8 tensor")
        sl = self.slots[self.head]
        n = int(host_frames.shape[0])
        if host_frames.shape[1:] != sl["d_in"].shape[1:] or not 1 <= n <= self.t.n_streams:
            raise ValueError("host_frames must be %s [n, %s] with 1 <= n <= %d, got %s"
                             % ("NV12" if self.nv12 else "RGB", ", ".join(map(str, sl["d_in"].shape[1:])),
                                self.t.n_streams, list(host_frames.shape)))
        self.t._check_sequence(sequence, ids, profiles, cameras)
        self.t._check_ids(ids, n, repeats=sequence)      # refuse bad ids / profiles / cameras before anything is enqueued
        self.t._check_profiles(profiles, n)
        self.t._check_cameras(cameras, n)
        self.t._check_starts(starts, ids, n, sequence)
        params = self.params if profiles is None else None
        rows_in, rows_out = self.rows_in, self.rows_out
        sl["n"] = n
        with torch.cuda.stream(self.s_in):
            self.s_in.wait_event(sl["e_run"])            # the kernels that last read this input buffer are done
            if self.inplace:
                a, b = rows_in
                self.t.copy_rows(sl["d_in"], host_frames, a, b, True)
                for ta, tb in _rows_minus(self.rows_text, (a, b)):      # text rows outside the rows already sent
                    self.t.copy_rows(sl["d_in"], host_frames, ta, tb, True)
                sl["frames"] = host_frames
            elif self.nv12 and not self.overlay:
                self.t.copy_rows(sl["d_in"], host_frames, rows_in[0], rows_in[1], True)
            else:
                sl["d_in"][:n].copy_(host_frames, non_blocking=True)
            sl["e_in"].record(self.s_in)
        bs = self._k & 1
        self._k += 1
        with torch.cuda.stream(self.s_front):
            self.s_front.wait_event(sl["e_in"])
            if self._set_free[bs] is not None:
                self.s_front.wait_event(self._set_free[bs])
            self.t.process_front_async(sl["d_in"][:n], bs, params=params, profiles=profiles, cameras=cameras)
            e_front = torch.cuda.Event()
            e_front.record(self.s_front)
        with torch.cuda.stream(self.s_run):
            self.s_run.wait_event(e_front)
            self.s_run.wait_event(sl["e_out"])           # the previous D2H out of this output buffer is done
            d_out = sl["d_in"][:n] if self.inplace else (sl["d_out"][:n] if self.overlay else None)
            self.t.process_back_async(sl["d_in"][:n], d_out, bs, params=params, results_dev=sl["d_res"], ids=ids,
                                      profiles=profiles, cameras=cameras, sequence=sequence, starts=starts)
            sl["e_run"].record(self.s_run)
        self._set_free[bs] = sl["e_run"]
        with torch.cuda.stream(self.s_out):
            self.s_out.wait_event(sl["e_run"])
            if self.inplace:
                a, b = rows_out
                if b > a:
                    self.t.copy_rows(host_frames, sl["d_in"][:n], a, b, False)
                for ta, tb in _rows_minus(self.rows_text, (a, b)):      # text rows outside the rows already fetched
                    self.t.copy_rows(host_frames, sl["d_in"][:n], ta, tb, False)
            elif self.overlay:
                sl["h_out"][:n].copy_(sl["d_out"][:n], non_blocking=True)
            sl["h_res"].copy_(sl["d_res"], non_blocking=True)
            sl["e_out"].record(self.s_out)
        sl["busy"] = True
        self.head = (self.head + 1) % self.depth
        self.inflight += 1

    def export_states(self, ids):
        """As ``DevicePipeline.export_states``, on the stream of the back halves."""
        return _on_stream(self.t, self.s_run, lambda: self.t.export_states(ids))

    def import_states(self, ids, records):
        """As ``DevicePipeline.import_states``, on the stream of the back halves."""
        return _on_stream(self.t, self.s_run, lambda: self.t.import_states(ids, records, check=False), records)

    def _collect(self, block):
        sl = self.slots[self.tail]
        if not sl["busy"]:
            return None
        if not block and not sl["e_out"].query():
            return None
        sl["e_out"].synchronize()
        n = sl["n"]
        res = sl["h_res"][:n * RESULT_DTYPE.itemsize].numpy().view(RESULT_DTYPE)
        out = sl.pop("frames") if self.inplace else (sl["h_out"][:n] if self.overlay else None)
        sl["busy"] = False
        self.tail = (self.tail + 1) % self.depth
        self.inflight -= 1
        return out, res

    def ready(self):
        """Finished batches (views into the pipeline's pinned buffers: consume before the slot is reused)."""
        while True:
            if self.inflight < self.depth:
                got = self._collect(block=False)
            else:
                got = self._collect(block=True)         # make room for the next submit
            if got is None:
                return
            yield got

    def drain(self):
        while self.inflight:
            yield self._collect(block=True)


class LaneTracker:
    """Drop-in for the reference ``LaneTracker`` (same constructor, lane_tracker.py:101).

    NumPy arrays in, NumPy arrays out; every computation runs on the GPU.  One deliberate difference from the
    reference: ``process``, ``draw_lane`` and ``print_failure`` never modify the caller's ``img`` (the reference's
    ``cv2.putText`` calls draw into the input array, lane_tracker.py:653-659, 668-672, and ``print_failure`` returns that
    same array); the returned frame is identical.  The debug views (``visualize_search``, ``split_view``) are rendered on
    the device from the buffers of the last ``process`` call.
    """

    # the second attempt's hard-coded search parameters (lane_tracker.py:1081-1099); the debug views of a frame
    # that went to attempt 2 are drawn with these, as in the reference
    _ATTEMPT2 = dict(window_width=30, window_height=40, ignore_bottom=30, bandwidth=30, partial=1.0)

    def __init__(self, img_size, warped_size, cam_matrix, dist_coeffs, warp_matrices, mpp_conversion,
                 n_fail=8, n_reset=4, n_average=2, print_frame_count=False, device=None):
        self.img_size = img_size
        self.warped_size = warped_size
        self.cam_matrix = cam_matrix
        self.dist_coeffs = dist_coeffs
        self.M, self.Minv = warp_matrices[0], warp_matrices[1]
        self.mppv, self.mpph = mpp_conversion[0], mpp_conversion[1]
        self.n_reset, self.n_fail, self.n_average = n_reset, n_fail, n_average
        self.print_frame_count = print_frame_count
        self._bt = BatchedLaneTracker(1, img_size, warped_size, cam_matrix, dist_coeffs, warp_matrices,
                                      mpp_conversion, n_fail, n_reset, n_average, print_frame_count, device)
        self._bt.set_capture(True)
        dev = self._bt.device
        w, h = self._bt.img_size
        self._in_host = torch.empty((1, h, w, 3), dtype=torch.uint8).pin_memory()
        self._out_host = torch.empty((1, h, w, 3), dtype=torch.uint8).pin_memory()
        self._in_dev = torch.empty((1, h, w, 3), dtype=torch.uint8, device=dev)
        self._out_dev = torch.empty((1, h, w, 3), dtype=torch.uint8, device=dev)
        # state attributes, lane_tracker.py:139-176
        self.last_detection = n_reset + 1
        self.detected_pixels = False
        self.valid_lane_lines = False
        self.left_fit_coeffs, self.right_fit_coeffs = [], []
        self.last_left_coeffs = self.last_right_coeffs = None
        self.left_avg_coeffs = self.right_avg_coeffs = None
        self.left_avg_y = np.array([])
        self.left_avg_x = np.array([])
        self.right_avg_y = np.array([])
        self.right_avg_x = np.array([])
        self.left_y = self.left_x = self.right_y = self.right_x = None
        self.left_window_centroids = self.right_window_centroids = None
        self.left_curve_radius = self.right_curve_radius = None
        self.average_curve_radius = None
        self.average_curve_radii = []
        self.eccentricity = None
        self.counter = 0
        self.success = 0
        self.last_result = None

    def get_success_ratio(self):
        return self.success / self.counter, self.success, self.counter

    def set_validity(self, **kw):
        """Extension: the check_validity windows the reference hard-codes (lane_tracker.py:588-593, 617)."""
        self._bt.set_validity(**kw)

    # ------------------------------------------------------------ helpers
    def _upload(self, arr, shape):
        a = np.ascontiguousarray(arr, dtype=np.uint8)
        if a.shape != shape:
            raise ValueError("expected an array of shape %s, got %s" % (shape, a.shape))
        return torch.from_numpy(a).to(self._bt.device)

    def _sync_state(self, res):
        st, lx, rx = self._bt.get_state(0)
        bh = self._bt.warped_size[1]
        self.last_detection = int(st.last_detection)
        self.counter, self.success = int(st.counter), int(st.success)
        self.left_fit_coeffs = [np.array([]) if st.ring_empty[i] else np.array(st.ring_left[i][:])
                                for i in range(st.ring_len)]
        self.right_fit_coeffs = [np.array([]) if st.ring_empty[i] else np.array(st.ring_right[i][:])
                                 for i in range(st.ring_len)]
        if st.has_last:
            self.last_left_coeffs = np.array(st.last_left[:])
            self.last_right_coeffs = np.array(st.last_right[:])
        if st.has_avg:
            self.left_avg_coeffs = np.array(st.left_avg[:])
            self.right_avg_coeffs = np.array(st.right_avg[:])
            self.left_avg_x = lx.astype(np.int64)
            self.right_avg_x = rx.astype(np.int64)
            self.left_avg_y = np.arange(bh - len(lx), bh, dtype=np.int64)
            self.right_avg_y = np.arange(bh - len(rx), bh, dtype=np.int64)
            self.average_curve_radius = int(st.average_curve_radius)
            self.eccentricity = float(st.eccentricity)
        self.average_curve_radii = [int(st.radii[i]) for i in range(st.radii_len)]
        if res is not None:
            self.detected_pixels = bool(res["detected_pixels"])
            self.valid_lane_lines = bool(res["valid_lane_lines"])
            if res["valid_lane_lines"]:
                self.left_curve_radius = int(res["left_curve_radius"])
                self.right_curve_radius = int(res["right_curve_radius"])
            # pixel sets / centroids are only replaced by a search that found pixels on both sides
            for attempt in range(int(res["attempts"])):
                det = res["first_detected"] if attempt == 0 else res["detected_pixels"]
                if int(res["attempts"]) == 1:
                    det = res["detected_pixels"]
                if det:
                    sides, cents = self._bt.read_capture(0, attempt)
                    (self.left_y, self.left_x), (self.right_y, self.right_x) = sides
                    if len(cents[0]) or len(cents[1]):
                        self.left_window_centroids, self.right_window_centroids = cents

    # ------------------------------------------------------------ methods
    def process(self, img, ksize_r=15, C_r=8, ksize_b=35, C_b=5, filter_type="bilateral", mask_noise=False,
                noise_thresh=140, ksize_noise=65, C_noise=10, window_width=30, window_height=40,
                search_range=20, mu=0.1, no_success_limit=8, start_slice=0.25, ignore_sides=360,
                ignore_bottom=30, bandwidth=25, partial=1.0, n_tries=2, visualize_search=False,
                split_view=False, diagnostics=False):
        """lane_tracker.py:876-1209.  Returns the annotated frame (new array); with ``visualize_search`` the tuple
        (frame, search visualisation), with ``split_view`` the three-panel canvas (lane_tracker.py:1161-1173).
        Unlike the reference, the text overlays are NOT also written into the caller's ``img`` (its in-place
        ``cv2.putText``, lane_tracker.py:653-659 / 668-672): the input array is left untouched."""
        debug = bool(visualize_search | split_view)
        band_coeffs = (self.last_left_coeffs, self.last_right_coeffs)      # what a band search of this frame uses
        p = make_params(ksize_r=ksize_r, C_r=C_r, ksize_b=ksize_b, C_b=C_b, filter_type=filter_type,
                        mask_noise=mask_noise, noise_thresh=noise_thresh, ksize_noise=ksize_noise,
                        C_noise=C_noise, window_width=window_width, window_height=window_height,
                        search_range=search_range, mu=mu, no_success_limit=no_success_limit,
                        start_slice=start_slice, ignore_sides=ignore_sides, ignore_bottom=ignore_bottom,
                        bandwidth=bandwidth, partial=partial, n_tries=n_tries)
        w, h = self._bt.img_size
        a = np.asarray(img)
        if a.shape != (h, w, 3) or a.dtype != np.uint8:
            raise ValueError("img must be uint8 [%d, %d, 3]" % (h, w))
        need = (2 * max(int(bandwidth), 30) - 1) * self._bt.warped_size[1]   # a band-search row: < 2 * bandwidth pixels
        if need > self._bt.geometry["pixel_capacity"]:
            self._bt.set_pixel_capacity(need)
        self._in_host[0].numpy()[...] = a
        self._in_dev.copy_(self._in_host, non_blocking=True)
        warped = self._bt.warp_frame(self._in_dev)[0] if debug else None   # lane_tracker.py:1035 (raw frame)
        self._bt.process_async(self._in_dev, self._out_dev, params=p)
        self._out_host.copy_(self._out_dev, non_blocking=True)
        res = self._bt.fetch_results(1)[0]
        self.last_result = res
        self._sync_state(res)
        if diagnostics:
            print("attempts=%d mode=%s detected=%s valid=%s" % (res["attempts"], "bs" if res["search_mode"] else "sws",
                                                                bool(res["detected_pixels"]), bool(res["valid_lane_lines"])))
        if not debug:
            return self._out_host[0].numpy().copy()
        # lane_tracker.py:1130-1138: the view of the LAST attempt, drawn with that attempt's parameters
        q = dict(window_width=window_width, window_height=window_height, ignore_bottom=ignore_bottom,
                 bandwidth=bandwidth, partial=partial)
        if int(res["attempts"]) == 2:
            q = self._ATTEMPT2
        mask = torch.from_numpy(self._bt.debug_read("mask", 0)).to(self._bt.device)
        if res["detected_pixels"]:
            lf, rf = np.array(res["left_fit"]), np.array(res["right_fit"])
            if res["search_mode"] == 0:
                vis = self._vis_sws(mask, lf, rf, q["window_width"], q["window_height"], q["ignore_bottom"])
            else:
                vis = self._vis_bs(mask, lf, rf, q["bandwidth"], q["partial"], band_coeffs)
        else:
            vis = mask                                                     # 2-D, as in the reference
        if visualize_search:
            return self._out_host[0].numpy().copy(), vis.cpu().numpy()
        return self._triple_split_view_dev([self._out_dev[0], warped, vis]).cpu().numpy()

    # ------------------------------------------------------------ debug views
    def window_mask(self, img, window_width, window_height, center, level, ignore_bottom):
        """lane_tracker.py:675-687."""
        output = np.zeros_like(img)
        r0, r1, c0, c1 = self._window_rect(img.shape[:2], window_width, window_height, center, level, ignore_bottom)
        output[r0:r1, c0:c1] = 1
        return output

    @staticmethod
    def _window_rect(shape, window_width, window_height, center, level, ignore_bottom):
        H, W = shape
        img_height = H - ignore_bottom
        rows = slice(int(img_height - (level + 1) * window_height), int(img_height - level * window_height)).indices(H)
        cols = slice(max(int(center - window_width / 2), 0), min(int(center + window_width / 2), W)).indices(W)
        return rows[0], max(rows[1], rows[0]), cols[0], max(cols[1], cols[0])

    def _vis_sws(self, mask, left_fit, right_fit, window_width, window_height, ignore_bottom):
        bw, bh = self._bt.warped_size
        rects = []
        for side, cents in enumerate((self.left_window_centroids, self.right_window_centroids)):
            for level, c in enumerate(cents):
                rects.append(self._window_rect((bh, bw), window_width, window_height, c, level, ignore_bottom) + (side,))
        return self._bt.visualize_search(mask, "sws", (self.left_y, self.left_x), (self.right_y, self.right_x),
                                         [left_fit, right_fit], rects=np.array(rects, dtype=np.int32).reshape(-1, 5))

    def _vis_bs(self, mask, left_fit, right_fit, bandwidth, partial, band_coeffs):
        return self._bt.visualize_search(mask, "bs", (self.left_y, self.left_x), (self.right_y, self.right_x),
                                         [left_fit, right_fit], band_fits=band_coeffs, bandwidth=bandwidth,
                                         partial=partial)

    def visualize_sliding_window_search(self, binary_img, left_fit_coeffs, right_fit_coeffs, window_width,
                                        window_height, ignore_bottom):
        """lane_tracker.py:689-729 (uses left/right_window_centroids and the lane pixel sets of the last search)."""
        return self._vis_sws(self._mask_dev(binary_img)[0], left_fit_coeffs, right_fit_coeffs, window_width,
                             window_height, ignore_bottom).cpu().numpy()

    def visualize_band_search(self, binary_img, left_fit_coeffs, right_fit_coeffs, bandwidth, partial):
        """lane_tracker.py:731-771 (the band is drawn around last_left_coeffs / last_right_coeffs)."""
        return self._vis_bs(self._mask_dev(binary_img)[0], left_fit_coeffs, right_fit_coeffs, bandwidth, partial,
                            (self.last_left_coeffs, self.last_right_coeffs)).cpu().numpy()

    def _triple_split_view_dev(self, images):
        from .utils import create_split_view
        img1_size = (int(images[0].shape[1]), int(images[0].shape[0]))
        img2_size = (int(images[1].shape[1]), int(images[1].shape[0]))
        positions = [(0, 0), (0, img1_size[1]), (round(0.5 * img1_size[0]), img1_size[1])]
        scale_factor = img2_size[0] / (0.5 * img1_size[0])
        scaled_size = (round(img2_size[0] / scale_factor), round(img2_size[1] / scale_factor))
        target_size = (img1_size[0], img1_size[1] + scaled_size[1])
        return create_split_view(target_size, images, positions, [img1_size, scaled_size, scaled_size],
                                 _device=self._bt.device, _numpy=False)

    def triple_split_view(self, images):
        """lane_tracker.py:773-793."""
        dev = [torch.as_tensor(np.ascontiguousarray(im, dtype=np.uint8)).to(self._bt.device) for im in images]
        return self._triple_split_view_dev(dev).cpu().numpy()

    def find_lane_points(self, img, ksize_r=15, C_r=8, ksize_b=35, C_b=5, filter_type="bilateral",
                         mask_noise=True, noise_thresh=140, ksize_noise=65, C_noise=10, window_width=30,
                         window_height=40, search_range=20, mu=0.1, no_success_limit=8, start_slice=0.25,
                         ignore_sides=360, ignore_bottom=30, bandwidth=30, partial=0.5, diagnostics=False):
        """lane_tracker.py:795-874."""
        w, h = self._bt.img_size
        frames = self._upload(img, (h, w, 3)).unsqueeze(0)
        self._bt.remap(frames, want_bv=False)
        mask = self._bt.filter_lane_points(None, filter_type, ksize_r, C_r, ksize_b, C_b, mask_noise,
                                           ksize_noise, C_noise, noise_thresh)[:1]
        if self.last_detection > self.n_reset:
            self._sws(mask, window_width, window_height, search_range, mu, no_success_limit, start_slice,
                      ignore_sides, ignore_bottom, partial)
            mode = "sws"
        else:
            self._bs(mask, bandwidth, ignore_bottom, partial)
            mode = "bs"
        return mask[0].cpu().numpy(), mode

    def filter_lane_points(self, img, filter_type="bilateral", ksize_r=25, C_r=8, ksize_b=35, C_b=5,
                           mask_noise=False, ksize_noise=65, C_noise=10, noise_thresh=135):
        """lane_tracker.py:183-240: bird's-eye RGB image -> binary mask {0,255}."""
        _filter_code(filter_type)
        bw, bh = self._bt.warped_size
        bv = self._upload(img, (bh, bw, 3)).unsqueeze(0)
        mask = self._bt.filter_lane_points(bv, filter_type, ksize_r, C_r, ksize_b, C_b, mask_noise,
                                           ksize_noise, C_noise, noise_thresh)
        return mask[0].cpu().numpy()

    def _mask_dev(self, img):
        bw, bh = self._bt.warped_size
        if isinstance(img, torch.Tensor):
            return img
        return self._upload(img, (bh, bw)).unsqueeze(0)

    def _sws(self, mask, *a):
        px, cents, det = self._bt.sliding_window_search(mask, *a)
        self.detected_pixels = bool(det[0])
        if det[0]:
            (self.left_y, self.left_x), (self.right_y, self.right_x) = px[0]
            self.left_window_centroids, self.right_window_centroids = cents[0]

    def _bs(self, mask, bandwidth, ignore_bottom, partial):
        coeffs = np.stack([self.last_left_coeffs, self.last_right_coeffs])[None]
        px, det = self._bt.band_search(mask, coeffs, bandwidth, ignore_bottom, partial)
        self.detected_pixels = bool(det[0])
        if det[0]:
            (self.left_y, self.left_x), (self.right_y, self.right_x) = px[0]

    def sliding_window_search(self, img, window_width, window_height, search_range, mu, no_success_limit,
                              start_slice=0.25, ignore_sides=360, ignore_bottom=30, partial=1, diagnostics=False):
        """lane_tracker.py:242-447."""
        self._sws(self._mask_dev(img), window_width, window_height, search_range, mu, no_success_limit,
                  start_slice, ignore_sides, ignore_bottom, partial)

    def band_search(self, img, bandwidth, ignore_bottom=30, partial=1, diagnostics=False):
        """lane_tracker.py:449-500."""
        if self.last_left_coeffs is None:
            raise TypeError("band_search needs last_left_coeffs / last_right_coeffs from a previous valid fit")
        self._bs(self._mask_dev(img), bandwidth, ignore_bottom, partial)

    def fit_poly(self):
        """lane_tracker.py:502-509."""
        f = self._bt.fit_poly([[(self.left_y, self.left_x), (self.right_y, self.right_x)]])
        return f[0, 0].copy(), f[0, 1].copy()

    def get_poly_points(self, left_fit_coeffs, right_fit_coeffs, partial=1):
        """lane_tracker.py:511-528."""
        xs, cnt = self._bt.get_poly_points(np.stack([left_fit_coeffs, right_fit_coeffs])[None], partial)
        xs, cnt = xs.cpu().numpy()[0], cnt.cpu().numpy()[0]
        bh = self._bt.warped_size[1]
        lx, rx = xs[0, :cnt[0]].astype(np.int64), xs[1, :cnt[1]].astype(np.int64)
        return (np.arange(bh - cnt[0], bh, dtype=np.int64), lx, np.arange(bh - cnt[1], bh, dtype=np.int64), rx)

    def check_validity(self, left_fit_coeffs, right_fit_coeffs, diagnostics=False):
        """lane_tracker.py:561-627."""
        valid, diffs = self._bt.check_validity(np.stack([left_fit_coeffs, right_fit_coeffs])[None])
        self.valid_lane_lines = bool(valid[0])
        if diagnostics:
            print("x1_diff == {:.2f}, x2_diff == {:.2f}, x3_diff == {:.2f}, valid == {}".format(*diffs[0], valid[0]))

    def get_curve_radius(self):
        """lane_tracker.py:530-549: curve radii in metres of the current lane pixel sets (left_x/left_y, right_x/right_y),
        appended to the running mean over n_average frames."""
        fits = self._bt.fit_poly([[(self.left_y, self.left_x), (self.right_y, self.right_x)]])
        radii, _ = self._bt.lane_metrics(fits)
        self.left_curve_radius, self.right_curve_radius = int(radii[0, 0]), int(radii[0, 1])
        average_curve_radius = int(0.5 * (self.left_curve_radius + self.right_curve_radius))
        self.average_curve_radii.append(average_curve_radius)
        if len(self.average_curve_radii) > self.n_average:
            self.average_curve_radii.pop(0)
        real_curve_radii = [float(r) for r in self.average_curve_radii if r > 0]
        self.average_curve_radius = int(_float64_mean(real_curve_radii))

    def get_eccentricity(self):
        """lane_tracker.py:551-559: lateral offset of the car from the lane centre in metres (left_avg_x / right_avg_x)."""
        bh = self._bt.warped_size[1]
        xs = np.zeros((1, 2, bh), dtype=np.int32)
        cnt = np.array([[len(self.left_avg_x), len(self.right_avg_x)]], dtype=np.int32)
        xs[0, 0, :cnt[0, 0]] = self.left_avg_x
        xs[0, 1, :cnt[0, 1]] = self.right_avg_x
        dev = self._bt.device
        _, ecc = self._bt.lane_metrics(np.zeros((1, 2, 3)), torch.as_tensor(xs).to(dev), torch.as_tensor(cnt).to(dev))
        self.eccentricity = float(ecc[0])

    def draw_lane(self, img):
        """lane_tracker.py:629-662: uses left_avg_x / right_avg_x, average_curve_radius, eccentricity.  Text first, then the
        blend over it, as in the reference; all on the device.  The caller's ``img`` is not modified (the reference draws
        its text into it)."""
        w, h = self._bt.img_size
        bh = self._bt.warped_size[1]
        frames = self._upload(img, (h, w, 3)).unsqueeze(0)
        if self._bt.text_enabled and self.average_curve_radius is not None and self.eccentricity is not None:
            self._bt.draw_text(frames, [0], [self.average_curve_radius], [self.eccentricity], [self.counter])
        xs = np.zeros((1, 2, bh), dtype=np.int32)
        cnt = np.array([[len(self.left_avg_x), len(self.right_avg_x)]], dtype=np.int32)
        xs[0, 0, :cnt[0, 0]] = self.left_avg_x
        xs[0, 1, :cnt[0, 1]] = self.right_avg_x
        out = self._bt.draw_lane(frames, torch.as_tensor(xs).to(self._bt.device),
                                 torch.as_tensor(cnt).to(self._bt.device))
        return out[0].cpu().numpy()

    def print_failure(self, img):
        """lane_tracker.py:664-673: the failure message (and frame number) on a copy of the frame, drawn on the device."""
        w, h = self._bt.img_size
        frames = self._upload(img, (h, w, 3)).unsqueeze(0)
        if self._bt.text_enabled:
            self._bt.draw_text(frames, [1], None, None, [self.counter])
        return frames[0].cpu().numpy()
