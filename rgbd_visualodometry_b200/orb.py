"""Host-side mirror of the operator interface the reference's front-end uses for its hot path.

  reference (C++)                                             this module
  ----------------------------------------------------------  -------------------------------------------
  cv::ORB::create(nfeatures, scaleFactor, nlevels)            ORB_create(nfeatures, scaleFactor, nlevels)
      src/frontend.cpp:35-37
  orb_->detectAndCompute(color_, Mat(), kps, desc)            ORB.detectAndCompute(image, None) -> (kps, desc)
      src/frontend.cpp:153
  matcher.match(query, train, matches)                        BFMatcher(NORM_HAMMING).match(query, train)
      src/frontend.cpp:187                                    (+ knnMatch(query, train, k <= 32), crossCheck=True,
                                                              radiusMatch(query, train, maxDistance))
  max(min_dis * match_ratio, 30) filter                       filter_matches(matches, match_ratio)
      src/frontend.cpp:190-211

Same names, argument meaning and empty-input behaviour as the OpenCV operators, so the parity tests read like
cv2 code.  Keypoints come back as a numpy structured array with cv::KeyPoint's seven fields (28-byte records,
KP_DTYPE); matches as DMATCH_DTYPE records (cv::DMatch, 16 bytes).  All arithmetic runs in liborbx.so on the
GPU; nothing here computes on the CPU.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib

KP_DTYPE = np.dtype([("x", "<f4"), ("y", "<f4"), ("size", "<f4"), ("angle", "<f4"), ("response", "<f4"),
                     ("octave", "<i4"), ("class_id", "<i4")])
DMATCH_DTYPE = np.dtype([("queryIdx", "<i4"), ("trainIdx", "<i4"), ("imgIdx", "<i4"), ("distance", "<f4")])
NORM_HAMMING = 6  # == cv2.NORM_HAMMING
MAX_KNN = 32      # == ORBX_MAX_KNN: the largest k of knnMatch

OK, E_ARG, E_CAPACITY, E_CUDA, E_NOMEM, E_UNSUPPORTED, E_INTERNAL, E_ORDER = 0, -1, -2, -3, -4, -5, -6, -7


class OrbxError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"orbx error {code}: {msg}")
        self.code = code


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class Context:
    """One orbx_ctx: a (GPU, stream) pair owning the device-resident buffers.  Not thread-safe."""

    def __init__(self, nfeatures=500, scale_factor=1.2, nlevels=8, max_w=640, max_h=480, max_batch=1, device=0):
        self.lib = _lib.load()
        h = C.c_void_p()
        rc = self.lib.orbx_create(C.byref(h), device, nfeatures, scale_factor, nlevels, max_w, max_h, max_batch)
        if rc != OK:
            raise OrbxError(rc, "orbx_create failed (no sm_100 CUDA device, bad arguments or out of memory)")
        self.h = h
        self.nfeatures, self.scale_factor, self.nlevels = nfeatures, scale_factor, nlevels
        self.max_w, self.max_h, self.max_batch, self.device = max_w, max_h, max_batch, device

    def close(self):
        if getattr(self, "h", None):
            self.lib.orbx_destroy(self.h)
            self.h = None

    __del__ = close

    def _check(self, rc):
        if rc != OK:
            raise OrbxError(rc, self.lib.orbx_last_error(self.h).decode())

    # ---- extraction -------------------------------------------------------------------------------------
    def detect_and_compute(self, image: np.ndarray, cap: int | None = None):
        """One HOST frame (H x W x 3 BGR or H x W gray, uint8) -> (keypoints[KP_DTYPE], descriptors[n, 32])."""
        k, d, n = self.detect_and_compute_batch([image], cap)
        return k[0, :n[0]].copy(), d[0, :n[0]].copy()

    def detect_and_compute_batch(self, images, cap: int | None = None):
        """Same-sized HOST frames -> (kps[B, cap], desc[B, cap, 32], counts[B]).  Grows cap on E_CAPACITY."""
        imgs = [np.ascontiguousarray(im, dtype=np.uint8) for im in images]
        b = len(imgs)
        if b == 0:
            return np.zeros((0, 0), KP_DTYPE), np.zeros((0, 0, 32), np.uint8), np.zeros(0, np.int32)
        h, w = imgs[0].shape[:2]
        ch = 1 if imgs[0].ndim == 2 else imgs[0].shape[2]
        cap = int(cap) if cap is not None else max(2 * self.nfeatures, 64)
        ptrs = (C.c_void_p * b)(*[im.ctypes.data for im in imgs])
        while True:
            kps = np.zeros((b, cap), KP_DTYPE)
            desc = np.zeros((b, cap, 32), np.uint8)
            n = np.zeros(b, np.int32)
            rc = self.lib.orbx_detect_and_compute_batch(self.h, ptrs, b, w, h, imgs[0].strides[0] if h else 0, ch,
                                                        _ptr(kps), _ptr(desc), cap, _ptr(n))
            if rc == E_CAPACITY:
                cap = int(n.max())
                continue
            self._check(rc)
            return kps, desc, n

    def submit_frame(self, image: np.ndarray):
        """Queue one HOST frame (returns at once; at most two in flight)."""
        im = np.ascontiguousarray(image, dtype=np.uint8)
        h, w = im.shape[:2]
        ch = 1 if im.ndim == 2 else im.shape[2]
        self._check(self.lib.orbx_submit_frame(self.h, _ptr(im), w, h, im.strides[0], ch))

    def collect_frame(self, cap: int | None = None):
        """Wait for the oldest submitted frame -> (keypoints, descriptors)."""
        cap = int(cap) if cap is not None else max(2 * self.nfeatures, 64)
        kps = np.zeros(cap, KP_DTYPE)
        desc = np.zeros((cap, 32), np.uint8)
        n = C.c_int(0)
        self._check(self.lib.orbx_collect_frame(self.h, _ptr(kps), _ptr(desc), cap, C.byref(n)))
        return kps[:n.value].copy(), desc[:n.value].copy()

    def extract_match_batch(self, images, maps, cap: int | None = None):
        """The front-end's per-frame pattern for a batch of HOST frames: extraction, then every map in `maps`
        ([M_j, 32] uint8 each) matched against each frame's own descriptors.  Returns (kps, desc, counts, [best_j[B, M_j]])."""
        imgs = [np.ascontiguousarray(im, dtype=np.uint8) for im in images]
        b = len(imgs)
        qs = [np.ascontiguousarray(m, np.uint8).reshape(-1, 32) for m in maps]
        h, w = imgs[0].shape[:2]
        ch = 1 if imgs[0].ndim == 2 else imgs[0].shape[2]
        cap = int(cap) if cap is not None else max(2 * self.nfeatures, 64)
        ptrs = (C.c_void_p * b)(*[im.ctypes.data for im in imgs])
        qptrs = (C.c_void_p * max(len(qs), 1))(*[q.ctypes.data for q in qs])
        nq = (C.c_int * max(len(qs), 1))(*[len(q) for q in qs])
        while True:
            kps = np.zeros((b, cap), KP_DTYPE)
            desc = np.zeros((b, cap, 32), np.uint8)
            n = np.zeros(b, np.int32)
            best = [np.zeros((b, len(q)), DMATCH_DTYPE) for q in qs]
            bptrs = (C.c_void_p * max(len(qs), 1))(*[x.ctypes.data for x in best])
            rc = self.lib.orbx_extract_match_batch(self.h, ptrs, b, w, h, imgs[0].strides[0] if h else 0, ch, _ptr(kps), _ptr(desc), cap,
                                                   _ptr(n), qptrs, nq, len(qs), bptrs)
            if rc == E_CAPACITY:
                cap = int(n.max())
                continue
            self._check(rc)
            return kps, desc, n, best

    def detect_and_compute_device(self, d_imgs_ptr: int, batch: int, w: int, h: int, step: int, frame_stride: int, channels: int,
                                  d_kps_ptr: int, d_desc_ptr: int, cap: int, d_counts_ptr: int):
        """Asynchronous, device-resident batch (raw device pointers, e.g. torch .data_ptr())."""
        self._check(self.lib.orbx_detect_and_compute_device(self.h, d_imgs_ptr, batch, w, h, step, frame_stride, channels,
                                                            d_kps_ptr, d_desc_ptr, cap, d_counts_ptr))

    # ---- matching -----------------------------------------------------------------------------------------
    def match(self, query: np.ndarray, train: np.ndarray) -> np.ndarray:
        q = np.ascontiguousarray(query, np.uint8).reshape(-1, 32)
        t = np.ascontiguousarray(train, np.uint8).reshape(-1, 32)
        out = np.zeros(max(len(q), 1), DMATCH_DTYPE)
        n = C.c_int(0)
        self._check(self.lib.orbx_match_hamming(self.h, _ptr(q), len(q), _ptr(t), len(t), _ptr(out), C.byref(n)))
        return out[:n.value]

    def knn_match2(self, query: np.ndarray, train: np.ndarray) -> np.ndarray:
        q = np.ascontiguousarray(query, np.uint8).reshape(-1, 32)
        t = np.ascontiguousarray(train, np.uint8).reshape(-1, 32)
        out = np.zeros((max(len(q), 1), 2), DMATCH_DTYPE)
        n = C.c_int(0)
        self._check(self.lib.orbx_match_hamming_knn2(self.h, _ptr(q), len(q), _ptr(t), len(t), _ptr(out), C.byref(n)))
        return out[:n.value]

    def knn_match(self, query: np.ndarray, train: np.ndarray, k: int) -> np.ndarray:
        """knnMatch(query, train, k), 1 <= k <= MAX_KNN: [nq, k] records, row i = query i's k nearest train rows by
        (distance, trainIdx); slots past the train set's size hold trainIdx = -1.  [0, k] when either set is empty."""
        q = np.ascontiguousarray(query, np.uint8).reshape(-1, 32)
        t = np.ascontiguousarray(train, np.uint8).reshape(-1, 32)
        out = np.zeros((max(len(q), 1), max(int(k), 1)), DMATCH_DTYPE)
        n = C.c_int(0)
        self._check(self.lib.orbx_match_hamming_knn(self.h, _ptr(q), len(q), _ptr(t), len(t), int(k), _ptr(out), C.byref(n)))
        return out[:n.value]

    def radius_match(self, query: np.ndarray, train: np.ndarray, max_distance: float):
        """radiusMatch(query, train, maxDistance): (records, offsets), query i's list = records[offsets[i]:offsets[i + 1]] in cv2's
        order (libstdc++ std::sort by distance of the rows in ascending trainIdx).  offsets is int64 [nq + 1]."""
        q = np.ascontiguousarray(query, np.uint8).reshape(-1, 32)
        t = np.ascontiguousarray(train, np.uint8).reshape(-1, 32)
        offsets = np.zeros(len(q) + 1, np.int64)
        n = C.c_int(0)
        cap = min(len(q) * len(t), max(1024, 16 * len(q)))
        while True:
            out = np.zeros(max(cap, 1), DMATCH_DTYPE)
            rc = self.lib.orbx_match_hamming_radius(self.h, _ptr(q), len(q), _ptr(t), len(t), float(max_distance), _ptr(out), cap,
                                                    _ptr(offsets), C.byref(n))
            if rc == E_CAPACITY:
                cap = n.value
                continue
            self._check(rc)
            return out[:n.value], offsets

    def match_crosscheck(self, query: np.ndarray, train: np.ndarray) -> np.ndarray:
        """BFMatcher(NORM_HAMMING, crossCheck=True).match: the mutual nearest pairs, ascending queryIdx."""
        q = np.ascontiguousarray(query, np.uint8).reshape(-1, 32)
        t = np.ascontiguousarray(train, np.uint8).reshape(-1, 32)
        out = np.zeros(max(len(q), 1), DMATCH_DTYPE)
        n = C.c_int(0)
        self._check(self.lib.orbx_match_hamming_crosscheck(self.h, _ptr(q), len(q), _ptr(t), len(t), _ptr(out), C.byref(n)))
        return out[:n.value]

    def match_device_crosscheck(self, d_query_ptr: int, nq: int, d_train_ptr: int, stride_rows: int, d_counts_ptr: int, nsets: int,
                                d_out_ptr: int, d_n_out_ptr: int):
        """Asynchronous, device-resident, ragged batch: set s's mutual pairs to d_out[s, :d_n_out[s]] ([nsets, nq] records)."""
        self._check(self.lib.orbx_match_hamming_device_crosscheck(self.h, d_query_ptr, nq, d_train_ptr, stride_rows, d_counts_ptr, nsets,
                                                                  d_out_ptr, d_n_out_ptr))

    def match_device(self, d_query_ptr: int, nq: int, d_train_ptr: int, nt: int, nsets: int, d_best_ptr: int, d_second_ptr: int = 0):
        self._check(self.lib.orbx_match_hamming_device(self.h, d_query_ptr, nq, d_train_ptr, nt, nsets, d_best_ptr,
                                                       d_second_ptr or None))

    def match_device_ragged(self, d_query_ptr: int, nq: int, d_train_ptr: int, stride_rows: int, d_counts_ptr: int, nsets: int,
                            d_best_ptr: int, d_second_ptr: int = 0):
        self._check(self.lib.orbx_match_hamming_device_ragged(self.h, d_query_ptr, nq, d_train_ptr, stride_rows, d_counts_ptr, nsets,
                                                              d_best_ptr, d_second_ptr or None))

    def match_device_pairwise(self, d_query_ptr: int, query_stride_rows: int, d_query_counts_ptr: int, d_train_ptr: int,
                              train_stride_rows: int, d_train_counts_ptr: int, npairs: int, d_best_ptr: int, d_second_ptr: int = 0):
        """Asynchronous, device-resident: pair p's own query set against its own train set ([npairs, query_stride_rows] records;
        slots past a pair's query count are not written)."""
        self._check(self.lib.orbx_match_hamming_device_pairwise(self.h, d_query_ptr, query_stride_rows, d_query_counts_ptr, d_train_ptr,
                                                                train_stride_rows, d_train_counts_ptr, npairs, d_best_ptr, d_second_ptr or None))

    def match_device_pairwise_crosscheck(self, d_query_ptr: int, query_stride_rows: int, d_query_counts_ptr: int, d_train_ptr: int,
                                         train_stride_rows: int, d_train_counts_ptr: int, npairs: int, d_out_ptr: int, d_n_out_ptr: int):
        """As match_device_pairwise with crossCheck: pair p's mutual pairs to d_out[p, :d_n_out[p]]."""
        self._check(self.lib.orbx_match_hamming_device_pairwise_crosscheck(self.h, d_query_ptr, query_stride_rows, d_query_counts_ptr,
                                                                           d_train_ptr, train_stride_rows, d_train_counts_ptr, npairs,
                                                                           d_out_ptr, d_n_out_ptr))

    def match_device_knn(self, d_query_ptr: int, nq: int, d_train_ptr: int, stride_rows: int, d_counts_ptr: int, nsets: int, k: int,
                         d_out_ptr: int):
        """Asynchronous, device-resident, ragged batch: knnMatch of the query set against every set, [nsets, nq, k] records."""
        self._check(self.lib.orbx_match_hamming_device_knn(self.h, d_query_ptr, nq, d_train_ptr, stride_rows, d_counts_ptr, nsets, int(k),
                                                           d_out_ptr))

    def match_device_pairwise_knn(self, d_query_ptr: int, query_stride_rows: int, d_query_counts_ptr: int, d_train_ptr: int,
                                  train_stride_rows: int, d_train_counts_ptr: int, npairs: int, k: int, d_out_ptr: int):
        """As match_device_pairwise with knnMatch: [npairs, query_stride_rows, k] records (slots past a pair's query count are
        not written)."""
        self._check(self.lib.orbx_match_hamming_device_pairwise_knn(self.h, d_query_ptr, query_stride_rows, d_query_counts_ptr, d_train_ptr,
                                                                    train_stride_rows, d_train_counts_ptr, npairs, int(k), d_out_ptr))

    def match_device_radius(self, d_query_ptr: int, nq: int, d_train_ptr: int, stride_rows: int, d_counts_ptr: int, nsets: int,
                            max_distance: float, d_out_ptr: int, cap: int, d_offsets_ptr: int):
        """Asynchronous, device-resident, ragged batch: radiusMatch of the query set against every set.  List s * nq + i at
        d_out[d_offsets[L] : d_offsets[L + 1]] (d_offsets: int64 [nsets * nq + 1], always complete); lists ending past cap
        records are not written."""
        self._check(self.lib.orbx_match_hamming_device_radius(self.h, d_query_ptr, nq, d_train_ptr, stride_rows, d_counts_ptr, nsets,
                                                              float(max_distance), d_out_ptr, int(cap), d_offsets_ptr))

    def match_device_pairwise_radius(self, d_query_ptr: int, query_stride_rows: int, d_query_counts_ptr: int, d_train_ptr: int,
                                     train_stride_rows: int, d_train_counts_ptr: int, npairs: int, max_distance: float, d_out_ptr: int,
                                     cap: int, d_offsets_ptr: int):
        """As match_device_radius, pairwise: list p * query_stride_rows + i (empty past pair p's query count)."""
        self._check(self.lib.orbx_match_hamming_device_pairwise_radius(self.h, d_query_ptr, query_stride_rows, d_query_counts_ptr,
                                                                       d_train_ptr, train_stride_rows, d_train_counts_ptr, npairs,
                                                                       float(max_distance), d_out_ptr, int(cap), d_offsets_ptr))

    def match_sets(self, query: np.ndarray, train: np.ndarray, counts: np.ndarray, knn2: bool = False):
        """One map (query [M,32]) against nsets frames' descriptor sets (train [S,cap,32], counts [S]); host buffers."""
        q = np.ascontiguousarray(query, np.uint8).reshape(-1, 32)
        t = np.ascontiguousarray(train, np.uint8)
        cnt = np.ascontiguousarray(counts, np.int32)
        s, cap = t.shape[0], t.shape[1]
        best = np.zeros((s, len(q)), DMATCH_DTYPE)
        second = np.zeros((s, len(q)), DMATCH_DTYPE) if knn2 else None
        self._check(self.lib.orbx_match_hamming_sets(self.h, _ptr(q), len(q), _ptr(t), cap, _ptr(cnt), s, _ptr(best), _ptr(second)))
        return (best, second) if knn2 else best

    # ---- map table / tracking (SURVEY 8(f)) -------------------------------------------------------------------
    def map_upsert(self, ids, desc=None, pos=None, norm=None, outlier=None):
        ids = np.ascontiguousarray(ids, np.int64)
        n = len(ids)
        d = None if desc is None else np.ascontiguousarray(desc, np.uint8).reshape(n, 32)
        p = None if pos is None else np.ascontiguousarray(pos, np.float64).reshape(n, 3)
        nv = None if norm is None else np.ascontiguousarray(norm, np.float64).reshape(n, 3)
        o = None if outlier is None else np.ascontiguousarray(outlier, np.uint8).reshape(n)
        self._check(self.lib.orbx_map_upsert(self.h, _ptr(ids), n, _ptr(d), _ptr(p), _ptr(nv), _ptr(o)))

    def map_upsert_from_frame(self, ids, frame: int, kp_index, pos=None, norm=None):
        ids = np.ascontiguousarray(ids, np.int64)
        n = len(ids)
        ki = np.ascontiguousarray(kp_index, np.int32).reshape(n)
        p = None if pos is None else np.ascontiguousarray(pos, np.float64).reshape(n, 3)
        nv = None if norm is None else np.ascontiguousarray(norm, np.float64).reshape(n, 3)
        self._check(self.lib.orbx_map_upsert_from_frame(self.h, _ptr(ids), n, frame, _ptr(ki), _ptr(p), _ptr(nv)))

    def map_erase(self, ids):
        ids = np.ascontiguousarray(ids, np.int64)
        self._check(self.lib.orbx_map_erase(self.h, _ptr(ids), len(ids)))

    def map_clear(self):
        self._check(self.lib.orbx_map_clear(self.h))

    @property
    def map_size(self) -> int:
        return int(self.lib.orbx_map_size(self.h))

    def track_match(self, ids, pose_Tcw, cam, cols: int, rows: int, train=None, frame: int = 0, match_ratio: float = 2.0):
        """FrontEnd::MatchKeyPointsInTrackingMap on the device.  Returns (cand, matches, min_dis, max_dis); matches'
        queryIdx index `cand`, whose entries index `ids`."""
        ids = np.ascontiguousarray(ids, np.int64)
        m = len(ids)
        T = np.ascontiguousarray(pose_Tcw, np.float64).reshape(12)
        K = np.ascontiguousarray(cam, np.float64).reshape(4)
        cand = np.zeros(max(m, 1), np.int32)
        out = np.zeros(max(m, 1), DMATCH_DTYPE)
        nc, nm = C.c_int(0), C.c_int(0)
        mn, mx = C.c_float(0), C.c_float(0)
        if train is not None:
            t = np.ascontiguousarray(train, np.uint8).reshape(-1, 32)
            tp, tn = _ptr(t), len(t)
            if tn == 0:
                tp = _ptr(np.zeros((1, 32), np.uint8))
        else:
            tp, tn = None, frame
        self._check(self.lib.orbx_track_match(self.h, _ptr(ids), m, _ptr(T), _ptr(K), cols, rows, tp, tn, match_ratio, _ptr(cand), C.byref(nc),
                                              _ptr(out), C.byref(nm), C.byref(mn), C.byref(mx)))
        return cand[:nc.value].copy(), out[:nm.value].copy(), mn.value, mx.value

    def backproject(self, kps: np.ndarray, depth: np.ndarray, depth_scale: float, cam, pose_Tcw):
        """Frame::GetDepth + Camera::Pixel2World for KP_DTYPE keypoints.  Returns (pos_w[n, 3], valid[n])."""
        k = np.ascontiguousarray(kps)
        d = np.ascontiguousarray(depth, np.uint16)
        n = len(k)
        T = np.ascontiguousarray(pose_Tcw, np.float64).reshape(12)
        K = np.ascontiguousarray(cam, np.float64).reshape(4)
        pos = np.zeros((max(n, 1), 3), np.float64)
        valid = np.zeros(max(n, 1), np.uint8)
        self._check(self.lib.orbx_backproject(self.h, _ptr(k), n, _ptr(d), d.shape[1], d.shape[0], d.strides[0], depth_scale, _ptr(K), _ptr(T),
                                              _ptr(pos), _ptr(valid)))
        return pos[:n], valid[:n].astype(bool)

    # ---- misc -----------------------------------------------------------------------------------------------
    def synchronize(self):
        self._check(self.lib.orbx_synchronize(self.h))

    @property
    def stream(self) -> int:
        return int(self.lib.orbx_stream(self.h) or 0)

    @property
    def launch_count(self) -> int:
        return int(self.lib.orbx_launch_count(self.h))

    def level_geometry(self, w: int, h: int):
        n = self.nlevels
        ws = np.zeros(n, np.int32); hs = np.zeros(n, np.int32); sc = np.zeros(n, np.float32); q = np.zeros(n, np.int32)
        self._check(self.lib.orbx_level_geometry(self.h, w, h, _ptr(ws), _ptr(hs), _ptr(sc), _ptr(q)))
        return ws, hs, sc, q

    def debug_level(self, frame: int, level: int, w: int, h: int) -> np.ndarray:
        out = np.zeros((h, w), np.uint8)
        self._check(self.lib.orbx_debug_read_level(self.h, frame, level, _ptr(out), out.size))
        return out

    def debug_fast(self, frame: int, level: int, cap: int = 1 << 20):
        x = np.zeros(cap, np.int32); y = np.zeros(cap, np.int32); s = np.zeros(cap, np.int32)
        n = C.c_int(0)
        self._check(self.lib.orbx_debug_read_fast(self.h, frame, level, _ptr(x), _ptr(y), _ptr(s), cap, C.byref(n)))
        return x[:n.value], y[:n.value], s[:n.value]

    def force_kernels(self, mode: int):
        """-1: pyramid / FAST kernel family by launch size (default); 0: warp-private TMA kernels; 1: CTA-cooperative kernels."""
        self._check(self.lib.orbx_debug_force_kernels(self.h, mode))

    def host_register(self, arr: np.ndarray):
        """Page-lock a long-lived host buffer (cudaHostRegister behind the C-ABI); pair with host_unregister."""
        self._check(self.lib.orbx_host_register(self.h, arr.ctypes.data, arr.nbytes))

    def host_unregister(self, arr: np.ndarray):
        self._check(self.lib.orbx_host_unregister(self.h, arr.ctypes.data))

    def set_profiling(self, on: bool):
        self._check(self.lib.orbx_set_profiling(self.h, 1 if on else 0))

    def stage_times(self) -> dict:
        names = (C.c_char_p * 8)(); ms = (C.c_float * 8)()
        n = self.lib.orbx_debug_stage_times(self.h, names, ms, 8)
        return {names[i].decode(): float(ms[i]) for i in range(max(n, 0))}


class ORB:
    """cv::ORB stand-in (only the parameters the reference sets; the rest are OpenCV's defaults)."""

    def __init__(self, nfeatures=500, scaleFactor=1.2, nlevels=8, device=0, kernels=-1):
        self.nfeatures, self.scaleFactor, self.nlevels, self.device = nfeatures, scaleFactor, nlevels, device
        self.kernels = kernels                  # orbx_debug_force_kernels mode (tests run both kernel families)
        self._ctx = None

    def _context(self, w, h, b=1):
        c = self._ctx
        if c is None or w > c.max_w or h > c.max_h or b > c.max_batch:
            if c is not None:
                c.close()
            self._ctx = c = Context(self.nfeatures, self.scaleFactor, self.nlevels, max(w, 1), max(h, 1), max(b, 1), self.device)
            if self.kernels >= 0:
                c.force_kernels(self.kernels)
        return c

    def detectAndCompute(self, image, mask=None):
        if mask is not None:
            raise OrbxError(E_UNSUPPORTED, "mask is not supported (the reference always passes Mat())")
        image = np.asarray(image)
        if image.size == 0:
            return np.zeros(0, KP_DTYPE), None              # cv2: ((), None)
        k, d = self._context(image.shape[1], image.shape[0]).detect_and_compute(image)
        return k, (d if len(k) else None)

    def detectAndComputeBatch(self, images):
        images = list(images)
        if not images:
            return np.zeros((0, 0), KP_DTYPE), np.zeros((0, 0, 32), np.uint8), np.zeros(0, np.int32)
        return self._context(images[0].shape[1], images[0].shape[0], len(images)).detect_and_compute_batch(images)


def ORB_create(nfeatures=500, scaleFactor=1.2, nlevels=8, device=0, kernels=-1) -> ORB:
    return ORB(nfeatures, scaleFactor, nlevels, device, kernels)


class BFMatcher:
    """cv::BFMatcher(NORM_HAMMING[, crossCheck]) stand-in on the tcgen05 int8 tensor cores.  With crossCheck, match keeps
    only the mutual nearest pairs (the reverse direction comes out of the same distance tiles); an empty train set gives
    no matches where cv2 raises."""

    def __init__(self, normType=NORM_HAMMING, crossCheck=False, device=0):
        if normType != NORM_HAMMING:
            raise OrbxError(E_UNSUPPORTED, "only NORM_HAMMING is implemented (what the hot path uses)")
        self.crossCheck = bool(crossCheck)
        self._ctx = Context(1, 1.2, 1, 64, 64, 1, device)

    def match(self, queryDescriptors, trainDescriptors):
        if queryDescriptors is None or trainDescriptors is None:
            return np.zeros(0, DMATCH_DTYPE)
        if self.crossCheck:
            return self._ctx.match_crosscheck(queryDescriptors, trainDescriptors)
        return self._ctx.match(queryDescriptors, trainDescriptors)

    def knnMatch(self, queryDescriptors, trainDescriptors, k=2):
        """[nq, k] records, row i = query i's k nearest train rows by (distance, trainIdx) as cv2's list for query i, padded
        with trainIdx = -1 records where cv2's list is shorter (k > number of train rows).  With crossCheck (k = 1 only, as
        cv2): the mutual pair, or a trainIdx = -1 record where cv2 gives []."""
        k = int(k)
        if k < 1:
            raise OrbxError(E_ARG, "knnMatch needs k >= 1")
        if k > MAX_KNN:
            raise OrbxError(E_UNSUPPORTED, f"knnMatch is implemented for k <= {MAX_KNN}")
        if self.crossCheck and k != 1:
            raise OrbxError(E_UNSUPPORTED, "knnMatch with crossCheck is implemented for k = 1 (cv2 asserts otherwise)")
        if queryDescriptors is None or trainDescriptors is None:
            return np.zeros((0, k), DMATCH_DTYPE)
        if self.crossCheck:
            nq = len(np.ascontiguousarray(queryDescriptors, np.uint8).reshape(-1, 32))
            pairs = self._ctx.match_crosscheck(queryDescriptors, trainDescriptors)
            if len(np.ascontiguousarray(trainDescriptors, np.uint8).reshape(-1, 32)) == 0:
                nq = 0                                      # an empty train set: no lists (as knn_match)
            out = np.zeros((nq, 1), DMATCH_DTYPE)
            out["queryIdx"][:, 0] = np.arange(nq)
            out["trainIdx"] = -1
            out[pairs["queryIdx"], 0] = pairs
            return out
        if k == 2:
            return self._ctx.knn_match2(queryDescriptors, trainDescriptors)
        return self._ctx.knn_match(queryDescriptors, trainDescriptors, k)

    def radiusMatch(self, queryDescriptors, trainDescriptors, maxDistance):
        """A list of nq DMATCH_DTYPE arrays (views of one buffer): query i's train rows at distance <= maxDistance, in cv2's
        order.  crossCheck does not apply, as in cv2.  maxDistance <= FLT_EPSILON or NaN raises (E_ARG) unless the query set is
        empty (cv2 returns no lists before it checks)."""
        if queryDescriptors is None or trainDescriptors is None or np.asarray(queryDescriptors).size == 0:
            return []
        rec, off = self._ctx.radius_match(queryDescriptors, trainDescriptors, maxDistance)
        return [rec[off[i]:off[i + 1]] for i in range(len(off) - 1)]


def filter_matches(matches: np.ndarray, match_ratio: float = 2.0) -> np.ndarray:
    """src/frontend.cpp:190-211: keep distance <= max(min_distance * match_ratio, 30)."""
    m = np.ascontiguousarray(matches.copy())
    n = _lib.load().orbx_filter_matches(_ptr(m), len(m), match_ratio)
    return m[:n]
