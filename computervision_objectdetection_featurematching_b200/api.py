"""Host-side mirror of the reference's hot-path calls on top of libcvgraft's C ABI.

    Context.match_knn2        <- cv::BFMatcher(NORM_L2).knnMatch(q, t, 2) + ratio test
                                 reference src/TestsDetector.cpp:59-72
    Context.match_cross_check <- cv::BFMatcher(NORM_L2, crossCheck=true).match(q, t)
    Context.find_homography   <- cv::findHomography(src, dst, RANSAC, 5.0, mask)    :77-78
    Context.estimate_affine2d <- cv::estimateAffine2D(src, dst, inliers, RANSAC)    (the other geometric checks)
    Context.estimate_affine_partial2d <- cv::estimateAffinePartial2D(src, dst, inliers, RANSAC)
    Context.detect_pairs      <- body of the view loop of detectAtScale             :58-95
                                 (detect_params(method=...): findHomography, estimateAffine2D or
                                 estimateAffinePartial2D as its geometric check; detect_params(cross_check=True):
                                 BFMatcher(NORM_L2, crossCheck=true).match instead of knnMatch + ratio test)
    Models                    <- ObjectModel descriptors resident in HBM            include/objectModel.hpp:11-16

Error behaviour follows OpenCV where the reference relies on it: find_homography raises for n < 4.
numpy arrays in, numpy arrays out; all compute happens on the GPU (no CPU fallback).
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import AffineParams, DetectParams, PairResult, RansacParams

ACCEPT, LT4_MATCHES, H_EMPTY, LT4_INLIERS, DET_REJECT = range(5)
RANSAC_NO_EARLY_STOP = 1
RANSAC_NO_REFINE = 2
FORCE_EXACT_MATCH = 1
MATCH_PAIR_MODE = 2
NITERS_ALL_ON_HOST = 4
PATH_TENSOR, PATH_EXACT, PATH_TENSOR_RERANK = 1, 2, 3   # cvg_last_match_path
VERIFY_HOMOGRAPHY, VERIFY_AFFINE, VERIFY_AFFINE_PARTIAL = range(3)   # cvg_detect_params.method & 0xFF
MATCH_CROSS_CHECK = 0x100                                             # cvg_detect_params.method flag (CVG_MATCH_CROSS_CHECK)

PAIR_DTYPE = np.dtype([("status", "<i4"), ("n_good", "<i4"), ("n_inliers", "<i4"), ("ransac_iters", "<i4"),
                       ("H", "<f8", (9,)), ("det", "<f8")])
assert PAIR_DTYPE.itemsize == C.sizeof(PairResult)


class CvgError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"cvgraft error {code}: {msg}")
        self.code = code


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _f32(a, cols):
    a = np.ascontiguousarray(a, dtype=np.float32)
    return a.reshape(-1, cols)


def ransac_params(threshold=5.0, max_iters=2000, confidence=0.995, flags=0):
    p = RansacParams()
    _lib.load().cvg_ransac_params_default(C.byref(p))
    p.threshold = threshold; p.max_iters = max_iters; p.confidence = confidence; p.flags = flags
    return p


def affine_params(threshold=3.0, max_iters=2000, confidence=0.99, refine_iters=10, flags=0):
    """cv2.estimateAffine2D's / estimateAffinePartial2D's ransacReprojThreshold, maxIters, confidence, refineIters
    (OpenCV's defaults)."""
    p = AffineParams()
    _lib.load().cvg_affine_params_default(C.byref(p))
    p.threshold = threshold; p.max_iters = max_iters; p.confidence = confidence; p.refine_iters = refine_iters
    p.flags = flags
    return p


def detect_params(ratio=0.9, min_inliers=4, det_lo=0.1, det_hi=10.0, ransac=None, method=VERIFY_HOMOGRAPHY,
                  refine_iters=10, cross_check=False):
    """Constants of the fused path.  method picks its geometric check: VERIFY_HOMOGRAPHY (findHomography), VERIFY_AFFINE
    (estimateAffine2D) or VERIFY_AFFINE_PARTIAL (estimateAffinePartial2D, refineIters = refine_iters).  The affine methods
    read ransac's threshold, max_iters and confidence as given: pass ransac_params(3.0, 2000, 0.99) for OpenCV's affine
    defaults.  cross_check=True sets MATCH_CROSS_CHECK in method: the correspondences are the mutual nearest neighbours of
    BFMatcher(NORM_L2, crossCheck=true).match (each view its own query matrix) and ratio is ignored."""
    p = DetectParams()
    _lib.load().cvg_detect_params_default(C.byref(p))
    p.ratio = ratio; p.min_inliers = min_inliers; p.det_lo = det_lo; p.det_hi = det_hi
    if ransac is not None:
        p.ransac = ransac
    p.method = method | (MATCH_CROSS_CHECK if cross_check else 0); p.refine_iters = refine_iters
    return p


class Models:
    """Model-view descriptors (+ keypoints) resident in HBM — the hook after src/ModelsDetector.cpp:80."""

    def __init__(self, ctx, handle, view_offsets):
        self.ctx, self.handle = ctx, handle
        self.view_offsets = np.asarray(view_offsets, np.int32)

    @property
    def n_views(self):
        return len(self.view_offsets) - 1

    @property
    def n_rows(self):
        return int(self.view_offsets[-1])

    def free(self):
        if self.handle:
            self.ctx.lib.cvg_models_free(self.ctx.handle, self.handle)
            self.handle = None


class Scenes:
    def __init__(self, ctx, handle, offsets, keep=None):
        self.ctx, self.handle = ctx, handle
        self.offsets = np.asarray(offsets, np.int64)
        self._keep = keep                      # host arrays an asynchronous upload is still reading

    def wait(self):
        """Block until an asynchronous upload has finished (optional: detect_scenes orders itself after it)."""
        self.ctx._check(self.ctx.lib.cvg_scenes_wait(self.ctx.handle, self.handle))
        self._keep = None

    @property
    def n_scenes(self):
        return len(self.offsets) - 1

    def free(self):
        if self.handle:
            self.ctx.lib.cvg_scenes_free(self.ctx.handle, self.handle)
            self.handle = None


class Job:
    """A fused call in flight (Context.submit_scenes); wait() returns what detect_scenes_inliers returns."""

    def __init__(self, ctx, handle, res, inl, off, S, V, keep):
        self.ctx, self.handle, self._res, self._inl, self._off, self._S, self._V, self._keep = ctx, handle, res, inl, off, S, V, keep

    def wait(self):
        if self.handle is None:
            raise RuntimeError("job already waited for")
        h, self.handle = self.handle, None
        self.ctx._check(self.ctx.lib.cvg_job_wait(self.ctx.handle, h))
        self._keep = None
        res = self._res[:self._S * self._V].reshape(self._S, self._V)
        if self._inl is None:
            return res, None, None
        return res, self._inl[:self._off[-1]], self._off


class Context:
    """device: one GPU index (cvg_create), or a list of GPU indices of this host (cvg_create_multi: model set replicated,
    scene batches dealt to the GPUs by cost, train-tile sharded match with one NCCL all-gather)."""

    def __init__(self, device=0, flags=0):
        self.lib = _lib.load()
        h = C.c_void_p()
        if isinstance(device, (list, tuple)):
            devs = (C.c_int * len(device))(*[int(d) for d in device])
            rc = self.lib.cvg_create_multi(C.byref(h), devs, len(device), flags)
        else:
            rc = self.lib.cvg_create(C.byref(h), device, flags)
        if rc:
            raise CvgError(rc, self.lib.cvg_last_error().decode())
        self.handle = h
        self.device = device

    @property
    def n_devices(self):
        return int(self.lib.cvg_num_devices(self.handle))

    @property
    def exchange_kind(self):
        """How the train-tile shards exchange their partial top-2: 'nccl', 'memcpy' (logical devices on one GPU), 'none'."""
        return self.lib.cvg_exchange_kind(self.handle).decode()

    def set_lanes(self, n):
        """Sub-batches of one synchronous fused call / jobs in flight (1 = strictly serial on the caller's thread, 0 = default)."""
        self._check(self.lib.cvg_set_lanes(self.handle, int(n)))

    def close(self):
        if self.handle:
            self.lib.cvg_destroy(self.handle)
            self.handle = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc):
        if rc:
            raise CvgError(rc, self.lib.cvg_last_error().decode())

    # ---- resident sets -----------------------------------------------------------------------
    def upload_models(self, descriptors, keypoints_xy, view_offsets, view_model=None):
        d = _f32(descriptors, 128)
        k = _f32(keypoints_xy, 2) if keypoints_xy is not None else None
        vo = np.ascontiguousarray(view_offsets, np.int32)
        vm = np.ascontiguousarray(view_model, np.int32) if view_model is not None else None
        h = C.c_void_p()
        self._check(self.lib.cvg_models_upload(self.handle, _ptr(d), _ptr(k), _ptr(vo), _ptr(vm), len(vo) - 1, C.byref(h)))
        return Models(self, h, vo)

    def upload_scenes(self, descriptors, keypoints_xy, offsets):
        d = _f32(descriptors, 128)
        k = _f32(keypoints_xy, 2) if keypoints_xy is not None else None
        off = np.ascontiguousarray(offsets, np.int64)
        h = C.c_void_p()
        self._check(self.lib.cvg_scenes_upload(self.handle, _ptr(d), _ptr(k), _ptr(off), len(off) - 1, C.byref(h)))
        return Scenes(self, h, off)

    def upload_scenes_async(self, descriptors, keypoints_xy, offsets):
        """Streaming upload on the context's copy stream: returns at once, overlaps a running detect_scenes.
        Pass pinned arrays for a truly asynchronous copy; they are kept alive by the returned handle."""
        d = _f32(descriptors, 128)
        k = _f32(keypoints_xy, 2) if keypoints_xy is not None else None
        off = np.ascontiguousarray(offsets, np.int64)
        h = C.c_void_p()
        self._check(self.lib.cvg_scenes_upload_async(self.handle, _ptr(d), _ptr(k), _ptr(off), len(off) - 1, C.byref(h)))
        return Scenes(self, h, off, keep=(d, k, off))

    def upload_scenes_u8_async(self, descriptors_u8, keypoints_xy, offsets):
        """Streaming upload of uint8 descriptor rows [N,128] (a quarter of the PCIe bytes of the fp32 form)."""
        d = np.ascontiguousarray(descriptors_u8, dtype=np.uint8).reshape(-1, 128)
        k = _f32(keypoints_xy, 2) if keypoints_xy is not None else None
        off = np.ascontiguousarray(offsets, np.int64)
        h = C.c_void_p()
        self._check(self.lib.cvg_scenes_upload_u8_async(self.handle, _ptr(d), _ptr(k), _ptr(off), len(off) - 1, C.byref(h)))
        return Scenes(self, h, off, keep=(d, k, off))

    # ---- match stage ---------------------------------------------------------------------------
    def match_knn2(self, query, train, ratio=0.9, view=-1):
        """query: Models (resident, optionally one view) or an [nq,128] array.  -> idx[nq,2] (-1 = absent),
        dist[nq,2], accept[nq]."""
        t = _f32(train, 128)
        if isinstance(query, Models):
            nq = query.n_rows if view < 0 else int(query.view_offsets[view + 1] - query.view_offsets[view])
        else:
            q = _f32(query, 128)
            nq = q.shape[0]
        idx = np.full((nq, 2), -1, np.int32); dist = np.zeros((nq, 2), np.float32); acc = np.zeros(nq, np.uint8)
        if isinstance(query, Models):
            rc = self.lib.cvg_match_knn2(self.handle, query.handle, view, _ptr(t), t.shape[0], ratio,
                                         _ptr(idx), _ptr(dist), _ptr(acc))
        else:
            rc = self.lib.cvg_match_knn2_raw(self.handle, _ptr(q), nq, _ptr(t), t.shape[0], ratio,
                                             _ptr(idx), _ptr(dist), _ptr(acc))
        self._check(rc)
        return idx, dist, acc

    def match_cross_check(self, query, train, view=-1):
        """BFMatcher(NORM_L2, crossCheck=True).match.  query: Models (resident; one view, or view=-1 for every view, each
        view its own query matrix) or an [nq,128] array.  -> idx[nq] (-1 = no match), dist[nq] (0 where idx is -1)."""
        t = _f32(train, 128)
        if isinstance(query, Models):
            nq = query.n_rows if view < 0 else int(query.view_offsets[view + 1] - query.view_offsets[view])
        else:
            q = _f32(query, 128)
            nq = q.shape[0]
        idx = np.full(nq, -1, np.int32); dist = np.zeros(nq, np.float32)
        if isinstance(query, Models):
            rc = self.lib.cvg_match_cross_check(self.handle, query.handle, view, _ptr(t), t.shape[0], _ptr(idx), _ptr(dist))
        else:
            rc = self.lib.cvg_match_cross_check_raw(self.handle, _ptr(q), nq, _ptr(t), t.shape[0], _ptr(idx), _ptr(dist))
        self._check(rc)
        return idx, dist

    @property
    def last_match_path(self):
        return self.lib.cvg_last_match_path(self.handle)

    @property
    def last_match_fallback_rows(self):
        """Rows of the last candidate-path call that were redone by the exact fallback kernel."""
        return int(self.lib.cvg_last_match_fallback_rows(self.handle))

    @property
    def last_match_guard_rows(self):
        """Rows of the last tensor-path call whose second distance reached 2048 and were redone exactly (cross-check calls:
        query rows plus train columns whose nearest distance reached 2048)."""
        return int(self.lib.cvg_last_match_guard_rows(self.handle))

    @property
    def last_sampler_serial_sets(self):
        """-1: the last verify call used the one-CTA-per-set sampler; else the sets the chunked sampler handed back."""
        return int(self.lib.cvg_last_sampler_serial_sets(self.handle))

    @property
    def stream(self):
        """cudaStream_t of the context as an int (all GPU work of this context is issued there)."""
        return int(self.lib.cvg_stream(self.handle) or 0)

    @property
    def launch_count(self):
        return int(self.lib.cvg_launch_count(self.handle))

    def selftest(self, which=0):
        """Device self test `which` (include/cvgraft.h); returns the number of mismatches (0 = pass)."""
        n = C.c_uint64(0)
        self._check(self.lib.cvg_selftest(self.handle, int(which), C.byref(n)))
        return int(n.value)

    def set_timing(self, on=True):
        self._check(self.lib.cvg_set_timing(self.handle, int(on)))

    def last_timing(self):
        a, b, c = C.c_float(), C.c_float(), C.c_float()
        self.lib.cvg_last_timing(self.handle, C.byref(a), C.byref(b), C.byref(c))
        h, n, p = C.c_float(), C.c_int(), C.c_uint64()
        self.lib.cvg_last_hyp_stats(self.handle, C.byref(h), C.byref(n), C.byref(p))
        sc = C.c_float()
        self.lib.cvg_last_score_ms(self.handle, C.byref(sc))
        return {"match_ms": a.value, "ransac_ms": b.value, "total_ms": c.value, "score_ms": sc.value,
                "hyp_ms": h.value, "hyp_launches": n.value, "scored_points": p.value}

    # ---- verify stage --------------------------------------------------------------------------
    def find_homography(self, src, dst, threshold=5.0, max_iters=2000, confidence=0.995, flags=0,
                        want_ransac_mask=False):
        """cv2.findHomography(src, dst, cv2.RANSAC, threshold, maxIters=, confidence=)
        -> (H 3x3 or None, mask uint8 [n]) (+ RANSAC-stage mask).  Raises for n < 4 like OpenCV."""
        s = _f32(src, 2); d = _f32(dst, 2)
        n = s.shape[0]
        if d.shape[0] != n:
            raise ValueError("src and dst must have the same number of points")
        H = np.zeros(9); mask = np.zeros(max(n, 1), np.uint8); found = C.c_int(0)
        rmask = np.zeros(max(n, 1), np.uint8) if want_ransac_mask else None
        p = ransac_params(threshold, max_iters, confidence, flags)
        self._check(self.lib.cvg_find_homography(self.handle, _ptr(s), _ptr(d), n, C.byref(p), _ptr(H), _ptr(mask),
                                                 C.byref(found), _ptr(rmask)))
        Hm = H.reshape(3, 3) if found.value else None
        return (Hm, mask[:n], rmask[:n]) if want_ransac_mask else (Hm, mask[:n])

    def find_homography_batch(self, src, dst, offsets, threshold=5.0, max_iters=2000, confidence=0.995, flags=0,
                              want_ransac_mask=False):
        s = _f32(src, 2); d = _f32(dst, 2)
        off = np.ascontiguousarray(offsets, np.int64)
        P = len(off) - 1
        H = np.zeros((P, 9)); mask = np.zeros(max(s.shape[0], 1), np.uint8)
        found = np.zeros(P, np.int32); iters = np.zeros(P, np.int32)
        rmask = np.zeros(max(s.shape[0], 1), np.uint8) if want_ransac_mask else None
        p = ransac_params(threshold, max_iters, confidence, flags)
        self._check(self.lib.cvg_find_homography_batch(self.handle, _ptr(s), _ptr(d), _ptr(off), P, C.byref(p),
                                                       _ptr(H), _ptr(mask), _ptr(found), _ptr(iters), _ptr(rmask)))
        out = {"H": H.reshape(P, 3, 3), "mask": mask[:s.shape[0]], "found": found.astype(bool), "iters": iters}
        if want_ransac_mask:
            out["ransac_mask"] = rmask[:s.shape[0]]
        return out

    def _affine(self, fn, src, dst, threshold, max_iters, confidence, refine_iters, flags):
        s = _f32(src, 2); d = _f32(dst, 2)
        n = s.shape[0]
        if d.shape[0] != n:
            raise ValueError("src and dst must have the same number of points")
        M = np.zeros(6); mask = np.zeros(max(n, 1), np.uint8); found = C.c_int(0)
        p = affine_params(threshold, max_iters, confidence, refine_iters, flags)
        self._check(fn(self.handle, _ptr(s), _ptr(d), n, C.byref(p), _ptr(M), _ptr(mask), C.byref(found)))
        return (M.reshape(2, 3) if found.value else None), mask[:n]

    def _affine_batch(self, fn, src, dst, offsets, threshold, max_iters, confidence, refine_iters, flags):
        s = _f32(src, 2); d = _f32(dst, 2)
        off = np.ascontiguousarray(offsets, np.int64)
        P = len(off) - 1
        M = np.zeros((max(P, 1), 6)); mask = np.zeros(max(s.shape[0], 1), np.uint8)
        found = np.zeros(max(P, 1), np.int32); iters = np.zeros(max(P, 1), np.int32)
        p = affine_params(threshold, max_iters, confidence, refine_iters, flags)
        self._check(fn(self.handle, _ptr(s), _ptr(d), _ptr(off), P, C.byref(p), _ptr(M), _ptr(mask), _ptr(found),
                       _ptr(iters)))
        return {"M": M[:P].reshape(P, 2, 3), "mask": mask[:s.shape[0]], "found": found[:P].astype(bool), "iters": iters[:P]}

    def estimate_affine2d(self, src, dst, threshold=3.0, max_iters=2000, confidence=0.99, refine_iters=10, flags=0):
        """cv2.estimateAffine2D(src, dst, method=cv2.RANSAC, ransacReprojThreshold=, maxIters=, confidence=, refineIters=)
        -> (M 2x3 or None, inlier mask uint8 [n]).  Raises for n = 0 like OpenCV."""
        return self._affine(self.lib.cvg_estimate_affine2d, src, dst, threshold, max_iters, confidence, refine_iters, flags)

    def estimate_affine2d_batch(self, src, dst, offsets, threshold=3.0, max_iters=2000, confidence=0.99, refine_iters=10,
                                flags=0):
        """estimate_affine2d for every set k = rows [offsets[k], offsets[k+1]) -> dict(M [P,2,3] (zeros where none),
        mask, found [P] bool, iters [P] RANSAC iterations)."""
        return self._affine_batch(self.lib.cvg_estimate_affine2d_batch, src, dst, offsets, threshold, max_iters, confidence,
                                  refine_iters, flags)

    def estimate_affine_partial2d(self, src, dst, threshold=3.0, max_iters=2000, confidence=0.99, refine_iters=10,
                                  flags=0):
        """cv2.estimateAffinePartial2D(src, dst, method=cv2.RANSAC, ...): the 4-DOF similarity [[a, -b, tx], [b, a, ty]]
        -> (M 2x3 or None, inlier mask uint8 [n]).  Raises for n = 0 like OpenCV."""
        return self._affine(self.lib.cvg_estimate_affine_partial2d, src, dst, threshold, max_iters, confidence,
                            refine_iters, flags)

    def estimate_affine_partial2d_batch(self, src, dst, offsets, threshold=3.0, max_iters=2000, confidence=0.99,
                                        refine_iters=10, flags=0):
        """estimate_affine_partial2d for every set k = rows [offsets[k], offsets[k+1]), with the outputs of
        estimate_affine2d_batch."""
        return self._affine_batch(self.lib.cvg_estimate_affine_partial2d_batch, src, dst, offsets, threshold, max_iters,
                                  confidence, refine_iters, flags)

    # ---- fused path ----------------------------------------------------------------------------
    def detect_pairs(self, models, scene_desc, scene_kpt_xy, scale=1.0, params=None, want_inliers=True):
        """All views of `models` against one scene: replaces the view loop src/TestsDetector.cpp:58-95.
        -> (per_view structured array, inlier_xy [k,2], inlier_offsets [V+1])."""
        t = _f32(scene_desc, 128); k = _f32(scene_kpt_xy, 2)
        p = params if params is not None else detect_params()
        V = models.n_views
        res = np.zeros(max(V, 1), PAIR_DTYPE)
        inl = np.zeros((max(models.n_rows, 1), 2), np.float32) if want_inliers else None
        ioff = np.zeros(V + 1, np.int32) if want_inliers else None
        self._check(self.lib.cvg_detect_pairs(self.handle, models.handle, _ptr(t), _ptr(k), t.shape[0], float(scale),
                                              C.byref(p), _ptr(res), _ptr(inl), _ptr(ioff)))
        if want_inliers:
            return res[:V], inl[:ioff[V]], ioff
        return res[:V], None, None

    def detect_scenes(self, models, scenes, scales=None, params=None):
        """Every view x every resident scene (no host->device input traffic). -> [S, V] structured array."""
        p = params if params is not None else detect_params()
        S, V = scenes.n_scenes, models.n_views
        res = np.zeros(max(S * V, 1), PAIR_DTYPE)
        sc = np.ascontiguousarray(scales, np.float32) if scales is not None else None
        self._check(self.lib.cvg_detect_scenes(self.handle, models.handle, scenes.handle, _ptr(sc), C.byref(p), _ptr(res)))
        return res[:S * V].reshape(S, V)

    def detect_scenes_inliers(self, models, scenes, scales=None, params=None):
        """detect_scenes + the inlier scene points of the accepted pairs -> ([S, V] results, xy [k,2], offsets [S*V+1])."""
        p = params if params is not None else detect_params()
        S, V = scenes.n_scenes, models.n_views
        res = np.zeros(max(S * V, 1), PAIR_DTYPE)
        sc = np.ascontiguousarray(scales, np.float32) if scales is not None else None
        inl = np.zeros((max(S * models.n_rows, 1), 2), np.float32)
        off = np.zeros(S * V + 1, np.int64)
        self._check(self.lib.cvg_detect_scenes_inliers(self.handle, models.handle, scenes.handle, _ptr(sc), C.byref(p),
                                                       _ptr(res), _ptr(inl), _ptr(off)))
        return res[:S * V].reshape(S, V), inl[:off[-1]], off

    def submit_scenes(self, models, scenes, scales=None, params=None, want_inliers=True):
        """Asynchronous detect_scenes_inliers: returns a Job at once (cvg_detect_scenes_submit); Job.wait() gives the results.
        A single-threaded caller keeps two or three jobs in flight to overlap them on the GPU."""
        p = params if params is not None else detect_params()
        S, V = scenes.n_scenes, models.n_views
        res = np.zeros(max(S * V, 1), PAIR_DTYPE)
        sc = np.ascontiguousarray(scales, np.float32) if scales is not None else None
        inl = np.zeros((max(S * models.n_rows, 1), 2), np.float32) if want_inliers else None
        off = np.zeros(S * V + 1, np.int64) if want_inliers else None
        h = C.c_void_p()
        self._check(self.lib.cvg_detect_scenes_submit(self.handle, models.handle, scenes.handle, _ptr(sc), C.byref(p),
                                                      _ptr(res), _ptr(inl), _ptr(off), C.byref(h)))
        return Job(self, h, res, inl, off, S, V, keep=(models, scenes, sc, p))

    def match_knn2_sharded(self, query, train, ratio=0.9):
        """Train-tile sharded knnMatch over the GPUs of a multi-device context (one all-gather + merge)."""
        q = _f32(query, 128); t = _f32(train, 128)
        nq = q.shape[0]
        idx = np.full((nq, 2), -1, np.int32); dist = np.zeros((nq, 2), np.float32); acc = np.zeros(nq, np.uint8)
        self._check(self.lib.cvg_match_knn2_sharded(self.handle, _ptr(q), nq, _ptr(t), t.shape[0], ratio,
                                                    _ptr(idx), _ptr(dist), _ptr(acc)))
        return idx, dist, acc

    def find_homography_sharded(self, src, dst, threshold=5.0, max_iters=2000, confidence=0.995, flags=0,
                                want_ransac_mask=False):
        """find_homography for one point set with the hypotheses of every round split over the GPUs of a multi-device
        context (one all-gather of inlier counts per round).  -> the dict find_homography_batch returns for one set:
        H 3x3, mask [n], found (bool), iters (int), and ransac_mask [n] when asked for.  Raises for n < 4 like OpenCV."""
        s = _f32(src, 2); d = _f32(dst, 2)
        n = s.shape[0]
        if d.shape[0] != n:
            raise ValueError("src and dst must have the same number of points")
        H = np.zeros(9); mask = np.zeros(max(n, 1), np.uint8); found = C.c_int(0); iters = np.zeros(1, np.int32)
        rmask = np.zeros(max(n, 1), np.uint8) if want_ransac_mask else None
        p = ransac_params(threshold, max_iters, confidence, flags)
        self._check(self.lib.cvg_find_homography_sharded(self.handle, _ptr(s), _ptr(d), n, C.byref(p), _ptr(H), _ptr(mask),
                                                         C.byref(found), _ptr(iters), _ptr(rmask)))
        out = {"H": H.reshape(3, 3), "mask": mask[:n], "found": bool(found.value), "iters": int(iters[0])}
        if want_ransac_mask:
            out["ransac_mask"] = rmask[:n]
        return out

    def last_exchange(self):
        """(exchange steps, their device ms on the first GPU) of the last find_homography_sharded call."""
        k, t = C.c_int(0), C.c_float(0)
        self._check(self.lib.cvg_last_exchange(self.handle, C.byref(k), C.byref(t)))
        return k.value, t.value

    # ---- device-pointer building blocks (multi-GPU train-tile shards) ---------------------------
    def dev_match_top2(self, query_ptr, n_query, train_ptr, n_train, index_base, dist_ptr, idx_ptr, stream=None):
        self._check(self.lib.cvg_dev_match_top2(self.handle, stream, query_ptr, n_query, train_ptr, n_train,
                                                index_base, dist_ptr, idx_ptr))

    def dev_merge_top2(self, dist_parts_ptr, idx_parts_ptr, n_parts, n_query, ratio, idx_ptr, dist_ptr, accept_ptr,
                       stream=None):
        self._check(self.lib.cvg_dev_merge_top2(self.handle, stream, dist_parts_ptr, idx_parts_ptr, n_parts, n_query,
                                                ratio, idx_ptr, dist_ptr, accept_ptr))
