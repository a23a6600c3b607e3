"""LikelihoodContext: a histogram resident on one B200 plus the batched evaluators over it.

Thin object wrapper over the C ABI (include/covest_b200.h).  Buffers may be numpy arrays (host;
the copies to and from the device are part of the call) or CUDA torch tensors (used in place).
"""
import ctypes
import math
import os

import numpy as np

from . import _capi


class DeviceError(RuntimeError):
    """An error reported by libcovest_b200 (bad argument or CUDA failure)."""


def default_device():
    for var in ('COVEST_B200_DEVICE', 'LOCAL_RANK'):
        v = os.environ.get(var)
        if v not in (None, ''):
            return int(v)
    return 0


def _is_torch_cuda(x):
    return hasattr(x, 'data_ptr') and hasattr(x, 'is_cuda') and x.is_cuda


def _host_out(n, dtype=np.float64):
    """A host output buffer of n values: page-locked when it is large and torch is at hand (the
    device -> host copy of 10^6 values is 4x faster into pinned memory), else a plain array."""
    if n >= (1 << 17):
        try:
            import torch
            if torch.cuda.is_available():
                return torch.empty(int(n), dtype=torch.float64, pin_memory=True).numpy()
        except Exception:
            pass
    return np.empty(n, dtype=dtype)


def _ptr(x):
    if x is None:
        return None
    if _is_torch_cuda(x):
        return ctypes.c_void_p(x.data_ptr())
    return ctypes.c_void_p(x.ctypes.data)


CUDA_STREAM_LEGACY = 1  # cudaStreamLegacy: the handle that names the default stream explicitly


def _stream_ptr(stream, like=None):
    """None -> NULL (the context's own stream, synchronised before a host-buffer call returns) --
    unless `like` is a torch CUDA tensor: work on device buffers is only enqueued, so it goes to
    torch's current stream of that device, where the caller's next torch operation is ordered
    behind it.  A torch stream or a raw cudaStream_t value is passed through; the default stream,
    whose raw value is 0, is named by cudaStreamLegacy so that it is not mistaken for "no stream
    given"."""
    if stream is None:
        if like is None or not _is_torch_cuda(like):
            return None
        import torch
        stream = torch.cuda.current_stream(like.device)
    value = stream.cuda_stream if hasattr(stream, 'cuda_stream') else int(stream)
    return ctypes.c_void_p(value if value else CUDA_STREAM_LEGACY)


def profile_segments(lens, keep_mask):
    """Number of segments of a lattice profile (cvb_lattice_profile): the product of the lengths of the
    axes whose bit is set in keep_mask.  The mask must keep at least one axis and name no axis beyond
    len(lens); the product must fit an int64."""
    keep_mask = int(keep_mask)
    if keep_mask <= 0 or keep_mask >> len(lens):
        raise ValueError('keep_mask must be a non-empty set of the bits 0..%d, not %d' % (len(lens) - 1, keep_mask))
    n_seg = 1
    for a, n in enumerate(lens):
        if keep_mask >> a & 1:
            n_seg *= int(n)
    if n_seg >= 1 << 63:
        raise ValueError('a profile of %d segments: more than an int64 counts' % n_seg)
    return n_seg


class LikelihoodContext:
    """Device copies of one histogram and its tables (models.py:19-31, :175-183 state)."""

    def __init__(self, model_kind, k, r, max_error, bin_j, bin_h, tail, threshold, bounds, comb,
                 pow3=None, device=None):
        self._lib = _capi.load()
        self._ctx = ctypes.c_void_p()
        self.n_param = 5 if model_kind == _capi.MODEL_REPEATS else 2
        self.n_bins = len(bin_j)
        self.device = default_device() if device is None else int(device)
        j = np.ascontiguousarray(bin_j, dtype=np.int32)
        h = np.ascontiguousarray(bin_h, dtype=np.float64)
        b = []
        for lo, hi in bounds:
            b += [math.nan if lo is None else float(lo), math.nan if hi is None else float(hi)]
        b = np.ascontiguousarray(b, dtype=np.float64)
        cm = np.ascontiguousarray([float(v) for v in comb[:max_error]], dtype=np.float64)
        if pow3 is None:
            pow3 = [1.0 if s == 0 else float(3 ** -s) for s in range(max_error)]
        p3 = np.ascontiguousarray(pow3, dtype=np.float64)
        thr = math.nan if threshold is None else float(threshold)
        rc = self._lib.cvb_ctx_create(int(model_kind), int(k), int(r), int(max_error), len(j),
                                      j.ctypes.data_as(_capi.c_int32_p),
                                      h.ctypes.data_as(_capi.c_double_p), float(tail), thr,
                                      b.ctypes.data_as(_capi.c_double_p),
                                      cm.ctypes.data_as(_capi.c_double_p),
                                      p3.ctypes.data_as(_capi.c_double_p), self.device,
                                      ctypes.byref(self._ctx))
        if rc != _capi.CVB_OK:
            msg = self._lib.cvb_last_error(None).decode()
            self._ctx = ctypes.c_void_p()
            raise DeviceError('cvb_ctx_create failed (%d): %s' % (rc, msg))

    # -- plumbing --------------------------------------------------------------------------
    def _check(self, rc, what):
        if rc != _capi.CVB_OK:
            raise DeviceError('%s failed (%d): %s' % (what, rc, self._lib.cvb_last_error(self._ctx).decode()))

    def close(self):
        if getattr(self, '_ctx', None) is not None and self._ctx.value:
            self._lib.cvb_ctx_destroy(self._ctx)
            self._ctx = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _points(self, points):
        if _is_torch_cuda(points):
            import torch
            if points.dtype != torch.float64 or not points.is_contiguous():
                raise ValueError('device points must be a contiguous float64 tensor')
            if points.numel() % self.n_param:
                raise ValueError('points must have %d columns' % self.n_param)
            return points, points.numel() // self.n_param
        pts = np.ascontiguousarray(points, dtype=np.float64).reshape(-1, self.n_param)
        return pts, len(pts)

    # -- evaluators ------------------------------------------------------------------------
    def loglik(self, points, out=None, stream=None):
        """compute_loglikelihood over the rows of `points` (models.py:100-117)."""
        pts, n = self._points(points)
        if out is None:
            if _is_torch_cuda(pts):
                import torch
                out = torch.empty(n, dtype=torch.float64, device=pts.device)
            else:
                out = _host_out(n)
        self._check(self._lib.cvb_loglik_batch(self._ctx, n, _ptr(pts), _ptr(out), _stream_ptr(stream, pts)),
                    'cvb_loglik_batch')
        return out

    def probs(self, points, clip=False, with_loglik=False, stream=None):
        """compute_probabilities over the rows of `points` (models.py:81-98, :211-242): an
        (n_points, n_bins) array whose columns follow the key order of `hist`."""
        pts, n = self._points(points)
        if _is_torch_cuda(pts):
            import torch
            out = torch.zeros((n, self.n_bins), dtype=torch.float64, device=pts.device)
            ll = torch.empty(n, dtype=torch.float64, device=pts.device) if with_loglik else None
        else:
            out = np.zeros((n, self.n_bins), dtype=np.float64)
            ll = np.empty(n, dtype=np.float64) if with_loglik else None
        self._check(self._lib.cvb_probs_batch(self._ctx, n, _ptr(pts), int(bool(clip)), _ptr(out),
                                              _ptr(ll), _stream_ptr(stream, pts)), 'cvb_probs_batch')
        return (out, ll) if with_loglik else out

    def topk(self, ll, points, k_best, stream=None):
        """Best-first (k_best, 1 + n_param) rows (loglik, params...)."""
        pts, n = self._points(points)
        if _is_torch_cuda(pts):
            import torch
            rows = torch.empty((k_best, 1 + self.n_param), dtype=torch.float64, device=pts.device)
            llb = ll
        else:
            rows = np.empty((k_best, 1 + self.n_param), dtype=np.float64)
            llb = np.ascontiguousarray(ll, dtype=np.float64)
        self._check(self._lib.cvb_topk(self._ctx, n, _ptr(llb), _ptr(pts), int(k_best), _ptr(rows),
                                       _stream_ptr(stream, pts)), 'cvb_topk')
        return rows

    def loglik_topk(self, points, k_best, want_ll=True, stream=None):
        """loglik + topk in one call (the batch crosses the bus once): (ll or None, rows)."""
        pts, n = self._points(points)
        if _is_torch_cuda(pts):
            import torch
            ll = torch.empty(n, dtype=torch.float64, device=pts.device) if want_ll else None
            rows = torch.empty((k_best, 1 + self.n_param), dtype=torch.float64, device=pts.device)
        else:
            ll = _host_out(n) if want_ll else None
            rows = np.empty((k_best, 1 + self.n_param), dtype=np.float64)
        self._check(self._lib.cvb_loglik_topk(self._ctx, n, _ptr(pts), _ptr(ll), int(k_best),
                                              _ptr(rows), _stream_ptr(stream, pts)), 'cvb_loglik_topk')
        return ll, rows

    def lattice_eval(self, axes, first=0, stride=1, count=None, want_ll=True, k_best=0,
                     out_ll=None, stream=None, block=1, out_rows=None):
        """Evaluate the Cartesian lattice of `axes` (one 1-D array per model parameter, last axis
        fastest), generating the points on the device: runs of `block` consecutive lattice
        indices, run j starting at (first + j*stride)*block -- with block = 1 the indices
        first + i*stride, i < count.  Returns (ll or None, rows or None).  `out_ll` / `out_rows`
        may be CUDA tensors: the call then only enqueues work (on `stream`, default torch's
        current stream)."""
        lens, vals, count = self._lattice_slice(axes, first, stride, block, count)
        ll = out_ll
        if ll is None and want_ll:
            ll = _host_out(count)
        rows = out_rows
        if rows is None and k_best > 0:
            rows = np.empty((k_best, 1 + self.n_param), dtype=np.float64)
        like = ll if _is_torch_cuda(ll) else rows
        self._check(self._lib.cvb_lattice_eval(self._ctx, lens.ctypes.data_as(_capi.c_int32_p),
                                               vals.ctypes.data_as(_capi.c_double_p), int(first),
                                               int(stride), int(block), int(count), _ptr(ll), int(k_best),
                                               _ptr(rows), _stream_ptr(stream, like)), 'cvb_lattice_eval')
        return ll, rows

    def _lattice_slice(self, axes, first, stride, block, count):
        """(axis lengths, concatenated axis values, count) of a lattice call; count None = every run
        of the slice up to the end of the lattice."""
        if len(axes) != self.n_param:
            raise ValueError('need %d axes' % self.n_param)
        lens = np.ascontiguousarray([len(a) for a in axes], dtype=np.int32)
        vals = np.ascontiguousarray(np.concatenate([np.asarray(a, dtype=np.float64).ravel() for a in axes]))
        total = int(np.prod(lens.astype(np.int64)))
        if count is None:
            runs = (total + block - 1) // block
            mine = max(0, (runs - first + stride - 1) // stride)
            count = mine * block
            if mine and (first + (mine - 1) * stride + 1) * block > total:
                count -= (first + (mine - 1) * stride + 1) * block - total
        return lens, vals, count

    def lattice_profile(self, axes, keep_mask, first=0, stride=1, block=1, count=None, out_rows=None, stream=None):
        """For every segment of the slice of lattice_eval (the points that share the values of the axes
        whose bit is set in `keep_mask`), the (loglik, params...) row of its best point: an
        (n_seg, 1 + n_param) array, n_seg = the product of the kept axes' lengths, segments numbered
        with the last kept axis fastest (include/covest_b200.h, cvb_lattice_profile).  `out_rows` may
        be a CUDA tensor: the call then only enqueues work (on `stream`, default torch's current
        stream)."""
        lens, vals, count = self._lattice_slice(axes, first, stride, block, count)
        keep_mask = int(keep_mask)
        n_seg = profile_segments(lens, keep_mask)
        rows = out_rows
        if rows is None:
            rows = np.empty((n_seg, 1 + self.n_param), dtype=np.float64)
        self._check(self._lib.cvb_lattice_profile(self._ctx, lens.ctypes.data_as(_capi.c_int32_p),
                                                  vals.ctypes.data_as(_capi.c_double_p), int(first), int(stride),
                                                  int(block), int(count), keep_mask, _ptr(rows),
                                                  _stream_ptr(stream, rows)), 'cvb_lattice_profile')
        return rows

    # -- measurement -----------------------------------------------------------------------
    def fp64_peak(self, kind=0, reps=5):
        """Measured FP64 throughput (TFLOP/s) of register-resident DFMA (0) / DMMA (1) chains, or of
        both running side by side (2)."""
        out = ctypes.c_double()
        self._check(self._lib.cvb_fp64_peak(self._ctx, int(kind), int(reps), ctypes.byref(out)),
                    'cvb_fp64_peak')
        return out.value

    def set_timing(self, on=True):
        self._check(self._lib.cvb_set_timing(self._ctx, int(bool(on))), 'cvb_set_timing')

    def last_kernel_ms(self):
        ms = ctypes.c_double()
        n = ctypes.c_int()
        self._check(self._lib.cvb_last_kernel_ms(self._ctx, ctypes.byref(ms), ctypes.byref(n)),
                    'cvb_last_kernel_ms')
        return ms.value, n.value

    def last_launches(self):
        """Kernels launched by the most recent call (needs no timing)."""
        n = ctypes.c_int()
        self._check(self._lib.cvb_last_kernel_ms(self._ctx, None, ctypes.byref(n)), 'cvb_last_kernel_ms')
        return n.value

    PATH_AUTO, PATH_PER_POINT, PATH_FACTORED, PATH_FACTORED_GEMM, PATH_FACTORED_PREFIX = 0, 1, 2, 3, 4
    PATH_TERM_BY_TERM = 5  # every point through the reference-order evaluation of faithful.cu (slow; a check)

    def set_path(self, mode):
        """Evaluation path of the repeats model: PATH_AUTO, PATH_PER_POINT, PATH_FACTORED (GEMM or
        prefix kernel by the sharing of q), PATH_FACTORED_GEMM or PATH_FACTORED_PREFIX
        (include/covest_b200.h, cvb_set_path)."""
        self._check(self._lib.cvb_set_path(self._ctx, int(mode)), 'cvb_set_path')

    def last_path_info(self):
        """Facts about the most recent evaluation (cvb_last_path_info)."""
        buf = (ctypes.c_double * 12)()
        self._check(self._lib.cvb_last_path_info(self._ctx, buf, 12), 'cvb_last_path_info')
        v = list(buf)
        return {'path': {1: 'per-point', 2: 'factored', 3: 'factored', 4: 'term-by-term'}.get(int(v[0]), 'none'),
                'kernel': {1: 'cv_loglik_kernel', 2: 'cvf_gemm_kernel', 3: 'cvf_prefix_kernel',
                           4: 'cv_faithful_kernel'}.get(int(v[0]), 'none'),
                'groups': int(v[1]), 'tiles': int(v[2]), 'items': int(v[3]), 'profile_doubles': int(v[4]),
                'plan_ms': v[5], 'profile_ms': v[6], 'gemm_ms': v[7], 'q_runs': int(v[8]),
                'refined_points': int(v[9]), 'analytic_plan': bool(v[10]), 'row_slots': int(v[11])}

    @property
    def sm_count(self):
        return self._lib.cvb_device_sm_count(self._ctx)
