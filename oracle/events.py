"""ctypes front-end of oracle/esr_oracle.c (TEST INFRASTRUCTURE ONLY; see that file's header).

Each function mirrors the reference call it restates:
  events_to_channels  <- dataloader/encodings.py:289-304 (+ :243-268)
  lift_coords         <- dataloader/h5dataset.py:508-528
  cnt2event           <- dataloader/cython_cnt2event/cnt2event.pyx:18-116
  event_redistribute  <- dataloader/cython_event_redistribute/event_redistribute.pyx:17-153
"""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "esr_oracle.c")
_SO = os.path.join(_HERE, "_build", "libesr_oracle.so")
_lib = None

_f32p = ctypes.POINTER(ctypes.c_float)
_f64p = ctypes.POINTER(ctypes.c_double)
_i64p = ctypes.POINTER(ctypes.c_int64)


def _stale(so):
    return not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(_SRC)


def build(force=False, so=_SO):
    if force or _stale(so):
        os.makedirs(os.path.dirname(so), exist_ok=True)
        subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fPIC", "-shared", _SRC, "-o", so, "-lm"])
    return so


def lib():
    global _lib
    if _lib is None:
        if not _stale(_SO):
            _lib = ctypes.CDLL(_SO)
        else:                       # not built, or older than its source: compile outside the tree, which may be read-only
            with tempfile.TemporaryDirectory() as d:
                _lib = ctypes.CDLL(build(so=os.path.join(d, "libesr_oracle.so")))
        _lib.oracle_total_events.restype = ctypes.c_int64
    return _lib


def _p(a, t):
    return a.ctypes.data_as(t)


def events_to_channels(xs, ys, ps, sensor_size):
    """xs, ys (float32 numpy, MUTATED in place like the reference), ps -> float32 [2,H,W]."""
    H, W = int(sensor_size[0]), int(sensor_size[1])
    assert xs.dtype == np.float32 and ys.dtype == np.float32
    ps = np.ascontiguousarray(ps, dtype=np.float32)
    out = np.zeros((2, H, W), dtype=np.float32)
    rc = lib().oracle_events_to_channels(_p(xs, _f32p), _p(ys, _f32p), _p(ps, _f32p),
                                         ctypes.c_int64(xs.shape[0]), H, W, _p(out, _f32p))
    assert rc == 0
    return out


def lift_coords(x, res_lr, res_hr):
    x = np.ascontiguousarray(x, dtype=np.float32)
    out = np.empty_like(x)
    lib().oracle_lift_coords(_p(x, _f32p), ctypes.c_int64(x.shape[0]), int(res_lr), int(res_hr), _p(out, _f32p))
    return out


def _random_stream(vals):
    """numpy's legacy global-RNG stream the reference consumes in mode 1 (np.random.seed(123) per call)."""
    n = lib().oracle_total_events(_p(vals, _f32p), ctypes.c_int64(vals.size))
    rs = np.random.RandomState(123)
    return rs.random_sample(int(n)) if n > 0 else np.zeros(1)


def _expand(fn, vals, dims, mode):
    vals = np.ascontiguousarray(vals, dtype=np.float32)
    B = vals.shape[0]
    lens = np.zeros(B, dtype=np.int64)
    maxlen = ctypes.c_int64(0)
    rnd = _random_stream(vals) if mode == 1 else None
    rp = _p(rnd, _f64p) if rnd is not None else None
    rc = fn(_p(vals, _f32p), *dims, int(mode), rp, _p(lens, _i64p), ctypes.byref(maxlen), None)
    if rc == -2:
        raise ValueError("negative dimensions are not allowed")
    assert rc == 0
    out = np.zeros((B, maxlen.value, 4), dtype=np.float32)
    rc = fn(_p(vals, _f32p), *dims, int(mode), rp, _p(lens, _i64p), ctypes.byref(maxlen), _p(out, _f32p))
    assert rc == 0
    return out


def cnt2event(event_cnt, mode=0):
    assert event_cnt.ndim == 4 and event_cnt.shape[1] == 2, "Wrong event count data!"
    B, _, H, W = event_cnt.shape
    return _expand(lib().oracle_cnt2event, event_cnt, (B, H, W), mode)


def event_redistribute(event_stack, mode=0):
    if event_stack.ndim == 5:
        B, P, C, H, W = event_stack.shape
    elif event_stack.ndim == 4:
        B, C, H, W = event_stack.shape
        P = 1
    else:
        raise Exception("wrong event stack")
    return _expand(lib().oracle_event_redistribute, event_stack, (B, P, C, H, W), mode)


def events_to_stack_no_polarity(xs, ys, ts, ps, B, sensor_size):
    """float32 numpy arrays (xs, ys, ps MUTATED in place like the reference) -> float32 [B,H,W]"""
    H, W = int(sensor_size[0]), int(sensor_size[1])
    n = len(ts)
    out = np.zeros((B, H, W), dtype=np.float32)
    if n <= 3 or float(ts.sum()) == 0:
        return out
    bounds = np.zeros(2 * B, dtype=np.int64)
    lib().oracle_time_bin_bounds(_p(np.ascontiguousarray(ts, np.float32), _f32p), ctypes.c_int64(n), int(B), _p(bounds, _i64p))
    for b in range(B):
        beg, end = int(bounds[2 * b]), int(bounds[2 * b + 1])
        sx, sy, sp = xs[beg:end], ys[beg:end], ps[beg:end]           # views: in-place side effects reach the caller
        lib().oracle_events_to_image_inplace(_p(sx, _f32p), _p(sy, _f32p), _p(sp, _f32p), ctypes.c_int64(len(sx)), H, W,
                                             _p(out[b], _f32p))
    return out


def events_to_voxel(xs, ys, ts, ps, num_bins, sensor_size):
    H, W = int(sensor_size[0]), int(sensor_size[1])
    out = np.zeros((num_bins, H, W), dtype=np.float32)
    ts = np.ascontiguousarray(ts, np.float32)
    ps = np.ascontiguousarray(ps, np.float32)
    rc = lib().oracle_events_to_voxel(_p(xs, _f32p), _p(ys, _f32p), _p(ts, _f32p), _p(ps, _f32p), ctypes.c_int64(len(xs)),
                                      int(num_bins), H, W, _p(out, _f32p))
    assert rc == 0
    return out
