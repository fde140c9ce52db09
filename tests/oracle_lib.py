"""ctypes binding of the CPU oracle (oracle/libm3tsz_oracle.so).

Test infrastructure only: importable from tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs.  The product package never
imports this module.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_DIR = os.path.join(_HERE, "..", "oracle")
_LIB_PATH = os.path.join(ORACLE_DIR, "libm3tsz_oracle.so")

UNIT_NONE, UNIT_S, UNIT_MS, UNIT_US, UNIT_NS = 0, 1, 2, 3, 4
OK, ERR_EOF = 0, 1
ERR_DOD_OVERFLOW = 4


def build_oracle(force=False):
    srcs = [os.path.join(ORACLE_DIR, f) for f in ("m3tsz_oracle.c", "m3tsz_merge_oracle.c",
                                                  "m3tsz_segment_oracle.c", "m3tsz_query_oracle.c",
                                                  "m3tsz_oracle.h")]
    if (not force and os.path.exists(_LIB_PATH)
            and os.path.getmtime(_LIB_PATH) >= max(os.path.getmtime(f) for f in srcs)):
        return _LIB_PATH
    subprocess.check_call(["make", "-C", ORACLE_DIR, "-s"])
    return _LIB_PATH


_lib = None

u8p = C.POINTER(C.c_uint8)
i64p = C.POINTER(C.c_int64)
u64p = C.POINTER(C.c_uint64)
f64p = C.POINTER(C.c_double)
i32p = C.POINTER(C.c_int32)
u32p = C.POINTER(C.c_uint32)


def lib():
    global _lib
    if _lib is not None:
        return _lib
    L = C.CDLL(build_oracle())
    vp = C.c_void_p
    sigs = {
        "m3o_ostream_new": (vp, []),
        "m3o_ostream_free": (None, [vp]),
        "m3o_ostream_reset": (None, [vp]),
        "m3o_ostream_write_bit": (None, [vp, C.c_int]),
        "m3o_ostream_write_byte": (None, [vp, C.c_uint8]),
        "m3o_ostream_write_bytes": (None, [vp, C.c_char_p, C.c_size_t]),
        "m3o_ostream_write_bits": (None, [vp, C.c_uint64, C.c_int]),
        "m3o_ostream_raw": (C.c_size_t, [vp, C.POINTER(u8p), C.POINTER(C.c_int)]),
        "m3o_istream_new": (vp, [C.c_char_p, C.c_size_t]),
        "m3o_istream_free": (None, [vp]),
        "m3o_istream_read_bits": (C.c_int, [vp, C.c_int, u64p]),
        "m3o_istream_peek_bits": (C.c_int, [vp, C.c_int, u64p]),
        "m3o_istream_remaining_bits_in_current_byte": (C.c_int, [vp]),
        "m3o_num_sig": (C.c_int, [C.c_uint64]),
        "m3o_sign_extend": (C.c_int64, [C.c_uint64, C.c_int]),
        "m3o_convert_to_int_float": (C.c_int, [C.c_double, C.c_int, f64p, C.POINTER(C.c_int),
                                               C.POINTER(C.c_int)]),
        "m3o_convert_from_int_float": (C.c_double, [C.c_double, C.c_int]),
        "m3o_initial_time_unit": (C.c_int, [C.c_int64, C.c_int]),
        "m3o_xxh64": (C.c_uint64, [C.c_char_p, C.c_size_t]),
        "m3o_write_dod_unit_unchanged": (C.c_int, [vp, C.c_int64, C.c_int64, C.c_int]),
        "m3o_write_dod_unit_changed": (None, [vp, C.c_int64, C.c_int64]),
        "m3o_write_xor": (None, [vp, C.c_uint64, C.c_uint64]),
        "m3o_encoder_new": (vp, [C.c_int64, C.c_int, C.c_int]),
        "m3o_encoder_free": (None, [vp]),
        "m3o_encoder_reset": (None, [vp, C.c_int64]),
        "m3o_encoder_encode": (C.c_int, [vp, C.c_int64, C.c_double, C.c_int, C.c_char_p, C.c_size_t]),
        "m3o_encoder_num_encoded": (C.c_int, [vp]),
        "m3o_encoder_last_encoded": (C.c_int, [vp, i64p, f64p]),
        "m3o_encoder_last_annotation_checksum": (C.c_int, [vp, u64p]),
        "m3o_encoder_len": (C.c_size_t, [vp]),
        "m3o_encoder_empty": (C.c_int, [vp]),
        "m3o_encoder_stream": (C.c_size_t, [vp, C.c_char_p, C.c_size_t]),
        "m3o_encoder_raw": (C.c_size_t, [vp, C.POINTER(u8p), C.POINTER(C.c_int)]),
        "m3o_encoder_close": (None, [vp]),
        "m3o_iter_new": (vp, [C.c_char_p, C.c_size_t, C.c_int, C.c_int]),
        "m3o_iter_free": (None, [vp]),
        "m3o_iter_reset": (None, [vp, C.c_char_p, C.c_size_t]),
        "m3o_iter_next": (C.c_int, [vp]),
        "m3o_iter_current": (None, [vp, i64p, f64p, C.POINTER(C.c_int), C.POINTER(u8p),
                                    C.POINTER(C.c_size_t)]),
        "m3o_iter_err": (C.c_int, [vp]),
        "m3o_iter_done": (C.c_int, [vp]),
        "m3o_iter_set_float_state": (None, [vp, C.c_uint64, C.c_uint64]),
        "m3o_iter_get_float_state": (None, [vp, u64p, u64p]),
        "m3o_iter_read_next_value": (None, [vp]),
        "m3o_iter_set_ts_state": (None, [vp, C.c_int, C.c_int64]),
        "m3o_iter_read_next_timestamp": (C.c_int, [vp]),
        "m3o_iter_read_first_timestamp": (C.c_int, [vp]),
        "m3o_iter_prev_time_delta": (C.c_int64, [vp]),
        "m3o_iter_read_annotation": (C.c_int, [vp, C.POINTER(u8p), C.POINTER(C.c_size_t)]),
        "m3o_iter_read_time_unit": (C.c_int, [vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
        "m3o_encode_series": (C.c_int64, [vp, vp, C.c_size_t, C.c_int64, C.c_int, C.c_int, C.c_int,
                                          vp, C.c_size_t]),
        "m3o_decode_series": (C.c_int64, [vp, C.c_size_t, C.c_int, C.c_int, vp, vp, C.c_size_t,
                                          C.POINTER(C.c_int)]),
        "m3o_decode_batch": (C.c_int, [vp, vp, C.c_size_t, C.c_int, C.c_int, vp, vp, C.c_size_t, vp,
                                       vp, C.c_int]),
        "m3o_encode_batch": (C.c_int, [vp, vp, C.c_size_t, C.c_size_t, vp, C.c_int, C.c_int, C.c_int,
                                       vp, C.c_size_t, vp, vp, C.c_int]),
        "m3o_downsample_series": (None, [vp, vp, C.c_size_t, C.c_int64, C.c_int64, C.c_size_t, vp, vp,
                                         vp, vp, vp]),
        "m3o_prom_convert_series": (C.c_size_t, [vp, vp, C.c_size_t, C.c_int64, C.c_int, C.c_double, C.c_int64,
                                                 vp, vp, C.c_size_t]),
        "m3o_gauge_value_of": (C.c_double, [C.c_int, C.c_double, C.c_int64, C.c_double, C.c_double,
                                            C.c_double]),
        "m3o_aggregate_tiles_series": (C.c_size_t, [vp, vp, C.c_size_t, C.c_int64, C.c_int64, C.c_size_t,
                                                    C.c_int, vp, vp]),
        "m3o_series_merge_batch": (None, [vp, vp, C.c_uint64, vp, vp, vp, vp, vp, C.c_uint64, C.c_int64,
                                          C.c_int64, C.c_int, vp, vp, C.c_uint64, vp, vp]),
        "m3o_adler32": (C.c_uint32, [C.c_char_p, C.c_size_t]),
        "m3o_adler32_batch": (None, [vp, vp, C.c_uint64, vp, vp, vp]),
    }
    for name, (res, args) in sigs.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


# ---------------------------------------------------------------------------
# pythonic wrappers
# ---------------------------------------------------------------------------
class OStream:
    def __init__(self):
        self.h = lib().m3o_ostream_new()

    def __del__(self):
        if getattr(self, "h", None):
            lib().m3o_ostream_free(self.h)
            self.h = None

    def write_bits(self, v, n):
        lib().m3o_ostream_write_bits(self.h, v & 0xFFFFFFFFFFFFFFFF, n)

    def write_bytes(self, b):
        lib().m3o_ostream_write_bytes(self.h, bytes(b), len(b))

    def raw(self):
        p = u8p()
        pos = C.c_int()
        n = lib().m3o_ostream_raw(self.h, C.byref(p), C.byref(pos))
        return (bytes(p[:n]) if n else b""), pos.value


class IStream:
    def __init__(self, data):
        self._data = bytes(data)
        self.h = lib().m3o_istream_new(self._data, len(self._data))

    def __del__(self):
        if getattr(self, "h", None):
            lib().m3o_istream_free(self.h)
            self.h = None

    def read_bits(self, n):
        out = C.c_uint64()
        err = lib().m3o_istream_read_bits(self.h, n, C.byref(out))
        return out.value, err

    def peek_bits(self, n):
        out = C.c_uint64()
        err = lib().m3o_istream_peek_bits(self.h, n, C.byref(out))
        return out.value, err

    def remaining_bits_in_current_byte(self):
        return lib().m3o_istream_remaining_bits_in_current_byte(self.h)


class Encoder:
    """Mirror of m3tsz.NewEncoder(start, nil, intOptimized, opts)."""

    def __init__(self, start_ns, int_optimized, default_unit=UNIT_S):
        self.h = lib().m3o_encoder_new(start_ns, int(int_optimized), default_unit)

    def __del__(self):
        if getattr(self, "h", None):
            lib().m3o_encoder_free(self.h)
            self.h = None

    def reset(self, start_ns):
        lib().m3o_encoder_reset(self.h, start_ns)

    def encode(self, ts_ns, value, unit=UNIT_S, annotation=b""):
        annotation = bytes(annotation or b"")
        return lib().m3o_encoder_encode(self.h, ts_ns, float(value), unit,
                                        annotation if annotation else None, len(annotation))

    def num_encoded(self):
        return lib().m3o_encoder_num_encoded(self.h)

    def last_encoded(self):
        t = C.c_int64()
        v = C.c_double()
        err = lib().m3o_encoder_last_encoded(self.h, C.byref(t), C.byref(v))
        return t.value, v.value, err

    def last_annotation_checksum(self):
        s = C.c_uint64()
        err = lib().m3o_encoder_last_annotation_checksum(self.h, C.byref(s))
        return s.value, err

    def len(self):
        return lib().m3o_encoder_len(self.h)

    def empty(self):
        return bool(lib().m3o_encoder_empty(self.h))

    def stream(self):
        n = lib().m3o_encoder_len(self.h)
        if n == 0:
            return None
        buf = C.create_string_buffer(n)
        got = lib().m3o_encoder_stream(self.h, buf, n)
        assert got == n
        return buf.raw

    def raw(self):
        p = u8p()
        pos = C.c_int()
        n = lib().m3o_encoder_raw(self.h, C.byref(p), C.byref(pos))
        return (bytes(p[:n]) if n else b""), pos.value

    def close(self):
        lib().m3o_encoder_close(self.h)


class Iterator:
    """Mirror of m3tsz.NewReaderIterator(reader, intOptimized, opts)."""

    def __init__(self, data, int_optimized, default_unit=UNIT_S):
        self._data = bytes(data)
        self.h = lib().m3o_iter_new(self._data, len(self._data), int(int_optimized), default_unit)

    def __del__(self):
        if getattr(self, "h", None):
            lib().m3o_iter_free(self.h)
            self.h = None

    def next(self):
        return bool(lib().m3o_iter_next(self.h))

    def current(self):
        t = C.c_int64()
        v = C.c_double()
        u = C.c_int()
        p = u8p()
        n = C.c_size_t()
        lib().m3o_iter_current(self.h, C.byref(t), C.byref(v), C.byref(u), C.byref(p), C.byref(n))
        ann = bytes(p[: n.value]) if n.value else b""
        return t.value, v.value, u.value, ann

    def err(self):
        return lib().m3o_iter_err(self.h)

    def done(self):
        return bool(lib().m3o_iter_done(self.h))


def decode_all(data, int_optimized, default_unit=UNIT_S):
    """Returns (list of (ts, value, unit, annotation), err)."""
    it = Iterator(data, int_optimized, default_unit)
    out = []
    while it.next():
        out.append(it.current())
    return out, it.err()


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def encode_series(ts, vals, start_ns, unit=UNIT_S, int_optimized=True, default_unit=UNIT_S):
    ts = np.ascontiguousarray(ts, dtype=np.int64)
    vals = np.ascontiguousarray(vals, dtype=np.float64)
    cap = 64 + 20 * len(ts)
    out = np.empty(cap, dtype=np.uint8)
    n = lib().m3o_encode_series(_ptr(ts), _ptr(vals), len(ts), int(start_ns), unit,
                                int(int_optimized), default_unit, _ptr(out), cap)
    if n < 0:
        raise ValueError("oracle encode error %d" % -n)
    return out[:n].tobytes()


def decode_series(data, int_optimized=True, default_unit=UNIT_S, cap=4096):
    buf = np.frombuffer(bytes(data), dtype=np.uint8)
    ts = np.empty(cap, dtype=np.int64)
    vals = np.empty(cap, dtype=np.float64)
    err = C.c_int()
    n = lib().m3o_decode_series(_ptr(buf), len(buf), int(int_optimized), default_unit, _ptr(ts),
                                _ptr(vals), cap, C.byref(err))
    return ts[: min(n, cap)].copy(), vals[: min(n, cap)].copy(), n, err.value


def encode_batch(ts, vals, start_ns, unit=UNIT_S, int_optimized=True, default_unit=UNIT_S,
                 out_stride=None, n_threads=1, bufs=None):
    """ts, vals: [S, P] arrays.  Returns (out[S, stride] uint8, out_len[S] uint64, status[S]).
    `bufs` = (out, out_len, status) reuses preallocated outputs (timing runs)."""
    ts = np.ascontiguousarray(ts, dtype=np.int64)
    vals = np.ascontiguousarray(vals, dtype=np.float64)
    S, P = ts.shape
    start = np.ascontiguousarray(np.broadcast_to(np.asarray(start_ns, dtype=np.int64), (S,)))
    if bufs is not None:
        out, out_len, status = bufs
        out_stride = out.shape[1]
    else:
        if out_stride is None:
            out_stride = 64 + 20 * P
        out = np.zeros((S, out_stride), dtype=np.uint8)
        out_len = np.zeros(S, dtype=np.uint64)
        status = np.zeros(S, dtype=np.int32)
    lib().m3o_encode_batch(_ptr(ts), _ptr(vals), S, P, _ptr(start), unit, int(int_optimized),
                           default_unit, _ptr(out), out_stride, _ptr(out_len), _ptr(status),
                           n_threads)
    return out, out_len, status


def decode_batch(streams, off, cap, int_optimized=True, default_unit=UNIT_S, n_threads=1, bufs=None):
    """streams: uint8 [total]; off: uint64 [S+1].  Returns ts[S,cap], vals[S,cap], n[S], status[S]."""
    streams = np.ascontiguousarray(streams, dtype=np.uint8)
    off = np.ascontiguousarray(off, dtype=np.uint64)
    S = len(off) - 1
    if bufs is not None:
        ts, vals, n, status = bufs
    else:
        ts = np.zeros((S, cap), dtype=np.int64)
        vals = np.zeros((S, cap), dtype=np.float64)
        n = np.zeros(S, dtype=np.uint32)
        status = np.zeros(S, dtype=np.int32)
    lib().m3o_decode_batch(_ptr(streams), _ptr(off), S, int(int_optimized), default_unit, _ptr(ts),
                           _ptr(vals), cap, _ptr(n), _ptr(status), n_threads)
    return ts, vals, n, status


def downsample_series(ts, vals, range_start_ns, window_ns, n_windows):
    ts = np.ascontiguousarray(ts, dtype=np.int64)
    vals = np.ascontiguousarray(vals, dtype=np.float64)
    s = np.empty(n_windows, dtype=np.float64)
    c = np.empty(n_windows, dtype=np.int64)
    mn = np.empty(n_windows, dtype=np.float64)
    mx = np.empty(n_windows, dtype=np.float64)
    last = np.empty(n_windows, dtype=np.float64)
    lib().m3o_downsample_series(_ptr(ts), _ptr(vals), len(ts), int(range_start_ns), int(window_ns),
                                n_windows, _ptr(s), _ptr(c), _ptr(mn), _ptr(mx), _ptr(last))
    return s, c, mn, mx, last


AGG_LAST, AGG_MIN, AGG_MAX, AGG_MEAN, AGG_COUNT, AGG_SUM = 1, 2, 3, 4, 6, 7  # aggregation.Type ids


def prom_convert_series(ts, vals, resolution_ns, handle_resets, tolerance=0.0, until_ns=0):
    """iteratorToPromResult over one decoded series -> (ts_ms int64[], values float64[])."""
    ts = np.ascontiguousarray(ts, dtype=np.int64)
    vals = np.ascontiguousarray(vals, dtype=np.float64)
    cap = len(ts) + 1
    to = np.zeros(cap, dtype=np.int64)
    vo = np.zeros(cap, dtype=np.float64)
    n = lib().m3o_prom_convert_series(_ptr(ts), _ptr(vals), len(ts), int(resolution_ns), int(bool(handle_resets)),
                                      float(tolerance), int(until_ns), _ptr(to), _ptr(vo), cap)
    return to[:n].copy(), vo[:n].copy()


def gauge_value_of(agg_type, s, c, mn, mx, last):
    return float(lib().m3o_gauge_value_of(int(agg_type), float(s), int(c), float(mn), float(mx), float(last)))


def aggregate_tiles_series(ts, vals, start_ns, step_ns, n_windows, agg_type):
    ts = np.ascontiguousarray(ts, dtype=np.int64)
    vals = np.ascontiguousarray(vals, dtype=np.float64)
    to = np.zeros(max(1, n_windows), dtype=np.int64)
    vo = np.zeros(max(1, n_windows), dtype=np.float64)
    n = lib().m3o_aggregate_tiles_series(_ptr(ts), _ptr(vals), len(ts), int(start_ns), int(step_ns),
                                         int(n_windows), int(agg_type), _ptr(to), _ptr(vo))
    return to[:n].copy(), vo[:n].copy()


def convert_to_int_float(v, cur_max_mult):
    val = C.c_double()
    mult = C.c_int()
    isf = C.c_int()
    err = lib().m3o_convert_to_int_float(float(v), cur_max_mult, C.byref(val), C.byref(mult),
                                         C.byref(isf))
    return val.value, mult.value, bool(isf.value), err


def series_merge_batch(ts, vals, n_points, seq_status, slice_off, replica_off, series_off, start=0, end=0,
                       strategy=0, out_cap=None):
    """Oracle of the iterator layer (iterators / multiReaderIterator / seriesIterator).
    ts, vals: [n_seq, cap]; returns (ts_out[S,out_cap], val_out, n_out[S], status[S])."""
    ts = np.ascontiguousarray(ts, dtype=np.int64)
    vals = np.ascontiguousarray(vals, dtype=np.float64)
    n_points = np.ascontiguousarray(n_points, dtype=np.uint32)
    seq_status = np.ascontiguousarray(seq_status, dtype=np.int32)
    slice_off = np.ascontiguousarray(slice_off, dtype=np.uint64)
    replica_off = np.ascontiguousarray(replica_off, dtype=np.uint64)
    series_off = np.ascontiguousarray(series_off, dtype=np.uint64)
    S = len(series_off) - 1
    cap = ts.shape[1] if ts.ndim == 2 and ts.shape[0] else 1
    if out_cap is None:
        out_cap = max(1, int(n_points.sum()))
    ts_out = np.zeros((S, out_cap), dtype=np.int64)
    val_out = np.zeros((S, out_cap), dtype=np.float64)
    n_out = np.zeros(S, dtype=np.uint32)
    status = np.zeros(S, dtype=np.int32)
    lib().m3o_series_merge_batch(_ptr(ts), _ptr(vals), cap, _ptr(n_points), _ptr(seq_status), _ptr(slice_off),
                                 _ptr(replica_off), _ptr(series_off), S, int(start), int(end), int(strategy),
                                 _ptr(ts_out), _ptr(val_out), out_cap, _ptr(n_out), _ptr(status))
    return ts_out, val_out, n_out, status


def adler32(data: bytes) -> int:
    """Segment checksum oracle (Adler-32 of the stream bytes)."""
    return int(lib().m3o_adler32(bytes(data), len(data)))


def adler32_batch(blob, offsets, expected=None):
    """Checksums of the CSR streams blob[offsets[s]:offsets[s+1]]; returns (checksums u32[S], status i32[S])."""
    blob = np.ascontiguousarray(np.frombuffer(bytes(blob), dtype=np.uint8)) if not isinstance(blob, np.ndarray) \
        else np.ascontiguousarray(blob, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    S = len(offsets) - 1
    out = np.zeros(S, dtype=np.uint32)
    status = np.zeros(S, dtype=np.int32)
    exp = None if expected is None else np.ascontiguousarray(expected, dtype=np.uint32)
    if len(blob) == 0:
        blob = np.zeros(1, dtype=np.uint8)
    lib().m3o_adler32_batch(_ptr(blob), _ptr(offsets), S, None if exp is None else _ptr(exp), _ptr(out),
                            _ptr(status))
    return out, status
