"""ctypes binding of libbbkio.so (include/bbk_io.h): the host-side file formats either side of the pass."""
import ctypes
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libbbkio.so")

_vp, _i32, _i64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64
SIGNATURES = {
    "bbkio_last_error": (None, [ctypes.c_char_p, ctypes.c_size_t]),
    "bbkio_write_significances": (ctypes.c_int, [ctypes.c_char_p, ctypes.POINTER(ctypes.c_char_p), _i32, _vp, _vp, _vp, _vp, _vp,
                                                 _vp, _vp, _i64, _i32, _i32, ctypes.POINTER(_i64)]),
    "bbkio_format_double": (ctypes.c_int, [ctypes.c_double, ctypes.c_char_p]),
    "bbkio_unpack_scores": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i64, _vp, _vp, _i32]),
    "bbkio_unpack_scores_keep": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _i32]),
    "bbkio_copy_bytes": (ctypes.c_int, [_vp, _vp, ctypes.c_size_t, _i32]),
    "bbkio_pack_records_bound": (ctypes.c_uint64, [_i64]),
    "bbkio_pack_records": (ctypes.c_int, [ctypes.POINTER(_vp), ctypes.POINTER(_vp), ctypes.POINTER(_vp), ctypes.POINTER(_i64), _i32, _vp,
                                          ctypes.c_uint64, ctypes.POINTER(ctypes.c_uint64), _i32]),
    "bbkio_check_records": (ctypes.c_int, [_vp, ctypes.c_uint64, _i64]),
    "bbkio_read_interactions": (ctypes.c_int, [ctypes.c_char_p, _i32, ctypes.POINTER(_vp)]),
    "bbkio_table_rows": (_i64, [_vp]),
    "bbkio_table_n_chrom": (_i32, [_vp]),
    "bbkio_table_chrom_name": (ctypes.c_char_p, [_vp, _i32]),
    "bbkio_table_copy": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "bbkio_table_free": (None, [_vp]),
}
_lib = None


class BbkIoError(RuntimeError):
    pass


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BbkIoError("%s not found: build it with `python -m blueberry_b200.build`" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _ptr(a):
    return None if a is None else ctypes.c_void_p(a.ctypes.data)


def write_significances(path, chrom_names, chr1, mid1, chr2, mid2, count, p, q=None, threads=0, level=1):
    """fithic.py:410-435 on arrays; returns the number of rows written (those with p <= 1)."""
    lib = load()
    n = len(p)
    names = (ctypes.c_char_p * len(chrom_names))(*[str(s).encode() for s in chrom_names])
    c1 = None if chr1 is None else np.ascontiguousarray(chr1, dtype=np.int32)
    c2 = None if chr2 is None else np.ascontiguousarray(chr2, dtype=np.int32)
    m1, m2 = np.ascontiguousarray(mid1, dtype=np.int64), np.ascontiguousarray(mid2, dtype=np.int64)
    cnt = np.ascontiguousarray(count, dtype=np.int64)
    pp = np.ascontiguousarray(p, dtype=np.float64)
    qq = None if q is None else np.ascontiguousarray(q, dtype=np.float64)
    rows = _i64(0)
    rc = lib.bbkio_write_significances(os.fsencode(path), names, len(chrom_names), _ptr(c1), _ptr(m1), _ptr(c2), _ptr(m2),
                                       _ptr(cnt), _ptr(pp), _ptr(qq), n, int(threads), int(level), ctypes.byref(rows))
    if rc != 0:
        buf = ctypes.create_string_buffer(512)
        lib.bbkio_last_error(buf, 512)
        raise BbkIoError("bbkio_write_significances failed (code %d): %s" % (rc, buf.value.decode(errors="replace")))
    return int(rows.value)


def _raise(lib, what, rc):
    buf = ctypes.create_string_buffer(512)
    lib.bbkio_last_error(buf, 512)
    msg = buf.value.decode(errors="replace")
    if rc == -4:
        # the reference's own failure for a malformed row: ValueError from the tuple unpack / int() (fithic.py:245-247)
        raise ValueError(msg.split(": ", 1)[-1])
    raise BbkIoError("%s failed (code %d): %s" % (what, rc, msg))


def read_interactions(path, threads=0):
    """fithic.py:243-247 on a whole file: returns (names, chr1, mid1, chr2, mid2, count) with chr1/chr2 int32 ids into
    `names` (order of first appearance), the rest int64.  One thread inflates, the others parse."""
    lib = load()
    handle = _vp()
    rc = lib.bbkio_read_interactions(os.fsencode(path), int(threads), ctypes.byref(handle))
    if rc != 0:
        _raise(lib, "bbkio_read_interactions", rc)
    try:
        n = int(lib.bbkio_table_rows(handle))
        names = [lib.bbkio_table_chrom_name(handle, i).decode() for i in range(int(lib.bbkio_table_n_chrom(handle)))]
        c1, c2 = np.empty(n, dtype=np.int32), np.empty(n, dtype=np.int32)
        m1, m2, cnt = np.empty(n, dtype=np.int64), np.empty(n, dtype=np.int64), np.empty(n, dtype=np.int64)
        rc = lib.bbkio_table_copy(handle, _ptr(c1), _ptr(m1), _ptr(c2), _ptr(m2), _ptr(cnt))
        if rc != 0:
            _raise(lib, "bbkio_table_copy", rc)
    finally:
        lib.bbkio_table_free(handle)
    return names, c1, m1, c2, m2, cnt


def format_double(x):
    buf = ctypes.create_string_buffer(64)
    n = load().bbkio_format_double(float(x), buf)
    return buf.raw[:n].decode()


def copy_bytes(dst_ptr, src_ptr, nbytes, threads=0):
    """memcpy by all cores (raw addresses)."""
    rc = load().bbkio_copy_bytes(ctypes.c_void_p(dst_ptr), ctypes.c_void_p(src_ptr), int(nbytes), int(threads))
    if rc != 0:
        _raise(load(), "bbkio_copy_bytes", rc)


def unpack_scores(codes, chunks, values_p, values_q, m, p_out=None, q_out=None, threads=0, want_q=True, keep_out=None):
    """The packed form of a pass' p / q columns (bbk_pack_scores) back into dense float64 columns, bit for bit.
    codes: uint32 words (16 rows each); chunks: the 24-byte chunk records as a uint8 / structured buffer; values_p / values_q:
    float64 lists.  All numpy arrays (or anything exposing ctypes.data through numpy).  Returns (p, q) (q None if not wanted)."""
    lib = load()
    m = int(m)
    p = p_out if p_out is not None else np.empty(m, dtype=np.float64)
    q = (q_out if q_out is not None else np.empty(m, dtype=np.float64)) if want_q else None
    if keep_out is not None:
        rc = lib.bbkio_unpack_scores_keep(_ptr(codes), _ptr(chunks), _ptr(values_p), _ptr(values_q), m, _ptr(p), _ptr(q), _ptr(keep_out),
                                          int(threads))
    else:
        rc = lib.bbkio_unpack_scores(_ptr(codes), _ptr(chunks), _ptr(values_p), _ptr(values_q), m, _ptr(p), _ptr(q), int(threads))
    if rc != 0:
        _raise(lib, "bbkio_unpack_scores", rc)
    return p, q



def pack_records_bound(rows):
    """The most bytes the packed records of `rows` layout rows can take (bbk.h, BbkRecHeader)."""
    return int(load().bbkio_pack_records_bound(int(rows)))


def pack_records(shards, out_ptr, capacity, threads=0):
    """The packed records of shards [(mid1, mid2, count), ...] (int32 columns, numpy or anything numpy views without a copy)
    laid out by layout_rows, written to the raw host address out_ptr (capacity bytes).  Returns the bytes written; raises
    ValueError when they do not fit."""
    lib = load()
    cols = [[np.ascontiguousarray(c, dtype=np.int32) for c in sh] for sh in shards]
    for c in cols:
        if not (len(c) == 3 and len(c[0]) == len(c[1]) == len(c[2])):
            raise ValueError("a shard is three int32 columns (mid1, mid2, count) of one length")
    n = len(cols)
    ptrs = [(_vp * max(n, 1))(*[c[j].ctypes.data for c in cols]) for j in range(3)]
    sizes = (_i64 * max(n, 1))(*[len(c[0]) for c in cols])
    used = ctypes.c_uint64(0)
    rc = lib.bbkio_pack_records(ptrs[0], ptrs[1], ptrs[2], sizes, n, ctypes.c_void_p(out_ptr), int(capacity), ctypes.byref(used), int(threads))
    if rc != 0:
        buf = ctypes.create_string_buffer(512)
        lib.bbkio_last_error(buf, 512)
        raise ValueError(buf.value.decode(errors="replace"))
    return int(used.value)


def check_records(buf_ptr, nbytes, rows):
    """Raise ValueError unless the nbytes at buf_ptr are packed records of `rows` rows that bbk_unpack_records may read."""
    lib = load()
    if lib.bbkio_check_records(ctypes.c_void_p(buf_ptr), int(nbytes), int(rows)) != 0:
        buf = ctypes.create_string_buffer(512)
        lib.bbkio_last_error(buf, 512)
        raise ValueError(buf.value.decode(errors="replace"))
