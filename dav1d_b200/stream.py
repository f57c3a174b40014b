"""Host glue for decoding AV1 elementary streams with the B200 back end behind a real dav1d front end.

`oracle/_ref/libdav1d_b200.so` is the unmodified dav1d library whose `f->bd_fn` hooks are the record emitters of
integration/dav1d/ (built by integration/dav1d/Makefile where the reference sources exist; like the rest of oracle/_ref/
it is shipped prebuilt to machines without them). This module binds its stream driver (dav1d's public API: dav1d_open / dav1d_send_data / dav1d_get_picture)
and points the hooks at dav1d_b200/libb200av1.so. No CPU fallback: without the CUDA library the decode fails."""
import ctypes as C
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOOKED_SO = os.path.join(ROOT, "oracle", "_ref", "libdav1d_b200.so")
LEVEL1_SO = os.path.join(ROOT, "oracle", "_ref", "libdav1d_b200_l1.so")
FAMILIES = {"itx": 1, "mc": 2, "ipred": 4, "loopfilter": 8, "cdef": 16, "looprestoration": 32, "filmgrain": 64}


class HookStats(C.Structure):
    _fields_ = [("frames", C.c_uint64), ("records", C.c_uint64), ("coefs", C.c_uint64), ("h2d_bytes", C.c_uint64),
                ("d2h_bytes", C.c_uint64), ("device_ms", C.c_double), ("intra_tx", C.c_uint64), ("pred", C.c_uint64),
                ("comp", C.c_uint64), ("warp", C.c_uint64), ("blend", C.c_uint64), ("itx", C.c_uint64),
                ("inter_frames", C.c_uint64), ("host_prep_ms", C.c_double), ("interintra", C.c_uint64), ("palette_bytes", C.c_uint64), ("ibc", C.c_uint64), ("scaled", C.c_uint64)]


def build_hooked(verbose=False):
    """(Re)build oracle/_ref/libdav1d_b200.so (+ the Level-1 variant) where the reference sources exist; a no-op elsewhere."""
    import subprocess
    r = subprocess.run(["make", "-j8", "-C", os.path.join(ROOT, "integration", "dav1d"), "all"], capture_output=True, text=True)
    if r.returncode:
        raise RuntimeError("integration/dav1d build failed:\n" + r.stderr[-3000:])
    if verbose:
        print(r.stdout[-500:])
    return HOOKED_SO


def plane_dims(w, h, layout):
    """(width, height) of the planes of a picture; layout = enum Dav1dPixelLayout (0 4:0:0, 1 4:2:0, 2 4:2:2, 3 4:4:4)"""
    if layout == 0:
        return [(w, h)]
    cw = w if layout == 3 else (w + 1) // 2
    ch = (h + 1) // 2 if layout == 1 else h
    return [(w, h), (cw, ch), (cw, ch)]


def decode_stream(dll, tus, n_threads=4, max_frame_delay=2, max_pics=64, apply_grain=0):
    """Decode a list of temporal units with `dll` (a CDLL exporting refdrv_decode_stream: the hooked library or the
    stock checker). Returns (n_pictures or negative dav1d error, info[n][4] = w, h, bpc, layout, packed pictures)."""
    data = b"".join(tus)
    sz = (C.c_uint64 * len(tus))(*[len(t) for t in tus])
    info = np.zeros(4 * max_pics, np.int32)
    # output size is not known before the sequence header is parsed by the decoder: bound it from the stream's own
    # sequence header (max_frame_width / height live in the first OBU_SEQ_HDR) -> the caller passes generous capacity
    cap = int(decode_stream.capacity)
    out = np.empty(cap, np.uint8)
    dll.refdrv_decode_stream.restype = C.c_int
    dll.refdrv_decode_stream.argtypes = [C.c_char_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_uint64,
                                         C.c_void_p, C.c_int]
    r = dll.refdrv_decode_stream(data, sz, len(tus), n_threads, max_frame_delay, apply_grain, out.ctypes.data, cap,
                                 info.ctypes.data, max_pics)
    n = 0
    for i in range(max(r, 0)):
        w, h, bpc, layout = (int(v) for v in info[4 * i:4 * i + 4])
        n += sum(pw * ph for pw, ph in plane_dims(w, h, layout)) * (2 if bpc > 8 else 1)
    return r, info[:4 * max(r, 0)].reshape(-1, 4).copy(), out[:n]


decode_stream.capacity = 256 << 20


class HookedDecoder:
    """dav1d front end + B200 back end. `backend` = path of the C-ABI library the hooks bind (default: the CUDA
    library); `serialize` = one device job at a time (for back ends that are not re-entrant)."""

    def __init__(self, backend=None, serialize=False):
        if not os.path.exists(HOOKED_SO):
            raise RuntimeError("oracle/_ref/libdav1d_b200.so missing (build() makes it where the reference sources exist)")
        if backend is None:
            from . import _lib
            _lib.get_lib()                       # builds / loads the CUDA library or raises
            backend = _lib.get_lib().path
        self.dll = C.CDLL(HOOKED_SO)
        if self.dll.b200hook_set_backend(backend.encode()) != 0:
            raise RuntimeError("b200hook_set_backend(%s) failed" % backend)
        self.dll.b200hook_set_serialize(1 if serialize else 0)

    def decode(self, tus, **kw):
        return decode_stream(self.dll, tus, **kw)

    def output_times_ns(self):
        """when each picture of the last decode() came out of dav1d_get_picture: nanoseconds since the call began"""
        buf = (C.c_uint64 * 4096)()
        self.dll.refdrv_output_times_ns.restype = C.c_int
        n = self.dll.refdrv_output_times_ns(buf, 4096)
        return [int(buf[i]) for i in range(n)]

    def stats(self, reset=False):
        s = HookStats()
        self.dll.b200hook_get_stats(C.byref(s), 1 if reset else 0)
        return {k: getattr(s, k) for k, _ in HookStats._fields_}

    def release(self):
        self.dll.b200hook_release()


class Level1Decoder:
    """dav1d with its own reconstruction code, but every DSP table slot (`Dav1dDSPContext`: itx, mc, ipred, loopfilter,
    cdef, looprestoration, filmgrain) overridden by libb200av1's Level-1 functions — the architecture-hook form of the
    drop-in (integration/dav1d/b200_level1.c). One kernel launch per DSP call: a parity harness, not a throughput path.
    `families` = iterable of FAMILIES keys (default: all seven)."""

    def __init__(self, backend=None, families=None):
        if not os.path.exists(LEVEL1_SO):
            raise RuntimeError("oracle/_ref/libdav1d_b200_l1.so missing (build() makes it where the reference sources exist)")
        if backend is None:
            from . import _lib
            backend = _lib.get_lib().path
        self.dll = C.CDLL(LEVEL1_SO)
        mask = sum(FAMILIES[f] for f in (families or FAMILIES))
        if self.dll.b200l1_set_backend(backend.encode(), mask) != 0:
            raise RuntimeError("b200l1_set_backend(%s) failed" % backend)

    def c_slots_left(self):
        """(slots still on dav1d's C functions after the back end's init, slots replaced): the first must be 0"""
        return int(self.dll.b200l1_c_slots_left()), int(self.dll.b200l1_slots_replaced())

    def decode(self, tus, **kw):
        kw.setdefault("n_threads", 1)            # the Level-1 thunks serialise on one lock anyway
        kw.setdefault("max_frame_delay", 1)
        return decode_stream(self.dll, tus, **kw)
