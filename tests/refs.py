"""Test-side access to the three checkers and the checkasm-style input generators.

  ref()     oracle/_ref/libdav1d_ref.so — the UNMODIFIED dav1d C path (+ oracle/refdriver);
            built by build() (oracle/Makefile) where the reference sources exist, shipped prebuilt elsewhere
  oracle()  oracle/liboracle.so — this repo's plain-C restatement (always buildable: gcc only)
  emu_lib() tests/emu: the CUDA sources compiled for the host fiber emulator (debug harness)
"""
import ctypes as C
import os
import subprocess
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
REF_SO = os.path.join(ORACLE_DIR, "_ref", "libdav1d_ref.so")
ORACLE_SO = os.path.join(ORACLE_DIR, "liboracle.so")

from dav1d_b200 import levels as L  # noqa: E402
from dav1d_b200.batch import ITX_BLOCK_DTYPE  # noqa: E402

_cache = {}


def _make(target):
    subprocess.run(["make", "-C", ORACLE_DIR, target], check=True, capture_output=True)


def have_ref():
    return os.path.exists(REF_SO)


def ref():
    if "ref" not in _cache:
        assert have_ref(), "oracle/_ref/libdav1d_ref.so missing (build() makes it where the reference sources exist)"
        lib = C.CDLL(REF_SO)
        lib.refdrv_scan.restype = C.POINTER(C.c_uint16)
        lib.refdrv_itx_add_batch.restype = C.c_double
        lib.refdrv_itx_add_batch.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                             C.POINTER(C.c_int32), C.c_int, C.c_int]
        _cache["ref"] = lib
    return _cache["ref"]


def oracle():
    if "oracle" not in _cache:
        _make("liboracle.so")
        lib = C.CDLL(ORACLE_SO)
        lib.oracle_inv_txfm_add.argtypes = [C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]
        lib.oracle_itx_add_batch.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                             C.POINTER(C.c_int32), C.c_int]
        _cache["oracle"] = lib
    return _cache["oracle"]


def emu_lib():
    """TEST-ONLY binding of the host-emulated build of the CUDA sources (see tests/emu/cuda_emu.h)."""
    if "emu" not in _cache:
        import importlib.util
        spec = importlib.util.spec_from_file_location("build_emu", os.path.join(ROOT, "tests", "emu", "build_emu.py"))
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        from dav1d_b200._lib import B200Lib
        _cache["emu"] = B200Lib(m.build())
    return _cache["emu"]


# ---------------------------------------------------------------- reference DSP tables
FT8 = C.CFUNCTYPE(None, C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_int)
FT16 = C.CFUNCTYPE(None, C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_int, C.c_int)


def ref_itx_table(bpc):
    """c.itxfm_add[tx][txtp] of the reference, as python callables (dst, stride, coeff, eob)."""
    key = ("itx", bpc)
    if key not in _cache:
        tbl = (C.c_void_p * (19 * 17))()
        if bpc == 8:
            ref().dav1d_itx_dsp_init_8bpc(tbl, 8)
        else:
            ref().dav1d_itx_dsp_init_16bpc(tbl, bpc)
        bdmax = (1 << bpc) - 1

        def wrap(p):
            if not p:
                return None
            if bpc == 8:
                f = FT8(p)
                return lambda d, s, c, e: f(d.ctypes.data, s, c.ctypes.data, e)
            f = FT16(p)
            return lambda d, s, c, e: f(d.ctypes.data, s, c.ctypes.data, e, bdmax)
        _cache[key] = [[wrap(tbl[tx * 17 + tp]) for tp in range(17)] for tx in range(19)]
    return _cache[key]


def oracle_itxfm_add(bpc):
    bdmax = (1 << bpc) - 1
    o = oracle()

    def mk(tx, tp):
        if not L.itx_defined(tx, tp):
            return None
        return lambda d, s, c, e: o.oracle_inv_txfm_add(d.ctypes.data, s, c.ctypes.data, e, tx, tp, bdmax)
    return [[mk(tx, tp) for tp in range(17)] for tx in range(19)]


# ---------------------------------------------------------------- checkasm-style generators
# 1-D type pairs as the checkasm generator sees them (reference tests/checkasm/itx.c:46-64)
_DCT, _ADST, _FLIPADST, _IDENTITY, _WHT = range(5)
_GEN_1D = [(_DCT, _DCT), (_DCT, _ADST), (_ADST, _DCT), (_ADST, _ADST), (_DCT, _FLIPADST), (_FLIPADST, _DCT),
           (_FLIPADST, _FLIPADST), (_FLIPADST, _ADST), (_ADST, _FLIPADST), (_IDENTITY, _IDENTITY),
           (_IDENTITY, _DCT), (_DCT, _IDENTITY), (_IDENTITY, _ADST), (_ADST, _IDENTITY),
           (_IDENTITY, _FLIPADST), (_FLIPADST, _IDENTITY), (_WHT, _WHT)]
_SCALE = [4.0, 4.0 * np.sqrt(0.5), 2.0, 2.0 * np.sqrt(0.5), 1.0, 0.5 * np.sqrt(0.5), 0.25, 0.125 * np.sqrt(0.5), 0.0625]
# TxClass per TxfmType (reference src/tables.c dav1d_tx_type_class): 2D / H / V
_TX_CLASS_2D, _TX_CLASS_H, _TX_CLASS_V = 0, 1, 2
SUBSH_ITERS = [2, 2, 3, 5, 5]   # reference tests/checkasm/itx.c:252


def _fwd_matrix(kind, sz):
    i = np.arange(sz)[:, None].astype(np.float64)
    j = np.arange(sz)[None, :].astype(np.float64)
    if kind == _DCT:
        m = np.cos(np.pi * (2 * j + 1) * i / (sz * 2.0))
        m[0] *= np.sqrt(0.5)
        return m
    if kind in (_ADST, _FLIPADST):
        if sz == 4:
            return np.sin(np.pi * (j + 1) * (2 * i + 1) / 9.0)
        return np.sin(np.pi * (2 * j + 1) * (2 * i + 1) / (sz * 4.0))
    if kind == _WHT:
        return None
    return np.eye(sz)


def _fwht4(v):
    t0 = v[0] + v[1]; t3 = v[3] - v[2]; t4 = (t0 - t3) * 0.5; t1 = t4 - v[1]; t2 = t4 - v[2]
    return np.array([t0 - t2, t2, t3 + t1, t1])


def scan_table(tx):
    """dav1d_scans[tx] (from the reference build when present, else the committed copy)."""
    key = ("scan", tx)
    if key not in _cache:
        sw, sh = L.tx_coef_dims(tx)
        gold = os.path.join(ROOT, "tests", "golden", "scans.npz")
        if have_ref():
            p = ref().refdrv_scan(tx)
            _cache[key] = np.array([p[i] for i in range(sw * sh)], np.int32)
        else:
            _cache[key] = np.load(gold)["tx%d" % tx].astype(np.int32)
    return _cache[key]


def tx_class(txtp):
    # reference src/tables.c: V_* are TX_CLASS_V, H_* are TX_CLASS_H, IDTX + 2-D types are 2D
    if txtp in (L.V_DCT, L.V_ADST, L.V_FLIPADST):
        return _TX_CLASS_V
    if txtp in (L.H_DCT, L.H_ADST, L.H_FLIPADST):
        return _TX_CLASS_H
    return _TX_CLASS_2D


def gen_itx_coefs(rng, tx, txtp, subsh, bitdepth_max):
    """Port of ftx() + copy_subcoefs() (reference tests/checkasm/itx.c:131-242): returns
    (coef[sw*sh] in the layout itxfm_add reads, eob). Coefficients come from a float forward
    transform of a random residual, then everything past a random eob inside the `subsh`
    sub-block is zeroed."""
    w, h = L.TX_W[tx], L.TX_H[tx]
    sw, sh = min(w, 32), min(h, 32)
    scale = _SCALE[int(np.log2(w * h)) - 4]
    k0 = _GEN_1D[txtp][0]
    resid = (rng.integers(0, 2 * bitdepth_max + 2, (h, w)) - bitdepth_max).astype(np.float64)
    if k0 == _WHT:
        temp = np.stack([_fwht4(r) for r in resid], 1) * scale          # temp[j*h+i]
        out = np.stack([_fwht4(t) for t in temp])                         # out[i*h + k]
    else:
        m = _fwd_matrix(k0, w)
        temp = (m @ resid.T) * scale                                       # [w][h]
        m2 = _fwd_matrix(k0, h)
        out = temp @ m2.T                                                  # out[i][k], i<w, k<h
    flat = out.reshape(-1)                                                 # out[i*h + k]
    buf = np.zeros(sw * sh, np.float64)
    for y in range(sh):
        buf[y * sw:(y + 1) * sw] = flat[y * w:y * w + sw]
    coef = np.floor(buf + 0.5)
    # C float->int conversion truncates toward zero
    coef = np.trunc(buf + 0.5).astype(np.int64)

    cls = tx_class(txtp) if txtp != L.WHT_WHT else _TX_CLASS_2D
    scan = scan_table(tx)
    sub_high = subsh * 8 - 1 if subsh > 0 else 0
    sub_low = sub_high - 8 if subsh > 1 else 0
    eob = 0
    n = 0
    while n < sw * sh:
        if cls == _TX_CLASS_2D:
            rc = int(scan[n]); rcx, rcy = rc % sh, rc // sh
        elif cls == _TX_CLASS_H:
            rcx, rcy = n % sh, n // sh
        else:
            rcx, rcy = n // sw, n % sw
        if rcx > sub_high or rcy > sub_high:
            break
        if not eob and (rcx > sub_low or rcy > sub_low):
            eob = n
        n += 1
    if eob:
        eob += int(rng.integers(0, 1 << 30)) % (n - eob - 1) if (n - eob - 1) > 0 else 0
    if cls == _TX_CLASS_2D:
        coef[scan[eob + 1:]] = 0
    elif cls == _TX_CLASS_H:
        coef[eob + 1:] = 0
    else:
        rcx, rcy = eob // sw, eob % sw
        while rcx < sh:
            rcy += 1
            while rcy < sw:
                coef[rcy * sh + rcx] = 0
                rcy += 1
            rcx += 1; rcy = -1
    return coef, eob


def coef_dtype(bpc):
    return np.int16 if bpc == 8 else np.int32


def pixel_dtype(bpc):
    return np.uint8 if bpc == 8 else np.uint16


# ---------------------------------------------------------------- mc
def ref_mc_ctx(bpc):
    """The reference's Dav1dMCDSPContext (C path) wrapped like dav1d_b200.dsp.MCDSPContext."""
    key = ("mc", bpc)
    if key not in _cache:
        from dav1d_b200 import dsp
        tbl = (C.c_void_p * 53)()
        (ref().dav1d_mc_dsp_init_8bpc if bpc == 8 else ref().dav1d_mc_dsp_init_16bpc)(tbl)

        class Ctx:
            pass
        c = Ctx()
        c._tbl = tbl
        for k, v in dsp.wrap_dsp_table(tbl, dsp.MC_LAYOUT, dsp.MC_PROTOS, bpc > 8, (1 << bpc) - 1).items():
            setattr(c, k, v)
        _cache[key] = c
    return _cache[key]


def oracle_mc_ctx(bpc):
    """oracle/mc.c behind the same member names / call signatures."""
    o = oracle()
    bd = (1 << bpc) - 1
    P, S, I = C.c_void_p, C.c_ssize_t, C.c_int

    def a(x):
        return x.ctypes.data if isinstance(x, np.ndarray) else x

    class Ctx:
        pass
    c = Ctx()
    c.mc = [(lambda d, ds, s, ss, w, h, mx, my, f=f: o.oracle_mc_put(P(a(d)), S(ds), P(a(s)), S(ss), w, h, mx, my, f, bd)) for f in range(10)]
    c.mct = [(lambda t, s, ss, w, h, mx, my, f=f: o.oracle_mc_prep(P(a(t)), P(a(s)), S(ss), w, h, mx, my, f, bd)) for f in range(10)]
    c.mc_scaled = [(lambda d, ds, s, ss, w, h, mx, my, dx, dy, f=f: o.oracle_mc_put_scaled(P(a(d)), S(ds), P(a(s)), S(ss), w, h, mx, my, dx, dy, f, bd)) for f in range(10)]
    c.mct_scaled = [(lambda t, s, ss, w, h, mx, my, dx, dy, f=f: o.oracle_mc_prep_scaled(P(a(t)), P(a(s)), S(ss), w, h, mx, my, dx, dy, f, bd)) for f in range(10)]
    c.avg = lambda d, ds, t1, t2, w, h: o.oracle_avg(P(a(d)), S(ds), P(a(t1)), P(a(t2)), w, h, bd)
    c.w_avg = lambda d, ds, t1, t2, w, h, wt: o.oracle_w_avg(P(a(d)), S(ds), P(a(t1)), P(a(t2)), w, h, wt, bd)
    c.mask = lambda d, ds, t1, t2, w, h, m: o.oracle_mask(P(a(d)), S(ds), P(a(t1)), P(a(t2)), w, h, P(a(m)), bd)
    c.w_mask = [(lambda d, ds, t1, t2, w, h, m, sign, l=l: o.oracle_w_mask(P(a(d)), S(ds), P(a(t1)), P(a(t2)), w, h, P(a(m)), sign, l, bd)) for l in range(3)]
    c.blend = lambda d, ds, t, w, h, m: o.oracle_blend(P(a(d)), S(ds), P(a(t)), w, h, P(a(m)), bd)
    c.blend_v = lambda d, ds, t, w, h: o.oracle_blend_v(P(a(d)), S(ds), P(a(t)), w, h, bd)
    c.blend_h = lambda d, ds, t, w, h: o.oracle_blend_h(P(a(d)), S(ds), P(a(t)), w, h, bd)
    c.warp8x8 = lambda d, ds, s, ss, abcd, mx, my: o.oracle_warp8x8(0, P(a(d)), S(ds), P(a(s)), S(ss), P(a(abcd)), mx, my, bd)
    c.warp8x8t = lambda t, ts, s, ss, abcd, mx, my: o.oracle_warp8x8(1, P(a(t)), S(ts), P(a(s)), S(ss), P(a(abcd)), mx, my, bd)
    c.emu_edge = lambda bw, bh, iw, ih, x, y, d, ds, r, rs: o.oracle_emu_edge(S(bw), S(bh), S(iw), S(ih), S(x), S(y), P(a(d)), S(ds), P(a(r)), S(rs), bd)
    c.resize = lambda d, ds, s, ss, dw, h, sw, dx, mx: o.oracle_resize(P(a(d)), S(ds), P(a(s)), S(ss), dw, h, sw, dx, mx, bd)
    return c
