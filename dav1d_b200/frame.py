"""Host side of the whole-frame job (include/b200av1.h, B200FrameJob).

FrameBuffers turns one frame's records (numpy arrays in dav1d's layouts, e.g. from synth.py — the
role dav1d's pass-1 entropy decode plays in a real integration) into device buffers + a B200FrameJob,
and runs it. `alloc` abstracts where the buffers live: torch CUDA tensors on the GPU, or plain numpy
when the same C ABI is bound to the test-only host emulator.
"""
import ctypes as C
import numpy as np

from . import _lib


class TorchAlloc:
    """device buffers as torch CUDA tensors (torch is plumbing: memory + streams only)"""

    def __init__(self, device=None):
        import torch
        self.torch = torch
        self.device = device if device is not None else torch.device("cuda", torch.cuda.current_device())

    def upload(self, a):
        t = self.torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).to(self.device)
        return t, t.data_ptr()

    def zeros(self, nbytes):
        t = self.torch.zeros(max(nbytes, 16), dtype=self.torch.uint8, device=self.device)
        return t, t.data_ptr()

    def download(self, t, like):
        return t.cpu().numpy()[:like.nbytes].view(like.dtype)

    def pinned(self, a):
        t = self.torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).pin_memory()
        return t, t.data_ptr()

    def sync(self):
        self.torch.cuda.synchronize()

    def stream(self):
        return self.torch.cuda.current_stream().cuda_stream

    def new_stream(self):
        s = self.torch.cuda.Stream(device=self.device)
        return s, s.cuda_stream


class NumpyAlloc:
    """'device' == host: only valid with the emulated library (tests/emu)"""

    def upload(self, a):
        c = np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()
        return c, c.ctypes.data

    def zeros(self, nbytes):
        c = np.zeros(max(nbytes, 16), np.uint8)
        return c, c.ctypes.data

    def download(self, t, like):
        return t[:like.nbytes].view(like.dtype)

    def pinned(self, a):
        return self.upload(a)

    def sync(self):
        pass

    def stream(self):
        return None

    def new_stream(self):
        return None, None


def band_plan(S, band_rows, compact=False, fused=False):
    """Cut a frame's records into horizontal bands of `band_rows` luma rows (a multiple of 64: blocks never straddle a
    band). Returns (S2, bands, need): S2 = shallow copy of S whose record arrays are stably sorted by band (the by-area
    order is kept inside a band), bands = list of dicts {y0, y1, last, <record list>: (first, count)} and need[k][ref] =
    (luma rows, chroma rows) of reference `ref` that band k's predictions read — the `lowest_pixel` of dav1d's
    check_tile (reference src/thread_task.c:415, src/decode.c lowest_pixel bookkeeping); expand = the compact coefficient
    stream and its band-sorted B200CoefBlock records when `compact`.
    Intra-machine records (S["intra_tx"]) are sorted by band too, keeping their wavefront order inside a band. A band may
    only depend on itself and the bands above it: ValueError when a record's bottom-left edge or an intra block copy's
    source reaches below its band (band edges must fall on superblock rows), and when the frame has predictions from
    scaled references (not band-sliced)."""
    assert band_rows % 64 == 0 and band_rows > 0
    H, off, stride = S["H"], S["off"], S["stride"]
    ssv = [0, S["ss_ver"], S["ss_ver"]]
    nb = -(-H // band_rows)
    S2 = dict(S)
    if nb > 1 and S.get("scaled") is not None and len(S["scaled"]):
        raise ValueError("band_plan: predictions from scaled references are not band-sliced (one band)")

    def luma_y(dst_off, plane):
        pl = np.asarray(plane).astype(np.int64)
        o = np.asarray(off, np.int64)[pl]; st = np.asarray(stride, np.int64)[pl]
        return ((np.asarray(dst_off).astype(np.int64) - o) // st) << np.asarray(ssv, np.int64)[pl]

    def sort_by_band(arr, y):
        band = (y // band_rows).astype(np.int64)
        assert not len(band) or (band.min() >= 0 and band.max() < nb)
        order = np.argsort(band, kind="stable")
        cnt = np.bincount(band, minlength=nb)
        first = np.concatenate([[0], np.cumsum(cnt)[:-1]])
        return arr[order], first, cnt, band[order]

    ranges, band_of = {}, {}
    # compound records first: they tell where the int16 predictions (op 1, addressed in `tmp`) belong
    tmp_y = {}
    for name in ("comp", "comp2"):
        a = S[name]
        y = luma_y(a["dst_off"], a["plane"]) if len(a) else np.zeros(0, np.int64)
        for t1, t2, yy in zip(a["tmp1_off"].tolist(), a["tmp2_off"].tolist(), y.tolist()):
            tmp_y[t1] = yy; tmp_y[t2] = yy
        S2[name], f, c, _ = sort_by_band(a, y)
        ranges[name] = (f, c)
    # blends (OBMC): they tell where the overlapped predictions (op 2, addressed in `px_tmp`) belong; 8x8 warps
    lap_y = {}
    for name in ("blend", "blend2", "warp"):
        if name in S:
            a = S[name]
            y = luma_y(a["dst_off"], a["plane"]) if len(a) else np.zeros(0, np.int64)
            if name != "warp":
                for t, yy in zip(a["tmp_off"].tolist(), y.tolist()):
                    lap_y[t] = yy
            S2[name], f, c, band_of[name] = sort_by_band(a, y)
            ranges[name] = (f, c)
    pname = "pred_single" if (fused and "cfused" in S) else "pred"
    a = S[pname]
    y = np.zeros(len(a), np.int64)
    put, prep, lap = a["op"] == 0, a["op"] == 1, a["op"] == 2
    if put.any():
        y[put] = luma_y(a["dst_off"][put], a["plane"][put])
    if prep.any():
        y[prep] = [tmp_y[t] for t in a["dst_off"][prep].tolist()]
    if lap.any():
        y[lap] = [lap_y[t] for t in a["dst_off"][lap].tolist()]
    S2[pname], f, c, pband = sort_by_band(a, y)
    ranges["pred"] = (f, c)
    for name in ("cfused", "cfused2"):
        if fused and name in S:
            a = S[name]
            S2[name], f, c, band_of[name] = sort_by_band(a, luma_y(a["dst_off"], a["plane"]) if len(a) else np.zeros(0, np.int64))
            ranges[name] = (f, c)
    iband = None
    it = S.get("intra_tx")
    if it is not None and len(it):
        S2["intra_tx"], f, c, iband = sort_by_band(it, it["y4"].astype(np.int64) * 4 << np.asarray(ssv, np.int64)[it["plane"]])
        ranges["intra"] = (f, c)
        _check_intra_bands(S2["intra_tx"], iband, band_rows, nb, S)
    S2["itx"] = {}
    itx_ranges = {}
    for tx in range(19):
        a = S["itx"][tx]
        S2["itx"][tx], f, c, _ = sort_by_band(a, luma_y(a["dst_off"], a["plane"]) if len(a) else np.zeros(0, np.int64))
        itx_ranges[tx] = (f, c)
    expand = None
    if compact:
        from . import synth
        cc, ex = synth.compact_coefs(S2)
        # compact_coefs emits its records size class after size class, each in the (band-sorted) order of S2["itx"][tx]
        per_tx = [np.repeat(np.arange(nb), itx_ranges[tx][1]) for tx in range(19) if len(S2["itx"][tx])]       # empty: every inter block skipped
        eb = np.concatenate(per_tx) if per_tx else np.zeros(0, np.int64)
        # ... followed by the intra records' blocks, size class after size class in the (band-sorted) order of S2["intra_tx"]
        if iband is not None:
            t = S2["intra_tx"]
            eb = np.concatenate([eb] + [iband[(t["tx"] == tx) & (t["eob"] >= 0)] for tx in range(19)]).astype(np.int64)
        assert len(eb) == len(ex)
        order = np.argsort(eb, kind="stable")
        cnt = np.bincount(eb, minlength=nb)
        expand = (cc, ex[order])
        ranges["expand"] = (np.concatenate([[0], np.cumsum(cnt)[:-1]]), cnt)
    bands = []
    for k in range(nb):
        b = {"y0": k * band_rows, "y1": min(H, (k + 1) * band_rows), "last": int(k == nb - 1)}
        for name, (f, c) in ranges.items():
            b[name] = (int(f[k]), int(c[k]))
        b["itx"] = [(int(itx_ranges[tx][0][k]), int(itx_ranges[tx][1][k])) for tx in range(19)]
        bands.append(b)
    # rows of each reference that a band reads: block bottom + 4 rows of filter support (8-tap: 3 above, 4 below)
    P = S2[pname]
    n_refs = len(S["refs"])
    need = np.zeros((nb, max(n_refs, 1), 2), np.int64)
    if len(P):
        low = P["src_y"].astype(np.int64) + P["h"] + 4
        cls = (P["plane"] > 0).astype(np.int64)
        np.maximum.at(need, (pband, P["ref"].astype(np.int64), cls), low)
    # warps read their reference directly (15 x 15 window: rows src_y - 3 .. src_y + 11); fused compound records carry
    # both references
    if "warp" in band_of and len(S2["warp"]):
        a = S2["warp"]
        np.maximum.at(need, (band_of["warp"], a["ref"].astype(np.int64), (a["plane"] > 0).astype(np.int64)),
                      a["src_y"].astype(np.int64) + 12)
    for name in ("cfused", "cfused2"):
        if name in band_of and len(S2[name]):
            a = S2[name]
            for i in range(2):
                np.maximum.at(need, (band_of[name], a["ref"][:, i].astype(np.int64), (a["plane"] > 0).astype(np.int64)),
                              a["src_y"][:, i].astype(np.int64) + a["h"] + 4)
    ph = [H, (H + ssv[1]) >> ssv[1]]
    need[:, :, 0] = np.minimum(need[:, :, 0], ph[0]); need[:, :, 1] = np.minimum(need[:, :, 1], ph[1])
    return S2, bands, need, expand


def _check_intra_bands(t, band, band_rows, nb, S):
    """ValueError when an intra record of a band-sliced frame depends on rows below its band (band = band index per record):
    the band's launch could never see them (the kernel would trap, or read pixels not yet reconstructed)."""
    if nb == 1:
        return
    from . import levels as L
    ssv = np.array([0, S["ss_ver"], S["ss_ver"]], np.int64)
    pl = t["plane"].astype(np.int64)
    y, th = t["y4"].astype(np.int64), np.asarray(L.TX_H, np.int64)[t["tx"]] // 4
    ye = t["yend4"].astype(np.int64)
    # first plane row (in 4-sample units for the edges, samples for the copies) below each record's band; none for the last band
    end_px = np.where(band < nb - 1, ((band + 1) * band_rows) >> ssv[pl], 1 << 30)
    flags = t["flags"].astype(np.int64)
    bl = (flags & 1 != 0) & (flags & 8 != 0) & (y + th < ye)
    reach = np.minimum(y + 2 * th, ye) * 4
    bad = bl & (reach > end_px)
    if bad.any():
        i = int(np.nonzero(bad)[0][0])
        raise ValueError("band_plan: intra record %d (plane %d, row %d) reads bottom-left rows down to %d, below its band "
                         "(band edges must fall on superblock rows)" % (i, pl[i], y[i] * 4, reach[i]))
    ibc = t["mode"] == 18
    if ibc.any():
        ph = np.array([S["h4"], S["h4"] >> S["ss_ver"], S["h4"] >> S["ss_ver"]], np.int64)[pl] * 4
        sy = t["luma_off"].astype(np.int64) >> 16
        last = np.minimum(sy + th * 4 - 1 + (t["cfl_h_pad"] != 0), ph - 1)
        bad = ibc & (last >= end_px)
        if bad.any():
            i = int(np.nonzero(bad)[0][0])
            raise ValueError("band_plan: intra block copy %d (plane %d) copies from row %d, below its band" % (i, pl[i], last[i]))


def run_batch(fbs, stream=None):
    """b200_frame_run_batch over several FrameBuffers (same library, same bit depth) on one stream: their intra
    stages share launches (frames are the parallel axis of intra decoding)."""
    lib = fbs[0].lib
    arr = (C.POINTER(_lib.FrameJob) * len(fbs))(*[C.pointer(fb.job) for fb in fbs])
    st = fbs[0].alloc.stream() if stream is None else stream
    lib.check(lib.b200_frame_run_batch(arr, len(fbs), st), "b200_frame_run_batch")


class FrameGroup:
    """Several FrameBuffers driven as one unit on one stream (b200_frame_run_batch / b200_frame_submit_host_batch)."""

    def __init__(self, fbs):
        self.fbs, self.lib = fbs, fbs[0].lib
        self.jobs = (C.POINTER(_lib.FrameJob) * len(fbs))(*[C.pointer(fb.job) for fb in fbs])
        self._stream = None
        self._host = False

    def stream(self):
        if self._stream is None:
            self._stream = self.fbs[0].alloc.new_stream()
        return self._stream[1]

    def run(self, stream=None):
        self.lib.check(self.lib.b200_frame_run_batch(self.jobs, len(self.fbs), self.stream() if stream is None else stream),
                       "b200_frame_run_batch")

    def submit_host(self):
        if not self._host:
            ups, downs = [], []
            for fb in self.fbs:
                fb.prepare_host(); fb._host = True
                ups += list(fb._ups); downs += list(fb._downs)
            self._ups = (_lib.Xfer * len(ups))(*ups); self._downs = (_lib.Xfer * len(downs))(*downs)
            self._host = True
        self.lib.check(self.lib.b200_frame_submit_host_batch(self.jobs, len(self.fbs), self._ups, len(self._ups), self._downs,
                                                             len(self._downs), self.stream()), "b200_frame_submit_host_batch")

    def wait(self):
        self.lib.check(self.lib.b200_frame_wait(self.stream()), "b200_frame_wait")


class FrameBuffers:
    def __init__(self, S, lib=None, alloc=None, run_lf=True, run_cdef=True, run_lr=True, intra_grid=0, compact=False, intra_sb=False, fused=False,
                 band_rows=0):
        self.bands = None
        expand = None
        if band_rows:            # records sorted by band + the B200FrameBand list (b200_frame_run_band)
            S, plan, self.band_need, expand = band_plan(S, band_rows, compact=compact, fused=fused)
            self.bands = (_lib.FrameBand * len(plan))()
            for k, b in enumerate(plan):
                fbn = self.bands[k]
                fbn.y0, fbn.y1, fbn.last = b["y0"], b["y1"], b["last"]
                for name in ("pred", "warp", "comp", "comp2", "blend", "blend2", "cfused", "cfused2", "expand", "intra"):
                    if name in b:
                        getattr(fbn, name)[0], getattr(fbn, name)[1] = b[name]
                for tx in range(19):
                    fbn.itx[tx][0], fbn.itx[tx][1] = b["itx"][tx]
        self.S, self.lib = S, lib or _lib.get_lib()
        self.alloc = alloc or TorchAlloc()
        A = self.alloc
        self.keep = {}
        px = S["pic"].itemsize

        def up(name, arr):
            self.keep[name] = A.upload(arr)
            return self.keep[name][1]

        def zeros(name, nbytes):
            self.keep[name] = A.zeros(nbytes)
            return self.keep[name][1]
        nbytes = S["pic"].nbytes
        refs = [up("ref%d" % i, r) for i, r in enumerate(S["refs"])]
        p0, p1, p2 = zeros("p0", nbytes), zeros("p1", nbytes), zeros("p2", nbytes)
        tmp = zeros("tmp", S["tmp_len"] * 2)
        mask = up("mask", S["mask"])
        j = _lib.FrameJob()
        j.bitdepth_max, j.zero_coefs = S["bd"], 0
        for i, r in enumerate(refs):
            j.mc.ref[i] = r
        ssh, ssv = [0, S["ss_hor"], S["ss_hor"]], [0, S["ss_ver"], S["ss_ver"]]
        for p in range(3):
            j.mc.ref_plane_off[p] = S["off"][p]; j.mc.ref_stride[p] = S["stride"][p]
            j.mc.ref_w[p] = (S["W"] + ssh[p]) >> ssh[p]; j.mc.ref_h[p] = (S["H"] + ssv[p]) >> ssv[p]
            j.mc.dst_stride[p] = S["stride"][p]; j.itx_stride[p] = S["stride"][p]
        j.mc.dst, j.mc.tmp, j.mc.mask, j.mc.px_tmp = p0, tmp, mask, (zeros("px_tmp", S["px_tmp_len"] * px) if S.get("px_tmp_len") else None)
        self.uploads = []          # (name, host array) re-sent per frame on the end-to-end path

        def rec(field_ptr, field_n, name, arr):
            if len(arr):
                setattr(j, field_ptr, up(name, arr)); setattr(j, field_n, len(arr))
                self.uploads.append((name, arr))
        if fused and "cfused" in S:      # compound blocks: both predictions + the combination in one kernel
            rec("d_pred", "n_pred", "pred", S["pred_single"])
            rec("d_cfused", "n_cfused", "cfused", S["cfused"])
            rec("d_cfused2", "n_cfused2", "cfused2", S["cfused2"])
        else:
            rec("d_pred", "n_pred", "pred", S["pred"])
            rec("d_comp", "n_comp", "comp", S["comp"])
            rec("d_comp2", "n_comp2", "comp2", S["comp2"])
        for name in ("warp", "blend", "blend2"):      # warped blocks; OBMC blends (stage 1: rows from above, stage 2: columns from the left)
            if name in S:
                rec("d_" + name, "n_" + name, name, S[name])
        for tx in range(19):
            a = S["itx"][tx]
            if len(a):
                j.d_itx[tx] = up("itx%d" % tx, a); j.n_itx[tx] = len(a)
                self.uploads.append(("itx%d" % tx, a))
        if compact:
            # the emitter ships coefficients 0 .. eob in scan order; the job zeroes + rebuilds the dense buffer
            from . import synth
            cc, ex = expand if expand is not None else synth.compact_coefs(S)
            j.d_coef = zeros("coef", S["coefs"].nbytes)
            j.coef_bytes = S["coefs"].nbytes
            j.d_ccoef = up("ccoef", cc); self.uploads.append(("ccoef", cc))
            if len(ex):
                j.d_expand = up("expand", ex); j.n_expand = len(ex); self.uploads.append(("expand", ex))
        else:
            j.d_coef = up("coef", S["coefs"]); self.uploads.append(("coef", S["coefs"]))
        if len(S["mask"]) > 1:
            self.uploads.append(("mask", S["mask"]))
        n_intra = 0
        if S.get("intra_tx") is not None and len(S["intra_tx"]):
            it = j.intra
            it.pic, it.d_coef, it.zero_coefs, it.grid = p0, j.d_coef, 0, intra_grid
            it.ss_hor, it.ss_ver = S["ss_hor"], S["ss_ver"]
            it.mask = mask                            # blend masks of inter-intra (II) records
            if S.get("intra_pal") is not None:       # colours + index maps of palette (PAL) records
                it.pal = up("intra_pal", S["intra_pal"]); self.uploads.append(("intra_pal", S["intra_pal"]))
            for p in range(3):
                it.stride[p] = S["stride"][p]; it.plane_off[p] = S["off"][p]
                it.w4[p] = S["w4"] >> ssh[p]; it.h4[p] = S["h4"] >> ssv[p]
            nb = self.lib.b200_intra_scratch_bytes(C.byref(it)) if hasattr(self.lib, "b200_intra_scratch_bytes") else 1 << 22
            it.scratch = zeros("intra_scratch", nb)
            if intra_sb:     # superblock-granular schedule (records grouped by 64x64 superblock)
                j.d_intra = up("intra_tx", S["intra_tx_sb"]); j.n_intra = len(S["intra_tx_sb"])
                self.uploads.append(("intra_tx", S["intra_tx_sb"]))
                it.sb = up("intra_sb", S["intra_sb"]); it.n_sb = len(S["intra_sb"])
                it.sb_w, it.sb_h = S["intra_sb_grid"]
                self.uploads.append(("intra_sb", S["intra_sb"]))
            else:
                j.d_intra = up("intra_tx", S["intra_tx"]); j.n_intra = len(S["intra_tx"])
                self.uploads.append(("intra_tx", S["intra_tx"]))
                if S.get("done_init") is not None:       # a frame that mixes inter and intra blocks: inter cells are final already
                    it.done_init = up("done_init", S["done_init"])
                    self.uploads.append(("done_init", S["done_init"]))
            n_intra = 1
            if self.bands is not None and len(self.bands) > 1:
                if (S["intra_tx"]["mode"] == 18).any() and (run_lf or run_cdef or run_lr):
                    raise ValueError("intra block copy reads the unfiltered picture above its band: its frames run with "
                                     "deblocking, CDEF and loop restoration off")
                # the rows each band saves for the band below (B200FrameBand.edge_top / edge_bottom): Y, U, V rows back to back
                eb = sum(S["stride"]) * px
                base = zeros("band_edges", eb * (len(self.bands) - 1))
                for k in range(len(self.bands) - 1):
                    self.bands[k].edge_bottom = self.bands[k + 1].edge_top = base + k * eb
        # post filters
        j.run_lf, j.run_cdef, j.run_lr = int(run_lf), int(run_cdef), int(run_lr)
        d_masks = up("masks", S["masks"]); self.uploads.append(("masks", S["masks"]))
        d_level = up("level", S["level"]); self.uploads.append(("level", S["level"]))
        d_lrm = up("lr_mask", S["lr_mask"]); self.uploads.append(("lr_mask", S["lr_mask"]))
        lf = j.lf
        lf.pic = p0
        for p in range(3):
            lf.plane_off[p] = S["off"][p]; lf.stride[p] = S["stride"][p]
        lf.w4, lf.h4, lf.sb128w, lf.b4_stride = S["w4"], S["h4"], S["sb128w"], S["b4_stride"]
        lf.ss_hor, lf.ss_ver, lf.sb128, lf.filter_y, lf.filter_uv = S["ss_hor"], S["ss_ver"], S["sb128"], 1, 1
        lf.mask, lf.level = d_masks, d_level
        for k in range(64):
            lf.lut.e[k], lf.lut.i[k] = int(S["lut_e"][k]), int(S["lut_i"][k])
        lf.lut.sharp[0], lf.lut.sharp[1] = S["lut_sharp"]
        cd = j.cdef
        cd.src, cd.dst = p0, p1
        for p in range(3):
            cd.plane_off[p] = S["off"][p]; cd.stride[p] = S["stride"][p]
        cd.bw, cd.bh, cd.sb128w, cd.ss_hor, cd.ss_ver, cd.damping = S["bw"], S["bh"], S["sb128w"], S["ss_hor"], S["ss_ver"], S["damping"]
        for i in range(8):
            cd.y_strength[i], cd.uv_strength[i] = S["y_strength"][i], S["uv_strength"][i]
        cd.mask = d_masks
        lr = j.lr
        lr.cdef, lr.dbl, lr.dst = (p1 if run_cdef else p0), p0, p2
        for p in range(3):
            lr.plane_off[p] = S["off"][p]; lr.stride[p] = S["stride"][p]
        lr.w, lr.h, lr.ss_hor, lr.ss_ver, lr.sb128 = S["W"], S["H"], S["ss_hor"], S["ss_ver"], S["sb128"]
        lr.sr_sb128w = (S["W"] + 127) >> 7
        lr.unit_size_log2[0], lr.unit_size_log2[1] = S["us"]
        lr.restore_planes, lr.lr_mask = S["rp"], d_lrm
        self.out_name = "p2" if run_lr else ("p1" if run_cdef else "p0")
        n_fg = 0
        self.ref_name = self.out_name          # the picture later frames predict from (never the grained copy)
        if S.get("fg") is not None:
            # film grain goes into a separate display copy; the un-grained picture stays the reference picture
            fg = j.fg
            j.run_fg = 1
            fg.in_, fg.out = self.keep[self.out_name][1], zeros("p3", nbytes)
            for p in range(3):
                fg.plane_off[p] = S["off"][p]; fg.stride[p] = S["stride"][p]
            fg.w, fg.h, fg.ss_hor, fg.ss_ver, fg.is_id = S["W"], S["H"], S["ss_hor"], S["ss_ver"], 0
            fg.data = S["fg"]
            fg.scratch = zeros("fg_scratch", 256 * 1024)
            self.ref_name, self.out_name = self.out_name, "p3"
            n_fg = 2
        self.job = j
        self.n_launches = (1 if j.n_pred else 0) + (1 if j.n_comp else 0) + (1 if j.n_comp2 else 0) + \
            (1 if j.n_warp else 0) + (1 if j.n_blend else 0) + (1 if j.n_blend2 else 0) + \
            (1 if j.n_cfused else 0) + (1 if j.n_cfused2 else 0) + \
            (1 if any(j.n_itx[tx] for tx in (4, 11, 12, 17, 18)) else 0) + \
            (1 if any(j.n_itx[tx] for tx in range(19) if tx not in (4, 11, 12, 17, 18)) else 0) + 2 * int(run_lf) + int(run_cdef) + int(run_lr) + n_fg + n_intra
        self._host = None

    # ---- device-resident run (records already in HBM) ----
    def run(self, stream=None):
        st = self.alloc.stream() if stream is None else stream
        self.lib.check(self.lib.b200_frame_run(C.byref(self.job), st), "b200_frame_run")

    # ---- band by band (b200_frame_run_band): same result as run(); what the frame pipeline over GPUs schedules ----
    def n_bands(self):
        return len(self.bands) if self.bands is not None else 0

    def run_band(self, k, stream=None):
        st = self.alloc.stream() if stream is None else stream
        self.lib.check(self.lib.b200_frame_run_band(C.byref(self.job), C.byref(self.bands[k]), st), "b200_frame_run_band")

    def run_band_phase(self, k, phases, stream=None):
        """1 = reconstruction of band k, 2 = its post filters (b200_frame_run_band_phase)"""
        st = self.alloc.stream() if stream is None else stream
        self.lib.check(self.lib.b200_frame_run_band_phase(C.byref(self.job), C.byref(self.bands[k]), phases, st), "b200_frame_run_band_phase")

    def run_bands(self, stream=None):
        for k in range(len(self.bands)):
            self.run_band(k, stream)

    def band_progress(self, k, plane):
        """rows of `plane` of the restored picture that are final after band k"""
        b = self.bands[k]
        return self.lib.b200_band_progress(C.byref(self.job), b.y1, b.last, plane)

    def set_refs(self, ptrs):
        for i, p in enumerate(ptrs):
            self.job.mc.ref[i] = p

    def output(self, name=None):
        return self.alloc.download(self.keep[name or self.out_name][0], self.S["pic"])

    def picture_ptr(self, name=None):
        return self.keep[name or self.out_name][1]

    # ---- end-to-end run: records from pinned host memory, picture back to the host ----
    def prepare_host(self):
        A = self.alloc
        ups = []
        self._host_keep = []
        for name, arr in self.uploads:
            t, p = A.pinned(arr)
            self._host_keep.append(t)
            ups.append((p, self.keep[name][1], arr.nbytes))
        out_t, out_p = A.pinned(np.zeros(self.S["pic"].nbytes, np.uint8))
        self._host_out = out_t
        self._ups = (_lib.Xfer * len(ups))(*[_lib.Xfer(h, d, n) for h, d, n in ups])
        self._downs = (_lib.Xfer * 1)(_lib.Xfer(out_p, self.keep[self.out_name][1], self.S["pic"].nbytes))
        self.h2d_bytes = sum(n for _, _, n in ups)
        self.d2h_bytes = self.S["pic"].nbytes

    def h2d_bytes_estimate(self):
        return sum(a.nbytes for _, a in self.uploads)

    def run_host(self, stream=None):
        if self._host is None:
            self.prepare_host(); self._host = True
        st = self.alloc.stream() if stream is None else stream
        self.lib.check(self.lib.b200_frame_run_host(C.byref(self.job), self._ups, len(self._ups), self._downs, 1, st),
                       "b200_frame_run_host")

    # frame-threaded variant: each FrameBuffers owns a stream; submit() returns at once, wait() joins
    def submit_host(self):
        if self._host is None:
            self.prepare_host(); self._host = True
        if getattr(self, "_own_stream", None) is None:
            self._own_stream = self.alloc.new_stream()
        self.lib.check(self.lib.b200_frame_submit_host(C.byref(self.job), self._ups, len(self._ups), self._downs, 1,
                                                       self._own_stream[1]), "b200_frame_submit_host")

    def wait(self):
        self.lib.check(self.lib.b200_frame_wait(self._own_stream[1]), "b200_frame_wait")

    def host_output(self):
        t = self._host_out
        a = t.numpy() if hasattr(t, "numpy") else t
        return a[:self.S["pic"].nbytes].view(self.S["pic"].dtype)
