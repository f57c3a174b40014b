"""Real-stream drop-in test: the same AV1 elementary stream decoded (a) by the stock reference (oracle/_ref, dav1d's own
CPU back end) and (b) by oracle/_ref/libdav1d_b200.so = the same dav1d front end with the f->bd_fn hooks emitting
B200 records and libb200av1 reconstructing + filtering every frame. Output pictures must be byte-identical.
Streams: dav1d_b200/obu.py (valid headers, random tile payloads: every intra tool, per-block delta q / lf, CDEF, LR).
CPU tests bind the hooks to the host emulator build of the CUDA sources; GPU tests bind the real library."""
import ctypes as C
import os

import numpy as np
import pytest

import refs
from dav1d_b200 import obu, stream

pytestmark = pytest.mark.skipif(not (os.path.exists(stream.HOOKED_SO) and refs.have_ref()),
                                reason="oracle/_ref/libdav1d_b200.so not built")


def _ref_decode(tus, **kw):
    assert refs.have_ref()
    return stream.decode_stream(C.CDLL(refs.REF_SO), tus, **kw)


def _check(dec, tus, expect_frames, **kw):
    r0, info0, out0 = _ref_decode(tus, **kw)
    assert r0 == expect_frames, "the stock reference could not decode the synthetic stream (%d)" % r0
    r1, info1, out1 = dec.decode(tus, **kw)
    assert r1 == r0, "hooked decoder returned %d" % r1
    assert np.array_equal(info0, info1)
    if not np.array_equal(out0, out1):
        d = np.nonzero(out0 != out1)[0]
        raise AssertionError("%d of %d output bytes differ, first at %d" % (len(d), len(out0), d[0]))
    st = dec.stats(reset=True)
    dec.last_stats = st
    assert st["frames"] >= min(expect_frames, 1) and st["records"] > 0


CASES_CPU = [
    # w, h, bpc, sb128, log2 tile cols, rows, frames
    (256, 192, 8, 0, 0, 0, 2),
    (256, 192, 10, 0, 1, 1, 2),
    (328, 250, 8, 1, 1, 0, 1),          # sizes that are not multiples of 8, 128x128 superblocks
    (640, 360, 8, 0, 2, 1, 2),
    (330, 250, 10, 1, 0, 1, 1),
]


@pytest.fixture(scope="module")
def emu_decoder():
    refs.emu_lib()
    import importlib.util
    spec = importlib.util.spec_from_file_location("build_emu", os.path.join(refs.ROOT, "tests", "emu", "build_emu.py"))
    m = importlib.util.module_from_spec(spec); spec.loader.exec_module(m)
    d = stream.HookedDecoder(backend=m.build(), serialize=True)
    yield d
    d.release()


@pytest.mark.emu
@pytest.mark.parametrize("case", CASES_CPU)
def test_stream_emu_matches_stock_dav1d(emu_decoder, case):
    w, h, bpc, sb128, lc, lr, nf = case
    tus = obu.intra_stream(hash(case) & 0xffff, w, h, n_frames=nf, bpc=bpc, sb128=sb128, log2_cols=lc, log2_rows=lr)
    _check(emu_decoder, tus, nf)


CASES_INTER_CPU = [
    # w, h, bpc, sb128, log2 tile cols, rows, frames (1 key frame + inter frames), per-block motion modes (OBMC, local warp)
    (320, 192, 8, 0, 0, 0, 3, 0),
    (320, 192, 10, 0, 1, 1, 4, 0),
    (640, 360, 8, 1, 1, 0, 3, 0),
    (330, 250, 8, 0, 0, 0, 5, 1),
    (320, 192, 10, 0, 1, 1, 4, 2),      # 2: inter-intra prediction as well
    (640, 360, 8, 1, 1, 0, 4, 2),
]


@pytest.mark.emu
@pytest.mark.parametrize("case", CASES_INTER_CPU)
def test_inter_stream_emu_matches_stock_dav1d(emu_decoder, case):
    """key frame + inter frames: single and compound references (average, distance weights, wedge and
    difference-weighted masks), sub-8x8 chroma, variable transform trees, intra blocks inside inter frames,
    references kept in device memory across frames and frame contexts"""
    w, h, bpc, sb128, lc, lr, nf, mm = case
    tus = obu.inter_stream(hash(case) & 0xffff, w, h, n_frames=nf, bpc=bpc, sb128=sb128, log2_cols=lc, log2_rows=lr, motion_modes=mm)
    _check(emu_decoder, tus, nf)
    if mm:
        assert emu_decoder.last_stats["blend"] > 0, "no OBMC block in the stream"
    if mm >= 2:
        assert emu_decoder.last_stats["interintra"] > 0, "no inter-intra block in the stream"


@pytest.mark.emu
@pytest.mark.parametrize("case", [(256, 192, 8, 2, 0), (320, 192, 10, 3, 1), (330, 250, 8, 4, 1)])
def test_film_grain_stream_emu_matches_stock_dav1d(emu_decoder, case):
    """film grain on the output copy (dav1d's apply_grain / delayed_fg tasks) runs as a device job on the HBM-resident
    picture: random scaling points, AR lags 0..3, overlap, chroma scaling from luma, 8 / 10 bit"""
    w, h, bpc, nf, inter = case
    gen = obu.inter_stream if inter else obu.intra_stream
    tus = gen(40 + (hash(case) & 0xff), w, h, n_frames=nf, bpc=bpc, film_grain=1)
    r0, _, with_grain = _ref_decode(tus, apply_grain=1)
    _, _, without = _ref_decode(tus, apply_grain=0)
    assert r0 == nf and not np.array_equal(with_grain, without), "the stream carries no visible grain"
    _check(emu_decoder, tus, nf, apply_grain=1)


@pytest.mark.emu
@pytest.mark.parametrize("case", [(256, 192, 8, 2, 0, 0), (320, 192, 10, 3, 1, 0), (640, 360, 8, 2, 0, 1)])
def test_screen_content_stream_emu_matches_stock_dav1d(emu_decoder, case):
    """allow_screen_content_tools: palette blocks (luma and chroma palettes, packed index maps) in key and inter frames"""
    w, h, bpc, nf, inter, sb128 = case
    gen = (lambda *a, **k: obu.inter_stream(*a, motion_modes=2, **k)) if inter else obu.intra_stream
    tus = gen(7, w, h, n_frames=nf, bpc=bpc, sb128=sb128, screen_content=1)
    _check(emu_decoder, tus, nf)
    assert emu_decoder.last_stats["palette_bytes"] > 0, "no palette block in the stream"


@pytest.mark.emu
@pytest.mark.parametrize("case", [("444", 8, 0, 0, 0), ("444", 10, 1, 1, 1), ("444", 12, 1, 0, 0), ("420", 12, 1, 1, 1),
                                  ("400", 8, 0, 0, 0), ("400", 10, 1, 1, 0), ("400", 12, 1, 0, 1)])
def test_other_layouts_and_12bit_stream_emu_matches_stock_dav1d(emu_decoder, case):
    """profile 1 (4:4:4) and profile 2 (12 bit) streams: same hooks, chroma at full resolution / 12-bit clipping ranges;
    monochrome (4:0:0): luma only, the device picture carries two dummy chroma planes for the frame-wide sweeps.
    (4:2:2 cannot be driven with random payloads: its illegal partitions make the decoder reject the tile.)"""
    layout, bpc, inter, fg, sc = case
    gen = (lambda *a, **k: obu.inter_stream(*a, motion_modes=2, **k)) if inter else obu.intra_stream
    tus = gen(5, 200, 136, n_frames=3, bpc=bpc, layout=layout, film_grain=fg, screen_content=sc)
    _check(emu_decoder, tus, 3, apply_grain=1)


@pytest.mark.emu
@pytest.mark.parametrize("case", [(8, 0, 0), (10, 1, 2)])
def test_hidden_frames_and_show_existing_emu_matches_stock_dav1d(emu_decoder, case):
    """frames decoded out of display order: hidden "future" frames referenced with backward prediction (which also makes
    skip mode available) and output later by show_existing_frame headers, film grain applied when they are shown"""
    bpc, fg, mm = case
    tus = obu.inter_stream(20 + bpc, 256, 192, n_frames=7, bpc=bpc, film_grain=fg, motion_modes=mm, hidden_every=2)
    assert len(tus) == 10
    _check(emu_decoder, tus, 10, apply_grain=1)


@pytest.mark.emu
def test_intra_only_frames_emu_matches_stock_dav1d(emu_decoder):
    """INTRA_ONLY frames between inter frames: intra coded, replace only the reference slots they name"""
    tus = obu.inter_stream(31, 256, 192, n_frames=8, bpc=10, film_grain=1, motion_modes=2, screen_content=1, intra_only_every=3)
    _check(emu_decoder, tus, 8, apply_grain=1)


@pytest.mark.emu
@pytest.mark.parametrize("case", [(8, 0), (10, 2)])
def test_global_motion_stream_emu_matches_stock_dav1d(emu_decoder, case):
    """non-identity global motion (translation, rotation-zoom, affine models written with the sub-exponential code):
    GLOBALMV blocks become warped predictions (warp8x8 into the picture, warp8x8t into the compound scratch)"""
    bpc, mm = case
    tus = obu.inter_stream(50 + bpc, 320, 192, n_frames=5, bpc=bpc, motion_modes=mm, global_motion=1)
    _check(emu_decoder, tus, 5)
    assert emu_decoder.last_stats["warp"] > 0, "no warped block in the stream"


@pytest.mark.emu
@pytest.mark.parametrize("seed", [70, 71, 75])
def test_segmentation_stream_emu_matches_stock_dav1d(emu_decoder, seed):
    """segmentation: per-segment quantiser deltas (down to qidx 0 = lossless segments: 4x4 Walsh-Hadamard blocks, loop
    filter off for them), loop-filter deltas, forced reference / skip / global motion"""
    if seed & 1:
        tus = obu.inter_stream(seed, 256, 192, n_frames=4, bpc=10, motion_modes=2, segmentation=1, global_motion=1)
    else:
        tus = obu.intra_stream(seed, 256, 192, n_frames=2, bpc=8, segmentation=1)
    _check(emu_decoder, tus, len(tus))


@pytest.mark.emu
def test_sequence_changes_within_one_decode(emu_decoder):
    """new sequence headers mid-stream (other picture size, other bit depth): per-frame geometry, buffers that grow, the
    8-bit and the 16-bit hook sets alternating on the same frame contexts"""
    tus = obu.inter_stream(1, 320, 192, n_frames=3, motion_modes=2) + obu.inter_stream(2, 200, 136, n_frames=3, motion_modes=1) + \
          obu.inter_stream(3, 456, 264, n_frames=3, bpc=10, motion_modes=2, film_grain=1)
    _check(emu_decoder, tus, 9, apply_grain=1)


@pytest.mark.emu
def test_abandoned_frames_do_not_poison_later_decodes(emu_decoder):
    """decoders closed while frames are still in flight (dav1d_close flushes them half way through pass 2): the frame
    contexts' slots keep half-emitted frames; later decodes must neither pick up their records nor run out of slots"""
    good = obu.inter_stream(1, 256, 192, n_frames=4, motion_modes=2)
    r0, _, out0 = _ref_decode(good)
    long_ = obu.inter_stream(2, 320, 256, n_frames=10, motion_modes=1, log2_cols=1, log2_rows=1)
    data = b"".join(long_)
    sz = (C.c_uint64 * len(long_))(*[len(t) for t in long_])
    dll = emu_decoder.dll
    dll.refdrv_decode_and_abandon.restype = C.c_int
    for k in range(14):                       # 14 x 8 frame contexts > the 64 slots of the hook's table
        assert dll.refdrv_decode_and_abandon(data, sz, 3 + k % 6, 8, 8) >= 0
        r1, _, out1 = emu_decoder.decode(good)
        assert r1 == r0 and np.array_equal(out0, out1), k
    emu_decoder.stats(reset=True)


@pytest.mark.emu
@pytest.mark.parametrize("seed", [6002, 6070, 6363])
def test_unused_references_are_not_waited_for(emu_decoder, seed):
    """a frame lists 7 references but its blocks may read only some of them; dav1d makes it wait only for those, so an
    unused reference may not even have started its second pass when the frame completes (found by fuzzing: the frame
    used to fail with "reference was not decoded"). Several repeats: the outcome depended on thread timing."""
    rng = np.random.default_rng(seed)
    w, h = int(rng.integers(4, 30)) * 8 + int(rng.choice([0, 0, 2, 6])), int(rng.integers(4, 22)) * 8 + int(rng.choice([0, 0, 4]))
    kw = dict(bpc=int(rng.choice([8, 10, 12])), sb128=int(rng.integers(0, 2)), log2_cols=int(rng.integers(0, 2)), log2_rows=int(rng.integers(0, 2)),
              film_grain=int(rng.integers(0, 2)), screen_content=int(rng.integers(0, 2)), layout=str(rng.choice(["420", "420", "444", "400"])),
              segmentation=int(rng.integers(0, 2)))
    tus = obu.inter_stream(seed, w, h, n_frames=int(rng.integers(2, 7)), motion_modes=int(rng.integers(0, 3)), global_motion=int(rng.integers(0, 2)),
                           hidden_every=int(rng.choice([0, 0, 2, 3])), intra_only_every=int(rng.choice([0, 0, 0, 4])), **kw)
    r0, _, out0 = _ref_decode(tus, apply_grain=1)
    assert r0 > 0
    for _ in range(6):
        r1, _, out1 = emu_decoder.decode(tus, apply_grain=1, n_threads=4, max_frame_delay=3)
        assert r1 == r0 and np.array_equal(out0, out1)
    emu_decoder.stats(reset=True)


@pytest.mark.parametrize("w,h,kw", [(256, 192, dict(bpc=8)), (328, 200, dict(bpc=10, log2_cols=1)), (192, 136, dict(bpc=12, layout="444")),
                                    (256, 192, dict(bpc=8, layout="400")), (320, 192, dict(bpc=8, film_grain=1))])
def test_super_resolution_key_frames_decode(emu_decoder, w, h, kw):
    """super-resolution (was refused until round 2): the frame is coded narrower, upscaled after CDEF by the job's resize stage
    (both the CDEF picture and the deblocked picture loop restoration reads), restored and output at full width"""
    for seed in range(3):
        tus = obu.intra_stream(900 + seed, w, h, n_frames=2, super_res=1, **kw)
        _check(emu_decoder, tus, 2, apply_grain=1)


@pytest.mark.parametrize("w,h,kw", [(256, 192, dict(bpc=8)), (328, 200, dict(bpc=10, log2_cols=1, motion_modes=1)),
                                    (192, 136, dict(bpc=12, layout="444", motion_modes=2)), (320, 192, dict(bpc=8, film_grain=1, intra_only_every=3))])
def test_super_resolution_inter_streams_decode(emu_decoder, w, h, kw):
    """inter frames with super-resolution: every reference is the upscaled picture of an earlier frame while the frame itself
    is coded narrower, so all of its predictions are scaled predictions"""
    n_scaled = 0
    for seed in range(2):
        tus = obu.inter_stream(950 + seed, w, h, n_frames=6, super_res=1, **kw)
        _check(emu_decoder, tus, 6, apply_grain=1)
        n_scaled += emu_decoder.last_stats["scaled"]
    assert n_scaled > 100


def test_monochrome_stream_decodes(emu_decoder):
    """4:0:0 (was refused in round 1): key frames through the hooked decoder, byte-identical to stock dav1d"""
    tus = obu.intra_stream(5, 128, 128, n_frames=2, layout="400")
    _check(emu_decoder, tus, 2)


def _valid_422(kind, w, h, bpc, want, **kw):
    """random tile payloads are only sometimes legal 4:2:2 streams (partitions whose chroma blocks would be 2 samples wide are
    forbidden, reference src/decode.c decode_sb): draw seeds until stock dav1d accepts `want` of them"""
    out = []
    for seed in range(400):
        tus = obu.intra_stream(seed, w, h, n_frames=1, bpc=bpc, layout="422", **kw) if kind == "intra" else \
            obu.inter_stream(seed, w, h, n_frames=3, bpc=bpc, layout="422", **kw)
        if _ref_decode(tus)[0] == (1 if kind == "intra" else 3):
            out.append(tus)
            if len(out) == want:
                break
    return out


@pytest.mark.parametrize("kind,w,h,bpc,kw", [("intra", 64, 64, 8, {}), ("intra", 128, 128, 10, dict(film_grain=1)), ("intra", 192, 128, 12, {}),
                                             ("inter", 64, 64, 10, dict(motion_modes=1)), ("inter", 128, 64, 8, dict(motion_modes=1, film_grain=1)),
                                             ("inter", 128, 64, 12, dict(motion_modes=2))])
def test_422_streams_decode(emu_decoder, kind, w, h, bpc, kw):
    """4:2:2 (ss_hor = 1, ss_ver = 0) key and inter frames through the hooked decoder, byte-identical to stock dav1d"""
    streams = _valid_422(kind, w, h, bpc, 3, **kw)
    assert len(streams) == 3
    for tus in streams:
        _check(emu_decoder, tus, 1 if kind == "intra" else 3, apply_grain=1)


def _valid_intrabc(w, h, want, n_frames=2, **kw):
    """random payloads in frames that allow intra block copy are legal only when no vector ends up inside the current
    superblock (reference src/decode.c:1286-1345 returns an error otherwise): draw seeds until stock dav1d accepts `want`"""
    out = []
    for seed in range(400):
        tus = obu.intra_stream(seed, w, h, n_frames=n_frames, screen_content=1, intrabc=1, **kw)
        if _ref_decode(tus)[0] == n_frames:
            out.append(tus)
            if len(out) == want:
                break
    return out


@pytest.mark.parametrize("w,h,kw", [(128, 128, dict(bpc=8)), (192, 128, dict(bpc=10)), (256, 192, dict(bpc=8, layout="444", log2_cols=1)),
                                    (384, 256, dict(bpc=12, sb128=1)), (320, 192, dict(bpc=10)), (128, 128, dict(bpc=8, layout="422")),
                                    (256, 256, dict(bpc=8, layout="400"))])
def test_intra_block_copy_streams_decode(emu_decoder, w, h, kw):
    """key frames with allow_intrabc (was refused in round 1): blocks predicted from the reconstructed part of the same picture
    go through the intra machine as IBC records (bilinear put, half-sample chroma phases included) + RESID records"""
    streams = _valid_intrabc(w, h, 3, **kw)
    assert len(streams) == 3
    n_ibc = 0
    for tus in streams:
        _check(emu_decoder, tus, 2)
        n_ibc += emu_decoder.last_stats["ibc"]
    assert n_ibc > 0, "no intra block copy block in any of the streams"


@pytest.mark.parametrize("w,h,sizes,kw", [(256, 192, [(192, 144), (256, 192), (160, 96)], dict(bpc=8)),
                                          (320, 192, [(256, 160), (320, 192), (200, 120), (320, 176)], dict(bpc=10, motion_modes=1, film_grain=1)),
                                          (256, 256, [(128, 128), (256, 256)], dict(bpc=8, motion_modes=2, layout="444")),
                                          (192, 136, [(96, 72), (192, 136), (144, 100)], dict(bpc=12, log2_cols=1))])
def test_scaled_reference_streams_decode(emu_decoder, w, h, sizes, kw):
    """inter frames coded at changing sizes (was refused in round 1): their references have other sizes, so predictions are
    B200McScaledBlock records (put, prep for compound blocks, pixel scratch for OBMC) against per-reference plane geometry
    (B200McFrame.ref_geom) — byte-identical to stock dav1d, which runs mc_scaled / mct_scaled there (src/recon_tmpl.c:991-1046)"""
    n_scaled = 0
    for seed in range(3):
        tus = obu.inter_stream(700 + seed, w, h, n_frames=6, sizes=sizes, **kw)
        _check(emu_decoder, tus, 6, apply_grain=1)
        n_scaled += emu_decoder.last_stats["scaled"]
    assert n_scaled > 100, "hardly any scaled prediction in the streams"


def test_film_grain_on_a_picture_that_is_not_resident(emu_decoder):
    """film grain on a picture without a device copy (decoded elsewhere and handed to dav1d_apply_grain, or after
    b200hook_release): the host picture is uploaded first instead of aborting the process (B200HOOK_FG_UPLOAD forces that path)"""
    tus = obu.inter_stream(77, 200, 136, n_frames=4, bpc=10, film_grain=1)
    r0, _, out0 = _ref_decode(tus, apply_grain=1)
    os.environ["B200HOOK_FG_UPLOAD"] = "1"
    try:
        r1, _, out1 = emu_decoder.decode(tus, apply_grain=1)
    finally:
        del os.environ["B200HOOK_FG_UPLOAD"]
    assert r0 == 4 and r1 == r0 and np.array_equal(out0, out1)
    emu_decoder.stats(reset=True)


@pytest.mark.parametrize("n_threads,delay", [(1, 1), (1, 0), (4, 1), (2, 0)])
def test_single_threaded_settings_decode(emu_decoder, n_threads, delay):
    """one thread / no frame delay used to put dav1d in single-pass mode, which the emitters cannot serve (every frame
    failed as unsupported): the hooked library's dav1d_open now keeps two frame contexts, and the pictures match"""
    tus = obu.inter_stream(11, 192, 136, n_frames=5, motion_modes=1, film_grain=1)
    r0, _, out0 = _ref_decode(tus, n_threads=1, max_frame_delay=1, apply_grain=1)
    r1, _, out1 = emu_decoder.decode(tus, n_threads=n_threads, max_frame_delay=delay, apply_grain=1)
    assert r0 == 5 and r1 == r0 and np.array_equal(out0, out1)
    emu_decoder.stats(reset=True)


@pytest.mark.emu
def test_stream_many_decoders_recycle_slots(emu_decoder):
    """frame contexts and host pictures of closed decoders must not exhaust the hook's tables (each decode opens a new
    dav1d context; the tables are recycled least-recently-used)"""
    tus = obu.inter_stream(5, 192, 128, n_frames=5, motion_modes=1)
    r0, _, out0 = _ref_decode(tus)
    for _ in range(20):
        r1, _, out1 = emu_decoder.decode(tus, n_threads=8, max_frame_delay=4)
        assert r1 == r0 and np.array_equal(out0, out1)
    emu_decoder.stats(reset=True)


def test_stream_without_backend_fails_loudly():
    """no CPU fallback: with no back end bound the hooked decoder reports an error instead of decoding (own process:
    the binding is process-wide state of the library)"""
    import subprocess, sys
    code = ("import ctypes as C, os, sys; sys.path.insert(0, %r); os.environ.pop('B200AV1_LIB', None)\n"
            "from dav1d_b200 import obu, stream\n"
            "dll = C.CDLL(stream.HOOKED_SO)\n"
            "r, _, _ = stream.decode_stream(dll, obu.intra_stream(1, 128, 128, n_frames=1))\n"
            "print('RESULT', r)\n") % refs.ROOT
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert "RESULT -" in out.stdout, out.stdout + out.stderr
    assert "no back end loaded" in out.stderr


CASES_GPU = [
    (640, 360, 8, 0, 1, 1, 3),
    (1920, 1080, 8, 0, 2, 1, 3),
    (1920, 1080, 10, 1, 1, 1, 2),
    (3840, 2160, 8, 0, 2, 2, 2),
    (1000, 602, 10, 0, 0, 0, 2),
]


CASES_INTER_GPU = [
    (640, 360, 8, 0, 1, 1, 4, 0),
    (1920, 1080, 8, 0, 2, 1, 4, 0),
    (1920, 1080, 10, 1, 1, 1, 3, 0),
    (3840, 2160, 8, 0, 2, 2, 3, 0),
    (1920, 1080, 8, 0, 2, 1, 6, 2),
    (1280, 720, 10, 1, 1, 0, 6, 2),
]


@pytest.fixture(scope="module")
def gpu_decoder():
    d = stream.HookedDecoder()
    yield d
    d.release()


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES_GPU)
def test_stream_gpu_matches_stock_dav1d(gpu_decoder, case):
    w, h, bpc, sb128, lc, lr, nf = case
    tus = obu.intra_stream(1000 + (hash(case) & 0xfff), w, h, n_frames=nf, bpc=bpc, sb128=sb128, log2_cols=lc, log2_rows=lr)
    _check(gpu_decoder, tus, nf)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES_INTER_GPU)
def test_inter_stream_gpu_matches_stock_dav1d(gpu_decoder, case):
    w, h, bpc, sb128, lc, lr, nf, mm = case
    tus = obu.inter_stream(2000 + (hash(case) & 0xfff), w, h, n_frames=nf, bpc=bpc, sb128=sb128, log2_cols=lc, log2_rows=lr, motion_modes=mm)
    _check(gpu_decoder, tus, nf)


@pytest.mark.gpu
def test_new_layouts_and_intra_block_copy_gpu(gpu_decoder):
    """round 2 on the device: 4:0:0 and 4:2:2 streams, key frames with intra block copy, one thread / no frame delay"""
    _check(gpu_decoder, obu.intra_stream(5, 256, 192, n_frames=2, layout="400"), 2)
    _check(gpu_decoder, obu.inter_stream(7, 320, 192, n_frames=4, layout="400", motion_modes=1, film_grain=1), 4, apply_grain=1)
    for kind, w, h, bpc, kw in (("intra", 128, 128, 10, dict(film_grain=1)), ("inter", 128, 64, 8, dict(motion_modes=1))):
        for tus in _valid_422(kind, w, h, bpc, 2, **kw):
            _check(gpu_decoder, tus, 1 if kind == "intra" else 3, apply_grain=1)
    n_ibc = 0
    for w, h, kw in ((320, 192, dict(bpc=10)), (256, 192, dict(bpc=8, layout="444", log2_cols=1)), (128, 128, dict(bpc=8, layout="422"))):
        for tus in _valid_intrabc(w, h, 2, **kw):
            _check(gpu_decoder, tus, 2)
            n_ibc += gpu_decoder.last_stats["ibc"]
    assert n_ibc > 0
    tus = obu.inter_stream(11, 192, 136, n_frames=5, motion_modes=1)
    _check(gpu_decoder, tus, 5, n_threads=1, max_frame_delay=1)


@pytest.mark.gpu
def test_stream_gpu_many_frames_in_flight(gpu_decoder):
    """8 frame contexts, 32 threads, decoders opened again and again (slot recycling), device jobs of several frames
    overlapping on their own streams"""
    tus = obu.inter_stream(77, 1280, 720, n_frames=10, log2_cols=1, log2_rows=1, motion_modes=2)
    r0, _, out0 = _ref_decode(tus, n_threads=16, max_frame_delay=8)
    assert r0 == 10
    for _ in range(12):
        r1, _, out1 = gpu_decoder.decode(tus, n_threads=32, max_frame_delay=8)
        assert r1 == r0 and np.array_equal(out0, out1)
    gpu_decoder.stats(reset=True)


@pytest.mark.gpu
@pytest.mark.parametrize("case", [(1920, 1080, 8, 3, 1), (3840, 2160, 10, 3, 1), (1280, 720, 10, 2, 0)])
def test_film_grain_stream_gpu_matches_stock_dav1d(gpu_decoder, case):
    w, h, bpc, nf, inter = case
    gen = (lambda *a, **k: obu.inter_stream(*a, motion_modes=2, **k)) if inter else obu.intra_stream
    tus = gen(60 + (hash(case) & 0xff), w, h, n_frames=nf, bpc=bpc, log2_cols=1, log2_rows=1, film_grain=1)
    _check(gpu_decoder, tus, nf, apply_grain=1)


@pytest.mark.gpu
@pytest.mark.parametrize("case", [(1280, 720, 8, 2, 0, 0), (1920, 1080, 10, 3, 1, 1)])
def test_screen_content_stream_gpu_matches_stock_dav1d(gpu_decoder, case):
    w, h, bpc, nf, inter, sb128 = case
    gen = (lambda *a, **k: obu.inter_stream(*a, motion_modes=2, **k)) if inter else obu.intra_stream
    tus = gen(9, w, h, n_frames=nf, bpc=bpc, sb128=sb128, log2_cols=1, log2_rows=1, screen_content=1)
    _check(gpu_decoder, tus, nf)


# ---------------------------------------------------------------------------------------------------------------
def test_synthetic_headers_are_accepted_by_the_stock_decoder():
    """the bit-level header writer (dav1d_b200/obu.py) against dav1d's own parser over many random parameter draws:
    tile layouts, quantiser / delta-q / delta-lf, loop filter, CDEF, restoration unit sizes, interpolation filters,
    reference lists (skip-mode signalling depends on the order hints), film grain parameters, screen content"""
    n = 0
    for seed in range(24):
        rng = np.random.default_rng(seed)
        w, h = int(rng.integers(3, 12)) * 16, int(rng.integers(3, 10)) * 16
        kw = dict(bpc=int(rng.choice([8, 10])), sb128=int(rng.integers(0, 2)), log2_cols=int(rng.integers(0, 2)),
                  log2_rows=int(rng.integers(0, 2)), film_grain=int(rng.integers(0, 2)), screen_content=int(rng.integers(0, 2)))
        if seed & 1:
            tus = obu.inter_stream(seed, w, h, n_frames=4, motion_modes=int(rng.integers(0, 3)), **kw)
        else:
            tus = obu.intra_stream(seed, w, h, n_frames=2, **kw)
        r, info, _ = _ref_decode(tus, apply_grain=1)
        assert r == len(tus), "seed %d: stock dav1d rejected the stream (%d)" % (seed, r)
        assert (info[:, 0] == w).all() and (info[:, 1] == h).all() and (info[:, 2] == kw["bpc"]).all()
        n += r
    assert n == 12 * 2 + 12 * 4


def test_hook_wavefront_sort_is_a_valid_order():
    """b200hook_wave_sort (integration/dav1d/b200_hooks.c): the order it produces must keep every intra record behind the
    records whose pixels its edge array reads (the kernel's ticket order requirement), for records in decode order"""
    from dav1d_b200 import synth, levels as L
    dll = C.CDLL(stream.HOOKED_SO)
    S = synth.make_intra_frame(np.random.default_rng(11), 8, 328, 200)
    tx = S["intra_tx_decode_order"]
    n = len(tx)
    out = np.zeros_like(tx)
    w4 = (C.c_int32 * 3)(S["w4"], S["w4"] >> 1, S["w4"] >> 1)
    h4 = (C.c_int32 * 3)(S["h4"], S["h4"] >> 1, S["h4"] >> 1)
    dll.b200hook_wave_sort.restype = C.c_int
    scratch, cap = C.c_void_p(), C.c_size_t(0)          # the caller keeps the sort's scratch buffer between frames (freed with libc below)
    for _ in range(2):                                   # the second call reuses the buffer
        waves = dll.b200hook_wave_sort(tx.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p), n, w4, h4, 1, 1, C.byref(scratch), C.byref(cap))
    assert scratch.value and cap.value >= 4 * (n + 1)
    C.CDLL(None).free(scratch)
    assert waves == S["intra_waves"], (waves, S["intra_waves"])          # same depth as the generator's own numbering
    # same multiset of records, and every record's dependency cells are owned by earlier records
    assert sorted(out.tobytes()[i * tx.itemsize:(i + 1) * tx.itemsize] for i in range(n)) == \
           sorted(tx.tobytes()[i * tx.itemsize:(i + 1) * tx.itemsize] for i in range(n))
    owner = [np.full((h4[p], w4[p]), -1, np.int64) for p in range(3)]
    for i in range(n):
        r = out[i]
        pl, x, y = int(r["plane"]), int(r["x4"]), int(r["y4"])
        tw, th = L.TX_W[r["tx"]] // 4, L.TX_H[r["tx"]] // 4
        fl = int(r["flags"])
        om = owner[pl]
        if fl & 1:
            rows = min(th, h4[pl] - y) + (min(th, h4[pl] - y - th) if (fl & 8) and y + th < h4[pl] else 0)
            assert (om[y:y + rows, x - 1] >= 0).all(), "record %d reads a left neighbour that comes later" % i
        if fl & 2:
            cols = min(tw, w4[pl] - x) + (min(tw, w4[pl] - x - tw) if (fl & 4) and x + tw < w4[pl] else 0)
            assert (om[y - 1, x:x + cols] >= 0).all(), "record %d reads a top neighbour that comes later" % i
        om[y:y + th, x:x + tw] = i


def test_cli_md5_y4m_and_obu_file_roundtrip(tmp_path, capsys):
    """python -m dav1d_b200.cli (the tools/dav1d.c analogue): synthetic stream -> .obu file -> split into temporal units
    -> decoded -> md5 / y4m; the md5 must be the one of the stock reference's output for the same file"""
    import importlib.util
    from dav1d_b200 import cli
    spec = importlib.util.spec_from_file_location("build_emu", os.path.join(refs.ROOT, "tests", "emu", "build_emu.py"))
    m = importlib.util.module_from_spec(spec); spec.loader.exec_module(m)
    emu = m.build()
    obu_file, y4m = str(tmp_path / "s.obu"), str(tmp_path / "o.y4m")
    assert cli.main(["--synth", "inter:208x144:10:3:grain,mm", "-w", obu_file]) == 0
    tus = cli.split_temporal_units(open(obu_file, "rb").read())
    assert len(tus) == 3 and b"".join(tus) == open(obu_file, "rb").read()
    common = ["-i", obu_file, "--backend", emu, "--one-job-at-a-time", "--threads", "4"]
    capsys.readouterr()
    assert cli.main(common + ["--muxer", "md5"]) == 0
    got = capsys.readouterr().out.split()[0]
    r0, info0, out0 = _ref_decode(tus, apply_grain=1)
    want, n = cli.md5_of(cli.frames_of(info0, out0))
    assert r0 == 3 and n == 3 and got == want
    # --frametimes: one line per output frame (nanoseconds since the previous one), and the "Decoded n/n frames - x fps" line of tools/dav1d.c
    ft = str(tmp_path / "ft.txt")
    assert cli.main(common + ["--muxer", "null", "--frametimes", ft]) == 0
    lines = open(ft).read().split()
    assert len(lines) == 3 and all(int(v) >= 0 for v in lines) and sum(map(int, lines)) > 0
    assert "Decoded 3/3 frames (100.0%) - " in capsys.readouterr().err
    # the same stream wrapped in IVF and in Annex B (size-less OBUs) demuxes to the same temporal units and the same md5
    ivf = b"DKIF" + (0).to_bytes(2, "little") + (32).to_bytes(2, "little") + b"AV01" + (208).to_bytes(2, "little") + \
          (144).to_bytes(2, "little") + (25).to_bytes(4, "little") + (1).to_bytes(4, "little") + (3).to_bytes(4, "little") + bytes(4)
    for k, tu in enumerate(tus):
        ivf += len(tu).to_bytes(4, "little") + k.to_bytes(8, "little") + tu
    ivf_file = str(tmp_path / "s.ivf")
    open(ivf_file, "wb").write(ivf)
    assert cli.demux(ivf) == tus
    assert cli.main(["-i", ivf_file] + common[2:] + ["--verify", want]) == 0
    assert cli.main(["-i", ivf_file] + common[2:] + ["--verify", "0" * 32]) == 2

    def annexb(tu):
        out, pos = bytearray(), 0
        while pos < len(tu):                      # strip the size fields, add obu_length prefixes; one frame unit per TU
            hdr = tu[pos]
            size, p = cli._leb128(tu, pos + 1)
            body = bytes([hdr & ~2]) + tu[p:p + size]
            out += obu.leb128(len(body)) + body
            pos = p + size
        fu = obu.leb128(len(out)) + bytes(out)
        return obu.leb128(len(fu)) + fu
    ab = b"".join(annexb(tu) for tu in tus)
    assert cli.split_annexb(ab) == tus
    assert cli.main(common + ["-o", y4m]) == 0
    assert open(y4m, "rb").read(64).startswith(b"YUV4MPEG2 W208 H144 F25:1 Ip C420p10\nFRAME\n")
    assert os.path.getsize(y4m) == len(b"YUV4MPEG2 W208 H144 F25:1 Ip C420p10\n") + 3 * (6 + 208 * 144 * 3)


# ---- committed golden streams: tests/golden/stream_*.obu + the md5 of the stock reference's output (make_stream_golden.py)
def _golden():
    import json
    from dav1d_b200 import cli
    g = json.load(open(os.path.join(refs.ROOT, "tests", "golden", "stream_golden.json")))
    return {k: (cli.demux(open(os.path.join(refs.ROOT, "tests", "golden", "stream_%s.obu" % k), "rb").read()), v) for k, v in g.items()}


def _md5(dec_result):
    from dav1d_b200 import cli
    n, info, packed = dec_result
    assert n > 0, n
    return cli.md5_of(cli.frames_of(info, packed))


def test_golden_streams_reference_md5():
    """the committed streams decode with the stock reference to the committed digests (pins the reference build and the files)"""
    for name, (tus, want) in _golden().items():
        assert len(tus) == want["temporal_units"] and sum(map(len, tus)) == want["bytes"]
        assert _md5(_ref_decode(tus, apply_grain=1)) == (want["md5"], want["frames"]), name


@pytest.mark.emu
def test_golden_streams_hooked_emu_md5(emu_decoder):
    for name, (tus, want) in _golden().items():
        assert _md5(emu_decoder.decode(tus, apply_grain=1)) == (want["md5"], want["frames"]), name
    emu_decoder.stats(reset=True)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["key_8bit_tiles", "inter_10bit_all_tools"])
def test_golden_streams_hooked_gpu_md5(gpu_decoder, name):
    """compares with no reference decode: the digest of the reference's output is committed"""
    tus, want = _golden()[name]
    assert _md5(gpu_decoder.decode(tus, apply_grain=1)) == (want["md5"], want["frames"])
    gpu_decoder.stats(reset=True)


# ---- Level 1 inside a real dav1d: Dav1dDSPContext filled by b200_*_dsp_init (integration/dav1d/b200_level1.c) ----------
def _level1_case(dec, launches):
    n0 = launches()
    for gen, kw in ((obu.intra_stream, dict(n_frames=1)),
                    (obu.inter_stream, dict(n_frames=3, bpc=10, motion_modes=2, film_grain=1, global_motion=1))):
        tus = gen(4, 136, 96, payload_bytes_per_sb64=600, **kw)
        r0, _, out0 = _ref_decode(tus, n_threads=1, max_frame_delay=1, apply_grain=1)
        r1, _, out1 = dec.decode(tus, apply_grain=1)
        assert r0 == len(tus) and r1 == r0 and np.array_equal(out0, out1), gen.__name__
    assert launches() - n0 > 1000, "the DSP calls did not reach the back end"
    # no slot that dav1d defines may be left on dav1d's own C function (it would run on the CPU and still "pass")
    left, replaced = dec.c_slots_left()
    assert left == 0 and replaced > 400, "Level-1 tables: %d slots still on dav1d's C functions (%d replaced)" % (left, replaced)


@pytest.mark.emu
def test_level1_tables_inside_dav1d_emu():
    """dav1d's own recon_tmpl.c / lf_apply / cdef_apply / lr_apply / fg_apply running on the B200 function tables (all seven
    families): decoded pictures identical to stock dav1d, thousands of kernel launches behind the DSP pointers"""
    import importlib.util
    spec = importlib.util.spec_from_file_location("build_emu", os.path.join(refs.ROOT, "tests", "emu", "build_emu.py"))
    m = importlib.util.module_from_spec(spec); spec.loader.exec_module(m)
    emu_path = m.build()
    emu = refs.emu_lib()
    _level1_case(stream.Level1Decoder(backend=emu_path), lambda: int(emu.b200_launch_count()))


@pytest.mark.emu
def test_level1_tables_inside_dav1d_many_streams_emu():
    """the same harness over randomly parameterised streams: 8 / 10 / 12 bit, 4:2:0 / 4:4:4 / 4:0:0, screen content (pal_pred),
    segmentation with lossless segments (the WHT slot), global motion (warp8x8 / warp8x8t), film grain"""
    emu = refs.emu_lib()
    dec = stream.Level1Decoder(backend=emu.path)
    for seed in range(5000, 5016):
        rng = np.random.default_rng(seed)
        w, h = int(rng.integers(4, 20)) * 8 + int(rng.choice([0, 0, 2, 6])), int(rng.integers(4, 14)) * 8 + int(rng.choice([0, 0, 4]))
        kw = dict(bpc=int(rng.choice([8, 10, 12])), sb128=int(rng.integers(0, 2)), log2_cols=int(rng.integers(0, 2)),
                  film_grain=int(rng.integers(0, 2)), screen_content=int(rng.integers(0, 2)), layout=str(rng.choice(["420", "420", "444", "400"])),
                  segmentation=int(rng.integers(0, 2)), payload_bytes_per_sb64=800)
        if seed % 3:
            tus = obu.inter_stream(seed, w, h, n_frames=int(rng.integers(2, 5)), motion_modes=int(rng.integers(0, 3)),
                                   global_motion=int(rng.integers(0, 2)), hidden_every=int(rng.choice([0, 2])), **kw)
        else:
            tus = obu.intra_stream(seed, w, h, n_frames=2, **kw)
        r0, _, out0 = _ref_decode(tus, n_threads=1, max_frame_delay=1, apply_grain=1)
        r1, _, out1 = dec.decode(tus, apply_grain=1)
        assert r0 > 0 and r1 == r0 and np.array_equal(out0, out1), (seed, kw)


@pytest.mark.gpu
def test_level1_tables_inside_dav1d_gpu():
    """own process: the Level-1 thunks have no error channel (like dav1d's DSP functions) and abort on a CUDA failure"""
    import subprocess, sys
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "import test_stream as T\n"
            "from dav1d_b200 import _lib, stream\n"
            "lib = _lib.get_lib()\n"
            "T._level1_case(stream.Level1Decoder(), lambda: int(lib.b200_launch_count()))\n"
            "print('LEVEL1 OK', lib.b200_launch_count())\n") % (refs.ROOT, os.path.join(refs.ROOT, "tests"))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900)
    assert "LEVEL1 OK" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]
