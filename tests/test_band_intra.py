"""Band-sliced execution of frames with intra-machine records (intra blocks, palette, inter-intra, intra block copy):
each band runs its own intra records after its inter stages, records on a band's first row read their top edge from the
rows the band above saved before its post filters (B200FrameBand.intra / edge_top / edge_bottom). Every banded run must
equal the whole-frame job and the oracle byte for byte; plans a band cannot satisfy are refused on the host."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import refs
from dav1d_b200 import _lib, frame, synth
import test_frame as TF
import test_intra as TI
import test_looprestoration as TLR
import test_multigpu as TMG

MOTION = dict(p_obmc=0.2, p_warp=0.15, p_ii=0.15)


def _emu():
    return dict(lib=refs.emu_lib(), alloc=frame.NumpyAlloc())


def post_oracle(S, recon, run_lf=True, run_cdef=True, run_lr=True):
    """the post-filter stages of test_frame.oracle_frame on a given reconstruction"""
    import test_loopfilter as TLF
    import test_cdef as TCD
    out = {"recon": recon.copy()}
    S2 = dict(S); S2["pic"] = recon.copy()
    pic = TLF.lf_frame_oracle(S2) if run_lf else S2["pic"]
    S2["pic"] = pic
    out["dbl"] = pic.copy()
    cd = TCD.cdef_frame_oracle(S2) if run_cdef else pic
    out["cdef"] = cd
    if run_lr:
        S3 = dict(S2); S3["cdef"], S3["dbl"] = cd, pic
        out["lr"] = TLR.lr_frame_oracle(S3)
    return out


def check_banded(S, exp, rows, **kw):
    fb = frame.FrameBuffers(S, band_rows=rows, **kw)
    assert fb.n_bands() == -(-S["H"] // rows)
    fb.run_bands()
    fb.alloc.sync()
    TF.check_frame(S, fb, exp)
    return fb


def pal_frame(rng, bpc, W, H, ssh=1, ssv=1):
    """an intra frame in which a share of the blocks are palette blocks (PAL + RESID records, test_intra.make_mixed)"""
    S = TI.make_mixed(synth.make_intra_frame(rng, bpc, W, H, ssh, ssv), rng, p_pal=0.3, p_ii=0.0)
    S["mixed_pic0"] = np.zeros_like(S["pic"])
    recon = TI.run_mixed(refs.oracle().oracle_intra_frame, S)
    S2 = dict(S); S2["intra_tx"] = S["mixed_tx"]; S2["intra_pal"] = S["mixed_pal"]
    return S2, recon


# ---------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.emu
@pytest.mark.parametrize("bpc,W,H,ssh,ssv,p_intra", [(8, 200, 264, 1, 1, 0.25), (10, 136, 200, 1, 1, 0.2),
                                                     (8, 136, 264, 1, 0, 0.15), (10, 136, 200, 0, 0, 0.25)])
def test_emu_mixed_frame_bands(bpc, W, H, ssh, ssv, p_intra):
    """mixed inter / intra frames at 64- and 128-row bands (compact upload; fused compound prediction) equal the oracle and
    the whole-frame job; every band with intra records costs one intra launch, every band boundary one edge-backup launch"""
    S = synth.make_inter_frame(np.random.default_rng(1100), bpc, W, H, ssh, ssv, p_intra=p_intra, film_grain=bpc > 8)
    assert len(S["intra_tx"]) > 15
    exp = TF.oracle_frame(S)
    kw = _emu()
    whole = frame.FrameBuffers(S, **kw)
    whole.run()
    TF.check_frame(S, whole, exp)
    lib = kw["lib"]
    S0 = dict(S); S0["intra_tx"] = S["intra_tx"][:0]
    for rows, opts in ((64, dict(compact=True)), (128, dict(compact=True)), (64, dict(fused=True, compact=True))):
        fb0 = frame.FrameBuffers(S0, band_rows=rows, **opts, **kw)
        n = lib.b200_launch_count(); fb0.run_bands(); inter_only = lib.b200_launch_count() - n
        fb = frame.FrameBuffers(S, band_rows=rows, **opts, **kw)
        n = lib.b200_launch_count(); fb.run_bands(); launches = lib.b200_launch_count() - n
        TF.check_frame(S, fb, exp)
        assert np.array_equal(fb.output("p2"), whole.output("p2"))
        nb = fb.n_bands()
        assert nb > 1 and sum(b.intra[1] for b in fb.bands) == len(S["intra_tx"])
        assert sum(1 for b in fb.bands if b.intra[1] > 0) > 1, "intra records in one band only"
        assert launches == inter_only + sum(1 for b in fb.bands if b.intra[1] > 0) + nb - 1


@pytest.mark.emu
@pytest.mark.parametrize("bpc,W,H", [(8, 264, 200), (10, 200, 264)])
def test_emu_motion_mode_frame_bands_with_intra(bpc, W, H):
    """OBMC, warps, inter-intra (II + RESID records) and intra blocks, cut into bands"""
    S = synth.make_inter_frame(np.random.default_rng(1120), bpc, W, H, p_intra=0.1, film_grain=bpc > 8, **MOTION)
    modes = S["intra_tx"]["mode"]
    assert (modes == 15).sum() > 5 and (modes == 16).sum() > 5 and len(S["warp"]) > 10
    exp = TF.oracle_frame(S)
    for rows in (64, 128):
        check_banded(S, exp, rows, compact=True, **_emu())


@pytest.mark.emu
@pytest.mark.parametrize("bpc,W,H,ssh,ssv", [(8, 200, 200, 1, 1), (10, 136, 264, 0, 0)])
def test_emu_palette_frame_bands(bpc, W, H, ssh, ssv):
    """palette blocks (PAL + RESID records) next to intra blocks, banded, deblocked / CDEF / LR after each band"""
    rng = np.random.default_rng(1140 + bpc)
    S, recon = pal_frame(rng, bpc, W, H, ssh, ssv)
    assert (S["intra_tx"]["mode"] == 17).sum() > 10
    exp = post_oracle(S, recon)
    for rows in (64, 128):
        check_banded(S, exp, rows, compact=rows == 64, **_emu())


@pytest.mark.emu
@pytest.mark.parametrize("bpc,W,H,ssh,ssv", [(8, 200, 264, 1, 1), (10, 264, 136, 1, 0), (12, 136, 200, 0, 0)])
def test_emu_intra_frame_bands(bpc, W, H, ssh, ssv):
    """intra-only frames (every block intra, CFL, filter-intra, bottom-left edges) cut into bands, with the post filters"""
    S = synth.make_intra_frame(np.random.default_rng(1160 + bpc + W), bpc, W, H, ssh, ssv)
    assert (S["intra_tx"]["flags"] & 8).any()
    exp = TF.oracle_frame(S)
    for rows, compact in ((64, True), (128, False)):
        fb = check_banded(S, exp, rows, compact=compact, **_emu())
        assert all(b.intra[1] > 0 for b in fb.bands)


@pytest.mark.emu
@pytest.mark.parametrize("bpc,W,H,ssh,ssv", [(8, 328, 264, 1, 1), (10, 200, 264, 0, 0)])
def test_emu_intra_block_copy_bands(bpc, W, H, ssh, ssv):
    """intra block copy across bands: sources in the bands above are read from the picture itself, which is never filtered
    in such frames (deblocking, CDEF and loop restoration off); asking for filters with banded copies is refused"""
    S = synth.make_intra_frame(np.random.default_rng(1180 + bpc + W), bpc, W, H, ssh, ssv, p_ibc=0.3)
    t = S["intra_tx"]
    ibc = t[t["mode"] == synth.MODE_IBC]
    rows = 64
    band = lambda yy, pl: (yy << (ssv if pl else 0)) // rows
    src_band = np.array([band(int(r["luma_off"]) >> 16, int(r["plane"])) for r in ibc])
    dst_band = np.array([band(int(r["y4"]) * 4, int(r["plane"])) for r in ibc])
    assert (src_band < dst_band).sum() > 5, "no copy from an earlier band"
    exp = TI.oracle_intra(S)
    off = dict(run_lf=False, run_cdef=False, run_lr=False)
    for rows_, compact in ((64, True), (128, False)):
        fb = frame.FrameBuffers(S, band_rows=rows_, compact=compact, **off, **_emu())
        fb.run_bands()
        ok, where = TI.planes_equal(S, exp, fb.output("p0"))
        assert ok, (rows_, where)
    with pytest.raises(ValueError, match="intra block copy"):
        frame.FrameBuffers(S, band_rows=64, **_emu())


@pytest.mark.emu
def test_emu_mixed_frame_band_progress():
    """after band k of a mixed frame the rows b200_band_progress reports hold their final values"""
    ssh = ssv = 1
    S = synth.make_inter_frame(np.random.default_rng(1200), 8, 200, 328, ssh, ssv, p_intra=0.25)
    exp = TF.oracle_frame(S)
    fb = frame.FrameBuffers(S, band_rows=64, compact=True, **_emu())
    final = exp["lr"]
    hs = [S["H"], (S["H"] + ssv) >> ssv, (S["H"] + ssv) >> ssv]
    ws = [S["W"], (S["W"] + ssh) >> ssh, (S["W"] + ssh) >> ssh]
    prev = [0, 0, 0]
    for k in range(fb.n_bands()):
        fb.run_band(k)
        got = fb.output("p2")
        for pl in range(3):
            rows = fb.band_progress(k, pl)
            assert prev[pl] <= rows <= hs[pl]
            prev[pl] = rows
            o, st = S["off"][pl], S["stride"][pl]
            a = got[o:o + hs[pl] * st].reshape(hs[pl], st)[:rows, :ws[pl]]
            b = final[o:o + hs[pl] * st].reshape(hs[pl], st)[:rows, :ws[pl]]
            assert np.array_equal(a, b), "band %d plane %d: rows reported final are not" % (k, pl)
    assert prev == hs


def _mixed_gop():
    return [synth.make_inter_frame(np.random.default_rng(1220 + k), 8, 200, 200, p_intra=0.2, p_obmc=0.2, p_warp=0.1, p_ii=0.1)
            for k in range(6)]


def _worker_emu_mixed_bands(rank, world, port, outdir):
    sys.path.insert(0, os.path.dirname(__file__))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        pics = TMG._decode_emu(rank, world, _mixed_gop(), band_rows=64)
        np.savez(os.path.join(outdir, "r%d.npz" % rank), **{str(k): v for k, v in pics.items()})
    finally:
        dist.destroy_process_group()


@pytest.mark.emu
@pytest.mark.parametrize("world", [2, 3])
def test_ranks_shard_mixed_frames_in_bands(tmp_path, world):
    """a dependent group of mixed frames (intra blocks, inter-intra, OBMC, warps) in 64-row bands over gloo ranks equals the
    oracle's chained decode"""
    port = 29500 + (os.getpid() + 41 + world * 5) % 2000
    mp.spawn(_worker_emu_mixed_bands, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    frames = _mixed_gop()
    exp = TMG.oracle_gop(frames)
    got = TMG._collect(str(tmp_path), world, len(frames))
    for k, (a, b) in enumerate(zip(exp, got)):
        assert TLR.picture_equal(frames[k], b, a), "frame %d" % k


@pytest.mark.emu
def test_bottom_left_edge_below_the_band_is_refused():
    """a record whose bottom-left edge reaches below its band (a band edge inside a 128x128 superblock): ValueError from the
    planner, before anything is allocated or launched"""
    S = synth.make_intra_frame(np.random.default_rng(1240), 8, 200, 200)
    t = S["intra_tx"].copy()
    th = np.asarray(synth._L.TX_H)[t["tx"]] // 4
    cand = np.nonzero((t["plane"] == 0) & (t["x4"] > 0) & ((t["y4"] + th) * 4 == 64))[0]
    assert len(cand)
    t["flags"][cand[0]] |= 8
    S2 = dict(S); S2["intra_tx"] = t
    frame.band_plan(S2, 128)                                    # inside one band: fine
    with pytest.raises(ValueError, match="bottom-left"):
        frame.band_plan(S2, 64)
    lib = refs.emu_lib()
    n = lib.b200_launch_count()
    with pytest.raises(ValueError, match="bottom-left"):
        frame.FrameBuffers(S2, band_rows=64, lib=lib, alloc=frame.NumpyAlloc())
    assert lib.b200_launch_count() == n


@pytest.mark.emu
def test_band_validation_in_the_library():
    """b200_frame_run_band_phase refuses, with -2 and before any launch: the superblock-granular intra schedule over several
    bands, an intra range outside the job's records, a missing edge_top / edge_bottom"""
    S = synth.make_intra_frame(np.random.default_rng(1260), 8, 136, 200)
    lib = refs.emu_lib()
    fb = frame.FrameBuffers(S, band_rows=64, intra_sb=True, lib=lib, alloc=frame.NumpyAlloc())
    n = lib.b200_launch_count()
    with pytest.raises(_lib.B200Error, match="superblock"):
        fb.run_band_phase(0, 1)
    fb = frame.FrameBuffers(S, band_rows=64, lib=lib, alloc=frame.NumpyAlloc())
    b = fb.bands[1]
    keep = (b.intra[0], b.intra[1], b.edge_top)
    b.intra[1] = len(S["intra_tx"])
    with pytest.raises(_lib.B200Error, match="outside"):
        fb.run_band_phase(1, 1)
    b.intra[1], b.edge_top = keep[1], None
    with pytest.raises(_lib.B200Error, match="edge_top"):
        fb.run_band_phase(1, 1)
    b.edge_top = keep[2]
    fb.bands[0].edge_bottom = None
    with pytest.raises(_lib.B200Error, match="edge_bottom"):
        fb.run_band_phase(0, 3)
    assert lib.b200_launch_count() == n


def test_need_covers_warps_and_fused_compound():
    """the reference rows a band reads include the warps' 15 x 15 windows and both predictions of fused compound records"""
    S = synth.make_inter_frame(np.random.default_rng(1280), 8, 264, 328, p_warp=0.3, p_compound=0.5)
    ph = [S["H"], (S["H"] + S["ss_ver"]) >> S["ss_ver"]]
    for fused in (False, True):
        S2, bands, need, _ = frame.band_plan(S, 64, fused=fused)
        w = S2["warp"]
        assert len(w) > 10
        for k, b in enumerate(bands):
            f, c = b["warp"]
            for r in w[f:f + c]:
                cls = int(r["plane"] > 0)
                assert need[k, r["ref"], cls] >= min(int(r["src_y"]) + 12, ph[cls])
        if fused:
            a = S2["cfused"]
            assert len(a)
            for k, b in enumerate(bands):
                f, c = b["cfused"]
                for r in a[f:f + c]:
                    cls = int(r["plane"] > 0)
                    for i in range(2):
                        assert need[k, r["ref"][i], cls] >= min(int(r["src_y"][i]) + int(r["h"]) + 4, ph[cls])
    # an inter-only frame without warps or fused records: the plan is what it was (prediction records only)
    S = synth.make_inter_frame(np.random.default_rng(1281), 8, 264, 200)
    ph = [S["H"], (S["H"] + S["ss_ver"]) >> S["ss_ver"]]
    S2, bands, need, _ = frame.band_plan(S, 64)
    P = S2["pred"]
    exp = np.zeros_like(need)
    for k, b in enumerate(bands):
        f, c = b["pred"]
        for r in P[f:f + c]:
            cls = int(r["plane"] > 0)
            exp[k, r["ref"], cls] = max(exp[k, r["ref"], cls], min(int(r["src_y"]) + int(r["h"]) + 4, ph[cls]))
    assert np.array_equal(need, exp)


def test_scaled_predictions_are_not_band_sliced():
    S = synth.make_inter_frame(np.random.default_rng(1290), 8, 136, 200)
    S2 = dict(S); S2["scaled"] = np.zeros(3, np.uint8)
    frame.band_plan(S2, 256)                                    # one band: the job runs them
    with pytest.raises(ValueError, match="scaled"):
        frame.band_plan(S2, 64)


# ---------------------------------------------------------------------------------------------------------- GPU
GPU_SIZES = [(8, 648, 520), (10, 1288, 720)]


@pytest.mark.gpu
@pytest.mark.parametrize("bpc,W,H", GPU_SIZES)
def test_gpu_mixed_frame_bands(bpc, W, H):
    S = synth.make_inter_frame(np.random.default_rng(1300 + bpc), bpc, W, H, p_intra=0.15, film_grain=bpc > 8)
    exp = TF.oracle_frame(S)
    for rows, opts in ((64, dict(compact=True)), (128, dict(compact=True)), (64, dict(fused=True, compact=True)), (192, {})):
        check_banded(S, exp, rows, **opts)


@pytest.mark.gpu
@pytest.mark.parametrize("bpc,W,H", GPU_SIZES)
def test_gpu_motion_mode_and_palette_frame_bands(bpc, W, H):
    S = synth.make_inter_frame(np.random.default_rng(1320 + bpc), bpc, W, H, p_intra=0.1, film_grain=bpc > 8, **MOTION)
    exp = TF.oracle_frame(S)
    for rows in (64, 128):
        check_banded(S, exp, rows, compact=True)
    S, recon = pal_frame(np.random.default_rng(1330 + bpc), bpc, W, H)
    exp = post_oracle(S, recon)
    check_banded(S, exp, 64, compact=True)


@pytest.mark.gpu
@pytest.mark.parametrize("bpc,W,H", GPU_SIZES)
def test_gpu_intra_frame_bands(bpc, W, H):
    S = synth.make_intra_frame(np.random.default_rng(1340 + bpc), bpc, W, H)
    exp = TF.oracle_frame(S)
    for rows in (64, 128):
        check_banded(S, exp, rows, compact=True)
    S = synth.make_intra_frame(np.random.default_rng(1350 + bpc), bpc, W, H, p_ibc=0.3)
    exp = TI.oracle_intra(S)
    fb = frame.FrameBuffers(S, band_rows=64, compact=True, run_lf=False, run_cdef=False, run_lr=False)
    fb.run_bands()
    fb.alloc.sync()
    ok, where = TI.planes_equal(S, exp, fb.output("p0"))
    assert ok, where


def _gpu_mixed_frames(n, seed, W=TMG.GW, H=TMG.GH):
    return [synth.make_inter_frame(np.random.default_rng(seed + k), 8, W, H, p_intra=0.15, p_obmc=0.1, p_warp=0.05, p_ii=0.1)
            for k in range(n)]


@pytest.mark.gpu
@pytest.mark.timeout(600)
def test_gpu_single_rank_pipeline_mixed_bands():
    """world = 1, two frames in flight (n_streams=2: band k+1's intra runs beside band k's deblock on the other stream), eager
    decode_gop and CUDA-graph replay of a GopPipeline, against the oracle's chained decode"""
    from dav1d_b200 import shard, get_lib
    lib = get_lib()
    frames = _gpu_mixed_frames(6, 1400)
    exp = TMG.oracle_gop(frames)

    def make(S, rows):
        return frame.FrameBuffers(S, band_rows=rows, compact=True)
    got = shard.decode_gop(frames, make, None, 0, 1, lib, band_rows=64, n_streams=2)
    for k in range(len(frames)):
        assert TLR.picture_equal(frames[k], got[k], exp[k]), ("eager", k)
    # graph replay: 4 resident sets, 10 frames (eager, captured + replayed, replayed)
    base = _gpu_mixed_frames(4, 1420)
    seq = [base[n % 4] for n in range(10)]
    exp = TMG.oracle_gop(seq)
    sets = [frame.FrameBuffers(S, band_rows=64, compact=True) for S in base]
    pipe = shard.GopPipeline(lib, 0, 1, sets, n_streams=2, graphs=True)
    for _ in range(10):
        pipe.submit()
    pipe.sync()
    for n in range(6, 10):
        assert TLR.picture_equal(seq[n], pipe.output(n), exp[n]), ("graph", n)


def _worker_gpu_mixed(rank, world, port, outdir):
    sys.path.insert(0, os.path.dirname(__file__))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from dav1d_b200 import shard, get_lib

        def make(S, rows):
            return frame.FrameBuffers(S, band_rows=rows, compact=True)
        pics = shard.decode_gop(_gpu_mixed_frames(6, 1440), make, dist, rank, world, get_lib(), exchange="peer", band_rows=64)
        np.savez(os.path.join(outdir, "r%d.npz" % rank), **{str(k): v for k, v in pics.items()})
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.timeout(300)
def test_gpu_ranks_shard_mixed_frames_in_bands(tmp_path):
    """two ranks, reference rows as peer-memory puts, mixed frames in 64-row bands"""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    port = 29500 + (os.getpid() + 57) % 2000
    mp.spawn(_worker_gpu_mixed, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    frames = _gpu_mixed_frames(6, 1440)
    exp = TMG.oracle_gop(frames)
    got = TMG._collect(str(tmp_path), 2, len(frames))
    for k in range(len(frames)):
        assert TLR.picture_equal(frames[k], got[k], exp[k]), "frame %d" % k
