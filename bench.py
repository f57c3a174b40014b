#!/usr/bin/env python3
"""bench.py — throughput of the B200 AV1 reconstruction + post-filter back end (BASELINE.json metric:
Mpixels/s recon+postfilter @ 4K).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic records, per GPU.

Workloads
  4k8_inter (default)  BASELINE config 2/3: one 3840x2160 8-bit 4:2:0 inter frame per GPU per step:
             prediction (put / prep + avg / w_avg / mask / w_mask from 2 reference pictures, 8-tap and
             bilinear, MVs that also leave the picture) -> inverse transforms (var-tx, 4x4..64x64) ->
             deblock (2 sweeps) -> CDEF -> loop restoration (Wiener + self-guided). Records are
             synthesised at the record level (no AV1 streams / encoder exist here, SURVEY.md §7.7).
             Mpixels = luma pixels (3840*2160 = 8.29 Mpx per frame).
  itx8x8     BASELINE config 0: 2^20 inv_txfm_add DCT_DCT 8x8 8-bit blocks (67.1 Mpx) per step.
Multi-GPU: ONE dependent stream of frames, frame n on rank n mod N (one frame per GPU per step, weak scaling); frame n
predicts from the restored pictures of frames n-1 and n-2, which other ranks produce. A frame job is cut into bands of
superblock rows; after each band the producer puts the rows that became final into its two consumers' landing buffers over
NVLink peer memory and raises their progress flag, and a band starts when the references have progressed past the lowest
row it reads (dav1d's check_tile rule; dav1d_b200/shard.py). Inside the timed region, also on the e2e leg.

--impl reference times dav1d's own C functions (oracle/_ref, unmodified reference sources, HAVE_ASM=0:
no nasm in this image) on the host cores: one frame per thread (dav1d's frame threading), all cores.

--dump-outputs DIR writes what the timed path computed in its last timed step (the pictures a caller of that path
receives) as DIR/<name>.npy in float32, so that two builds can be compared output for output: the inputs are seeded and
the number of frames decoded before it is fixed by the arguments. Above 64 MB in all, every array is cut down to the
same seeded sample of its elements.
"""
import os as _os
# up to 32 hardware work queues, so that the frames in flight (one stream each) really run side by side: with the
# default of 8, kernels of streams that share a queue are dispatched one after the other
_os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
import argparse
import contextlib
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

ITX_DT = np.dtype([("dst_off", "<u4"), ("coef_off", "<u4"), ("eob", "<i2"), ("txtp", "u1"), ("plane", "u1")])
W4K, H4K = 3840, 2160


# ------------------------------------------------------------------------------ itx8x8 workload
def fdct_matrix(n):
    i = np.arange(n)[:, None].astype(np.float64)
    j = np.arange(n)[None, :].astype(np.float64)
    m = np.cos(np.pi * (2 * j + 1) * i / (2.0 * n))
    m[0] *= np.sqrt(0.5)
    return m


def make_itx8x8(seed, n_blocks, plane_w):
    """BASELINE config 0 records (vectorised port of the checkasm generator's distribution:
    random +-255 residual -> float forward DCT x 2.0 -> round; eob uniform over the dc-only /
    full classes; reference tests/checkasm/itx.c:185-242)."""
    from dav1d_b200 import synth
    rng = np.random.default_rng(seed)
    m = fdct_matrix(8)
    coefs = np.empty((n_blocks, 64), np.int16)
    eobs = np.empty(n_blocks, np.int16)
    order = synth.scan_table(1)          # dav1d_scans[TX_8X8]: scan position -> coefficient index
    inv = np.empty(64, np.int32)
    inv[order] = np.arange(64)
    chunk = 1 << 16
    for s in range(0, n_blocks, chunk):
        e = min(n_blocks, s + chunk)
        resid = rng.integers(-255, 256, (e - s, 8, 8)).astype(np.float64)
        out = np.einsum("ij,njk,lk->nil", m, resid.transpose(0, 2, 1), m) * 2.0   # [n][x][y]
        c = np.trunc(out.reshape(e - s, 64) + 0.5).astype(np.int64)
        dc_only = rng.integers(0, 2, e - s) == 0
        eob = np.where(dc_only, 0, rng.integers(1, 63, e - s))
        c[inv[None, :] > eob[:, None]] = 0
        coefs[s:e] = c.astype(np.int16)
        eobs[s:e] = eob
    per_row = plane_w // 8
    blocks = np.zeros(n_blocks, ITX_DT)
    i = np.arange(n_blocks)
    blocks["dst_off"] = (i // per_row) * 8 * plane_w + (i % per_row) * 8
    blocks["coef_off"] = i * 64
    blocks["eob"] = eobs
    blocks["txtp"] = 0
    rows = (n_blocks + per_row - 1) // per_row * 8
    pic = rng.integers(0, 256, (rows, plane_w), dtype=np.uint8)
    return blocks, coefs.reshape(-1), pic


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during the timed region: ONE long-running
    `nvidia-smi ... -lms 200` process (the recipe of B200_PROFILING.md) read by this thread, so that the run is
    not perturbed by a process spawn + driver attach per sample."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.proc = index, False, [], None
        self.marks = []

    def mark(self):
        """remember how many samples had arrived (called at the start and the end of the device-timed region)"""
        self.marks.append(len(self.samples))

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                f = [x.strip() for x in line.strip().split(",")]
                if len(f) >= 6:
                    self.samples.append(f)
                if self.stop_flag:
                    break
        except Exception:
            pass
        finally:
            self.stop()

    def stop(self):
        self.stop_flag = True
        p = self.proc
        if p is not None and p.poll() is None:
            try:
                p.terminate()          # exactly the process this object started
            except Exception:
                pass

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(int(float(s[0])) for s in self.samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(s[2 + k].lower().startswith("active") for s in self.samples)]
        out = {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(float(self.samples[0][1])), "reasons": reasons,
               "samples": len(sm)}
        if len(self.marks) >= 2:
            out["samples_in_timed_region"] = self.marks[1] - self.marks[0]
        return out


def host_threads():
    """threads the CPU arm may really use: the scheduler affinity set capped by the cgroup CPU quota (os.cpu_count() reports the
    machine, not the container: round 1's arm ran 64 threads on a box that gave it a quarter of that)"""
    try:
        aff = len(os.sched_getaffinity(0))
    except Exception:
        aff = os.cpu_count() or 1
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = max(1, int(float(q) / float(per) + 0.5))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = max(1, int(q / per + 0.5))
        except Exception:
            pass
    n = min(aff, quota) if quota else aff
    return max(1, n), {"os_cpu_count": os.cpu_count(), "affinity": aff, "cgroup_quota": quota}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# stage name (stage_times) -> key of frame_algorithmic_bytes
STAGE_BYTES_KEY = {"pred": "mc", "warp": "warp", "blend": "blend", "comp": "comp", "itx": "itx", "intra": "intra", "deblock": "deblock",
                   "cdef": "cdef", "lr": "lr", "fg": "fg"}
STAGE_NAMES = tuple(STAGE_BYTES_KEY)          # every name stage_times() can return


def frame_algorithmic_bytes(S, fused=False):
    """SURVEY.md §8(d) accounting for one frame, per stage (bytes); px = bytes per pixel."""
    px = S["pic"].itemsize
    cps = S["coefs"].itemsize
    ssh, ssv = [0, S["ss_hor"], S["ss_hor"]], [0, S["ss_ver"], S["ss_ver"]]
    samples = sum(((S["W"] + ssh[p]) >> ssh[p]) * ((S["H"] + ssv[p]) >> ssv[p]) for p in range(3))
    fused = fused and "cfused" in S
    b = S["pred_single"] if fused else S["pred"]
    foot = ((b["w"].astype(np.int64) + 7 * (b["mx"] != 0)) * (b["h"].astype(np.int64) + 7 * (b["my"] != 0))).sum() * px
    out = (b["w"].astype(np.int64) * b["h"] * np.where(b["op"] == 1, 2, px)).sum()
    if fused:      # a fused compound block: two footprints read + one block written (SURVEY §8d)
        c = np.concatenate([S["cfused"], S["cfused2"]])
        w_, h_ = c["w"].astype(np.int64), c["h"].astype(np.int64)
        comp = (sum((w_ + 7 * (c["mx"][:, k] != 0)) * (h_ + 7 * (c["my"][:, k] != 0)) for k in range(2)) * px + w_ * h_ * px).sum() if len(c) else 0
    else:
        c = np.concatenate([S["comp"], S["comp2"]])
        comp = (c["w"].astype(np.int64) * c["h"] * (4 + px)).sum()
    # 8x8 warps: 15x15 window read + 8x8 written; blends: prediction (pixel scratch) read + picture read-modify-write
    warp = len(S["warp"]) * (15 * 15 + 64) * px if "warp" in S else 0
    blend = sum(int((S[n]["w"].astype(np.int64) * S[n]["h"]).sum()) * 3 * px for n in ("blend", "blend2") if n in S)
    itx = 0
    from dav1d_b200 import levels as L
    for tx in range(19):
        n = len(S["itx"][tx])
        sw, sh = L.tx_coef_dims(tx)
        itx += n * (sw * sh * cps + 2 * L.TX_W[tx] * L.TX_H[tx] * px)
    luma = S["W"] * S["H"]
    intra = 0
    if S.get("intra_tx") is not None and len(S["intra_tx"]):
        t = S["intra_tx"]
        tw = np.array(L.TX_W)[t["tx"]].astype(np.int64); th = np.array(L.TX_H)[t["tx"]].astype(np.int64)
        coded = t["eob"] >= 0
        # prediction written + edge read; residual: coefficients read + picture read-modify-write
        intra = int(((tw * th + 2 * (tw + th) + 1) * px).sum() +
                    ((np.minimum(tw, 32) * np.minimum(th, 32) * cps + 2 * tw * th * px) * coded).sum())
    return {"intra": intra, "mc": int(foot + out), "warp": int(warp), "blend": int(blend), "comp": int(comp), "itx": int(itx), "deblock": int(4 * samples * px),
            "cdef": int(2 * samples * px), "lr": int(2 * samples * px),
            "fg": int((2 * samples + luma) * px) if S.get("fg") is not None else 0,   # + luma re-read by the chroma planes
            "samples": int(samples)}


FRAME_WORKLOADS = {
    "4k8_inter": dict(bpc=8, W=3840, H=2160, fg=False, dtype="u8/i16->i32",
                      desc="one 3840x2160 8-bit 4:2:0 inter frame per GPU per step: prediction (put/prep+compound, 2 refs) + "
                           "inverse transforms + deblock + CDEF + loop restoration (BASELINE configs[2])"),
    "4k8_mixed": dict(bpc=8, W=3840, H=2160, fg=False, dtype="u8/i16->i32", p_intra=0.10, p_obmc=0.10, p_warp=0.05, p_ii=0.05,
                      desc="4k8_inter with the block mix of real inter frames: 10 % of the blocks intra coded, and of the single-reference "
                           "blocks 10 % with overlapped block motion compensation, 5 % warped, 5 % inter-intra: the inter stages (incl. warp "
                           "and the two blend stages), then the dependency-driven intra kernel on top of them (done map pre-marked for the "
                           "inter cells), then the post filters"),
    "4k10_full": dict(bpc=10, W=3840, H=2160, fg=True, dtype="u16/i32->i32",
                      desc="one 3840x2160 10-bit 4:2:0 inter frame per GPU per step, full pipeline: prediction + inverse "
                           "transforms + deblock + CDEF + loop restoration + film grain (BASELINE configs[3])"),
    "8k10_full": dict(bpc=10, W=7680, H=4320, fg=True, dtype="u16/i32->i32",
                      desc="one 7680x4320 10-bit 4:2:0 inter frame per GPU per step, full pipeline incl. film grain "
                           "(BASELINE configs[4]: with --gpus N the frames of one dependent stream go round the ranks and every "
                           "restored picture reaches the two ranks that predict from it band by band over NVLink)"),
    "1080p8_intra": dict(bpc=8, W=1920, H=1080, fg=False, dtype="u8/i16->i32", intra=True, frames_per_step=int(os.environ.get("B200_INTRA_FPS", "96")),
                         desc="one 1920x1080 8-bit 4:2:0 intra-only frame per GPU per step: device-side edge preparation + "
                              "intra prediction + inverse transforms (dependency-driven kernel) + deblock (BASELINE configs[1]); a step is %s "
                              "independent frames in flight, 24 per launch / stream (an intra frame is a ~1000-deep dependency chain, "
                              "so frames, like dav1d's frame threads, are the parallel axis)" % os.environ.get("B200_INTRA_FPS", "96")),
}


def make_workload_frame(name, seed):
    from dav1d_b200 import synth
    wl = FRAME_WORKLOADS[name]
    if wl.get("intra"):
        return synth.make_intra_frame(np.random.default_rng(seed), wl["bpc"], wl["W"], wl["H"])
    return synth.make_inter_frame(np.random.default_rng(seed), wl["bpc"], wl["W"], wl["H"], film_grain=wl["fg"],
                                  **{k: wl[k] for k in ("p_intra", "p_obmc", "p_warp", "p_ii") if k in wl})


def workload_buffers(name, S, **kw):
    from dav1d_b200 import frame
    if FRAME_WORKLOADS[name].get("intra"):
        # frames in flight x CTAs per frame <= the 592 CTAs (4 per SM) that can be resident at once
        sb = bool(int(os.environ.get("B200_INTRA_SB", "1"))) and kw.get("lib") is None      # superblock-granular schedule
        return frame.FrameBuffers(S, run_cdef=False, run_lr=False, intra_grid=int(os.environ.get("B200_INTRA_GRID", "8")),
                                  intra_sb=sb, **kw)
    return frame.FrameBuffers(S, **kw)


# ... compound blocks go through prep + compound (the fused prediction kernel, B200_FUSED=1, measured slower: the stages
# are instruction bound, not HBM bound, so saving the int16 round trip does not pay: 114 us vs 33 + 29 us at 4K)
OURS = dict(compact=True, fused=bool(int(os.environ.get("B200_FUSED", "0"))))    # our arm ships coefficients 0 .. eob in scan order (the reference arm needs the dense plane)


# ------------------------------------------------------------------------------ reference arm / cpu baseline
def cpu_reps(S, n_threads, target_s=20.0):
    """frames per thread so that the CPU sample is ~target_s of CPU work (the C path does ~27 Mpixels/s per thread)"""
    return max(1, int(round(target_s / (n_threads * S["W"] * S["H"] / 27e6))))


def cpu_frames(S, n_threads, reps, use_ref=True):
    """`n_threads` frames in parallel, one per thread (frame threading), each through the reference's own
    functions (oracle/refdriver refdrv_frame_run) or, when oracle/_ref is absent, the oracle port."""
    import refs
    from dav1d_b200 import frame
    if use_ref and refs.have_ref():
        fn = refs.ref().refdrv_frame_run_8bpc if S["bpc"] == 8 else refs.ref().refdrv_frame_run_16bpc
        kind = "reference"
    else:
        import test_frame
        fn, kind = None, "port"
    intra_only = S.get("intra_tx") is not None and not len(S["pred"])
    wl = next((k for k, v in FRAME_WORKLOADS.items() if v.get("intra")), None) if intra_only else "4k8_inter"
    fbs = [workload_buffers(wl, S, lib=object(), alloc=frame.NumpyAlloc()) for _ in range(n_threads)] if fn else None

    def work(i):
        for _ in range(reps):
            if fn:
                fn(C.byref(fbs[i].job))
            else:
                test_frame.oracle_frame(S)
    ths = [threading.Thread(target=work, args=(i,)) for i in range(n_threads)]
    t0 = time.perf_counter()
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    dt = time.perf_counter() - t0
    return n_threads * reps * S["W"] * S["H"] / dt / 1e6, dt, kind


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from dav1d_b200 import synth
    ncores, thr_info = host_threads()
    arm_note = None
    if args.workload == "itx8x8":
        import refs
        n = 1 << 18
        blocks, coefs, pic = make_itx8x8(1, n, 8192)
        st = (C.c_int32 * 3)(8192, 8192, 8192)
        lib = refs.ref()

        def step():
            return lib.refdrv_itx_add_batch(255, 1, blocks.ctypes.data, n, coefs.ctypes.data, pic.ctypes.data, st, 0, ncores)
        for _ in range(args.warmup):
            step()
        t = [step() for _ in range(args.steps)]
        ms = 1e3 * sum(t) / len(t)
        val = n * 64 / (ms * 1e-3) / 1e6
        wl = ("itx8x8: 2^20 inv_txfm_add DCT_DCT 8x8 8-bit blocks per GPU per step (BASELINE config 0), "
              "checkasm-style coefficients, 8192x8192 plane")
        arm_note = "a sample of 2^18 of the 2^20 blocks per step"
        sample = "2^18 blocks/step, %d threads" % ncores
        kind = "reference"
    else:
        S = make_workload_frame(args.workload, 1)
        nthr = min(ncores, 64)
        for _ in range(args.warmup):
            cpu_frames(S, nthr, 1)
        vals, dts = [], []
        for _ in range(args.steps):
            v, dt, kind = cpu_frames(S, nthr, 1)
            vals.append(v); dts.append(dt)
        val = float(np.mean(vals)); ms = 1e3 * float(np.mean(dts))
        wl = "%s: %s" % (args.workload, FRAME_WORKLOADS[args.workload]["desc"])
        arm_note = "%d independent frames of this workload per step, one per host thread (dav1d's frame threading without its inter-frame waits: an upper bound for the CPU)" % nthr
        sample = "%d whole frames per step (one per thread; usable host threads: %r), dav1d C path HAVE_ASM=0 (no nasm in the image: not the AVX2 / AVX-512 path)" % (nthr, thr_info)
        ncores = nthr
    line = {"impl": "reference", "metric": "Mpixels/s", "value": val, "unit": "Mpixels/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": FRAME_WORKLOADS.get(args.workload, {"dtype": "u8/i16->i32"})["dtype"], "data": "synthetic",
            "config": {"workload": wl, "l2": "n/a (host)"},
            "arm_note": arm_note,
            "cpu_baseline": {"value": val, "unit": "Mpixels/s", "cores": ncores, "kind": kind, "sample": sample, "host": thr_info},
            "e2e": {"value": val, "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ------------------------------------------------------------------------------ real streams behind dav1d's front end
STREAM_WORKLOADS = {
    "stream1080p8": dict(W=1920, H=1080, bpc=8, frames=8, log2_cols=2, log2_rows=1,
                         desc="AV1 elementary stream, 8 key frames 1920x1080 8-bit 4:2:0, 4x2 tiles (valid headers, random tile "
                              "payloads: dav1d_b200/obu.py) decoded through dav1d's public API; front end (OBU parsing, entropy "
                              "decoding, threading) = unmodified dav1d on the host, back end = f->bd_fn record emitters + "
                              "libb200av1 (intra reconstruction, deblock, CDEF, loop restoration)"),
    "stream1080p8_inter": dict(W=1920, H=1080, bpc=8, frames=16, log2_cols=2, log2_rows=1, inter=1,
                               desc="AV1 elementary stream, 1 key frame + 15 inter frames 1920x1080 8-bit 4:2:0, 4x2 tiles (valid headers, "
                                    "random tile payloads: single / compound references incl. wedge and difference-weighted masks, OBMC, "
                                    "locally warped motion, inter-intra, transform trees, intra blocks) decoded through dav1d's public API; host front "
                                    "end = unmodified dav1d, back end = f->bd_fn record emitters + libb200av1, references resident in HBM"),
    "stream4k8_inter": dict(W=3840, H=2160, bpc=8, frames=8, log2_cols=2, log2_rows=2, inter=1,
                            desc="AV1 elementary stream, 1 key frame + 7 inter frames 3840x2160 8-bit 4:2:0, 4x4 tiles, all inter tools of "
                                 "stream1080p8_inter, decoded through dav1d's public API (host front end = unmodified dav1d, back end = libb200av1)"),
    # the same streams with statistics closer to encoder-made video: 60 % skipped blocks, half of the coded transform blocks all zero,
    # short end-of-block positions, 10 % intra blocks (tests/streamgen.py: the reference decoder chooses and range-encodes the symbols)
    "stream1080p8_sparse": dict(W=1920, H=1080, bpc=8, frames=16, log2_cols=2, log2_rows=1, inter=1,
                                gen=dict(p_skip=0.6, p_txskip=0.5, eob_draws=4, p_intra=0.1),
                                desc="AV1 elementary stream, 1 key frame + 15 inter frames 1920x1080 8-bit 4:2:0, 4x2 tiles, every tool of "
                                     "stream1080p8_inter, symbols chosen by the stream generator (60 % skipped blocks, 50 % all-zero transform "
                                     "blocks, short end-of-block positions, 10 % intra blocks) instead of a random payload; decoded through dav1d's public API"),
    "stream4k8_sparse": dict(W=3840, H=2160, bpc=8, frames=8, log2_cols=2, log2_rows=2, inter=1,
                             gen=dict(p_skip=0.6, p_txskip=0.5, eob_draws=4, p_intra=0.1),
                             desc="AV1 elementary stream, 1 key frame + 7 inter frames 3840x2160 8-bit 4:2:0, 4x4 tiles, the statistics of "
                                  "stream1080p8_sparse; decoded through dav1d's public API"),
    "stream4k10": dict(W=3840, H=2160, bpc=10, frames=6, log2_cols=2, log2_rows=2, inter=1, film_grain=1,
                       desc="AV1 elementary stream, 1 key frame + 5 inter frames 3840x2160 10-bit 4:2:0, 4x4 tiles, all inter tools of "
                            "stream1080p8_inter plus film grain on every frame (the full pipeline of BASELINE configs[3]) decoded through "
                            "dav1d's public API (host front end = unmodified dav1d, back end incl. film grain = libb200av1)"),
}


def run_stream(args):
    """e2e = pixels / wall time of the whole decode (dav1d_send_data -> pictures out); value = pixels / time spent in the
    device jobs (record upload + kernels + picture download, from the hooks' own clock). Reference arm = the stock
    reference decoding the same stream with the same number of threads."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    from dav1d_b200 import obu, stream
    W = STREAM_WORKLOADS[args.workload]
    nthr = int(os.environ.get("B200_STREAM_THREADS", min(host_threads()[0], 32)))     # dav1d worker threads, both arms
    mfd = min(8, W["frames"], nthr)
    gen = (lambda *a, **k: obu.inter_stream(*a, motion_modes=2, **k)) if W.get("inter") else obu.intra_stream
    fg = int(W.get("film_grain", 0))
    build = lambda: gen(100 + rank, W["W"], W["H"], n_frames=W["frames"], bpc=W["bpc"], log2_cols=W["log2_cols"], log2_rows=W["log2_rows"], film_grain=fg)
    if W.get("gen"):
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import streamgen                 # workload synthesis only (test infrastructure): the generator is not on any measured path
        tus = streamgen.generate(build, seed=100 + rank, check=False, **W["gen"])[0]
    else:
        tus = build()
    px = W["W"] * W["H"] * W["frames"]
    stream.decode_stream.capacity = (W["W"] * W["H"] * 3 // 2) * (2 if W["bpc"] > 8 else 1) * W["frames"] + (1 << 20)
    steps = args.steps
    wl = "%s: %s; %d dav1d threads, %d frames in flight" % (args.workload, W["desc"], nthr, mfd)
    if args.impl == "reference":
        if rank != 0:
            return
        import refs
        dll = C.CDLL(refs.REF_SO)
        for _ in range(min(args.warmup, 1)):
            stream.decode_stream(dll, tus, n_threads=nthr, max_frame_delay=mfd, apply_grain=fg)
        dts = []
        for _ in range(steps):
            t0 = time.perf_counter()
            r, _, _ = stream.decode_stream(dll, tus, n_threads=nthr, max_frame_delay=mfd, apply_grain=fg)
            dts.append(time.perf_counter() - t0)
            assert r == W["frames"], r
        ms = 1e3 * float(np.mean(dts)); val = px / (ms * 1e-3) / 1e6
        emit({"impl": "reference", "metric": "Mpixels/s", "value": val, "unit": "Mpixels/s", "n_gpus": args.gpus, "steps": steps,
              "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
              "dtype": "u8/i16->i32" if W["bpc"] == 8 else "u16/i32", "data": "synthetic", "config": {"workload": wl, "l2": "n/a (host)"},
              "cpu_baseline": {"value": val, "unit": "Mpixels/s", "cores": nthr, "kind": "reference",
                               "sample": "the whole stream per step, stock dav1d (C path, HAVE_ASM=0), %d threads" % nthr},
              "e2e": {"value": val, "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0})
        return
    torch, dist, world, rank, local = dist_setup()
    from dav1d_b200 import get_lib
    lib = get_lib()
    dec = stream.HookedDecoder()
    for _ in range(max(args.warmup, 3) if steps > 1 else 1):
        r, _, _ = dec.decode(tus, n_threads=nthr, max_frame_delay=mfd, apply_grain=fg)
        assert r == W["frames"], "hooked decode failed: %d" % r
    dec.stats(reset=True)
    before = lib.b200_launch_count()
    sampler = ClockSampler(local); sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        r, _, out = dec.decode(tus, n_threads=nthr, max_frame_delay=mfd, apply_grain=fg)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    sampler.stop()
    st = dec.stats()
    if args.dump_outputs and rank == 0:            # every picture of the last decode, packed plane after plane
        dump_outputs(args.dump_outputs, {"pictures": out.view(np.uint16) if W["bpc"] > 8 else out})
    if world > 1:
        tt = torch.tensor([dt], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
    launches = lib.b200_launch_count() - before
    ms = 1e3 * dt / steps
    e2e = world * px / (ms * 1e-3) / 1e6
    dev_ms = st["device_ms"] / max(st["frames"], 1)
    value = world * W["W"] * W["H"] / (dev_ms * 1e-3) / 1e6
    pxb = 2 if W["bpc"] > 8 else 1
    S_ = W["W"] * W["H"] * 3 // 2
    alg = st["coefs"] / max(st["frames"], 1) * (2 * pxb) + S_ * pxb * (1 + 2 + 4 + 2 + 2)   # coefs + pred write + itx rmw + deblock + cdef + lr
    peak, src = measured_peak()
    # the CPU arm beside it (bounded: one decode of the same stream by the stock reference)
    cpu = None
    if rank == 0:
        import refs
        dll = C.CDLL(refs.REF_SO)
        t1 = time.perf_counter(); rr, _, ref_out = stream.decode_stream(dll, tus, n_threads=nthr, max_frame_delay=mfd, apply_grain=fg); tc = time.perf_counter() - t1
        assert rr == W["frames"] and np.array_equal(ref_out, out), "stream bench: output differs from the stock reference"
        cpu = {"value": px / tc / 1e6, "unit": "Mpixels/s", "cores": nthr, "kind": "reference",
               "sample": "one decode of the same stream by stock dav1d (C path, HAVE_ASM=0), %d threads, %.2f s; outputs compared byte for byte" % (nthr, tc)}
    if rank == 0:
        emit({"metric": "Mpixels/s", "value": value, "unit": "Mpixels/s", "n_gpus": world, "steps": steps, "warmup": max(args.warmup, 3),
              "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
              "dtype": "u8/i16->i32" if W["bpc"] == 8 else "u16/i32", "data": "synthetic",
              "config": {"workload": wl, "l2": "every frame's records and pictures are fresh (uploaded per frame)",
                         "value_is": "pixels / time inside the per-frame device jobs (H2D of records + kernels + D2H of the picture), host clock",
                         "records_per_frame": {k: st[k] // max(st["frames"], 1) for k in ("intra_tx", "pred", "comp", "warp", "blend", "itx")},
                         "host_ms_per_frame": {"completion_before_job (mask fix-ups, wavefront sort, staging)": st["host_prep_ms"] / max(st["frames"], 1),
                                               "device_job": dev_ms, "whole_decode_wall": ms / W["frames"]}},
              "roofline": {"bound": "hbm", "kernel": "frame job (intra reconstruction + deblock + CDEF + LR, incl. PCIe copies)",
                           "achieved": alg / (dev_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                           "frac": alg / (dev_ms * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": src},
              "cpu_baseline": cpu,
              "e2e": {"value": e2e, "unit": "Mpixels/s", "h2d_bytes_per_step": st["h2d_bytes"] // steps, "d2h_bytes_per_step": st["d2h_bytes"] // steps},
              "gpu_launches": int(launches), "clocks": sampler.summary()})
    dec.release()


# ------------------------------------------------------------------------------ our arm
def dist_setup():
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return torch, dist, world, rank, local


def run_ours_frame(args):
    torch, dist, world, rank, local = dist_setup()
    from dav1d_b200 import synth, frame, get_lib
    lib = get_lib()
    # frames in flight for the device-resident measurement: consecutive frames go round-robin to this many streams (the
    # device-side analogue of dav1d's frame threads, n_fc): one frame's kernel tails and launch gaps are filled by the
    # next frame's kernels. Every frame set always runs on the same stream (nsets is a multiple of the stream count).
    n_streams = max(1, int(os.environ.get("B200_FRAMES_IN_FLIGHT", "2")))
    nsets = max(24, FRAME_WORKLOADS[args.workload].get("frames_per_step", 1)) if FRAME_WORKLOADS[args.workload].get("intra") else int(os.environ.get("B200_NSETS", "3" if args.workload == "8k10_full" else "6"))
    if not FRAME_WORKLOADS[args.workload].get("intra"):
        nsets = -(-nsets // n_streams) * n_streams
    side = [torch.cuda.Stream() for _ in range(n_streams)] if n_streams > 1 else []
    fbs, Ss = [], []
    for k in range(nsets):
        # at most 8 distinct synthetic frames; every set still owns its device buffers (that is what defeats L2)
        S = make_workload_frame(args.workload, 1 + rank * 16 + k) if k < 8 else Ss[k % 8]
        Ss.append(S)
        fbs.append(workload_buffers(args.workload, S, **OURS))
    fps = FRAME_WORKLOADS[args.workload].get("frames_per_step", 1)
    px_per_step = fps * FRAME_WORKLOADS[args.workload]["W"] * FRAME_WORKLOADS[args.workload]["H"]
    GROUP = 24
    groups = [frame.FrameGroup(fbs[g:g + GROUP]) for g in range(0, nsets, GROUP)] if fps > 1 else []
    ev_go = torch.cuda.Event() if fps > 1 else None
    ev_done = [torch.cuda.Event() for _ in groups]
    gather, pending = None, [None] * nsets
    if world > 1:   # reference-picture exchange buffers (one per frame set): every rank's restored picture
        gather = [torch.empty(world * Ss[0]["pic"].nbytes, dtype=torch.uint8, device="cuda") for _ in range(nsets)]

    def step(i):
        if fps > 1:      # fps frames in flight: groups of 24 frames, one batched job per group on its own stream
            cur = torch.cuda.current_stream()
            ev_go.record(cur)
            for k, g in enumerate(groups):
                g.stream()
                gs = g._stream[0]                 # torch stream object of the group
                gs.wait_event(ev_go)
                g.run()
                ev_done[k].record(gs)
                cur.wait_event(ev_done[k])
            return
        k = i % nsets
        fb = fbs[k]
        ctx = torch.cuda.stream(side[k % n_streams]) if side else contextlib.nullcontext()
        with ctx:
            if pending[k] is not None:      # the exchange that still reads this frame set's picture (issued nsets steps ago)
                pending[k].wait()
            fb.run()
            if world > 1:
                # the exchange of frame i overlaps the reconstruction of frame i + 1 (NCCL stream; un-grained picture)
                pending[k] = dist.all_gather_into_tensor(gather[k], fb.keep[fb.ref_name][0][:Ss[0]["pic"].nbytes], async_op=True)

    def sync_all():
        for k in range(nsets):
            if pending[k] is not None:
                pending[k].wait(); pending[k] = None
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    sync_all()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = lib.b200_launch_count()
    ev = [torch.cuda.Event(enable_timing=True)]
    ev[0].record()
    main = torch.cuda.current_stream()
    for s_ in side:
        s_.wait_stream(main)            # the timed region starts on every stream after ev[0]
    for i in range(args.steps):
        step(i)
    for k in range(nsets):              # the timed region ends when the last exchanges have landed too
        if pending[k] is not None:
            pending[k].wait(); pending[k] = None
    for s_ in side:
        main.wait_stream(s_)            # ... and when every stream has drained
    ev_end = torch.cuda.Event(enable_timing=True)
    ev_end.record()
    sync_all()
    launches = lib.b200_launch_count() - launches0
    if args.dump_outputs and rank == 0:            # the displayed pictures of the frames of the last timed step
        last = range(nsets) if fps > 1 else [(args.steps - 1) % nsets]
        arrays = {}
        for k in last:
            arrays.update(picture_arrays("picture%d_" % k if fps > 1 else "picture_", Ss[k], fbs[k].output()))
        dump_outputs(args.dump_outputs, arrays)
    total_ms = ev[0].elapsed_time(ev_end)
    t = torch.tensor([total_ms], device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = float(t.item()) / args.steps
    value = world * px_per_step / (ms_per_step * 1e-3) / 1e6

    # per-stage device times (CUDA events around each stage's launches, same stream, same rotation)
    stage_ms = stage_times(torch, lib, fbs, nsets)

    # end to end: records from pinned host memory through b200_frame_run_host, picture back to the host
    # nsets frames in flight, one stream each (the GPU-side analogue of dav1d's frame threads): every step
    # copies that frame's records host->device and its restored picture device->host.
    units = groups if fps > 1 else fbs                      # what is submitted at once: a group of 24 frames or one frame
    per_unit = GROUP if fps > 1 else 1
    e2e_steps = max(4 * len(units), min(args.steps, 400) // per_unit)     # many more submissions than units in flight
    for i in range(2 * len(units)):
        if i >= len(units):
            units[i % len(units)].wait()
        units[i % len(units)].submit_host()
    for u in units:
        u.wait()
    sync_all()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        if i >= len(units):
            units[i % len(units)].wait()
        units[i % len(units)].submit_host()
    for u in units:
        u.wait()
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
    t = torch.tensor([e2e_ms], device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_val = world * per_unit * (px_per_step // fps) / (float(t.item()) * 1e-3) / 1e6
    sampler.stop()
    sampler.join(timeout=2)

    if rank == 0:
        peak, peak_src = measured_peak()
        alg = frame_algorithmic_bytes(Ss[0], fused=bool(fbs[0].job.n_cfused))
        stages = {}
        for name, ms in stage_ms.items():
            key = STAGE_BYTES_KEY[name]
            stages[name] = {"ms": ms, "algorithmic_bytes": alg[key], "GBps": alg[key] / (ms * 1e-3) / 1e9 if ms > 0 else None}
        dom = max(stage_ms, key=lambda k: stage_ms[k])
        traffic = None
        tp = os.path.join(ROOT, "profiles", "frame_traffic.json")
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get(dom)
        achieved = stages[dom]["GBps"]
        run_keys = STAGE_BYTES_KEY
        total_alg = sum(alg[run_keys[k]] for k in stage_ms)
        recon_ms = sum(v for k, v in stage_ms.items() if k in ("pred", "warp", "blend", "comp", "itx", "intra"))
        post_ms = sum(v for k, v in stage_ms.items() if k in ("deblock", "cdef", "lr", "fg"))
        split = {"recon": {"ms": recon_ms, "Mpixels/s": px_per_step / (recon_ms * 1e-3) / 1e6,
                           "GBps": sum(alg[run_keys[k]] for k in stage_ms if k in ("pred", "warp", "blend", "comp", "itx", "intra")) / (recon_ms * 1e-3) / 1e9},
                 "postfilter": {"ms": post_ms, "Mpixels/s": px_per_step / (post_ms * 1e-3) / 1e6,
                                "GBps": sum(alg[run_keys[k]] for k in stage_ms if k in ("deblock", "cdef", "lr", "fg")) / (post_ms * 1e-3) / 1e9}}
        nthr = min(host_threads()[0], 32)
        cr = cpu_reps(Ss[0], nthr)
        v, dt, kind = cpu_frames(Ss[0], nthr, cr)
        cpu = {"value": v, "unit": "Mpixels/s", "cores": nthr, "kind": kind,
               "sample": "%d whole frames of this workload, %d per thread on %d threads (frame threading), dav1d C path HAVE_ASM=0 (no nasm in image), %.1f s wall, ~%.0f s of CPU work" % (nthr * cr, cr, nthr, dt, dt * nthr)}
        line = {"metric": "Mpixels/s", "value": value, "unit": "Mpixels/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": FRAME_WORKLOADS[args.workload]["dtype"], "data": "synthetic",
                "config": {"workload": "%s: %s" % (args.workload, FRAME_WORKLOADS[args.workload]["desc"]),
                           "frames_in_flight": n_streams, "l2": "%d rotating frame sets (~%d MB) > 126 MB L2" % (nsets, nsets * ((2 + len(Ss[0]["refs"]) + fbs[0].job.run_cdef + fbs[0].job.run_lr + fbs[0].job.run_fg) * Ss[0]["pic"].nbytes + Ss[0]["coefs"].nbytes) // 1000000),
                           "records": {"pred_blocks": int(len(Ss[0]["pred"])), "compound": int(len(Ss[0]["comp"]) + len(Ss[0]["comp2"])),
                                       "tx_blocks": int(sum(len(a) for a in Ss[0]["itx"].values())), "coefs": int(len(Ss[0]["coefs"])),
                                       "intra_tx_blocks": int(len(Ss[0].get("intra_tx", []))), "intra_waves": int(Ss[0].get("intra_waves", 0))},
                           "compound": "fused: both predictions + avg/w_avg/mask/w_mask in one kernel, int16 intermediates stay on the SM",
                           "upload": "per coded transform block the coefficients 0..eob in scan order (expanded on the device inside the timed job) + block records + masks/levels",
                           "exchange": "all_gather of each rank's restored picture per step (NCCL, asynchronous: overlaps the next frame)" if world > 1 else "none"},
                "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                             "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                             "whole_frame": {"algorithmic_bytes": total_alg, "GBps": total_alg / (ms_per_step * 1e-3) / 1e9,
                                             "frac": total_alg / (ms_per_step * 1e-3) / 1e9 / peak},
                             "stages": stages, "split": split},
                "cpu_baseline": cpu,
                "e2e": {"value": e2e_val, "unit": "Mpixels/s", "h2d_bytes_per_step": int(fbs[0].h2d_bytes),
                        "d2h_bytes_per_step": int(fbs[0].d2h_bytes)},
                "gpu_launches": int(launches), "clocks": sampler.summary()}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def picture_planes(S, pic):
    """the visible area of each plane of a picture of frame S, as 2-D views"""
    ssh, ssv = [0, S["ss_hor"], S["ss_hor"]], [0, S["ss_ver"], S["ss_ver"]]
    out = []
    for pl in range(3):
        h, w = (S["H"] + ssv[pl]) >> ssv[pl], (S["W"] + ssh[pl]) >> ssh[pl]
        o, st = S["off"][pl], S["stride"][pl]
        out.append(pic[o:o + h * st].reshape(h, st)[:, :w])
    return out


def planes_differ(S, a, b):
    """first (plane, row) where the visible area of two pictures of frame S differs, or None"""
    for pl, (A, B) in enumerate(zip(picture_planes(S, a), picture_planes(S, b))):
        if not np.array_equal(A, B):
            return pl, int(np.where((A != B).any(axis=1))[0][0])
    return None


def picture_arrays(prefix, S, pic):
    return {"%s%s" % (prefix, n): p for n, p in zip(("y", "u", "v"), picture_planes(S, pic))}


def dev_to_numpy(lib, ptr, like):
    out = np.empty_like(like)
    lib.check(lib.b200_copy_async(out.ctypes.data, ptr, out.nbytes, None), "b200_copy_async")
    lib.check(lib.b200_frame_wait(None), "b200_frame_wait")
    return out


def run_ours_gop(args):
    """the inter workloads: one dependent stream of frames over the ranks (dav1d_b200/shard.py)"""
    torch, dist, world, rank, local = dist_setup()
    from dav1d_b200 import frame, shard, get_lib
    lib = get_lib()
    wl = FRAME_WORKLOADS[args.workload]
    W, H = wl["W"], wl["H"]
    px_per_frame = W * H
    whole = -(-H // 64) * 64
    # bands: one GPU decodes whole frames (nothing to wait for: stream order is the dependency); over several GPUs a frame
    # is cut into bands of superblock rows so that frame n+1 starts on its GPU while frame n is still being decoded
    # ... the band height: a band of frame n+1 may start once frame n has restored ~144 luma rows more than the band's bottom
    # (motion reach + filter taps + the rows the post filters still hold back), i.e. frame n+1 trails frame n by about
    # (144 + band) rows; N ranks stay busy when N such lags fit into a frame, hence ~H / 3N rows per band — as few bands as
    # that allows, because every band is a dozen more (small) launches
    n_bands = min(2 * world + 1, max(2, H // 256))          # ... and no more than ~256-row bands: a band costs ~55 us of launch chain
    # ... from 4 ranks on the stream is bound by the frame-to-frame lag (one band period + the launch chains of a band's
    # reconstruction and post filters + 2 bands of work), not by GPU time: measured at N=4 (profiles/r02_bench_n4_*): 4K
    # 0.369 / 0.282 / 0.315 ms per frame with 128 / 192 / 320-row bands, 8K 0.686 / 0.606 with 128 / 192, 0.558 with 320 (N=8)
    default_rows = whole if world == 1 else -(-H // n_bands) if world < 4 else (192 if H <= 2160 else 320)
    if wl.get("p_intra") or wl.get("p_ii"):
        default_rows = whole             # intra-machine records form a dependency graph over the frame: such frames are not cut into bands
    band_rows = int(os.environ.get("B200_BAND_ROWS", str(default_rows)))
    band_rows = min(whole, max(64, -(-band_rows // 64) * 64))
    n_streams = max(1, int(os.environ.get("B200_FRAMES_IN_FLIGHT", "1" if world == 1 else "2")))
    nsets = int(os.environ.get("B200_NSETS", "3" if args.workload == "8k10_full" else "6"))
    # a banded frame is hundreds of launches, waits and copies: replayed as one CUDA graph per frame (the host would otherwise
    # be the bottleneck: ~100 us of launch calls per band)
    graphs = bool(int(os.environ.get("B200_GRAPHS", "1" if -(-H // band_rows) > 1 else "0")))
    mult = n_streams * (2 if graphs and n_streams % 2 else 1)       # graph replay: an even number of sets (fixed landing slots per set)
    nsets = -(-nsets // mult) * mult
    distinct = min(nsets, int(os.environ.get("B200_DISTINCT", "2" if args.workload == "8k10_full" else "3")))
    Ss = [make_workload_frame(args.workload, 1 + rank * 16 + k) for k in range(distinct)]
    sets = [workload_buffers(args.workload, Ss[k % distinct], band_rows=band_rows, **OURS) for k in range(nsets)]
    x = shard.PeerExchange(lib, dist, rank, world, Ss[0]["pic"].nbytes, 2) if world > 1 else None
    # programmatic dependent launch pays on one chain of whole-frame launches; parked CTAs hurt when chains share the GPU
    lib.b200_set_pdl(1 if (-(-H // band_rows) == 1 and n_streams == 1) else 0)
    pipe = shard.GopPipeline(lib, rank, world, sets, exchange=x, n_refs=2, n_streams=n_streams, graphs=graphs)
    main = torch.cuda.current_stream()
    tstreams = [t for t, _ in pipe.streams] + ([pipe.copy_stream[0]] if pipe.copy_stream[0] is not None else []) + \
               [t for t, _ in (pipe.post_streams or [])]

    def sync_all():
        pipe.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- parity before timing: this rank's first frame (global frame `rank`) against the reference's own functions
    # (oracle/_ref: dav1d's C path over the same records), given the references this rank holds for it — synthetic ones
    # before the stream starts, otherwise the rows its producers put into the landing buffers
    pipe.submit()
    sync_all()
    parity = None
    if not int(os.environ.get("B200_SKIP_PARITY", "0")):
        import refs
        if refs.have_ref():
            S0 = dict(Ss[0])
            S0["refs"] = []
            for d in (1, 2):
                kind, mseq = pipe.ref_source(rank, d)
                S0["refs"].append(Ss[0]["refs"][d - 1] if kind == "own" else
                                  dev_to_numpy(lib, x.landing_ptr(d, mseq % shard.K_SLOTS) if kind == "remote" else sets[mseq % nsets].picture_ptr(pipe.ref_name), Ss[0]["pic"]))
            fbr = workload_buffers(args.workload, S0, lib=object(), alloc=frame.NumpyAlloc())
            fn = refs.ref().refdrv_frame_run_8bpc if S0["bpc"] == 8 else refs.ref().refdrv_frame_run_16bpc
            fn(C.byref(fbr.job))
            bad = planes_differ(S0, sets[0].output(pipe.ref_name), fbr.output(fbr.ref_name))
            if bad is None and fbr.out_name != fbr.ref_name:
                bad = planes_differ(S0, sets[0].output(sets[0].out_name), fbr.output(fbr.out_name))
            ok = torch.tensor([0 if bad is None else 1], device="cuda")
            if world > 1:
                dist.all_reduce(ok, op=dist.ReduceOp.MAX)
            if int(ok.item()):
                raise SystemExit("bench: parity check failed on rank %d: frame %d differs from the reference at (plane, row) %r" % (rank, rank, bad))
            parity = "frame n = rank of the stream on every rank (%dx%d, the bench workload itself), restored%s picture byte-identical to dav1d's C functions (oracle/_ref) given the same records and references" % (W, H, " and grained" if wl["fg"] else "")
        else:
            parity = "skipped: oracle/_ref not built"

    def block(nframes):
        for _ in range(nframes):
            pipe.submit()

    # every set runs twice before timing: buffers touched, and with graphs each set's schedule captured (on its 2nd frame)
    args.warmup = max(args.warmup, 2 * nsets)
    block(args.warmup)
    sync_all()
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.15)
    put0 = pipe.bytes_put
    launches0 = lib.b200_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.mark()
    ev0.record(main)
    for t in tstreams:
        t.wait_stream(main)             # the timed region starts on every stream after ev0
    block(args.steps)
    for t in tstreams:
        main.wait_stream(t)             # ... and ends when every stream (incl. the puts) has drained
    ev1.record(main)
    sync_all()
    sampler.mark()
    launches = lib.b200_launch_count() - launches0
    t = torch.tensor([ev0.elapsed_time(ev1)], device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = float(t.item()) / args.steps
    value = world * px_per_frame / (ms_per_step * 1e-3) / 1e6
    put_per_frame = (pipe.bytes_put - put0) // max(1, args.steps)
    if args.dump_outputs and rank == 0:            # the displayed picture of this rank's last timed frame
        last = pipe.submitted - 1
        dump_outputs(args.dump_outputs, picture_arrays("picture_", Ss[last % nsets % distinct], pipe.output(last, sets[0].out_name)))

    stage_ms = stage_times(torch, lib, sets, nsets)

    # ---- end to end: the same stream of frames, every frame's records from pinned host memory (H2D) and its output picture
    # back to the host (D2H), the reference exchange between the GPUs included; host clock, max over ranks
    pipe.enable_host_io()
    block(max(2, nsets)); sync_all()
    e2e_frames = max(2 * nsets, int(0.4 / max(ms_per_step * 1e-3, 1e-5) / 2))
    t0 = time.perf_counter()
    block(e2e_frames)
    pipe.sync()
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_frames
    t = torch.tensor([e2e_ms], device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_val = world * px_per_frame / (float(t.item()) * 1e-3) / 1e6
    sampler.stop()
    sampler.join(timeout=2)
    sync_all()

    if rank == 0:
        peak, peak_src = measured_peak()
        fb0 = sets[0]
        alg = frame_algorithmic_bytes(fb0.S, fused=bool(fb0.job.n_cfused))
        key = STAGE_BYTES_KEY
        stages = {n: {"ms": ms, "algorithmic_bytes": alg[key[n]], "GBps": alg[key[n]] / (ms * 1e-3) / 1e9 if ms > 0 else None,
                      "frac": alg[key[n]] / (ms * 1e-3) / 1e9 / peak if ms > 0 else None} for n, ms in stage_ms.items()}
        tot_ms = sum(stage_ms.values())
        # the kernel the roofline object is about: the stage furthest from the roofline among those that matter (>= 10 % of the frame)
        cand = [n for n in stages if stage_ms[n] >= 0.10 * tot_ms] or list(stages)
        dom = min(cand, key=lambda n: stages[n]["frac"])
        traffic = None
        tp = os.path.join(ROOT, "profiles", "frame_traffic.json")
        if os.path.exists(tp):
            tj = json.load(open(tp))
            traffic = (tj.get(args.workload) or {}).get(dom) if isinstance(tj.get(args.workload), dict) else None
        total_alg = sum(alg[key[k]] for k in stage_ms)
        grp = lambda names: {"ms": sum(stage_ms[k] for k in stage_ms if k in names),
                             "Mpixels/s": px_per_frame / (sum(stage_ms[k] for k in stage_ms if k in names) * 1e-3) / 1e6,
                             "GBps": sum(alg[key[k]] for k in stage_ms if k in names) / (sum(stage_ms[k] for k in stage_ms if k in names) * 1e-3) / 1e9}
        split = {"recon": grp(("pred", "warp", "blend", "comp", "itx", "intra")), "postfilter": grp(("deblock", "cdef", "lr", "fg"))}
        cpu = None
        if world == 1:
            nthr, thr_info = host_threads()
            nthr = min(nthr, 32)
            cr = cpu_reps(Ss[0], nthr)
            v, dt, kind = cpu_frames(Ss[0], nthr, cr)
            cpu = {"value": v, "unit": "Mpixels/s", "cores": nthr, "kind": kind, "host": thr_info,
                   "sample": "%d whole frames of this workload, %d per thread on %d threads (frame threading), dav1d C path HAVE_ASM=0 (no nasm in image), %.1f s wall, ~%.0f s of CPU work" % (nthr * cr, cr, nthr, dt, dt * nthr)}
        line = {"metric": "Mpixels/s", "value": value, "unit": "Mpixels/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": wl["dtype"], "data": "synthetic",
                "config": {"workload": "%s: %s" % (args.workload, wl["desc"]),
                           "stream": "one dependent stream: frame n on rank n mod %d predicts from the restored pictures of frames n-1 and n-2" % world,
                           "timed_region_ms": ms_per_step * args.steps,
                           "frames_in_flight_per_gpu": n_streams, "band_rows": band_rows, "bands_per_frame": pipe.nb,
                           "cuda_graphs": "one graph launch per frame (bands, waits, puts captured once per frame set; flag values derived on the device from the frame's sequence word)" if graphs else "off",
                           "l2": "%d rotating frame sets per GPU (~%d MB) > 126 MB L2" % (nsets, nsets * ((2 + 2 + fb0.job.run_cdef + fb0.job.run_lr + fb0.job.run_fg) * Ss[0]["pic"].nbytes + Ss[0]["coefs"].nbytes) // 1000000),
                           "records": {"pred_blocks": int(len(Ss[0]["pred"])), "compound": int(len(Ss[0]["comp"]) + len(Ss[0]["comp2"])),
                                       "tx_blocks": int(sum(len(a) for a in Ss[0]["itx"].values())), "coefs": int(len(Ss[0]["coefs"])),
                                       "intra_tx_blocks": int(len(Ss[0].get("intra_tx", [])) if Ss[0].get("intra_tx") is not None else 0)},
                           "upload": "per coded transform block the coefficients 0..eob in scan order (expanded on the device inside the timed job) + block records + masks/levels",
                           "exchange": ("per band, the producer puts the restored rows that became final into the landing buffers of the ranks decoding frames n+1 and n+2 "
                                        "(cudaMemcpyAsync over NVLink peer memory, CUDA IPC) and raises their progress flag; consumers wait on the flag value of the lowest row a band reads "
                                        "(dav1d check_tile rule); %d bytes put per frame per rank, inside the timed region and inside e2e" % put_per_frame) if world > 1 else "none (one GPU: stream order is the dependency)",
                           "exchange_bytes_per_step": int(put_per_frame) * world,
                           "parity_checked": parity,
                           "roofline_kernel_rule": "stage with the lowest HBM fraction among stages >= 10 % of the frame time"},
                "parity_checked": parity,
                "roofline": {"bound": "hbm", "kernel": dom, "achieved": stages[dom]["GBps"], "peak": peak, "unit": "GB/s",
                             "frac": stages[dom]["frac"], "traffic": traffic, "peak_source": peak_src,
                             "whole_frame": {"algorithmic_bytes": total_alg, "GBps": total_alg / (ms_per_step * 1e-3) / 1e9,
                                             "frac": total_alg / (ms_per_step * 1e-3) / 1e9 / peak},
                             "stages": stages, "split": split},
                "cpu_baseline": cpu,
                "e2e": {"value": e2e_val, "unit": "Mpixels/s", "h2d_bytes_per_step": int(fb0.h2d_bytes) * world,
                        "d2h_bytes_per_step": int(fb0.d2h_bytes) * world, "frames_timed": e2e_frames},
                "gpu_launches": int(launches), "clocks": sampler.summary()}
        emit(line)
    if x is not None:
        x.close()
    if world > 1:
        dist.destroy_process_group()


def stage_times(torch, lib, fbs, nsets, reps=6):
    """average device time of each stage of the frame job (events on the launching stream)"""
    from dav1d_b200 import _lib
    j0 = fbs[0].job
    stages = []
    if j0.n_pred:
        stages.append(("pred", lambda j, bd, st: lib.b200_mc_batch(bd, C.byref(j.mc), j.d_pred, j.n_pred, st)))
    if j0.n_warp:
        stages.append(("warp", lambda j, bd, st: lib.b200_mc_warp_batch(bd, C.byref(j.mc), j.d_warp, j.n_warp, st)))
    if j0.n_blend or j0.n_blend2:
        stages.append(("blend", lambda j, bd, st: (lib.b200_mc_blend_batch(bd, C.byref(j.mc), j.d_blend, j.n_blend, st),
                                                   lib.b200_mc_blend_batch(bd, C.byref(j.mc), j.d_blend2, j.n_blend2, st))))
    if j0.n_cfused or j0.n_cfused2:
        stages.append(("comp", lambda j, bd, st: (lib.b200_mc_comp_fused_batch(bd, C.byref(j.mc), j.d_cfused, j.n_cfused, st),
                                                  lib.b200_mc_comp_fused_batch(bd, C.byref(j.mc), j.d_cfused2, j.n_cfused2, st))))
    if j0.n_comp or j0.n_comp2:
        stages.append(("comp", lambda j, bd, st: (lib.b200_mc_comp_batch(bd, C.byref(j.mc), j.d_comp, j.n_comp, st),
                                                  lib.b200_mc_comp_batch(bd, C.byref(j.mc), j.d_comp2, j.n_comp2, st))))
    if any(j0.n_itx[t] for t in range(19)):
        stages.append(("itx", lambda j, bd, st: lib.b200_itx_add_frame(bd, j.d_itx, j.n_itx, j.d_coef, j.mc.dst, j.itx_stride, 0, st)))
    if j0.n_intra:
        stages.append(("intra", lambda j, bd, st: lib.b200_intra_frame(bd, C.byref(j.intra), j.d_intra, j.n_intra, st)))
    if j0.run_lf:
        stages.append(("deblock", lambda j, bd, st: lib.b200_lf_frame(bd, C.byref(j.lf), st)))
    if j0.run_cdef:
        stages.append(("cdef", lambda j, bd, st: lib.b200_cdef_frame(bd, C.byref(j.cdef), st)))
    if j0.run_lr:
        stages.append(("lr", lambda j, bd, st: lib.b200_lr_frame(bd, C.byref(j.lr), st)))
    if j0.run_fg:   # grain templates + scaling LUT, then the blend; in the job the preparation runs on a side stream beside reconstruction
        stages.append(("fg", lambda j, bd, st: (lib.b200_fg_prep(bd, C.byref(j.fg), st), lib.b200_fg_apply(bd, C.byref(j.fg), st))))
    acc = {n: 0.0 for n, _ in stages}
    st = torch.cuda.current_stream().cuda_stream
    for r in range(reps):
        fb = fbs[r % nsets]
        j = fb.job
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(stages) + 1)]
        evs[0].record()
        for k, (_, fn) in enumerate(stages):
            fn(j, j.bitdepth_max, st)
            evs[k + 1].record()
        torch.cuda.synchronize()
        if r >= 1:
            for k, (n, _) in enumerate(stages):
                acc[n] += evs[k].elapsed_time(evs[k + 1])
    return {n: acc[n] / (reps - 1) for n in acc}


def run_ours_itx(args):
    torch, dist, world, rank, local = dist_setup()
    from dav1d_b200 import batch, get_lib
    lib = get_lib()
    n_blocks, plane_w, nsets = 1 << 20, 8192, 3
    px_per_step = n_blocks * 64
    sets, host = [], None
    for k in range(nsets):
        blocks, coefs, pic = make_itx8x8(1 + rank * 16 + k, n_blocks, plane_w)
        if k == 0:
            host = (blocks, coefs, pic)
        sets.append((torch.from_numpy(blocks.view(np.uint8)).cuda(), torch.from_numpy(coefs).cuda(),
                     torch.from_numpy(pic).cuda()))
    strides = [plane_w] * 3

    def step(i):
        b, c, p = sets[i % nsets]
        batch.itx_add_batch(255, 1, b, c, p, strides)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
    for i in range(args.warmup):
        step(i)
    sync_all()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = lib.b200_launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    ev[0].record()
    for i in range(args.steps):
        step(i)
        ev[i + 1].record()
    sync_all()
    launches = lib.b200_launch_count() - launches0
    if args.dump_outputs and rank == 0:            # the picture the last timed step wrote into
        dump_outputs(args.dump_outputs, {"picture": sets[(args.steps - 1) % nsets][2].cpu().numpy()})
    total_ms = ev[0].elapsed_time(ev[-1])
    kern_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    t = torch.tensor([total_ms], device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = float(t.item()) / args.steps
    value = world * px_per_step / (ms_per_step * 1e-3) / 1e6
    hb = torch.from_numpy(host[0].view(np.uint8)).pin_memory()
    hc = torch.from_numpy(host[1]).pin_memory()
    hp = torch.from_numpy(host[2].copy()).pin_memory()
    e2e_steps = max(3, min(args.steps, 10))
    for _ in range(2):
        batch.itx_add_batch_host(255, 1, hb, hc, hp, strides)
    sync_all()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        batch.itx_add_batch_host(255, 1, hb, hc, hp, strides)
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
    t = torch.tensor([e2e_ms], device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_val = world * px_per_step / (float(t.item()) * 1e-3) / 1e6
    sampler.stop()
    sampler.join(timeout=2)
    if rank == 0:
        import refs
        peak, peak_src = measured_peak()
        alg_bytes = n_blocks * 256
        k_ms = sum(kern_ms) / len(kern_ms)
        achieved = alg_bytes / (k_ms * 1e-3) / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "itx8x8_traffic.json")
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get("dram_bytes_per_launch")
        n = 1 << 18
        blocks, coefs, pic = make_itx8x8(1, n, 8192)
        st = (C.c_int32 * 3)(8192, 8192, 8192)
        ncores = host_threads()[0]
        lib_r = refs.ref()
        lib_r.refdrv_itx_add_batch(255, 1, blocks.ctypes.data, n, coefs.ctypes.data, pic.ctypes.data, st, 0, ncores)
        reps, tot = 0, 0.0
        while tot < 3.0 and reps < 200:
            tot += lib_r.refdrv_itx_add_batch(255, 1, blocks.ctypes.data, n, coefs.ctypes.data, pic.ctypes.data, st, 0, ncores)
            reps += 1
        cpu = {"value": reps * n * 64 / tot / 1e6, "unit": "Mpixels/s", "cores": ncores, "kind": "reference",
               "sample": "2^18 of the 2^20 blocks x %d reps, dav1d C path HAVE_ASM=0 (no nasm in image), %d threads" % (reps, ncores)}
        line = {"metric": "Mpixels/s", "value": value, "unit": "Mpixels/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u8/i16->i32", "data": "synthetic",
                "config": {"workload": "itx8x8: 2^20 inv_txfm_add DCT_DCT 8x8 8-bit blocks per GPU per step (BASELINE config 0), "
                                       "checkasm-style coefficients, 8192x8192 plane",
                           "l2": "3 rotating input sets (576 MB) > 126 MB L2", "blocks_per_step_per_gpu": n_blocks},
                "roofline": {"bound": "hbm", "kernel": "itx_add_kernel<8,8>", "achieved": achieved, "peak": peak,
                             "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": k_ms},
                "cpu_baseline": cpu,
                "e2e": {"value": e2e_val, "unit": "Mpixels/s", "h2d_bytes_per_step": int(hb.numel() + hc.numel() * 2 + hp.numel()),
                        "d2h_bytes_per_step": int(hp.numel())},
                "gpu_launches": int(launches), "clocks": sampler.summary()}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


_JSON_OUT = None


def emit(line):
    """the one JSON line, on the process's real stdout"""
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


DUMP_BYTES = 64 << 20


def dump_outputs(dirname, arrays):
    """arrays (name -> numpy) as dirname/<name>.npy in float32; above DUMP_BYTES in all, each array is cut down to the
    same fixed seeded sample of its flattened elements (sorted indices)"""
    os.makedirs(dirname, exist_ok=True)
    total = sum(a.size for a in arrays.values()) * 4
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float32)
        if total > DUMP_BYTES:
            keep = max(1, a.size * DUMP_BYTES // total)
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(dirname, name + ".npy"), a)


def main():
    # stdout carries the JSON line and nothing else: libraries that print to fd 1 (e.g. NCCL's version banner) go to stderr
    global _JSON_OUT
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path computed in its last step as DIR/<name>.npy (float32, at most 64 MB)")
    ap.add_argument("--workload", default="4k8_inter", choices=["4k8_inter", "4k8_mixed", "4k10_full", "8k10_full", "1080p8_intra", "itx8x8"] + sorted(STREAM_WORKLOADS))
    args = ap.parse_args()
    if args.workload in STREAM_WORKLOADS:
        return run_stream(args)
    if args.impl == "reference":
        run_reference(args)                  # every step is bounded (one frame per host thread); --steps / --warmup are honoured
    else:
        args.warmup = max(args.warmup, 3)
        if args.workload == "itx8x8":
            run_ours_itx(args)
        elif FRAME_WORKLOADS[args.workload].get("intra"):
            run_ours_frame(args)
        else:
            run_ours_gop(args)


if __name__ == "__main__":
    main()
