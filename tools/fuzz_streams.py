#!/usr/bin/env python3
"""Fuzz the hooked decoder against stock dav1d on the CPU: randomly parameterised synthetic streams (every header option of
dav1d_b200/obu.py drawn at random: bit depth, layout, superblock size, tiles, film grain, screen content + intra block copy,
motion modes, global motion, segmentation, hidden / intra-only frames, changing frame sizes, super-resolution), decoded with
random thread counts / frames in flight through oracle/_ref/libdav1d_b200.so bound to the host-emulator build of the CUDA
sources, and through oracle/_ref (stock dav1d); every output picture must be byte-identical. Streams the stock decoder rejects
(random payloads are not always legal, e.g. 4:2:2 or intra block copy) are skipped. Every other stream goes through the stream
generator first (tests/streamgen.py: symbols chosen and range-encoded by the reference decoder itself), with a random policy for
skipped blocks / sparse coefficients / intra share — and, for 4:2:2, frames of any size, since the generator avoids the
partitions that are illegal there.
usage: tools/fuzz_streams.py [n_streams] [first_seed] [big | level1]
   big: frames up to 1000x560 instead of 420x290;  level1: small frames through oracle/_ref/libdav1d_b200_l1.so instead — dav1d's
   own reconstruction code on the B200 function tables (every Dav1dDSPContext slot incl. mc_scaled / resize / emu_edge / warp / blend),
   one emulated kernel launch per DSP call"""
import importlib.util
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import refs                      # noqa: E402
from dav1d_b200 import obu, stream   # noqa: E402
import test_stream as TS         # noqa: E402
import streamgen                 # noqa: E402


BIG = len(sys.argv) > 3 and sys.argv[3] == "big"
LEVEL1 = len(sys.argv) > 3 and sys.argv[3] == "level1"


def draw(seed):
    rng = np.random.default_rng(seed)
    inter = rng.random() < 0.65
    layout = str(rng.choice(["420", "420", "420", "444", "400", "422"]))
    use_gen = streamgen.have_generator() and rng.random() < 0.5
    small = layout == "422" and not use_gen
    w = int(rng.integers(8, 18 if small or LEVEL1 else 125 if BIG else 52)) * 8 + int(rng.choice([0, 0, 2, 6]))
    h = int(rng.integers(8, 14 if LEVEL1 else 18 if small else 70 if BIG else 36)) * 8 + int(rng.choice([0, 0, 4]))
    kw = dict(bpc=int(rng.choice([8, 10, 12])), sb128=int(rng.integers(0, 2)), log2_cols=int(rng.integers(0, 3)), log2_rows=int(rng.integers(0, 2)),
              film_grain=int(rng.integers(0, 2)), layout=layout)
    sc = int(rng.random() < 0.3)
    if inter:
        kw.update(n_frames=int(rng.integers(2, 8)), motion_modes=int(rng.integers(0, 3)), global_motion=int(rng.integers(0, 2)),
                  hidden_every=int(rng.choice([0, 0, 2, 3])), intra_only_every=int(rng.choice([0, 0, 0, 4])), segmentation=int(rng.integers(0, 2)),
                  screen_content=sc)
        u = rng.random()
        if u < 0.25 and not kw["hidden_every"]:
            # frame sizes within a factor 2 of each other (every pair of frames may meet as frame and reference)
            ws = sorted({w, max(16, (w * 3 // 4) & ~1), max(16, (w * 5 // 8) & ~1)}); hs = sorted({h, max(16, (h * 3 // 4) & ~1), max(16, (h * 5 // 8) & ~1)})
            kw["sizes"] = [(int(rng.choice(ws)), int(rng.choice(hs))) for _ in range(4)]
        elif u < 0.45:
            kw["super_res"] = 1
        return "inter", w, h, kw, use_gen
    kw.update(n_frames=int(rng.integers(1, 4)), screen_content=sc, segmentation=int(rng.integers(0, 2)))
    u = rng.random()
    if sc and u < 0.5:
        kw["intrabc"] = 1
    elif u < 0.7 or not sc and u < 0.4:
        kw["super_res"] = 1
    return "intra", w, h, kw, use_gen


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 100
    first = int(sys.argv[2]) if len(sys.argv) > 2 else 1
    refs.emu_lib()
    spec = importlib.util.spec_from_file_location("build_emu", os.path.join(ROOT, "tests", "emu", "build_emu.py"))
    m = importlib.util.module_from_spec(spec); spec.loader.exec_module(m)
    dec = stream.Level1Decoder(backend=m.build()) if LEVEL1 else stream.HookedDecoder(backend=m.build(), serialize=True)
    ok = skipped = bad = 0
    kinds = {}
    t0 = time.time()
    for seed in range(first, first + n):
        kind, w, h, kw, use_gen = draw(seed)
        build = lambda: (obu.inter_stream if kind == "inter" else obu.intra_stream)(seed, w, h, **kw)
        if use_gen:
            prng = np.random.default_rng(seed + 13)
            pol = dict(p_skip=float(prng.choice([-1, 0.3, 0.7, 0.9])), p_intra=float(prng.choice([-1, 0.02, 0.2, 0.6])),
                       p_txskip=float(prng.choice([-1, 0.5, 0.8])), eob_draws=int(prng.choice([1, 2, 6])))
            try:
                tus = streamgen.generate(build, seed=seed, check=False, apply_grain=1, layout422=kw["layout"] == "422", tries=6, **pol)[0]
            except RuntimeError:
                skipped += 1
                continue
        else:
            tus = build()
        r0, i0, o0 = TS._ref_decode(tus, apply_grain=1)
        if r0 <= 0:
            skipped += 1
            continue
        rng = np.random.default_rng(seed + 7)
        thr = int(rng.choice([1, 2, 3, 4, 8, 16])); mfd = int(rng.choice([1, 2, 4, 8]))
        if LEVEL1:
            r1, i1, o1 = dec.decode(tus, apply_grain=1)
            st = dict(ibc=0, scaled="sizes" in kw or ("super_res" in kw and kind == "inter"), interintra=0, warp=0, blend=0, palette_bytes=0)
        else:
            r1, i1, o1 = dec.decode(tus, apply_grain=1, n_threads=thr, max_frame_delay=mfd)
            st = dec.stats(reset=True)
        if r1 == r0 and np.array_equal(i0, i1) and np.array_equal(o0, o1):
            ok += 1
            for k in ("ibc", "scaled", "interintra", "warp", "blend", "palette_bytes"):
                kinds[k] = kinds.get(k, 0) + int(st[k] > 0)
            for k in ("super_res", "sizes"):
                kinds[k] = kinds.get(k, 0) + int(k in kw)
            kinds["generated"] = kinds.get("generated", 0) + int(use_gen)
            kinds[kw["layout"]] = kinds.get(kw["layout"], 0) + 1
        else:
            bad += 1
            print("MISMATCH seed %d: %s %dx%d %r threads %d delay %d -> stock %d frames, hooked %d" % (seed, kind, w, h, kw, thr, mfd, r0, r1), flush=True)
    if LEVEL1:
        print("level 1: %d emulated kernel launches behind the DSP tables; slots (left on C, replaced) = %r" % (int(refs.emu_lib().b200_launch_count()), dec.c_slots_left()))
    print("fuzz: %d streams identical, %d rejected by stock dav1d (skipped), %d MISMATCHES in %.0f s; streams with: %s"
          % (ok, skipped, bad, time.time() - t0, ", ".join("%s %d" % kv for kv in sorted(kinds.items()))))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
