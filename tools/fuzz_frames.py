#!/usr/bin/env python3
"""Fuzz the frame job against the oracle on the CPU: random synthetic frames (dav1d_b200/synth.py: bit depth, chroma layout, frame
size, compound / skip / intra / OBMC / warp / inter-intra rates, film grain; intra-only frames with intra block copy) through the
host-emulator build of the CUDA sources — whole-frame job, compact coefficient upload, fused compound prediction, band-sliced
execution with random band heights (intra-only frames too, filters off) — compared with oracle/*.c stage by stage (tests/test_frame.py::check_frame).
usage: tools/fuzz_frames.py [n_frames] [first_seed]"""
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import refs                                   # noqa: E402
from dav1d_b200 import frame, synth           # noqa: E402
import test_frame as TF                       # noqa: E402
import test_intra as TI                       # noqa: E402


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 60
    first = int(sys.argv[2]) if len(sys.argv) > 2 else 1
    lib, bad, kinds, t0 = refs.emu_lib(), 0, {}, time.time()
    for seed in range(first, first + n):
        rng = np.random.default_rng(seed)
        bpc = int(rng.choice([8, 10, 12]))
        ssh, ssv = [(1, 1), (1, 1), (0, 0), (1, 0)][int(rng.integers(0, 4))]
        W, H = int(rng.integers(9, 56)) * 8, int(rng.integers(9, 44)) * 8
        try:
            if rng.random() < 0.25:
                S = synth.make_intra_frame(rng, bpc, W, H, ssh, ssv, p_ibc=float(rng.choice([0, 0.3])))
                exp = TI.oracle_intra(S)
                got = TI.run_lib(lib, frame.NumpyAlloc(), S, order=str(rng.choice(["intra_tx", "intra_tx_decode_order"])), compact=bool(rng.integers(0, 2)))
                ok, where = TI.planes_equal(S, exp, got)
                assert ok, where
                # band by band (intra block copy reads the unfiltered picture: the filters are off here, as in such frames)
                fb = frame.FrameBuffers(S, lib=lib, alloc=frame.NumpyAlloc(), run_lf=False, run_cdef=False, run_lr=False,
                                        band_rows=64 * int(rng.integers(1, 4)), compact=bool(rng.integers(0, 2)))
                fb.run_bands()
                ok, where = TI.planes_equal(S, exp, fb.output("p0"))
                assert ok, ("bands", where)
                kind = "intra"
            else:
                mixed = rng.random() < 0.5
                kw = dict(p_compound=float(rng.choice([0, 0.3, 0.7])), p_skip=float(rng.choice([0, 0.25, 0.8])), film_grain=bool(rng.integers(0, 2)))
                if mixed:
                    kw.update(p_intra=float(rng.choice([0, 0.1, 0.4])), p_obmc=float(rng.choice([0, 0.2])), p_warp=float(rng.choice([0, 0.2])),
                              p_ii=float(rng.choice([0, 0.2])))
                S = synth.make_inter_frame(rng, bpc, W, H, ssh, ssv, **kw)
                exp = TF.oracle_frame(S)
                whole = -(-H // 64) * 64
                variants = [dict(), dict(compact=True), dict(fused=True), dict(band_rows=whole, compact=True),
                            dict(band_rows=64 * int(rng.integers(1, 4)), compact=bool(rng.integers(0, 2)), fused=bool(rng.integers(0, 2)))]
                for v in variants:
                    fb = frame.FrameBuffers(S, lib=lib, alloc=frame.NumpyAlloc(), **v)
                    fb.run_bands() if v.get("band_rows") else fb.run()
                    TF.check_frame(S, fb, exp)
                kind = "mixed" if mixed else "inter"
            kinds[kind] = kinds.get(kind, 0) + 1
        except AssertionError as e:
            bad += 1
            print("MISMATCH seed %d: bpc %d %dx%d ss %d%d: %s" % (seed, bpc, W, H, ssh, ssv, str(e)[:200]), flush=True)
    print("fuzz_frames: %d frames, %d MISMATCHES in %.0f s (%s)" % (n, bad, time.time() - t0, ", ".join("%s %d" % kv for kv in sorted(kinds.items()))))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
