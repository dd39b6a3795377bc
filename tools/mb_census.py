#!/usr/bin/env python3
"""Macroblock census of the bench workload, on the CPU: what InterKernel gets to do per macroblock.

  mb_census.py [--streams 2] [--frames 30] [--synth-args "..."]

Generates the streams bench.py decodes (same generator settings, seeds 7122+k), parses them with the host
parser and counts, over all inter frames: intra / whole-macroblock / SPLIT macroblocks, the whole ones by
how many axes of their vector are fractional, and for macroblocks with a residual the number of coded
blocks (= blocks the residual transform runs on; more than 8 take a second pass of the warp), the number of
blocks with AC coefficients, and the Y2 blocks.  Prints one table; needs no GPU."""
import argparse
import collections
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (SYNTH_ARGS: the workload this census describes)
import vp8_b200  # noqa: E402
from vp8_b200 import _capi  # noqa: E402

IS_INTER, HAS_Y2, MODE_SHIFT, SPLIT = 0x1, 0x100, 3, 4


def popcount(x):
    return np.bitwise_count(x.astype(np.uint32)).astype(np.int64)


def census_frame(d, c, coded_hist, ac_hist):
    n = d.hdr.mb_rows * d.hdr.mb_cols
    raw = np.ctypeslib.as_array(_capi.C.cast(d.mbs, _capi.C.POINTER(_capi.C.c_uint32)), shape=(n * 8,)).reshape(n, 8)
    flags, mask, off = raw[:, 0], raw[:, 1], raw[:, 2].astype(np.int64)
    mv = raw[:, 3]
    mvr = ((mv & 0xffff).astype(np.int64) ^ 0x8000) - 0x8000
    mvc = ((mv >> 16).astype(np.int64) ^ 0x8000) - 0x8000
    inter = (flags & IS_INTER) != 0
    split = inter & (((flags >> MODE_SHIFT) & 7) == SPLIT)
    whole = inter & ~split
    frac = ((mvr & 7) != 0).astype(int) + ((mvc & 7) != 0).astype(int)
    c["mb"] += n
    c["intra"] += int((~inter).sum())
    c["split"] += int(split.sum())
    for k, name in enumerate(["whole, whole-pel", "whole, fractional in one axis", "whole, fractional in both axes"]):
        c[name] += int((whole & (frac == k)).sum())
    res = inter & (mask != 0)
    c["inter with residual"] += int(res.sum())
    c["inter with Y2 coded"] += int((res & ((flags & HAS_Y2) != 0) & ((mask & 1) != 0)).sum())
    nb = max(1, d.hdr.n_payload_blocks)
    pay = np.ctypeslib.as_array(d.payload, shape=(nb * 16,)).reshape(nb, 16)
    coded = np.zeros(n, np.int64)
    ac = np.zeros(n, np.int64)
    for b in range(1, 25):  # blocks 0..23; bit 0 is Y2
        has = res & (((mask >> b) & 1) != 0)
        at = off + popcount(mask & ((1 << b) - 1))
        blk = pay[np.where(has, at, 0)]
        coded += has
        ac += has & np.any(blk[:, 1:] != 0, axis=1)
    for v in coded[res]:
        coded_hist[int(v)] += 1
    for v in ac[res]:
        ac_hist[min(int(v), 9)] += 1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=2)
    ap.add_argument("--frames", type=int, default=30)
    ap.add_argument("--synth-args", default=bench.SYNTH_ARGS)
    a = ap.parse_args()
    args = a.synth_args.replace("--frames 30", f"--frames {a.frames}").split()
    c, coded_hist, ac_hist = collections.Counter(), collections.Counter(), collections.Counter()
    with tempfile.TemporaryDirectory() as tmp:
        for k in range(a.streams):
            path = os.path.join(tmp, f"s{k}.ivf")
            subprocess.check_call([bench.SYNTH] + args + ["--seed", str(7122 + k), "--out", path])
            ps = vp8_b200.Parser()
            for payload in vp8_b200.read_ivf(path)[1]:
                f = ps.parse(payload)
                d = f.desc()
                if not d.hdr.key_frame:
                    c["inter frames"] += 1
                    census_frame(d, c, coded_hist, ac_hist)
                f.close()
            ps.close()
    tot, nres = c["mb"], max(1, c["inter with residual"])
    print(f"{a.streams} streams, {c['inter frames']} inter frames, {tot} macroblocks ({a.synth_args})")
    print("share of all macroblocks:")
    for k in ["intra", "whole, whole-pel", "whole, fractional in one axis", "whole, fractional in both axes", "split",
              "inter with residual", "inter with Y2 coded"]:
        print(f"  {k:32s} {100.0 * c[k] / max(1, tot):6.2f} %")
    mean = sum(k * v for k, v in coded_hist.items()) / nres
    print(f"inter macroblocks with a residual: coded blocks (transformed, Y2 apart), mean {mean:.2f}")
    for k in sorted(coded_hist):
        print(f"  {k:2d} {100.0 * coded_hist[k] / nres:6.2f} %")
    print(f"  more than 8 (second transform pass): {100.0 * sum(v for k, v in coded_hist.items() if k > 8) / nres:.2f} %")
    print("  blocks with AC coefficients (9 = 9 or more):")
    for k in sorted(ac_hist):
        print(f"  {k:2d} {100.0 * ac_hist[k] / nres:6.2f} %")


if __name__ == "__main__":
    main()
