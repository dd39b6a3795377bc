#!/usr/bin/env python3
"""Records the golden MD5s of the inter-frame encoder test (tests/test_encoder_inter.py).

For every case of test_inter_encoder_matches_oracle_and_decoders (picture size x 16x16 / B_PRED key frame x
quantiser) the encoder runs on cuda:0 on the test's seeded scene, one key frame and four inter frames; the MD5 of
the IVF it writes and of each frame it reconstructs go to tests/golden/enc/encoder_inter_frames.json.  These are
the encoder's own output: the test uses them to hold later builds to it (a regression pin), not as reference output.

Before a case is recorded, every inter frame's records and coefficient blocks have to equal
oracle_encode_inter_frame's (oracle_inter/enc_inter_oracle.c), host parser + oracle have to decode the IVF to the
reconstructions, and so does the unmodified reference decoder when it has been built (oracle/_ref/decode,
oracle/Makefile).

Needs a B200 and a built tree (__graft_entry__.build()):
    python tests/golden/make_inter_encoder_goldens.py [--out PATH]
"""
import argparse
import ctypes as C
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import helpers  # noqa: E402
import test_encoder_inter as ti  # noqa: E402
import vp8_b200  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=ti.INTER_GOLDEN)
    args = ap.parse_args()
    have_ref = os.path.exists(helpers.REF_DECODE)
    lib = ti._oracle_lib()
    out = {}
    eng = vp8_b200.Engine(0)
    try:
        for w, h in ti.SIZES:
            n_mb = ((w + 15) // 16) * ((h + 15) // 16)
            for bpred in (False, True):
                for q, lf in ti.QUANTISERS:
                    key = ti._case_key(w, h, bpred, q)
                    payloads, recons, frames, imgs = ti.encode_sequence(eng, w, h, q, lf, bpred, seed=q + w)
                    ps, dec = vp8_b200.Parser(), lib.oracle_create()
                    try:
                        for t, p in enumerate(payloads):
                            d = frames[t].desc()
                            if t > 0:
                                recs, pay = ti._oracle_inter(lib, dec, imgs[t], w, h, q, lf)
                                for m in range(n_mb):
                                    a, b = d.mbs[m], recs[m]
                                    nb = bin(a.coef_mask).count("1")
                                    if (a.flags & ~ti.MODE_BITS, a.coef_mask, a.mv[0], a.mv[1]) != (b.flags, b.coef_mask, b.mv[0], b.mv[1]) or \
                                            d.payload[a.coef_offset * 16:(a.coef_offset + nb) * 16] != pay[b.coef_offset * 16:(b.coef_offset + nb) * 16]:
                                        raise SystemExit(f"{key}: frame {t} macroblock {m} differs from the oracle")
                            back = ps.parse(p)
                            if lib.oracle_decode_frame(dec, C.byref(back.desc())) != 0:
                                raise SystemExit(f"{key}: the oracle refuses frame {t}")
                            back.close()
                    finally:
                        lib.oracle_destroy(dec)
                        ps.close()
                    ivf = vp8_b200.ivf_bytes(w, h, payloads)
                    if helpers.oracle_decode_ivf(ivf) != recons:
                        raise SystemExit(f"{key}: the oracle decodes the stream to other frames")
                    if have_ref:
                        with tempfile.TemporaryDirectory() as td:
                            path = os.path.join(td, "e.ivf")
                            with open(path, "wb") as fh:
                                fh.write(ivf)
                            if helpers.ref_decode_ivf(path) != b"".join(recons):
                                raise SystemExit(f"{key}: the reference decoder decodes the stream to other frames")
                    out[key] = {"ivf_md5": helpers.md5(ivf), "frame_md5": [helpers.md5(r) for r in recons],
                                "bytes": [len(p) for p in payloads]}
                    for f in frames:
                        f.close()
    finally:
        eng.close()
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print(len(out), "cases ->", args.out, "(checked by the oracle%s)" % (" and the reference decoder" if have_ref else ""))


if __name__ == "__main__":
    sys.exit(main())
