#!/usr/bin/env python3
"""Records the golden MD5s of the key-frame encoder test (tests/test_encoder.py).

For every case of test_encoder_matches_oracle_and_reference_decoder (picture size x 16x16 / B_PRED modes x
quantiser) the encoder runs on cuda:0 on the test's seeded picture; the MD5 of the bitstream it writes and
of the frame it reconstructs go to tests/golden/enc/encoder_key_frames.json.  These are the encoder's own
output: the test uses them to hold later builds to it (a regression pin), not as reference output.

Before a case is recorded, the host parser + oracle have to decode its bitstream to the reconstructed frame,
and so does the unmodified reference decoder when it has been built (oracle/_ref/decode, oracle/Makefile).
The committed file was recorded without the reference decoder.

Needs a B200 and a built tree (__graft_entry__.build()):
    python tests/golden/make_encoder_goldens.py [--out PATH]
"""
import argparse
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import helpers  # noqa: E402
import test_encoder as te  # noqa: E402
import vp8_b200  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=te.ENC_GOLDEN)
    args = ap.parse_args()
    have_ref = os.path.exists(helpers.REF_DECODE)
    out = {}
    eng = vp8_b200.Engine(0)
    orc = helpers.Oracle()
    try:
        for w, h in te.SIZES:
            for bpred in (False, True):
                for q, lf in te.QUANTISERS:
                    key = te.golden_key(w, h, bpred, q)
                    st = eng.open_stream()
                    (fr,) = eng.encode_key_frames([st], [te._image(w, h, 7 + q)], w, h, q, loop_filter_level=lf, bpred=bpred)
                    data, recon = fr.write_bitstream(), st.read_frame()
                    back = vp8_b200.Parser().parse(data)
                    if orc.decode(back) != recon:
                        raise SystemExit(f"{key}: the oracle decodes the bitstream to another frame")
                    back.close()
                    if have_ref:
                        with tempfile.TemporaryDirectory() as td:
                            path = os.path.join(td, "e.ivf")
                            vp8_b200.write_ivf(path, w, h, [data])
                            if helpers.ref_decode_ivf(path) != recon:
                                raise SystemExit(f"{key}: the reference decoder decodes the bitstream to another frame")
                    out[key] = {"bitstream_md5": helpers.md5(data), "frame_md5": helpers.md5(recon)}
                    fr.close()
                    st.close()
    finally:
        orc.close()
        eng.close()
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print(len(out), "cases ->", args.out, "(checked by the oracle%s)" % (" and the reference decoder" if have_ref else ""))


if __name__ == "__main__":
    sys.exit(main())
