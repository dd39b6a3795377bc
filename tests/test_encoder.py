"""Row f4 (encoder).  CPU tier: the key-frame writer is the inverse of the parser.  GPU tier: the closed-loop encoder
kernel against the pinned oracle, against the unmodified reference DECODER (what it reconstructs is what a decoder makes
of its bitstream) and against the source (quality follows the quantiser)."""
import ctypes as C
import json
import os
import tempfile

import numpy as np
import pytest

import helpers

SIZES = [(176, 144), (65, 33), (320, 240), (1280, 720)]
QUANTISERS = ((100, 20), (40, 12), (8, 0))  # (q_index, loop filter level), coarse to fine
# MD5s of the bitstream the encoder wrote and of the frame it reconstructed, per case, recorded from the encoder itself
# by tests/golden/make_encoder_goldens.py: they pin its output against regressions, they are not reference output
ENC_GOLDEN = os.path.join(helpers.ROOT, "tests", "golden", "enc", "encoder_key_frames.json")


def golden_key(w, h, bpred, q):
    return f"{w}x{h}-{'bpred' if bpred else '16x16'}-q{q}"


def _image(w, h, seed):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    y = 128 + 70 * np.sin(xx / 11.0 + seed) * np.cos(yy / 13.0) + 25 * ((xx // 24 + yy // 20) % 2) + rng.integers(-5, 6, (h, w))
    cw, ch = (w + 1) // 2, (h + 1) // 2
    cy, cx = np.mgrid[0:ch, 0:cw]
    u = 118 + 40 * np.sin(cx / 9.0) + rng.integers(-3, 4, (ch, cw))
    v = 135 + 40 * np.cos(cy / 7.0) + rng.integers(-3, 4, (ch, cw))
    planes = [np.clip(p, 0, 255).astype(np.uint8) for p in (y, u, v)]
    return b"".join(p.tobytes() for p in planes)


def _psnr(a, b, n):
    a = np.frombuffer(a, np.uint8)[:n].astype(float)
    b = np.frombuffer(b, np.uint8)[:n].astype(float)
    mse = float(np.mean((a - b) ** 2))
    return 99.0 if mse == 0 else 10 * np.log10(255.0 ** 2 / mse)


def test_writer_is_the_inverse_of_the_parser(built):
    """Key frames of the synthesiser (16x16 and B_PRED modes, skipped macroblocks, all token categories) parsed,
    written, parsed again: same macroblock records, same coefficient blocks."""
    import vp8_b200
    for args in ("--width 176 --height 144 --frames 1 --seed 3 --segmentation 0 --lf-deltas 0 --log2-parts 0",
                 "--width 65 --height 33 --frames 1 --seed 4 --segmentation 0 --lf-deltas 0 --log2-parts 0 --q 5",
                 "--width 320 --height 192 --frames 1 --seed 5 --segmentation 0 --lf-deltas 0 --log2-parts 0 --pct-skip 70 --lf 0"):
        key = vp8_b200.read_ivf(helpers.synth_stream(args))[1][0]
        a = vp8_b200.Parser().parse(key)
        written = a.write_bitstream()
        b = vp8_b200.Parser().parse(written)
        da, db = a.desc(), b.desc()
        for name in ("width", "height", "mb_cols", "mb_rows", "key_frame", "filter_type", "loop_filter_level", "sharpness_level", "q_index",
                     "n_coef_blocks"):
            assert getattr(da.hdr, name) == getattr(db.hdr, name), name
        n_mb = da.hdr.mb_cols * da.hdr.mb_rows
        for m in range(n_mb):
            x, y = da.mbs[m], db.mbs[m]
            assert (x.flags, x.coef_mask, x.aux[0], x.aux[1]) == (y.flags, y.coef_mask, y.aux[0], y.aux[1]), m
            nb = bin(x.coef_mask).count("1")
            assert da.payload[x.coef_offset * 16:(x.coef_offset + nb) * 16] == db.payload[y.coef_offset * 16:(y.coef_offset + nb) * 16], m
        a.close()
        b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("bpred", [False, True], ids=["16x16", "bpred"])
@pytest.mark.parametrize("size", SIZES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_encoder_matches_oracle_and_reference_decoder(built, size, bpred):
    import vp8_b200
    from vp8_b200 import _capi
    w, h = size
    with open(ENC_GOLDEN) as f:
        gold = json.load(f)
    eng = vp8_b200.Engine(0)
    orc = C.CDLL(helpers.ORACLE_SO)
    try:
        last_psnr = None
        for q, lf in QUANTISERS:
            img = _image(w, h, 7 + q)
            st = eng.open_stream()
            (fr,) = eng.encode_key_frames([st], [img], w, h, q, loop_filter_level=lf, bpred=bpred)
            recon = st.read_frame()
            d = fr.desc()
            cols, rows = d.hdr.mb_cols, d.hdr.mb_rows
            # (1) the oracle encoder on the same padded planes: same modes, same coefficient blocks
            cw, ch = (w + 1) // 2, (h + 1) // 2
            y = np.frombuffer(img, np.uint8, w * h).reshape(h, w)
            u = np.frombuffer(img, np.uint8, cw * ch, w * h).reshape(ch, cw)
            v = np.frombuffer(img, np.uint8, cw * ch, w * h + cw * ch).reshape(ch, cw)
            pad = lambda p, ph, pw: np.ascontiguousarray(np.pad(p, ((0, ph - p.shape[0]), (0, pw - p.shape[1])), mode="edge"))
            sy, su, sv = pad(y, rows * 16, cols * 16), pad(u, rows * 8, cols * 8), pad(v, rows * 8, cols * 8)
            dq = (C.c_int16 * 6)(*d.hdr.dq[0])
            mbs = (_capi.MbInfo * (cols * rows))()
            payload = (C.c_int16 * (cols * rows * 25 * 16))()
            ry, ru, rv = np.zeros_like(sy), np.zeros_like(su), np.zeros_like(sv)
            assert orc.oracle_encode_key_frame2(C.c_void_p(sy.ctypes.data), C.c_void_p(su.ctypes.data), C.c_void_p(sv.ctypes.data), cols, rows, dq,
                                                lf, mbs, payload, C.c_void_p(ry.ctypes.data), C.c_void_p(ru.ctypes.data),
                                                C.c_void_p(rv.ctypes.data), int(bpred)) == 0
            for m in range(cols * rows):
                a, b = d.mbs[m], mbs[m]
                assert (a.flags, a.coef_mask, a.coef_offset, a.aux[0], a.aux[1]) == (b.flags, b.coef_mask, b.coef_offset, b.aux[0], b.aux[1]), (q, m)
                nb = bin(a.coef_mask).count("1")
                assert d.payload[a.coef_offset * 16:(a.coef_offset + nb) * 16] == payload[b.coef_offset * 16:(b.coef_offset + nb) * 16], (q, m)
            # (2) the bitstream and the frame are the recorded ones (ENC_GOLDEN, a regression pin), and the oracle decodes
            # the bitstream to the frame the encoder holds; the oracle is tied to the reference decoder only through its
            # golden-vector MD5s.  Where the UNMODIFIED reference decoder has been built (from sources outside the
            # repository, oracle/Makefile) it has to decode the bitstream to that frame as well
            data = fr.write_bitstream()
            want = gold[golden_key(w, h, bpred, q)]
            assert helpers.md5(data) == want["bitstream_md5"], (size, q)
            assert helpers.md5(recon) == want["frame_md5"], (size, q)
            back = vp8_b200.Parser().parse(data)
            oracle = helpers.Oracle()
            assert oracle.decode(back) == recon, (size, q)
            oracle.close()
            if os.path.exists(helpers.REF_DECODE):
                with tempfile.TemporaryDirectory() as td:
                    path = os.path.join(td, "e.ivf")
                    vp8_b200.write_ivf(path, w, h, [data])
                    ref = helpers.ref_decode_ivf(path)
                assert ref == recon, (size, q)
            # (3) our own parser reads the records back
            db = back.desc()
            for m in range(cols * rows):
                assert (db.mbs[m].flags, db.mbs[m].coef_mask, db.mbs[m].aux[0], db.mbs[m].aux[1]) == \
                       (d.mbs[m].flags, d.mbs[m].coef_mask, d.mbs[m].aux[0], d.mbs[m].aux[1]), (q, m)
            back.close()
            # (4) finer quantisers are closer to the source
            p = _psnr(recon, img, w * h)
            assert p > 24, (size, q, p)
            if last_psnr is not None:
                assert p > last_psnr, (size, q, p, last_psnr)
            last_psnr = p
            fr.close()
            st.close()
    finally:
        eng.close()


@pytest.mark.gpu
def test_encoder_batch_and_decode_continues(built):
    """Eight streams encoded in one call; each stream then decodes inter frames on top of the encoded key frame like
    any decoder state (here: the same key frame decoded from the written bitstream gives the same picture)."""
    import vp8_b200
    eng = vp8_b200.Engine(0)
    try:
        w, h = 208, 160
        imgs = [_image(w, h, 30 + k) for k in range(8)]
        streams = [eng.open_stream() for _ in imgs]
        frames = eng.encode_key_frames(streams, imgs, w, h, 30, loop_filter_level=16, sharpness=2)
        for st, fr in zip(streams, frames):
            recon = st.read_frame()
            st2 = eng.open_stream()
            assert st2.decode(fr.write_bitstream())
            assert st2.read_frame() == recon
            st2.close()
            fr.close()
            st.close()
    finally:
        eng.close()
