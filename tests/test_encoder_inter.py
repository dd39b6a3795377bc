"""Inter-frame encoding (row f4).  CPU tier: the writer is the inverse of the parser for inter frames too (and refuses
what it cannot write), and the CPU restatement of the motion search finds a whole-pixel pan.  GPU tier: the encoder
kernel against that restatement (oracle_inter/enc_inter_oracle.c) bit for bit, the written bitstream against the reconstruction the engine holds
(host parser -> oracle, the engine's own host and device parse, the reference decoder where it has been built), the
quality of the search, batch independence, the refusals, encode_ivf and a regression pin."""
import ctypes as C
import json
import os
import subprocess
import tempfile

import numpy as np
import pytest

import helpers

SIZES = [(176, 144), (65, 33), (320, 240), (1280, 720)]
QUANTISERS = ((100, 20), (40, 12), (8, 0))  # (q_index, loop filter level), coarse to fine
N_INTER = 4
# MD5s of the bitstream and of the reconstruction per case, recorded from the encoder itself on a B200 by
# tests/golden/make_inter_encoder_goldens.py: a regression pin, not reference output
INTER_GOLDEN = os.path.join(helpers.ROOT, "tests", "golden", "enc", "encoder_inter_frames.json")
SYNTH_INTER = ("--width 176 --height 144 --frames 12 --seed 11",
               "--width 65 --height 33 --frames 10 --seed 12 --q 5 --key-interval 6",
               "--width 320 --height 192 --frames 14 --seed 13 --pct-intra 30 --lf 0")
SYNTH_FIXED = " --pct-split 0 --segmentation 0 --lf-deltas 0 --log2-parts 0"


# ---------------------------------------------------------------------------------------------- bindings ----
# The oracle decoder together with the CPU restatement of the inter-frame encoder (oracle_inter/enc_inter_oracle.c,
# built by build.sh): one library, so that the encoder predicts from that decoder's LAST frame.
ORACLE_INTER_SO = os.path.join(helpers.ROOT, "oracle_inter", "_build", "liboracle_inter.so")


def _oracle_lib():
    helpers.ensure_built()
    if not os.path.exists(ORACLE_INTER_SO):
        subprocess.check_call([os.path.join(helpers.ROOT, "build.sh")], cwd=helpers.ROOT)
    lib = C.CDLL(ORACLE_INTER_SO)
    lib.oracle_create.restype = C.c_void_p
    lib.oracle_destroy.argtypes = [C.c_void_p]
    lib.oracle_decode_frame.argtypes = [C.c_void_p, C.c_void_p]
    lib.oracle_encode_key_frame2.restype = C.c_int
    lib.oracle_encode_inter_frame.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int16),
                                              C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.oracle_encode_inter_frame.restype = C.c_int
    return lib


def _padded_planes(img, w, h):
    """Source planes padded to whole macroblocks by edge replication (what the engine encodes)."""
    cols, rows = (w + 15) // 16, (h + 15) // 16
    cw, ch = (w + 1) // 2, (h + 1) // 2
    y = np.frombuffer(img, np.uint8, w * h).reshape(h, w)
    u = np.frombuffer(img, np.uint8, cw * ch, w * h).reshape(ch, cw)
    v = np.frombuffer(img, np.uint8, cw * ch, w * h + cw * ch).reshape(ch, cw)
    pad = lambda p, ph, pw: np.ascontiguousarray(np.pad(p, ((0, ph - p.shape[0]), (0, pw - p.shape[1])), mode="edge"))
    return pad(y, rows * 16, cols * 16), pad(u, rows * 8, cols * 8), pad(v, rows * 8, cols * 8)


def _oracle_inter(lib, dec, img, w, h, q, lf, search_range=16):
    """oracle_encode_inter_frame on oracle decoder `dec`: (records, payload)."""
    from vp8_b200 import _capi
    cols, rows = (w + 15) // 16, (h + 15) // 16
    sy, su, sv = _padded_planes(img, w, h)
    dq = (C.c_int16 * 6)()
    dq_ref = _dq(q)
    for i in range(6):
        dq[i] = dq_ref[i]
    mbs = (_capi.MbInfo * (cols * rows))()
    payload = (C.c_int16 * (cols * rows * 25 * 16))()
    assert lib.oracle_encode_inter_frame(dec, sy.ctypes.data, su.ctypes.data, sv.ctypes.data, cols, rows, dq, q, lf, search_range,
                                         C.cast(mbs, C.c_void_p), C.cast(payload, C.c_void_p)) == 0
    return mbs, payload


_DC_Q = [4, 5, 6, 7, 8, 9, 10, 10, 11, 12, 13, 14, 15, 16, 17, 17, 18, 19, 20, 20, 21, 21, 22, 22, 23, 23, 24, 25, 25, 26, 27, 28, 29, 30,
         31, 32, 33, 34, 35, 36, 37, 37, 38, 39, 40, 41, 42, 43, 44, 45, 46, 46, 47, 48, 49, 50, 51, 52, 53, 54, 55, 56, 57, 58, 59, 60, 61,
         62, 63, 64, 65, 66, 67, 68, 69, 70, 71, 72, 73, 74, 75, 76, 76, 77, 78, 79, 80, 81, 82, 83, 84, 85, 86, 87, 88, 89, 91, 93, 95, 96,
         98, 100, 101, 102, 104, 106, 108, 110, 112, 114, 116, 118, 122, 124, 126, 128, 130, 132, 134, 136, 138, 140, 143, 145, 148, 151,
         154, 157]
_AC_Q = [4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26, 27, 28, 29, 30, 31, 32, 33, 34, 35, 36, 37,
         38, 39, 40, 41, 42, 43, 44, 45, 46, 47, 48, 49, 50, 51, 52, 53, 54, 55, 56, 57, 58, 60, 62, 64, 66, 68, 70, 72, 74, 76, 78, 80, 82,
         84, 86, 88, 90, 92, 94, 96, 98, 100, 102, 104, 106, 108, 110, 112, 114, 116, 119, 122, 125, 128, 131, 134, 137, 140, 143, 146, 149,
         152, 155, 158, 161, 164, 167, 170, 173, 177, 181, 185, 189, 193, 197, 201, 205, 209, 213, 217, 221, 225, 229, 234, 239, 245, 249,
         254, 259, 264, 269, 274, 279, 284]


def _dq(q):
    """Factors of q_index without deltas (RFC 6386 section 14.1), VP8R_DQ_* order."""
    return [_DC_Q[q], _AC_Q[q], 2 * _DC_Q[q], max(8, (_AC_Q[q] * 101581) >> 16), min(132, _DC_Q[q]), _AC_Q[q]]


def _texture(h, w, seed):
    """Smoothed random texture: every 16x16 block is distinctive, whole-pixel shifts are unambiguous."""
    rng = np.random.default_rng(seed)
    t = rng.integers(0, 256, (h + 2, w + 2)).astype(float)
    t = (t[:-2, :-2] + t[1:-1, :-2] + t[2:, :-2] + t[:-2, 1:-1] + 2 * t[1:-1, 1:-1] + t[2:, 1:-1] + t[:-2, 2:] + t[1:-1, 2:] + t[2:, 2:]) / 10
    return np.clip((t - 128) * 2.2 + 128, 0, 255)


def _i420(y, u, v):
    return b"".join(np.clip(p, 0, 255).astype(np.uint8).tobytes() for p in (y, u, v))


def _pan_picture(w, h, t, step, seed=5):
    """Frame t of a texture panned by `step` = (dy, dx) whole pixels per frame: frame t at (x, y) shows the texture
    at (x + t*dx, y + t*dy), so the true vector of every macroblock is (dy, dx)."""
    margin = 64
    big = _texture(h + 2 * margin, w + 2 * margin, seed)
    oy, ox = margin + t * step[0], margin + t * step[1]
    y = big[oy:oy + h, ox:ox + w]
    cw, ch = (w + 1) // 2, (h + 1) // 2
    return _i420(y, np.full((ch, cw), 120.0), np.full((ch, cw), 136.0))


def _scene(w, h, t, seed):
    """Frame t of a seeded scene: a texture under a sub-pixel global pan, a rectangle moving on its own, noise."""
    rng = np.random.default_rng(seed * 1000 + t)
    yy, xx = np.mgrid[0:h, 0:w].astype(float)
    px, py = xx + 0.75 * t, yy - 0.5 * t
    y = 128 + 55 * np.sin(px / 7.3 + seed) * np.cos(py / 9.1) + 30 * np.sin((px + 2 * py) / 4.7) + rng.integers(-3, 4, (h, w))
    rx, ry = (w // 5 + 3 * t) % max(w - w // 4, 1), (h // 4 + 2 * t) % max(h - h // 4, 1)
    y[ry:ry + h // 4, rx:rx + w // 4] = 40 + 25 * ((xx[ry:ry + h // 4, rx:rx + w // 4] // 4) % 2)
    cw, ch = (w + 1) // 2, (h + 1) // 2
    cy, cx = np.mgrid[0:ch, 0:cw].astype(float)
    u = 118 + 35 * np.sin((cx + 0.375 * t) / 6.1) + rng.integers(-2, 3, (ch, cw))
    v = 135 + 35 * np.cos((cy - 0.25 * t) / 5.3) + rng.integers(-2, 3, (ch, cw))
    return _i420(y, u, v)


def _records(desc, n_mb, mode_mask=0xFFFFFFFF):
    return [(m.flags & mode_mask, m.coef_mask, m.mv[0], m.mv[1], m.aux[0], m.aux[1]) for m in (desc.mbs[i] for i in range(n_mb))]


def _blocks(desc, n_mb):
    out = []
    for i in range(n_mb):
        m = desc.mbs[i]
        nb = bin(m.coef_mask).count("1")
        out.append(desc.payload[m.coef_offset * 16:(m.coef_offset + nb) * 16])
    return out


MODE_BITS = 7 << 3  # VP8R_MB_MODE_SHIFT


# ---------------------------------------------------------------------------------------------- CPU tier ----
@pytest.mark.parametrize("args", SYNTH_INTER, ids=["qcif", "odd", "qvga-intra30"])
def test_writer_round_trip_inter_frames(built, args):
    """Synthetic streams with intra macroblocks in inter frames, golden and altref references, sign bias and hidden
    altref frames: parse, write, parse the written frame with a second parser -> the same records (mode bits
    included) and coefficient blocks; host parser -> oracle decodes the written stream to the original's frames."""
    import vp8_b200
    _, payloads = vp8_b200.read_ivf(helpers.synth_stream(args + SYNTH_FIXED))
    pa, pb = vp8_b200.Parser(), vp8_b200.Parser()
    oa, ob = helpers.Oracle(), helpers.Oracle()
    seen_inter = seen_intra_in_inter = seen_golden = seen_hidden = 0
    try:
        for k, p in enumerate(payloads):
            a = pa.parse(p)
            written = a.write_bitstream()
            b = pb.parse(written)
            da, db = a.desc(), b.desc()
            for name in ("width", "height", "key_frame", "show_frame", "filter_type", "loop_filter_level", "sharpness_level", "q_index",
                         "refresh_last", "refresh_golden", "refresh_altref", "copy_to_golden", "copy_to_altref", "sign_bias_golden",
                         "sign_bias_altref", "n_coef_blocks", "n_inter_mbs"):
                assert getattr(da.hdr, name) == getattr(db.hdr, name), (k, name)
            assert [list(r) for r in da.hdr.dq] == [list(r) for r in db.hdr.dq], k
            n_mb = da.hdr.mb_cols * da.hdr.mb_rows
            assert _records(da, n_mb) == _records(db, n_mb), k
            assert _blocks(da, n_mb) == _blocks(db, n_mb), k
            assert oa.decode(a) == ob.decode(b), k
            if not da.hdr.key_frame:
                seen_inter += 1
                seen_intra_in_inter += da.hdr.n_inter_mbs < n_mb
                seen_golden += any((da.mbs[i].flags >> 1) & 3 in (2, 3) for i in range(n_mb))
                seen_hidden += not da.hdr.show_frame
            a.close()
            b.close()
    finally:
        oa.close()
        ob.close()
    assert seen_inter and seen_intra_in_inter and seen_golden, (seen_inter, seen_intra_in_inter, seen_golden)


def test_writer_refuses_split_and_contradicting_vectors(built):
    import vp8_b200
    from vp8_b200._capi import Vp8rError
    # a SPLIT frame
    _, payloads = vp8_b200.read_ivf(helpers.synth_stream("--width 96 --height 64 --frames 4 --seed 21 --pct-split 60" + SYNTH_FIXED.replace(
        " --pct-split 0", "")))
    ps = vp8_b200.Parser()
    refused = False
    for p in payloads:
        f = ps.parse(p)
        if f.desc().hdr.n_split_mbs:
            with pytest.raises(Vp8rError) as e:
                f.write_bitstream()
            assert e.value.code == 1  # VP8R_ERR_INVALID_ARG
            refused = True
        f.close()
    assert refused
    # a record whose vector contradicts its mode: ZERO with a non-zero vector
    _, payloads = vp8_b200.read_ivf(helpers.synth_stream("--width 96 --height 64 --frames 3 --seed 22" + SYNTH_FIXED))
    ps = vp8_b200.Parser()
    ps.parse(payloads[0]).close()
    f = ps.parse(payloads[1])
    d = f.desc()
    n_mb = d.hdr.mb_cols * d.hdr.mb_rows
    m = next(i for i in range(n_mb) if d.mbs[i].flags & 1)
    d.mbs[m].flags = (d.mbs[m].flags & ~MODE_BITS) | (2 << 3)  # MV_ZERO
    d.mbs[m].mv[0], d.mbs[m].mv[1] = 8, -16
    with pytest.raises(Vp8rError) as e:
        f.write_bitstream()
    assert e.value.code == 1
    f.close()


def test_oracle_search_finds_a_whole_pixel_pan(built):
    """A textured picture, key frame at q=8 through the oracle (encoder, then decoder), then the same texture moved by
    (3, -5) pixels: the oracle's search returns the true vector for >= 90 % of the macroblocks whose displaced block
    lies inside the frame."""
    from vp8_b200 import _capi
    lib = _oracle_lib()
    w, h, q, step = 176, 144, 8, (3, -5)
    cols, rows = w // 16, h // 16
    dq = _dq(q)
    img0 = _pan_picture(w, h, 0, step)
    sy, su, sv = _padded_planes(img0, w, h)
    mbs = (_capi.MbInfo * (cols * rows))()
    payload = (C.c_int16 * (cols * rows * 25 * 16))()
    ry, ru, rv = np.zeros_like(sy), np.zeros_like(su), np.zeros_like(sv)
    assert lib.oracle_encode_key_frame2(C.c_void_p(sy.ctypes.data), C.c_void_p(su.ctypes.data), C.c_void_p(sv.ctypes.data), cols, rows,
                                        (C.c_int16 * 6)(*dq), 0, mbs, payload, C.c_void_p(ry.ctypes.data), C.c_void_p(ru.ctypes.data),
                                        C.c_void_p(rv.ctypes.data), 0) == 0
    desc = _capi.FrameDesc()
    desc.hdr.width, desc.hdr.height, desc.hdr.mb_cols, desc.hdr.mb_rows = w, h, cols, rows
    desc.hdr.key_frame = desc.hdr.show_frame = 1
    desc.hdr.refresh_last = desc.hdr.refresh_golden = desc.hdr.refresh_altref = 1
    for i in range(6):
        desc.hdr.dq[0][i] = dq[i]
    desc.mbs = C.cast(mbs, C.POINTER(_capi.MbInfo))
    desc.payload = C.cast(payload, C.POINTER(C.c_int16))
    dec = lib.oracle_create()
    try:
        assert lib.oracle_decode_frame(dec, C.byref(desc)) == 0
        recs, _ = _oracle_inter(lib, dec, _pan_picture(w, h, 1, step), w, h, q, 0)
    finally:
        lib.oracle_destroy(dec)
    hits = total = 0
    for r in range(rows):
        for c in range(cols):
            y0, x0 = 16 * r + step[0], 16 * c + step[1]
            if y0 < 0 or x0 < 0 or y0 + 16 > h or x0 + 16 > w:
                continue
            total += 1
            hits += (recs[r * cols + c].mv[0], recs[r * cols + c].mv[1]) == (8 * step[0], 8 * step[1])
    assert total > 50 and hits >= 0.9 * total, (hits, total)


# ---------------------------------------------------------------------------------------------- GPU tier ----
def _case_key(w, h, bpred, q):
    return f"{w}x{h}-{'bpred' if bpred else '16x16'}-q{q}"


def encode_sequence(eng, w, h, q, lf, bpred, seed):
    """One key frame and N_INTER inter frames of the seeded scene on one stream: (payloads, reconstructions,
    frames, images); the frames are open ParsedFrames (the caller closes them)."""
    imgs = [_scene(w, h, t, seed) for t in range(N_INTER + 1)]
    st = eng.open_stream()
    payloads, recons, frames = [], [], []
    try:
        for t, img in enumerate(imgs):
            if t == 0:
                (f,) = eng.encode_key_frames([st], [img], w, h, q, loop_filter_level=lf, bpred=bpred)
            else:
                (f,) = eng.encode_inter_frames([st], [img], w, h, q, loop_filter_level=lf)
            payloads.append(f.write_bitstream())
            recons.append(st.read_frame())
            frames.append(f)
    finally:
        st.close()
    return payloads, recons, frames, imgs


@pytest.mark.gpu
@pytest.mark.parametrize("bpred", [False, True], ids=["16x16", "bpred"])
@pytest.mark.parametrize("size", SIZES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_inter_encoder_matches_oracle_and_decoders(built, size, bpred):
    import vp8_b200
    w, h = size
    n_mb = ((w + 15) // 16) * ((h + 15) // 16)
    with open(INTER_GOLDEN) as f:
        gold = json.load(f)
    lib = _oracle_lib()
    eng = vp8_b200.Engine(0)
    try:
        for q, lf in QUANTISERS:
            payloads, recons, frames, imgs = encode_sequence(eng, w, h, q, lf, bpred, seed=q + w)
            # (4) device records and blocks against the oracle, predicting from the oracle's decode of the stream
            # (5) host parser -> oracle decodes the written stream to the engine's reconstructions
            # (7) the re-parsed records equal the device records, mode bits included
            ps = vp8_b200.Parser()
            dec = lib.oracle_create()
            orc = helpers.Oracle()
            try:
                for t, (p, fr) in enumerate(zip(payloads, frames)):
                    d = fr.desc()
                    if t > 0:
                        recs, pay = _oracle_inter(lib, dec, imgs[t], w, h, q, lf)
                        for m in range(n_mb):
                            a, b = d.mbs[m], recs[m]
                            assert (a.flags & ~MODE_BITS, a.coef_mask, a.coef_offset, a.mv[0], a.mv[1]) == \
                                   (b.flags, b.coef_mask, b.coef_offset, b.mv[0], b.mv[1]), (q, t, m)
                            nb = bin(a.coef_mask).count("1")
                            assert d.payload[a.coef_offset * 16:(a.coef_offset + nb) * 16] == pay[b.coef_offset * 16:(b.coef_offset + nb) * 16], \
                                (q, t, m)
                    back = ps.parse(p)
                    db = back.desc()
                    assert _records(db, n_mb) == _records(d, n_mb), (q, t)
                    assert _blocks(db, n_mb) == _blocks(d, n_mb), (q, t)
                    assert orc.decode(back) == recons[t], (q, t)
                    assert lib.oracle_decode_frame(dec, C.byref(db)) == 0
                    back.close()
                    if t > 0:
                        # (9) inter frames are smaller than the sequence's key frame
                        assert len(p) < len(payloads[0]), (q, t, len(p), len(payloads[0]))
            finally:
                lib.oracle_destroy(dec)
                orc.close()
                ps.close()
            ivf = vp8_b200.ivf_bytes(w, h, payloads)
            # (6) a fresh engine stream, host parse and device parse
            st = eng.open_stream()
            for t, p in enumerate(payloads):
                assert st.decode(p)
                assert st.read_frame() == recons[t], (q, t)
            st.close()
            pd = vp8_b200.Parser()
            pd.set_defer_tokens(True)
            pd.set_defer_modes(True)
            st = eng.open_stream()
            for t, p in enumerate(payloads):
                fr = pd.parse(p, pinned=True)
                eng.reconstruct_batch([st], [fr])
                eng.sync()
                assert st.read_frame() == recons[t], (q, t, "device parse")
                fr.close()
            st.close()
            pd.close()
            # (5) the unmodified reference decoder, where it has been built
            if os.path.exists(helpers.REF_DECODE):
                with tempfile.TemporaryDirectory() as td:
                    path = os.path.join(td, "e.ivf")
                    with open(path, "wb") as fh:
                        fh.write(ivf)
                    assert helpers.ref_decode_ivf(path) == b"".join(recons), (size, q)
            # (13) regression pin
            want = gold[_case_key(w, h, bpred, q)]
            assert helpers.md5(ivf) == want["ivf_md5"], (size, q)
            assert [helpers.md5(r) for r in recons] == want["frame_md5"], (size, q)
            for f in frames:
                f.close()
    finally:
        eng.close()


@pytest.mark.gpu
def test_inter_encoder_finds_a_whole_pixel_pan(built):
    """(8) q=8, a texture panned by whole pixels: >= 90 % of the interior macroblocks get the true vector."""
    import vp8_b200
    w, h, step = 320, 240, (-2, 6)
    cols, rows = w // 16, h // 16
    eng = vp8_b200.Engine(0)
    try:
        st = eng.open_stream()
        eng.encode_key_frames([st], [_pan_picture(w, h, 0, step)], w, h, 8, bpred=False)[0].close()
        (fr,) = eng.encode_inter_frames([st], [_pan_picture(w, h, 1, step)], w, h, 8)
        d = fr.desc()
        hits = total = 0
        for r in range(1, rows - 1):
            for c in range(1, cols - 1):
                total += 1
                hits += (d.mbs[r * cols + c].mv[0], d.mbs[r * cols + c].mv[1]) == (8 * step[0], 8 * step[1])
        fr.close()
        st.close()
    finally:
        eng.close()
    assert hits >= 0.9 * total, (hits, total)


@pytest.mark.gpu
def test_inter_encoder_batch_is_independent(built):
    """(10) Eight streams in one call write the same bytes as each stream encoded alone."""
    import vp8_b200
    w, h = 208, 160
    eng = vp8_b200.Engine(0)
    try:
        keys = [_scene(w, h, 0, 40 + k) for k in range(8)]
        nexts = [_scene(w, h, 1 + k % 3, 40 + k) for k in range(8)]
        streams = [eng.open_stream() for _ in range(8)]
        for f in eng.encode_key_frames(streams, keys, w, h, 30, loop_filter_level=10):
            f.close()
        batch = eng.encode_inter_frames(streams, nexts, w, h, 30, loop_filter_level=10, search_range=12)
        together = [(f.write_bitstream(), st.read_frame()) for f, st in zip(batch, streams)]
        for f in batch:
            f.close()
        for k in range(8):
            st = eng.open_stream()
            eng.encode_key_frames([st], [keys[k]], w, h, 30, loop_filter_level=10)[0].close()
            (f,) = eng.encode_inter_frames([st], [nexts[k]], w, h, 30, loop_filter_level=10, search_range=12)
            assert (f.write_bitstream(), st.read_frame()) == together[k], k
            f.close()
            st.close()
        for st in streams:
            st.close()
    finally:
        eng.close()


@pytest.mark.gpu
def test_inter_encoder_refusals(built):
    """(11) No frame to predict from, another size, search_range 3 and 25, a stream twice in one call."""
    import vp8_b200
    from vp8_b200._capi import Vp8rError
    w, h = 64, 48
    eng = vp8_b200.Engine(0)
    try:
        img = _scene(w, h, 0, 1)
        fresh = eng.open_stream()
        with pytest.raises(Vp8rError) as e:
            eng.encode_inter_frames([fresh], [img], w, h, 40)
        assert e.value.code == 5  # VP8R_ERR_STATE
        st = eng.open_stream()
        eng.encode_key_frames([st], [img], w, h, 40)[0].close()
        other = _scene(80, 48, 1, 1)
        with pytest.raises(Vp8rError) as e:
            eng.encode_inter_frames([st], [other], 80, 48, 40)
        assert e.value.code == 5
        for rng_ in (3, 25):
            with pytest.raises(Vp8rError) as e:
                eng.encode_inter_frames([st], [img], w, h, 40, search_range=rng_)
            assert e.value.code == 1  # VP8R_ERR_INVALID_ARG
        with pytest.raises(Vp8rError) as e:
            eng.encode_inter_frames([st, st], [img, img], w, h, 40)
        assert e.value.code == 1
        # the stream is untouched by the refusals
        (f,) = eng.encode_inter_frames([st], [img], w, h, 40)
        f.close()
        st.close()
        fresh.close()
    finally:
        eng.close()


@pytest.mark.gpu
def test_encode_ivf_round_trips_through_decode_ivf(built):
    """(12) encode_ivf with a key frame every third frame: decode_ivf gives back the reconstructions the encoder
    held, frame by frame."""
    import vp8_b200
    w, h = 96, 80
    imgs = [_scene(w, h, t, 9) for t in range(7)]
    eng = vp8_b200.Engine(0)
    try:
        data = vp8_b200.encode_ivf(imgs, w, h, 36, key_interval=3, loop_filter_level=8, engine=eng)
        _, payloads = vp8_b200.read_ivf(data)
        ps = vp8_b200.Parser()
        kinds = []
        for p in payloads:
            f = ps.parse(p)
            kinds.append(f.desc().hdr.key_frame)
            f.close()
        assert kinds == [1, 0, 0, 1, 0, 0, 1]
        # the reconstructions the encoder held: the same calls on one stream
        st = eng.open_stream()
        recons = []
        for t, img in enumerate(imgs):
            if t % 3 == 0:
                f = eng.encode_key_frames([st], [img], w, h, 36, loop_filter_level=8)[0]
            else:
                f = eng.encode_inter_frames([st], [img], w, h, 36, loop_filter_level=8)[0]
            f.close()
            recons.append(st.read_frame())
        st.close()
        assert vp8_b200.decode_ivf(data, engine=eng) == recons
        with tempfile.TemporaryDirectory() as td:
            path = os.path.join(td, "x.ivf")
            assert vp8_b200.encode_ivf(imgs, w, h, 36, path=path, key_interval=3, loop_filter_level=8, engine=eng) == data
            assert open(path, "rb").read() == data
    finally:
        eng.close()
