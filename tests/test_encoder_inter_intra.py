"""Intra macroblocks of inter frames (VP8R_ENC_INTRA_MBS, EncodeIntraMbsKernel).

CPU tier: oracle_encode_inter_frame2 (oracle_inter/enc_inter_oracle.c) with flags 0 equals oracle_encode_inter_frame; a
numpy restatement checks every intra / inter decision on the oracle's final unfiltered reconstruction; the oracle's
records decode, through the oracle decoder, to its closed-loop reconstruction; and the decision does what it is for on
four fixtures (a scene cut, an object entering the picture, a pan that uncovers content at one edge, a static picture).
GPU tier: the kernel against the oracle, record for record and block for block, the written stream against the
engine's reconstruction on every decode path, chains, batches, device sources, flags 0 and the refusals."""
import ctypes as C
import os
import tempfile

import numpy as np
import pytest

import helpers
from test_encoder_inter import QUANTISERS as QUANTISERS_INTER, SIZES as SIZES_INTER
from test_encoder_inter import MODE_BITS, _dq, _i420, _oracle_lib, _padded_planes, _pan_picture, _scene, _texture

INTRA_MBS, BPRED = 2, 1
UNDECIDED = 0xFFFFFFFF  # oracle intra_err of a macroblock the skip rule did not decide
IS_INTER = 1
SEARCH = 8  # the fixtures move by at most 6 pixels
FIXTURES = ("cut", "enter", "pan", "static")


def _bias(y1_ac):
    """vp8r_enc_intra_bias (vp8_b200/csrc/cuda/enc_cost.h) restated."""
    return y1_ac * y1_ac


def fixture(kind, w, h, seed=0):
    """(key picture, next picture) of one fixture, cropped I420 bytes."""
    cw, ch = (w + 1) // 2, (h + 1) // 2
    if kind == "cut":  # the next picture is an unrelated texture
        t = _texture(ch, cw, 78 + seed)
        return _scene(w, h, 0, 3 + seed), _i420(_texture(h, w, 77 + seed), 0.4 * (t - 128) + 110, 0.4 * (128 - t) + 140)
    if kind == "enter":  # a textured rectangle over the middle third of the columns
        nxt = _scene(w, h, 1, 5 + seed)
        y = np.frombuffer(nxt, np.uint8, w * h).reshape(h, w).astype(float)
        y[:, w // 3:2 * w // 3] = _texture(h, w, 55 + seed)[:, w // 3:2 * w // 3]
        return _scene(w, h, 0, 5 + seed), np.clip(y, 0, 255).astype(np.uint8).tobytes() + nxt[w * h:]
    if kind == "pan":  # 6 pixels to the left: new content at the right edge
        return _pan_picture(w, h, 0, (0, 6), seed=5 + seed), _pan_picture(w, h, 1, (0, 6), seed=5 + seed)
    img = _scene(w, h, 0, 9 + seed)
    return img, img


def _lib():
    lib = _oracle_lib()
    lib.oracle_encode_inter_frame2.restype = C.c_int
    lib.oracle_encode_inter_frame2.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int16), C.c_int,
                                               C.c_int, C.c_int, C.c_uint, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                               C.c_void_p, C.c_void_p]
    lib.oracle_frame_bytes.restype = C.c_size_t
    lib.oracle_frame_bytes.argtypes = [C.c_void_p]
    lib.oracle_write_i420.restype = C.c_size_t
    lib.oracle_write_i420.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    return lib


def _desc(mbs, payload, w, h, q, lf, key):
    from vp8_b200 import _capi
    d = _capi.FrameDesc()
    d.hdr.width, d.hdr.height, d.hdr.mb_cols, d.hdr.mb_rows = w, h, (w + 15) // 16, (h + 15) // 16
    d.hdr.key_frame, d.hdr.show_frame, d.hdr.loop_filter_level, d.hdr.q_index = key, 1, lf, q
    d.hdr.refresh_last = 1
    d.hdr.refresh_golden = d.hdr.refresh_altref = key
    for i, v in enumerate(_dq(q)):
        d.hdr.dq[0][i] = v
    d.mbs = C.cast(mbs, C.POINTER(_capi.MbInfo))
    d.payload = C.cast(payload, C.POINTER(C.c_int16))
    return d


def _decoded(lib, dec):
    buf = (C.c_uint8 * lib.oracle_frame_bytes(dec))()
    lib.oracle_write_i420(dec, buf, len(buf))
    return bytes(buf)


def oracle_key(lib, img, w, h, q, lf):
    """An oracle decoder holding the oracle's key-frame encode of img (B_PRED on) as LAST."""
    from vp8_b200 import _capi
    cols, rows = (w + 15) // 16, (h + 15) // 16
    sy, su, sv = _padded_planes(img, w, h)
    mbs = (_capi.MbInfo * (cols * rows))()
    payload = (C.c_int16 * (cols * rows * 25 * 16))()
    ry, ru, rv = np.zeros_like(sy), np.zeros_like(su), np.zeros_like(sv)
    assert lib.oracle_encode_key_frame2(C.c_void_p(sy.ctypes.data), C.c_void_p(su.ctypes.data), C.c_void_p(sv.ctypes.data), cols, rows,
                                        (C.c_int16 * 6)(*_dq(q)), lf, mbs, payload, C.c_void_p(ry.ctypes.data), C.c_void_p(ru.ctypes.data),
                                        C.c_void_p(rv.ctypes.data), 1) == 0
    dec = lib.oracle_create()
    assert lib.oracle_decode_frame(dec, C.byref(_desc(mbs, payload, w, h, q, lf, 1))) == 0
    return dec


def oracle_inter(lib, dec, img, w, h, q, lf, flags, search_range=SEARCH):
    """oracle_encode_inter_frame2 against dec's LAST: dict of records, payload, inter_err, intra_err (UNDECIDED for the
    macroblocks of the skip rule) and the unfiltered reconstruction planes (macroblock aligned), plus the padded source
    planes."""
    from vp8_b200 import _capi
    cols, rows = (w + 15) // 16, (h + 15) // 16
    sy, su, sv = _padded_planes(img, w, h)
    mbs = (_capi.MbInfo * (cols * rows))()
    payload = (C.c_int16 * (cols * rows * 25 * 16))()
    err, ierr = (C.c_uint32 * (cols * rows))(), (C.c_uint32 * (cols * rows))()
    ry, ru, rv = np.zeros_like(sy), np.zeros_like(su), np.zeros_like(sv)
    assert lib.oracle_encode_inter_frame2(dec, sy.ctypes.data, su.ctypes.data, sv.ctypes.data, cols, rows, (C.c_int16 * 6)(*_dq(q)), q, lf,
                                          search_range, flags, C.cast(mbs, C.c_void_p), C.cast(payload, C.c_void_p),
                                          C.cast(err, C.c_void_p), C.cast(ierr, C.c_void_p), ry.ctypes.data, ru.ctypes.data,
                                          rv.ctypes.data) == 0
    return dict(mbs=mbs, payload=payload, err=np.array(err, np.int64), intra_err=np.array(ierr, np.int64), ry=ry, ru=ru, rv=rv, sy=sy, cols=cols, rows=rows)


def rec_array(mbs, n):
    """Records as an (n, 8) uint32 array: flags, coef_mask, coef_offset, mv, aux[0], aux[1], reserved."""
    return np.frombuffer(C.string_at(C.addressof(mbs.contents) if hasattr(mbs, "contents") else C.addressof(mbs), 32 * n),
                         np.uint32).reshape(n, 8).copy()


def block_list(recs, payload):
    pay = np.ctypeslib.as_array(payload, (int(recs[:, 2].max() + 25) * 16,)) if len(recs) else None
    return [pay[o * 16:(o + bin(m).count("1")) * 16].tobytes() for m, o in zip(recs[:, 1], recs[:, 2])]


def intra_mask(recs):
    return (recs[:, 0] & IS_INTER) == 0


def _predict16(ry, r, c):
    """The four 16x16 predictions of macroblock (r, c) on plane ry (key-frame edge rules): {mode: 16x16 array}."""
    above = ry[16 * r - 1, 16 * c:16 * c + 16].astype(np.int64) if r else np.full(16, 127, np.int64)
    left = ry[16 * r:16 * r + 16, 16 * c - 1].astype(np.int64) if c else np.full(16, 129, np.int64)
    P = (int(ry[16 * r - 1, 16 * c - 1]) if c else 129) if r else 127
    if r and c:
        dc = (above.sum() + left.sum() + 16) >> 5
    elif r:
        dc = (above.sum() + 8) >> 4
    elif c:
        dc = (left.sum() + 8) >> 4
    else:
        dc = 128
    return {1: np.tile(above, (16, 1)), 2: np.tile(left[:, None], (1, 16)), 0: np.full((16, 16), dc, np.int64),
            3: np.clip(left[:, None] + above[None, :] - P, 0, 255)}


def best16(o, r, c):
    """(first minimum mode in V, H, DC, TM order, its error) of macroblock (r, c) on the oracle's final reconstruction."""
    src = o["sy"][16 * r:16 * r + 16, 16 * c:16 * c + 16].astype(np.int64)
    preds = _predict16(o["ry"], r, c)
    best = None
    for mode in (1, 2, 0, 3):
        e = int(((preds[mode] - src) ** 2).sum())
        if best is None or e < best[1]:
            best = (mode, e)
    return best


# --------------------------------------------------------------------------------------------- CPU tier ----
@pytest.mark.parametrize("size", SIZES_INTER, ids=lambda s: f"{s[0]}x{s[1]}")
def test_flags_zero_is_the_all_inter_pass(built, size):
    """The inter fixtures of test_encoder_inter.py (its sizes, quantisers and scene): with flags 0,
    oracle_encode_inter_frame2 codes every macroblock inter with the records and blocks of oracle_encode_inter_frame,
    its step-2 reconstruction is what the oracle decoder makes of those records (loop filter 0), and inter_err is the
    squared error of the source against that reconstruction less the decoded residual, i.e. of the prediction."""
    from test_encoder_inter import _oracle_inter
    lib = _lib()
    w, h = size
    cw, ch = (w + 1) // 2, (h + 1) // 2
    for q, _ in QUANTISERS_INTER:
        key, nxt = _scene(w, h, 0, q + w), _scene(w, h, 1, q + w)
        dec = oracle_key(lib, key, w, h, q, 0)
        try:
            mbs, payload = _oracle_inter(lib, dec, nxt, w, h, q, 0)
            o = oracle_inter(lib, dec, nxt, w, h, q, 0, 0, search_range=16)
            n = o["cols"] * o["rows"]
            a, b = rec_array(mbs, n), rec_array(o["mbs"], n)
            assert (a == b).all() and not intra_mask(b).any(), q
            assert block_list(a, payload) == block_list(b, o["payload"]), q
            assert (o["intra_err"] == UNDECIDED).all(), q
            assert lib.oracle_decode_frame(dec, C.byref(_desc(o["mbs"], o["payload"], w, h, q, 0, 0))) == 0
            assert _decoded(lib, dec) == o["ry"][:h, :w].tobytes() + o["ru"][:ch, :cw].tobytes() + o["rv"][:ch, :cw].tobytes(), q
        finally:
            lib.oracle_destroy(dec)


@pytest.mark.parametrize("bpred", [False, True], ids=["16x16", "bpred"])
@pytest.mark.parametrize("q", [0, 20, 60, 127])
@pytest.mark.parametrize("kind", FIXTURES)
def test_oracle_decisions_match_numpy(built, kind, q, bpred):
    """Every macroblock against the 16x16 errors rebuilt from the oracle's final unfiltered reconstruction (which holds
    the final pixels of every neighbour) and the oracle's inter_err and intra_err:
    - a macroblock is intra iff intra_err + bias < inter_err (strict: a tie stays inter);
    - one the skip rule passed over has inter_err <= bias and stays inter;
    - intra_err is best16, or with B_PRED a trial total strictly below best16, and a B_PRED macroblock has exactly that;
    - a 16x16 intra macroblock has the first minimum of V, H, DC, TM as its mode, and HAS_Y2."""
    lib = _lib()
    w, h, lf = 96, 64, 10
    key, nxt = fixture(kind, w, h)
    dec = oracle_key(lib, key, w, h, q, lf)
    try:
        o = oracle_inter(lib, dec, nxt, w, h, q, lf, INTRA_MBS | (BPRED if bpred else 0))
    finally:
        lib.oracle_destroy(dec)
    cols, rows = o["cols"], o["rows"]
    recs = rec_array(o["mbs"], cols * rows)
    bias = _bias(_dq(q)[1])
    n_intra = {False: 0, True: 0}  # 16x16, B_PRED
    for r in range(rows):
        for c in range(cols):
            m = r * cols + c
            mode, e16 = best16(o, r, c)
            rec = recs[m]
            is_intra = not rec[0] & IS_INTER
            ymode = (rec[0] >> 3) & 7
            inter_err, intra_err = o["err"][m], o["intra_err"][m]
            if intra_err == UNDECIDED:
                assert inter_err <= bias and not is_intra, (m, inter_err, bias)
                continue
            assert is_intra == (intra_err + bias < inter_err), (m, intra_err, bias, inter_err)
            assert intra_err == e16 or (bpred and intra_err < e16), (m, intra_err, e16)
            if is_intra:
                assert rec[3] == 0 and (rec[0] >> 1) & 3 == 0, (m, "intra record carries a vector or a reference")
                assert (ymode == 4) == (intra_err < e16), (m, ymode, intra_err, e16)
                if ymode != 4:
                    assert ymode == mode, (m, ymode, mode)
                    assert rec[0] & 0x100, m  # VP8R_MB_HAS_Y2
            n_intra[ymode == 4] += is_intra
    if kind == "cut" and q in (20, 60):
        assert n_intra[True if bpred else False] > 0, n_intra


TIE_Q = 12  # y1_ac 16, bias 256


def tie_fixture(pattern):
    """A 16x16 frame whose macroblock ties exactly: LAST is a key frame of flat 127 (which reconstructs to flat 127 at
    q 12), the next luma has mean exactly 128 and DC (128) as its best 16x16 mode.  Every vector predicts flat 127, so
    inter_err - SSE(DC) = sum(2s - 255) = 256 = y1_ac^2 = bias, with inter_err > bias: the gate, not the skip rule,
    decides, and a tie stays inter."""
    i = np.arange(16)
    y = {"halves": np.where(i[None, :] < 8, 127, 129).repeat(16, 0),
         "checker": np.where((i[:, None] + i[None, :]) % 2, 127, 129),
         "rows": np.where(i[:, None] % 2, 126, 130).repeat(16, 1)}[pattern]
    flat_chroma = bytes([128]) * 128
    return np.full(256, 127, np.uint8).tobytes() + flat_chroma, y.astype(np.uint8).tobytes() + flat_chroma


# B_PRED beats DC on "halves" and "rows", so only "checker" ties with it
TIES = [("halves", 0), ("checker", 0), ("rows", 0), ("checker", BPRED)]


@pytest.mark.parametrize("pattern,bpred", TIES)
def test_exact_ties_stay_inter(built, pattern, bpred):
    lib = _lib()
    key, nxt = tie_fixture(pattern)
    bias = _bias(_dq(TIE_Q)[1])
    dec = oracle_key(lib, key, 16, 16, TIE_Q, 0)
    try:
        assert _decoded(lib, dec)[:256] == bytes([127]) * 256
        o = oracle_inter(lib, dec, nxt, 16, 16, TIE_Q, 0, INTRA_MBS | bpred)
    finally:
        lib.oracle_destroy(dec)
    _, e16 = best16(o, 0, 0)
    assert o["err"][0] == e16 + bias == o["intra_err"][0] + bias and o["err"][0] > bias, (o["err"][0], e16, o["intra_err"][0])
    assert not intra_mask(rec_array(o["mbs"], 1)).any()


def test_oracle_records_decode_to_its_reconstruction(built):
    """The oracle's records, intra macroblocks included, decoded by the oracle decoder (loop filter 0): exactly the
    closed-loop reconstruction the oracle coded against; with a loop filter the decode of the records through the
    writer and the parser is covered on the GPU tier."""
    lib = _lib()
    for kind in FIXTURES:
        for bpred in (False, True):
            w, h, q = 72, 56, 40
            key, nxt = fixture(kind, w, h)
            dec = oracle_key(lib, key, w, h, q, 0)
            try:
                o = oracle_inter(lib, dec, nxt, w, h, q, 0, INTRA_MBS | (BPRED if bpred else 0))
                assert lib.oracle_decode_frame(dec, C.byref(_desc(o["mbs"], o["payload"], w, h, q, 0, 0))) == 0
                got = _decoded(lib, dec)
            finally:
                lib.oracle_destroy(dec)
            cw, ch = (w + 1) // 2, (h + 1) // 2
            want = o["ry"][:h, :w].tobytes() + o["ru"][:ch, :cw].tobytes() + o["rv"][:ch, :cw].tobytes()
            assert got == want, (kind, bpred)


# Fractions of intra macroblocks on 176x144 at loop-filter level 8, measured with the oracle (bias y1_ac^2):
#   cut, B_PRED: 100 % at q 20 and 60;  cut, 16x16 only: 43 % / 45 % (a random texture is no easier to predict from its
#   neighbours than from an unrelated picture; the cut frame then goes intra where 16x16 prediction wins);
#   static: 0 at every q;  pan: no interior macroblock.
@pytest.mark.parametrize("q", [20, 60])
def test_outcomes(built, q):
    lib = _lib()
    w, h, lf = 176, 144, 8
    cols, rows = w // 16, h // 16
    frac = {}
    for kind in FIXTURES:
        for bpred in (False, True):
            key, nxt = fixture(kind, w, h)
            dec = oracle_key(lib, key, w, h, q, lf)
            try:
                o = oracle_inter(lib, dec, nxt, w, h, q, lf, INTRA_MBS | (BPRED if bpred else 0))
            finally:
                lib.oracle_destroy(dec)
            intra = intra_mask(rec_array(o["mbs"], cols * rows))
            frac[kind, bpred] = intra.mean()
            if kind == "pan":
                assert not intra.reshape(rows, cols)[1:-1, 1:-1].any(), bpred
            if kind == "static":
                assert not intra.any(), bpred
    assert frac["cut", True] >= 0.9, frac
    assert frac["cut", False] >= 0.4, frac
    assert frac["enter", True] >= 0.3, frac


# --------------------------------------------------------------------------------------------- GPU tier ----
def _engine_case(eng, lib, w, h, q, lf, key, nxt, flags, check_decoders=True):
    """Key frame then one inter frame with `flags` on a fresh stream; checks device records and blocks against the
    oracle (mode bits masked on inter macroblocks), the re-parsed records against the device's, and the written
    stream against the engine's reconstruction (host parser -> oracle, the engine's host and device parse, the
    reference decoder where built).  Returns (inter frame bytes, intra fraction, reconstruction, inter frame, key frame)."""
    import vp8_b200
    n = ((w + 15) // 16) * ((h + 15) // 16)
    st = eng.open_stream()
    (kf,) = eng.encode_key_frames([st], [key], w, h, q, loop_filter_level=lf)
    kdata = kf.write_bitstream()
    kf.close()
    intra_mbs, bpred = bool(flags & INTRA_MBS), bool(flags & BPRED)
    (fr,) = eng.encode_inter_frames([st], [nxt], w, h, q, loop_filter_level=lf, search_range=SEARCH, intra_mbs=intra_mbs, bpred=bpred)
    recon = st.read_frame()
    st.close()
    data = fr.write_bitstream()
    d = fr.desc()
    got = rec_array(d.mbs, n)
    ps = vp8_b200.Parser()
    orc = helpers.Oracle()
    dec = lib.oracle_create()
    try:
        kback = ps.parse(kdata)
        assert lib.oracle_decode_frame(dec, C.byref(kback.desc())) == 0
        orc.decode(kback)
        kback.close()
        o = oracle_inter(lib, dec, nxt, w, h, q, lf, flags)
        want = rec_array(o["mbs"], n)
        inter = ~intra_mask(want)
        masked = got.copy()
        masked[inter, 0] &= ~np.uint32(MODE_BITS)
        assert (masked[:, :6] == want[:, :6]).all(), np.nonzero((masked[:, :6] != want[:, :6]).any(1))[0][:8]
        assert block_list(got, d.payload) == block_list(want, o["payload"])
        assert d.hdr.n_inter_mbs == int(inter.sum())
        back = ps.parse(data)
        db = back.desc()
        fields = [0, 1, 3, 4, 5]  # the parser stores the blocks packed: coef_offset differs
        assert (rec_array(db.mbs, n)[:, fields] == got[:, fields]).all()
        assert block_list(rec_array(db.mbs, n), db.payload) == block_list(got, d.payload)
        assert orc.decode(back) == recon
        back.close()
    finally:
        lib.oracle_destroy(dec)
        orc.close()
        ps.close()
    fr.close()
    if check_decoders:
        check_decode_paths(eng, w, h, [kdata, data], recon)
    return len(data), float((~inter).mean()), recon, data, kdata


def check_decode_paths(eng, w, h, payloads, last):
    """The engine's host parse and device parse, and the reference decoder where built, decode `payloads` to `last`."""
    import vp8_b200
    st = eng.open_stream()
    for p in payloads:
        assert st.decode(p)
    assert st.read_frame() == last, "host parse"
    st.close()
    pd = vp8_b200.Parser()
    pd.set_defer_tokens(True)
    pd.set_defer_modes(True)
    st = eng.open_stream()
    for p in payloads:
        fr = pd.parse(p, pinned=True)
        eng.reconstruct_batch([st], [fr])
        eng.sync()
        fr.close()
    assert st.read_frame() == last, "device parse"
    st.close()
    pd.close()
    if os.path.exists(helpers.REF_DECODE):
        with tempfile.TemporaryDirectory() as td:
            path = os.path.join(td, "e.ivf")
            with open(path, "wb") as fh:
                fh.write(vp8_b200.ivf_bytes(w, h, payloads))
            assert helpers.ref_decode_ivf(path)[-len(last):] == last, "reference decoder"


@pytest.mark.gpu
@pytest.mark.parametrize("bpred", [False, True], ids=["16x16", "bpred"])
@pytest.mark.parametrize("size", [(16, 16), (65, 33), (176, 144), (1280, 720), (1920, 1080)], ids=lambda s: f"{s[0]}x{s[1]}")
def test_kernel_matches_oracle_and_decoders(built, size, bpred):
    import vp8_b200
    w, h = size
    lib = _lib()
    eng = vp8_b200.Engine(0)
    sizes = {}
    try:
        for kind in FIXTURES:
            key, nxt = fixture(kind, w, h)
            for q in (0, 20, 60, 127):
                lf = 0 if q == 0 else 12
                flags = INTRA_MBS | (BPRED if bpred else 0)
                size_on, frac = _engine_case(eng, lib, w, h, q, lf, key, nxt, flags, check_decoders=w * h <= 1280 * 720 or q == 20)[:2]
                sizes[kind, q] = (size_on, frac)
                if kind == "static":
                    # at q 0 the bias is 16, below the noise of a few flat macroblocks: 15 of 8160 at 1920x1080
                    assert frac == 0 if q else frac < 0.005, (q, frac)
        if bpred and w >= 176:
            # a scene cut: nearly all intra, and smaller than the same frame coded all inter
            for q in (20, 60):
                key, nxt = fixture("cut", w, h)
                size_off = _engine_case(eng, lib, w, h, q, 12, key, nxt, 0, check_decoders=False)[0]
                assert sizes["cut", q][1] >= 0.9 and sizes["cut", q][0] < size_off, (q, sizes["cut", q], size_off)
    finally:
        eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("pattern,bpred", TIES)
def test_kernel_keeps_exact_ties_inter(built, pattern, bpred):
    """The exact ties of test_exact_ties_stay_inter on the device: records equal the oracle's, and the macroblock is
    inter."""
    import vp8_b200
    lib = _lib()
    eng = vp8_b200.Engine(0)
    try:
        key, nxt = tie_fixture(pattern)
        frac = _engine_case(eng, lib, 16, 16, TIE_Q, 0, key, nxt, INTRA_MBS | bpred)[1]
        assert frac == 0
    finally:
        eng.close()


def _levels_picture(w, h, n_levels):
    """An inter picture whose intra macroblocks form exactly n_levels dependency levels: the key picture everywhere
    except an unrelated texture over the first rows and columns that make up those levels (macroblock (r, c) is at
    level c + 2r)."""
    key = _scene(w, h, 0, 21)
    y = np.frombuffer(key, np.uint8, w * h).reshape(h, w).copy()
    tex = _texture(h, w, 91)
    cols, rows = w // 16, h // 16
    for r in range(rows):
        for c in range(cols):
            if c + 2 * r < n_levels:
                y[16 * r:16 * r + 16, 16 * c:16 * c + 16] = tex[16 * r:16 * r + 16, 16 * c:16 * c + 16]
    return key, y.tobytes() + key[w * h:]


@pytest.mark.gpu
def test_intra_levels_around_the_flat_limit(built):
    """An all-intra inter frame at 1920x1080 (far beyond FrameParser::kMaxFlatIntraLevels = 48 levels), and inter
    frames whose intra macroblocks form 47..50 levels: device records against the oracle, and every decode path."""
    import vp8_b200
    lib = _lib()
    eng = vp8_b200.Engine(0)
    try:
        key, _ = fixture("cut", 1920, 1080)
        frac = _engine_case(eng, lib, 1920, 1080, 20, 8, key, _i420(_texture(1080, 1920, 4), np.full((540, 960), 100.0),
                                                                            np.full((540, 960), 150.0)), INTRA_MBS | BPRED)[1]
        assert frac > 0.99, frac
        for n_levels in (47, 48, 49, 50):
            key, nxt = _levels_picture(640, 480, n_levels)
            data, kdata = _engine_case(eng, lib, 640, 480, 20, 8, key, nxt, INTRA_MBS | BPRED)[3:]
            ps = vp8_b200.Parser()
            ps.parse(kdata).close()
            fr = ps.parse(data)
            d = fr.desc()
            region = (np.arange(40)[None, :] + 2 * np.arange(30)[:, None] < n_levels).reshape(-1)
            assert (intra_mask(rec_array(d.mbs, 1200)) == region).all(), n_levels
            # the host parser's level table: n levels up to kMaxFlatIntraLevels (48), 0 (the wavefront fallback) above
            assert d.hdr.n_intra_levels == (n_levels if n_levels <= 48 else 0), (d.hdr.n_intra_levels, n_levels)
            fr.close()
            ps.close()
    finally:
        eng.close()


@pytest.mark.gpu
def test_chain_with_cuts(built):
    """Ten frames with a cut every third one on one stream: each inter frame's records equal the oracle's predicting
    from the oracle's decode of the stream so far, and the stream decodes to the engine's reconstructions."""
    import vp8_b200
    w, h, q, lf = 176, 144, 30, 10
    imgs = [_scene(w, h, t % 3, 60 + t // 3) for t in range(10)]
    lib = _lib()
    eng = vp8_b200.Engine(0)
    st = eng.open_stream()
    dec = lib.oracle_create()
    ps = vp8_b200.Parser()
    payloads, recons, seen = [], [], 0
    try:
        for t, img in enumerate(imgs):
            if t == 0:
                (f,) = eng.encode_key_frames([st], [img], w, h, q, loop_filter_level=lf)
            else:
                (f,) = eng.encode_inter_frames([st], [img], w, h, q, loop_filter_level=lf, search_range=SEARCH, intra_mbs=True)
                o = oracle_inter(lib, dec, img, w, h, q, lf, INTRA_MBS | BPRED)
                n = o["cols"] * o["rows"]
                got, want = rec_array(f.desc().mbs, n), rec_array(o["mbs"], n)
                got[~intra_mask(want), 0] &= ~np.uint32(MODE_BITS)
                assert (got[:, :6] == want[:, :6]).all(), t
                seen += int(intra_mask(want).sum())
            payloads.append(f.write_bitstream())
            recons.append(st.read_frame())
            f.close()
            back = ps.parse(payloads[-1])
            assert lib.oracle_decode_frame(dec, C.byref(back.desc())) == 0
            assert _decoded(lib, dec) == recons[-1], t
            back.close()
    finally:
        lib.oracle_destroy(dec)
        ps.close()
        st.close()
    try:
        assert seen > 0
        s2 = eng.open_stream()
        for t, p in enumerate(payloads):
            assert s2.decode(p)
            assert s2.read_frame() == recons[t], t
        s2.close()
    finally:
        eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("filt", ["scalar", "swar"])
def test_batch_independence(built, filt):
    """1, 7 and 130 frames per call, fixtures mixed: each frame equals the same frame encoded alone."""
    w, h, q, lf = 96, 64, 30, 12
    engines = helpers.Engines()
    eng = engines.get({"VP8R_FILTER": filt})
    try:
        for n in (1, 7, 130):
            pairs = [fixture(FIXTURES[k % 4], w, h, seed=k % 5) for k in range(n)]
            streams = [eng.open_stream() for _ in range(n)]
            for f in eng.encode_key_frames(streams, [p[0] for p in pairs], w, h, q, loop_filter_level=lf):
                f.close()
            batch = eng.encode_inter_frames(streams, [p[1] for p in pairs], w, h, q, loop_filter_level=lf, search_range=SEARCH,
                                            intra_mbs=True)
            together = [(f.write_bitstream(), s.read_frame()) for f, s in zip(batch, streams)]
            for f in batch:
                f.close()
            for s in streams:
                s.close()
            for k in sorted({0, n // 2, n - 1} | set(range(min(n, 8)))):
                st = eng.open_stream()
                eng.encode_key_frames([st], [pairs[k][0]], w, h, q, loop_filter_level=lf)[0].close()
                (f,) = eng.encode_inter_frames([st], [pairs[k][1]], w, h, q, loop_filter_level=lf, search_range=SEARCH, intra_mbs=True)
                assert (f.write_bitstream(), st.read_frame()) == together[k], (n, k)
                f.close()
                st.close()
    finally:
        engines.close()


@pytest.mark.gpu
def test_device_sources_equal_the_host_path(built):
    """vp8r_encode_inter_frames_device_ex with I420, NV12 and RGB tensors: the host path on their I420."""
    import torch
    import vp8_b200
    w, h, q = 96, 64, 30
    cw, ch = w // 2, h // 2
    eng = vp8_b200.Engine(0)
    try:
        key, nxt = fixture("cut", w, h)
        a = np.frombuffer(nxt, np.uint8)
        uv = np.stack([a[w * h:w * h + cw * ch], a[w * h + cw * ch:]], -1).reshape(-1)
        rng = np.random.default_rng(3)
        rgb = np.clip(np.repeat(a[:w * h].reshape(h, w, 1), 3, -1).astype(int) + rng.integers(-30, 31, (h, w, 3)), 0, 255).astype(np.uint8)
        sources = {"i420": a[None], "nv12": np.concatenate([a[:w * h], uv])[None], "rgb": rgb[None]}
        for layout, arr in sources.items():
            dev = torch.from_numpy(arr.copy()).cuda()
            coded = bytes(eng.convert_to_i420(dev, layout, w, h).cpu().numpy()[0])
            outs = []
            for src, lay in ((dev, layout), ([coded], "i420")):
                st = eng.open_stream()
                eng.encode_key_frames([st], [key], w, h, q, loop_filter_level=8)[0].close()
                (f,) = eng.encode_inter_frames([st], src, w, h, q, loop_filter_level=8, search_range=SEARCH, layout=lay, intra_mbs=True)
                outs.append((f.write_bitstream(), st.read_frame()))
                f.close()
                st.close()
            assert outs[0] == outs[1], layout
    finally:
        eng.close()


@pytest.mark.gpu
def test_flags_zero_is_byte_identical(built):
    """vp8r_encode_inter_frames_ex with flags 0 and vp8r_encode_inter_frames write the same records and blocks."""
    import vp8_b200
    w, h, q = 176, 144, 30
    eng = vp8_b200.Engine(0)
    lib = eng._lib
    try:
        outs = []
        for fn in ("plain", "ex"):
            key, nxt = fixture("cut", w, h)
            st = eng.open_stream()
            eng.encode_key_frames([st], [key], w, h, q, loop_filter_level=8)[0].close()
            if fn == "plain":
                (f,) = eng._encode(lib.vp8r_encode_inter_frames, lib.vp8r_encode_inter_frames_device, [st], [nxt], "i420", w, h, q, 8, 0,
                                   SEARCH)
            else:
                (f,) = eng.encode_inter_frames([st], [nxt], w, h, q, loop_filter_level=8, search_range=SEARCH)
            outs.append((f.write_bitstream(), st.read_frame(), rec_array(f.desc().mbs, 99).tobytes()))
            f.close()
            st.close()
        assert outs[0] == outs[1]
    finally:
        eng.close()


@pytest.mark.gpu
def test_refusals_leave_the_streams_working(built):
    import vp8_b200
    from vp8_b200._capi import Vp8rError
    w, h, q = 64, 48, 40
    eng = vp8_b200.Engine(0)
    try:
        key, nxt = fixture("cut", w, h)
        st = eng.open_stream()
        eng.encode_key_frames([st], [key], w, h, q)[0].close()
        for flags in (4, 0x80000000, BPRED):
            with pytest.raises(Vp8rError) as e:
                eng._encode(eng._lib.vp8r_encode_inter_frames_ex, eng._lib.vp8r_encode_inter_frames_device_ex, [st], [nxt], "i420", w, h,
                            q, 0, 0, SEARCH, flags)
            assert e.value.code == 1
        (f,) = eng.encode_inter_frames([st], [nxt], w, h, q, search_range=SEARCH, intra_mbs=True)
        got = (f.write_bitstream(), st.read_frame())
        f.close()
        st.close()
        st = eng.open_stream()
        eng.encode_key_frames([st], [key], w, h, q)[0].close()
        (f,) = eng.encode_inter_frames([st], [nxt], w, h, q, search_range=SEARCH, intra_mbs=True)
        assert (f.write_bitstream(), st.read_frame()) == got
        f.close()
        st.close()
    finally:
        eng.close()


@pytest.mark.gpu
def test_encode_ivf_with_a_cut_round_trips(built):
    import vp8_b200
    w, h = 96, 80
    imgs = [_scene(w, h, t % 3, 9 + t // 3) for t in range(7)]
    eng = vp8_b200.Engine(0)
    try:
        data = vp8_b200.encode_ivf(imgs, w, h, 36, loop_filter_level=8, engine=eng, search_range=SEARCH, intra_mbs=True)
        st = eng.open_stream()
        recons, n_intra = [], 0
        for t, img in enumerate(imgs):
            if t == 0:
                f = eng.encode_key_frames([st], [img], w, h, 36, loop_filter_level=8)[0]
            else:
                f = eng.encode_inter_frames([st], [img], w, h, 36, loop_filter_level=8, search_range=SEARCH, intra_mbs=True)[0]
                d = f.desc().hdr
                n_intra += d.mb_cols * d.mb_rows - d.n_inter_mbs
            f.close()
            recons.append(st.read_frame())
        st.close()
        assert n_intra > 0
        assert vp8_b200.decode_ivf(data, engine=eng) == recons
    finally:
        eng.close()
