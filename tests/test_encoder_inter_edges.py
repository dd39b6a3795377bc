"""The inter-frame encoder at the edges of its input space, and inter frames written into decoded streams.

CPU tier: a numpy restatement of the full-pel search checks the oracle's (oracle_inter/enc_inter_oracle.c) at both ends
of the search range, on flat, striped (equal costs, so the tie rule decides) and far-panned content; the writer codes
inter frames against the probability context of a parser that has parsed a real stream (vp80-02-inter-14xx), and a
vector coded NEW against a clamped predictor survives the round trip.

GPU tier, every comparison exact against the oracle (records, blocks) and through every decoder (host parser ->
oracle, the engine's host parse, its device parse, the reference decoder where it has been built): vectors at the
edge of the search window for R = 4, 5, 23, 24 on frames of one to 99 macroblocks, quantiser / filter / content
extremes, ties, chains of ten inter frames with large vectors, and inter frames encoded on top of decoded streams.
Every case asserts that it reached the edge it is named for."""
import ctypes as C
import os
import tempfile
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import helpers
from test_encoder_inter import MODE_BITS, SYNTH_FIXED, _blocks, _dq, _i420, _oracle_inter, _oracle_lib, _padded_planes, _records

DIRS = [(-1, -1), (-1, 0), (-1, 1), (0, -1), (0, 1), (1, -1), (1, 0), (1, 1)]  # (dy, dx) of the eight pans
IS_INTER, REF_LAST, MV_NEAREST, MV_NEAR, MV_ZERO, MV_NEW = 1, 1 << 1, 0, 1, 2, 3
# kProbMvRef (RFC 6386 section 18.3): row cnt[i] gives the probability of mode-tree node i
PROB_MV_REF = [[7, 1, 1, 143], [14, 18, 14, 107], [135, 64, 57, 68], [60, 56, 128, 65], [159, 134, 128, 34], [234, 188, 128, 28]]
# md5 of the context-free bytes of the synthetic inter frames below (CONTEXT_SYNTH), written by the writer as it was
# before it took a context: vp8r_frame_write_bitstream and write_bitstream(context=None) must not change them
CONTEXT_FREE_MD5 = {(176, 144): "055960f3cc3790b849939f01076be61e", (96, 96): "a5a65b69f7d45fd0492f57ed3190be83",
                    (200, 200): "ff0f449a7059a44965f0ad787c56529a"}


def _lib():
    lib = _oracle_lib()
    lib.oracle_search_full_pel.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int16)]
    lib.oracle_search_full_pel.restype = C.c_int
    lib.oracle_frame_bytes.argtypes = [C.c_void_p]
    lib.oracle_frame_bytes.restype = C.c_size_t
    lib.oracle_write_i420.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    lib.oracle_write_i420.restype = C.c_size_t
    lib.oracle_decode_frame.restype = C.c_int
    return lib


def _oracle_image(lib, dec):
    """The cropped I420 image of the oracle decoder's latest frame."""
    n = lib.oracle_frame_bytes(dec)
    buf = (C.c_uint8 * n)()
    lib.oracle_write_i420(dec, buf, n)
    return bytes(buf)


# ------------------------------------------------------------------------------------------------ content ----
def _analytic(h, w, oy, ox, seed=0):
    """A smooth texture defined everywhere, sampled at (y + oy, x + ox): sub-pixel pans of it are exact."""
    yy, xx = np.mgrid[0:h, 0:w].astype(float)
    y, x = yy + oy, xx + ox
    return (128 + 48 * np.sin(x / 5.3 + y / 17.0 + seed) + 38 * np.cos(y / 4.1 - x / 23.0 + 0.5 * seed)
            + 28 * np.sin((x + 1.6 * y) / 3.3 + 2.0 * seed))


def _far_pan(w, h, t, R, d, seed=0):
    """Frame t of the texture panned by R + 0.75 px per frame in direction d = (dy, dx): the true vector of every
    macroblock, (R + 0.75) * d, lies outside the full-pel window, so the search stops at its edge and the sub-pel
    refinement steps out to +-(4R + 3) quarter pels."""
    s = t * (R + 0.75)
    cw, ch = (w + 1) // 2, (h + 1) // 2
    y = _analytic(h, w, s * d[0], s * d[1], seed)
    u = 128 + 0.5 * (_analytic(ch, cw, s * d[0] / 2, s * d[1] / 2, seed + 1) - 128)
    v = 128 + 0.5 * (_analytic(ch, cw, s * d[0] / 2, s * d[1] / 2, seed + 2) - 128)
    return _i420(y, u, v)


def _flat(w, h, level):
    cw, ch = (w + 1) // 2, (h + 1) // 2
    return _i420(np.full((h, w), float(level)), np.full((ch, cw), 128.0), np.full((ch, cw), 128.0))


def _stripes(w, h, shift):
    """Vertical stripes of period 8 (four dark, four bright columns), moved right by `shift` px: every candidate
    offset that is a multiple of 8 away from the true one costs the same SAD, and dy does not change it."""
    xx = np.arange(w) - shift
    y = np.tile(np.where((xx // 4) % 2 == 0, 40.0, 210.0), (h, 1))
    cw, ch = (w + 1) // 2, (h + 1) // 2
    return _i420(y, np.full((ch, cw), 100.0), np.full((ch, cw), 150.0))


def _checkerboard(w, h, cell, phase):
    yy, xx = np.mgrid[0:h, 0:w]
    y = np.where(((yy // cell) + (xx // cell) + phase) % 2 == 0, 0.0, 255.0)
    cw, ch = (w + 1) // 2, (h + 1) // 2
    cy, cx = np.mgrid[0:ch, 0:cw]
    u = np.where(((cy // cell) + (cx // cell) + phase) % 2 == 0, 255.0, 0.0)
    return _i420(y, u, 255.0 - u)


def _negative(img):
    return bytes(255 - b for b in img)


# ---------------------------------------------------------------------------- neighbour vectors, restated ----
def _near_mvs(ctx, r, c, cols, rows):
    """RFC 6386 section 18.3 for a macroblock predicting from LAST among LAST-only neighbours (sign biases 0).
    ctx[(r, c)] = (mode, (mvr, mvc)) of the macroblocks coded so far.  Returns (best, nearest, near, cnt, raw):
    best / nearest / near clamped to 16 px beyond the frame as the decoder clamps them, raw the same before the clamp."""
    cnt, mv, ptr = [0, 0, 0, 0], [(0, 0)] * 4, 0
    above, left, aboveleft = ctx.get((r - 1, c)), ctx.get((r, c - 1)), ctx.get((r - 1, c - 1))
    if above:
        if above[1] != (0, 0):
            ptr += 1
            mv[ptr] = above[1]
        cnt[ptr] += 2
    for nb, wgt in ((left, 2), (aboveleft, 1)):
        if not nb:
            continue
        if nb[1] != (0, 0):
            if mv[ptr] != nb[1]:
                ptr += 1
                mv[ptr] = nb[1]
            cnt[ptr] += wgt
        else:
            cnt[0] += wgt
    if cnt[3] and mv[ptr] == mv[1]:
        cnt[1] += 1
    cnt[3] = 0  # no SPLIT neighbours
    if cnt[2] > cnt[1]:
        cnt[1], cnt[2] = cnt[2], cnt[1]
        mv[1], mv[2] = mv[2], mv[1]
    if cnt[1] >= cnt[0]:
        mv[0] = mv[1]
    top, bottom, lft, rgt = -r * 128, (rows - 1 - r) * 128, -c * 128, (cols - 1 - c) * 128
    clamp = lambda v: (min(max(v[0], top - 128), bottom + 128), min(max(v[1], lft - 128), rgt + 128))
    return clamp(mv[0]), clamp(mv[1]), clamp(mv[2]), cnt, (mv[0], mv[1], mv[2])


def _assign_modes(vectors, cols, rows):
    """The encoder's mode choice restated: the cheapest mode consistent with each vector under the mode tree's
    probabilities.  Returns per macroblock (mode, best, best_was_clamped, nearest_or_near_was_clamped)."""
    ctx, out = {}, []
    for r in range(rows):
        for c in range(cols):
            v = vectors[r * cols + c]
            best, nearest, near, cnt, raw = _near_mvs(ctx, r, c, cols, rows)
            p = [PROB_MV_REF[cnt[i]][i] for i in range(4)]
            w_zero, w_nearest, w_near = p[0] << 24, (256 - p[0]) * p[1] << 16, (256 - p[0]) * (256 - p[1]) * p[2] << 8
            mode, wbest = MV_NEW, 0
            if v == nearest and w_nearest > wbest:
                mode, wbest = MV_NEAREST, w_nearest
            if v == near and w_near > wbest:
                mode, wbest = MV_NEAR, w_near
            if v == (0, 0) and w_zero > wbest:
                mode, wbest = MV_ZERO, w_zero
            ctx[(r, c)] = (mode, v)
            out.append((mode, best, best != raw[0], nearest != raw[1] or near != raw[2]))
    return out


# --------------------------------------------------------------------------------------------- CPU tier ----
def _oracle_key(lib, img, w, h, q):
    """An oracle decoder holding the oracle's key-frame encode of img (quantiser q, no loop filter) as LAST."""
    from vp8_b200 import _capi
    cols, rows = (w + 15) // 16, (h + 15) // 16
    sy, su, sv = _padded_planes(img, w, h)
    mbs = (_capi.MbInfo * (cols * rows))()
    payload = (C.c_int16 * (cols * rows * 25 * 16))()
    ry, ru, rv = np.zeros_like(sy), np.zeros_like(su), np.zeros_like(sv)
    dq = _dq(q)
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
    assert lib.oracle_decode_frame(dec, C.byref(desc)) == 0
    return dec


def _numpy_full_pel(last, src, R, y1_ac):
    """The full-pel search restated: for every macroblock the argmin over |dy|, |dx| <= R of SAD against the
    edge-clamped LAST plane + lambda * bits(v), the lowest index (dy + R) * (2R + 1) + dx + R on a tie."""
    lam = 1 + (y1_ac >> 4)
    bits = lambda q: 2 * abs(q).bit_length() + 1 if q else 0
    offs = range(-R, R + 1)
    pen = np.array([[lam * (bits(4 * dy) + bits(4 * dx)) for dx in offs] for dy in offs], np.int64)
    pad = np.pad(last.astype(np.int64), R, mode="edge")
    rows, cols = last.shape[0] // 16, last.shape[1] // 16
    out, ties = [], 0
    for r in range(rows):
        for c in range(cols):
            blk = src[16 * r:16 * r + 16, 16 * c:16 * c + 16].astype(np.int64)
            win = np.lib.stride_tricks.sliding_window_view(pad[16 * r:16 * r + 16 + 2 * R, 16 * c:16 * c + 16 + 2 * R], (16, 16))
            cost = np.abs(win - blk).sum(axis=(2, 3)) + pen
            i = int(np.argmin(cost))  # first minimum in raster order = lowest index
            ties += int((cost == cost.flat[i]).sum()) > 1
            out.append((i // (2 * R + 1) - R, i % (2 * R + 1) - R))
    return out, ties


@pytest.mark.parametrize("R", [4, 24])
@pytest.mark.parametrize("content", ["flat", "stripes", "far-pan"])
def test_oracle_full_pel_search_matches_numpy(built, content, R):
    """The oracle's full-pel stage (the one the kernel restates) against the numpy argmin, every macroblock of a
    64x48 frame whose LAST is the oracle's key-frame encode at q = 20."""
    lib = _lib()
    w, h, q = 64, 48, 20
    if content == "flat":
        imgs = (_flat(w, h, 90), _flat(w, h, 97))
    elif content == "stripes":
        imgs = (_stripes(w, h, 0), _stripes(w, h, 4))
    else:
        imgs = (_analytic(h, w, 0, 0), _analytic(h, w, R - 1, -R))
        imgs = tuple(_i420(y, np.full((h // 2, w // 2), 128.0), np.full((h // 2, w // 2), 128.0)) for y in imgs)
    dec = _oracle_key(lib, imgs[0], w, h, q)
    try:
        last = np.frombuffer(_oracle_image(lib, dec), np.uint8, w * h).reshape(h, w)
        sy, _, _ = _padded_planes(imgs[1], w, h)
        mv = (C.c_int16 * (2 * (w // 16) * (h // 16)))()
        assert lib.oracle_search_full_pel(dec, C.c_void_p(sy.ctypes.data), w // 16, h // 16, _dq(q)[1], R, mv) == 0
    finally:
        lib.oracle_destroy(dec)
    got = [(mv[2 * m], mv[2 * m + 1]) for m in range(len(mv) // 2)]
    want, ties = _numpy_full_pel(last, sy, R, _dq(q)[1])
    assert got == want
    # the edge each content is for
    if content == "flat":
        assert set(want) == {(0, 0)}
    elif content == "stripes":
        # the interior macroblocks' minimum is shared by several candidates (at the frame's edges the clamp breaks
        # the symmetry), and the lowest index took it: -4 before +4
        assert ties >= len(want) // 2 and (0, -4) in want, (ties, want)
    else:
        assert any(abs(dy) == R or abs(dx) == R for dy, dx in want), want


# The writer against a decoding parser's context: (vector, frames of its prefix) and a synthetic stream of its size
CONTEXT_VECTORS = [("vp80-02-inter-1402", 3), ("vp80-02-inter-1412", 4), ("vp80-02-inter-1418", 5), ("vp80-02-inter-1424", 3)]
CONTEXT_SYNTH = {(176, 144): "--width 176 --height 144 --frames 6 --seed 31",
                 (96, 96): "--width 96 --height 96 --frames 6 --seed 32 --pct-intra 20",
                 (200, 200): "--width 200 --height 200 --frames 6 --seed 33 --hidden-altref 1"}


def _vector_payloads(name):
    import vp8_b200
    return vp8_b200.read_ivf(os.path.join(helpers.VEC_DIR, name + ".ivf"))[1]


def _parser_after(payloads):
    import vp8_b200
    ps = vp8_b200.Parser()
    for p in payloads:
        ps.parse(p).close()
    return ps


def _synthetic_inter_frames(w, h):
    """The inter frames of CONTEXT_SYNTH's stream of this size as parsed (writable: no SPLIT, segmentation or
    loop-filter deltas), with their context-free bytes."""
    import vp8_b200
    _, payloads = vp8_b200.read_ivf(helpers.synth_stream(CONTEXT_SYNTH[(w, h)] + SYNTH_FIXED))
    ps, out = vp8_b200.Parser(), []
    for p in payloads:
        f = ps.parse(p)
        if f.desc().hdr.key_frame:
            f.close()
            continue
        out.append(f)
    return out


def _header_fields(d):
    return tuple(getattr(d.hdr, n) for n in ("width", "height", "key_frame", "show_frame", "filter_type", "loop_filter_level",
                                              "sharpness_level", "q_index", "refresh_last", "refresh_golden", "refresh_altref",
                                              "copy_to_golden", "copy_to_altref", "sign_bias_golden", "sign_bias_altref",
                                              "n_coef_blocks", "n_inter_mbs"))


@pytest.mark.parametrize("vector,k", CONTEXT_VECTORS, ids=[v[0][-4:] for v in CONTEXT_VECTORS])
def test_writer_codes_inter_frames_in_a_decoded_streams_context(built, vector, k):
    """Inter frames written against a parser that has parsed the first k frames of a real stream parse, with a second
    parser that has parsed the same frames (and then every written frame before it), to the original records and
    blocks; written without a context they give the bytes they always gave."""
    import vp8_b200
    from vp8_b200._capi import Vp8rError
    prefix = _vector_payloads(vector)[:k]
    key = vp8_b200.Parser().parse(prefix[0])
    w, h = key.desc().hdr.width, key.desc().hdr.height
    key.close()
    ctx, follower = _parser_after(prefix), _parser_after(prefix)
    frames = _synthetic_inter_frames(w, h)
    differs = 0
    plain = b""
    for t, f in enumerate(frames):
        d = f.desc()
        n_mb = d.hdr.mb_cols * d.hdr.mb_rows
        free = f.write_bitstream()
        assert f.write_bitstream(context=None) == free
        plain += free
        written = f.write_bitstream(context=ctx)
        differs += written != free
        back = follower.parse(written)
        db = back.desc()
        assert _header_fields(db) == _header_fields(d), t
        assert _records(db, n_mb) == _records(d, n_mb), t
        assert _blocks(db, n_mb) == _blocks(d, n_mb), t
        back.close()
        # writing does not change the context
        assert f.write_bitstream(context=ctx) == written, t
        f.close()
    assert differs, "the prefix left the default context: nothing was tested"
    assert helpers.md5(plain) == CONTEXT_FREE_MD5[(w, h)], (w, h)
    # the context-free bytes of the first frame do not parse to its records in this stream (what the context is for)
    f = _synthetic_inter_frames(w, h)[0]
    d = f.desc()
    n_mb = d.hdr.mb_cols * d.hdr.mb_rows
    other = _parser_after(prefix)
    try:
        back = other.parse(f.write_bitstream())
        assert _records(back.desc(), n_mb) != _records(d, n_mb) or _blocks(back.desc(), n_mb) != _blocks(d, n_mb)
    except Vp8rError:
        pass
    f.close()


def test_writer_refuses_a_context_without_key_frame_or_of_another_size(built):
    import vp8_b200
    from vp8_b200._capi import Vp8rError
    frames = _synthetic_inter_frames(176, 144)
    fresh = vp8_b200.Parser()
    with pytest.raises(Vp8rError) as e:
        frames[0].write_bitstream(context=fresh)
    assert e.value.code == 5  # VP8R_ERR_STATE
    other = _parser_after(_vector_payloads("vp80-02-inter-1412")[:2])  # 96x96
    with pytest.raises(Vp8rError) as e:
        frames[0].write_bitstream(context=other)
    assert e.value.code == 5
    # a key frame resets the context: it is written the same with any context, even one that could not take it
    _, payloads = vp8_b200.read_ivf(helpers.synth_stream(CONTEXT_SYNTH[(176, 144)] + SYNTH_FIXED))
    key = vp8_b200.Parser().parse(payloads[0])
    assert key.desc().hdr.key_frame
    assert key.write_bitstream(context=fresh) == key.write_bitstream(context=other) == key.write_bitstream()
    for f in frames + [key]:
        f.close()


def test_new_vectors_coded_against_clamped_predictors_round_trip(built):
    """Vectors up to 28 px beyond the frame in every direction: the decoder clamps the neighbours' vectors to 16 px
    beyond the frame before it uses them as predictors, so NEAREST / NEAR select the clamped vector and NEW codes its
    delta from the clamped best.  Modes chosen by the restated rule, written, parsed: the same vectors and modes."""
    import vp8_b200
    _, payloads = vp8_b200.read_ivf(helpers.synth_stream("--width 64 --height 48 --frames 2 --seed 41 --pct-intra 0" + SYNTH_FIXED))
    ps = vp8_b200.Parser()
    ps.parse(payloads[0]).close()
    f = ps.parse(payloads[1])
    d = f.desc()
    cols, rows = d.hdr.mb_cols, d.hdr.mb_rows
    n_mb = cols * rows
    assert all(d.mbs[m].flags & IS_INTER for m in range(n_mb))
    # every macroblock points far out of the frame on the side it is nearest to, some exactly at the clamp bound
    rng = np.random.default_rng(7)
    vectors = []
    for r in range(rows):
        for c in range(cols):
            vr = (-(16 * r + 16 + int(rng.integers(-4, 13))) if r < rows / 2 else 16 * (rows - r) + int(rng.integers(-4, 13))) * 8
            vc = (-(16 * c + 16 + int(rng.integers(-4, 13))) if c < cols / 2 else 16 * (cols - c) + int(rng.integers(-4, 13))) * 8
            vectors.append((vr + 2 * int(rng.integers(0, 4)), vc - 2 * int(rng.integers(0, 4))))
    # plus a few that repeat a neighbour's clamped vector, so that NEAREST / NEAR of a clamped vector occur
    plan = _assign_modes(vectors, cols, rows)
    for m in (cols + 1, 2 * cols - 1, n_mb - 1):
        vectors[m] = plan[m][1]
        plan = _assign_modes(vectors, cols, rows)
    for m in range(n_mb):
        mb = d.mbs[m]
        mb.flags = (mb.flags & ~(MODE_BITS | (3 << 1))) | REF_LAST | (plan[m][0] << 3)
        mb.mv[0], mb.mv[1] = vectors[m]
    new_clamped = sum(p[0] == MV_NEW and p[2] for p in plan)
    reused_clamped = sum(p[0] in (MV_NEAREST, MV_NEAR) and p[3] for p in plan)
    assert new_clamped >= 3 and reused_clamped >= 1, (new_clamped, reused_clamped)
    back = vp8_b200.Parser()
    back.parse(payloads[0]).close()
    b = back.parse(f.write_bitstream())
    assert _records(b.desc(), n_mb) == _records(d, n_mb)
    assert [((b.desc().mbs[m].flags >> 3) & 7) for m in range(n_mb)] == [p[0] for p in plan]
    b.close()
    f.close()


# --------------------------------------------------------------------------------------------- GPU tier ----
def _oracle_many(lib, decs, imgs, w, h, q, lf, R):
    """oracle_encode_inter_frame for several streams at once (ctypes releases the GIL: one thread per stream)."""
    with ThreadPoolExecutor(max_workers=min(len(decs), os.cpu_count() or 1)) as pool:
        return list(pool.map(lambda a: _oracle_inter(lib, a[0], a[1], w, h, q, lf, R), zip(decs, imgs)))


def _check_decoders(eng, lib, payloads, recons, w, h, what):
    """The stream `payloads` decodes to `recons` (one image per frame) through the engine's host parse, its device
    parse and, where it has been built, the reference decoder (host parser -> oracle is checked frame by frame by
    the caller)."""
    import vp8_b200
    st = eng.open_stream()
    for t, p in enumerate(payloads):
        st.decode(p)
        assert st.read_frame() == recons[t], (what, t, "engine host parse")
    st.close()
    pd = vp8_b200.Parser()
    pd.set_defer_modes(True)
    st = eng.open_stream()
    for t, p in enumerate(payloads):
        fr = pd.parse(p, pinned=True)
        eng.reconstruct_batch([st], [fr])
        eng.sync()
        assert st.read_frame() == recons[t], (what, t, "engine device parse")
        fr.close()
    st.close()
    pd.close()
    if os.path.exists(helpers.REF_DECODE):
        shown = []
        ps = vp8_b200.Parser()
        for p, r in zip(payloads, recons):
            f = ps.parse(p)
            if f.desc().hdr.show_frame:
                shown.append(r)
            f.close()
        with tempfile.TemporaryDirectory() as td:
            path = os.path.join(td, "e.ivf")
            with open(path, "wb") as fh:
                fh.write(vp8_b200.ivf_bytes(w, h, payloads))
            assert helpers.ref_decode_ivf(path) == b"".join(shown), (what, "reference decoder")


def _compare_with_oracle(d, recs, pay, n_mb, what):
    for m in range(n_mb):
        a, b = d.mbs[m], recs[m]
        assert (a.flags & ~MODE_BITS, a.coef_mask, a.coef_offset, a.mv[0], a.mv[1]) == \
               (b.flags, b.coef_mask, b.coef_offset, b.mv[0], b.mv[1]), (what, m)
        nb = bin(a.coef_mask).count("1")
        assert d.payload[a.coef_offset * 16:(a.coef_offset + nb) * 16] == pay[b.coef_offset * 16:(b.coef_offset + nb) * 16], (what, m)


def _run_streams(eng, lib, seqs, w, h, q, lf=0, sharpness=0, R=16):
    """Encodes n streams in lock-step, one call per time step: seqs[k][0] as a key frame, the rest as inter frames.
    Every inter frame of every stream: device records (mode bits masked) and blocks equal the oracle's, predicting
    from the oracle's decode of the written stream; the re-parsed records (mode bits included) and blocks equal the
    device's; the device's modes equal the restated mode choice; the written stream decodes to the engine's
    reconstructions through host parser -> oracle, the engine's host and device parse and the reference decoder.
    Returns per stream and inter frame a dict: vectors, modes, blocks, coef_masks, new_clamped (NEW vectors coded
    against a clamped best) and last (the I420 image the frame predicted from)."""
    import vp8_b200
    n, cols, rows = len(seqs), (w + 15) // 16, (h + 15) // 16
    n_mb = cols * rows
    streams = [eng.open_stream() for _ in range(n)]
    decs = [lib.oracle_create() for _ in range(n)]
    parsers = [vp8_b200.Parser() for _ in range(n)]
    payloads, recons, out = [[] for _ in range(n)], [[] for _ in range(n)], [[] for _ in range(n)]
    try:
        for t in range(len(seqs[0])):
            imgs = [s[t] for s in seqs]
            if t == 0:
                frames = eng.encode_key_frames(streams, imgs, w, h, q, loop_filter_level=lf, sharpness=sharpness)
            else:
                frames = eng.encode_inter_frames(streams, imgs, w, h, q, loop_filter_level=lf, sharpness=sharpness, search_range=R)
                want = _oracle_many(lib, decs, imgs, w, h, q, lf, R)
            for k, f in enumerate(frames):
                what = (w, h, q, lf, R, k, t)
                d = f.desc()
                if t > 0:
                    recs, pay = want[k]
                    _compare_with_oracle(d, recs, pay, n_mb, what)
                    vectors = [(d.mbs[m].mv[0], d.mbs[m].mv[1]) for m in range(n_mb)]
                    plan = _assign_modes(vectors, cols, rows)
                    modes = [(d.mbs[m].flags >> 3) & 7 for m in range(n_mb)]
                    assert modes == [p[0] for p in plan], what
                    out[k].append(dict(vectors=vectors, modes=modes, blocks=_blocks(d, n_mb), last=recons[k][-1],
                                       coef_masks=[d.mbs[m].coef_mask for m in range(n_mb)],
                                       new_clamped=sum(p[0] == MV_NEW and p[2] for p in plan)))
                p = f.write_bitstream()
                payloads[k].append(p)
                recons[k].append(streams[k].read_frame())
                back = parsers[k].parse(p)
                db = back.desc()
                assert _records(db, n_mb) == _records(d, n_mb), what
                assert _blocks(db, n_mb) == _blocks(d, n_mb), what
                assert lib.oracle_decode_frame(decs[k], C.byref(db)) == 0
                assert _oracle_image(lib, decs[k]) == recons[k][-1], (what, "host parser -> oracle")
                back.close()
                f.close()
        for k in range(n):
            _check_decoders(eng, lib, payloads[k], recons[k], w, h, (w, h, q, lf, R, k))
    finally:
        for dec in decs:
            lib.oracle_destroy(dec)
        for st in streams:
            st.close()
        for ps in parsers:
            ps.close()
    return out


EDGE_SIZES = [(16, 16), (17, 17), (33, 18), (65, 33), (176, 144)]


@pytest.mark.gpu
@pytest.mark.parametrize("R", [4, 5, 23, 24])
def test_search_window_edges(built, R):
    """The texture panned by R + 0.75 px per frame in each of the eight directions, one stream per direction, two inter
    frames, on frames of one to 99 macroblocks: the refinement reaches +-(8R + 6) in 1/8 pel (the window's last staged
    rows and columns), and for R >= 17 vectors more than 16 px beyond the frame reach the decoder's clamp, so that
    NEW vectors are coded against clamped predictors."""
    import vp8_b200
    lib = _lib()
    eng = vp8_b200.Engine(0)
    clamped_new = 0
    try:
        for w, h in EDGE_SIZES:
            seqs = [[_far_pan(w, h, t, R, d, seed=R) for t in range(3)] for d in DIRS]
            res = _run_streams(eng, lib, seqs, w, h, 20, lf=8, R=R)
            largest = max(abs(c) for frames in res for fr in frames for v in fr["vectors"] for c in v)
            if (w, h) != (16, 16) or R + 3 < 16:
                # (one macroblock under a pan of 16 px or more sees none of its content in LAST)
                assert largest == 8 * R + 6, (w, h, largest)
            assert largest <= 8 * R + 6, (w, h, largest)
            clamped_new += sum(fr["new_clamped"] for frames in res for fr in frames)
    finally:
        eng.close()
    if R >= 17:
        assert clamped_new >= 1, clamped_new


@pytest.mark.gpu
@pytest.mark.parametrize("q", [0, 127])
def test_quantiser_and_content_extremes(built, q):
    """Residuals of +-255: sources that are the negative of the key frame, and saturated 0 / 255 checkerboards whose
    cells are larger than the search window, at q 0 and 127, loop-filter level 0 and 63, sharpness 0 and 7.  At q = 0
    coefficients need DCT_CAT6 tokens (>= 67) and Y2 DC values pass 2000."""
    import vp8_b200
    lib = _lib()
    w, h, R = 96, 64, 6
    tex = _i420(_analytic(h, w, 0, 0, 3), np.full((h // 2, w // 2), 60.0), np.full((h // 2, w // 2), 200.0))
    seqs = [[tex, _negative(tex), tex],
            [_checkerboard(w, h, 32, 0), _checkerboard(w, h, 32, 1), _checkerboard(w, h, 32, 0)],
            [_checkerboard(w, h, 32, 1), _negative(tex), _checkerboard(w, h, 32, 1)]]
    eng = vp8_b200.Engine(0)
    largest, y2_dc = 0, 0
    try:
        for lf, sharpness in ((0, 0), (63, 7), (63, 0), (0, 7)):
            res = _run_streams(eng, lib, seqs, w, h, q, lf=lf, sharpness=sharpness, R=R)
            for frames in res:
                for fr in frames:
                    largest = max([largest] + [abs(v) for b in fr["blocks"] for v in b])
                    # the first stored block of a macroblock is its Y2 block when bit 0 of its mask is set
                    y2_dc = max([y2_dc] + [abs(b[0]) for b, m in zip(fr["blocks"], fr["coef_masks"]) if m & 1])
    finally:
        eng.close()
    if q == 0:
        assert largest >= 67 and y2_dc > 2000, (largest, y2_dc)
    else:
        assert largest >= 1, largest


@pytest.mark.gpu
@pytest.mark.parametrize("R", [4, 24])
def test_ties_on_the_device(built, R):
    """Flat sources (every candidate costs the same SAD) and period-8 stripes moved by half a period (candidates
    four pixels left and right cost the same): the device's vectors are the oracle's, and each lies within the
    sub-pel refinement's reach (3 quarter pels) of the lowest-index full-pel minimum that the numpy search finds on
    the LAST frame the device predicted from."""
    import vp8_b200
    lib = _lib()
    w, h = 64, 48
    eng = vp8_b200.Engine(0)
    try:
        res = _run_streams(eng, lib, [[_flat(w, h, 90), _flat(w, h, 97), _flat(w, h, 60)],
                                      [_stripes(w, h, 0), _stripes(w, h, 4), _stripes(w, h, 8)]], w, h, 20, R=R)
    finally:
        eng.close()
    flat, stripes = res
    assert all(v == (0, 0) for fr in flat for v in fr["vectors"])
    tied = 0
    for t, fr in enumerate(stripes):
        last = np.frombuffer(fr["last"], np.uint8, w * h).reshape(h, w)
        src, _, _ = _padded_planes(_stripes(w, h, 4 * (t + 1)), w, h)
        want, ties = _numpy_full_pel(last, src, R, _dq(20)[1])
        tied += ties
        for m, ((dy, dx), v) in enumerate(zip(want, fr["vectors"])):
            assert abs(v[0] - 8 * dy) <= 6 and abs(v[1] - 8 * dx) <= 6, (t, m, (dy, dx), v)
    assert tied >= 1, tied


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(176, 144), (640, 360)], ids=lambda s: f"{s[0]}x{s[1]}")
def test_long_chains_of_far_pans(built, size):
    """Twelve streams of different far pans at R = 24 in one call per frame, ten inter frames each: every LAST after
    the first is an encoded inter frame with vectors at the window's edge, and every frame of every stream is
    compared."""
    import vp8_b200
    lib = _lib()
    w, h = size
    R = 24
    seqs = [[_far_pan(w, h, t, R, DIRS[k % 8], seed=k) for t in range(11)] for k in range(12)]
    eng = vp8_b200.Engine(0)
    try:
        res = _run_streams(eng, lib, seqs, w, h, 30 + 4 * (w // 176), lf=10, R=R)
    finally:
        eng.close()
    for k, frames in enumerate(res):
        assert len(frames) == 10
        # the edge is reached in the last frame of the chain too, predicting from nine encoded inter frames
        assert max(abs(c) for v in frames[-1]["vectors"] for c in v) == 8 * R + 6, k


# Decoded streams to encode on: (vector or synthetic stream, frames decoded before the encoder takes over)
DECODED = [("vp80-01-intra-1400", 3), ("vp80-02-inter-1402", 3), ("vp80-02-inter-1412", 4), ("vp80-02-inter-1418", 5),
           ("vp80-02-inter-1424", 3), ("vp80-03-segmentation-1403", 4), ("vp80-05-sharpness-1428", 3), ("hidden-altref", None)]
HIDDEN_SYNTH = "--width 96 --height 64 --frames 12 --seed 51 --hidden-altref 1 --altref-period 4"


def _decoded_source(name):
    import vp8_b200
    if name == "hidden-altref":
        payloads = vp8_b200.read_ivf(helpers.synth_stream(HIDDEN_SYNTH))[1]
        ps = vp8_b200.Parser()
        hidden = [not ps.parse(p).desc().hdr.show_frame for p in payloads]
        k = hidden.index(True, 1) + 1  # right after the first hidden frame
        assert k + 3 <= len(payloads)
        return payloads, k
    return _vector_payloads(name), dict(DECODED)[name]


@pytest.mark.gpu
@pytest.mark.parametrize("name", [d[0] for d in DECODED])
def test_encoding_on_decoded_streams(built, name):
    """A stream is decoded up to frame k (engine host parse, engine device parse, oracle), then three inter frames are
    encoded on top of it from the decoded pictures that follow in the same stream.  Device records and blocks equal
    the oracle's on both engine streams; the frames are written with the decoding parser as context, and the prefix's
    bytes followed by them decode, by every path, to the encoder's reconstructions."""
    import vp8_b200
    lib = _lib()
    payloads, k = _decoded_source(name)
    # the pictures: the oracle's decode of the whole stream
    ps, dec = vp8_b200.Parser(), lib.oracle_create()
    pictures = []
    for p in payloads[:k + 3]:
        f = ps.parse(p)
        assert lib.oracle_decode_frame(dec, C.byref(f.desc())) == 0
        pictures.append(_oracle_image(lib, dec))
        w, h = f.desc().hdr.width, f.desc().hdr.height
        f.close()
    lib.oracle_destroy(dec)
    ps.close()
    q, lf, R = 36, 12, 16
    cols, rows = (w + 15) // 16, (h + 15) // 16
    n_mb = cols * rows
    eng = vp8_b200.Engine(0)
    dec = lib.oracle_create()
    host, dev = vp8_b200.Parser(), vp8_b200.Parser()
    dev.set_defer_modes(True)
    try:
        sh, sd = eng.open_stream(), eng.open_stream()
        for t, p in enumerate(payloads[:k]):
            fh = host.parse(p)
            assert lib.oracle_decode_frame(dec, C.byref(fh.desc())) == 0
            fd = dev.parse(p, pinned=True)
            eng.reconstruct_batch([sh, sd], [fh, fd])
            eng.sync()
            assert sh.read_frame() == sd.read_frame() == _oracle_image(lib, dec), (name, t)
            fh.close()
            fd.close()
        written, recons = [], []
        for t in range(3):
            img = pictures[k + t]
            fh, fd = eng.encode_inter_frames([sh, sd], [img, img], w, h, q, loop_filter_level=lf, search_range=R)
            recs, pay = _oracle_inter(lib, dec, img, w, h, q, lf, R)
            _compare_with_oracle(fh.desc(), recs, pay, n_mb, (name, t, "host-parsed stream"))
            _compare_with_oracle(fd.desc(), recs, pay, n_mb, (name, t, "device-parsed stream"))
            data = fh.write_bitstream(context=host)
            assert fd.write_bitstream(context=dev) == data, (name, t)
            written.append(data)
            recons.append(sh.read_frame())
            assert sd.read_frame() == recons[-1], (name, t)
            # the oracle follows the written frame, parsed in the stream's context
            check = _parser_after(payloads[:k] + written[:-1])
            back = check.parse(data)
            assert _records(back.desc(), n_mb) == _records(fh.desc(), n_mb), (name, t)
            assert _blocks(back.desc(), n_mb) == _blocks(fh.desc(), n_mb), (name, t)
            assert lib.oracle_decode_frame(dec, C.byref(back.desc())) == 0
            assert _oracle_image(lib, dec) == recons[-1], (name, t, "host parser -> oracle")
            back.close()
            check.close()
            fh.close()
            fd.close()
        sh.close()
        sd.close()
        # the whole stream: the prefix decodes to the oracle's pictures, the encoded frames to the reconstructions
        _check_decoders(eng, lib, payloads[:k] + written, pictures[:k] + recons, w, h, name)
    finally:
        lib.oracle_destroy(dec)
        host.close()
        dev.close()
        eng.close()
