"""The key-frame encoder (EncodeIntraKernel) at the edges of its input space.

CPU tier: the oracle's key frame (oracle_encode_key_frame2) against a numpy restatement of its decisions, every
macroblock: the 16x16 luma and 8x8 chroma modes from predictors built on the oracle's unfiltered reconstruction with
the frame-border rules (127 above row 0, 129 left of column 0, P = 127 or 129), first minimum in the order V, H, DC,
TM; the B_PRED trial replayed sub-block by sub-block in a closed loop (edge arrays restated with the decoder's rules,
the right column reading the macroblock row above, the ten errors from oracle_pick_sub_mode), with its sub-modes,
blocks and reconstruction equal to the oracle's where it coded B_PRED and its total never below the best 16x16 error
where it did not.  The inputs are built to tie (flat, striped, checkered and small-alphabet pictures and their
negatives) and the ties they reach are counted and asserted.

GPU tier, every comparison exact: device records and blocks against the oracle, the re-parsed records against the
device's, the written stream through host parser -> oracle, the engine's host and device parse and the reference
decoder (where it has been built) against the engine's reconstruction.  Cases: the tie inputs at q 0, 20 and 127;
saturated residuals at q 0 and 127 with loop-filter and sharpness extremes; frames of one macroblock row or column, of
16, 17 and 33 rows (the kernel's warps each take every sixteenth row) up to 1080p and 4K; batches of 1 to 149 frames
under both loop-filter forms; calls of changing size on one engine's staging slots."""
import ctypes as C

import numpy as np
import pytest

import helpers
from test_encoder_inter import _blocks, _dq, _i420, _oracle_lib, _padded_planes, _records
from test_encoder_inter_edges import _analytic, _check_decoders, _checkerboard, _flat, _negative, _stripes

ORDER = (1, 2, 0, 3)  # the 16x16 / chroma candidates in decision order, vp8r.h numbering: V, H, DC, TM
MODE_SHIFT, UVMODE_SHIFT = 3, 6
B_LD, B_VL = 4, 7
TIE_SIZE = (80, 48)


# ------------------------------------------------------------------------------------------------ content ----
def _hstripes(w, h):
    """Horizontal stripes of period 8 (four dark rows, four bright)."""
    y = np.tile(np.where((np.arange(h) // 4) % 2 == 0, 40.0, 210.0)[:, None], (1, w))
    cw, ch = (w + 1) // 2, (h + 1) // 2
    return _i420(y, np.full((ch, cw), 150.0), np.full((ch, cw), 100.0))


def _pieces(w, h, seed, cell=4):
    """Piecewise-constant picture over a small alphabet (cells of `cell` px in luma, cell / 2 in chroma): equal
    neighbours make predictors coincide, so that the decisions tie."""
    rng = np.random.default_rng(seed)
    alphabet = np.array([0.0, 127.0, 128.0, 129.0, 255.0])
    cw, ch = (w + 1) // 2, (h + 1) // 2
    grid = lambda ph, pw, k: np.kron(alphabet[rng.integers(0, 5, (-(-ph // k), -(-pw // k)))], np.ones((k, k)))[:ph, :pw]
    return _i420(grid(h, w, cell), grid(ch, cw, max(cell // 2, 1)), grid(ch, cw, max(cell // 2, 1)))


def _texture(w, h, seed):
    cw, ch = (w + 1) // 2, (h + 1) // 2
    return _i420(_analytic(h, w, 0, 0, seed), 128 + 0.6 * (_analytic(ch, cw, 3, 1, seed + 1) - 128),
                 128 + 0.6 * (_analytic(ch, cw, 1, 5, seed + 2) - 128))


def _noise(w, h, seed):
    """Saturated noise: every sample 0 or 255."""
    rng = np.random.default_rng(seed)
    return rng.choice(np.array([0, 255], np.uint8), helpers.i420_bytes(w, h)).tobytes()


# Seeds of the piecewise-constant tie inputs, fixed so that the tie counts the tests assert are reproducible
PIECE_SEEDS = (3, 11, 24)


def _tie_inputs(w, h):
    base = [("flat%d" % v, _flat(w, h, v)) for v in (0, 127, 128, 129, 255)]
    base += [("vstripes", _stripes(w, h, 0)), ("hstripes", _hstripes(w, h)), ("checker4", _checkerboard(w, h, 4, 0)),
             ("checker16", _checkerboard(w, h, 16, 1))]
    base += [("pieces%d" % s, _pieces(w, h, s, 4 if k < 2 else 8)) for k, s in enumerate(PIECE_SEEDS)]
    return base + [("neg-" + name, _negative(img)) for name, img in base]


# ------------------------------------------------------------------------------------------------- oracle ----
def _oracle_key(lib, img, w, h, q, bpred, lf=0):
    from vp8_b200 import _capi
    cols, rows = (w + 15) // 16, (h + 15) // 16
    sy, su, sv = _padded_planes(img, w, h)
    mbs = (_capi.MbInfo * (cols * rows))()
    payload = (C.c_int16 * (cols * rows * 25 * 16))()
    ry, ru, rv = np.zeros_like(sy), np.zeros_like(su), np.zeros_like(sv)
    assert lib.oracle_encode_key_frame2(C.c_void_p(sy.ctypes.data), C.c_void_p(su.ctypes.data), C.c_void_p(sv.ctypes.data), cols, rows,
                                        (C.c_int16 * 6)(*_dq(q)), lf, mbs, payload, C.c_void_p(ry.ctypes.data),
                                        C.c_void_p(ru.ctypes.data), C.c_void_p(rv.ctypes.data), int(bpred)) == 0
    return dict(mbs=mbs, payload=payload, src=(sy, su, sv), rec=(ry, ru, rv), cols=cols, rows=rows)


def _rec_array(mbs, n_mb):
    """flags, coef_mask, coef_offset, mv, aux[0], aux[1] of every record (vp8r_mb_info as uint32)."""
    return np.ctypeslib.as_array(C.cast(mbs, C.POINTER(C.c_uint32)), shape=(n_mb * 8,)).reshape(n_mb, 8)[:, :6].copy()


def _block_array(payload, n_mb):
    """The payload as [macroblock][stored block][coefficient] (coef_offset = 25 * macroblock on both sides)."""
    return np.ctypeslib.as_array(C.cast(payload, C.POINTER(C.c_int16)), shape=(n_mb * 25 * 16,)).reshape(n_mb, 25, 16).copy()


def _stored(recs):
    """Number of stored blocks of each macroblock."""
    return np.array([bin(int(m)).count("1") for m in recs[:, 1]])


# ------------------------------------------------------------------------------------- numpy restatement ----
def _mb_errors(src, rec, r, c, n, P=None):
    """Squared errors of the V, H, DC and TM predictions of the n x n block (r, c) of one plane, predicted from the
    reconstruction `rec` with the decoder's frame-border rules (P: another top-left value for TM)."""
    s = src[n * r:n * r + n, n * c:n * c + n].astype(np.int64)
    above = rec[n * r - 1, n * c:n * c + n].astype(np.int64) if r else np.full(n, 127)
    left = rec[n * r:n * r + n, n * c - 1].astype(np.int64) if c else np.full(n, 129)
    if P is None:
        P = 127 if r == 0 else (129 if c == 0 else int(rec[n * r - 1, n * c - 1]))
    if r == 0 and c == 0:
        dc = 128
    else:
        shf = (3 if n == 16 else 2) + (r > 0) + (c > 0)
        dc = (int(above.sum()) * (r > 0) + int(left.sum()) * (c > 0) + (1 << (shf - 1))) >> shf
    preds = (np.broadcast_to(above, (n, n)), np.broadcast_to(left[:, None], (n, n)), np.full((n, n), dc),
             np.clip(left[:, None] + above[None, :] - P, 0, 255))
    return [int(((s - p) ** 2).sum()) for p in preds]


def _avg3(x, y, z):
    return (x + 2 * y + z + 2) >> 2


def _avg2(x, y):
    return (x + y + 1) >> 1


def _predict_b(mode, A, L, P):
    """The ten 4x4 predictors (RFC 6386 section 12.3), A = above[0..7], L = left[0..3]: o[row][column]."""
    E = [L[3], L[2], L[1], L[0], P, A[0], A[1], A[2], A[3]]
    o = np.zeros((4, 4), np.int64)
    if mode == 0:  # B_DC
        o[:] = (sum(A[:4]) + sum(L) + 4) >> 3
    elif mode == 1:  # B_TM
        o[:] = np.clip(np.array(L)[:, None] + np.array(A[:4])[None, :] - P, 0, 255)
    elif mode == 2:  # B_VE
        o[:] = [_avg3(P if j == 0 else A[j - 1], A[j], A[j + 1]) for j in range(4)]
    elif mode == 3:  # B_HE
        o[:] = np.array([_avg3(P if i == 0 else L[i - 1], L[i], L[min(i + 1, 3)]) for i in range(4)])[:, None]
    elif mode == 4:  # B_LD
        for i in range(4):
            for j in range(4):
                o[i, j] = _avg3(A[i + j], A[i + j + 1], A[min(i + j + 2, 7)])
    elif mode == 5:  # B_RD: down-right diagonals over E
        for i in range(4):
            for j in range(4):
                o[i, j] = _avg3(E[3 - i + j], E[4 - i + j], E[5 - i + j])
    elif mode == 6:  # B_VR
        o[3, 0] = _avg3(E[1], E[2], E[3])
        o[2, 0] = _avg3(E[2], E[3], E[4])
        o[3, 1] = o[1, 0] = _avg3(E[3], E[4], E[5])
        o[2, 1] = o[0, 0] = _avg2(E[4], E[5])
        o[3, 2] = o[1, 1] = _avg3(E[4], E[5], E[6])
        o[2, 2] = o[0, 1] = _avg2(E[5], E[6])
        o[3, 3] = o[1, 2] = _avg3(E[5], E[6], E[7])
        o[2, 3] = o[0, 2] = _avg2(E[6], E[7])
        o[1, 3] = _avg3(E[6], E[7], E[8])
        o[0, 3] = _avg2(E[7], E[8])
    elif mode == 7:  # B_VL
        o[0, 0] = _avg2(A[0], A[1])
        o[1, 0] = _avg3(A[0], A[1], A[2])
        o[2, 0] = o[0, 1] = _avg2(A[1], A[2])
        o[1, 1] = o[3, 0] = _avg3(A[1], A[2], A[3])
        o[2, 1] = o[0, 2] = _avg2(A[2], A[3])
        o[3, 1] = o[1, 2] = _avg3(A[2], A[3], A[4])
        o[2, 2] = o[0, 3] = _avg2(A[3], A[4])
        o[3, 2] = o[1, 3] = _avg3(A[3], A[4], A[5])
        o[2, 3] = _avg3(A[4], A[5], A[6])
        o[3, 3] = _avg3(A[5], A[6], A[7])
    elif mode == 8:  # B_HD
        o[3, 0] = _avg2(E[0], E[1])
        o[3, 1] = _avg3(E[0], E[1], E[2])
        o[2, 0] = o[3, 2] = _avg2(E[1], E[2])
        o[2, 1] = o[3, 3] = _avg3(E[1], E[2], E[3])
        o[2, 2] = o[1, 0] = _avg2(E[2], E[3])
        o[2, 3] = o[1, 1] = _avg3(E[2], E[3], E[4])
        o[1, 2] = o[0, 0] = _avg2(E[3], E[4])
        o[1, 3] = o[0, 1] = _avg3(E[3], E[4], E[5])
        o[0, 2] = _avg3(E[4], E[5], E[6])
        o[0, 3] = _avg3(E[5], E[6], E[7])
    else:  # 9: B_HU
        o[0, 0] = _avg2(L[0], L[1])
        o[0, 1] = _avg3(L[0], L[1], L[2])
        o[0, 2] = o[1, 0] = _avg2(L[1], L[2])
        o[0, 3] = o[1, 1] = _avg3(L[1], L[2], L[3])
        o[1, 2] = o[2, 0] = _avg2(L[2], L[3])
        o[1, 3] = o[2, 1] = _avg3(L[2], L[3], L[3])
        o[2, 2] = o[2, 3] = o[3, 0] = o[3, 1] = o[3, 2] = o[3, 3] = L[3]
    return o


def _int16(x):
    return ((np.asarray(x, np.int64) + 32768) & 0xFFFF) - 32768


def _sub_edges(ry, r, c, cols, rec, i, j):
    """Edge arrays (above[8], left[4], P) of sub-block (i, j) of macroblock (r, c) as the decoder gathers them:
    `rec` holds the macroblock's own sub-blocks reconstructed so far, `ry` the reconstructed luma around it.  The
    right column's above-right pixels come from the macroblock row above in every sub-block row, and from pixel 15
    of that row in the frame's last column."""
    y0, x0 = 16 * r, 16 * c
    top = lambda k: 127 if r == 0 else int(ry[y0 - 1, x0 + k])  # the row above the macroblock, k = -1 .. 19
    A = [top(4 * j + k) if i == 0 else int(rec[4 * i - 1, 4 * j + k]) for k in range(4)]
    if j == 3:
        A += [top(15 if c + 1 == cols else 16 + k) for k in range(4)]
    else:
        A += [top(4 * j + 4 + k) if i == 0 else int(rec[4 * i - 1, 4 * j + 4 + k]) for k in range(4)]
    L = [(129 if c == 0 else int(ry[y0 + 4 * i + k, x0 - 1])) if j == 0 else int(rec[4 * i + k, 4 * j - 1]) for k in range(4)]
    if i and j:
        P = int(rec[4 * i - 1, 4 * j - 1])
    elif i:
        P = 129 if c == 0 else int(ry[y0 + 4 * i - 1, x0 - 1])
    elif j:
        P = top(4 * j - 1)
    else:
        P = 127 if r == 0 else (129 if c == 0 else int(ry[y0 - 1, x0 - 1]))
    return A, L, P


def _bpred_trial(lib, sy, ry, r, c, cols, dq):
    """The B_PRED trial of macroblock (r, c) replayed: per sub-block in raster order the first minimum of the ten
    errors (oracle_pick_sub_mode, checked against the numpy predictors), the residual through the oracle's forward
    transform and quantiser, the decoder's way back.  Returns (total of the sixteen best errors, modes, the ten errors
    per sub-block, the 16x16 reconstruction, the sixteen quantised blocks)."""
    rec = np.zeros((16, 16), np.int64)
    total, modes, errs, qblocks = 0, [], [], []
    err = (C.c_uint32 * 10)()
    for i in range(4):
        for j in range(4):
            A, L, P = _sub_edges(ry, r, c, cols, rec, i, j)
            target = sy[16 * r + 4 * i:16 * r + 4 * i + 4, 16 * c + 4 * j:16 * c + 4 * j + 4].astype(np.int64)
            lib.oracle_pick_sub_mode((C.c_int * 8)(*A), (C.c_int * 4)(*L), P, (C.c_uint8 * 16)(*target.ravel().tolist()), err)
            e = list(err)
            preds = [_predict_b(m, A, L, P) for m in range(10)]
            assert e == [int(((target - p) ** 2).sum()) for p in preds], (r, c, i, j)
            mode = e.index(min(e))
            total += e[mode]
            modes.append(mode)
            errs.append(e)
            t = (C.c_int16 * 16)(*(target - preds[mode]).ravel().tolist())
            lib.oracle_fdct4x4(t)
            lib.oracle_quantize(t, dq[0], dq[1])
            qb = np.array(t[:], np.int64)
            qblocks.append(qb)
            v = _int16(qb * np.array([dq[0]] + [dq[1]] * 15))
            if v[1:].any():
                vv = (C.c_int16 * 16)(*v.tolist())
                lib.oracle_idct4x4(vv)
                res = np.array(vv[:], np.int64).reshape(4, 4)
            else:
                res = _int16((v[0] + 4) >> 3)
            rec[4 * i:4 * i + 4, 4 * j:4 * j + 4] = np.clip(_int16(preds[mode] + res), 0, 255)
    return total, modes, errs, rec, qblocks


def _restate(lib, o, q, bpred):
    """Checks every decision of the oracle's key frame `o` against the restatement; returns the edges reached."""
    sy, su, sv = o["src"]
    ry, ru, rv = o["rec"]
    cols, rows = o["cols"], o["rows"]
    n_mb = cols * rows
    recs, blocks = _rec_array(o["mbs"], n_mb), _block_array(o["payload"], n_mb)
    dq = _dq(q)
    first = lambda e: ORDER[e.index(min(e))]
    tie_not_v = lambda e: e.count(min(e)) >= 2 and e[0] > min(e)
    n = dict(luma_tie=0, chroma_tie=0, cross_half=0, inside_half=0, bpred_equal=0, bpred_equal_nonzero=0, bpred_mbs=0,
             ld_vl_right=0, p_left=0)
    for r in range(rows):
        for c in range(cols):
            m = r * cols + c
            flags = int(recs[m, 0])
            ymode, uvmode = (flags >> MODE_SHIFT) & 7, (flags >> UVMODE_SHIFT) & 3
            ey = _mb_errors(sy, ry, r, c, 16)
            ec = [a + b for a, b in zip(_mb_errors(su, ru, r, c, 8), _mb_errors(sv, rv, r, c, 8))]
            assert uvmode == first(ec), ("chroma", r, c, ec)
            n["luma_tie"] += tie_not_v(ey)
            n["chroma_tie"] += tie_not_v(ec)
            if c == 0 and r > 0:
                # in column 0, TM with P = 129 predicts what V does; with P = 127 instead it would be 2 brighter
                wrong = lambda plane, rec_, k: _mb_errors(plane, rec_, r, c, k, P=127)[3]
                n["p_left"] += wrong(sy, ry, 16) < min(ey) or wrong(su, ru, 8) + wrong(sv, rv, 8) < min(ec)
            best16 = min(ey)
            if not bpred:
                assert ymode == first(ey), ("luma", r, c, ey)
                continue
            total, modes, errs, rec, qblocks = _bpred_trial(lib, sy, ry, r, c, cols, dq)
            if ymode != 4:
                assert ymode == first(ey), ("luma", r, c, ey)
                assert total >= best16, ("B_PRED total below the best 16x16 error but not coded", r, c, total, best16)
                n["bpred_equal"] += total == best16
                n["bpred_equal_nonzero"] += total == best16 > 0
                continue
            n["bpred_mbs"] += 1
            aux = int(recs[m, 4]) | int(recs[m, 5]) << 32
            assert [(aux >> (4 * b)) & 15 for b in range(16)] == modes, ("sub-modes", r, c)
            assert total < best16, ("B_PRED coded but not strictly better", r, c, total, best16)
            assert np.array_equal(rec, ry[16 * r:16 * r + 16, 16 * c:16 * c + 16]), ("B_PRED reconstruction", r, c)
            mask = int(recs[m, 1])
            assert [bool(mask >> (b + 1) & 1) for b in range(16)] == [bool(qb.any()) for qb in qblocks] and not mask & 1, (r, c)
            stored = [qb for qb in qblocks if qb.any()]
            assert all(np.array_equal(blocks[m, k], qb) for k, qb in enumerate(stored)), ("B_PRED blocks", r, c)
            for e in errs:
                n["cross_half"] += min(e[:5]) == min(e[5:])
                n["inside_half"] += any(e[h:h + 5].count(min(e[h:h + 5])) >= 2 and e[h:h + 5].index(min(e[h:h + 5])) > 0 for h in (0, 5))
            n["ld_vl_right"] += c + 1 == cols and r > 0 and any(modes[4 * i + 3] in (B_LD, B_VL) for i in range(4))
    return n


def _add(total, n):
    for k, v in n.items():
        total[k] = total.get(k, 0) + v
    return total


def _assert_ties(n, q):
    """The ties the tie inputs are built for: luma and chroma decisions settled by the order H < DC < TM (V not
    among the tied), sub-block minima shared across the two half-warps and inside one half (won by a later mode of
    that half), and B_PRED totals equal to the best 16x16 error: 0 == 0 on flat areas at every q, non-zero equal
    totals from q 20 on (at q 0 the trial's reconstruction is close to exact and its later sub-blocks predict too
    well to tie)."""
    assert n["luma_tie"] >= 8 and n["chroma_tie"] >= 8, n
    assert n["cross_half"] >= 1 and n["inside_half"] >= 1, n
    assert n["bpred_equal"] >= 1, n
    if q > 0:
        assert n["bpred_equal_nonzero"] >= 1, n


def _lib():
    lib = _oracle_lib()
    lib.oracle_pick_sub_mode.restype = C.c_int
    return lib


# --------------------------------------------------------------------------------------------- CPU tier ----
@pytest.mark.parametrize("q", [0, 20, 127])
def test_decisions_restated_on_tie_inputs(built, q):
    """Every macroblock of the tie inputs, B_PRED off and on: the oracle's decisions are the restated ones, and the
    inputs reach every kind of tie."""
    lib = _lib()
    w, h = TIE_SIZE
    n = {}
    for bpred in (False, True):
        for name, img in _tie_inputs(w, h):
            got = _restate(lib, _oracle_key(lib, img, w, h, q, bpred), q, bpred)
            if bpred:
                _add(n, got)
    _assert_ties(n, q)


CPU_SIZES = [(16, 16), (17, 17), (16, 64), (64, 16), (33, 49), (320, 240)]


@pytest.mark.parametrize("size", CPU_SIZES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_decisions_restated_at_frame_edges(built, size):
    """Frames one macroblock wide or tall, where the border rules overlap, and a 320x240 frame: textured and
    piecewise-constant pictures at q 4 and 60.  Below row 0, macroblocks in column 0 are reached where TM with the wrong
    top-left value (127 instead of 129) would have won; in the one-column frame and at 320x240, B_PRED macroblocks
    in the last column use B_LD / B_VL in their right column (above-right copied from pixel 15 of the row above)."""
    lib = _lib()
    w, h = size
    n = {}
    for q in (4, 60):
        for img in (_texture(w, h, 5 + q), _pieces(w, h, 40 + q, 8), _negative(_texture(w, h, 6 + q))):
            for bpred in (False, True):
                _add(n, _restate(lib, _oracle_key(lib, img, w, h, q, bpred), q, bpred))
    if h > 16:
        assert n["p_left"] >= 1, n
    if size in ((16, 64), (320, 240)):
        assert n["ld_vl_right"] >= 1, n


# --------------------------------------------------------------------------------------------- GPU tier ----
def _compare(recs, blocks, orecs, oblocks, what):
    bad = np.nonzero((recs != orecs).any(axis=1))[0]
    assert not bad.size, (what, "record of macroblock", int(bad[0]), recs[bad[0]].tolist(), orecs[bad[0]].tolist())
    valid = np.arange(25)[None, :] < _stored(recs)[:, None]
    bad = np.nonzero(((blocks != oblocks).any(axis=2) & valid).any(axis=1))[0]
    assert not bad.size, (what, "blocks of macroblock", int(bad[0]))


def _encode(eng, imgs, w, h, q, lf=0, sharpness=0, bpred=True):
    """One call of encode_key_frames on fresh streams: per picture the device records and blocks (numpy), the written
    bitstream and the reconstruction."""
    streams = [eng.open_stream() for _ in imgs]
    out = []
    try:
        n_mb = ((w + 15) // 16) * ((h + 15) // 16)
        for f, st in zip(eng.encode_key_frames(streams, imgs, w, h, q, loop_filter_level=lf, sharpness=sharpness, bpred=bpred), streams):
            d = f.desc()
            out.append(dict(recs=_rec_array(d.mbs, n_mb), blocks=_block_array(d.payload, n_mb), data=f.write_bitstream(),
                            recon=st.read_frame(), records=_records(d, n_mb), coded=_blocks(d, n_mb)))
            f.close()
    finally:
        for st in streams:
            st.close()
    return out


def _encode_and_check(eng, lib, imgs, w, h, q, lf=0, sharpness=0, bpred=True):
    """_encode, and every frame exact against the oracle and through every decoder."""
    import vp8_b200
    n_mb = ((w + 15) // 16) * ((h + 15) // 16)
    out = _encode(eng, imgs, w, h, q, lf, sharpness, bpred)
    ps, orc = vp8_b200.Parser(), helpers.Oracle()
    try:
        for k, (img, fr) in enumerate(zip(imgs, out)):
            what = (w, h, q, lf, sharpness, bpred, k)
            o = _oracle_key(lib, img, w, h, q, bpred, lf)
            _compare(fr["recs"], fr["blocks"], _rec_array(o["mbs"], n_mb), _block_array(o["payload"], n_mb), what)
            back = ps.parse(fr["data"])
            assert _records(back.desc(), n_mb) == fr["records"], what
            assert _blocks(back.desc(), n_mb) == fr["coded"], what
            assert orc.decode(back) == fr["recon"], (what, "host parser -> oracle")
            back.close()
            _check_decoders(eng, lib, [fr["data"]], [fr["recon"]], w, h, what)
    finally:
        orc.close()
        ps.close()
    return out


def _extremes(frames):
    """Largest coefficient, largest Y2 DC, largest coefficient of a B_PRED macroblock."""
    big = y2 = bp = 0
    for fr in frames:
        recs, blocks = fr["recs"], fr["blocks"]
        valid = np.arange(25)[None, :] < _stored(recs)[:, None]
        per_mb = np.where(valid[:, :, None], np.abs(blocks), 0).max(axis=(1, 2))
        big = max(big, int(per_mb.max()))
        has_y2 = (recs[:, 1] & 1) == 1
        if has_y2.any():
            y2 = max(y2, int(np.abs(blocks[has_y2, 0, 0]).max()))
        is_bp = ((recs[:, 0] >> MODE_SHIFT) & 7) == 4
        if is_bp.any():
            bp = max(bp, int(per_mb[is_bp].max()))
    return big, y2, bp


@pytest.mark.gpu
@pytest.mark.parametrize("q", [0, 20, 127])
def test_ties_on_the_device(built, q):
    """The tie inputs, one call each with B_PRED off and on: the device takes every tied decision the way the oracle
    does (whose ties are re-counted here from the restatement)."""
    import vp8_b200
    lib = _lib()
    w, h = TIE_SIZE
    inputs = [img for _, img in _tie_inputs(w, h)]
    n = {}
    for img in inputs:
        _add(n, _restate(lib, _oracle_key(lib, img, w, h, q, True), q, True))
    _assert_ties(n, q)
    eng = vp8_b200.Engine(0)
    try:
        for bpred in (False, True):
            _encode_and_check(eng, lib, inputs, w, h, q, lf=20, sharpness=2, bpred=bpred)
    finally:
        eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("q", [0, 127])
def test_quantiser_and_content_extremes(built, q):
    """Residuals of +-255: 0 / 255 checkerboards of 16-px cells (every neighbour of a macroblock has the other
    colour), 4-px checkerboards, 0 / 255 noise and the negative of a texture, at q 0 and 127 under loop-filter
    levels 0 and 63 and sharpness 0 and 7.  At q 0: DCT_CAT6 coefficients (>= 67), Y2 DC values above 2000 with
    B_PRED off, B_PRED macroblocks with coefficients of 67 or more with it on."""
    import vp8_b200
    lib = _lib()
    w, h = 96, 64
    imgs = [_checkerboard(w, h, 16, 0), _checkerboard(w, h, 16, 1), _checkerboard(w, h, 4, 0), _noise(w, h, 8),
            _negative(_texture(w, h, 3))]
    eng = vp8_b200.Engine(0)
    seen = {}
    try:
        for lf, sharpness in ((0, 0), (63, 7), (63, 0), (0, 7)):
            for bpred in (False, True):
                big, y2, bp = _extremes(_encode_and_check(eng, lib, imgs, w, h, q, lf, sharpness, bpred))
                seen[bpred] = tuple(max(a, b) for a, b in zip(seen.get(bpred, (0, 0, 0)), (big, y2, bp)))
    finally:
        eng.close()
    if q == 0:
        assert seen[False][0] >= 67 and seen[False][1] > 2000, seen
        assert seen[True][2] >= 67, seen
    else:
        assert seen[False][0] >= 1 and seen[True][0] >= 1, seen


GEOMETRY = [(1, 1), (15, 15), (16, 16), (17, 17), (16, 256), (16, 272), (16, 528), (272, 16), (33, 513), (1920, 1080),
            (3840, 2160)]


@pytest.mark.gpu
@pytest.mark.parametrize("size", GEOMETRY, ids=lambda s: f"{s[0]}x{s[1]}")
def test_frame_geometry(built, size):
    """One macroblock; one column of 16, 17 and 33 rows (the sixteen warps of the CTA wrap around to row 16, 32);
    one row of 17 columns; 1080p and 4K (68 and 135 rows, 120 and 240 columns).  A textured and a piecewise-constant
    (tie) picture in one call, B_PRED off and on."""
    import vp8_b200
    lib = _lib()
    w, h = size
    imgs = [_texture(w, h, 11), _pieces(w, h, 12, 4)]
    eng = vp8_b200.Engine(0)
    try:
        for bpred in (False, True):
            _encode_and_check(eng, lib, imgs, w, h, 24, lf=16, sharpness=3, bpred=bpred)
    finally:
        eng.close()


@pytest.mark.gpu
def test_batch_geometry(built, monkeypatch):
    """Calls of 1, 127, 128 and 149 frames (one CTA per frame; more frames than the B200 has SMs) of different
    pictures: every frame equals the same picture encoded in a call of one and the oracle's encode.  From 128 frames
    on the engine filters the batch with FilterSwarKernel; the 149-frame call under VP8R_FILTER=scalar and =swar
    gives the same reconstructions."""
    import vp8_b200
    lib = _lib()
    w, h, q, lf = 48, 32, 30, 24
    imgs = [(_pieces(w, h, 100 + k, 4 << (k % 2)) if k % 3 == 0 else _texture(w, h, 100 + k)) for k in range(149)]
    eng = vp8_b200.Engine(0)
    try:
        single = [_encode(eng, [img], w, h, q, lf, 5)[0] for img in imgs]
        for n in (1, 127, 128):
            for k, fr in enumerate(_encode(eng, imgs[:n], w, h, q, lf, 5)):
                assert (fr["records"], fr["coded"], fr["data"], fr["recon"]) == \
                       (single[k]["records"], single[k]["coded"], single[k]["data"], single[k]["recon"]), (n, k)
        full = _encode_and_check(eng, lib, imgs, w, h, q, lf, 5)
        for k, fr in enumerate(full):
            assert (fr["data"], fr["recon"]) == (single[k]["data"], single[k]["recon"]), (149, k)
    finally:
        eng.close()
    for form in ("scalar", "swar"):
        monkeypatch.setenv("VP8R_FILTER", form)
        e = vp8_b200.Engine(0)
        try:
            got = _encode(e, imgs, w, h, q, lf, 5)
        finally:
            e.close()
        assert [fr["recon"] for fr in got] == [fr["recon"] for fr in full], form
        assert [fr["data"] for fr in got] == [fr["data"] for fr in full], form


@pytest.mark.gpu
def test_staging_slots_across_sizes(built):
    """Eleven calls of changing size on one engine (more than its eight staging slots, so slots are taken again by
    calls of another size): each equals the same call on a fresh engine, records, blocks, bitstream and
    reconstruction."""
    import vp8_b200
    calls = [(16, 16), (3840, 2160), (65, 33), (3840, 2160), (17, 17), (48, 32), (1920, 1080), (16, 16), (130, 98),
             (3840, 2160), (33, 17)]
    eng = vp8_b200.Engine(0)
    try:
        for k, (w, h) in enumerate(calls):
            imgs = [_texture(w, h, 200 + k), _pieces(w, h, 300 + k, 8)]
            args = (w, h, 20 + 7 * k, 4 * k, k % 8, k % 2 == 0)
            got = _encode(eng, imgs, *args)
            fresh = vp8_b200.Engine(0)
            try:
                want = _encode(fresh, imgs, *args)
            finally:
                fresh.close()
            for i, (a, b) in enumerate(zip(got, want)):
                assert (a["records"], a["coded"], a["data"], a["recon"]) == (b["records"], b["coded"], b["data"], b["recon"]), (k, w, h, i)
    finally:
        eng.close()
