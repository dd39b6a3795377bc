"""Decode parity at the syntax extremes that ordinary streams never reach: coefficients whose dequantised int16 value
wraps to zero and the whole DCT_CAT6 range, motion vectors far beyond the frame (chroma sums that wrap in int16),
probability updates and frames that do not refresh them, frames without the skip flag, inter frames whose intra
macroblocks need 47 to 50 dependency levels, and loop-filter bands and groups of eight frames at 12 to 25
macroblock rows.

Every case first asserts, from the host parser's records (numpy over desc().mbs / payload / hdr.dq), that its
stream reaches the edge it is built for, and that the same stream without the vp8synth option does not.  The GPU
cases then require every decode path that applies to equal host parser -> oracle byte for byte."""
import ctypes as C
import os

import numpy as np
import pytest

import helpers

VP8R_MB_IS_INTER, VP8R_MB_LF_INNER, VP8R_MB_SKIP_COEF = 0x1, 0x20000, 0x40000
MODE_SPLIT = 4
CAT6_BASE = 67


def wrap_args(q, seg, lp):
    """Quantiser indices with a factor that is a multiple of 32 (q 28), 64 (57) or 128 (87: Y and chroma AC; 113:
    Y DC), with segmentation also in the segment rows around them; single big coefficients per block."""
    return (f"--width 176 --height 144 --frames 5 --seed {300 + q + lp} --q {q} --segmentation {seg} --log2-parts {lp} "
            f"--pct-big-coef 100 --coef-density 1 --pct-empty-block 30 --pct-skip 10 --pct-split 20 --pct-intra 20")


WRAP = {f"q{q}-seg{seg}-p{1 << lp}": wrap_args(q, seg, lp) for q, seg in ((28, 0), (57, 0), (87, 0), (87, 1), (113, 1))
        for lp in (0, 2)}
LONG_4K = "--width 3840 --height 2160 --frames 3 --seed 61 --log2-parts 3 --pct-split 30 --pct-new 60 --pct-long-mv 60 " \
          "--pct-skip 60 --coef-density 2 --pct-empty-block 80 --altref-period 0 --golden-period 0"
LONG_SMALL = {f"{w}x{h}": f"--width {w} --height {h} --frames 6 --seed {70 + w} --pct-split 30 --pct-new 60 --pct-long-mv 60"
              for w, h in ((16, 16), (33, 17))}
PROBS = {f"p{1 << lp}": f"--width 176 --height 144 --frames 8 --seed {90 + lp} --log2-parts {lp} --prob-updates 20 "
                        f"--no-skip-flag --pct-split 20 --pct-intra 20 --pct-big-coef 5 --altref-period 3"
         for lp in (0, 3)}
LEVEL_COLS = (19, 20, 21, 22)  # x 15 rows: an all-intra inter frame has C + 2R - 2 = 47, 48, 49, 50 levels


def level_args(cols, bpred):
    return f"--width {cols * 16} --height 240 --frames 3 --seed {cols} --pct-intra 100 --pct-bpred {bpred}"


def band_args(rows, k):
    """Stream k of the loop-filter band set: simple and normal filter, sharpness 0 and 7, level 63 with deltas."""
    return (f"--width 48 --height {rows * 16} --frames 3 --seed {400 + rows * 20 + k} --lf 63 --lf-deltas 1 "
            f"--filter-type {k % 2} --sharpness {7 * ((k // 2) % 2)} --pct-intra 20 --pct-split 20 --golden-period 2")


def without(args, option):
    """The same generator settings with `option` (and its value) left out."""
    toks = args.split()
    i = toks.index(option)
    return " ".join(toks[:i] + toks[i + (1 if option == "--no-skip-flag" else 2):])


ALL_STREAMS = {**{"wrap-" + k: v for k, v in WRAP.items()}, **{"long-" + k: v for k, v in LONG_SMALL.items()},
               **{"probs-" + k: v for k, v in PROBS.items()},
               **{f"levels-{c}-bpred{b}": level_args(c, b) for c in LEVEL_COLS for b in (0, 100)},
               **{f"bands-{r}-{k}": band_args(r, k) for r in (12, 13, 24, 25) for k in range(4)}}


def payloads_of(args):
    import vp8_b200
    return vp8_b200.read_ivf(helpers.synth_stream(args))[1]


def host_frames(args, fn, **parse):
    """fn(desc, mbs, payload) for every frame of the stream, host parse (full unless `parse` defers a half)."""
    import vp8_b200
    ps = vp8_b200.Parser()
    if parse.get("tokens"):
        ps.set_defer_tokens(True)
    if parse.get("modes"):
        ps.set_defer_modes(True)
    out = []
    for p in payloads_of(args):
        fr = ps.parse(p)
        d = fr.desc()
        n = d.hdr.mb_cols * d.hdr.mb_rows if not d.hdr.modes_deferred else 0
        mbs = np.ctypeslib.as_array(d.mbs, shape=(n,)).copy() if n else None
        pl = np.ctypeslib.as_array(d.payload, shape=(d.hdr.n_payload_blocks * 16,)).copy() if d.hdr.n_payload_blocks else \
            np.zeros(0, np.int16)
        out.append(fn(d, mbs, pl))
        fr.close()
    ps.close()
    return out


# ---- what a stream reaches, from the host parser's records -------------------------------------------------------
def coef_stats(args):
    """(blocks whose every coefficient dequantises to int16 0, of those the ones with a coded right or lower neighbour
    in their plane, OR of the DCT_CAT6 extra values, largest |coefficient|) over the stream."""
    def one(d, mbs, pl):
        cols, rows = d.hdr.mb_cols, d.hdr.mb_rows
        dq = np.array(d.hdr.dq, dtype=np.int32)
        # coded / wrapped blocks per plane on the block grid of the frame: Y 4x4 per macroblock, U and V 2x2
        coded = {p: np.zeros((rows * s, cols * s), bool) for p, s in (("Y", 4), ("U", 2), ("V", 2))}
        wrapped = {p: np.zeros_like(g) for p, g in coded.items()}
        n_wrapped = 0
        cat6, big = 0, 0
        for i, m in enumerate(mbs):
            mask = int(m["coef_mask"])
            if not mask:
                continue
            r, c = divmod(i, cols)
            seg = (int(m["flags"]) >> 9) & 3
            at = int(m["coef_offset"])
            for b in range(25):
                if not mask >> b & 1:
                    continue
                blk = pl[at * 16:at * 16 + 16].astype(np.int32)
                at += 1
                dc, ac = (2, 3) if b == 0 else ((0, 1) if b <= 16 else (4, 5))
                f = np.full(16, dq[seg][ac])
                f[0] = dq[seg][dc]
                prod = (blk * f).astype(np.int16)
                nz = blk != 0
                a = np.abs(blk[nz])
                big = max(big, int(a.max()))
                for v in a[a >= CAT6_BASE]:
                    cat6 |= int(v) - CAT6_BASE
                w = bool(np.all(prod[nz] == 0))
                n_wrapped += w
                if b == 0:
                    continue
                if b <= 16:
                    plane, s, k = "Y", 4, b - 1
                else:
                    plane, s, k = ("U" if b <= 20 else "V"), 2, (b - 17) % 4
                y, x = r * s + k // s, c * s + k % s
                coded[plane][y, x] = True
                wrapped[plane][y, x] = w
        near = 0
        for p in coded:
            g, wr = coded[p], wrapped[p]
            right = np.zeros_like(g)
            right[:, :-1] = g[:, 1:]
            below = np.zeros_like(g)
            below[:-1, :] = g[1:, :]
            near += int(np.sum(wr & (right | below)))
        return n_wrapped, near, cat6, big

    per = host_frames(args, lambda d, mbs, pl: one(d, mbs, pl) if mbs is not None else (0, 0, 0, 0))
    return (sum(p[0] for p in per), sum(p[1] for p in per), int(np.bitwise_or.reduce([p[2] for p in per])),
            max(p[3] for p in per))


def mv_stats(args):
    """(non-SPLIT vectors with |4 mv| > 32767, SPLIT chroma sums of four vectors beyond int16, prediction windows
    wholly beyond the 32-px border) over the stream."""
    def one(d, mbs, pl):
        if d.hdr.key_frame:
            return 0, 0, 0
        cols, rows = d.hdr.mb_cols, d.hdr.mb_rows
        inter = (mbs["flags"] & VP8R_MB_IS_INTER) != 0
        split = inter & (((mbs["flags"] >> 3) & 7) == MODE_SPLIT)
        whole = inter & ~split
        mv = mbs["mv"].astype(np.int32)
        wrap = int(np.sum(np.any(np.abs(4 * mv[whole]) > 32767, axis=1)))
        r, c = np.divmod(np.arange(cols * rows), cols)
        # a 16x16 window (plus the six-tap reach) that starts and ends beyond the border of the reference frame
        y0, x0 = 16 * r + (mv[:, 0] >> 3), 16 * c + (mv[:, 1] >> 3)
        out = (x0 + 19 < -32) | (x0 - 2 >= 16 * cols + 32) | (y0 + 19 < -32) | (y0 - 2 >= 16 * rows + 32)
        beyond = int(np.sum(out & whole))
        sums = 0
        for i in np.flatnonzero(split):
            sub = pl[int(mbs["aux"][i][0]) * 16:int(mbs["aux"][i][0]) * 16 + 32].astype(np.int32).reshape(4, 4, 2)
            quad = sub.reshape(2, 2, 2, 2, 2).sum(axis=(1, 3))  # the four vectors of each 8x8 chroma quarter
            sums += int(np.sum(np.abs(quad) > 32767))
            sy, sx = 16 * r[i] + 4 * np.arange(4)[:, None] + (sub[..., 0] >> 3), 16 * c[i] + 4 * np.arange(4)[None, :] + (sub[..., 1] >> 3)
            beyond += int(np.sum((sx + 7 < -32) | (sx - 2 >= 16 * cols + 32) | (sy + 7 < -32) | (sy - 2 >= 16 * rows + 32)))
        return wrap, sums, beyond

    per = host_frames(args, one)
    return tuple(sum(p[k] for p in per) for k in range(3))


class ModeHdr(C.Structure):
    _fields_ = [("first_off", C.c_uint32), ("first_size", C.c_uint32), ("bitpos", C.c_uint32),
                ("value", C.c_uint8), ("range", C.c_uint8), ("key_frame", C.c_uint8), ("segmentation_enabled", C.c_uint8),
                ("update_segment_map", C.c_uint8), ("mb_no_skip_coeff", C.c_uint8), ("prob_skip_false", C.c_uint8),
                ("prob_intra", C.c_uint8), ("prob_last", C.c_uint8), ("prob_gf", C.c_uint8), ("sign_bias", C.c_uint8 * 4),
                ("segment_tree_probs", C.c_uint8 * 3), ("segment_abs", C.c_uint8), ("segment_lf", C.c_int8 * 4),
                ("lf_adj_enable", C.c_uint8), ("frame_lf_level", C.c_uint8), ("ref_lf_delta", C.c_int8 * 4),
                ("mode_lf_delta", C.c_int8 * 4), ("ymode_probs", C.c_uint8 * 4), ("uvmode_probs", C.c_uint8 * 3),
                ("pad0", C.c_uint8), ("mv_probs", C.c_uint8 * 38), ("pad1", C.c_uint8 * 70)]


assert C.sizeof(ModeHdr) == 160


def deferred_headers(d):
    """(vp8r_mode_hdr or None, vp8r_token_hdr) of a frame parsed with deferred tokens or modes."""
    from vp8_b200._capi import TokenHdr
    base = C.addressof(d.payload.contents)
    th = C.cast(base + d.hdr.tokens_at * 32, C.POINTER(TokenHdr)).contents
    mh = C.cast(base + d.hdr.modes_at * 32, C.POINTER(ModeHdr)).contents if d.hdr.modes_deferred else None
    return mh, th


def prob_stats(args):
    """(frames with updated token probabilities, with updated MV probabilities, with updated 16x16 / chroma mode
    probabilities, without the skip flag), from the frame headers of the device-parse hand-over."""
    def one(d, mbs, pl):
        mh, th = deferred_headers(d)
        return (bytes(th.coef_probs), bytes(mh.mv_probs), bytes(mh.ymode_probs) + bytes(mh.uvmode_probs),
                mh.mb_no_skip_coeff, d.hdr.key_frame)

    per = host_frames(args, one, modes=True)
    dflt = host_frames("--width 16 --height 16 --frames 2 --seed 1", one, modes=True)[1]  # an inter frame's defaults
    return (sum(p[0] != dflt[0] for p in per), sum(p[1] != dflt[1] for p in per if not p[4]),
            sum(p[2] != dflt[2] for p in per if not p[4]), sum(p[3] == 0 for p in per))


def intra_levels(args):
    return host_frames(args, lambda d, mbs, pl: None if d.hdr.key_frame else
                       (d.hdr.n_intra_levels, int(np.sum((mbs["flags"] & VP8R_MB_IS_INTER) == 0)), d.hdr.mb_cols * d.hdr.mb_rows))


# ---- CPU tier ------------------------------------------------------------------------------------------------------
def test_new_options_are_deterministic(built):
    """The same settings and seed give the same bytes; the options change the stream (so they are not ignored)."""
    for name, args in [("wrap", WRAP["q87-seg0-p1"]), ("long", LONG_SMALL["33x17"]), ("probs", PROBS["p1"])]:
        a, b = helpers.synth_stream(args), helpers.synth_stream(args)
        assert a == b, name
    for option, args in [("--pct-big-coef", WRAP["q87-seg0-p1"]), ("--pct-long-mv", LONG_SMALL["33x17"]),
                         ("--prob-updates", PROBS["p1"]), ("--no-skip-flag", PROBS["p1"])]:
        assert helpers.synth_stream(args) != helpers.synth_stream(without(args, option)), option


def test_wrap_to_zero_and_cat6_reached(built):
    """Blocks whose coefficients all dequantise to int16 0 (512 x 128 and the like: the context they hand to their
    neighbours must say "zero"), with coded neighbours to the right or below; every DCT_CAT6 extra bit; |coef| 2048.
    Without --pct-big-coef none of it happens."""
    wrapped = near = cat6 = 0
    big = 0
    for args in WRAP.values():
        w, n, c6, b = coef_stats(args)
        wrapped, near, cat6, big = wrapped + w, near + n, cat6 | c6, max(big, b)
        w0, n0, c60, b0 = coef_stats(without(args, "--pct-big-coef"))
        assert w0 == 0 and b0 < 300, args
    assert wrapped >= 50 and near > 0
    assert cat6 == 0x7ff and big >= 2048


def test_long_vectors_reached(built):
    """4K: non-SPLIT vectors and SPLIT chroma sums that wrap in int16, windows wholly beyond the border; 16x16 and
    33x17: windows wholly beyond the border.  Without --pct-long-mv no vector wraps."""
    wrap, sums, beyond = mv_stats(LONG_4K)
    assert wrap > 0 and sums > 0 and beyond > 0
    assert mv_stats(without(LONG_4K, "--pct-long-mv"))[:2] == (0, 0)
    for args in LONG_SMALL.values():
        assert mv_stats(args)[2] > 0, args
        assert mv_stats(without(args, "--pct-long-mv"))[2] == 0, args


def test_probability_updates_reached(built):
    """Token, MV and mode probability updates and frames without the skip flag, as the device parse receives them;
    without --prob-updates / --no-skip-flag the tables stay at their defaults and every frame has the flag."""
    for args in PROBS.values():
        coef, mv, modes, noskip = prob_stats(args)
        assert coef > 0 and mv > 0 and modes > 0 and noskip == len(payloads_of(args))
        assert prob_stats(without(without(args, "--prob-updates"), "--no-skip-flag")) == (0, 0, 0, 0)


def test_intra_level_boundary_reached(built):
    """All-intra inter frames of 19..22 x 15 macroblocks: 47 and 48 levels take the level path, 49 and 50 do not
    (n_intra_levels 0: the wavefront)."""
    for bpred in (0, 100):
        for cols, want in zip(LEVEL_COLS, (47, 48, 0, 0)):
            for lv, n_intra, n_mb in filter(None, intra_levels(level_args(cols, bpred))):
                assert n_intra == n_mb and lv == want, (cols, bpred)


def test_deferred_parse_matches_full_parse_at_extremes(built):
    """With deferred tokens and with deferred modes, the host half of the parse equals the full parse field by field
    on every new stream (frame header, quantisers, macroblock records up to the fields the device fills in), and the
    token probabilities handed to the device are the same in both deferred forms."""
    hdr_fields = ("width", "height", "mb_cols", "mb_rows", "key_frame", "version", "show_frame", "filter_type",
                  "loop_filter_level", "sharpness_level", "refresh_last", "refresh_golden", "refresh_altref",
                  "copy_to_golden", "copy_to_altref", "sign_bias_golden", "sign_bias_altref", "q_index")

    def full(d, mbs, pl):
        return {f: getattr(d.hdr, f) for f in hdr_fields + ("n_inter_mbs", "n_split_mbs", "n_intra_levels")}, \
            bytes(d.hdr.dq), mbs, pl

    def tokens(d, mbs, pl):
        mh, th = deferred_headers(d)
        return {f: getattr(d.hdr, f) for f in hdr_fields + ("n_inter_mbs", "n_split_mbs", "n_intra_levels")}, \
            bytes(d.hdr.dq), mbs, pl, bytes(th.coef_probs)

    def modes(d, mbs, pl):
        mh, th = deferred_headers(d)
        return {f: getattr(d.hdr, f) for f in hdr_fields}, bytes(d.hdr.dq), bytes(th.coef_probs), mh.key_frame

    for name, args in ALL_STREAMS.items():
        fa, fb, fc = host_frames(args, full), host_frames(args, tokens, tokens=True), host_frames(args, modes, modes=True)
        assert len(fa) == len(fb) == len(fc)
        for k, (a, b, c) in enumerate(zip(fa, fb, fc)):
            assert a[0] == b[0] and a[1] == b[1], (name, k)
            assert {f: a[0][f] for f in hdr_fields} == c[0] and a[1] == c[1] and c[3] == a[0]["key_frame"], (name, k)
            assert b[4] == c[2], (name, k)
            ma, mb = a[2], b[2]
            assert np.array_equal(ma["flags"] & np.uint32(~VP8R_MB_LF_INNER & 0xffffffff),
                                  mb["flags"] & np.uint32(~(VP8R_MB_LF_INNER | VP8R_MB_SKIP_COEF) & 0xffffffff)), (name, k)
            assert not np.any(mb["coef_mask"]) and not np.any(mb["coef_offset"])
            assert np.all(ma["coef_mask"][(mb["flags"] & VP8R_MB_SKIP_COEF) != 0] == 0)
            inter = (ma["flags"] & VP8R_MB_IS_INTER) != 0
            assert np.array_equal(ma["mv"][inter], mb["mv"][inter]), (name, k)
            split = inter & (((ma["flags"] >> 3) & 7) == MODE_SPLIT)
            for i in np.flatnonzero(split):
                sa, sb = int(ma["aux"][i][0]) * 16, int(mb["aux"][i][0]) * 16
                assert np.array_equal(a[3][sa:sa + 32], b[3][sb:sb + 32]), (name, k, i)
            assert np.array_equal(ma["aux"][~split], mb["aux"][~split]), (name, k)


@pytest.mark.parametrize("name", sorted(ALL_STREAMS) + ["long-4k"])
def test_reference_decoder_equals_oracle_at_extremes(built, tmp_path, name):
    """The compiled, unmodified reference decoder against host parser -> oracle on every new stream: the only check
    of the oracle itself on these quirks (skipped where the reference decoder has not been built)."""
    if not os.path.exists(helpers.REF_DECODE):
        pytest.skip("oracle/_ref/decode not built")
    ivf = helpers.synth_stream(LONG_4K if name == "long-4k" else ALL_STREAMS[name])
    p = tmp_path / "s.ivf"
    p.write_bytes(ivf)
    assert helpers.ref_decode_ivf(str(p)) == b"".join(helpers.oracle_decode_ivf(ivf))


# ---- GPU tier ------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def engines(built):
    e = helpers.Engines()
    yield e
    e.close()


HOST = dict(env={})


def device_paths(env=None):
    """Tokens on the device, and macroblock headers + tokens on the device."""
    env = env or {}
    return [dict(env=env, tokens_on_device=True), dict(env=env, device_parse=True, depth=3)]


def check_paths(engines, named_args, paths, check_last=False):
    """Decodes the streams of `named_args` as one batch on every path; all frames must equal the oracle."""
    from vp8_b200 import _capi
    names = list(named_args)
    payloads = [payloads_of(named_args[n]) for n in names]
    want = [helpers.oracle_checksums(_capi.load(), p) for p in payloads]
    last = [helpers.oracle_frames(p)[-1][0] for p in payloads] if check_last else None
    for path in paths:
        bad = helpers.decode_on_path(engines.get(path["env"]), payloads, want, path, names, last_frames=last)
        assert not bad, (path, bad[:4])


@pytest.mark.gpu
@pytest.mark.parametrize("parts", [1, 4])
def test_wrap_to_zero_contexts_on_every_token_path(engines, parts):
    """Blocks that dequantise to zero hand "zero" to their neighbours, and the whole CAT6 range decodes, on the host
    parse and in the device token decoder."""
    streams = {k: v for k, v in WRAP.items() if k.endswith(f"-p{parts}")}
    check_paths(engines, streams, [HOST] + device_paths())


@pytest.mark.gpu
def test_long_vectors(engines):
    """Vectors beyond the frame and chroma sums that wrap in int16, host and device parse; the 4K frames by checksum,
    the last frame byte for byte."""
    streams = {"4k": LONG_4K, **LONG_SMALL}
    paths = [HOST, dict(env={}, device_parse=True, depth=3)]
    check_paths(engines, streams, paths, check_last=True)


@pytest.mark.gpu
def test_intra_level_boundary(engines):
    """47, 48, 49 and 50 intra levels in one batch: per-level launches on the host-parsed records, the device-built
    level table (IntraLevelsKernel) against the wavefront fallback on the device-parsed ones."""
    streams = {f"{c}-bpred{b}": level_args(c, b) for c in LEVEL_COLS for b in (0, 100)}
    paths = [HOST, dict(env={}, device_parse=True, depth=3)]
    check_paths(engines, streams, paths)


@pytest.mark.gpu
@pytest.mark.parametrize("rows", [12, 13, 24, 25])
def test_filter_bands_and_groups(engines, rows):
    """The packed-lane loop filter hands over between bands of 12 macroblock rows and packs eight frames per warp:
    batches of 1, 7, 8, 9 and 17 frames of one geometry mixing the simple and normal filter and sharpness 0 and 7 at
    level 63 with deltas, SWAR form and scalar form."""
    streams = {f"{rows}-{k}": band_args(rows, k) for k in range(17)}
    for n in (1, 7, 8, 9, 17):
        part = dict(list(streams.items())[:n])
        check_paths(engines, part, [dict(env={"VP8R_FILTER": "swar"}), dict(env={"VP8R_FILTER": "scalar"})])


@pytest.mark.gpu
def test_probability_updates_and_no_skip_flag_on_device_parse(engines):
    """Updated token, MV and mode probabilities (and frames that drop their updates) and frames without the skip flag,
    decoded with the macroblock headers and tokens on the device, and on the host."""
    for args in PROBS.values():
        assert all(prob_stats(args)[:3])
    check_paths(engines, {f"probs-{k}": v for k, v in PROBS.items()}, [HOST] + device_paths({"VP8R_FILTER": "swar"}))
