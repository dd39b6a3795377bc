"""The residual transform of the reconstruction kernels on its edges: the DC-only shortcut for Y blocks fed by
Y2 alone, and macroblocks with more coded blocks than one pass of the warp transforms (8), decoded and compared
with the oracle frame by frame."""
import ctypes as C

import numpy as np
import pytest

import helpers

# dense residuals: every block coded, ~16 coefficients each, Y2 in every non-SPLIT macroblock; three versions
# (six-tap, bilinear, full-pixel chroma) and three quantizers
DENSE = [f"--width 176 --height 144 --frames 6 --seed {31 + v} --version {v} --q {q} --pct-split 60 --pct-skip 0 "
         f"--coef-density 16 --pct-empty-block 0" for v, q in [(0, 4), (1, 60), (3, 127)]]


def test_dc_only_idct_matches_oracle(built):
    """A block whose only non-zero input is its DC inverse-transforms to (dc + 4) >> 3 on all 16 outputs, for every
    int16 DC: the kernels write that instead of running the IDCT on such blocks."""
    orc = helpers.Oracle()
    blk = (C.c_int16 * 16)()
    bad = []
    for dc in range(-32768, 32768):
        C.memset(blk, 0, C.sizeof(blk))
        blk[0] = dc
        orc.lib.oracle_idct4x4(blk)
        want = np.int16((dc + 4) >> 3)
        if any(v != want for v in blk):
            bad.append(dc)
    orc.close()
    assert not bad, bad[:8]


def _coded_blocks_per_mb(data):
    """Coded blocks (Y2 apart) of every inter macroblock with a residual, and how many of those had Y2 coded."""
    import vp8_b200
    counts, y2 = [], 0
    ps = vp8_b200.Parser()
    for p in vp8_b200.read_ivf(data)[1]:
        f = ps.parse(p)
        d = f.desc()
        n = d.hdr.mb_rows * d.hdr.mb_cols
        raw = np.ctypeslib.as_array(C.cast(d.mbs, C.POINTER(C.c_uint32)), shape=(n * 8,)).reshape(n, 8)
        for flags, mask in zip(raw[:, 0], raw[:, 1]):  # vp8r_mb_info starts with flags, coef_mask
            if flags & 1 and mask:
                counts.append(bin(int(mask) >> 1).count("1"))
                y2 += bool(flags & 0x100 and mask & 1)
        f.close()
    ps.close()
    return counts, y2


@pytest.mark.parametrize("args", DENSE)
def test_dense_streams_need_a_second_pass(built, args):
    """The dense streams below do reach the second transform pass, up to all 24 blocks, with Y2 coded."""
    counts, y2 = _coded_blocks_per_mb(helpers.synth_stream(args))
    assert sum(c > 8 for c in counts) > len(counts) // 2
    assert max(counts) == 24
    assert y2 > 0


@pytest.mark.gpu
def test_dense_residuals_match_oracle(built):
    """Every frame of the dense streams equals the oracle's."""
    import vp8_b200
    eng = vp8_b200.Engine(0)
    try:
        for args in DENSE:
            ps, orc, st = vp8_b200.Parser(), helpers.Oracle(), eng.open_stream()
            for k, p in enumerate(vp8_b200.read_ivf(helpers.synth_stream(args))[1]):
                fr = ps.parse(p)
                want = orc.decode(fr)
                fr.close()
                st.decode(p)
                assert st.read_frame() == want, f"{args}: frame {k}"
            st.close()
            orc.close()
            ps.close()
    finally:
        eng.close()
