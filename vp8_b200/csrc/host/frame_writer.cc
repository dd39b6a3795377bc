#include "frame_writer.h"

#include <cstring>

#include "bool_writer.h"
#include "frame_parser.h"
#include "near_mvs.h"
#include "vp8r.h"

namespace vp8r {
namespace {

#include "vp8_prob_tables.inc"

enum { DC_PRED = 0, V_PRED, H_PRED, TM_PRED, B_PRED };
const int8_t kTreeYModeKey[8] = {-B_PRED, 2, 4, 6, -DC_PRED, -V_PRED, -H_PRED, -TM_PRED};
const int8_t kTreeYMode[8] = {-DC_PRED, 2, 4, 6, -V_PRED, -H_PRED, -TM_PRED, -B_PRED};
const int8_t kTreeMvRef[8] = {-MV_ZERO, 2, -MV_NEAREST, 4, -MV_NEAR, 6, -MV_NEW, -MV_SPLIT};
const int8_t kTreeSmallMv[14] = {2, 8, 4, 6, -0, -1, -2, -3, 10, 12, -4, -5, -6, -7};
const int8_t kTreeUvMode[6] = {-DC_PRED, 2, -V_PRED, 4, -H_PRED, -TM_PRED};
const int8_t kTreeBMode[18] = {0, 2, -1, 4, -2, 6, 8, 12, -3, 10, -5, -6, -4, 14, -7, 16, -8, -9};
const uint8_t kProbYModeKey[4] = {145, 156, 163, 128};
const uint8_t kProbUvModeKey[3] = {142, 114, 183};
const uint8_t kProbYModeDefault[4] = {112, 86, 140, 37};
const uint8_t kProbUvModeDefault[3] = {162, 101, 204};
const uint8_t kProbBModeInter[9] = {120, 90, 79, 133, 87, 85, 80, 111, 151};
const uint8_t kProbMvRef[6][4] = {{7, 1, 1, 143},   {14, 18, 14, 107}, {135, 64, 57, 68},
                                  {60, 56, 128, 65}, {159, 134, 128, 34}, {234, 188, 128, 28}};
const uint8_t kZigzag[16] = {0, 1, 4, 8, 5, 2, 3, 6, 9, 12, 13, 10, 7, 11, 14, 15};
const uint8_t kBand[17] = {0, 1, 2, 3, 6, 4, 5, 6, 6, 6, 6, 6, 6, 6, 6, 7, 0};
const uint8_t kCat1[] = {159, 0}, kCat2[] = {165, 145, 0}, kCat3[] = {173, 148, 140, 0};
const uint8_t kCat4[] = {176, 155, 140, 135, 0}, kCat5[] = {180, 157, 141, 134, 130, 0};
const uint8_t kCat6[] = {254, 254, 243, 230, 196, 177, 153, 140, 133, 130, 129, 0};
const uint8_t *const kCatProbs[6] = {kCat1, kCat2, kCat3, kCat4, kCat5, kCat6};
const int kCatBase[7] = {5, 7, 11, 19, 35, 67, 2115};
const int kCatBits[6] = {1, 2, 3, 4, 5, 11};

// One block of tokens (RFC 6386 section 13; the mirror of FrameParser::ReadCoefTokens): `blk` holds the quantised
// coefficients in raster order, scan position n is blk[kZigzag[n]].  No end-of-block right after a zero token.
// Returns whether any coefficient from `first` on is non-zero.  A magnitude above DCT_CAT6's range cannot be coded.
// `coef` holds the token probabilities of the frame's context.
bool WriteBlock(BoolWriter &bw, const uint8_t (*coef)[8][3][11], int type, int ctx, int first, const int16_t *blk,
                bool *too_large) {
  int last = -1;
  for (int n = first; n < 16; ++n)
    if (blk[kZigzag[n]]) last = n;
  auto probs = [&](int n, int cx) { return coef[type][kBand[n]][cx]; };
  bool prev_zero = false;
  int n = first;
  for (; n <= last; ++n) {
    const uint8_t *p = probs(n, ctx);
    const int v = blk[kZigzag[n]], a = v < 0 ? -v : v;
    if (!prev_zero) bw.Put(p[0], 1);
    if (a == 0) {
      bw.Put(p[1], 0);
      prev_zero = true;
      ctx = 0;
      continue;
    }
    bw.Put(p[1], 1);
    if (a == 1) {
      bw.Put(p[2], 0);
    } else {
      bw.Put(p[2], 1);
      if (a <= 4) {
        bw.Put(p[3], 0);
        if (a == 2) {
          bw.Put(p[4], 0);
        } else {
          bw.Put(p[4], 1);
          bw.Put(p[5], a == 4);
        }
      } else {
        if (a >= kCatBase[6]) {
          *too_large = true;
          return true;
        }
        bw.Put(p[3], 1);
        int cat = 0;
        while (a >= kCatBase[cat + 1]) ++cat;
        if (cat < 2) {
          bw.Put(p[6], 0);
          bw.Put(p[7], cat == 1);
        } else {
          bw.Put(p[6], 1);
          if (cat < 4) {
            bw.Put(p[8], 0);
            bw.Put(p[9], cat == 3);
          } else {
            bw.Put(p[8], 1);
            bw.Put(p[10], cat == 5);
          }
        }
        const int extra = a - kCatBase[cat];
        for (int i = 0; i < kCatBits[cat]; ++i) bw.Put(kCatProbs[cat][i], (extra >> (kCatBits[cat] - 1 - i)) & 1);
      }
    }
    bw.Put(128, v < 0);
    prev_zero = false;
    ctx = a > 1 ? 2 : 1;
  }
  if (n < 16) bw.Put(probs(n, ctx)[0], 0);  // end of block (never right after a zero: `last` is non-zero)
  return last >= 0;
}

// One motion-vector component in quarter-pel units (the mirror of FrameParser::ReadMvComponent).
void WriteMvComponent(BoolWriter &bw, const uint8_t *p, int v) {
  const int x = v < 0 ? -v : v;
  if (x < 8) {
    bw.Put(p[0], 0);
    bw.Tree(kTreeSmallMv, 14, p + 2, x);
  } else {
    bw.Put(p[0], 1);
    for (int i = 0; i < 3; ++i) bw.Put(p[9 + i], (x >> i) & 1);
    for (int i = 9; i > 3; --i) bw.Put(p[9 + i], (x >> i) & 1);
    if (x & 0xFFF0) bw.Put(p[9 + 3], (x >> 3) & 1);
  }
  if (x) bw.Put(p[1], v < 0);
}

// The context of a stream right after a key frame: the default token, motion-vector and 16x16 / chroma mode
// probabilities (FrameParser::LoadDefaults).
EntropyTables DefaultTables() {
  EntropyTables t;
  std::memcpy(t.coef, kCoefDefault, sizeof(t.coef));
  std::memcpy(t.mv, kMvDefault, sizeof(t.mv));
  std::memcpy(t.ymode, kProbYModeDefault, sizeof(t.ymode));
  std::memcpy(t.uvmode, kProbUvModeDefault, sizeof(t.uvmode));
  return t;
}

// P(bit == 0) out of 256 for `zeros` of `total` decisions, kept inside 1..255 (how prob_skip_false is chosen).
int ProbOf(size_t zeros, size_t total) {
  const int p = int(256 * zeros / (total ? total : 1));
  return p < 1 ? 1 : (p > 255 ? 255 : p);
}

// The five quantiser deltas (y_dc, y2_dc, y2_ac, uv_dc, uv_ac) under which q_index gives the factors dq; the
// smallest magnitude wins, positive before negative.  False when no deltas in -15..15 give them.
bool FindQuantDeltas(int q_index, const int16_t dq[6], int delta[5]) {
  static const int kColumn[5] = {VP8R_DQ_Y1_DC, VP8R_DQ_Y2_DC, VP8R_DQ_Y2_AC, VP8R_DQ_UV_DC, VP8R_DQ_UV_AC};
  int16_t f[6];
  for (int i = 0; i < 5; ++i) delta[i] = 0;
  DequantFactors(q_index, delta, f);
  if (f[VP8R_DQ_Y1_AC] != dq[VP8R_DQ_Y1_AC]) return false;
  for (int i = 0; i < 5; ++i) {
    bool found = false;
    for (int m = 0; m <= 15 && !found; ++m)
      for (int sgn = 1; sgn >= -1 && !found; sgn -= 2) {
        int d[5] = {0, 0, 0, 0, 0};
        d[i] = sgn * m;
        DequantFactors(q_index, d, f);
        if (f[kColumn[i]] == dq[kColumn[i]]) {
          delta[i] = d[i];
          found = true;
        }
      }
    if (!found) return false;
  }
  return true;
}

}  // namespace

int AssignInterModes(vp8r_mb_info *mbs, int cols, int rows, std::string *err) {
  std::vector<MbCtx> ctx(size_t(cols) * rows, MbCtx{0, 0, 0, Mv{0, 0}});
  const bool sign_bias[4] = {false, false, false, false};
  for (int r = 0; r < rows; ++r)
    for (int c = 0; c < cols; ++c) {
      const int idx = r * cols + c;
      vp8r_mb_info &mb = mbs[idx];
      if (!(mb.flags & VP8R_MB_IS_INTER)) continue;
      const int ref = int((mb.flags >> VP8R_MB_REF_SHIFT) & 3);
      const NearMvs nm = FindNearMvs(ctx.data(), r, c, cols, rows, ref, sign_bias);
      const Mv v{mb.mv[0], mb.mv[1]};
      // probability of each mode's path through the mode tree, all scaled to 256^4 (exact comparison)
      uint64_t p[4];
      for (int i = 0; i < 4; ++i) p[i] = kProbMvRef[nm.cnt[i]][i];
      const uint64_t w_zero = p[0] << 24, w_nearest = (256 - p[0]) * p[1] << 16,
                     w_near = (256 - p[0]) * (256 - p[1]) * p[2] << 8;
      int mode = MV_NEW;
      uint64_t w = 0;
      if (v == nm.nearest && w_nearest > w) mode = MV_NEAREST, w = w_nearest;
      if (v == nm.near && w_near > w) mode = MV_NEAR, w = w_near;
      if (!v.nonzero() && w_zero > w) mode = MV_ZERO, w = w_zero;
      if (mode == MV_NEW) {
        const int dr = v.r - nm.best.r, dc = v.c - nm.best.c;
        if ((dr | dc) & 1 || dr / 2 > 1023 || dr / 2 < -1023 || dc / 2 > 1023 || dc / 2 < -1023) {
          if (err) *err = "motion vector too far from its predictor to be coded";
          return VP8R_ERR_INVALID_ARG;
        }
      }
      mb.flags = (mb.flags & ~(7u << VP8R_MB_MODE_SHIFT)) | (uint32_t(mode) << VP8R_MB_MODE_SHIFT);
      ctx[idx] = MbCtx{1, uint8_t(ref), uint8_t(mode), v};
    }
  return VP8R_OK;
}

int WriteFrame(const vp8r_frame &f, const FrameParser *context, std::vector<uint8_t> *out, std::string *err) {
  const vp8r_frame_hdr &h = f.hdr;
  auto fail = [&](const char *what, int code = VP8R_ERR_INVALID_ARG) {
    if (err) *err = what;
    return code;
  };
  if (!f.blob) return fail("vp8r_frame_write_bitstream: the frame has no host arrays");
  if (h.tokens_deferred || h.modes_deferred) return fail("vp8r_frame_write_bitstream: the frame holds raw partitions, not macroblock records");
  const int cols = h.mb_cols, rows = h.mb_rows;
  if (cols <= 0 || rows <= 0 || size_t(cols) * rows != f.n_mb) return fail("vp8r_frame_write_bitstream: inconsistent frame size");
  if (h.version > 3) return fail("vp8r_frame_write_bitstream: unknown bitstream version");
  const bool key = h.key_frame != 0;
  // A key frame resets the decoder's context to the defaults; an inter frame is coded in the one it is decoded in.
  static const EntropyTables kDefaults = DefaultTables();
  const EntropyTables *probs = &kDefaults;
  if (context && !key) {
    if (!context->have_key()) return fail("vp8r_frame_write_bitstream_in: the context parser has not parsed a key frame", VP8R_ERR_STATE);
    if (context->width() != h.width || context->height() != h.height)
      return fail("vp8r_frame_write_bitstream_in: the context parser's frame size differs from the frame's", VP8R_ERR_STATE);
    probs = &context->probs();
  }
  const vp8r_mb_info *mbs = f.mbs();
  const int16_t *payload = f.payload();
  int qdelta[5];
  if (!FindQuantDeltas(h.q_index, h.dq[0], qdelta)) return fail("vp8r_frame_write_bitstream: no quantiser deltas give the frame's factors");

  // Per-frame probabilities from the frame's own counts: P(bit == 0) of the skip flag (0 = coded), of is_inter
  // (0 = intra), of the reference (0 = last) and of golden / altref (0 = golden).
  size_t n_skip = 0, n_intra = 0, n_last = 0, n_golden = 0, n_altref = 0;
  for (size_t i = 0; i < f.n_mb; ++i) {
    n_skip += mbs[i].coef_mask == 0;
    if (!(mbs[i].flags & VP8R_MB_IS_INTER)) ++n_intra;
    else {
      const int ref = int((mbs[i].flags >> VP8R_MB_REF_SHIFT) & 3);
      n_last += ref == 1;
      n_golden += ref == 2;
      n_altref += ref == 3;
    }
  }
  const int prob_skip = ProbOf(f.n_mb - n_skip, f.n_mb);
  const int prob_intra = ProbOf(n_intra, f.n_mb), prob_last = ProbOf(n_last, f.n_mb - n_intra);
  const int prob_gf = ProbOf(n_golden, n_golden + n_altref);

  BoolWriter hdr, tok;
  if (key) {
    hdr.Lit(1, 0);  // color space
    hdr.Lit(1, 0);  // clamping type: the reconstruction clamps
  }
  hdr.Lit(1, 0);  // segmentation_enabled
  hdr.Lit(1, h.filter_type ? 1u : 0u);
  hdr.Lit(6, h.loop_filter_level);
  hdr.Lit(3, h.sharpness_level);
  hdr.Lit(1, 0);  // loop_filter_adj_enable
  hdr.Lit(2, 0);  // one DCT partition
  hdr.Lit(7, h.q_index);
  for (int i = 0; i < 5; ++i) {
    hdr.Lit(1, qdelta[i] != 0);
    if (qdelta[i]) hdr.SignedLit(4, qdelta[i]);
  }
  if (!key) {
    hdr.Lit(1, h.refresh_golden ? 1u : 0u);
    hdr.Lit(1, h.refresh_altref ? 1u : 0u);
    if (!h.refresh_golden) hdr.Lit(2, h.copy_to_golden);
    if (!h.refresh_altref) hdr.Lit(2, h.copy_to_altref);
    hdr.Lit(1, h.sign_bias_golden ? 1u : 0u);
    hdr.Lit(1, h.sign_bias_altref ? 1u : 0u);
  }
  hdr.Lit(1, 1);  // refresh_entropy_probs
  if (!key) hdr.Lit(1, h.refresh_last ? 1u : 0u);
  for (int i = 0; i < 1056; ++i) hdr.Put(kCoefUpdate[i], 0);  // keep the context's token probabilities
  hdr.Lit(1, 1);                                             // mb_no_skip_coeff
  hdr.Lit(8, uint32_t(prob_skip));
  if (!key) {
    hdr.Lit(8, uint32_t(prob_intra));
    hdr.Lit(8, uint32_t(prob_last));
    hdr.Lit(8, uint32_t(prob_gf));
    hdr.Lit(1, 0);                                         // keep the context's 16x16 luma mode probabilities
    hdr.Lit(1, 0);                                         // ... its chroma mode probabilities
    for (int i = 0; i < 38; ++i) hdr.Put(kMvUpdate[i], 0);  // ... and its motion-vector probabilities
  }

  const bool sign_bias[4] = {false, false, h.sign_bias_golden != 0, h.sign_bias_altref != 0};
  std::vector<MbCtx> ctx(key ? 0 : f.n_mb, MbCtx{0, 0, 0, Mv{0, 0}});
  std::vector<uint8_t> above_b(size_t(cols) * 4, 0), nz_ay(size_t(cols) * 4, 0), nz_au(size_t(cols) * 2, 0), nz_av(size_t(cols) * 2, 0),
      nz_ay2(size_t(cols), 0);
  bool too_large = false;
  for (int r = 0; r < rows; ++r) {
    uint8_t left_b[4] = {0, 0, 0, 0};
    uint8_t nz_ly[4] = {0, 0, 0, 0}, nz_lu[2] = {0, 0}, nz_lv[2] = {0, 0}, nz_ly2 = 0;
    for (int c = 0; c < cols; ++c) {
      const int idx = r * cols + c;
      const vp8r_mb_info &mb = mbs[idx];
      const bool inter = (mb.flags & VP8R_MB_IS_INTER) != 0;
      if (inter && key) return fail("vp8r_frame_write_bitstream: inter macroblock in a key frame");
      if ((mb.flags >> VP8R_MB_QSEG_SHIFT) & 3) return fail("vp8r_frame_write_bitstream: macroblock of a segment (segmentation is not written)");
      if (int((mb.flags >> VP8R_MB_LF_SHIFT) & 63) != h.loop_filter_level)
        return fail("vp8r_frame_write_bitstream: macroblock filter level differs from the frame's (loop-filter deltas are not written)");
      const int ymode = int((mb.flags >> VP8R_MB_MODE_SHIFT) & 7), uvmode = int((mb.flags >> VP8R_MB_UVMODE_SHIFT) & 3);
      if (inter && ymode == MV_SPLIT) return fail("vp8r_frame_write_bitstream: SPLIT macroblocks cannot be written");
      const bool has_y2 = inter || ymode != B_PRED;
      if (has_y2 != ((mb.flags & VP8R_MB_HAS_Y2) != 0) || ymode > B_PRED) return fail("vp8r_frame_write_bitstream: inconsistent macroblock mode");
      const bool skip = mb.coef_mask == 0;
      hdr.Put(prob_skip, skip);
      if (!key) hdr.Put(prob_intra, inter);
      if (inter) {
        const int ref = int((mb.flags >> VP8R_MB_REF_SHIFT) & 3);
        if (ref == 0) return fail("vp8r_frame_write_bitstream: inter macroblock without a reference frame");
        hdr.Put(prob_last, ref != 1);
        if (ref != 1) hdr.Put(prob_gf, ref == 3);
        const NearMvs nm = FindNearMvs(ctx.data(), r, c, cols, rows, ref, sign_bias);
        const Mv v{mb.mv[0], mb.mv[1]};
        bool ok;
        int dr = 0, dc = 0;
        switch (ymode) {
          case MV_NEAREST: ok = v == nm.nearest; break;
          case MV_NEAR: ok = v == nm.near; break;
          case MV_ZERO: ok = !v.nonzero(); break;
          default:
            dr = v.r - nm.best.r;
            dc = v.c - nm.best.c;
            ok = !((dr | dc) & 1) && dr / 2 <= 1023 && dr / 2 >= -1023 && dc / 2 <= 1023 && dc / 2 >= -1023;
            break;
        }
        if (!ok) return fail("vp8r_frame_write_bitstream: motion vector contradicts its mode");
        uint8_t p[4];
        for (int i = 0; i < 4; ++i) p[i] = kProbMvRef[nm.cnt[i]][i];
        hdr.Tree(kTreeMvRef, 8, p, ymode);
        if (ymode == MV_NEW) {
          WriteMvComponent(hdr, probs->mv[0], dr / 2);
          WriteMvComponent(hdr, probs->mv[1], dc / 2);
        }
        ctx[size_t(idx)] = MbCtx{1, uint8_t(ref), uint8_t(ymode), v};
      } else {
        hdr.Tree(key ? kTreeYModeKey : kTreeYMode, 8, key ? kProbYModeKey : probs->ymode, ymode);
        if (ymode == B_PRED) {
          for (int i = 0; i < 4; ++i)
            for (int j = 0; j < 4; ++j) {
              const int b = i * 4 + j, m = int((mb.aux[b >> 3] >> ((b & 7) * 4)) & 15);
              if (m > 9) return fail("vp8r_frame_write_bitstream: invalid sub-block mode");
              if (key) {
                hdr.Tree(kTreeBMode, 18, &kKfBmode[(size_t(above_b[size_t(c) * 4 + j]) * 10 + left_b[i]) * 9], m);
                above_b[size_t(c) * 4 + j] = left_b[i] = uint8_t(m);
              } else {
                hdr.Tree(kTreeBMode, 18, kProbBModeInter, m);
              }
            }
        } else if (key) {
          static const uint8_t implied[4] = {0, 2, 3, 1};  // DC->B_DC, V->B_VE, H->B_HE, TM->B_TM (RFC 6386 11.3)
          for (int i = 0; i < 4; ++i) above_b[size_t(c) * 4 + i] = left_b[i] = implied[ymode];
        }
        hdr.Tree(kTreeUvMode, 6, key ? kProbUvModeKey : probs->uvmode, uvmode);
      }

      if (!skip) {
        const int16_t *dq = h.dq[0];
        // stored blocks follow each other in increasing block number; absent blocks are all zero
        static const int16_t kZeroBlock[16] = {0};
        const int16_t *next = payload + size_t(mb.coef_offset) * 16;
        const int16_t *blk[25];
        for (int b = 0; b < 25; ++b) {
          if ((mb.coef_mask >> b) & 1) {
            blk[b] = next;
            next += 16;
          } else {
            blk[b] = kZeroBlock;
          }
        }
        // The token contexts of later blocks are "non-zero after dequantisation" (FrameParser::ReadCoefTokens: a
        // product that wraps to 0 in int16 counts as zero there).
        auto dq_nz = [](const int16_t *q, int first, int dc_f, int ac_f) {
          for (int k = first; k < 16; ++k)
            if (int16_t(q[k] * (k == 0 ? dc_f : ac_f)) != 0) return true;
          return false;
        };
        uint32_t raw = 0, nz = 0;  // bit 0: Y2, 1..16: Y, 17..20: U, 21..24: V
        if (has_y2) {
          if (WriteBlock(tok, probs->coef, 1, nz_ay2[size_t(c)] + nz_ly2, 0, blk[0], &too_large)) raw |= 1;
          if (dq_nz(blk[0], 0, dq[VP8R_DQ_Y2_DC], dq[VP8R_DQ_Y2_AC])) nz |= 1;
          nz_ay2[size_t(c)] = nz_ly2 = uint8_t(nz & 1);
        }
        for (int b = 0; b < 16; ++b) {
          const int i = b >> 2, j = b & 3;
          const int a = i ? int((raw >> (b - 3)) & 1) : nz_ay[size_t(c) * 4 + j];
          const int l = j ? int((raw >> b) & 1) : nz_ly[i];
          if (WriteBlock(tok, probs->coef, has_y2 ? 0 : 3, a + l, has_y2 ? 1 : 0, blk[1 + b], &too_large)) raw |= 2u << b;
          if (dq_nz(blk[1 + b], has_y2 ? 1 : 0, dq[VP8R_DQ_Y1_DC], dq[VP8R_DQ_Y1_AC])) nz |= 2u << b;
        }
        for (int pl = 0; pl < 2; ++pl) {
          uint8_t *na = pl ? &nz_av[size_t(c) * 2] : &nz_au[size_t(c) * 2];
          uint8_t *nl = pl ? nz_lv : nz_lu;
          const int base = 17 + 4 * pl;
          for (int b = 0; b < 4; ++b) {
            const int i = b >> 1, j = b & 1;
            const int a = i ? int((raw >> (base + b - 2)) & 1) : na[j];
            const int l = j ? int((raw >> (base + b - 1)) & 1) : nl[i];
            if (WriteBlock(tok, probs->coef, 2, a + l, 0, blk[base + b], &too_large)) raw |= 1u << (base + b);
            if (dq_nz(blk[base + b], 0, dq[VP8R_DQ_UV_DC], dq[VP8R_DQ_UV_AC])) nz |= 1u << (base + b);
          }
        }
        if (too_large) return fail("vp8r_frame_write_bitstream: a coefficient exceeds the largest token (2048 + 66)");
        for (int j = 0; j < 4; ++j) nz_ay[size_t(c) * 4 + j] = uint8_t((nz >> (13 + j)) & 1);
        for (int i = 0; i < 4; ++i) nz_ly[i] = uint8_t((nz >> (4 + i * 4)) & 1);
        for (int j = 0; j < 2; ++j) {
          nz_au[size_t(c) * 2 + j] = uint8_t((nz >> (19 + j)) & 1);
          nz_av[size_t(c) * 2 + j] = uint8_t((nz >> (23 + j)) & 1);
        }
        for (int i = 0; i < 2; ++i) {
          nz_lu[i] = uint8_t((nz >> (18 + i * 2)) & 1);
          nz_lv[i] = uint8_t((nz >> (22 + i * 2)) & 1);
        }
      } else {
        if (has_y2) nz_ay2[size_t(c)] = nz_ly2 = 0;
        for (int j = 0; j < 4; ++j) nz_ay[size_t(c) * 4 + j] = nz_ly[j] = 0;
        for (int j = 0; j < 2; ++j) nz_au[size_t(c) * 2 + j] = nz_av[size_t(c) * 2 + j] = nz_lu[j] = nz_lv[j] = 0;
      }
    }
  }

  const std::vector<uint8_t> first = hdr.Finish(), tokens = tok.Finish();
  if (first.size() >= (1u << 19)) return fail("vp8r_frame_write_bitstream: first partition too large for the frame tag");
  out->clear();
  const uint32_t tag = (key ? 0u : 1u) | (uint32_t(h.version) << 1) | (uint32_t(h.show_frame ? 1 : 0) << 4) |
                       (uint32_t(first.size()) << 5);
  out->push_back(uint8_t(tag));
  out->push_back(uint8_t(tag >> 8));
  out->push_back(uint8_t(tag >> 16));
  if (key) {
    const uint8_t sc[3] = {0x9d, 0x01, 0x2a};
    out->insert(out->end(), sc, sc + 3);
    out->push_back(uint8_t(h.width));
    out->push_back(uint8_t((h.width >> 8) & 0x3f));
    out->push_back(uint8_t(h.height));
    out->push_back(uint8_t((h.height >> 8) & 0x3f));
  }
  out->insert(out->end(), first.begin(), first.end());
  out->insert(out->end(), tokens.begin(), tokens.end());
  return VP8R_OK;
}

}  // namespace vp8r
