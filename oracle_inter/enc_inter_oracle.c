/*
 * enc_inter_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE (liboracle_inter.so; only tests/ load it).
 *
 * CPU restatement of the inter-frame encoder's macroblock path (K_encode_inter, vp8_b200/csrc/cuda/enc_kernels.cu),
 * next to the decoder restatement it predicts from.  It is compiled as one unit with oracle/recon_oracle.c (which
 * brings oracle/enc_oracle.c along), so that it uses that file's inter prediction (predict_inter4x4, the reference's
 * six-tap filter and edge clamp) and reads the LAST frame of an oracle_decoder directly: the library exports the whole
 * oracle API plus oracle_encode_inter_frame, and a test uses one library for the decoder and the encoder.
 * The cost (lambda, vector bits, refinement ring) comes from the header the kernel uses.
 */
#include "../oracle/recon_oracle.c"
#include "../vp8_b200/csrc/cuda/enc_cost.h"

int oracle_encode_inter_frame(const oracle_decoder *d, const uint8_t *sy, const uint8_t *su, const uint8_t *sv, int cols, int rows,
                              const int16_t dq[6], int q_index, int lf_level, int search_range, vp8r_mb_info *mbs, int16_t *payload);
int oracle_search_full_pel(const oracle_decoder *d, const uint8_t *sy, int cols, int rows, int y1_ac, int search_range,
                           int16_t *mv);

/* Six-tap prediction of the 16x16 luma block of macroblock (r, c) for the vector (mvr, mvc) in 1/8 pel, as the
 * decoder predicts it (predict_inter4x4 per 4x4 block, reference clamped at the plane's edges). */
static void enc_predict_luma(const ofrm *ref, int r, int c, int mvr, int mvc, uint8_t pred[256]) {
  for (int b = 0; b < 16; b++)
    predict_inter4x4(pred + (b >> 2) * 64 + (b & 3) * 4, 16, ref->y, ref->ys, ref->yh, ref->ys, 16 * r + 4 * (b >> 2),
                     16 * c + 4 * (b & 3), mvr, mvc, k_sixtap);
}

/* Full-pel search of macroblock (r, c) over |dy|, |dx| <= R: the minimum of (cost << 12) | index with
 * index = (dy + R) * (2R + 1) + dx + R, reference pixels clamped to the MB-aligned plane. */
static uint32_t enc_full_pel(const ofrm *ref, const uint8_t *src, int ys, int r, int c, int R, int lambda) {
  const int span = 2 * R + 1;
  uint32_t best = 0xffffffffu;
  for (int i = 0; i < span * span; i++) {
    const int dy = i / span - R, dx = i % span - R;
    uint32_t sad = 0;
    for (int y = 0; y < 16; y++)
      for (int x = 0; x < 16; x++) {
        int dd = (int)src[y * ys + x] - ref_px(ref->y, ref->ys, ref->yh, ref->ys, 16 * r + y + dy, 16 * c + x + dx);
        sad += (uint32_t)(dd < 0 ? -dd : dd);
      }
    const uint32_t key = ((sad + (uint32_t)(lambda * vp8r_enc_mv_bits(4 * dy, 4 * dx))) << 12) | (uint32_t)i;
    if (key < best) best = key;
  }
  return best;
}

static uint32_t enc_sad16(const uint8_t *src, int ss, const uint8_t pred[256]) {
  uint32_t sad = 0;
  for (int y = 0; y < 16; y++)
    for (int x = 0; x < 16; x++) {
      int d = (int)src[y * ss + x] - (int)pred[y * 16 + x];
      sad += (uint32_t)(d < 0 ? -d : d);
    }
  return sad;
}

/* The inter-frame encoder's macroblock path (K_encode_inter, vp8_b200/csrc/cuda/enc_kernels.cu) restated: for every
 * macroblock, full-pel search over |dy|, |dx| <= search_range against d's LAST frame (which is macroblock aligned),
 * minimum of (cost << 12) | index with index = (dy + R) * (2R + 1) + dx + R; then half-pel and quarter-pel
 * refinement over the eight neighbours of the best in enc_cost.h's ring order (the centre wins a tie, then the lowest
 * neighbour); then the luma and chroma prediction of the vector, residual, forward DCT / WHT and quantisation.
 * Writes records WITHOUT mode bits (IS_INTER, ref LAST, HAS_Y2, lf_level, LF_INNER exactly when coef_mask != 0;
 * mv in 1/8 pel) and the non-zero blocks at payload block 25*m.  Source planes: strides cols*16 / cols*8.
 * Returns 0, or -1 when d has no LAST frame of this size. */
int oracle_encode_inter_frame(const oracle_decoder *d, const uint8_t *sy, const uint8_t *su, const uint8_t *sv, int cols, int rows,
                              const int16_t dq[6], int q_index, int lf_level, int search_range, vp8r_mb_info *mbs, int16_t *payload) {
  (void)q_index; /* lambda is a function of the luma AC factor of q_index, dq[VP8R_DQ_Y1_AC] */
  const ofrm *ref = d->ref[1];
  if (!d->have_frame || !ref || ref->cols != cols || ref->rows != rows) return -1;
  const int ys = cols * 16, cs = cols * 8, R = search_range, span = 2 * R + 1;
  const int lambda = vp8r_enc_lambda(dq[VP8R_DQ_Y1_AC]);
  uint8_t pred[256];
  for (int r = 0; r < rows; r++)
    for (int c = 0; c < cols; c++) {
      const int m = r * cols + c;
      const uint8_t *src = sy + (size_t)(16 * r) * ys + 16 * c;
      const uint32_t best = enc_full_pel(ref, src, ys, r, c, R, lambda);
      int qr = 4 * ((int)(best & 4095u) / span - R), qc = 4 * ((int)(best & 4095u) % span - R);
      uint32_t centre = best >> 12;
      /* half pel, quarter pel */
      for (int step = 2; step >= 1; step >>= 1) {
        uint32_t kbest = centre << 4;
        for (int k = 0; k < 8; k++) {
          const int cr = qr + step * vp8r_enc_ring_dr(k), cc = qc + step * vp8r_enc_ring_dc(k);
          enc_predict_luma(ref, r, c, 2 * cr, 2 * cc, pred);
          const uint32_t cost = enc_sad16(src, ys, pred) + (uint32_t)(lambda * vp8r_enc_mv_bits(cr, cc));
          const uint32_t key = (cost << 4) | (uint32_t)(k + 1);
          if (key < kbest) kbest = key;
        }
        const int won = (int)(kbest & 15u);
        if (won) {
          qr += step * vp8r_enc_ring_dr(won - 1);
          qc += step * vp8r_enc_ring_dc(won - 1);
        }
        centre = kbest >> 4;
      }
      const int mvr = 2 * qr, mvc = 2 * qc;
      /* prediction of the vector: luma, and chroma with the decoder's derivation (predict_inter_mb) */
      enc_predict_luma(ref, r, c, mvr, mvc, pred);
      uint8_t cpred[2][64];
      {
        const int16_t sr = (int16_t)(4 * mvr), sc = (int16_t)(4 * mvc);
        const int dr = sr >= 0 ? (sr + 4) / 8 : (sr - 4) / 8, dc = sc >= 0 ? (sc + 4) / 8 : (sc - 4) / 8;
        for (int b = 0; b < 4; b++) {
          const int i = b >> 1, j = b & 1;
          predict_inter4x4(cpred[0] + i * 32 + j * 4, 8, ref->u, ref->cs, ref->ch, ref->cs, 8 * r + 4 * i, 8 * c + 4 * j, dr, dc, k_sixtap);
          predict_inter4x4(cpred[1] + i * 32 + j * 4, 8, ref->v, ref->cs, ref->ch, ref->cs, 8 * r + 4 * i, 8 * c + 4 * j, dr, dc, k_sixtap);
        }
      }
      int16_t blk[25][16];
      for (int b = 0; b < 24; b++) {
        const uint8_t *s, *p;
        int st, pst;
        if (b < 16) {
          s = src + (size_t)(4 * (b >> 2)) * ys + 4 * (b & 3), st = ys;
          p = pred + 4 * (b >> 2) * 16 + 4 * (b & 3), pst = 16;
        } else {
          const int k = (b - 16) & 3;
          s = (b < 20 ? su : sv) + (size_t)(8 * r + 4 * (k >> 1)) * cs + 8 * c + 4 * (k & 1), st = cs;
          p = cpred[b >= 20] + 4 * (k >> 1) * 8 + 4 * (k & 1), pst = 8;
        }
        for (int i = 0; i < 4; i++)
          for (int j = 0; j < 4; j++) blk[b + 1][i * 4 + j] = (int16_t)((int)s[i * st + j] - (int)p[i * pst + j]);
        oracle_fdct4x4(blk[b + 1]);
      }
      for (int b = 0; b < 16; b++) blk[0][b] = blk[b + 1][0];
      oracle_fwht4x4(blk[0]);
      oracle_quantize(blk[0], dq[VP8R_DQ_Y2_DC], dq[VP8R_DQ_Y2_AC]);
      for (int b = 1; b <= 16; b++) {
        oracle_quantize(blk[b], dq[VP8R_DQ_Y1_DC], dq[VP8R_DQ_Y1_AC]);
        blk[b][0] = 0; /* the DC travels in the Y2 block */
      }
      for (int b = 17; b <= 24; b++) oracle_quantize(blk[b], dq[VP8R_DQ_UV_DC], dq[VP8R_DQ_UV_AC]);
      vp8r_mb_info *mb = &mbs[m];
      memset(mb, 0, sizeof(*mb));
      mb->coef_offset = (uint32_t)m * 25u;
      int16_t *dst = payload + (size_t)mb->coef_offset * 16;
      for (int b = 0; b < 25; b++) {
        int any = 0;
        for (int i = 0; i < 16; i++) any |= blk[b][i] != 0;
        if (any) {
          mb->coef_mask |= 1u << b;
          memcpy(dst, blk[b], 32);
          dst += 16;
        }
      }
      mb->flags = VP8R_MB_IS_INTER | (1u << VP8R_MB_REF_SHIFT) | VP8R_MB_HAS_Y2 | ((uint32_t)lf_level << VP8R_MB_LF_SHIFT) |
                  (mb->coef_mask ? VP8R_MB_LF_INNER : 0u);
      mb->mv[0] = (int16_t)mvr;
      mb->mv[1] = (int16_t)mvc;
    }
  return 0;
}

/* The full-pel stage alone, as oracle_encode_inter_frame runs it (lambda from the luma AC factor y1_ac): mv[2m],
 * mv[2m+1] = (dy, dx) in whole pixels of macroblock m.  Returns 0, or -1 when d has no LAST frame of this size. */
int oracle_search_full_pel(const oracle_decoder *d, const uint8_t *sy, int cols, int rows, int y1_ac, int search_range,
                           int16_t *mv) {
  const ofrm *ref = d->ref[1];
  if (!d->have_frame || !ref || ref->cols != cols || ref->rows != rows) return -1;
  const int ys = cols * 16, R = search_range, span = 2 * R + 1, lambda = vp8r_enc_lambda(y1_ac);
  for (int r = 0; r < rows; r++)
    for (int c = 0; c < cols; c++) {
      const int i = (int)(enc_full_pel(ref, sy + (size_t)(16 * r) * ys + 16 * c, ys, r, c, R, lambda) & 4095u);
      mv[2 * (r * cols + c)] = (int16_t)(i / span - R);
      mv[2 * (r * cols + c) + 1] = (int16_t)(i % span - R);
    }
  return 0;
}
