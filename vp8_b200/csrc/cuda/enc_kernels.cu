// K_encode: closed-loop key-frame encoder (row f4 of SURVEY.md section 8): intra mode decision by squared error,
// forward DCT / WHT, quantisation, and the decoder's own reconstruction, one warp per macroblock.
//
// Replaces (the reference only sketches its encoder; these are the functions it has):
//   PickIntraModeLuma / PickIntraModeChroma, PickIntraSubBlockModeSB/MB (B_PRED)   src/encode_frame.cc:30-76,109-238
//   TransformResidual, QuantizeResidualValue                      src/residual.cc:5-40,96-108
//   DCT, WHT, Quantize                                            src/dct.cc:5-65, src/quantizer.cc:5-8
// and produces the SAME per-macroblock arrays the decode path consumes (vp8r_mb_info + coefficient blocks), so that
// the loop filter and the reference-buffer bookkeeping of the decoder run on them unchanged and a host writer
// (host/frame_writer.cc) can turn them into a VP8 key frame.
//
// Mapping: one CTA per frame, one warp per macroblock row, rows advance as a wavefront (a macroblock is predicted
// from RECONSTRUCTED pixels of its left / above neighbours, so row r may do column c once row r-1 has finished
// column c+1).  Lane b < 24 owns 4x4 block b (16 Y raster, 4 U, 4 V), lane 24 the Y2 block.  Everything of a block
// stays in the lane's registers: source pixels, the four candidate predictions and their errors (summed over the
// warp with REDUX), residual, forward DCT, quantisation, dequantisation, inverse DCT, reconstruction.
#include "enc_cost.h"
#include "recon_kernels.h"

namespace vp8r {

namespace {

__device__ __forceinline__ int s16e(int x) { return (int)(short)x; }
__device__ __forceinline__ int clamp255e(int x) { return min(max(x, 0), 255); }

// src/dct.cc:5-32: rows first (inputs << 3), then columns; int16 between and after the passes.
__device__ __forceinline__ void Fdct4x4(int *m) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int *r = m + 4 * i;
    const int a = (r[0] + r[3]) << 3, b = (r[1] + r[2]) << 3, c = (r[1] - r[2]) << 3, d = (r[0] - r[3]) << 3;
    r[0] = s16e(a + b);
    r[2] = s16e(a - b);
    r[1] = s16e((c * 2217 + d * 5352 + 14500) >> 12);
    r[3] = s16e((d * 2217 - c * 5352 + 7500) >> 12);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int a = m[i] + m[12 + i], b = m[4 + i] + m[8 + i], c = m[4 + i] - m[8 + i], d = m[i] - m[12 + i];
    m[i] = s16e((a + b + 7) >> 4);
    m[8 + i] = s16e((a - b + 7) >> 4);
    m[4 + i] = s16e(((c * 2217 + d * 5352 + 12000) >> 16) + (d != 0 ? 1 : 0));
    m[12 + i] = s16e((d * 2217 - c * 5352 + 51000) >> 16);
  }
}

// src/dct.cc:34-65
__device__ __forceinline__ void Fwht4x4(int *m) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int *r = m + 4 * i;
    const int a = (r[0] + r[2]) << 2, d = (r[1] + r[3]) << 2, c = (r[1] - r[3]) << 2, b = (r[0] - r[2]) << 2;
    r[0] = s16e(a + d + (a != 0 ? 1 : 0));
    r[1] = s16e(b + c);
    r[2] = s16e(b - c);
    r[3] = s16e(a - d);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int a = m[i] + m[8 + i], d = m[4 + i] + m[12 + i], c = m[4 + i] - m[12 + i], b = m[i] - m[8 + i];
    int a2 = a + d, b2 = b + c, c2 = b - c, d2 = a - d;
    a2 += a2 < 0;
    b2 += b2 < 0;
    c2 += c2 < 0;
    d2 += d2 < 0;
    m[i] = s16e((a2 + 3) >> 3);
    m[4 + i] = s16e((b2 + 3) >> 3);
    m[8 + i] = s16e((c2 + 3) >> 3);
    m[12 + i] = s16e((d2 + 3) >> 3);
  }
}

// The decoder's inverse transforms (src/dct.cc:67-133), as in recon_kernels.cu.
__device__ __forceinline__ void IdctE(int *m) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int a = m[i] + m[8 + i], b = m[i] - m[8 + i];
    int t1 = (m[4 + i] * 35468) >> 16;
    int t2 = m[12 + i] + ((m[12 + i] * 20091) >> 16);
    int c = t1 - t2;
    t1 = m[4 + i] + ((m[4 + i] * 20091) >> 16);
    t2 = (m[12 + i] * 35468) >> 16;
    int d = t1 + t2;
    m[i] = s16e(a + d);
    m[12 + i] = s16e(a - d);
    m[4 + i] = s16e(b + c);
    m[8 + i] = s16e(b - c);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int *r = m + 4 * i;
    int a = r[0] + r[2], b = r[0] - r[2];
    int t1 = (r[1] * 35468) >> 16;
    int t2 = r[3] + ((r[3] * 20091) >> 16);
    int c = t1 - t2;
    t1 = r[1] + ((r[1] * 20091) >> 16);
    t2 = (r[3] * 35468) >> 16;
    int d = t1 + t2;
    r[0] = s16e((a + d + 4) >> 3);
    r[3] = s16e((a - d + 4) >> 3);
    r[1] = s16e((b + c + 4) >> 3);
    r[2] = s16e((b - c + 4) >> 3);
  }
}
__device__ __forceinline__ void IwhtE(int *m) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int a = m[i] + m[12 + i], b = m[4 + i] + m[8 + i];
    int c = m[4 + i] - m[8 + i], d = m[i] - m[12 + i];
    m[i] = s16e(a + b);
    m[4 + i] = s16e(c + d);
    m[8 + i] = s16e(a - b);
    m[12 + i] = s16e(d - c);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int *r = m + 4 * i;
    int a = r[0] + r[3], b = r[1] + r[2];
    int c = r[1] - r[2], d = r[0] - r[3];
    r[0] = s16e((a + b + 3) >> 3);
    r[1] = s16e((c + d + 3) >> 3);
    r[2] = s16e((a - b + 3) >> 3);
    r[3] = s16e((d - c + 3) >> 3);
  }
}

constexpr int kEncWarps = 16;

// Per-warp scratch.  tile: the B_PRED trial's view of the macroblock, as the decoder's PredictBpred lays it out: row 0 =
// the pixel row above (columns -1..19 at bytes 3..23), byte 3 of rows 1..16 = the column to the left, the macroblock
// itself at rows 1..16, bytes 4..19.
struct __align__(16) EncScratch {
  short y2[16];
  short xfer[16];            // one 4x4 block on its way between the pixel lanes and the transform lane
  short cand[16][16];        // quantised blocks of the B_PRED trial
  unsigned char tile[17][32];
};

// B_PRED gather table, as recon_kernels.cu's c_bpred_lut: [mode][pixel] -> i0 | i1<<4 | i2<<8 | kind<<12 over the edge
// array E = {L3,L2,L1,L0,P,A0..A7}; kind 0: (E[i0]+2E[i1]+E[i2]+2)>>2, 1: (E[i0]+E[i2]+1)>>1, 2: DC, 3: TM.
__constant__ unsigned short c_enc_bpred_lut[10 * 16];

// Prediction of this lane's 4x4 block for one 16x16 / 8x8 mode (src/intra_predict.cc:6-98): aw = the four pixels
// above the block's columns in the macroblock's top edge, l[k] = the pixel left of row k in its left edge.
__device__ __forceinline__ void PredictRows(int mode, unsigned aw, const int *l, int P, int dc, unsigned *rows) {
  if (mode == 1) {
    rows[0] = rows[1] = rows[2] = rows[3] = aw;
  } else if (mode == 2) {
#pragma unroll
    for (int k = 0; k < 4; ++k) rows[k] = (unsigned)l[k] * 0x01010101u;
  } else if (mode == 0) {
    rows[0] = rows[1] = rows[2] = rows[3] = (unsigned)dc * 0x01010101u;
  } else {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      unsigned o = 0;
#pragma unroll
      for (int x = 0; x < 4; ++x) o |= (unsigned)clamp255e(l[k] + (int)((aw >> (8 * x)) & 0xff) - P) << (8 * x);
      rows[k] = o;
    }
  }
}

__device__ __forceinline__ unsigned Sse4(const unsigned *rows, const unsigned *src) {
  unsigned e = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const unsigned d = __vabsdiffu4(rows[k], src[k]);  // |difference| per pixel
    e = __dp4a(d, d, e);                               // sum of squares
  }
  return e;
}


// B_PRED trial of one macroblock by one warp (src/encode_frame.cc:109-202 for the decision, the decoder's PredictBpred
// for the edges): sub-block by sub-block in raster order, closed loop inside the macroblock.  Lanes 0..15 are the
// pixels of the sub-block and try modes 0..4, lanes 16..31 the same pixels for modes 5..9; lane 0 transforms.
// Returns the sum of the sixteen best prediction errors; s.cand holds the quantised blocks (DC in place), s.tile the
// reconstruction, aux[2] the sixteen sub-block modes.
__device__ __forceinline__ unsigned BpredTrial(const DevFrameJob &job, int r, int c, int lane, const unsigned (&src)[4],
                                               int f_dc, int f_ac, EncScratch &s, const unsigned short *lut, unsigned (&aux)[2]) {
  const int pitch = job.pitch_y;
  const uint8_t *mbp = job.cur.y + (ptrdiff_t)(r * 16) * pitch + c * 16;
  if (lane < 21) {
    const int col = lane - 1;
    int v;
    if (r == 0) v = 127;
    else if (col < 0) v = c == 0 ? 129 : *reinterpret_cast<const volatile uint8_t *>(mbp - pitch - 1);
    else if (col >= 16 && c + 1 == job.mb_cols) v = *reinterpret_cast<const volatile uint8_t *>(mbp - pitch + 15);
    else v = *reinterpret_cast<const volatile uint8_t *>(mbp - pitch + col);
    s.tile[0][4 + col] = (unsigned char)v;
  }
  if (lane < 16) s.tile[1 + lane][3] = (unsigned char)(c == 0 ? 129 : *reinterpret_cast<const volatile uint8_t *>(mbp + (ptrdiff_t)lane * pitch - 1));
  __syncwarp();

  const int px = lane & 3, py = (lane >> 2) & 3, half = lane >> 4;
  unsigned total = 0;
  aux[0] = aux[1] = 0;
  for (int b = 0; b < 16; ++b) {
    const int i = b >> 2, j = b & 3;
    int E = 0;  // edge array, one entry per lane 0..12
    if (lane < 4) E = s.tile[1 + 4 * i + (3 - lane)][3 + 4 * j];
    else if (lane < 9) E = s.tile[4 * i][3 + 4 * j + (lane - 4)];
    else if (lane < 13) E = s.tile[(j == 3) ? 0 : 4 * i][3 + 4 * j + (lane - 4)];
    const int dc_in = (lane < 4 || (lane >= 5 && lane < 9)) ? E : 0;
    const int dc = (int)(__reduce_add_sync(0xffffffffu, (unsigned)dc_in) + 4u) >> 3;
    // this lane's source pixel: block b's rows live in lane b
    const unsigned w0 = __shfl_sync(0xffffffffu, src[0], b), w1 = __shfl_sync(0xffffffffu, src[1], b);
    const unsigned w2 = __shfl_sync(0xffffffffu, src[2], b), w3 = __shfl_sync(0xffffffffu, src[3], b);
    const unsigned wsel = py == 0 ? w0 : (py == 1 ? w1 : (py == 2 ? w2 : w3));
    const int pix = (int)((wsel >> (8 * px)) & 0xffu);
    unsigned best_lo = 0xffffffffu, best_hi = 0xffffffffu;
    int mode_lo = 0, mode_hi = 5, v_best = 0;
#pragma unroll 1
    for (int t = 0; t < 5; ++t) {
      const unsigned e = lut[(t + 5 * half) * 16 + (lane & 15)];
      const int x0 = __shfl_sync(0xffffffffu, E, e & 15), x1 = __shfl_sync(0xffffffffu, E, (e >> 4) & 15);
      const int x2 = __shfl_sync(0xffffffffu, E, (e >> 8) & 15);
      const int kind = e >> 12;
      int v;
      if (kind == 0) v = (x0 + 2 * x1 + x2 + 2) >> 2;
      else if (kind == 1) v = (x0 + x2 + 1) >> 1;
      else if (kind == 2) v = dc;
      else v = clamp255e(x0 + x1 - x2);
      const int d = v - pix;
      const unsigned se = (unsigned)(d * d);
      const unsigned e_lo = __reduce_add_sync(0xffffffffu, half ? 0u : se), e_hi = __reduce_add_sync(0xffffffffu, half ? se : 0u);
      if (e_lo < best_lo) {
        best_lo = e_lo;
        mode_lo = t;
        if (!half) v_best = v;
      }
      if (e_hi < best_hi) {
        best_hi = e_hi;
        mode_hi = t + 5;
        if (half) v_best = v;
      }
    }
    const bool hi_wins = best_hi < best_lo;  // the ten modes in order, a later one only when strictly better
    const int mode = hi_wins ? mode_hi : mode_lo;
    total += hi_wins ? best_hi : best_lo;
    const int pred = __shfl_sync(0xffffffffu, v_best, (lane & 15) + (hi_wins ? 16 : 0));
    if (b < 8) aux[0] |= (unsigned)mode << (4 * b);
    else aux[1] |= (unsigned)mode << (4 * (b - 8));
    if (lane < 16) s.xfer[lane] = (short)(pix - pred);
    __syncwarp();
    if (lane == 0) {  // forward transform, quantisation, and the decoder's way back
      int m[16];
#pragma unroll
      for (int k = 0; k < 16; ++k) m[k] = s.xfer[k];
      Fdct4x4(m);
      m[0] = s16e(m[0] / f_dc);
#pragma unroll
      for (int k = 1; k < 16; ++k) m[k] = s16e(m[k] / f_ac);
      uint4 *cand = reinterpret_cast<uint4 *>(s.cand[b]);
      unsigned w[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) w[k] = ((unsigned)m[2 * k] & 0xffffu) | ((unsigned)m[2 * k + 1] << 16);
      cand[0] = make_uint4(w[0], w[1], w[2], w[3]);
      cand[1] = make_uint4(w[4], w[5], w[6], w[7]);
      m[0] = s16e(m[0] * f_dc);
#pragma unroll
      for (int k = 1; k < 16; ++k) m[k] = s16e(m[k] * f_ac);
      IdctE(m);  // (a block with only its DC comes out as (dc + 4) >> 3 everywhere, the decoder's short cut)
#pragma unroll
      for (int k = 0; k < 16; ++k) s.xfer[k] = (short)m[k];
    }
    __syncwarp();
    if (lane < 16) s.tile[1 + 4 * i + py][4 + 4 * j + px] = (unsigned char)clamp255e(s16e(pred + s.xfer[lane]));
    __syncwarp();
  }
  return total;
}

// What one lane of an intra warp owns for the whole frame: lane b < 24 the 4x4 block b (16 Y raster, 4 U, 4 V),
// lane 24 the Y2 block; the plane it predicts into and the source plane it reads; its quantiser factors.
struct IntraLane {
  bool luma, is_block;
  int n4, first, bi, bj, pitch, spitch, n, f_dc, f_ac;
  uint8_t *plane;
  const uint8_t *splane;
};

__device__ __forceinline__ IntraLane MakeIntraLane(const DevFrameJob &job, int lane) {
  IntraLane L;
  L.luma = lane < 16;
  L.n4 = L.luma ? 4 : 2;
  L.first = L.luma ? 0 : (lane < 20 ? 16 : 20);
  const int b = lane - L.first;
  L.bi = L.luma ? (b >> 2) : (b >> 1);
  L.bj = L.luma ? (b & 3) : (b & 1);
  L.pitch = L.luma ? job.pitch_y : job.pitch_c;
  L.spitch = L.luma ? job.enc_src_pitch_y : job.enc_src_pitch_c;
  L.plane = L.luma ? job.cur.y : (lane < 20 ? job.cur.u : job.cur.v);
  L.splane = L.luma ? job.enc_src[0] : (lane < 20 ? job.enc_src[1] : job.enc_src[2]);
  L.n = L.luma ? 16 : 8;
  L.is_block = lane < 24;
  const int16_t *dq = job.dq[0];
  L.f_dc = lane == 24 ? dq[VP8R_DQ_Y2_DC] : (L.luma ? dq[VP8R_DQ_Y1_DC] : dq[VP8R_DQ_UV_DC]);
  L.f_ac = lane == 24 ? dq[VP8R_DQ_Y2_AC] : (L.luma ? dq[VP8R_DQ_Y1_AC] : dq[VP8R_DQ_UV_AC]);
  return L;
}

// One macroblock of the closed-loop intra coder, by one warp, once its left, above-left, above and above-right
// neighbours are final in job.cur: the mode decision on those neighbours, then the commit (residual, forward
// transforms, quantisation, record and blocks, the decoder's reconstruction in place).  kGated (intra macroblocks of
// inter frames): the commit happens only when the macroblock's intra error plus vp8r_enc_intra_bias is strictly below
// inter_err; otherwise nothing of the frame is touched.  Returns whether it committed.
template <bool kGated>
__device__ __forceinline__ bool EncodeIntraMb(const DevFrameJob &job, const IntraLane &L, int lane, int r, int c, bool try_bpred,
                                              EncScratch &s, const unsigned short *lut, unsigned inter_err) {
  const bool luma = L.luma, is_block = L.is_block;
  const int n4 = L.n4, first = L.first, bi = L.bi, bj = L.bj, pitch = L.pitch, spitch = L.spitch, n = L.n;
  const int f_dc = L.f_dc, f_ac = L.f_ac;
  const int cols = job.mb_cols;
  short *const y2_slot = s.y2;
  const int16_t *dq = job.dq[0];
  uint8_t *mbp = L.plane + (ptrdiff_t)(r * n) * pitch + c * n;
  const uint8_t *sp = L.splane + (ptrdiff_t)(r * n + 4 * bi) * spitch + c * n + 4 * bj;
  const bool have_above = r > 0, have_left = c > 0;
  unsigned src[4] = {0, 0, 0, 0}, aw = 0x7f7f7f7fu;
  int l[4] = {129, 129, 129, 129};
  int P = have_above ? (have_left ? 0 : 129) : 127;
  if (is_block) {
#pragma unroll
    for (int k = 0; k < 4; ++k) src[k] = *reinterpret_cast<const unsigned *>(sp + (ptrdiff_t)k * spitch);
    if (have_above) aw = *reinterpret_cast<const volatile unsigned *>(mbp - pitch + 4 * bj);
    if (have_left) {
#pragma unroll
      for (int k = 0; k < 4; ++k) l[k] = *reinterpret_cast<const volatile uint8_t *>(mbp + (ptrdiff_t)(4 * bi + k) * pitch - 1);
    }
    if (have_above && have_left) P = *reinterpret_cast<const volatile uint8_t *>(mbp - pitch - 1);
  }
  // DC value: sums over the whole top edge / left edge of the plane's macroblock
  int dc = 128;
  {
    const int sum_a = (int)__dp4a(aw, 0x01010101u, 0u), sum_l = l[0] + l[1] + l[2] + l[3];
    int tot_a = 0, tot_l = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int va = __shfl_sync(0xffffffffu, sum_a, first + (k < n4 ? k : 0));
      const int vl = __shfl_sync(0xffffffffu, sum_l, first + (k < n4 ? k * n4 : 0));
      if (k < n4) {
        tot_a += va;
        tot_l += vl;
      }
    }
    if (have_above || have_left) {
      const int shf = (luma ? 3 : 2) + (have_above ? 1 : 0) + (have_left ? 1 : 0);
      dc = ((have_above ? tot_a : 0) + (have_left ? tot_l : 0) + (1 << (shf - 1))) >> shf;
    }
  }
  // ---- mode decision: V, H, DC, TM in the reference's order, a later one only when strictly better ----
  int ymode = 0, uvmode = 0;
  unsigned best_y = 0xffffffffu;
  {
    unsigned best_c = 0xffffffffu;
    const int order[4] = {1, 2, 0, 3};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      unsigned rows4[4];
      PredictRows(order[k], aw, l, P, dc, rows4);
      const unsigned e = is_block ? Sse4(rows4, src) : 0u;
      const unsigned ey = __reduce_add_sync(0xffffffffu, luma ? e : 0u);
      const unsigned ec = __reduce_add_sync(0xffffffffu, luma ? 0u : e);
      if (ey < best_y) best_y = ey, ymode = order[k];
      if (ec < best_c) best_c = ec, uvmode = order[k];
    }
  }
  // ---- B_PRED last, only when strictly better than the best 16x16 mode (src/encode_frame.cc:233-237) ----
  bool bpred = false;
  unsigned aux[2] = {0, 0};
  unsigned intra_err = best_y;
  if (try_bpred) {
    const int y1_dc = dq[VP8R_DQ_Y1_DC], y1_ac = dq[VP8R_DQ_Y1_AC];
    const unsigned total = BpredTrial(job, r, c, lane, src, y1_dc, y1_ac, s, lut, aux);
    bpred = total < best_y;
    if (bpred) ymode = 4, intra_err = total;
  }
  // ---- intra or inter: strict, so a tie stays inter (warp-uniform: both errors are warp sums) ----
  if (kGated && !(intra_err + (unsigned)vp8r_enc_intra_bias(dq[VP8R_DQ_Y1_AC]) < inter_err)) return false;
  // ---- residual, forward transform, quantisation ----
  unsigned pred[4];
  PredictRows(luma ? ymode : uvmode, aw, l, P, dc, pred);
  int m[16];
  if (bpred && lane <= 24) {  // luma blocks were quantised in the trial (DC in place); there is no Y2 block
#pragma unroll
    for (int i = 0; i < 16; ++i) m[i] = (luma) ? s.cand[lane][i] : 0;
  }
  if (!(bpred && (luma || lane == 24))) {
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
      for (int x = 0; x < 4; ++x) m[4 * k + x] = (int)((src[k] >> (8 * x)) & 0xff) - (int)((pred[k] >> (8 * x)) & 0xff);
    if (is_block) Fdct4x4(m);
  }
  if (!bpred) {
    if (luma) y2_slot[lane] = (short)m[0];
    __syncwarp();
    if (lane == 24) {
#pragma unroll
      for (int i = 0; i < 16; ++i) m[i] = y2_slot[i];
      Fwht4x4(m);
    }
    __syncwarp();
  }
  bool nz = false;
  if (lane <= 24) {
    if (!(bpred && (luma || lane == 24))) {
      m[0] = luma ? 0 : s16e(m[0] / f_dc);  // a luma block's DC travels in the Y2 block
#pragma unroll
      for (int i = 1; i < 16; ++i) m[i] = s16e(m[i] / f_ac);
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) nz |= m[i] != 0;
  }
  const unsigned lanes_nz = __ballot_sync(0xffffffffu, nz);
  const unsigned coef_mask = ((lanes_nz & 0x00ffffffu) << 1) | ((lanes_nz >> 24) & 1u);
  const int mb_index = r * cols + c;
  const unsigned coef_offset = (unsigned)mb_index * 25u;
  if (nz) {
    const int blk = lane < 24 ? lane + 1 : 0;
    const int at = __popc(coef_mask & ((1u << blk) - 1u));
    int4 *dst = reinterpret_cast<int4 *>(const_cast<int16_t *>(job.payload) + (size_t)(coef_offset + at) * 16);
    unsigned w[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) w[i] = ((unsigned)m[2 * i] & 0xffffu) | ((unsigned)m[2 * i + 1] << 16);
    dst[0] = make_int4((int)w[0], (int)w[1], (int)w[2], (int)w[3]);
    dst[1] = make_int4((int)w[4], (int)w[5], (int)w[6], (int)w[7]);
  }
  if (lane == 0) {
    const unsigned flags = ((unsigned)ymode << VP8R_MB_MODE_SHIFT) | ((unsigned)uvmode << VP8R_MB_UVMODE_SHIFT) |
                           (bpred ? 0u : VP8R_MB_HAS_Y2) | ((unsigned)job.lf_level << VP8R_MB_LF_SHIFT) |
                           ((coef_mask || bpred) ? VP8R_MB_LF_INNER : 0u);
    int4 *rec = reinterpret_cast<int4 *>(const_cast<vp8r_mb_info *>(job.mbs) + mb_index);
    rec[0] = make_int4((int)flags, (int)coef_mask, (int)coef_offset, 0);
    rec[1] = make_int4(bpred ? (int)aux[0] : 0, bpred ? (int)aux[1] : 0, 0, 0);
  }
  // ---- reconstruction, exactly as the decoder does it from the stored blocks (WarpResidual) ----
  if (lane <= 24) {
    m[0] = s16e(m[0] * f_dc);
#pragma unroll
    for (int i = 1; i < 16; ++i) m[i] = s16e(m[i] * f_ac);
  }
  bool any = nz && is_block;
  if (bpred) {  // the luma reconstruction stands in the trial's tile
    if (lane < 16) {
      const unsigned *t = reinterpret_cast<const unsigned *>(&s.tile[1 + lane][4]);
      *reinterpret_cast<uint4 *>(mbp + (ptrdiff_t)lane * pitch) = make_uint4(t[0], t[1], t[2], t[3]);
    }
  }
  if (coef_mask & 1u) {
    if (lane == 24) {
      IwhtE(m);
#pragma unroll
      for (int i = 0; i < 16; ++i) y2_slot[i] = (short)m[i];
    }
    __syncwarp();
    if (luma) {
      m[0] = y2_slot[lane];
      any = true;
    }
    __syncwarp();
  }
  if (is_block && !(bpred && luma)) {
    if (any) IdctE(m);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      unsigned v = pred[k];
      if (any) {
        unsigned o = 0;
#pragma unroll
        for (int x = 0; x < 4; ++x) o |= (unsigned)clamp255e(s16e((int)((v >> (8 * x)) & 0xff) + m[4 * k + x])) << (8 * x);
        v = o;
      }
      *reinterpret_cast<unsigned *>(mbp + (ptrdiff_t)(4 * bi + k) * pitch + 4 * bj) = v;
    }
  }
  return true;
}

// Shared memory of the intra wavefront kernels: one progress word per macroblock row, the B_PRED gather table, then
// one EncScratch per warp.
__device__ __forceinline__ void IntraWavefrontSetup(const DevFrameJob &job, unsigned char *smem, volatile int *&progress,
                                                    unsigned short *&lut, EncScratch *&scratch) {
  const int rows = job.mb_rows;
  progress = reinterpret_cast<volatile int *>(smem);
  lut = reinterpret_cast<unsigned short *>(smem + ((rows * 4 + 15) & ~15));
  scratch = reinterpret_cast<EncScratch *>(reinterpret_cast<unsigned char *>(lut) + 320);
  for (int i = threadIdx.x; i < rows; i += blockDim.x) progress[i] = 0;
  for (int i = threadIdx.x; i < 160; i += blockDim.x) lut[i] = c_enc_bpred_lut[i];
  __syncthreads();
}

// Row r may work on column c once row r-1 has finished column c+1 (its above-right neighbour).
__device__ __forceinline__ void WaitForRowAbove(volatile int *progress, int r, int c, int cols) {
  if (r > 0) {
    const int need = min(c + 2, cols);
    while (progress[r - 1] < need) __nanosleep(100);
    __threadfence_block();
  }
}

__device__ __forceinline__ void PublishColumn(volatile int *progress, int r, int c, int lane) {
  __syncwarp();
  __threadfence_block();
  if (lane == 0) progress[r] = c + 1;
}

}  // namespace

__global__ void __launch_bounds__(kEncWarps * 32) EncodeIntraKernel(const DevFrameJob *__restrict__ jobs) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const DevFrameJob &job = jobs[blockIdx.x];
  if (!job.enc_src[0]) return;
  volatile int *progress;
  unsigned short *lut;
  EncScratch *scratch;
  IntraWavefrontSetup(job, smem_raw, progress, lut, scratch);
  const bool try_bpred = (job.enc_flags & VP8R_ENC_BPRED) != 0;
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;  // from lane 0: known to be warp-uniform
  const IntraLane L = MakeIntraLane(job, lane);
  const int rows = job.mb_rows, cols = job.mb_cols;
  for (int r = warp; r < rows; r += kEncWarps) {
    for (int c = 0; c < cols; ++c) {
      WaitForRowAbove(progress, r, c, cols);
      EncodeIntraMb<false>(job, L, lane, r, c, try_bpred, scratch[warp], lut, 0u);
      PublishColumn(progress, r, c, lane);
    }
  }
}

// K_encode_intra_mbs: the intra macroblocks of inter frames (VP8R_ENC_INTRA_MBS).  Runs after K_encode_inter and
// K_inter, on the unfiltered reconstruction they left, in EncodeIntraKernel's wavefront: a macroblock is decided on
// its final neighbours (inter ones as K_inter made them, intra ones as this pass made them) and, when it goes intra,
// overwrites its inter record, blocks and reconstruction in place.  No inter macroblock reads pixels of its own frame,
// so nothing else changes.
__global__ void __launch_bounds__(kEncWarps * 32) EncodeIntraMbsKernel(const DevFrameJob *__restrict__ jobs) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const DevFrameJob &job = jobs[blockIdx.x];
  if (!job.enc_src[0] || !(job.enc_flags & VP8R_ENC_INTRA_MBS)) return;
  volatile int *progress;
  unsigned short *lut;
  EncScratch *scratch;
  IntraWavefrontSetup(job, smem_raw, progress, lut, scratch);
  const bool try_bpred = (job.enc_flags & VP8R_ENC_BPRED) != 0;
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const IntraLane L = MakeIntraLane(job, lane);
  const int rows = job.mb_rows, cols = job.mb_cols;
  const unsigned bias = (unsigned)vp8r_enc_intra_bias(job.dq[0][VP8R_DQ_Y1_AC]);
  for (int r = warp; r < rows; r += kEncWarps) {
    for (int c = 0; c < cols; ++c) {
      const unsigned inter_err = job.enc_inter_err[r * cols + c];
      // Skip rule: intra_err + bias >= bias >= inter_err can never win the strict comparison, so such a macroblock
      // stays inter without a decision, and it reads no neighbour, so it need not wait for the row above either.
      if (!(inter_err <= bias)) {
        WaitForRowAbove(progress, r, c, cols);
        EncodeIntraMb<true>(job, L, lane, r, c, try_bpred, scratch[warp], lut, inter_err);
      }
      PublishColumn(progress, r, c, lane);
    }
  }
}

// ------------------------------------------------------------------------------------------------------------------
// K_encode_inter: inter frames whose macroblocks all predict from LAST with one vector each.  No pixel of such a frame
// depends on another pixel of the same frame, so every macroblock is searched and transformed on its own, one warp
// each, all frames of the batch in one launch; the reconstruction is the decoder's own K_inter on the records written
// here (the host assigns the modes afterwards, from the vectors).
//
// Per macroblock: the source luma and a window of the LAST luma plane (rows -(R+3) .. 15+R+3, columns -32 .. 47
// around the macroblock; the surface's 32-pixel border makes any clamp unnecessary for R <= 24) are staged in shared
// memory by 128-bit loads.  Full-pel search over |dy|, |dx| <= R, candidates split over the lanes, SAD by
// vabsdiff4-with-accumulate, cost = SAD + lambda * R(v) (enc_cost.h), minimum of (cost << 12) | candidate index by
// REDUX (ties: the lowest index, index = (dy + R) * (2R + 1) + dx + R).  Then half-pel and quarter-pel refinement:
// the eight neighbours of the current best (enc_cost.h's ring order, the centre kept on a tie), four lanes per
// candidate, the prediction computed exactly as the decoder computes it (six-tap, horizontal pass over the rows
// -2..+3 around each output row, rounding (x + 64) >> 7 and a clamp to 0..255 after each pass; whole-pel
// positions are the identity filter).  Finally the prediction of luma and of chroma (the decoder's chroma vector
// of a non-SPLIT macroblock), residual, forward DCT / WHT and quantisation as in K_encode.
namespace {

constexpr int kEncInterWarps = 4;
constexpr int kEncSearchMax = 24;
constexpr int kWinTop = kEncSearchMax + 3;       // window row of the macroblock's first row
constexpr int kWinRows = 16 + 2 * kWinTop;       // 70
constexpr int kWinLeft = 32;                     // window column of the macroblock's first column
constexpr int kWinW = 16 + 2 * kWinLeft;         // 80 bytes: five 128-bit words per row

struct __align__(16) EncInterScratch {
  unsigned char win[kWinRows][kWinW];
  unsigned src[64];                 // source luma, row y at words 4y..4y+3
  unsigned pred[64];                // luma prediction of the chosen vector, same layout
  unsigned char cpred[2][8][8];     // U, V prediction
  short y2[16];
};

__constant__ int c_enc_sixtap[8][6] = {  // RFC 6386 section 14.4 (src/inter_predict.h:18-27)
    {0, 0, 128, 0, 0, 0},  {0, -6, 123, 12, -1, 0},   {2, -11, 108, 36, -8, 1}, {0, -9, 93, 50, -6, 0},
    {3, -16, 77, 77, -16, 3}, {0, -6, 50, 93, -9, 0}, {1, -8, 36, 108, -11, 2}, {0, -1, 12, 123, -6, 0}};

__device__ __forceinline__ unsigned Vabsdiff4Add(unsigned a, unsigned b, unsigned c) {
  unsigned d;
  asm("vabsdiff4.u32.u32.u32.add %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}

__device__ __forceinline__ int Tap6(const int *t, int p0, int p1, int p2, int p3, int p4, int p5) {
  return clamp255e((t[0] * p0 + t[1] * p1 + t[2] * p2 + t[3] * p3 + t[4] * p4 + t[5] * p5 + 64) >> 7);
}

// Luma prediction of rows y0..y0+NR-1, columns x0..x0+NC-1 (NC a multiple of 4) of the macroblock for the vector
// (mr, mc) in 1/8 pel, from the staged window.  kStore: into s.pred; otherwise returns the SAD against s.src.
template <int NR, int NC, bool kStore>
__device__ __forceinline__ unsigned PredictLuma(EncInterScratch &s, int mr, int mc, int y0, int x0) {
  int th[6], tv[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    th[k] = c_enc_sixtap[mc & 7][k];
    tv[k] = c_enc_sixtap[mr & 7][k];
  }
  const int row0 = kWinTop + y0 + (mr >> 3) - 2, col0 = kWinLeft + x0 + (mc >> 3) - 2;
  unsigned sad = 0;
#pragma unroll 1
  for (int x4 = 0; x4 < NC; x4 += 4) {
    unsigned out[NR];
#pragma unroll
    for (int y = 0; y < NR; ++y) out[y] = 0;
#pragma unroll
    for (int xx = 0; xx < 4; ++xx) {
      const unsigned char *w = &s.win[row0][col0 + x4 + xx];
      int h[NR + 5];
#pragma unroll
      for (int i = 0; i < NR + 5; ++i) {
        const unsigned char *q = w + i * kWinW;
        h[i] = Tap6(th, q[0], q[1], q[2], q[3], q[4], q[5]);
      }
#pragma unroll
      for (int y = 0; y < NR; ++y) out[y] |= (unsigned)Tap6(tv, h[y], h[y + 1], h[y + 2], h[y + 3], h[y + 4], h[y + 5]) << (8 * xx);
    }
#pragma unroll
    for (int y = 0; y < NR; ++y) {
      const int at = 4 * (y0 + y) + ((x0 + x4) >> 2);
      if (kStore) s.pred[at] = out[y];
      else sad = Vabsdiff4Add(out[y], s.src[at], sad);
    }
  }
  return sad;
}

}  // namespace

__global__ void __launch_bounds__(kEncInterWarps * 32) EncodeInterKernel(const DevFrameJob *__restrict__ jobs) {
  __shared__ EncInterScratch s_scratch[kEncInterWarps];
  const DevFrameJob &job = jobs[blockIdx.z];
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int mb_r = blockIdx.y, mb_c = blockIdx.x * kEncInterWarps + warp, cols = job.mb_cols;
  if (!job.enc_src[0] || mb_r >= job.mb_rows || mb_c >= cols) return;
  EncInterScratch &s = s_scratch[warp];
  const int R = job.enc_search_range;

  // ---- stage the source macroblock and the search window ----
  {
    const int sp = job.enc_src_pitch_y;
    if (lane < 16)
      reinterpret_cast<uint4 *>(s.src)[lane] =
          *reinterpret_cast<const uint4 *>(job.enc_src[0] + (ptrdiff_t)(mb_r * 16 + lane) * sp + mb_c * 16);
    const int r_lo = kWinTop - (R + 3), n_rows = 16 + 2 * (R + 3);
    const uint8_t *ref = job.ref[1].y + (ptrdiff_t)(mb_r * 16 - kWinTop) * job.pitch_y + mb_c * 16 - kWinLeft;
    for (int i = lane; i < n_rows * 5; i += 32) {
      const int row = r_lo + i / 5, q = i % 5;
      reinterpret_cast<uint4 *>(s.win[row])[q] = *reinterpret_cast<const uint4 *>(ref + (ptrdiff_t)row * job.pitch_y + 16 * q);
    }
  }
  __syncwarp();
  const int lambda = vp8r_enc_lambda(job.dq[0][VP8R_DQ_Y1_AC]);

  // ---- full-pel search ----
  unsigned best = 0xffffffffu;
  {
    const int span = 2 * R + 1, n_cand = span * span;
#pragma unroll 1
    for (int i = lane; i < n_cand; i += 32) {
      const int dy = i / span - R, dx = i - (i / span) * span - R;
      const int col = kWinLeft + dx;
      const unsigned sh = (col & 3) * 8;
      unsigned sad = 0;
#pragma unroll 4
      for (int y = 0; y < 16; ++y) {
        const unsigned *p = reinterpret_cast<const unsigned *>(s.win[kWinTop + dy + y]) + (col >> 2);
        const unsigned a0 = p[0], a1 = p[1], a2 = p[2], a3 = p[3], a4 = p[4];
        sad = Vabsdiff4Add(__funnelshift_r(a0, a1, sh), s.src[4 * y + 0], sad);
        sad = Vabsdiff4Add(__funnelshift_r(a1, a2, sh), s.src[4 * y + 1], sad);
        sad = Vabsdiff4Add(__funnelshift_r(a2, a3, sh), s.src[4 * y + 2], sad);
        sad = Vabsdiff4Add(__funnelshift_r(a3, a4, sh), s.src[4 * y + 3], sad);
      }
      const unsigned cost = sad + (unsigned)(lambda * vp8r_enc_mv_bits(4 * dy, 4 * dx));
      best = min(best, (cost << 12) | (unsigned)i);
    }
    best = __reduce_min_sync(0xffffffffu, best);
  }
  const int span = 2 * R + 1, bi = (int)(best & 4095u);
  int qr = 4 * (bi / span - R), qc = 4 * (bi % span - R);  // quarter pel
  unsigned centre = best >> 12;

  // ---- half-pel, then quarter-pel refinement: four lanes per neighbour, rows 4*(lane&3) .. +3 ----
#pragma unroll 1
  for (int step = 2; step >= 1; step >>= 1) {
    const int k = lane >> 2, part = lane & 3;
    const int cr = qr + step * vp8r_enc_ring_dr(k), cc = qc + step * vp8r_enc_ring_dc(k);
    unsigned sad = PredictLuma<4, 16, false>(s, 2 * cr, 2 * cc, 4 * part, 0);
    sad += __shfl_xor_sync(0xffffffffu, sad, 1);
    sad += __shfl_xor_sync(0xffffffffu, sad, 2);
    const unsigned cost = sad + (unsigned)(lambda * vp8r_enc_mv_bits(cr, cc));
    const unsigned key = __reduce_min_sync(0xffffffffu, min((cost << 4) | (unsigned)(k + 1), centre << 4));
    const int won = (int)(key & 15u);
    if (won) {
      qr += step * vp8r_enc_ring_dr(won - 1);
      qc += step * vp8r_enc_ring_dc(won - 1);
    }
    centre = key >> 4;
  }
  const int mvr = 2 * qr, mvc = 2 * qc;  // 1/8 pel, as vp8r_mb_info.mv

  // ---- prediction of the chosen vector: luma row lane>>1, half lane&1; chroma plane lane>>4, row, half ----
  PredictLuma<1, 8, true>(s, mvr, mvc, lane >> 1, 8 * (lane & 1));
  {
    // chroma vector of a non-SPLIT macroblock (src/inter_predict.cc:116-144), as K_inter derives it
    const int sr = s16e(4 * mvr), sc = s16e(4 * mvc);
    const int ar = (abs(sr) + 4) >> 3, ac = (abs(sc) + 4) >> 3;
    const int cmr = sr < 0 ? -ar : ar, cmc = sc < 0 ? -ac : ac;
    const int pl = lane >> 4, y = (lane >> 1) & 7, x0 = 4 * (lane & 1);
    int th[6], tv[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      th[k] = c_enc_sixtap[cmc & 7][k];
      tv[k] = c_enc_sixtap[cmr & 7][k];
    }
    const uint8_t *base = (pl ? job.ref[1].v : job.ref[1].u) + (ptrdiff_t)(mb_r * 8 + y + (cmr >> 3) - 2) * job.pitch_c + mb_c * 8 + x0 +
                          (cmc >> 3) - 2;
#pragma unroll
    for (int xx = 0; xx < 4; ++xx) {
      int h[6];
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        const uint8_t *q = base + (ptrdiff_t)i * job.pitch_c + xx;
        h[i] = Tap6(th, __ldg(q), __ldg(q + 1), __ldg(q + 2), __ldg(q + 3), __ldg(q + 4), __ldg(q + 5));
      }
      s.cpred[pl][y][x0 + xx] = (unsigned char)Tap6(tv, h[0], h[1], h[2], h[3], h[4], h[5]);
    }
  }
  __syncwarp();
  if (job.enc_flags & VP8R_ENC_INTRA_MBS) {  // inter_err: the luma squared error of the prediction, for K_encode_intra_mbs
    unsigned e = 0;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const unsigned d = __vabsdiffu4(s.pred[lane + 32 * k], s.src[lane + 32 * k]);
      e = __dp4a(d, d, e);
    }
    e = __reduce_add_sync(0xffffffffu, e);
    if (lane == 0) job.enc_inter_err[mb_r * cols + mb_c] = e;
  }

  // ---- residual, forward transform, quantisation (lane b < 24: block b; lane 24: Y2) ----
  const bool luma = lane < 16, is_block = lane < 24;
  const int16_t *dq = job.dq[0];
  const int f_dc = lane == 24 ? dq[VP8R_DQ_Y2_DC] : (luma ? dq[VP8R_DQ_Y1_DC] : dq[VP8R_DQ_UV_DC]);
  const int f_ac = lane == 24 ? dq[VP8R_DQ_Y2_AC] : (luma ? dq[VP8R_DQ_Y1_AC] : dq[VP8R_DQ_UV_AC]);
  int m[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) m[i] = 0;
  if (is_block) {
    unsigned src[4], pred[4];
    if (luma) {
      const int bi4 = lane >> 2, bj = lane & 3;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        src[k] = s.src[4 * (4 * bi4 + k) + bj];
        pred[k] = s.pred[4 * (4 * bi4 + k) + bj];
      }
    } else {
      const int pl = lane >= 20, b = (lane - 16) & 3, bi2 = b >> 1, bj = b & 1;
      const int sp = job.enc_src_pitch_c;
      const uint8_t *sp_base = job.enc_src[1 + pl] + (ptrdiff_t)(mb_r * 8 + 4 * bi2) * sp + mb_c * 8 + 4 * bj;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        src[k] = *reinterpret_cast<const unsigned *>(sp_base + (ptrdiff_t)k * sp);
        pred[k] = *reinterpret_cast<const unsigned *>(&s.cpred[pl][4 * bi2 + k][4 * bj]);
      }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
      for (int x = 0; x < 4; ++x) m[4 * k + x] = (int)((src[k] >> (8 * x)) & 0xff) - (int)((pred[k] >> (8 * x)) & 0xff);
    Fdct4x4(m);
  }
  if (luma) s.y2[lane] = (short)m[0];
  __syncwarp();
  if (lane == 24) {
#pragma unroll
    for (int i = 0; i < 16; ++i) m[i] = s.y2[i];
    Fwht4x4(m);
  }
  bool nz = false;
  if (lane <= 24) {
    m[0] = luma ? 0 : s16e(m[0] / f_dc);  // a luma block's DC travels in the Y2 block
#pragma unroll
    for (int i = 1; i < 16; ++i) m[i] = s16e(m[i] / f_ac);
#pragma unroll
    for (int i = 0; i < 16; ++i) nz |= m[i] != 0;
  }
  const unsigned lanes_nz = __ballot_sync(0xffffffffu, nz);
  const unsigned coef_mask = ((lanes_nz & 0x00ffffffu) << 1) | ((lanes_nz >> 24) & 1u);
  const int mb_index = mb_r * cols + mb_c;
  const unsigned coef_offset = (unsigned)mb_index * 25u;
  if (nz) {
    const int blk = lane < 24 ? lane + 1 : 0;
    const int at = __popc(coef_mask & ((1u << blk) - 1u));
    int4 *dst = reinterpret_cast<int4 *>(const_cast<int16_t *>(job.payload) + (size_t)(coef_offset + at) * 16);
    unsigned w[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) w[i] = ((unsigned)m[2 * i] & 0xffffu) | ((unsigned)m[2 * i + 1] << 16);
    dst[0] = make_int4((int)w[0], (int)w[1], (int)w[2], (int)w[3]);
    dst[1] = make_int4((int)w[4], (int)w[5], (int)w[6], (int)w[7]);
  }
  if (lane == 0) {
    const unsigned flags = VP8R_MB_IS_INTER | (1u << VP8R_MB_REF_SHIFT) | VP8R_MB_HAS_Y2 | ((unsigned)job.lf_level << VP8R_MB_LF_SHIFT) |
                           (coef_mask ? VP8R_MB_LF_INNER : 0u);
    const unsigned mv = ((unsigned)mvr & 0xffffu) | ((unsigned)mvc << 16);
    int4 *rec = reinterpret_cast<int4 *>(const_cast<vp8r_mb_info *>(job.mbs) + mb_index);
    rec[0] = make_int4((int)flags, (int)coef_mask, (int)coef_offset, (int)mv);
    rec[1] = make_int4(0, 0, 0, 0);
  }
}

cudaError_t InitEncodeTables(const unsigned short *bpred_lut) {
  return cudaMemcpyToSymbol(c_enc_bpred_lut, bpred_lut, sizeof(unsigned short) * 160);
}

cudaError_t LaunchEncodeIntra(const DevFrameJob *jobs, int n_frames, int max_rows, cudaStream_t st) {
  const size_t smem = ((size_t(max_rows) * 4 + 15) & ~size_t(15)) + 320 + sizeof(EncScratch) * kEncWarps;
  EncodeIntraKernel<<<n_frames, kEncWarps * 32, smem, st>>>(jobs);
  return cudaGetLastError();
}

cudaError_t LaunchEncodeIntraMbs(const DevFrameJob *jobs, int n_frames, int max_rows, cudaStream_t st) {
  const size_t smem = ((size_t(max_rows) * 4 + 15) & ~size_t(15)) + 320 + sizeof(EncScratch) * kEncWarps;
  EncodeIntraMbsKernel<<<n_frames, kEncWarps * 32, smem, st>>>(jobs);
  return cudaGetLastError();
}

cudaError_t LaunchEncodeInter(const DevFrameJob *jobs, int n_frames, int max_cols, int max_rows, cudaStream_t st) {
  if (max_rows > 65535 || n_frames > 65535) return cudaErrorInvalidValue;
  dim3 grid((max_cols + kEncInterWarps - 1) / kEncInterWarps, max_rows, n_frames);
  EncodeInterKernel<<<grid, kEncInterWarps * 32, 0, st>>>(jobs);
  return cudaGetLastError();
}

}  // namespace vp8r
