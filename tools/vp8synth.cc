// vp8synth -- writes syntactically valid VP8 (RFC 6386) streams in an IVF container for the
// 1080p / 4K workloads of BASELINE.json.  The reference's own encoder is a 28-line stub that
// does not compile (src/encode.cc:12) and its bool encoder has empty WriteByte/AddOne
// (src/bool_encoder.h:72-73), so the synthetic streams have to come from here.
//
// It is an OPEN-LOOP synthesiser, not a video encoder: every decision (modes, motion vectors,
// coefficients, reference updates) is drawn from std::mt19937 (seed 7122 by default, the seed the
// reference's unit tests use, test/dct_test.h:19) with tunable statistics, and written with the
// default entropy tables (or, with --prob-updates, with the tables its own header updates).  What
// makes a stream a valid test input is that the unmodified reference decoder decodes it; its output is then the golden (tests/golden/synthetic/*.md5).
//
// Stand-alone on purpose: links neither the product parser nor anything under oracle/.
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <string>
#include <vector>

#include "../vp8_b200/csrc/host/bool_writer.h"

namespace {
using vp8r::BoolWriter;

#include "../vp8_b200/csrc/host/vp8_prob_tables.inc"

// ----------------------------------------------------------------------------- syntax tables --
enum { DC_PRED = 0, V_PRED, H_PRED, TM_PRED, B_PRED };
enum { MV_NEAREST = 0, MV_NEAR, MV_ZERO, MV_NEW, MV_SPLIT };
const int8_t kTreeYModeKey[8] = {-B_PRED, 2, 4, 6, -DC_PRED, -V_PRED, -H_PRED, -TM_PRED};
const int8_t kTreeYMode[8] = {-DC_PRED, 2, 4, 6, -V_PRED, -H_PRED, -TM_PRED, -B_PRED};
const int8_t kTreeUvMode[6] = {-DC_PRED, 2, -V_PRED, 4, -H_PRED, -TM_PRED};
const int8_t kTreeBMode[18] = {0, 2, -1, 4, -2, 6, 8, 12, -3, 10, -5, -6, -4, 14, -7, 16, -8, -9};
const int8_t kTreeSegment[6] = {2, 4, -0, -1, -2, -3};
const int8_t kTreeMvRef[8] = {-MV_ZERO, 2, -MV_NEAREST, 4, -MV_NEAR, 6, -MV_NEW, -MV_SPLIT};
const int8_t kTreeSplit[6] = {-3, 2, -2, 4, -0, -1};
const int8_t kTreeSubMv[6] = {-0, 2, -1, 4, -2, -3};  // left, above, zero, new
const int8_t kTreeSmallMv[14] = {2, 8, 4, 6, -0, -1, -2, -3, 10, 12, -4, -5, -6, -7};
const uint8_t kProbYModeKey[4] = {145, 156, 163, 128};
const uint8_t kProbUvModeKey[3] = {142, 114, 183};
const uint8_t kProbYMode[4] = {112, 86, 140, 37};
const uint8_t kProbUvMode[3] = {162, 101, 204};
const uint8_t kProbBModeInter[9] = {120, 90, 79, 133, 87, 85, 80, 111, 151};
const uint8_t kProbSplit[3] = {110, 111, 150};
const uint8_t kProbSubMv[5][3] = {{147, 136, 18}, {106, 145, 1}, {179, 121, 1}, {223, 1, 34}, {208, 1, 1}};
const uint8_t kProbMvRef[6][4] = {{7, 1, 1, 143},   {14, 18, 14, 107}, {135, 64, 57, 68},
                                  {60, 56, 128, 65}, {159, 134, 128, 34}, {234, 188, 128, 28}};
const uint8_t kSplitCount[4] = {2, 2, 4, 16};
const uint8_t kSplitMap[4][16] = {{0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 1, 1, 1, 1},
                                  {0, 0, 1, 1, 0, 0, 1, 1, 0, 0, 1, 1, 0, 0, 1, 1},
                                  {0, 0, 1, 1, 0, 0, 1, 1, 2, 2, 3, 3, 2, 2, 3, 3},
                                  {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15}};
const uint8_t kSplitHead[4][16] = {{0, 8}, {0, 2}, {0, 2, 8, 10}, {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15}};
const uint8_t kZigzag[16] = {0, 1, 4, 8, 5, 2, 3, 6, 9, 12, 13, 10, 7, 11, 14, 15};
const uint8_t kBand[17] = {0, 1, 2, 3, 6, 4, 5, 6, 6, 6, 6, 6, 6, 6, 6, 7, 0};
const uint8_t kCat1[] = {159, 0}, kCat2[] = {165, 145, 0}, kCat3[] = {173, 148, 140, 0};
const uint8_t kCat4[] = {176, 155, 140, 135, 0}, kCat5[] = {180, 157, 141, 134, 130, 0};
const uint8_t kCat6[] = {254, 254, 243, 230, 196, 177, 153, 140, 133, 130, 129, 0};
const uint8_t *const kCatProbs[6] = {kCat1, kCat2, kCat3, kCat4, kCat5, kCat6};
const int kCatBase[7] = {5, 7, 11, 19, 35, 67, 2115};
const int kCatBits[6] = {1, 2, 3, 4, 5, 11};
// Quantiser lookup tables (RFC 6386 section 14.1): the writer derives the above / left token contexts from the
// dequantised values, as the decoder does.
const uint8_t kDcQ[128] = {
    4,   5,   6,   7,   8,   9,   10,  10,  11,  12,  13,  14,  15,  16,  17,  17,  18,  19,  20,
    20,  21,  21,  22,  22,  23,  23,  24,  25,  25,  26,  27,  28,  29,  30,  31,  32,  33,  34,
    35,  36,  37,  37,  38,  39,  40,  41,  42,  43,  44,  45,  46,  46,  47,  48,  49,  50,  51,
    52,  53,  54,  55,  56,  57,  58,  59,  60,  61,  62,  63,  64,  65,  66,  67,  68,  69,  70,
    71,  72,  73,  74,  75,  76,  76,  77,  78,  79,  80,  81,  82,  83,  84,  85,  86,  87,  88,
    89,  91,  93,  95,  96,  98,  100, 101, 102, 104, 106, 108, 110, 112, 114, 116, 118, 122, 124,
    126, 128, 130, 132, 134, 136, 138, 140, 143, 145, 148, 151, 154, 157};
const uint16_t kAcQ[128] = {
    4,   5,   6,   7,   8,   9,   10,  11,  12,  13,  14,  15,  16,  17,  18,  19,  20,  21,  22,
    23,  24,  25,  26,  27,  28,  29,  30,  31,  32,  33,  34,  35,  36,  37,  38,  39,  40,  41,
    42,  43,  44,  45,  46,  47,  48,  49,  50,  51,  52,  53,  54,  55,  56,  57,  58,  60,  62,
    64,  66,  68,  70,  72,  74,  76,  78,  80,  82,  84,  86,  88,  90,  92,  94,  96,  98,  100,
    102, 104, 106, 108, 110, 112, 114, 116, 119, 122, 125, 128, 131, 134, 137, 140, 143, 146, 149,
    152, 155, 158, 161, 164, 167, 170, 173, 177, 181, 185, 189, 193, 197, 201, 205, 209, 213, 217,
    221, 225, 229, 234, 239, 245, 249, 254, 259, 264, 269, 274, 279, 284};

struct Mv {
  int r = 0, c = 0;
  bool operator==(const Mv &o) const { return r == o.r && c == o.c; }
  bool operator!=(const Mv &o) const { return !(*this == o); }
  bool nz() const { return r || c; }
};

struct Options {
  int width = 1920, height = 1080, frames = 30, key_interval = 0 /* 0 = first frame only */;
  uint32_t seed = 7122;
  int q = 40, lf_level = 24, sharpness = 0, filter_type = 0, version = 0, log2_parts = 0;
  int segmentation = 1, lf_deltas = 1, golden_period = 7, altref_period = 11, hidden_altref = 1;
  int pct_intra = 8, pct_split = 10, pct_new = 30, pct_skip = 35, pct_bpred = 25;
  int coef_density = 6;  // expected non-zero coefficients per coded block (x2)
  int pct_empty_block = 45;  // blocks without any coefficient inside a non-skipped macroblock
  // Syntax extremes, all off by default (an option at 0 draws nothing from the RNG, so the streams of
  // the manifest stay byte-identical):
  int pct_big_coef = 0;   // share of the non-zero coefficients made DCT_CAT6 magnitudes (67..2114, 512*k)
  int pct_long_mv = 0;    // share of the NEW deltas aimed 64 px beyond a frame corner
  int prob_updates = 0;   // per-probability update chance (coefficients, MVs), mode updates, non-refreshed frames
  int no_skip_flag = 0;   // mb_no_skip_coeff = 0: every macroblock carries its tokens
  std::string out = "synth.ivf";
};

class Synth {
 public:
  explicit Synth(const Options &o) : opt_(o), rng_(o.seed) {
    cols_ = (o.width + 15) / 16;
    rows_ = (o.height + 15) / 16;
  }

  std::vector<uint8_t> Frame(int index) {
    const bool key = index == 0 || (opt_.key_interval > 0 && index % opt_.key_interval == 0);
    key_ = key;
    if (key) probs_ = Probs();
    BoolWriter hdr;
    const int n_parts = 1 << opt_.log2_parts;
    std::vector<BoolWriter> parts(n_parts);

    // ---- frame header (RFC 6386 section 9 / 19.2) ----
    if (key) {
      hdr.Lit(1, 0);  // color space
      hdr.Lit(1, 0);  // clamping type
      seg_map_.assign(size_t(cols_) * rows_, 0);
      std::memset(ref_lf_delta_, 0, sizeof(ref_lf_delta_));
      std::memset(mode_lf_delta_, 0, sizeof(mode_lf_delta_));
      have_seg_data_ = false;
    }
    const bool seg = opt_.segmentation != 0;
    bool update_map = false;
    hdr.Lit(1, seg);
    if (seg) {
      update_map = key || Pct(30);
      const bool update_data = key || !have_seg_data_ || Pct(20);
      hdr.Lit(1, update_map);
      hdr.Lit(1, update_data);
      if (update_data) {
        seg_abs_ = Pct(30);
        hdr.Lit(1, seg_abs_);
        for (int i = 0; i < 4; ++i) {
          int v = seg_abs_ ? Clamp(opt_.q + Range(-12, 12), 0, 127) : Range(-10, 10);
          seg_q_[i] = v;
          hdr.Lit(1, 1);
          hdr.SignedLit(7, v);
        }
        for (int i = 0; i < 4; ++i) {
          int v = seg_abs_ ? Clamp(opt_.lf_level + Range(-8, 8), 0, 63) : Range(-6, 6);
          hdr.Lit(1, 1);
          hdr.SignedLit(6, v);
        }
        have_seg_data_ = true;
      }
      if (update_map)
        for (int i = 0; i < 3; ++i) {
          seg_tree_probs_[i] = uint8_t(Range(64, 200));
          hdr.Lit(1, 1);
          hdr.Lit(8, seg_tree_probs_[i]);
        }
    }
    hdr.Lit(1, opt_.filter_type);
    hdr.Lit(6, uint32_t(opt_.lf_level));
    hdr.Lit(3, uint32_t(opt_.sharpness));
    const bool lf_adj = opt_.lf_deltas != 0;
    hdr.Lit(1, lf_adj);
    if (lf_adj) {
      const bool upd = key || Pct(15);
      hdr.Lit(1, upd);
      if (upd) {
        for (int i = 0; i < 4; ++i) {
          int v = Range(-4, 4);
          hdr.Lit(1, 1);
          hdr.SignedLit(6, v);
        }
        for (int i = 0; i < 4; ++i) {
          int v = Range(-4, 4);
          hdr.Lit(1, 1);
          hdr.SignedLit(6, v);
        }
      }
    }
    hdr.Lit(2, uint32_t(opt_.log2_parts));
    hdr.Lit(7, uint32_t(opt_.q));
    const int deltas[5] = {Range(-3, 3), 0, Range(-2, 2), Range(-3, 3), 0};
    for (int i = 0; i < 5; ++i) {
      hdr.Lit(1, deltas[i] != 0);
      if (deltas[i]) hdr.SignedLit(4, deltas[i]);
    }
    for (int s = 0; s < 4; ++s) {  // dequantisation factors per segment: Y1 DC, AC, Y2 DC, AC, UV DC, AC
      const int q = Clamp(seg ? (seg_abs_ ? seg_q_[s] : opt_.q + seg_q_[s]) : opt_.q, 0, 127);
      auto qi = [&](int d) { return Clamp(q + d, 0, 127); };
      dq_[s][0] = kDcQ[qi(deltas[0])];
      dq_[s][1] = kAcQ[q];
      dq_[s][2] = kDcQ[qi(deltas[1])] * 2;
      dq_[s][3] = std::max(8, int(kAcQ[qi(deltas[2])]) * 155 / 100);
      dq_[s][4] = std::min(132, int(kDcQ[qi(deltas[3])]));
      dq_[s][5] = kAcQ[qi(deltas[4])];
    }
    bool show = true, refresh_entropy = true;
    bool sign_bias[4] = {false, false, false, false};
    if (key) {
      hdr.Lit(1, 1);  // refresh_entropy_probs
    } else {
      bool refresh_g = opt_.golden_period > 0 && index % opt_.golden_period == 0;
      bool refresh_a = opt_.altref_period > 0 && index % opt_.altref_period == 0;
      int copy_g = 0, copy_a = 0;
      if (!refresh_g && Pct(4)) copy_g = 1 + int(rng_() % 2);
      if (!refresh_a && Pct(4)) copy_a = 1 + int(rng_() % 2);
      bool refresh_last = true;
      if (refresh_a && opt_.hidden_altref) {  // a hidden alt-ref frame: decoded, not shown
        show = false;
        refresh_last = false;
      }
      sign_bias[2] = Pct(10);
      sign_bias[3] = Pct(50);
      hdr.Lit(1, refresh_g);
      hdr.Lit(1, refresh_a);
      if (!refresh_g) hdr.Lit(2, uint32_t(copy_g));
      if (!refresh_a) hdr.Lit(2, uint32_t(copy_a));
      hdr.Lit(1, sign_bias[2]);
      hdr.Lit(1, sign_bias[3]);
      refresh_entropy = !(opt_.prob_updates && Pct(opt_.prob_updates));
      hdr.Lit(1, refresh_entropy);
      hdr.Lit(1, refresh_last);
    }
    // The updates of a frame that does not refresh the entropy context last for that frame only.
    const Probs saved = probs_;
    for (int i = 0; i < 1056; ++i) {
      const bool upd = opt_.prob_updates && Pct(opt_.prob_updates);
      hdr.Put(kCoefUpdate[i], upd);
      if (upd) {
        probs_.coef[i] = uint8_t(Range(1, 255));
        hdr.Lit(8, probs_.coef[i]);
      }
    }
    const int prob_skip = 255 - (opt_.pct_skip * 255) / 100;
    hdr.Lit(1, !opt_.no_skip_flag);  // mb_no_skip_coeff
    if (!opt_.no_skip_flag) hdr.Lit(8, uint32_t(Clamp(prob_skip, 1, 255)));
    // prob_intra = P(bit == 0) = P(macroblock is intra), out of 256.
    const int prob_intra = Clamp((opt_.pct_intra * 256) / 100, 1, 255);
    const int prob_last = 200, prob_gf = 128;
    if (!key) {
      hdr.Lit(8, uint32_t(prob_intra));
      hdr.Lit(8, prob_last);
      hdr.Lit(8, prob_gf);
      const bool upd_y = opt_.prob_updates && Pct(50), upd_uv = opt_.prob_updates && Pct(50);
      hdr.Lit(1, upd_y);
      if (upd_y)
        for (int i = 0; i < 4; ++i) hdr.Lit(8, probs_.ymode[i] = uint8_t(Range(1, 255)));
      hdr.Lit(1, upd_uv);
      if (upd_uv)
        for (int i = 0; i < 3; ++i) hdr.Lit(8, probs_.uvmode[i] = uint8_t(Range(1, 255)));
      for (int i = 0; i < 38; ++i) {
        const bool upd = opt_.prob_updates && Pct(opt_.prob_updates);
        hdr.Put(kMvUpdate[i], upd);
        if (upd) {
          const int v = Range(0, 127);
          hdr.Lit(7, uint32_t(v));
          probs_.mv[i] = uint8_t(v ? v << 1 : 1);
        }
      }
    }

    // ---- macroblocks ----
    ctx_.assign(size_t(cols_) * rows_, MbCtx());
    sub_mvs_.assign(size_t(cols_) * rows_ * 16, Mv());
    above_b_.assign(size_t(cols_) * 4, 0);
    nz_ay_.assign(size_t(cols_) * 4, 0);
    nz_au_.assign(size_t(cols_) * 2, 0);
    nz_av_.assign(size_t(cols_) * 2, 0);
    nz_ay2_.assign(size_t(cols_), 0);
    // a smooth global motion for this frame plus per-macroblock jitter, quarter-pel units
    const int pan_r = Range(-12, 12), pan_c = Range(-16, 16);
    if (opt_.pct_long_mv) {  // the point the long deltas aim at: 64 px beyond one corner of the frame
      far_r_ = Pct(50) ? -64 : rows_ * 16 + 64;
      far_c_ = Pct(50) ? -64 : cols_ * 16 + 64;
    }

    for (int r = 0; r < rows_; ++r) {
      uint8_t left_b[4] = {0, 0, 0, 0};
      uint8_t nz_ly[4] = {0, 0, 0, 0}, nz_lu[2] = {0, 0}, nz_lv[2] = {0, 0}, nz_ly2 = 0;
      BoolWriter &tok = parts[n_parts > 1 ? r % n_parts : 0];
      for (int c = 0; c < cols_; ++c) {
        const int idx = r * cols_ + c;
        if (update_map) {
          int s = ((r / 8) + (c / 8) + int(rng_() % 2)) & 3;
          seg_map_[idx] = uint8_t(s);
          hdr.Tree(kTreeSegment, 6, seg_tree_probs_, s);
        }
        const bool skip = !opt_.no_skip_flag && Pct(opt_.pct_skip);
        if (!opt_.no_skip_flag) hdr.Put(Clamp(prob_skip, 1, 255), skip);
        bool inter = false;
        if (!key) {
          inter = !Pct(opt_.pct_intra);
          hdr.Put(prob_intra, inter);
        }
        bool has_y2 = true;
        if (inter) {
          int ref = 1;
          if (Pct(22)) ref = 2 + int(rng_() % 2);
          hdr.Put(prob_last, ref != 1);
          if (ref != 1) hdr.Put(prob_gf, ref == 3);
          has_y2 = WriteInterMb(hdr, r, c, idx, ref, sign_bias, pan_r, pan_c);
        } else {
          int ymode = Pct(opt_.pct_bpred) ? B_PRED : int(rng_() % 4);
          if (key) hdr.Tree(kTreeYModeKey, 8, kProbYModeKey, ymode);
          else hdr.Tree(kTreeYMode, 8, probs_.ymode, ymode);
          if (ymode == B_PRED) {
            has_y2 = false;
            for (int i = 0; i < 4; ++i)
              for (int j = 0; j < 4; ++j) {
                int m = int(rng_() % 10);
                if (key) {
                  hdr.Tree(kTreeBMode, 18, &kKfBmode[(above_b_[c * 4 + j] * 10 + left_b[i]) * 9], m);
                  above_b_[c * 4 + j] = left_b[i] = uint8_t(m);
                } else {
                  hdr.Tree(kTreeBMode, 18, kProbBModeInter, m);
                }
              }
          } else if (key) {
            static const uint8_t implied[4] = {0, 2, 3, 1};  // DC->B_DC, V->B_VE, H->B_HE, TM->B_TM
            for (int i = 0; i < 4; ++i) above_b_[c * 4 + i] = left_b[i] = implied[ymode];
          }
          int uvmode = int(rng_() % 4);
          hdr.Tree(kTreeUvMode, 6, key ? kProbUvModeKey : probs_.uvmode, uvmode);
        }

        // ---- residual tokens ----
        if (!skip) {
          // Inside the macroblock the contexts follow the coded tokens; the ones handed to the next macroblocks
          // follow the dequantised int16 values (a product that wraps to 0 counts as zero).
          uint32_t nz = 0, dnz = 0;  // bit 0: Y2, 1..16: Y, 17..20: U, 21..24: V
          const int *dq = dq_[seg ? seg_map_[idx] : 0];
          if (has_y2) {
            int coefs[16];
            MakeCoefs(coefs, 0, /*dc_bias=*/true, 3);
            if (WriteBlock(tok, 1, nz_ay2_[c] + nz_ly2, 0, coefs)) nz |= 1;
            if (DequantNz(coefs, dq[2], dq[3])) dnz |= 1;
            nz_ay2_[c] = nz_ly2 = uint8_t(dnz & 1);
          }
          for (int b = 0; b < 16; ++b) {
            int i = b >> 2, j = b & 3;
            int a = i ? int((nz >> (b - 3)) & 1) : nz_ay_[c * 4 + j];
            int l = j ? int((nz >> b) & 1) : nz_ly[i];
            int coefs[16];
            MakeCoefs(coefs, has_y2 ? 1 : 0, !has_y2, 2);
            if (WriteBlock(tok, has_y2 ? 0 : 3, a + l, has_y2 ? 1 : 0, coefs)) nz |= 2u << b;
            if (DequantNz(coefs, dq[0], dq[1])) dnz |= 2u << b;
          }
          for (int pl = 0; pl < 2; ++pl) {
            uint8_t *na = pl ? &nz_av_[c * 2] : &nz_au_[c * 2];
            uint8_t *nl = pl ? nz_lv : nz_lu;
            int base = 17 + 4 * pl;
            for (int b = 0; b < 4; ++b) {
              int i = b >> 1, j = b & 1;
              int a = i ? int((nz >> (base + b - 2)) & 1) : na[j];
              int l = j ? int((nz >> (base + b - 1)) & 1) : nl[i];
              int coefs[16];
              MakeCoefs(coefs, 0, true, 2);
              if (WriteBlock(tok, 2, a + l, 0, coefs)) nz |= 1u << (base + b);
              if (DequantNz(coefs, dq[4], dq[5])) dnz |= 1u << (base + b);
            }
          }
          for (int j = 0; j < 4; ++j) nz_ay_[c * 4 + j] = uint8_t((dnz >> (13 + j)) & 1);
          for (int i = 0; i < 4; ++i) nz_ly[i] = uint8_t((dnz >> (4 + i * 4)) & 1);
          for (int j = 0; j < 2; ++j) {
            nz_au_[c * 2 + j] = uint8_t((dnz >> (19 + j)) & 1);
            nz_av_[c * 2 + j] = uint8_t((dnz >> (23 + j)) & 1);
          }
          for (int i = 0; i < 2; ++i) {
            nz_lu[i] = uint8_t((dnz >> (18 + i * 2)) & 1);
            nz_lv[i] = uint8_t((dnz >> (22 + i * 2)) & 1);
          }
        } else {
          if (has_y2) nz_ay2_[c] = nz_ly2 = 0;
          for (int j = 0; j < 4; ++j) nz_ay_[c * 4 + j] = nz_ly[j] = 0;
          for (int j = 0; j < 2; ++j) nz_au_[c * 2 + j] = nz_av_[c * 2 + j] = nz_lu[j] = nz_lv[j] = 0;
        }
      }
    }

    // ---- assemble: tag | first partition | partition sizes | DCT partitions ----
    std::vector<uint8_t> first = hdr.Finish();
    std::vector<std::vector<uint8_t>> pb;
    for (auto &p : parts) pb.push_back(p.Finish());
    if (!refresh_entropy) probs_ = saved;
    std::vector<uint8_t> out;
    uint32_t tag = (key ? 0u : 1u) | (uint32_t(opt_.version) << 1) | (uint32_t(show) << 4) | (uint32_t(first.size()) << 5);
    out.push_back(uint8_t(tag));
    out.push_back(uint8_t(tag >> 8));
    out.push_back(uint8_t(tag >> 16));
    if (key) {
      const uint8_t sc[3] = {0x9d, 0x01, 0x2a};
      out.insert(out.end(), sc, sc + 3);
      out.push_back(uint8_t(opt_.width));
      out.push_back(uint8_t(opt_.width >> 8));
      out.push_back(uint8_t(opt_.height));
      out.push_back(uint8_t(opt_.height >> 8));
    }
    out.insert(out.end(), first.begin(), first.end());
    for (int i = 0; i + 1 < n_parts; ++i) {
      uint32_t n = uint32_t(pb[i].size());
      out.push_back(uint8_t(n));
      out.push_back(uint8_t(n >> 8));
      out.push_back(uint8_t(n >> 16));
    }
    for (auto &p : pb) out.insert(out.end(), p.begin(), p.end());
    return out;
  }

 private:
  struct Probs {  // the entropy context: token, motion-vector and inter-frame 16x16 / chroma mode probabilities
    uint8_t coef[1056], mv[38], ymode[4], uvmode[3];
    Probs() {
      std::memcpy(coef, kCoefDefault, sizeof(coef));
      std::memcpy(mv, kMvDefault, sizeof(mv));
      std::memcpy(ymode, kProbYMode, sizeof(ymode));
      std::memcpy(uvmode, kProbUvMode, sizeof(uvmode));
    }
  };
  struct MbCtx {
    bool inter = false;
    int ref = 0, mode = 0;
    Mv mv;
  };

  static int Clamp(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }
  bool Pct(int p) { return int(rng_() % 100) < p; }
  int Range(int lo, int hi) { return lo + int(rng_() % uint32_t(hi - lo + 1)); }

  // Sparse, low-frequency-weighted coefficients in zig-zag order; no int16 wrap after dequant unless
  // --pct-big-coef asks for DCT_CAT6 magnitudes: half of them over the whole 11-bit range, half multiples
  // of 512, whose product with a factor that is a multiple of 128 (or 1024 with 64, 2048 with 32) wraps to 0.
  void MakeCoefs(int *z, int first, bool allow_dc, int amp) {
    std::memset(z, 0, sizeof(int) * 16);
    if (Pct(opt_.pct_empty_block)) return;  // uncoded block
    int n = 1 + int(rng_() % uint32_t(opt_.coef_density));
    for (int k = 0; k < n; ++k) {
      int pos = first + int((rng_() % 16) * (rng_() % 16) / 16);  // skewed to low frequencies
      if (pos > 15) pos = 15;
      if (pos == 0 && !allow_dc) continue;
      int mag = 1 + int(rng_() % uint32_t(amp));
      if (Pct(3)) mag += int(rng_() % 40);  // occasionally exercise the DCT_CAT tokens
      if (Pct(1)) mag = 67 + int(rng_() % 200);
      if (opt_.pct_big_coef && Pct(opt_.pct_big_coef)) mag = Pct(50) ? Range(67, 2114) : 512 * Range(1, 4);
      z[pos] = Pct(50) ? mag : -mag;
    }
  }

  // Whether any coefficient of a block is non-zero after dequantisation in int16 (z in zig-zag order, z[0] the DC).
  static bool DequantNz(const int *z, int dc_f, int ac_f) {
    for (int n = 0; n < 16; ++n)
      if (int16_t(z[n] * (n ? ac_f : dc_f)) != 0) return true;
    return false;
  }

  // Writes one block; returns whether any coefficient is non-zero.  No trailing zero tokens.
  bool WriteBlock(BoolWriter &bw, int type, int ctx, int first, const int *z) {
    int last = -1;
    for (int n = first; n < 16; ++n)
      if (z[n]) last = n;
    const uint8_t *base = &probs_.coef[size_t(type) * 8 * 3 * 11];
    auto probs = [&](int n, int cx) { return base + (size_t(kBand[n]) * 3 + cx) * 11; };
    bool prev_zero = false;
    int n = first;
    for (; n <= last; ++n) {
      const uint8_t *p = probs(n, ctx);
      int v = z[n], a = v < 0 ? -v : v;
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
          int extra = a - kCatBase[cat];
          for (int i = 0; i < kCatBits[cat]; ++i) bw.Put(kCatProbs[cat][i], (extra >> (kCatBits[cat] - 1 - i)) & 1);
        }
      }
      bw.Put(128, v < 0);
      prev_zero = false;
      ctx = a > 1 ? 2 : 1;
    }
    if (n < 16) bw.Put(probs(n, ctx)[0], 0);  // end of block (never right after a zero: last is non-zero)
    (void)kZigzag;
    return last >= 0;
  }

  void WriteMvComponent(BoolWriter &bw, const uint8_t *p, int a) {
    int x = a < 0 ? -a : a;
    if (x < 8) {
      bw.Put(p[0], 0);
      bw.Tree(kTreeSmallMv, 14, p + 2, x);
    } else {
      bw.Put(p[0], 1);
      for (int i = 0; i < 3; ++i) bw.Put(p[9 + i], (x >> i) & 1);
      for (int i = 9; i > 3; --i) bw.Put(p[9 + i], (x >> i) & 1);
      if (x & 0xFFF0) bw.Put(p[9 + 3], (x >> 3) & 1);
    }
    if (x) bw.Put(p[1], a < 0);
  }

  // Inter MB header with the neighbour search of RFC 6386 section 18.3; returns has_y2.
  bool WriteInterMb(BoolWriter &bw, int r, int c, int idx, int ref, const bool *sign_bias, int pan_r, int pan_c) {
    int cnt[4] = {0, 0, 0, 0};
    Mv near_mvs[4];
    int ptr = 0;
    auto flip = [&](Mv v, int other) {
      if (sign_bias[other] != sign_bias[ref]) {
        v.r = -v.r;
        v.c = -v.c;
      }
      return v;
    };
    const MbCtx *ab = r > 0 ? &ctx_[idx - cols_] : nullptr;
    const MbCtx *lf = c > 0 ? &ctx_[idx - 1] : nullptr;
    const MbCtx *al = (r > 0 && c > 0) ? &ctx_[idx - cols_ - 1] : nullptr;
    if (ab && ab->inter) {
      if (ab->mv.nz()) near_mvs[++ptr] = flip(ab->mv, ab->ref);
      cnt[ptr] += 2;
    }
    if (lf && lf->inter) {
      if (lf->mv.nz()) {
        Mv v = flip(lf->mv, lf->ref);
        if (near_mvs[ptr] != v) near_mvs[++ptr] = v;
        cnt[ptr] += 2;
      } else {
        cnt[0] += 2;
      }
    }
    if (al && al->inter) {
      if (al->mv.nz()) {
        Mv v = flip(al->mv, al->ref);
        if (near_mvs[ptr] != v) near_mvs[++ptr] = v;
        cnt[ptr] += 1;
      } else {
        cnt[0] += 1;
      }
    }
    if (cnt[3] && near_mvs[ptr] == near_mvs[1]) ++cnt[1];
    cnt[3] = ((ab && ab->inter && ab->mode == MV_SPLIT) ? 2 : 0) + ((lf && lf->inter && lf->mode == MV_SPLIT) ? 2 : 0) +
             ((al && al->inter && al->mode == MV_SPLIT) ? 1 : 0);
    if (cnt[2] > cnt[1]) {
      std::swap(cnt[1], cnt[2]);
      std::swap(near_mvs[1], near_mvs[2]);
    }
    if (cnt[1] >= cnt[0]) near_mvs[0] = near_mvs[1];
    auto clamp2 = [&](Mv v) {
      int tl = -(c * 16) * 8 - 128, tr = ((cols_ - 1 - c) * 16) * 8 + 128;
      int tt = -(r * 16) * 8 - 128, tb = ((rows_ - 1 - r) * 16) * 8 + 128;
      v.c = Clamp(v.c, tl, tr);
      v.r = Clamp(v.r, tt, tb);
      return v;
    };
    Mv best = clamp2(near_mvs[0]), nearest = clamp2(near_mvs[1]), near = clamp2(near_mvs[2]);

    int mode;
    int roll = int(rng_() % 100);
    if (roll < opt_.pct_split) mode = MV_SPLIT;
    else if (roll < opt_.pct_split + opt_.pct_new) mode = MV_NEW;
    else if (roll < opt_.pct_split + opt_.pct_new + 25) mode = MV_NEAREST;
    else if (roll < opt_.pct_split + opt_.pct_new + 35) mode = MV_NEAR;
    else mode = MV_ZERO;
    uint8_t p[4];
    for (int i = 0; i < 4; ++i) p[i] = kProbMvRef[cnt[i]][i];
    bw.Tree(kTreeMvRef, 8, p, mode);

    const uint8_t *mvp_r = &probs_.mv[0], *mvp_c = &probs_.mv[19];
    // A delta that steers the final vector towards the frame's global pan (quarter-pel units).
    auto new_delta = [&](const Mv &base_mv, int *dr, int *dc) {
      int want_r = pan_r + Range(-6, 6), want_c = pan_c + Range(-6, 6);
      if (Pct(3)) {  // occasional long vectors: exercise the border clamps
        want_r += Range(-400, 400);
        want_c += Range(-400, 400);
      }
      if (opt_.pct_long_mv && Pct(opt_.pct_long_mv)) {  // at the frame's far point, as far as one delta gets
        want_r = 4 * (far_r_ - r * 16);
        want_c = 4 * (far_c_ - c * 16);
      }
      *dr = Clamp(want_r - base_mv.r / 2, -1023, 1023);
      *dc = Clamp(want_c - base_mv.c / 2, -1023, 1023);
    };
    Mv *sub = &sub_mvs_[size_t(idx) * 16];
    Mv mbmv;
    if (mode == MV_NEAREST) mbmv = nearest;
    else if (mode == MV_NEAR) mbmv = near;
    else if (mode == MV_NEW) {
      int dr, dc;
      new_delta(best, &dr, &dc);
      WriteMvComponent(bw, mvp_r, dr);
      WriteMvComponent(bw, mvp_c, dc);
      mbmv.r = int16_t(dr * 2 + best.r);
      mbmv.c = int16_t(dc * 2 + best.c);
    } else if (mode == MV_SPLIT) {
      int layout = int(rng_() % 4);
      bw.Tree(kTreeSplit, 6, kProbSplit, layout);
      for (int part = 0; part < kSplitCount[layout]; ++part) {
        int k = kSplitHead[layout][part];
        Mv lmv = (k & 3) ? sub[k - 1] : (c == 0 ? Mv() : sub_mvs_[size_t(idx - 1) * 16 + k + 3]);
        Mv amv = (k >= 4) ? sub[k - 4] : (r == 0 ? Mv() : sub_mvs_[size_t(idx - cols_) * 16 + k + 12]);
        int cx;
        if (lmv == amv) cx = amv.nz() ? 3 : 4;
        else if (!amv.nz()) cx = 2;
        else if (!lmv.nz()) cx = 1;
        else cx = 0;
        int sm = int(rng_() % 4);
        bw.Tree(kTreeSubMv, 6, kProbSubMv[cx], sm);
        Mv v;
        if (sm == 0) v = lmv;
        else if (sm == 1) v = amv;
        else if (sm == 3) {
          int dr, dc;
          new_delta(best, &dr, &dc);
          WriteMvComponent(bw, mvp_r, dr);
          WriteMvComponent(bw, mvp_c, dc);
          v.r = int16_t(dr * 2 + best.r);
          v.c = int16_t(dc * 2 + best.c);
        }
        for (int b = 0; b < 16; ++b)
          if (kSplitMap[layout][b] == part) sub[b] = v;
      }
      mbmv = sub[15];
    }
    if (mode != MV_SPLIT)
      for (int b = 0; b < 16; ++b) sub[b] = mbmv;
    ctx_[idx].inter = true;
    ctx_[idx].ref = ref;
    ctx_[idx].mode = mode;
    ctx_[idx].mv = mbmv;
    return mode != MV_SPLIT;
  }

  Options opt_;
  std::mt19937 rng_;
  int cols_, rows_;
  bool key_ = true;
  std::vector<uint8_t> seg_map_;
  bool have_seg_data_ = false;
  int seg_abs_ = 0, seg_q_[4] = {0, 0, 0, 0};
  int dq_[4][6] = {};
  uint8_t seg_tree_probs_[3] = {128, 128, 128};
  int ref_lf_delta_[4], mode_lf_delta_[4];
  Probs probs_;
  int far_r_ = 0, far_c_ = 0;
  std::vector<MbCtx> ctx_;
  std::vector<Mv> sub_mvs_;
  std::vector<uint8_t> above_b_, nz_ay_, nz_au_, nz_av_, nz_ay2_;
};

void Put32(std::vector<uint8_t> &v, uint32_t x) {
  for (int i = 0; i < 4; ++i) v.push_back(uint8_t(x >> (8 * i)));
}

}  // namespace

int main(int argc, char **argv) {
  Options o;
  for (int i = 1; i < argc; ++i) {
    std::string a = argv[i];
    auto next = [&]() -> const char * {
      if (i + 1 >= argc) {
        std::fprintf(stderr, "missing value for %s\n", a.c_str());
        std::exit(2);
      }
      return argv[++i];
    };
    if (a == "--width") o.width = std::atoi(next());
    else if (a == "--height") o.height = std::atoi(next());
    else if (a == "--frames") o.frames = std::atoi(next());
    else if (a == "--seed") o.seed = uint32_t(std::strtoul(next(), nullptr, 10));
    else if (a == "--key-interval") o.key_interval = std::atoi(next());
    else if (a == "--q") o.q = std::atoi(next());
    else if (a == "--lf") o.lf_level = std::atoi(next());
    else if (a == "--sharpness") o.sharpness = std::atoi(next());
    else if (a == "--filter-type") o.filter_type = std::atoi(next());
    else if (a == "--version") o.version = std::atoi(next());
    else if (a == "--log2-parts") o.log2_parts = std::atoi(next());
    else if (a == "--segmentation") o.segmentation = std::atoi(next());
    else if (a == "--lf-deltas") o.lf_deltas = std::atoi(next());
    else if (a == "--golden-period") o.golden_period = std::atoi(next());
    else if (a == "--altref-period") o.altref_period = std::atoi(next());
    else if (a == "--hidden-altref") o.hidden_altref = std::atoi(next());
    else if (a == "--pct-intra") o.pct_intra = std::atoi(next());
    else if (a == "--pct-split") o.pct_split = std::atoi(next());
    else if (a == "--pct-new") o.pct_new = std::atoi(next());
    else if (a == "--pct-skip") o.pct_skip = std::atoi(next());
    else if (a == "--pct-bpred") o.pct_bpred = std::atoi(next());
    else if (a == "--coef-density") o.coef_density = std::max(1, std::atoi(next()));
    else if (a == "--pct-empty-block") o.pct_empty_block = std::atoi(next());
    else if (a == "--pct-big-coef") o.pct_big_coef = std::atoi(next());
    else if (a == "--pct-long-mv") o.pct_long_mv = std::atoi(next());
    else if (a == "--prob-updates") o.prob_updates = std::atoi(next());
    else if (a == "--no-skip-flag") o.no_skip_flag = 1;
    else if (a == "--out") o.out = next();
    else {
      std::fprintf(stderr,
                   "usage: vp8synth --width W --height H --frames N --seed S [--key-interval K] [--q Q] [--lf L]\n"
                   "       [--sharpness S] [--filter-type 0|1] [--version 0..3] [--log2-parts 0..3] [--segmentation 0|1]\n"
                   "       [--lf-deltas 0|1] [--golden-period N] [--altref-period N] [--hidden-altref 0|1]\n"
                   "       [--pct-intra P] [--pct-split P] [--pct-new P] [--pct-skip P] [--pct-bpred P]\n"
                   "       [--coef-density N] [--pct-empty-block P] [--pct-big-coef P] [--pct-long-mv P]\n"
                   "       [--prob-updates P] [--no-skip-flag] --out file.ivf\n"
                   "  --pct-big-coef P   P %% of the non-zero coefficients become DCT_CAT6 magnitudes: half uniform over\n"
                   "                     67..2114 (all 11 extra bits), half from {512, 1024, 1536, 2048}\n"
                   "  --pct-long-mv P    P %% of the NEW deltas (macroblock and SPLIT partition) aim 64 px beyond a frame\n"
                   "                     corner chosen per frame, clamped to +-1023, the range of the long form\n"
                   "  --prob-updates P   each token and MV probability is updated with chance P %%; inter frames may\n"
                   "                     update the 16x16 and chroma mode probabilities; P %% of the inter frames\n"
                   "                     set refresh_entropy_probs = 0\n"
                   "  --no-skip-flag     mb_no_skip_coeff = 0\n");
      return 2;
    }
  }
  if (o.width < 1 || o.width > 16383 || o.height < 1 || o.height > 16383 || o.frames < 1) {
    std::fprintf(stderr, "bad dimensions\n");
    return 2;
  }
  Synth s(o);
  std::vector<uint8_t> file;
  const char sig[4] = {'D', 'K', 'I', 'F'};
  file.insert(file.end(), sig, sig + 4);
  file.push_back(0); file.push_back(0);    // version
  file.push_back(32); file.push_back(0);   // header length
  const char fourcc[4] = {'V', 'P', '8', '0'};
  file.insert(file.end(), fourcc, fourcc + 4);
  file.push_back(uint8_t(o.width)); file.push_back(uint8_t(o.width >> 8));
  file.push_back(uint8_t(o.height)); file.push_back(uint8_t(o.height >> 8));
  Put32(file, 30);
  Put32(file, 1);
  Put32(file, uint32_t(o.frames));
  Put32(file, 0);
  for (int k = 0; k < o.frames; ++k) {
    std::vector<uint8_t> fr = s.Frame(k);
    Put32(file, uint32_t(fr.size()));
    Put32(file, uint32_t(k));
    Put32(file, 0);
    file.insert(file.end(), fr.begin(), fr.end());
  }
  FILE *f = std::fopen(o.out.c_str(), "wb");
  if (!f || std::fwrite(file.data(), 1, file.size(), f) != file.size()) {
    std::fprintf(stderr, "cannot write %s\n", o.out.c_str());
    return 1;
  }
  std::fclose(f);
  return 0;
}
