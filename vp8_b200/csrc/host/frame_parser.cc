#include "frame_parser.h"

#include <algorithm>
#include <cstring>

namespace vp8r {
namespace {

#include "vp8_prob_tables.inc"

// ---- small fixed tables of RFC 6386 (reference: src/bitstream_const.h, src/quantizer.h) ----
enum { DC_PRED = 0, V_PRED, H_PRED, TM_PRED, B_PRED };
enum { B_DC = 0, B_TM, B_VE, B_HE, B_LD, B_RD, B_VR, B_VL, B_HD, B_HU };
enum { SUB_LEFT = 0, SUB_ABOVE, SUB_ZERO, SUB_NEW };

// Trees: entry > 0 is the next node index, entry <= 0 is a negated leaf (RFC 6386 section 8.1).
const int8_t kTreeYModeKey[8] = {-B_PRED, 2, 4, 6, -DC_PRED, -V_PRED, -H_PRED, -TM_PRED};
const int8_t kTreeYMode[8] = {-DC_PRED, 2, 4, 6, -V_PRED, -H_PRED, -TM_PRED, -B_PRED};
const int8_t kTreeUvMode[6] = {-DC_PRED, 2, -V_PRED, 4, -H_PRED, -TM_PRED};
const int8_t kTreeBMode[18] = {-B_DC, 2,  -B_TM, 4,  -B_VE, 6,  8,     12, -B_HE,
                               10,    -B_RD, -B_VR, -B_LD, 14, -B_VL, 16, -B_HD, -B_HU};
const int8_t kTreeSegment[6] = {2, 4, -0, -1, -2, -3};
const int8_t kTreeMvRef[8] = {-MV_ZERO, 2, -MV_NEAREST, 4, -MV_NEAR, 6, -MV_NEW, -MV_SPLIT};
const int8_t kTreeSplit[6] = {-3, 2, -2, 4, -0, -1};  // 3: sixteenths, 2: quarters, 0: top/bottom, 1: left/right
const int8_t kTreeSubMv[6] = {-SUB_LEFT, 2, -SUB_ABOVE, 4, -SUB_ZERO, -SUB_NEW};
const int8_t kTreeSmallMv[14] = {2, 8, 4, 6, -0, -1, -2, -3, 10, 12, -4, -5, -6, -7};

const uint8_t kProbYModeKey[4] = {145, 156, 163, 128};
const uint8_t kProbUvModeKey[3] = {142, 114, 183};
const uint8_t kProbYModeDefault[4] = {112, 86, 140, 37};
const uint8_t kProbUvModeDefault[3] = {162, 101, 204};
const uint8_t kProbBModeInter[9] = {120, 90, 79, 133, 87, 85, 80, 111, 151};
const uint8_t kProbSplit[3] = {110, 111, 150};
const uint8_t kProbSubMv[5][3] = {{147, 136, 18}, {106, 145, 1}, {179, 121, 1}, {223, 1, 34}, {208, 1, 1}};
const uint8_t kProbMvRef[6][4] = {{7, 1, 1, 143},   {14, 18, 14, 107}, {135, 64, 57, 68},
                                  {60, 56, 128, 65}, {159, 134, 128, 34}, {234, 188, 128, 28}};

// Which partition each 4x4 block belongs to, and the first block (raster) of each partition.
const uint8_t kSplitCount[4] = {2, 2, 4, 16};
const uint8_t kSplitMap[4][16] = {{0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 1, 1, 1, 1},
                                  {0, 0, 1, 1, 0, 0, 1, 1, 0, 0, 1, 1, 0, 0, 1, 1},
                                  {0, 0, 1, 1, 0, 0, 1, 1, 2, 2, 3, 3, 2, 2, 3, 3},
                                  {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15}};
const uint8_t kSplitHead[4][16] = {{0, 8}, {0, 2}, {0, 2, 8, 10},
                                   {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15}};

const uint8_t kZigzag[16] = {0, 1, 4, 8, 5, 2, 3, 6, 9, 12, 13, 10, 7, 11, 14, 15};
const uint8_t kBand[17] = {0, 1, 2, 3, 6, 4, 5, 6, 6, 6, 6, 6, 6, 6, 6, 7, 0};
// Extra-bit probabilities of the DCT_CAT tokens (zero terminated) and their base values.
const uint8_t kCat1[] = {159, 0};
const uint8_t kCat2[] = {165, 145, 0};
const uint8_t kCat3[] = {173, 148, 140, 0};
const uint8_t kCat4[] = {176, 155, 140, 135, 0};
const uint8_t kCat5[] = {180, 157, 141, 134, 130, 0};
const uint8_t kCat6[] = {254, 254, 243, 230, 196, 177, 153, 140, 133, 130, 129, 0};
const uint8_t *const kCatProbs[6] = {kCat1, kCat2, kCat3, kCat4, kCat5, kCat6};
const int16_t kCatBase[6] = {5, 7, 11, 19, 35, 67};

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

inline int ClampQ(int q) { return q < 0 ? 0 : (q > 127 ? 127 : q); }

// Dequantisation factors for one quantiser index (src/quantizer.cc:15-53).
void BuildDequant(int q, const int delta[5], int16_t out[6]) {
  // delta order: y_dc, y2_dc, y2_ac, uv_dc, uv_ac
  out[VP8R_DQ_Y1_DC] = int16_t(kDcQ[ClampQ(q + delta[0])]);
  out[VP8R_DQ_Y1_AC] = int16_t(kAcQ[q]);
  out[VP8R_DQ_Y2_DC] = int16_t(kDcQ[ClampQ(q + delta[1])] * 2);
  int y2ac = (int(kAcQ[ClampQ(q + delta[2])]) * 101581) >> 16;
  out[VP8R_DQ_Y2_AC] = int16_t(y2ac < 8 ? 8 : y2ac);
  int uvdc = kDcQ[ClampQ(q + delta[3])];
  out[VP8R_DQ_UV_DC] = int16_t(uvdc > 132 ? 132 : uvdc);
  out[VP8R_DQ_UV_AC] = int16_t(kAcQ[ClampQ(q + delta[4])]);
}

}  // namespace

void DequantFactors(int q_index, const int delta[5], int16_t out[6]) { BuildDequant(ClampQ(q_index), delta, out); }

void DequantFactorsForIndex(int q_index, int16_t out[6]) {
  const int zero[5] = {0, 0, 0, 0, 0};
  BuildDequant(ClampQ(q_index), zero, out);
}

namespace {

inline int ReadSigned(BoolReader &br, int bits) {  // magnitude then sign
  int v = int(br.Literal(bits));
  return br.Bit128() ? -v : v;
}

}  // namespace

void FrameParser::LoadDefaults() {
  std::memcpy(probs_.coef, kCoefDefault, sizeof(probs_.coef));
  std::memcpy(probs_.mv, kMvDefault, sizeof(probs_.mv));
  std::memcpy(probs_.ymode, kProbYModeDefault, sizeof(probs_.ymode));
  std::memcpy(probs_.uvmode, kProbUvModeDefault, sizeof(probs_.uvmode));
  std::memset(segment_tree_probs_, 0, sizeof(segment_tree_probs_));
  std::memset(ref_lf_delta_, 0, sizeof(ref_lf_delta_));
  std::memset(mode_lf_delta_, 0, sizeof(mode_lf_delta_));
  segment_abs_ = 0;
  std::memset(segment_quant_, 0, sizeof(segment_quant_));
  std::memset(segment_lf_, 0, sizeof(segment_lf_));
}

void FrameParser::Reset() {
  have_key_ = false;
  width_ = height_ = mb_cols_ = mb_rows_ = 0;
  LoadDefaults();
  segment_map_.clear();
  error_.clear();
}

bool FrameParser::EnsurePayload(vp8r_frame *out, size_t blocks_needed) {
  size_t bytes = out->mb_bytes() + blocks_needed * 32;
  if (bytes <= out->blob_cap) return true;
  return out->Reserve(bytes, out->used_bytes());
}

// Frame tag + frame header (src/bitstream_parser.cc:12-318).
int FrameParser::ParseHeader(const uint8_t *data, size_t size, vp8r_frame *out) {
  if (size < 3) return Fail(VP8R_ERR_TRUNCATED, "frame shorter than its 3-byte tag");
  uint32_t tag = uint32_t(data[0]) | (uint32_t(data[1]) << 8) | (uint32_t(data[2]) << 16);
  key_frame_ = !(tag & 1);
  version_ = int((tag >> 1) & 7);
  int show = int((tag >> 4) & 1);
  size_t first_size = (tag >> 5) & 0x7FFFF;
  if (version_ > 3) return Fail(VP8R_ERR_UNSUPPORTED, "experimental bitstream version (>3)");
  size_t tag_size = key_frame_ ? 10 : 3;
  if (key_frame_) {
    if (size < 10) return Fail(VP8R_ERR_TRUNCATED, "key frame shorter than its 10-byte tag");
    if (data[3] != 0x9d || data[4] != 0x01 || data[5] != 0x2a)
      return Fail(VP8R_ERR_BITSTREAM, "incorrect key-frame start code");
    width_ = (int(data[6]) | (int(data[7]) << 8)) & 0x3FFF;
    height_ = (int(data[8]) | (int(data[9]) << 8)) & 0x3FFF;  // scaling bits ignored (bitstream_parser.cc:32,35)
    if (width_ == 0 || height_ == 0) return Fail(VP8R_ERR_BITSTREAM, "zero frame dimension");
  } else if (!have_key_) {
    return Fail(VP8R_ERR_STATE, "inter frame before the first key frame");
  }
  // The reference's SubSpan needs at least one byte after the first partition (src/utils.h:78-83).
  if (tag_size + first_size >= size) return Fail(VP8R_ERR_TRUNCATED, "first partition exceeds the frame");
  first_.Init(data + tag_size, first_size);
  first_.MarkUsed();
  first_data_ = data + tag_size;
  first_size_ = first_size;
  BoolReader &br = first_;

  if (key_frame_) {
    LoadDefaults();  // a key frame rebuilds the whole context (bitstream_parser.cc:43-56)
    mb_cols_ = (width_ + 15) / 16;
    mb_rows_ = (height_ + 15) / 16;
    segment_map_.assign(size_t(mb_cols_) * mb_rows_, 0);
    have_key_ = true;
    int color_space = br.Bit128();
    int clamping = br.Bit128();
    if (color_space || clamping) return Fail(VP8R_ERR_UNSUPPORTED, "unsupported color_space / clamping_type");
  }

  vp8r_frame_hdr &h = out->hdr;
  std::memset(&h, 0, sizeof(h));
  h.width = uint16_t(width_);
  h.height = uint16_t(height_);
  h.mb_cols = uint16_t(mb_cols_);
  h.mb_rows = uint16_t(mb_rows_);
  h.key_frame = key_frame_;
  h.version = uint8_t(version_);
  h.show_frame = uint8_t(show);

  segmentation_enabled_ = br.Bit128();
  update_segment_map_ = false;
  if (segmentation_enabled_) {  // bitstream_parser.cc:153-200
    update_segment_map_ = br.Bit128();
    bool update_data = br.Bit128();
    if (update_data) {
      segment_abs_ = br.Bit128();
      for (int i = 0; i < 4; ++i) segment_quant_[i] = br.Bit128() ? int16_t(ReadSigned(br, 7)) : 0;
      for (int i = 0; i < 4; ++i) segment_lf_[i] = br.Bit128() ? int16_t(ReadSigned(br, 6)) : 0;
    }
    if (update_segment_map_) {
      for (int i = 0; i < 3; ++i) segment_tree_probs_[i] = br.Bit128() ? uint8_t(br.Literal(8)) : 255;
    }
  }
  h.filter_type = uint8_t(br.Bit128());
  frame_lf_level_ = int(br.Literal(6));
  h.loop_filter_level = uint8_t(frame_lf_level_);
  h.sharpness_level = uint8_t(br.Literal(3));
  lf_adj_enable_ = br.Bit128();  // bitstream_parser.cc:202-227
  if (lf_adj_enable_ && br.Bit128()) {
    for (int i = 0; i < 4; ++i)
      if (br.Bit128()) ref_lf_delta_[i] = int8_t(ReadSigned(br, 6));
    for (int i = 0; i < 4; ++i)
      if (br.Bit128()) mode_lf_delta_[i] = int8_t(ReadSigned(br, 6));
  }

  // DCT partitions (bitstream_parser.cc:72-86).
  n_dct_parts_ = 1 << br.Literal(2);
  size_t sizes_at = tag_size + first_size;
  size_t off = sizes_at + 3 * size_t(n_dct_parts_ - 1);
  if (off >= size && n_dct_parts_ > 1) return Fail(VP8R_ERR_TRUNCATED, "partition size table exceeds the frame");
  for (int i = 0; i < 8; ++i) {
    dct_[i].Init(nullptr, 0);
    dct_data_[i] = nullptr;
    dct_size_[i] = 0;
  }
  for (int i = 0; i + 1 < n_dct_parts_; ++i) {
    const uint8_t *s = data + sizes_at + 3 * i;
    size_t count = size_t(s[0]) | (size_t(s[1]) << 8) | (size_t(s[2]) << 16);
    if (off + count >= size) return Fail(VP8R_ERR_TRUNCATED, "DCT partition exceeds the frame");
    dct_[i].Init(data + off, count);
    dct_data_[i] = data + off;
    dct_size_[i] = count;
    off += count;
  }
  if (off < size && size - off >= 2) {
    dct_[n_dct_parts_ - 1].Init(data + off, size - off);
    dct_data_[n_dct_parts_ - 1] = data + off;
    dct_size_[n_dct_parts_ - 1] = size - off;
  }

  // Quantiser indices (bitstream_parser.cc:229-273).
  y_ac_qi_ = int(br.Literal(7));
  int delta[5];
  for (int i = 0; i < 5; ++i) delta[i] = br.Bit128() ? ReadSigned(br, 4) : 0;
  int n_seg = segmentation_enabled_ ? 4 : 1;
  for (int s = 0; s < n_seg; ++s) {
    int q = y_ac_qi_;
    if (segmentation_enabled_) q = segment_abs_ ? segment_quant_[s] : segment_quant_[s] + q;  // decode_frame.cc:102-109
    BuildDequant(ClampQ(q), delta, h.dq[s]);
  }

  bool refresh_entropy;
  if (key_frame_) {
    refresh_entropy = br.Bit128();
    h.refresh_golden = h.refresh_altref = h.refresh_last = 1;
  } else {
    h.refresh_golden = uint8_t(br.Bit128());
    h.refresh_altref = uint8_t(br.Bit128());
    if (!h.refresh_golden) h.copy_to_golden = uint8_t(br.Literal(2));
    if (!h.refresh_altref) h.copy_to_altref = uint8_t(br.Literal(2));
    h.sign_bias_golden = uint8_t(br.Bit128());
    h.sign_bias_altref = uint8_t(br.Bit128());
    refresh_entropy = br.Bit128();
    h.refresh_last = uint8_t(br.Bit128());
  }
  sign_bias_[0] = sign_bias_[1] = false;
  sign_bias_[2] = h.sign_bias_golden;
  sign_bias_[3] = h.sign_bias_altref;
  refresh_entropy_ = refresh_entropy;  // consumed by Parse()
  h.q_index = uint8_t(y_ac_qi_);

  return VP8R_OK;
}

int16_t FrameParser::ReadMvComponent(const uint8_t *p) {  // bitstream_parser.cc:441-464
  BoolReader &br = first_;
  int a = 0;
  if (br.Bit(p[0])) {
    for (int i = 0; i < 3; ++i) a += br.Bit(p[9 + i]) << i;
    for (int i = 9; i > 3; --i) a += br.Bit(p[9 + i]) << i;
    if (!(a & 0xFFF0) || br.Bit(p[9 + 3])) a += 8;
  } else {
    a = br.Tree(kTreeSmallMv, p + 2);
  }
  if (a && br.Bit(p[1])) a = -a;
  return int16_t(a);
}

// One 4x4 block of tokens (bitstream_parser.cc:572-621).  Coefficients are written de-zigzagged
// into dst[16] (zeroed here once the block is known to be non-empty).  Returns 1 when any
// coefficient is non-zero (a block of explicit zero tokens returns 0 and leaves zeros in dst).
// *nz_after_dequant mirrors what the reference later derives from the DEQUANTISED int16 values
// (decode_frame.cc:6-47): a product that wraps to 0 in int16 counts as zero there.
int FrameParser::ReadCoefTokens(BoolReader &br, int type, int ctx, int first, int dc_f, int ac_f,
                                int16_t *dst, bool *nz_after_dequant) {
  const uint8_t(*bands)[3][11] = probs_.coef[type];
  int n = first;
  const uint8_t *p = bands[kBand[n]][ctx];
  int any = 0;
  bool dq_any = false;
  std::memset(dst, 0, 32);
  bool first_symbol = true;
  while (n < 16) {
    if (!first_symbol && !br.Bit(p[0])) break;  // end of block (not coded right after a zero token;
                                                // the block's first end-of-block test is in ReadCoefBlock)
    first_symbol = false;
    while (!br.Bit(p[1])) {    // zero token(s)
      if (++n == 16) goto done;
      p = bands[kBand[n]][0];
    }
    int v;
    if (!br.Bit(p[2])) {
      v = 1;
    } else if (!br.Bit(p[3])) {
      v = !br.Bit(p[4]) ? 2 : 3 + br.Bit(p[5]);
    } else {
      int cat;
      if (!br.Bit(p[6])) {
        cat = br.Bit(p[7]);
      } else if (!br.Bit(p[8])) {
        cat = 2 + br.Bit(p[9]);
      } else {
        cat = 4 + br.Bit(p[10]);
      }
      int extra = 0;
      for (const uint8_t *q = kCatProbs[cat]; *q; ++q) extra = extra + extra + br.Bit(*q);
      v = kCatBase[cat] + extra;
    }
    int next_ctx = v > 1 ? 2 : 1;
    if (br.Bit128()) v = -v;
    dst[kZigzag[n]] = int16_t(v);
    any = 1;
    if (int16_t(v * (n == 0 ? dc_f : ac_f)) != 0) dq_any = true;
    ++n;
    p = bands[kBand[n]][next_ctx];
  }
done:
  *nz_after_dequant = dq_any;
  return any;
}

// Inter macroblock header: neighbour search, mode, motion vectors
// (src/inter_predict.cc:8-81,146-244; src/bitstream_parser.cc:354-390).
void FrameParser::ParseInterMb(int r, int c, int idx, int ref, vp8r_mb_info *mb, vp8r_frame *out,
                               bool *split) {
  BoolReader &br = first_;
  const NearMvs nm = FindNearMvs(mbctx_.data(), r, c, mb_cols_, mb_rows_, ref, sign_bias_);
  uint8_t p[4];
  for (int i = 0; i < 4; ++i) p[i] = kProbMvRef[nm.cnt[i]][i];
  int mode = br.Tree(kTreeMvRef, p);
  const Mv best = nm.best, nearest = nm.nearest, near = nm.near;

  Mv *sub = &sub_mvs_[size_t(idx) * 16];
  Mv mbmv{0, 0};
  *split = false;
  switch (mode) {
    case MV_NEAREST: mbmv = nearest; break;
    case MV_NEAR: mbmv = near; break;
    case MV_ZERO: break;
    case MV_NEW: {
      int16_t dr = int16_t(ReadMvComponent(probs_.mv[0]) * 2);
      int16_t dc = int16_t(ReadMvComponent(probs_.mv[1]) * 2);
      mbmv = Mv{int16_t(dr + best.r), int16_t(dc + best.c)};  // no re-clamp (inter_predict.cc:224-228)
      break;
    }
    default: {  // MV_SPLIT
      *split = true;
      int layout = br.Tree(kTreeSplit, kProbSplit);
      const Mv zero{0, 0};
      for (int part = 0; part < kSplitCount[layout]; ++part) {
        int k = kSplitHead[layout][part];
        // a neighbouring macroblock's sub-block vector: stored only for SPLIT macroblocks, otherwise
        // its one vector (zero for intra macroblocks)
        auto neighbour = [&](int i, int b) {
          const MbCtx &m = mbctx_[i];
          return (m.is_inter && m.mode == MV_SPLIT) ? sub_mvs_[size_t(i) * 16 + b] : m.mv;
        };
        Mv lmv = (k & 3) ? sub[k - 1] : (c == 0 ? zero : neighbour(idx - 1, k + 3));
        Mv amv = (k >= 4) ? sub[k - 4] : (r == 0 ? zero : neighbour(idx - mb_cols_, k + 12));
        int ctx;  // src/inter_predict.h:42-43, src/inter_predict.cc:112-114
        if (lmv == amv) ctx = amv.nonzero() ? 3 : 4;
        else if (!amv.nonzero()) ctx = 2;
        else if (!lmv.nonzero()) ctx = 1;
        else ctx = 0;
        int sm = br.Tree(kTreeSubMv, kProbSubMv[ctx]);
        Mv v;
        if (sm == SUB_LEFT) v = lmv;
        else if (sm == SUB_ABOVE) v = amv;
        else if (sm == SUB_ZERO) v = zero;
        else {
          int16_t dr = int16_t(ReadMvComponent(probs_.mv[0]) * 2);
          int16_t dc = int16_t(ReadMvComponent(probs_.mv[1]) * 2);
          v = Mv{int16_t(dr + best.r), int16_t(dc + best.c)};
        }
        for (int b = 0; b < 16; ++b)
          if (kSplitMap[layout][b] == part) sub[b] = v;
      }
      mbmv = sub[15];
      break;
    }
  }

  mbctx_[idx] = MbCtx{1, uint8_t(ref), uint8_t(mode), mbmv};
  mb->flags |= VP8R_MB_IS_INTER | (uint32_t(ref) << VP8R_MB_REF_SHIFT) | (uint32_t(mode) << VP8R_MB_MODE_SHIFT);
  mb->mv[0] = mbmv.r;
  mb->mv[1] = mbmv.c;
  if (*split) {
    uint32_t at = out->hdr.n_payload_blocks;
    int16_t *dst = out->payload() + size_t(at) * 16;
    for (int b = 0; b < 16; ++b) {
      dst[2 * b] = sub[b].r;
      dst[2 * b + 1] = sub[b].c;
    }
    mb->aux[0] = at;
    out->hdr.n_payload_blocks += 2;
    out->hdr.n_split_mbs++;
  }
  out->hdr.n_inter_mbs++;
}

// Per-macroblock syntax in raster order (decode_frame.cc:98-170 with the pixel work removed).
int FrameParser::ParseMacroblocks(vp8r_frame *out) {
  BoolReader &br = first_;
  const int cols = mb_cols_, rows = mb_rows_;
  const size_t n_mb = size_t(cols) * rows;
  vp8r_frame_hdr &h = out->hdr;

  mbctx_.assign(n_mb, MbCtx{0, 0, 0, Mv{0, 0}});
  if (!key_frame_ && sub_mvs_.size() < n_mb * 16) sub_mvs_.resize(n_mb * 16);  // written for SPLIT macroblocks only
  above_bmodes_.assign(size_t(cols) * 4, B_DC);
  nz_above_y_.assign(size_t(cols) * 4, 0);
  nz_above_u_.assign(size_t(cols) * 2, 0);
  nz_above_v_.assign(size_t(cols) * 2, 0);
  nz_above_y2_.assign(size_t(cols), 0);

  for (int r = 0; r < rows; ++r) {
    uint8_t left_bmodes[4] = {B_DC, B_DC, B_DC, B_DC};
    uint8_t nz_left_y[4] = {0, 0, 0, 0}, nz_left_u[2] = {0, 0}, nz_left_v[2] = {0, 0};
    uint8_t nz_left_y2 = 0;
    BoolReader &tok = dct_[n_dct_parts_ > 1 ? (r % n_dct_parts_) : 0];  // bitstream_parser.cc:468-477

    for (int c = 0; c < cols; ++c) {
      const int idx = r * cols + c;
      if (!EnsurePayload(out, size_t(h.n_payload_blocks) + 27)) return Fail(VP8R_ERR_NOMEM, "out of host memory");
      vp8r_mb_info *mb = &out->mbs()[idx];
      std::memset(mb, 0, sizeof(*mb));

      // --- pre-header (bitstream_parser.cc:320-352) ---
      int seg;
      if (update_segment_map_) {
        seg = br.Tree(kTreeSegment, segment_tree_probs_);
        segment_map_[idx] = uint8_t(seg);
      } else {
        seg = segment_map_[idx];
      }
      int skip = mb_no_skip_coeff_ ? br.Bit(prob_skip_false_) : 0;
      int is_inter = key_frame_ ? 0 : br.Bit(prob_intra_);

      int ymode = DC_PRED;
      bool split = false, bpred = false;
      int ref = 0, inter_mode = 0;
      if (is_inter) {
        ref = br.Bit(prob_last_) ? 2 + br.Bit(prob_gf_) : 1;
        ParseInterMb(r, c, idx, ref, mb, out, &split);
        inter_mode = int((mb->flags >> VP8R_MB_MODE_SHIFT) & 7);
      } else {
        ymode = key_frame_ ? br.Tree(kTreeYModeKey, kProbYModeKey) : br.Tree(kTreeYMode, probs_.ymode);
        bpred = ymode == B_PRED;
        if (bpred) {  // intra_predict.cc:176-183
          uint8_t *above = &above_bmodes_[size_t(c) * 4];
          uint32_t packed[2] = {0, 0};
          for (int i = 0; i < 4; ++i) {
            for (int j = 0; j < 4; ++j) {
              int m;
              if (key_frame_) {
                m = br.Tree(kTreeBMode, &kKfBmode[(above[j] * 10 + left_bmodes[i]) * 9]);
                above[j] = left_bmodes[i] = uint8_t(m);
              } else {
                m = br.Tree(kTreeBMode, kProbBModeInter);
              }
              int b = i * 4 + j;
              packed[b >> 3] |= uint32_t(m) << ((b & 7) * 4);
            }
          }
          mb->aux[0] = packed[0];
          mb->aux[1] = packed[1];
        } else if (key_frame_) {
          static const uint8_t implied[4] = {B_DC, B_VE, B_HE, B_TM};  // intra_predict.h:19-26
          for (int i = 0; i < 4; ++i) above_bmodes_[size_t(c) * 4 + i] = left_bmodes[i] = implied[ymode];
        }
        int uvmode = key_frame_ ? br.Tree(kTreeUvMode, kProbUvModeKey) : br.Tree(kTreeUvMode, probs_.uvmode);
        mb->flags |= (uint32_t(ymode) << VP8R_MB_MODE_SHIFT) | (uint32_t(uvmode) << VP8R_MB_UVMODE_SHIFT);
      }

      // --- residual tokens (bitstream_parser.cc:466-537) ---
      const bool has_y2 = is_inter ? !split : !bpred;
      const int qseg = segmentation_enabled_ ? seg : 0;
      const int16_t *dq = h.dq[qseg];
      uint32_t mask = 0;
      mb->coef_offset = h.n_payload_blocks;
      if (defer_tokens_) {
        // The device token decoder fills coef_mask / coef_offset and completes VP8R_MB_LF_INNER.
        mb->coef_offset = 0;
        if (skip) mb->flags |= VP8R_MB_SKIP_COEF;
      } else if (!skip) {
        tok.MarkUsed();
        int16_t *dst = out->payload() + size_t(h.n_payload_blocks) * 16;
        uint32_t stored = 0;
        bool dqnz;
        uint32_t raw = 0;  // raw non-zero flags, bit b as in coef_mask
        uint32_t dqf = 0;  // non-zero after dequantisation
        if (has_y2) {
          int ctx = nz_above_y2_[c] + nz_left_y2;
          if (ReadCoefBlock(tok, 1, ctx, 0, dq[VP8R_DQ_Y2_DC], dq[VP8R_DQ_Y2_AC], dst, &dqnz)) {
            raw |= 1;
            dst += 16;
            ++stored;
          }
          if (dqnz) dqf |= 1;
        }
        const int ytype = has_y2 ? 0 : 3, yfirst = has_y2 ? 1 : 0;
        for (int b = 0; b < 16; ++b) {
          int i = b >> 2, j = b & 3;
          int a = i ? int((raw >> (b - 3)) & 1) : nz_above_y_[c * 4 + j];  // block b-4 is bit b-3
          int l = j ? int((raw >> b) & 1) : nz_left_y[i];                  // block b-1 is bit b
          if (ReadCoefBlock(tok, ytype, a + l, yfirst, dq[VP8R_DQ_Y1_DC], dq[VP8R_DQ_Y1_AC], dst, &dqnz)) {
            raw |= 2u << b;
            dst += 16;
            ++stored;
          }
          if (dqnz) dqf |= 2u << b;
        }
        for (int plane = 0; plane < 2; ++plane) {
          uint8_t *na = plane ? &nz_above_v_[c * 2] : &nz_above_u_[c * 2];
          uint8_t *nl = plane ? nz_left_v : nz_left_u;
          int base = 17 + plane * 4;
          for (int b = 0; b < 4; ++b) {
            int i = b >> 1, j = b & 1;
            int a = i ? int((raw >> (base + b - 2)) & 1) : na[j];
            int l = j ? int((raw >> (base + b - 1)) & 1) : nl[i];
            if (ReadCoefBlock(tok, 2, a + l, 0, dq[VP8R_DQ_UV_DC], dq[VP8R_DQ_UV_AC], dst, &dqnz)) {
              raw |= 1u << (base + b);
              dst += 16;
              ++stored;
            }
            if (dqnz) dqf |= 1u << (base + b);
          }
        }
        mask = raw;
        h.n_payload_blocks += stored;
        h.n_coef_blocks += stored;
        // Export contexts for the neighbours: post-dequant flags (decode_frame.cc:6-47).
        if (has_y2) nz_above_y2_[c] = nz_left_y2 = uint8_t(dqf & 1);
        for (int j = 0; j < 4; ++j) nz_above_y_[c * 4 + j] = uint8_t((dqf >> (1 + 12 + j)) & 1);
        for (int i = 0; i < 4; ++i) nz_left_y[i] = uint8_t((dqf >> (1 + i * 4 + 3)) & 1);
        for (int j = 0; j < 2; ++j) {
          nz_above_u_[c * 2 + j] = uint8_t((dqf >> (17 + 2 + j)) & 1);
          nz_above_v_[c * 2 + j] = uint8_t((dqf >> (21 + 2 + j)) & 1);
        }
        for (int i = 0; i < 2; ++i) {
          nz_left_u[i] = uint8_t((dqf >> (17 + i * 2 + 1)) & 1);
          nz_left_v[i] = uint8_t((dqf >> (21 + i * 2 + 1)) & 1);
        }
      } else {
        if (has_y2) nz_above_y2_[c] = nz_left_y2 = 0;
        for (int j = 0; j < 4; ++j) nz_above_y_[c * 4 + j] = nz_left_y[j] = 0;
        for (int j = 0; j < 2; ++j) nz_above_u_[c * 2 + j] = nz_above_v_[c * 2 + j] = nz_left_u[j] = nz_left_v[j] = 0;
      }
      mb->coef_mask = mask;

      // --- loop-filter level of this MB (bitstream_parser.cc:539-568) ---
      int lvl = frame_lf_level_;
      if (segmentation_enabled_) {
        lvl = segment_abs_ ? segment_lf_[seg] : lvl + segment_lf_[seg];
        lvl = lvl < 0 ? 0 : (lvl > 63 ? 63 : lvl);
      }
      if (lf_adj_enable_) {
        lvl += ref_lf_delta_[ref];
        if (ref == 0) {
          if (bpred) lvl += mode_lf_delta_[0];
        } else if (inter_mode == MV_ZERO) {
          lvl += mode_lf_delta_[1];
        } else if (inter_mode == MV_SPLIT) {
          lvl += mode_lf_delta_[3];
        } else {
          lvl += mode_lf_delta_[2];
        }
        lvl = lvl < 0 ? 0 : (lvl > 63 ? 63 : lvl);
      }
      // Inner edges: decode_frame.cc:149, intra_predict.cc:362, inter_predict.cc:206.
      bool inner = (!skip && mask != 0) || bpred || split;
      mb->flags |= (has_y2 ? VP8R_MB_HAS_Y2 : 0) | (uint32_t(qseg) << VP8R_MB_QSEG_SHIFT) |
                   (uint32_t(lvl) << VP8R_MB_LF_SHIFT) | (inner ? VP8R_MB_LF_INNER : 0);
    }
  }
  return VP8R_OK;
}

// Dependency levels of the intra macroblocks of an inter frame (see vp8r_frame_hdr.n_intra_levels).
// Intra prediction reads the left, above-left, above and (B_PRED) above-right macroblocks; inter
// neighbours are complete before any intra MB is touched, so only intra neighbours order the work.
bool FrameParser::BuildIntraLevels(vp8r_frame *out) {
  vp8r_frame_hdr &h = out->hdr;
  const int cols = mb_cols_, rows = mb_rows_;
  const size_t n_mb = size_t(cols) * rows;
  const size_t n_intra = n_mb - h.n_inter_mbs;
  h.n_intra_levels = 0;
  h.intra_levels_at = 0;
  if (n_intra == 0) return true;
  levels_.assign(n_mb, 0);  // 0 = inter, k>0 = intra of level k-1
  const vp8r_mb_info *mbs = out->mbs();
  unsigned max_level = 0;
  for (int r = 0; r < rows; ++r)
    for (int c = 0; c < cols; ++c) {
      const size_t i = size_t(r) * cols + c;
      if (mbs[i].flags & VP8R_MB_IS_INTER) continue;
      unsigned lv = 0;
      if (c > 0) lv = std::max<unsigned>(lv, levels_[i - 1]);
      if (r > 0) {
        lv = std::max<unsigned>(lv, levels_[i - cols]);
        if (c > 0) lv = std::max<unsigned>(lv, levels_[i - cols - 1]);
        if (c + 1 < cols) lv = std::max<unsigned>(lv, levels_[i - cols + 1]);
      }
      levels_[i] = uint16_t(lv + 1);
      max_level = std::max(max_level, lv + 1);
    }
  if (max_level > kMaxFlatIntraLevels) return true;  // scheduled as a wavefront instead
  // counting sort by level into the tail of the payload
  const size_t table_bytes = (size_t(max_level) + 1 + n_intra) * 4;
  const size_t blocks = (table_bytes + 31) / 32;
  if (!EnsurePayload(out, size_t(h.n_payload_blocks) + blocks)) return false;
  mbs = out->mbs();
  uint32_t *tab = reinterpret_cast<uint32_t *>(out->payload() + size_t(h.n_payload_blocks) * 16);
  std::memset(tab, 0, blocks * 32);
  cursor_.assign(max_level, 0);
  for (size_t i = 0; i < n_mb; ++i)
    if (levels_[i]) cursor_[levels_[i] - 1]++;
  tab[0] = 0;
  for (unsigned k = 0; k < max_level; ++k) {
    tab[k + 1] = tab[k] + cursor_[k];
    cursor_[k] = tab[k];  // becomes the write cursor of level k
  }
  uint32_t *idx = tab + max_level + 1;
  for (size_t i = 0; i < n_mb; ++i)
    if (levels_[i]) idx[cursor_[levels_[i] - 1]++ ] = uint32_t(i);
  h.n_intra_levels = max_level;
  h.intra_levels_at = h.n_payload_blocks;
  h.n_payload_blocks += uint32_t(blocks);
  return true;
}

// Deferred tokens: token header (partition table + the probabilities in force) and the raw bytes of
// the DCT partitions, appended to the payload so that the frame still travels as one blob.
bool FrameParser::AttachTokenPartitions(vp8r_frame *out) {
  vp8r_frame_hdr &h = out->hdr;
  static_assert(sizeof(vp8r_token_hdr) == 1152, "vp8r_token_hdr layout");
  static_assert(sizeof(vp8r_mode_hdr) == 160, "vp8r_mode_hdr layout");
  size_t raw = 0;
  for (int i = 0; i < n_dct_parts_; ++i) raw += (dct_size_[i] + 3) & ~size_t(3);
  const size_t first_at = raw;
  if (defer_modes_) raw += (first_size_ + 3) & ~size_t(3);
  const size_t raw_padded = (raw + 16 + 31) & ~size_t(31);
  const size_t mode_bytes = defer_modes_ ? sizeof(vp8r_mode_hdr) : 0;
  const size_t blocks = (mode_bytes + sizeof(vp8r_token_hdr) + raw_padded) / 32;
  if (!EnsurePayload(out, size_t(h.n_payload_blocks) + blocks)) return false;
  uint8_t *base = reinterpret_cast<uint8_t *>(out->payload() + size_t(h.n_payload_blocks) * 16);
  vp8r_token_hdr *th = reinterpret_cast<vp8r_token_hdr *>(base + mode_bytes);
  std::memset(th, 0, 96);
  th->n_parts = uint32_t(n_dct_parts_);
  uint8_t *dst = reinterpret_cast<uint8_t *>(th) + sizeof(vp8r_token_hdr);
  size_t at = 0;
  auto put = [&](const uint8_t *src, size_t n) {
    if (n) std::memcpy(dst + at, src, n);
    size_t end = at + n;
    at = (end + 3) & ~size_t(3);
    std::memset(dst + end, 0, at - end);
  };
  for (int i = 0; i < n_dct_parts_; ++i) {
    th->part_off[i] = uint32_t(at);
    th->part_size[i] = uint32_t(dct_size_[i]);
    put(dct_data_[i], dct_size_[i]);
  }
  if (defer_modes_) put(first_data_, first_size_);
  std::memset(dst + at, 0, raw_padded - at);
  th->raw_bytes = uint32_t(raw_padded);
  std::memcpy(th->coef_probs, probs_.coef, sizeof(th->coef_probs));
  h.tokens_deferred = 1;
  h.tokens_at = h.n_payload_blocks + uint32_t(mode_bytes / 32);
  if (defer_modes_) {
    vp8r_mode_hdr *mh = reinterpret_cast<vp8r_mode_hdr *>(base);
    std::memset(mh, 0, sizeof(*mh));
    first_.Prime();
    mh->first_off = uint32_t(first_at);
    mh->first_size = uint32_t(first_size_);
    mh->bitpos = uint32_t(first_.Shifts() + 8);
    mh->value = uint8_t(first_.Top8());
    mh->range = uint8_t(first_.Range());
    mh->key_frame = key_frame_;
    mh->segmentation_enabled = segmentation_enabled_;
    mh->update_segment_map = update_segment_map_;
    mh->mb_no_skip_coeff = mb_no_skip_coeff_;
    mh->prob_skip_false = uint8_t(prob_skip_false_);
    mh->prob_intra = uint8_t(prob_intra_);
    mh->prob_last = uint8_t(prob_last_);
    mh->prob_gf = uint8_t(prob_gf_);
    for (int i = 0; i < 4; ++i) {
      mh->sign_bias[i] = sign_bias_[i];
      mh->segment_lf[i] = int8_t(segment_lf_[i]);
      mh->ref_lf_delta[i] = ref_lf_delta_[i];
      mh->mode_lf_delta[i] = mode_lf_delta_[i];
      mh->ymode_probs[i] = probs_.ymode[i];
    }
    for (int i = 0; i < 3; ++i) {
      mh->segment_tree_probs[i] = segment_tree_probs_[i];
      mh->uvmode_probs[i] = probs_.uvmode[i];
    }
    mh->segment_abs = uint8_t(segment_abs_);
    mh->lf_adj_enable = lf_adj_enable_;
    mh->frame_lf_level = uint8_t(frame_lf_level_);
    std::memcpy(mh->mv_probs, probs_.mv, sizeof(mh->mv_probs));
    h.modes_deferred = 1;
    h.modes_at = h.n_payload_blocks;
  }
  h.n_payload_blocks += uint32_t(blocks);
  return true;
}

int FrameParser::Parse(const uint8_t *data, size_t size, vp8r_frame *out) {
  if (!data || !out) return Fail(VP8R_ERR_INVALID_ARG, "null argument");
  out->DropDeviceCopy();
  int rc = ParseHeader(data, size, out);
  if (rc != VP8R_OK) return rc;
  BoolReader &br = first_;
  const bool refresh_entropy = refresh_entropy_;

  // Probability updates of a frame with refresh_entropy_probs == 0 are dropped at its end
  // (bitstream_parser.cc:116-141,276-284,302-309).
  EntropyTables saved;
  if (!refresh_entropy) saved = probs_;

  for (int i = 0; i < 4; ++i)  // token probabilities, bitstream_parser.cc:275-299
    for (int j = 0; j < 8; ++j)
      for (int k = 0; k < 3; ++k)
        for (int l = 0; l < 11; ++l)
          if (br.Bit(kCoefUpdate[((i * 8 + j) * 3 + k) * 11 + l])) probs_.coef[i][j][k][l] = uint8_t(br.Literal(8));
  mb_no_skip_coeff_ = br.Bit128();
  prob_skip_false_ = mb_no_skip_coeff_ ? int(br.Literal(8)) : 0;
  if (!key_frame_) {
    prob_intra_ = int(br.Literal(8));
    prob_last_ = int(br.Literal(8));
    prob_gf_ = int(br.Literal(8));
    if (br.Bit128())
      for (int i = 0; i < 4; ++i) probs_.ymode[i] = uint8_t(br.Literal(8));
    if (br.Bit128())
      for (int i = 0; i < 3; ++i) probs_.uvmode[i] = uint8_t(br.Literal(8));
    for (int i = 0; i < 2; ++i)  // bitstream_parser.cc:301-318
      for (int j = 0; j < 19; ++j)
        if (br.Bit(kMvUpdate[i * 19 + j])) {
          int x = int(br.Literal(7));
          probs_.mv[i][j] = uint8_t(x ? x << 1 : 1);
        }
  }

  const bool fits_device = size_t(mb_cols_) * mb_rows_ <= kMaxDeferMbs;
  defer_modes_ = want_defer_modes_ && fits_device;
  defer_tokens_ = (want_defer_tokens_ || want_defer_modes_) && fits_device;
  out->n_mb = defer_modes_ ? 0 : size_t(mb_cols_) * mb_rows_;  // deferred modes: no host MB records
  out->hdr.n_coef_blocks = out->hdr.n_payload_blocks = 0;
  if (!out->Reserve(out->mb_bytes() + 64 * 1024, 0)) return Fail(VP8R_ERR_NOMEM, "out of host memory");
  if (defer_modes_) {
    const bool ok = AttachTokenPartitions(out);
    if (!refresh_entropy) probs_ = saved;
    return ok ? int(VP8R_OK) : Fail(VP8R_ERR_NOMEM, "out of host memory");
  }

  rc = ParseMacroblocks(out);
  bool ok = rc == VP8R_OK;
  if (ok && !key_frame_) ok = BuildIntraLevels(out);
  if (ok && defer_tokens_) ok = AttachTokenPartitions(out);  // needs this frame's probabilities
  if (!refresh_entropy) probs_ = saved;
  if (rc != VP8R_OK) return rc;
  if (!ok) return Fail(VP8R_ERR_NOMEM, "out of host memory");

  if (first_.Overrun()) return Fail(VP8R_ERR_TRUNCATED, "first partition read past its end");
  for (int i = 0; i < n_dct_parts_; ++i)
    if (dct_[i].Overrun()) return Fail(VP8R_ERR_TRUNCATED, "DCT partition read past its end");
  return VP8R_OK;
}

}  // namespace vp8r
