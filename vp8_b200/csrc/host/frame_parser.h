// Pure host parser: compressed VP8 frame -> vp8r_frame (per-macroblock mode / motion-vector /
// coefficient arrays).  It never touches a pixel.
//
// The reference interleaves these reads with reconstruction (src/decode_frame.cc:98-170); the
// split is legal because every syntax element depends only on previously parsed syntax
// (b-mode contexts: src/intra_predict.cc:176-183; neighbour MVs: src/inter_predict.cc:22-68;
// token contexts: src/bitstream_parser.cc:500-534, src/decode_frame.cc:111-130).
#ifndef VP8R_HOST_FRAME_PARSER_H_
#define VP8R_HOST_FRAME_PARSER_H_

#include <cstdint>
#include <string>
#include <vector>

#include "bool_reader.h"
#include "near_mvs.h"
#include "parsed_frame.h"
#include "vp8r.h"

namespace vp8r {

struct EntropyTables {
  uint8_t coef[4][8][3][11];
  uint8_t mv[2][19];
  uint8_t ymode[4];
  uint8_t uvmode[3];
};

// Dequantisation (= quantisation) factors of one quantiser index without deltas, in VP8R_DQ_* order
// (src/quantizer.cc:15-53).  Used by the encoder, which writes frames with one quantiser.
void DequantFactorsForIndex(int q_index, int16_t out[6]);
// The same with the frame header's five quantiser deltas (y_dc, y2_dc, y2_ac, uv_dc, uv_ac).
void DequantFactors(int q_index, const int delta[5], int16_t out[6]);

class FrameParser {
 public:
  FrameParser() { Reset(); }
  void Reset();

  // Returns a vp8r_status; on failure `error()` describes it.
  int Parse(const uint8_t *data, size_t size, vp8r_frame *out);
  const std::string &error() const { return error_; }
  // Deferred tokens: parse the first partition only and attach the DCT partitions to the frame for
  // the device-side token decoder (vp8r_frame_hdr.tokens_deferred).  Survives Reset().
  void set_defer_tokens(bool on) { want_defer_tokens_ = on; }
  // Deferred modes: parse the frame header only; the per-macroblock syntax is decoded on the device
  // too (vp8r_frame_hdr.modes_deferred).  Implies deferred tokens.
  void set_defer_modes(bool on) { want_defer_modes_ = on; }

  // The context the next frame of the stream is parsed in (read by the bitstream writer): whether a key frame has
  // been seen, the size it set, and the token / motion-vector / mode probabilities (after a frame with
  // refresh_entropy_probs = 0, those from before that frame).
  bool have_key() const { return have_key_; }
  int width() const { return width_; }
  int height() const { return height_; }
  const EntropyTables &probs() const { return probs_; }

 private:
  int Fail(int code, const std::string &msg) {
    error_ = msg;
    return code;
  }
  void LoadDefaults();
  bool refresh_entropy_ = true;  // of the frame being parsed (ParseHeader -> Parse)
  int ParseHeader(const uint8_t *data, size_t size, vp8r_frame *out);
  int ParseMacroblocks(vp8r_frame *out);
  void ParseInterMb(int r, int c, int idx, int ref, vp8r_mb_info *mb, vp8r_frame *out, bool *split);
  int16_t ReadMvComponent(const uint8_t *p);
  // Most blocks are empty: their first symbol is the end-of-block branch.  That test is inlined
  // into the macroblock loop; only non-empty blocks pay for the call into the token loop.
  inline int ReadCoefBlock(BoolReader &br, int type, int ctx, int first, int dc_f, int ac_f, int16_t *dst,
                           bool *nz_after_dequant) {
    static constexpr uint8_t kFirstBand[2] = {0, 1};  // band of coefficient 0 / coefficient 1
    if (!br.Bit(probs_.coef[type][kFirstBand[first]][ctx][0])) {
      *nz_after_dequant = false;
      return 0;
    }
    return ReadCoefTokens(br, type, ctx, first, dc_f, ac_f, dst, nz_after_dequant);
  }
  int ReadCoefTokens(BoolReader &br, int type, int ctx, int first, int dc_f, int ac_f, int16_t *dst,
                     bool *nz_after_dequant);
  bool EnsurePayload(vp8r_frame *out, size_t blocks_needed);
  bool BuildIntraLevels(vp8r_frame *out);
  bool AttachTokenPartitions(vp8r_frame *out);
  static constexpr unsigned kMaxFlatIntraLevels = 48;
  // Largest frame (macroblocks) whose tokens / modes are deferred: the device parse kernel keeps two
  // bytes per macroblock in shared memory.  Larger frames are parsed on the host as usual.
  static constexpr size_t kMaxDeferMbs = 65536;

  // ---- state that persists between frames (ParserContext, src/bitstream_parser.h:124-182) ----
  bool have_key_ = false;
  int width_ = 0, height_ = 0, mb_cols_ = 0, mb_rows_ = 0;
  EntropyTables probs_;
  uint8_t segment_tree_probs_[3];
  int8_t ref_lf_delta_[4], mode_lf_delta_[4];
  int segment_abs_ = 0;
  int16_t segment_quant_[4], segment_lf_[4];
  std::vector<uint8_t> segment_map_;

  // ---- per-frame scratch ----
  BoolReader first_;
  BoolReader dct_[8];
  const uint8_t *dct_data_[8] = {};  // start / size of each DCT partition inside the compressed frame
  size_t dct_size_[8] = {};
  int n_dct_parts_ = 1;
  bool defer_tokens_ = false, defer_modes_ = false;          // what the caller asked for
  bool want_defer_tokens_ = false, want_defer_modes_ = false;
  const uint8_t *first_data_ = nullptr;  // first partition inside the compressed frame
  size_t first_size_ = 0;
  bool key_frame_ = false;
  int version_ = 0;
  bool segmentation_enabled_ = false, update_segment_map_ = false;
  bool lf_adj_enable_ = false;
  bool mb_no_skip_coeff_ = false;
  int prob_skip_false_ = 0, prob_intra_ = 0, prob_last_ = 0, prob_gf_ = 0;
  int frame_lf_level_ = 0;
  int y_ac_qi_ = 0;
  bool sign_bias_[4] = {false, false, false, false};
  std::vector<MbCtx> mbctx_;          // per MB of the frame
  std::vector<Mv> sub_mvs_;           // 16 per MB (zero for intra MBs; src/decode.cc:71)
  std::vector<uint8_t> above_bmodes_; // 4 per MB column (key frames)
  std::vector<uint8_t> nz_above_y_, nz_above_u_, nz_above_v_, nz_above_y2_;  // per 4x4 column
  std::vector<uint16_t> levels_;      // intra dependency level + 1 per MB (0 = inter)
  std::vector<uint32_t> cursor_;
  std::string error_;
};

}  // namespace vp8r

struct vp8r_parser {
  vp8r::FrameParser impl;
};

#endif  // VP8R_HOST_FRAME_PARSER_H_
