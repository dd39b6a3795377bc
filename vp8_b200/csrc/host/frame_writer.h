// Bitstream writer: the inverse of FrameParser for the frames the encoder produces (row f4).
#ifndef VP8R_HOST_FRAME_WRITER_H_
#define VP8R_HOST_FRAME_WRITER_H_

#include <cstdint>
#include <string>
#include <vector>

#include "parsed_frame.h"

namespace vp8r {

class FrameParser;

// Serialises a parsed-frame structure into a VP8 frame (RFC 6386 sections 9, 19.2, 19.3, 13): frame tag (+ start
// code and dimensions of a key frame), first partition (headers, "keep the token / mode / motion-vector
// probabilities", per-macroblock skip flag, modes and motion vectors), one token partition.  The probabilities are
// those the frame will be decoded with: the defaults for a key frame or when `context` is null, else the context
// parser's current ones (the stream's state after what that parser has parsed).  The frame carries no updates and
// sets refresh_entropy_probs, so the context is the same after it.  VP8R_ERR_STATE: for an inter frame, a context
// parser that has not parsed a key frame or whose frame size differs.  Frames it can write: one DCT partition, no
// segmentation, no loop-filter deltas, quantiser factors that q_index and five deltas reproduce; key frames with intra macroblocks, inter frames with intra macroblocks
// and inter macroblocks of any reference coded NEAREST / NEAR / ZERO / NEW (SPLIT is refused, and so is a vector
// that contradicts its mode).  Parsing the result with FrameParser gives back the same macroblock records and
// coefficient blocks.  Returns VP8R_OK or an error code with *err set.
int WriteFrame(const vp8r_frame &f, const FrameParser *context, std::vector<uint8_t> *out, std::string *err);

// Mode bits of the inter macroblocks of a frame whose records carry vectors but no modes (the encoder's): walking
// the macroblocks in raster order, each vector gets the cheapest mode consistent with it under the mode tree's
// probabilities (NEAREST if it equals the nearest vector, NEAR if the near one, ZERO if it is zero; the most probable
// of those that apply, else NEW).  The vector itself is never changed.  Sign biases are taken as 0.
// VP8R_ERR_INVALID_ARG when a NEW vector lies too far from its predictor (|delta| > 1023 quarter pels).
int AssignInterModes(vp8r_mb_info *mbs, int cols, int rows, std::string *err);

}  // namespace vp8r

#endif  // VP8R_HOST_FRAME_WRITER_H_
