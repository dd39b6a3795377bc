// Neighbour motion-vector search of an inter macroblock (RFC 6386 section 18.3; src/inter_predict.cc:8-93 of the
// reference): the best / nearest / near vectors and the mode contexts `cnt` that select the probabilities of the
// mode tree.  One copy, shared by the parser (which reads the mode) and the writer (which codes it).
#ifndef VP8R_HOST_NEAR_MVS_H_
#define VP8R_HOST_NEAR_MVS_H_

#include <cstdint>
#include <utility>

namespace vp8r {

enum { MV_NEAREST = 0, MV_NEAR, MV_ZERO, MV_NEW, MV_SPLIT };

// {row, col} in 1/8 pel (quarter-pel values doubled), as vp8r_mb_info.mv.
struct Mv {
  int16_t r, c;
  bool operator==(const Mv &o) const { return r == o.r && c == o.c; }
  bool operator!=(const Mv &o) const { return !(*this == o); }
  bool nonzero() const { return (r | c) != 0; }
};

// What later macroblocks need to know about an earlier one of the same frame.
struct MbCtx {
  uint8_t is_inter;
  uint8_t ref;   // 0 intra, 1 last, 2 golden, 3 altref
  uint8_t mode;  // inter: MV_* mode
  Mv mv;         // representative MV (block 15 for SPLIT), src/inter_predict.cc:232-233
};

struct NearMvs {
  Mv best, nearest, near;  // clamped (ClampMV2, src/inter_predict.cc:83-93,201-203)
  int cnt[4];              // mode contexts: row i of kProbMvRef gives the probability of tree node i
};

// Macroblock (r, c) of a cols x rows frame that predicts from `ref`; `ctx` holds the already coded macroblocks in
// raster order, sign_bias[k] the sign bias of reference frame k.
inline NearMvs FindNearMvs(const MbCtx *ctx, int r, int c, int cols, int rows, int ref, const bool sign_bias[4]) {
  const int idx = r * cols + c;
  int cnt[4] = {0, 0, 0, 0};
  Mv mv[4] = {{0, 0}, {0, 0}, {0, 0}, {0, 0}};
  int ptr = 0;
  auto flip = [&](Mv v, int other_ref) {
    if (sign_bias[other_ref] != sign_bias[ref]) return Mv{int16_t(-v.r), int16_t(-v.c)};
    return v;
  };
  const MbCtx *above = r > 0 ? &ctx[idx - cols] : nullptr;
  const MbCtx *left = c > 0 ? &ctx[idx - 1] : nullptr;
  const MbCtx *aboveleft = (r > 0 && c > 0) ? &ctx[idx - cols - 1] : nullptr;
  if (above && above->is_inter) {
    Mv v = above->mv;
    if (v.nonzero()) mv[++ptr] = flip(v, above->ref);
    cnt[ptr] += 2;
  }
  if (left && left->is_inter) {
    Mv v = left->mv;
    if (v.nonzero()) {
      v = flip(v, left->ref);
      if (mv[ptr] != v) mv[++ptr] = v;
      cnt[ptr] += 2;
    } else {
      cnt[0] += 2;
    }
  }
  if (aboveleft && aboveleft->is_inter) {
    Mv v = aboveleft->mv;
    if (v.nonzero()) {
      v = flip(v, aboveleft->ref);
      if (mv[ptr] != v) mv[++ptr] = v;
      cnt[ptr] += 1;
    } else {
      cnt[0] += 1;
    }
  }
  if (cnt[3] && mv[ptr] == mv[1]) ++cnt[1];
  cnt[3] = ((above && above->is_inter && above->mode == MV_SPLIT) ? 2 : 0) +
           ((left && left->is_inter && left->mode == MV_SPLIT) ? 2 : 0) +
           ((aboveleft && aboveleft->is_inter && aboveleft->mode == MV_SPLIT) ? 1 : 0);
  if (cnt[2] > cnt[1]) {
    std::swap(cnt[1], cnt[2]);
    std::swap(mv[1], mv[2]);
  }
  if (cnt[1] >= cnt[0]) mv[0] = mv[1];

  const int to_top = -(r * 16) * 8, to_bottom = ((rows - 1 - r) * 16) * 8;
  const int to_left = -(c * 16) * 8, to_right = ((cols - 1 - c) * 16) * 8;
  auto clamp2 = [&](Mv v) {
    if (v.c < to_left - 128) v.c = int16_t(to_left - 128);
    else if (v.c > to_right + 128) v.c = int16_t(to_right + 128);
    if (v.r < to_top - 128) v.r = int16_t(to_top - 128);
    else if (v.r > to_bottom + 128) v.r = int16_t(to_bottom + 128);
    return v;
  };
  NearMvs out;
  out.best = clamp2(mv[0]);
  out.nearest = clamp2(mv[1]);
  out.near = clamp2(mv[2]);
  for (int i = 0; i < 4; ++i) out.cnt[i] = cnt[i];
  return out;
}

}  // namespace vp8r

#endif  // VP8R_HOST_NEAR_MVS_H_
