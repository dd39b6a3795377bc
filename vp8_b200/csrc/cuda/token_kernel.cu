// K_tokens: device-side decode of the DCT token partitions (frames parsed with deferred tokens).
//
// Replaces, for those frames, the residual half of the host parser: ResidualTokens / the token
// loop of src/bitstream_parser.cc:466-537,572-621 driven by the bool decoder of
// src/bool_decoder.cc:13-41, plus the non-zero context hand-over of src/decode_frame.cc:6-47,111-130.
//
// Parallelism is what the bitstream offers: a bool-coded partition is a serial chain, but the
// 1/2/4/8 DCT partitions of a frame are separate chains (MB row r lives in partition r % n) that
// only meet through the "above" non-zero context, and frames of different streams are independent.
// One CTA per frame, one warp per partition with a single working lane; rows advance as a pipeline:
// row r may decode macroblock c once row r-1 has published c.  With a few hundred frames per batch
// that is ~1000 independent chains on 148 SMs, each bound by the latency of its own dependent
// integer chain (~25 instructions per boolean), which is what a GPU thread is slow at and many
// GPU threads together are fast at.
//
// Output: coefficient blocks (de-zigzagged int16, not dequantised) into the frame's device
// coefficient area, row r compact inside its own region starting at block r * cols * 25;
// coef_mask / coef_offset / VP8R_MB_LF_INNER of every vp8r_mb_info are completed in place.
//
// Deferred modes (vp8r_frame_hdr.modes_deferred): K_modes, a kernel of its own with one single-lane warp per
// frame, reads the per-macroblock syntax of the first partition (segment id, skip flag, intra modes incl. the 16
// B_PRED sub-modes, reference frame, the near/nearest/best motion-vector search, NEW and SPLIT vectors) in raster
// order, writes the vp8r_mb_info records the reconstruction kernels consume, computes the loop-filter level of
// every macroblock and the intra dependency levels of inter frames.  Replaces ParseMacroblocks / ParseInterMb /
// BuildIntraLevels of host/frame_parser.cc, i.e. src/bitstream_parser.cc:320-464,539-568,
// src/inter_predict.cc:8-244, src/intra_predict.cc:176-183 of the reference.
//
// A header chain is the longest serial chain of a frame (~29 ms for 1080p against ~12 ms for a token partition)
// and needs nothing of the frame before it EXCEPT the persistent segment map.  So the map is taken out of the
// chain: K_modes never touches it, and K_segments, a one-thread-per-macroblock kernel the engine runs in batch
// order, stores the ids of frames that code a map and patches segment / loop-filter level into the records of
// frames that inherit it.  That leaves the header kernels of consecutive time steps free to run side by side
// (one engine stream per batch slot), which is where the parse throughput comes from: a 32-thread CTA with
// ~14 KB of shared memory lets sixteen chains share an SM instead of five frame-CTAs that each wait for their
// slowest chain.
#include "recon_kernels.h"

namespace vp8r {

namespace host_tables {
#include "../host/vp8_prob_tables.inc"
}

namespace {

enum { DC_PRED = 0, V_PRED, H_PRED, TM_PRED, B_PRED };
enum { MV_NEAREST = 0, MV_NEAR, MV_ZERO, MV_NEW, MV_SPLIT };
enum { B_DC = 0, B_TM, B_VE, B_HE, B_LD, B_RD, B_VR, B_VL, B_HD, B_HU };
enum { SUB_LEFT = 0, SUB_ABOVE, SUB_ZERO, SUB_NEW };

// Fixed trees and probabilities of the macroblock header (RFC 6386 sections 8.1, 9.3, 11.2-11.5,
// 16.3, 17; reference: src/bitstream_const.h).  Copied to shared memory by every CTA.
struct ModeTables {
  signed char tree_ymode_key[8], tree_ymode[8], tree_uvmode[6], tree_bmode[18], tree_segment[6], tree_mvref[8],
      tree_split[6], tree_submv[6], tree_smallmv[14];
  unsigned char prob_ymode_key[4], prob_uvmode_key[3], prob_bmode_inter[9], prob_split[3], prob_submv[5][3],
      prob_mvref[6][4];
  unsigned char split_count[4], split_head[4][16];
  unsigned short split_mask[4][16];  // [layout][partition]: the sub-blocks it covers
  unsigned char kf_bmode[900];
};
__constant__ ModeTables c_mode_tables;

const ModeTables kModeTablesInit = {
    {-B_PRED, 2, 4, 6, -DC_PRED, -V_PRED, -H_PRED, -TM_PRED},
    {-DC_PRED, 2, 4, 6, -V_PRED, -H_PRED, -TM_PRED, -B_PRED},
    {-DC_PRED, 2, -V_PRED, 4, -H_PRED, -TM_PRED},
    {-B_DC, 2, -B_TM, 4, -B_VE, 6, 8, 12, -B_HE, 10, -B_RD, -B_VR, -B_LD, 14, -B_VL, 16, -B_HD, -B_HU},
    {2, 4, -0, -1, -2, -3},
    {-MV_ZERO, 2, -MV_NEAREST, 4, -MV_NEAR, 6, -MV_NEW, -MV_SPLIT},
    {-3, 2, -2, 4, -0, -1},
    {-SUB_LEFT, 2, -SUB_ABOVE, 4, -SUB_ZERO, -SUB_NEW},
    {2, 8, 4, 6, -0, -1, -2, -3, 10, 12, -4, -5, -6, -7},
    {145, 156, 163, 128},
    {142, 114, 183},
    {120, 90, 79, 133, 87, 85, 80, 111, 151},
    {110, 111, 150},
    {{147, 136, 18}, {106, 145, 1}, {179, 121, 1}, {223, 1, 34}, {208, 1, 1}},
    {{7, 1, 1, 143}, {14, 18, 14, 107}, {135, 64, 57, 68}, {60, 56, 128, 65}, {159, 134, 128, 34}, {234, 188, 128, 28}},
    {2, 2, 4, 16},
    {{0, 8}, {0, 2}, {0, 2, 8, 10}, {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15}},
    {{0x00ff, 0xff00},
     {0x3333, 0xcccc},
     {0x0033, 0x00cc, 0x3300, 0xcc00},
     {0x0001, 0x0002, 0x0004, 0x0008, 0x0010, 0x0020, 0x0040, 0x0080, 0x0100, 0x0200, 0x0400, 0x0800, 0x1000, 0x2000,
      0x4000, 0x8000}},
    {0}};

__constant__ unsigned char c_band[17] = {0, 1, 2, 3, 6, 4, 5, 6, 6, 6, 6, 6, 6, 6, 6, 7, 0};
__constant__ unsigned char c_zigzag[16] = {0, 1, 4, 8, 5, 2, 3, 6, 9, 12, 13, 10, 7, 11, 14, 15};
// DCT_CAT extra-bit probabilities, 12 per category, zero terminated (src/bitstream_const.h:89-90).
__constant__ unsigned char c_cat[6][12] = {{159, 0},
                                           {165, 145, 0},
                                           {173, 148, 140, 0},
                                           {176, 155, 140, 135, 0},
                                           {180, 157, 141, 134, 130, 0},
                                           {254, 254, 243, 230, 196, 177, 153, 140, 133, 130, 129, 0}};
__constant__ short c_cat_base[6] = {5, 7, 11, 19, 35, 67};

// RFC 6386 section 7 boolean decoder, 64-bit left-aligned window refilled 32 bits at a time with
// aligned loads.  Produces the bit sequence of src/bool_decoder.cc:13-41.
struct BoolDec {
  const unsigned *next, *end;  // next aligned word to append / first word without a byte of the partition
  unsigned long long win;      // upcoming bits, left aligned
  int avail;                   // valid bits in win
  unsigned range;              // 128..255
  int loaded;                  // bytes appended so far (for the over-read test)

  // The reader is bounded to ITS partition at word granularity: past the last word that holds partition bytes it
  // sees zeros, like the reference's byte-at-a-time reader and the host reader (it must not walk into the next
  // partition).  Up to three bytes behind the end may come from the neighbour inside that last word; they cannot
  // reach a decision of a frame that is kept: a reader that needs them has consumed more bytes than the partition
  // has, which BytesConsumed() reports and which stops the frame (JobFailed).  A mask for those bytes was
  // measured: +8 % parse-kernel time for the extra compare at every refill site.
  __device__ __forceinline__ void Bound(const unsigned char *lim) {
    end = reinterpret_cast<const unsigned *>(lim + ((4u - ((unsigned)(size_t)lim & 3u)) & 3u));
  }
  __device__ __forceinline__ unsigned Word(const unsigned *p) const { return p < end ? __ldg(p) : 0u; }
  __device__ __forceinline__ unsigned Byte(const unsigned char *p) const {
    return p < reinterpret_cast<const unsigned char *>(end) ? (unsigned)*p : 0u;
  }

  __device__ __forceinline__ void Refill() {
    const unsigned w0 = Word(next);
    unsigned w = w0;
    ++next;
    w = __byte_perm(w, 0, 0x0123);  // big endian
    win |= (unsigned long long)w << (32 - avail);
    avail += 32;
    loaded += 4;
  }
  __device__ __forceinline__ void Init(const unsigned char *raw, unsigned off, const unsigned char *lim) {
    const unsigned mis = off & 3u;
    next = reinterpret_cast<const unsigned *>(raw + (off - mis));
    Bound(lim);
    unsigned w = Word(next);
    ++next;
    w = __byte_perm(w, 0, 0x0123) << (8 * mis);
    win = (unsigned long long)w << 32;
    avail = 32 - 8 * (int)mis;
    loaded = 4 - (int)mis;
    range = 255;
    Refill();
  }
  // Resumes a decoder handed over by the host after the frame headers (vp8r_mode_hdr): the window
  // is `value` (8 bits) followed by the raw stream from bit `bitpos` of the partition on.
  __device__ __forceinline__ void InitAt(const unsigned char *raw, unsigned part_off, unsigned bitpos, unsigned value,
                                         unsigned rng, const unsigned char *lim) {
    unsigned at = part_off + (bitpos >> 3);  // byte offset in the raw section
    const unsigned sub = bitpos & 7u;
    Bound(lim);
    win = (unsigned long long)value << 56;
    avail = 8;
    unsigned b = Byte(raw + at);
    ++at;
    win |= (unsigned long long)(b & (0xffu >> sub)) << (48 + sub);
    avail += 8 - (int)sub;
    while (at & 3u) {
      b = Byte(raw + at);
      ++at;
      win |= (unsigned long long)b << (56 - avail);
      avail += 8;
    }
    next = reinterpret_cast<const unsigned *>(raw + at);
    loaded = (int)(at - part_off);
    range = rng;
    if (avail <= 32) Refill();
  }
  // Walks an RFC 6386 tree: positive entries are next-node indices, entries <= 0 negated leaves.
  __device__ __forceinline__ int Tree(const signed char *tree, const unsigned char *probs) {
    int i = 0;
    do {
      i = tree[i + Bit(probs[i >> 1])];
    } while (i > 0);
    return -i;
  }
  // One boolean, probability prob/256 of being 0.
  __device__ __forceinline__ int Bit(unsigned prob) {
    const unsigned split = 1u + (((range - 1u) * prob) >> 8);
    const unsigned big = split << 24;
    unsigned hi = (unsigned)(win >> 32);
    const int bit = hi >= big;
    if (bit) {
      hi -= big;
      range -= split;
    } else {
      range = split;
    }
    const int sh = __clz(range) - 24;
    range <<= sh;
    win = (((unsigned long long)hi << 32) | (unsigned)win) << sh;
    avail -= sh;
    if (avail <= 32) Refill();
    return bit;
  }
  // Bytes the reference's byte-at-a-time reader would have consumed (see host/bool_reader.h).
  __device__ __forceinline__ int BytesConsumed() const { return 2 + ((8 * loaded - avail) >> 3); }
};

struct TokenShared {
  unsigned char probs[4 * 8 * 3 * 11];
  int progress[8];      // progress[w]: macroblocks finished by partition w, counted along its rows
  short blk[8][16];     // staging of the block being decoded, one per warp
};

// Tokens of one block whose first symbol was not end-of-block (src/bitstream_parser.cc:572-621).
// Returns bit 0: some coefficient is non-zero; bit 1: some coefficient is non-zero after the
// reference's int16 dequantisation (src/decode_frame.cc:6-47).
__device__ __forceinline__ int ReadTokens(BoolDec &bd, const unsigned char *probs, int type, int ctx, int first,
                                          int dc_f, int ac_f, short *blk) {
  const unsigned char *bands = probs + type * (8 * 3 * 11);
  int n = first;
  const unsigned char *p = bands + (c_band[n] * 3 + ctx) * 11;
  int any = 0, dq_any = 0;
  bool first_symbol = true;
  while (n < 16) {
    if (!first_symbol && !bd.Bit(p[0])) break;
    first_symbol = false;
    bool ended = false;
    while (!bd.Bit(p[1])) {
      if (++n == 16) {
        ended = true;
        break;
      }
      p = bands + (c_band[n] * 3) * 11;
    }
    if (ended) break;
    int v;
    if (!bd.Bit(p[2])) {
      v = 1;
    } else if (!bd.Bit(p[3])) {
      v = !bd.Bit(p[4]) ? 2 : 3 + bd.Bit(p[5]);
    } else {
      int cat;
      if (!bd.Bit(p[6])) cat = bd.Bit(p[7]);
      else if (!bd.Bit(p[8])) cat = 2 + bd.Bit(p[9]);
      else cat = 4 + bd.Bit(p[10]);
      int extra = 0;
      const unsigned char *q = c_cat[cat];
      for (unsigned pq = *q; pq; pq = *++q) extra = extra + extra + bd.Bit(pq);
      v = c_cat_base[cat] + extra;
    }
    const int next_ctx = v > 1 ? 2 : 1;
    if (bd.Bit(128)) v = -v;
    blk[c_zigzag[n]] = (short)v;
    any = 1;
    if ((short)(v * (n == 0 ? dc_f : ac_f)) != 0) dq_any = 2;
    ++n;
    p = bands + (c_band[n] * 3 + next_ctx) * 11;
  }
  return any | dq_any;
}

}  // namespace

constexpr int kTokenWarps = 8;           // token partitions
constexpr int kMaxFlatLevels = 48;       // as FrameParser::kMaxFlatIntraLevels
constexpr int kMaxLevelMbs = 96 * 1024;  // frames with more macroblocks use the intra wavefront kernel

// Shared memory of K_tokens: TokenShared, then the above-context of every macroblock column.
__host__ __device__ inline size_t TokenSmem(int cols) {
  return ((sizeof(TokenShared) + 15) & ~size_t(15)) + ((size_t(cols) * 2 + 15) & ~size_t(15));
}
// Shared memory of K_modes.
struct ModeLayout {
  size_t tabs, fp, sub, mbctx, above_sub, above_bmodes, levels, cnt, total;
};
__host__ __device__ inline ModeLayout MakeModeLayout(int cols, int n_mb) {
  ModeLayout l;
  size_t at = 0;
  l.tabs = at; at += (sizeof(ModeTables) + 15) & ~size_t(15);
  l.fp = at; at += 64;
  l.sub = at; at += 64;
  l.mbctx = at; at += size_t(cols) * 2 * 8;
  l.above_sub = at; at += size_t(cols) * 16;
  l.above_bmodes = at; at += (size_t(cols) * 4 + 15) & ~size_t(15);
  l.cnt = at; at += ((kMaxFlatLevels + 2) * 4 + 15) & ~size_t(15);
  l.levels = at; at += (size_t(n_mb <= kMaxLevelMbs ? n_mb : 0) + 15) & ~size_t(15);
  l.total = at;
  return l;
}

__device__ __forceinline__ int PackMv(int r, int c) { return (r & 0xffff) | (c << 16); }
__device__ __forceinline__ int MvRow(int v) { return (int)(short)(v & 0xffff); }
__device__ __forceinline__ int MvCol(int v) { return v >> 16; }

// Motion-vector component (src/bitstream_parser.cc:441-464).
__device__ __forceinline__ int ReadMvComponent(BoolDec &bd, const unsigned char *p, const signed char *tree_small) {
  int a = 0;
  if (bd.Bit(p[0])) {
    for (int i = 0; i < 3; ++i) a += bd.Bit(p[9 + i]) << i;
    for (int i = 9; i > 3; --i) a += bd.Bit(p[9 + i]) << i;
    if (!(a & 0xFFF0) || bd.Bit(p[9 + 3])) a += 8;
  } else {
    a = bd.Tree(tree_small, p + 2);
  }
  if (a && bd.Bit(p[1])) a = -a;
  return (int)(short)a;
}

// Loop-filter level of a macroblock (src/bitstream_parser.cc:539-568).  mode_delta: the mode_lf_delta entry that
// applies (B_PRED: [0], ZERO: [1], SPLIT: [3], other inter modes: [2]; 0 for the other intra modes).
__device__ __forceinline__ int MbFilterLevel(int frame_lf, bool seg_enabled, bool seg_abs, int seg_lf, bool lf_adj,
                                             int ref_delta, int ref, int mode_delta) {
  int lvl = frame_lf;
  if (seg_enabled) {
    lvl = seg_abs ? seg_lf : lvl + seg_lf;
    lvl = lvl < 0 ? 0 : (lvl > 63 ? 63 : lvl);
  }
  if (lf_adj) {
    lvl += ref_delta + mode_delta;
    (void)ref;
    lvl = lvl < 0 ? 0 : (lvl > 63 ? 63 : lvl);
  }
  return lvl;
}

// The macroblock-header pass of one frame by one thread (see the file comment).
__device__ void ModeThread(const DevFrameJob &job, const vp8r_token_hdr *th, unsigned char *smem) {
  const vp8r_mode_hdr *mhp = reinterpret_cast<const vp8r_mode_hdr *>(job.mode_hdr);
  const int cols = job.mb_cols, rows = job.mb_rows, n_mb = cols * rows;
  const ModeLayout lay = MakeModeLayout(cols, n_mb);
  const ModeTables &T = *reinterpret_cast<const ModeTables *>(smem + lay.tabs);
  uint2 *mbctx = reinterpret_cast<uint2 *>(smem + lay.mbctx);        // [2][cols]: x = 1 | ref<<1 | mode<<3 (0: intra), y = mv
  int *above_sub = reinterpret_cast<int *>(smem + lay.above_sub);      // [cols][4]: bottom-row sub-block MVs of the MB above
  unsigned char *above_bmodes = smem + lay.above_bmodes;               // [cols*4] (key frames)
  unsigned *cnt = reinterpret_cast<unsigned *>(smem + lay.cnt);        // macroblocks per dependency level
  unsigned char *levels = smem + lay.levels;                           // [n_mb]: 0 inter, k intra of level k-1
  const bool have_levels = n_mb <= kMaxLevelMbs;

  // frame parameters to registers
  const bool key = mhp->key_frame != 0, seg_enabled = mhp->segmentation_enabled != 0, update_map = mhp->update_segment_map != 0;
  const bool no_skip = mhp->mb_no_skip_coeff != 0, lf_adj = mhp->lf_adj_enable != 0, seg_abs = mhp->segment_abs != 0;
  const unsigned prob_skip = mhp->prob_skip_false, prob_intra = mhp->prob_intra, prob_last = mhp->prob_last, prob_gf = mhp->prob_gf;
  const int frame_lf = mhp->frame_lf_level;
  unsigned sign_bias = 0;
  for (int i = 0; i < 4; ++i) sign_bias |= (unsigned)(mhp->sign_bias[i] != 0) << i;
  int *sub = reinterpret_cast<int *>(smem + lay.sub);  // sub-block motion vectors of the current SPLIT macroblock
  unsigned char *fp = smem + lay.fp;                   // [0..3] ymode, [4..6] uvmode, [8..10] segment tree, [16..53] mv
  for (int i = 0; i < 4; ++i) fp[i] = mhp->ymode_probs[i];
  for (int i = 0; i < 3; ++i) fp[4 + i] = mhp->uvmode_probs[i], fp[8 + i] = mhp->segment_tree_probs[i];
  for (int i = 0; i < 38; ++i) fp[16 + i] = (&mhp->mv_probs[0][0])[i];
  int seg_lf[4], ref_delta[4], mode_delta[4];
  for (int i = 0; i < 4; ++i) seg_lf[i] = mhp->segment_lf[i], ref_delta[i] = mhp->ref_lf_delta[i], mode_delta[i] = mhp->mode_lf_delta[i];

  const unsigned char *raw = reinterpret_cast<const unsigned char *>(th) + sizeof(vp8r_token_hdr);
  BoolDec bd;
  bd.InitAt(raw, mhp->first_off, mhp->bitpos, mhp->value, mhp->range, raw + mhp->first_off + mhp->first_size);

  vp8r_mb_info *mbs = const_cast<vp8r_mb_info *>(job.mbs);
  int16_t *payload = const_cast<int16_t *>(job.payload);
  unsigned n_inter = 0, n_split = 0, max_level = 0;
  bool level_overflow = !have_levels;

  for (int r = 0; r < rows; ++r) {
    uint2 *ctx_cur = mbctx + (r & 1) * cols;
    const uint2 *ctx_abv = mbctx + ((r & 1) ^ 1) * cols;
    uint2 left_ctx = make_uint2(0, 0), aboveleft_ctx = make_uint2(0, 0);
    int left_sub[4] = {0, 0, 0, 0};
    unsigned left_bmodes = 0;  // 4 x 4 bits, B_DC = 0
    unsigned left_level = 0, aboveleft_level = 0;
    const int to_top = -(r * 16) * 8, to_bottom = ((rows - 1 - r) * 16) * 8;

    for (int c = 0; c < cols; ++c) {
      const int idx = r * cols + c;
      const uint2 above_ctx = r > 0 ? ctx_abv[c] : make_uint2(0, 0);
      // --- pre-header (src/bitstream_parser.cc:320-352) ---
      // Without a coded map the id is inherited from the persistent map: K_segments fills it in (and the level
      // that hangs on it) after this kernel; nothing else of the syntax depends on it.
      const int seg = update_map ? bd.Tree(T.tree_segment, fp + 8) : 0;
      const int skip = no_skip ? bd.Bit(prob_skip) : 0;
      const int is_inter = key ? 0 : bd.Bit(prob_intra);

      unsigned flags = 0, aux0 = 0, aux1 = 0;
      int mbmv = 0, ref = 0, inter_mode = 0;
      bool split = false, bpred = false;
      if (is_inter) {
        ref = bd.Bit(prob_last) ? 2 + bd.Bit(prob_gf) : 1;
        // ---- neighbour search (src/inter_predict.cc:8-81) ----
        int cn[4] = {0, 0, 0, 0};
        int mv[4] = {0, 0, 0, 0};
        int ptr = 0;
        const unsigned my_bias = (sign_bias >> ref) & 1u;
        auto flip = [&](int v, unsigned other_ref) {
          if (((sign_bias >> other_ref) & 1u) != my_bias) return PackMv(-MvRow(v), -MvCol(v));
          return v;
        };
        if (above_ctx.x & 1u) {
          int v = (int)above_ctx.y;
          if (v) mv[++ptr] = flip(v, (above_ctx.x >> 1) & 3u);
          cn[ptr] += 2;
        }
        if (left_ctx.x & 1u) {
          int v = (int)left_ctx.y;
          if (v) {
            v = flip(v, (left_ctx.x >> 1) & 3u);
            if (mv[ptr] != v) mv[++ptr] = v;
            cn[ptr] += 2;
          } else {
            cn[0] += 2;
          }
        }
        if (aboveleft_ctx.x & 1u) {
          int v = (int)aboveleft_ctx.y;
          if (v) {
            v = flip(v, (aboveleft_ctx.x >> 1) & 3u);
            if (mv[ptr] != v) mv[++ptr] = v;
            cn[ptr] += 1;
          } else {
            cn[0] += 1;
          }
        }
        if (cn[3] && mv[ptr] == mv[1]) ++cn[1];
        auto is_split = [](uint2 x) { return (x.x & 1u) && ((x.x >> 3) & 7u) == MV_SPLIT; };
        cn[3] = (is_split(above_ctx) ? 2 : 0) + (is_split(left_ctx) ? 2 : 0) + (is_split(aboveleft_ctx) ? 1 : 0);
        if (cn[2] > cn[1]) {
          int t = cn[1]; cn[1] = cn[2]; cn[2] = t;
          t = mv[1]; mv[1] = mv[2]; mv[2] = t;
        }
        if (cn[1] >= cn[0]) mv[0] = mv[1];
        unsigned char p[4];
        for (int i = 0; i < 4; ++i) p[i] = T.prob_mvref[cn[i]][i];
        int i = 0;  // kTreeMvRef walk with the four context-selected probabilities
        do {
          i = T.tree_mvref[i + bd.Bit(p[i >> 1])];
        } while (i > 0);
        inter_mode = -i;
        // best / nearest / near are always clamped (src/inter_predict.cc:83-93,201-203)
        const int to_left = -(c * 16) * 8, to_right = ((cols - 1 - c) * 16) * 8;
        auto clamp2 = [&](int v) {
          int vr = MvRow(v), vc = MvCol(v);
          vc = vc < to_left - 128 ? to_left - 128 : (vc > to_right + 128 ? to_right + 128 : vc);
          vr = vr < to_top - 128 ? to_top - 128 : (vr > to_bottom + 128 ? to_bottom + 128 : vr);
          return PackMv(vr, vc);
        };
        const int best = clamp2(mv[0]), nearest = clamp2(mv[1]), near = clamp2(mv[2]);
        auto read_new = [&]() {
          const int dr = (int)(short)(ReadMvComponent(bd, fp + 16, T.tree_smallmv) * 2);
          const int dc = (int)(short)(ReadMvComponent(bd, fp + 16 + 19, T.tree_smallmv) * 2);
          return PackMv(dr + MvRow(best), dc + MvCol(best));  // no re-clamp (src/inter_predict.cc:224-228)
        };
        switch (inter_mode) {
          case MV_NEAREST: mbmv = nearest; break;
          case MV_NEAR: mbmv = near; break;
          case MV_ZERO: break;
          case MV_NEW: mbmv = read_new(); break;
          default: {  // MV_SPLIT (src/inter_predict.cc:146-184)
            split = true;
            const int layout = bd.Tree(T.tree_split, T.prob_split);
            const int n_part = T.split_count[layout];
            for (int part = 0; part < n_part; ++part) {
              const int k = T.split_head[layout][part];
              const int lmv = (k & 3) ? sub[k - 1] : left_sub[k >> 2];
              const int amv = (k >= 4) ? sub[k - 4] : (r == 0 ? 0 : above_sub[c * 4 + k]);
              int sctx;
              if (lmv == amv) sctx = amv ? 3 : 4;
              else if (!amv) sctx = 2;
              else if (!lmv) sctx = 1;
              else sctx = 0;
              const int sm = bd.Tree(T.tree_submv, T.prob_submv[sctx]);
              int v;
              if (sm == SUB_LEFT) v = lmv;
              else if (sm == SUB_ABOVE) v = amv;
              else if (sm == SUB_ZERO) v = 0;
              else v = read_new();
              const unsigned members = T.split_mask[layout][part];
#pragma unroll
              for (int b = 0; b < 16; ++b)
                if ((members >> b) & 1u) sub[b] = v;
            }
            mbmv = sub[15];
            break;
          }
        }
        flags = VP8R_MB_IS_INTER | ((unsigned)ref << VP8R_MB_REF_SHIFT) | ((unsigned)inter_mode << VP8R_MB_MODE_SHIFT);
        if (split) {
          // the 16 vectors go to this frame's split area: two payload blocks per SPLIT macroblock
          const unsigned at = job.split_base + 2u * n_split;
          int *dst = reinterpret_cast<int *>(payload + (size_t)at * 16);
          for (int b = 0; b < 16; b += 4) *reinterpret_cast<int4 *>(dst + b) = make_int4(sub[b], sub[b + 1], sub[b + 2], sub[b + 3]);
          aux0 = at;
          ++n_split;
        }
        ++n_inter;
      } else {
        const int ymode = key ? bd.Tree(T.tree_ymode_key, T.prob_ymode_key) : bd.Tree(T.tree_ymode, fp);
        bpred = ymode == B_PRED;
        if (bpred) {  // src/intra_predict.cc:176-183
          unsigned char *abm = above_bmodes + c * 4;
          unsigned lb = left_bmodes;
          for (int i = 0; i < 4; ++i)
            for (int j = 0; j < 4; ++j) {
              int m;
              if (key) {
                const int l = (int)((lb >> (4 * i)) & 15u);
                m = bd.Tree(T.tree_bmode, T.kf_bmode + (abm[j] * 10 + l) * 9);
                abm[j] = (unsigned char)m;
                lb = (lb & ~(15u << (4 * i))) | ((unsigned)m << (4 * i));
              } else {
                m = bd.Tree(T.tree_bmode, T.prob_bmode_inter);
              }
              const int b = i * 4 + j;
              if (b < 8) aux0 |= (unsigned)m << (b * 4);
              else aux1 |= (unsigned)m << ((b - 8) * 4);
            }
          left_bmodes = lb;
        } else if (key) {
          const unsigned implied = ymode == DC_PRED ? B_DC : (ymode == V_PRED ? B_VE : (ymode == H_PRED ? B_HE : B_TM));
          for (int i = 0; i < 4; ++i) above_bmodes[c * 4 + i] = (unsigned char)implied;
          left_bmodes = implied * 0x1111u;
        }
        const int uvmode = key ? bd.Tree(T.tree_uvmode, T.prob_uvmode_key) : bd.Tree(T.tree_uvmode, fp + 4);
        flags = ((unsigned)ymode << VP8R_MB_MODE_SHIFT) | ((unsigned)uvmode << VP8R_MB_UVMODE_SHIFT);
      }

      // --- loop-filter level (src/bitstream_parser.cc:539-568), flags ---
      const bool has_y2 = is_inter ? !split : !bpred;
      const int qseg = seg_enabled ? seg : 0;
      const int lvl = MbFilterLevel(frame_lf, seg_enabled, seg_abs, seg_lf[seg], lf_adj, ref_delta[ref], ref,
                                    ref == 0 ? (bpred ? mode_delta[0] : 0)
                                             : mode_delta[inter_mode == MV_ZERO ? 1 : (inter_mode == MV_SPLIT ? 3 : 2)]);
      flags |= (has_y2 ? VP8R_MB_HAS_Y2 : 0u) | ((unsigned)qseg << VP8R_MB_QSEG_SHIFT) | ((unsigned)lvl << VP8R_MB_LF_SHIFT) |
               ((bpred || split) ? VP8R_MB_LF_INNER : 0u) | (skip ? VP8R_MB_SKIP_COEF : 0u);

      // --- intra dependency level (BuildIntraLevels of the host parser) ---
      unsigned level = 0;
      if (!key && !is_inter && have_levels) {
        unsigned lv = left_level;
        if (r > 0) {
          lv = max(lv, (unsigned)levels[idx - cols]);
          lv = max(lv, aboveleft_level);
          if (c + 1 < cols) lv = max(lv, (unsigned)levels[idx - cols + 1]);
        }
        level = lv + 1;
        if (level > (unsigned)kMaxFlatLevels) {
          level_overflow = true;
          level = kMaxFlatLevels;  // keeps the byte array in range; the table is not used then
        } else {
          cnt[level - 1]++;
        }
        max_level = max(max_level, level);
      }
      if (have_levels) {
        aboveleft_level = r > 0 ? levels[idx - cols] : 0u;
        levels[idx] = (unsigned char)level;
      }
      left_level = level;

      // --- the macroblock record ---
      int4 *rec = reinterpret_cast<int4 *>(mbs + idx);
      rec[0] = make_int4((int)flags, 0, 0, mbmv);
      rec[1] = make_int4((int)aux0, (int)aux1, 0, 0);

      // --- contexts for the macroblocks to come ---
      aboveleft_ctx = above_ctx;
      const uint2 me = is_inter ? make_uint2(1u | ((unsigned)ref << 1) | ((unsigned)inter_mode << 3), (unsigned)mbmv) : make_uint2(0, 0);
      ctx_cur[c] = me;
      left_ctx = me;
      if (!key) {
        if (split) {
          for (int k = 0; k < 4; ++k) above_sub[c * 4 + k] = sub[12 + k], left_sub[k] = sub[4 * k + 3];
        } else {
          for (int k = 0; k < 4; ++k) above_sub[c * 4 + k] = mbmv, left_sub[k] = mbmv;
        }
      }
    }
  }

  // --- intra dependency levels -> table for the level-scheduled intra kernel ---
  DevFrameDyn *dyn = job.dyn;
  unsigned n_levels = 0;
  const unsigned n_intra = (unsigned)n_mb - n_inter;
  if (!key && n_intra > 0 && !level_overflow) {
    unsigned *tab = job.level_table;  // max_level+1 offsets, then the macroblock indices
    unsigned run = 0;
    for (unsigned k = 0; k < max_level; ++k) {
      tab[k] = run;
      const unsigned n = cnt[k];
      cnt[k] = run;  // becomes the write cursor
      run += n;
    }
    tab[max_level] = run;
    unsigned *out = tab + max_level + 1;
    for (int i = 0; i < n_mb; ++i) {
      const unsigned lv = levels[i];
      if (lv) out[cnt[lv - 1]++] = (unsigned)i;
    }
    n_levels = max_level;
  }
  dyn->n_inter = (int)n_inter;
  dyn->n_intra = (int)n_intra;
  dyn->n_intra_levels = (int)n_levels;
  dyn->n_split = (int)n_split;
  if (bd.BytesConsumed() > (int)mhp->first_size && job.status) {
    atomicOr(job.status, 2);
    if (job.status_host) atomicOr(job.status_host, 2);
  }
}

// K_modes: one 32-thread CTA per frame with deferred modes; lane 0 walks the first partition.
__global__ void __launch_bounds__(32) ModeKernel(const DevFrameJob *__restrict__ jobs) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const DevFrameJob &job = jobs[blockIdx.x];
  if (!job.tok_hdr || !job.mode_hdr) return;
  const int cols = job.mb_cols, rows = job.mb_rows;
  const ModeLayout lay = MakeModeLayout(cols, cols * rows);
  for (int i = threadIdx.x; i < (int)(sizeof(ModeTables) + 3) / 4; i += 32)
    reinterpret_cast<unsigned *>(smem_raw + lay.tabs)[i] = reinterpret_cast<const unsigned *>(&c_mode_tables)[i];
  for (int i = threadIdx.x; i < cols * 4; i += 32) smem_raw[lay.above_bmodes + i] = B_DC;
  for (int i = threadIdx.x; i < kMaxFlatLevels + 2; i += 32) reinterpret_cast<unsigned *>(smem_raw + lay.cnt)[i] = 0;
  __syncwarp();
  if (threadIdx.x != 0) return;
  ModeThread(job, reinterpret_cast<const vp8r_token_hdr *>(job.tok_hdr), smem_raw);
}

// K_segments: the persistent segment map of every stream, in batch order (see the file comment).  One thread per
// macroblock.  A frame that codes a map (update_mb_segmentation_map) stores its ids; a key frame without one
// clears the map (the parser context restarts, host/frame_parser.cc); an inter frame with segmentation but no
// coded map takes its ids from the map and gets segment and loop-filter level patched into its records.
__global__ void __launch_bounds__(256) SegmentKernel(const DevFrameJob *__restrict__ jobs) {
  const DevFrameJob &job = jobs[blockIdx.y];
  if (!job.mode_hdr || JobFailed(job)) return;
  const vp8r_mode_hdr *mh = reinterpret_cast<const vp8r_mode_hdr *>(job.mode_hdr);
  const int n_mb = job.mb_cols * job.mb_rows;
  const int idx = blockIdx.x * 256 + threadIdx.x;
  if (idx >= n_mb) return;
  unsigned char *segmap = job.segment_map;
  vp8r_mb_info *mbs = const_cast<vp8r_mb_info *>(job.mbs);
  if (mh->update_segment_map) {
    segmap[idx] = (unsigned char)((mbs[idx].flags >> VP8R_MB_QSEG_SHIFT) & 3u);
  } else if (mh->key_frame) {
    segmap[idx] = 0;
  } else if (mh->segmentation_enabled) {
    const int seg = segmap[idx] & 3;
    unsigned flags = mbs[idx].flags;
    const int ref = (int)((flags >> VP8R_MB_REF_SHIFT) & 3u), mode = (int)((flags >> VP8R_MB_MODE_SHIFT) & 7u);
    const int lvl = MbFilterLevel(mh->frame_lf_level, true, mh->segment_abs != 0, mh->segment_lf[seg], mh->lf_adj_enable != 0,
                                  mh->ref_lf_delta[ref], ref,
                                  ref == 0 ? (mode == B_PRED ? mh->mode_lf_delta[0] : 0)
                                           : mh->mode_lf_delta[mode == MV_ZERO ? 1 : (mode == MV_SPLIT ? 3 : 2)]);
    flags &= ~((3u << VP8R_MB_QSEG_SHIFT) | (63u << VP8R_MB_LF_SHIFT));
    flags |= ((unsigned)seg << VP8R_MB_QSEG_SHIFT) | ((unsigned)lvl << VP8R_MB_LF_SHIFT);
    mbs[idx].flags = flags;
  }
}

// K_tokens.  Block = (most DCT partitions of any frame in the batch) warps.  Only one lane per warp works, but
// registers are allocated for all 32: the trimmed block keeps a batch's footprint small enough to share the SMs
// with the reconstruction kernels of the previous time step.  (A register cap was tried: spills in the serial
// chain cost more than the occupancy won.)
// kBlockWarps / kMinBlocks: launch bounds (measured in profiles/r2_summary.md).
template <int kBlockWarps, int kMinBlocks>
__global__ void __launch_bounds__(kBlockWarps * 32, kMinBlocks) TokenKernel(const DevFrameJob *__restrict__ jobs) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const DevFrameJob &job = jobs[blockIdx.x];
  if (!job.tok_hdr) return;
  TokenShared &sh = *reinterpret_cast<TokenShared *>(smem_raw);
  const vp8r_token_hdr *th = reinterpret_cast<const vp8r_token_hdr *>(job.tok_hdr);
  const int cols = job.mb_cols, rows = job.mb_rows;
  // above-context per macroblock column: bits 0-3 Y (column j), 4-5 U, 6-7 V, 8 Y2
  unsigned short *above = reinterpret_cast<unsigned short *>(smem_raw + ((sizeof(TokenShared) + 15) & ~size_t(15)));
  for (int i = threadIdx.x; i < (int)sizeof(sh.probs) / 4; i += blockDim.x)
    reinterpret_cast<unsigned *>(sh.probs)[i] = __ldg(reinterpret_cast<const unsigned *>(th->coef_probs) + i);
  for (int i = threadIdx.x; i < cols; i += blockDim.x) above[i] = 0;
  if (threadIdx.x < 8) sh.progress[threadIdx.x] = 0;
  for (int i = threadIdx.x; i < 8 * 16; i += blockDim.x) (&sh.blk[0][0])[i] = 0;
  __syncthreads();

  const int warp = (int)(threadIdx.x >> 5);  // = the partition of this thread
  if ((threadIdx.x & 31) != 0) return;
  const int n_parts = (int)__ldg(&th->n_parts);
  if (warp >= n_parts) return;

  const unsigned char *raw = reinterpret_cast<const unsigned char *>(th) + sizeof(vp8r_token_hdr);
  const unsigned raw_bytes = __ldg(&th->raw_bytes);
  const unsigned part_size = __ldg(&th->part_size[warp]);
  BoolDec bd;
  bd.Init(raw, __ldg(&th->part_off[warp]), raw + __ldg(&th->part_off[warp]) + part_size);
  bool used = false;

  vp8r_mb_info *mbs = const_cast<vp8r_mb_info *>(job.mbs);
  short *const blk = sh.blk[warp];
  volatile int *const prog = sh.progress;
  const int prev_warp = (warp + n_parts - 1) % n_parts;
  int16_t *const coef_area = const_cast<int16_t *>(job.payload) + (size_t)job.coef_base * 16;

  int k = 0;  // index of the row among this partition's rows
  for (int r = warp; r < rows; r += n_parts, ++k) {
    unsigned left = 0;  // bits 0-3 Y (row i), 4-5 U, 6-7 V, 8 Y2
    unsigned stored_row = 0;
    const unsigned row_base = (unsigned)r * (unsigned)cols * 25u;
    // what the previous row's partition must have reached before macroblock c of this row:
    // its progress counts macroblocks along its own rows; row r-1 is its row (warp ? k : k-1).
    const int prev_row_base = (warp ? k : k - 1) * cols;
    for (int c = 0; c < cols; ++c) {
      const size_t idx = (size_t)r * cols + c;
      const unsigned flags = mbs[idx].flags;
      if (r > 0 && n_parts > 1) {
        const int need = prev_row_base + c + 1;
        while (prog[prev_warp] < need) __nanosleep(100);
        __threadfence_block();
      }
      const bool has_y2 = (flags & VP8R_MB_HAS_Y2) != 0;
      unsigned abv = above[c];
      unsigned mask = 0;
      unsigned new_above, new_left;
      if (flags & VP8R_MB_SKIP_COEF) {
        // no tokens: contexts are cleared, except Y2's when the macroblock has no Y2 block
        new_above = has_y2 ? 0u : (abv & 0x100u);
        new_left = has_y2 ? 0u : (left & 0x100u);
      } else {
        used = true;
        const short *dq = job.dq[(flags >> VP8R_MB_QSEG_SHIFT) & 3];
        unsigned raw_nz = 0, dq_nz = 0;  // bit b as in coef_mask
        unsigned stored = 0;
        int16_t *out = coef_area + (size_t)(row_base + stored_row) * 16;
        const int ytype = has_y2 ? 0 : 3, yfirst = has_y2 ? 1 : 0;
        // Neighbour contexts as two bit sets indexed by block: ca / cl bit b = "the block above / to the
        // left of block b is non-zero".  Seeded with the neighbouring macroblocks' flags for the blocks on
        // the top row / left column of each plane; inside the macroblock a non-zero block sets the bits of
        // the blocks below and to the right of it (raw flags, src/bitstream_parser.cc:500-534).
        unsigned ca = ((abv >> 8) & 1u) | ((abv & 0xfu) << 1) | (((abv >> 4) & 3u) << 17) | (((abv >> 6) & 3u) << 21);
        unsigned cl = ((left >> 8) & 1u) | ((left & 1u) << 1) | (((left >> 1) & 1u) << 5) | (((left >> 2) & 1u) << 9) |
                      (((left >> 3) & 1u) << 13) | (((left >> 4) & 1u) << 17) | (((left >> 5) & 1u) << 19) |
                      (((left >> 6) & 1u) << 21) | (((left >> 7) & 1u) << 23);
        constexpr unsigned kInnerAboveY = 0x0001ffe0u, kInnerAboveC = (3u << 19) | (3u << 23);  // blocks whose upper neighbour is in this MB
        constexpr unsigned kInnerLeft = 0x0001dddcu | (1u << 18) | (1u << 20) | (1u << 22) | (1u << 24);  // ... left neighbour
        const unsigned char *const pb_y2 = sh.probs + ((1 * 8 + 0) * 3) * 11;
        const unsigned char *const pb_y = sh.probs + ((ytype * 8 + yfirst) * 3) * 11;  // band of coefficient `first` is `first`
        const unsigned char *const pb_uv = sh.probs + ((2 * 8 + 0) * 3) * 11;
        for (int b = has_y2 ? 0 : 1; b < 25; ++b) {
          const int ctx = (int)(((ca >> b) & 1u) + ((cl >> b) & 1u));
          const unsigned char *p = (b == 0 ? pb_y2 : (b <= 16 ? pb_y : pb_uv)) + ctx * 11;
          if (!bd.Bit(p[0])) continue;
          int type, first, dc_f, ac_f;
          if (b == 0) {
            type = 1; first = 0; dc_f = dq[VP8R_DQ_Y2_DC]; ac_f = dq[VP8R_DQ_Y2_AC];
          } else if (b <= 16) {
            type = ytype; first = yfirst; dc_f = dq[VP8R_DQ_Y1_DC]; ac_f = dq[VP8R_DQ_Y1_AC];
          } else {
            type = 2; first = 0; dc_f = dq[VP8R_DQ_UV_DC]; ac_f = dq[VP8R_DQ_UV_AC];
          }
          const int res = ReadTokens(bd, sh.probs, type, ctx, first, dc_f, ac_f, blk);
          if (res & 1) {
            raw_nz |= 1u << b;
            ca |= b <= 16 ? (16u << b) & kInnerAboveY : (4u << b) & kInnerAboveC;
            cl |= (2u << b) & kInnerLeft;
            uint4 lo = *reinterpret_cast<const uint4 *>(blk), hi = *reinterpret_cast<const uint4 *>(blk + 8);
            *reinterpret_cast<uint4 *>(out + stored * 16) = lo;
            *reinterpret_cast<uint4 *>(out + stored * 16 + 8) = hi;
            *reinterpret_cast<uint4 *>(blk) = make_uint4(0, 0, 0, 0);
            *reinterpret_cast<uint4 *>(blk + 8) = make_uint4(0, 0, 0, 0);
            ++stored;
          }
          if (res & 2) dq_nz |= 1u << b;
        }
        mask = raw_nz;
        // contexts handed to the neighbours: post-dequant flags
        new_above = ((dq_nz >> 13) & 0xfu) | (((dq_nz >> 19) & 3u) << 4) | (((dq_nz >> 23) & 3u) << 6);
        new_left = ((dq_nz >> 4) & 1u) | (((dq_nz >> 8) & 1u) << 1) | (((dq_nz >> 12) & 1u) << 2) | (((dq_nz >> 16) & 1u) << 3) |
                   (((dq_nz >> 18) & 1u) << 4) | (((dq_nz >> 20) & 1u) << 5) | (((dq_nz >> 22) & 1u) << 6) |
                   (((dq_nz >> 24) & 1u) << 7);
        if (has_y2) {
          new_above |= (dq_nz & 1u) << 8;
          new_left |= (dq_nz & 1u) << 8;
        } else {
          new_above |= abv & 0x100u;
          new_left |= left & 0x100u;
        }
        // complete the macroblock record
        if (mask) {
          mbs[idx].coef_mask = mask;
          mbs[idx].coef_offset = job.coef_base + row_base + stored_row;
          mbs[idx].flags = flags | VP8R_MB_LF_INNER;
        }
        stored_row += stored;
      }
      above[c] = (unsigned short)new_above;
      left = new_left;
      if (n_parts > 1) {
        __threadfence_block();
        prog[warp] = k * cols + c + 1;
      }
    }
  }
  if (used && bd.BytesConsumed() > (int)part_size && job.status) {
    atomicOr(job.status, 1);
    if (job.status_host) atomicOr(job.status_host, 1);
  }
}

cudaError_t InitParseTables() {
  ModeTables t = kModeTablesInit;
  static_assert(sizeof(t.kf_bmode) == sizeof(host_tables::kKfBmode), "kf_bmode size");
  for (size_t i = 0; i < sizeof(t.kf_bmode); ++i) t.kf_bmode[i] = host_tables::kKfBmode[i];
  (void)host_tables::kCoefDefault; (void)host_tables::kCoefUpdate; (void)host_tables::kMvDefault; (void)host_tables::kMvUpdate;
  return cudaMemcpyToSymbol(c_mode_tables, &t, sizeof(t));
}

namespace {
// cudaFuncAttributeMaxDynamicSharedMemorySize belongs to the (function, device) pair: one high-water mark each.
template <typename K>
cudaError_t EnsureSmem(K kernel, size_t smem, size_t *marks) {
  int dev = 0;
  cudaGetDevice(&dev);
  size_t &mark = marks[dev & 63];
  if (smem > 48 * 1024 && smem > mark) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    mark = smem;
  }
  return cudaSuccess;
}
}  // namespace

cudaError_t LaunchModes(const DevFrameJob *jobs, int n_frames, int max_cols, int max_mbs, cudaStream_t st) {
  const size_t smem = MakeModeLayout(max_cols, max_mbs).total;
  static size_t marks[64] = {};
  cudaError_t e = EnsureSmem(ModeKernel, smem, marks);
  if (e != cudaSuccess) return e;
  ModeKernel<<<n_frames, 32, smem, st>>>(jobs);
  return cudaGetLastError();
}

cudaError_t LaunchSegments(const DevFrameJob *jobs, int n_frames, int max_mbs, cudaStream_t st) {
  SegmentKernel<<<dim3((max_mbs + 255) / 256, n_frames), 256, 0, st>>>(jobs);
  return cudaGetLastError();
}

cudaError_t LaunchTokens(const DevFrameJob *jobs, int n_frames, int max_cols, int max_parts, cudaStream_t st) {
  max_parts = max_parts < 1 ? 1 : (max_parts > kTokenWarps ? kTokenWarps : max_parts);
  const size_t smem = TokenSmem(max_cols);
  // (min blocks 0 = "unspecified" makes ptxas settle on 48 registers with spills for this kernel; 1 gives 72, none)
  const bool narrow = max_parts <= 4;
  void (*kernel)(const DevFrameJob *) = narrow ? TokenKernel<4, 1> : TokenKernel<kTokenWarps, 1>;
  static size_t marks[2][64] = {};
  cudaError_t e = EnsureSmem(kernel, smem, marks[narrow]);
  if (e != cudaSuccess) return e;
  kernel<<<n_frames, max_parts * 32, smem, st>>>(jobs);
  return cudaGetLastError();
}

}  // namespace vp8r
