/*
 * vp8r.h -- C ABI of the B200-native VP8 frame-reconstruction engine (libvp8r.so).
 *
 * This is the drop-in boundary for the reference decoder's frame-reconstruction path.
 * The reference (TaWeiTu/vp8) has no FFI layer of its own; its de-facto boundary is the body
 * of the per-frame loop in src/decode.cc:50-77:
 *
 *     ReadFrameTagHeader()            src/bitstream_parser.cc:12-151   -> vp8r_parser_parse()
 *     InitSignBias() + DecodeFrame()  src/loop.h:13-17, src/decode_frame.cc:175-187
 *     RefreshRefFrames()              src/loop.h:19-46                 -> vp8r_reconstruct_batch()
 *     YUV<WRITE>::WriteFrame()        src/yuv.cc:6-28                  -> vp8r_stream_read_frame()
 *
 * In the reference, parsing and pixel reconstruction are interleaved per macroblock
 * (src/decode_frame.cc:98-170).  Here they are split: a pure host parser (bool decoder, headers,
 * per-macroblock syntax, motion-vector derivation, token decode) emits the arrays declared below,
 * and hand-written sm_100a CUDA kernels consume them (dequantisation + inverse WHT/DCT, 6-tap /
 * bilinear motion compensation, intra prediction, normal/simple loop filter).  Reference frames
 * (last / golden / altref) stay resident in HBM; there is no CPU fallback for the pixel path.
 *
 * Conventions: plain C types only, no exceptions or exit() across the boundary; every call
 * returns a vp8r_status and vp8r_last_error() gives a thread-local message (the reference
 * prints and exit(1)s in ensure(), src/utils.h:9-13, or throws std::out_of_range from
 * SpanReader, src/utils.h:62-66).
 */
#ifndef VP8R_H_
#define VP8R_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define VP8R_API
#else
#define VP8R_API __attribute__((visibility("default")))
#endif

typedef enum vp8r_status {
  VP8R_OK = 0,
  VP8R_ERR_INVALID_ARG = 1,
  VP8R_ERR_BITSTREAM = 2,   /* bad start code etc.  (reference: ensure(), bitstream_parser.cc:24-29) */
  VP8R_ERR_UNSUPPORTED = 3, /* version > 3, color_space / clamping_type != 0 (bitstream_parser.cc:47-48) */
  VP8R_ERR_TRUNCATED = 4,   /* a partition was read past its end (reference: std::out_of_range) */
  VP8R_ERR_STATE = 5,       /* inter frame before any key frame, stream/engine mismatch, ... */
  VP8R_ERR_CUDA = 6,
  VP8R_ERR_NOMEM = 7
} vp8r_status;

/* ---------------------------------------------------------------------------------------------
 * Parsed-frame description: what the host parser emits and the kernels consume.
 * All arithmetic inputs are integers; nothing here is floating point.
 * ------------------------------------------------------------------------------------------- */

/* Per-macroblock record, raster order, 32 bytes (two 128-bit loads on the device). */
typedef struct vp8r_mb_info {
  uint32_t flags;       /* VP8R_MB_* bit fields below */
  uint32_t coef_mask;   /* bit b: block b has >=1 non-zero coefficient stored.
                           b = 0: Y2, 1..16: Y raster, 17..20: U, 21..24: V
                           (block order of src/residual.cc:42-94) */
  uint32_t coef_offset; /* index, in units of one block (16 int16), of this MB's first stored
                           block in vp8r_frame_desc.coeffs; stored blocks follow in increasing b */
  int16_t mv[2];        /* {row, col} luma motion vector in 1/8-pel units (quarter-pel values
                           doubled, src/bitstream_parser.cc:360-361); non-SPLIT inter MBs */
  uint32_t aux[2];      /* intra B_PRED: 16 sub-block modes, 4 bits each, block i at bits 4i
                           (aux[0] holds blocks 0..7).  inter SPLIT: aux[0] = index (same units as
                           coef_offset) of two payload blocks holding this MB's 16 luma motion
                           vectors as int16 {row,col} pairs in raster order */
  uint32_t reserved[2];
} vp8r_mb_info;

#define VP8R_MB_IS_INTER      0x00000001u
#define VP8R_MB_REF_SHIFT     1  /* 2 bits: 1 last, 2 golden, 3 altref (0 for intra) */
#define VP8R_MB_MODE_SHIFT    3  /* 3 bits: intra 0 DC,1 V,2 H,3 TM,4 B_PRED ; inter 0 NEAREST,1 NEAR,2 ZERO,3 NEW,4 SPLIT */
#define VP8R_MB_UVMODE_SHIFT  6  /* 2 bits: 0 DC,1 V,2 H,3 TM (intra only) */
#define VP8R_MB_HAS_Y2        0x00000100u
#define VP8R_MB_QSEG_SHIFT    9  /* 2 bits: row of vp8r_frame_hdr.dq used by this MB */
#define VP8R_MB_LF_SHIFT      11 /* 6 bits: loop-filter level of this MB (0 = not filtered) */
#define VP8R_MB_LF_INNER      0x00020000u /* filter the inner (sub-block) edges too */
#define VP8R_MB_SKIP_COEF     0x00040000u /* mb_skip_coeff: the MB has no tokens in its DCT partition
                                             (only meaningful in frames with deferred tokens) */

/* Dequantisation factor columns of vp8r_frame_hdr.dq (src/quantizer.cc:15-53). */
enum { VP8R_DQ_Y1_DC = 0, VP8R_DQ_Y1_AC, VP8R_DQ_Y2_DC, VP8R_DQ_Y2_AC, VP8R_DQ_UV_DC, VP8R_DQ_UV_AC };

typedef struct vp8r_frame_hdr {
  uint16_t width, height;     /* display size of the stream (last key frame's tag) */
  uint16_t mb_cols, mb_rows;  /* ceil(width/16), ceil(height/16) */
  uint8_t key_frame;
  uint8_t version;            /* 0: six-tap; 1,2: bilinear; 3: bilinear + full-pixel chroma */
  uint8_t show_frame;
  uint8_t filter_type;        /* 0 normal loop filter, 1 simple (luma only) */
  uint8_t loop_filter_level;  /* frame level; 0 disables the loop filter for the frame */
  uint8_t sharpness_level;
  uint8_t refresh_last, refresh_golden, refresh_altref; /* key frames: all 1 */
  uint8_t copy_to_golden, copy_to_altref;               /* 0 none, 1 last, 2 other (loop.h:19-46) */
  uint8_t sign_bias_golden, sign_bias_altref;
  uint8_t q_index;            /* quantiser index of the frame (y_ac_qi, 0..127) */
  uint8_t modes_deferred;     /* 1: see modes_at below (implies tokens_deferred) */
  uint8_t tokens_deferred;    /* 1: see tokens_at below */
  int16_t dq[4][6];           /* dequant factors per segment (row 0 only when segmentation is off) */
  uint32_t n_coef_blocks;     /* coefficient blocks stored in payload[] */
  uint32_t n_payload_blocks;  /* all 32-byte payload blocks (coefficients + SPLIT motion vectors) */
  uint32_t n_inter_mbs;       /* informational */
  uint32_t n_split_mbs;       /* informational */
  /* Dependency levels of the intra macroblocks of an inter frame (0 when the frame has none or too
   * many levels, e.g. key frames, which are scheduled as a wavefront instead).  An intra MB of
   * level L only neighbours (left, above-left, above, above-right) intra MBs of lower levels, so
   * all MBs of one level can be predicted concurrently.  The table lives in the payload at block
   * `intra_levels_at`: n_intra_levels+1 uint32 offsets, then the MB indices sorted by level. */
  uint32_t n_intra_levels;
  uint32_t intra_levels_at;
  /* Deferred tokens (vp8r_parser_set_defer_tokens): the host parsed the first partition only.
   * coef_mask / coef_offset of every MB are 0, VP8R_MB_LF_INNER only covers B_PRED / SPLIT, and the
   * payload carries, at block `tokens_at`, a vp8r_token_hdr followed by the raw bytes of the
   * DCT partitions; the engine's token kernel (one thread per partition, rows pipelined through
   * the above-context as in src/bitstream_parser.cc:466-537) fills the rest on the device. */
  uint32_t tokens_at;
  /* Deferred modes (vp8r_parser_set_defer_modes): the host parsed the frame header only (tag, segment /
   * filter / quantiser headers, probability updates).  There are NO host vp8r_mb_info records
   * (vp8r_frame_desc.mbs is empty); the payload carries a vp8r_mode_hdr at block `modes_at`, the
   * vp8r_token_hdr at `tokens_at`, and the raw bytes of the first partition and the DCT partitions.
   * The engine's parse kernel reads the per-macroblock syntax (src/bitstream_parser.cc:320-464,
   * src/inter_predict.cc:8-244, src/intra_predict.cc:176-183) on the device, one thread per frame,
   * running ahead of the token threads, and builds the intra dependency levels there too. */
  uint32_t modes_at;
} vp8r_frame_hdr;

/* Per-frame parser state handed to the device-side macroblock-header decoder (160 bytes). */
typedef struct vp8r_mode_hdr {
  uint32_t first_off;   /* byte offset of the first partition inside the raw section (4-byte aligned) */
  uint32_t first_size;  /* bytes */
  uint32_t bitpos;      /* bit index, from the start of the first partition, of the first stream bit
                           behind the 8 bits held in `value` (bool decoder hand-over after the headers) */
  uint8_t value, range; /* bool decoder state: top 8 bits of the window, current range (128..255) */
  uint8_t key_frame, segmentation_enabled, update_segment_map, mb_no_skip_coeff;
  uint8_t prob_skip_false, prob_intra, prob_last, prob_gf;
  uint8_t sign_bias[4];            /* by reference frame id; [2] golden, [3] altref */
  uint8_t segment_tree_probs[3];
  uint8_t segment_abs;
  int8_t segment_lf[4];
  uint8_t lf_adj_enable, frame_lf_level;
  int8_t ref_lf_delta[4], mode_lf_delta[4];
  uint8_t ymode_probs[4], uvmode_probs[3];
  uint8_t pad0;
  uint8_t mv_probs[2][19];
  uint8_t pad1[160 - 12 - 10 - 4 - 4 - 4 - 2 - 8 - 8 - 38];
} vp8r_mode_hdr;

/* Header of the deferred-token section of the payload (32-byte aligned, 1152 bytes). */
typedef struct vp8r_token_hdr {
  uint32_t n_parts;        /* 1, 2, 4 or 8 DCT partitions; MB row r uses partition r % n_parts */
  uint32_t part_off[8];    /* byte offset of each partition inside the raw section */
  uint32_t part_size[8];   /* bytes */
  uint32_t raw_bytes;      /* size of the raw section (follows this header, zero padded by >= 16 B) */
  uint32_t reserved[6];
  uint8_t coef_probs[4][8][3][11]; /* token probabilities in force for this frame */
} vp8r_token_hdr;

typedef struct vp8r_frame_desc {
  vp8r_frame_hdr hdr;
  const vp8r_mb_info *mbs;    /* mb_rows*mb_cols records */
  const int16_t *payload;     /* n_payload_blocks*16 int16.  Coefficient blocks: raster order
                                 inside the block (already de-zigzagged), NOT dequantised.
                                 SPLIT MBs: their 16 motion vectors (2 blocks) precede their
                                 coefficient blocks. */
} vp8r_frame_desc;

/* ---------------------------------------------------------------------------------------------
 * Host parser (no GPU needed).  Replaces BitstreamParser + the syntax-driven halves of
 * IntraPredict / InterPredict (src/intra_predict.cc:176-178,398-399; src/inter_predict.cc:8-244).
 * One parser per stream: it carries the probability / segmentation state between frames
 * (ParserContext, src/bitstream_parser.h:124-182).
 * ------------------------------------------------------------------------------------------- */
typedef struct vp8r_parser vp8r_parser;
typedef struct vp8r_frame vp8r_frame; /* owns the arrays behind one vp8r_frame_desc */

VP8R_API vp8r_parser *vp8r_parser_create(void);
VP8R_API void vp8r_parser_destroy(vp8r_parser *p);
/* Discards all inter-frame state (as a fresh ParserContext does, src/decode.cc:43). */
VP8R_API void vp8r_parser_reset(vp8r_parser *p);

/* pinned != 0: arrays live in CUDA pinned host memory (needs a GPU); 0: plain heap. */
VP8R_API vp8r_frame *vp8r_frame_create(int pinned);
VP8R_API void vp8r_frame_destroy(vp8r_frame *f);
VP8R_API int vp8r_frame_get_desc(const vp8r_frame *f, vp8r_frame_desc *out);

/* on != 0: later vp8r_parser_parse calls read the first partition only (headers, modes, motion
 * vectors) and attach the DCT partitions for the engine's device-side token decoder; see
 * vp8r_frame_hdr.tokens_at.  Over-reads of a DCT partition are then reported by
 * vp8r_engine_sync() instead of the parse call. */
VP8R_API void vp8r_parser_set_defer_tokens(vp8r_parser *p, int on);

/* on != 0: later vp8r_parser_parse calls read the frame header only; the per-macroblock syntax of the
 * first partition and the DCT partitions are decoded by the engine's parse kernel (implies deferred
 * tokens; see vp8r_frame_hdr.modes_at).  The stream's segment map then lives on the device, so a
 * stream must not switch this mode between key frames.  Over-reads of the first partition are
 * reported by vp8r_engine_sync(). */
VP8R_API void vp8r_parser_set_defer_modes(vp8r_parser *p, int on);

/* Parses one compressed frame (the payload of one IVF frame record) into `out`. */
VP8R_API int vp8r_parser_parse(vp8r_parser *p, const uint8_t *data, size_t size, vp8r_frame *out);

/* Parses frame i with parsers[i] into out[i] for i < n, using up to n_threads host threads
 * (parsers must be distinct).  status (nullable) receives the per-frame result; the return value
 * is the first failure. */
VP8R_API int vp8r_parse_batch(int n, vp8r_parser *const *parsers, const uint8_t *const *data,
                              const size_t *sizes, vp8r_frame *const *out, int n_threads, int *status);

/* Peeks at the 3-byte frame tag: key-frame flag (bit 0 of byte 0 clear, bitstream_parser.cc:19-20).
 * Used to cut a stream at key frames (src/display.cc:64-67 does the same to seek). */
VP8R_API int vp8r_is_key_frame(const uint8_t *data, size_t size);

/* ---------------------------------------------------------------------------------------------
 * Engine: device surfaces + CUDA kernels.  One engine per GPU (per process); any number of
 * streams; frames of DIFFERENT streams are reconstructed together in one batched launch.
 * ------------------------------------------------------------------------------------------- */
typedef struct vp8r_engine vp8r_engine;
typedef struct vp8r_stream vp8r_stream;

/* cuda_stream: a cudaStream_t to launch on (e.g. torch's current stream), or NULL for a private
 * non-blocking stream owned by the engine. */
VP8R_API int vp8r_engine_create(int device, void *cuda_stream, vp8r_engine **out);
VP8R_API void vp8r_engine_destroy(vp8r_engine *e);
VP8R_API int vp8r_engine_sync(vp8r_engine *e);

/* Fences for pipelining host work against the asynchronous device work: a ticket marks everything
 * submitted to the engine so far; vp8r_engine_wait blocks the host until that work is done (so a
 * pinned vp8r_frame or output buffer can be reused).  At most 16 tickets are outstanding; waiting
 * on an older one waits for nothing (a later fence was recorded over it - callers keep <= 16). */
VP8R_API int vp8r_engine_fence(vp8r_engine *e, uint64_t *ticket);
VP8R_API int vp8r_engine_wait(vp8r_engine *e, uint64_t ticket);

VP8R_API int vp8r_stream_open(vp8r_engine *e, vp8r_stream **out);
VP8R_API void vp8r_stream_close(vp8r_stream *s);

/* Copies a parsed frame's arrays to HBM once, so later vp8r_reconstruct_batch() calls on it
 * start with inputs resident on the device (kernel-only measurements, replays). */
VP8R_API int vp8r_frame_upload(vp8r_engine *e, vp8r_frame *f);

/* Frees the host arrays of an uploaded frame (the header stays readable; vp8r_frame_get_desc then
 * fails).  For replays of many resident frames: a 1080p frame holds ~0.9 MB of host memory. */
VP8R_API int vp8r_frame_release_host(vp8r_frame *f);

/* DecodeFrame + RefreshRefFrames for n frames of n distinct streams, asynchronously on the
 * engine's CUDA stream.  frames[i] not uploaded are staged host->device inside the call. */
VP8R_API int vp8r_reconstruct_batch(vp8r_engine *e, int n, vp8r_stream *const *streams,
                                    vp8r_frame *const *frames);

/* Size in bytes of the cropped I420 image of the stream's most recent frame
 * (w*h + 2*ceil(w/2)*ceil(h/2), src/yuv.cc:6-28); 0 before the first frame. */
VP8R_API size_t vp8r_stream_frame_bytes(const vp8r_stream *s);
VP8R_API int vp8r_stream_dims(const vp8r_stream *s, int *width, int *height);

/* YUV<WRITE>::WriteFrame: crop + pack the most recently reconstructed frame of each stream into
 * caller memory (Y, U, V planes back to back).  `dst[i]` may be pinned or pageable host memory.
 * Asynchronous on the engine's stream when `async` != 0 (dst must then be pinned and stay valid
 * until vp8r_engine_sync()). */
VP8R_API int vp8r_read_batch(vp8r_engine *e, int n, vp8r_stream *const *streams,
                             uint8_t *const *dst, const size_t *cap, int async);
VP8R_API int vp8r_stream_read_frame(vp8r_stream *s, uint8_t *dst, size_t cap);
/* Same output, but cropped and packed ON THE DEVICE (one kernel for all n frames) and moved with
 * ONE contiguous copy: frame i lands at dst + i*stride (stride >= frame bytes).  For many streams
 * this replaces 3*n pitched copies per time step. */
VP8R_API int vp8r_read_batch_packed(vp8r_engine *e, int n, vp8r_stream *const *streams, uint8_t *dst,
                                    size_t stride, int async);
/* Output layouts of the packed read-back.  I420 is what YUV<WRITE>::WriteFrame writes (src/yuv.cc:6-28); NV12
 * (Y plane, then one plane of interleaved U,V pairs: the layout display engines and hardware encoders take) has
 * the same number of bytes. */
#define VP8R_LAYOUT_I420 0
#define VP8R_LAYOUT_NV12 1
/* vp8r_read_batch_packed with the layout chosen by the caller. */
VP8R_API int vp8r_read_batch_packed_as(vp8r_engine *e, int n, vp8r_stream *const *streams, uint8_t *dst,
                                       size_t stride, int async, int layout);

/* Layouts only the device read-back below writes: BT.601 limited-range RGB of the cropped frame (the matrix of a VP8
 * stream, color_space 0), 3*w*h bytes, chroma point-sampled (the sample at (x>>1, y>>1) serves its 2x2 pixels).  Per
 * pixel, c = Y-16, d = U-128, e = V-128, with an arithmetic shift and a clamp to 0..255:
 *   R = (298c + 409e + 128) >> 8,  G = (298c - 100d - 208e + 128) >> 8,  B = (298c + 516d + 128) >> 8 */
#define VP8R_LAYOUT_RGB24      2  /* per pixel R,G,B bytes, rows of 3*w bytes (HWC) */
#define VP8R_LAYOUT_RGB_PLANAR 3  /* R plane, G plane, B plane, each w*h bytes (CHW) */
/* Writes the most recent frame of streams[i] to dst + i*stride in DEVICE memory of the engine's device, for consumers
 * on the GPU (nothing crosses PCIe).  layout: VP8R_LAYOUT_I420 / _NV12 (vp8r_stream_frame_bytes(s) bytes, as the packed
 * read-back writes them) or VP8R_LAYOUT_RGB24 / _RGB_PLANAR (3*w*h bytes).  Asynchronous on the engine's stream, behind
 * its reconstruction kernels.
 *
 * consumer_stream: the cudaStream_t the caller reads dst on (e.g. torch's current stream).  NULL or the engine's own
 * stream: nothing extra.  Otherwise, without blocking the host:
 *   1. before the conversion the engine's stream waits for the work submitted to consumer_stream so far, so that dst
 *      is not overwritten while earlier consumer work may still read it.  This wait also holds back every later
 *      kernel on the engine's stream (the next time steps' reconstruction) until that consumer work has finished;
 *   2. after the conversion consumer_stream waits for it, so work submitted there afterwards sees the frames.
 * VP8R_ERR_INVALID_ARG: null engine / streams / dst, n <= 0, an unknown layout, stride smaller than a frame, dst not
 * device memory of the engine's device (pinned, pageable and managed memory are refused); VP8R_ERR_STATE: a stream of
 * another engine or without a frame. */
VP8R_API int vp8r_read_batch_device(vp8r_engine *e, int n, vp8r_stream *const *streams, void *dst, size_t stride,
                                    int layout, void *consumer_stream);

/* ---- encoder (SURVEY.md section 8 row f4; the reference only sketches one: src/encode_frame.cc:30-244,
 * src/residual.cc:5-40,96-108, src/dct.cc:5-65, src/quantizer.cc:5-8; its encode.cc does not compile) ----
 *
 * vp8r_encode_key_frames: one KEY frame for each of n different streams, all of size width x height, from cropped
 * I420 images in host memory (i420[k]: Y, U, V planes back to back, as vp8r_stream_read_frame delivers them).  On the
 * device, per macroblock and in a closed loop: 16x16 luma and chroma intra mode by squared error (candidates V, H,
 * DC, TM in that order, a later one only when strictly better: PickIntraModeLuma / PickIntraModeChroma), residual,
 * forward DCT / WHT, quantisation by the factors of q_index, and the decoder's reconstruction + loop filter, so that
 * stream k afterwards holds exactly the frame a decoder makes of the result (vp8r_stream_read_frame returns it, and
 * inter frames decoded next predict from it).  out[k] receives the macroblock records and coefficient blocks (the
 * same structure the parser produces); vp8r_frame_write_bitstream turns it into a VP8 frame.  Synchronous. */
#define VP8R_ENC_BPRED 1u /* flags: B_PRED is a candidate for every macroblock: its sixteen sub-block modes are picked
                            one after the other on the reconstructed neighbours (ten predictors by squared error, in
                            enum order, a later one only when strictly better: PickIntraSubBlockModeSB), and the
                            macroblock is coded B_PRED when the sum of their errors is strictly below the best 16x16
                            mode's (PickIntraModeLuma, src/encode_frame.cc:204-238) */
VP8R_API int vp8r_encode_key_frames(vp8r_engine *e, int n, vp8r_stream *const *streams, const uint8_t *const *i420,
                                    int width, int height, int q_index, int loop_filter_level, int sharpness,
                                    unsigned flags, vp8r_frame *const *out);
/* vp8r_encode_inter_frames: one INTER frame for each of n different streams, from cropped I420 images in host memory
 * (the same conventions as vp8r_encode_key_frames).  Every macroblock predicts from the stream's current LAST frame
 * (made by vp8r_encode_key_frames, by an earlier inter encode or by decoding) with one motion vector; there are no
 * intra or SPLIT macroblocks.  On the device, one warp per macroblock: full-pel search over +-search_range whole pixels
 * around the zero vector, then half-pel and quarter-pel refinement, by cost = luma SAD + lambda(q) * bits(vector)
 * (the lowest candidate index wins a tie), residual, forward DCT / WHT and quantisation; the decoder's own inter
 * reconstruction, loop filter and border extension then run on the records, so that stream k afterwards holds exactly
 * the frame a decoder makes of the written bitstream.  The host then gives every vector the cheapest mode consistent
 * with it (NEAREST / NEAR / ZERO / NEW).  out[k]: complete records (mode bits included, coef_offset = 25*mb) and
 * coefficient blocks, n_coef_blocks and n_inter_mbs set; header: show_frame 1, refresh_last 1, golden and altref
 * neither refreshed nor copied, sign biases 0, version 0.  References move as for a decoded inter frame.  Synchronous.
 * VP8R_ERR_INVALID_ARG: the key-frame call's argument checks, or search_range outside 4..24; VP8R_ERR_STATE: a stream
 * without a frame, whose frame is not width x height, or that has failed. */
VP8R_API int vp8r_encode_inter_frames(vp8r_engine *e, int n, vp8r_stream *const *streams, const uint8_t *const *i420,
                                      int width, int height, int q_index, int loop_filter_level, int sharpness,
                                      int search_range, vp8r_frame *const *out);
/* ---- encoder input from device memory ----
 * Frames already on the GPU (decoded frames, a model's output, rendered images) encode without crossing PCIe.  The
 * source layouts are the VP8R_LAYOUT_* constants read as input formats: VP8R_LAYOUT_I420 (cropped Y, U, V planes back to
 * back: the bytes of the host path and of vp8r_read_batch_device), VP8R_LAYOUT_NV12 (Y plane, then interleaved U,V
 * pairs), VP8R_LAYOUT_RGB24 (HWC) and VP8R_LAYOUT_RGB_PLANAR (CHW), 3*w*h bytes.  RGB becomes I420 by BT.601 limited
 * range in integers, with arithmetic shifts and no clamp (Y lands in 16..235, U and V in 16..240):
 *   Y = ((66R + 129G + 25B + 128) >> 8) + 16                 per pixel
 *   U = ((-38R' - 74G' + 112B' + 128) >> 8) + 128            per chroma sample
 *   V = ((112R' - 94G' - 18B' + 128) >> 8) + 128
 * where R', G', B' are the channel means (s + 2) >> 2 over the pixels (2i+a, 2j+b), a, b in {0, 1}, of chroma sample
 * (i, j), pixel coordinates clamped to w-1 / h-1 (odd sizes replicate the edge pixels).  Each component is within 1 of
 * the rounded floating-point BT.601 matrix.  Whatever the layout, the encoder codes exactly what the host path codes for
 * the cropped I420 image of the frame (vp8r_convert_to_i420_device returns it).
 *
 * vp8r_encode_key_frames_device / vp8r_encode_inter_frames_device: vp8r_encode_key_frames / vp8r_encode_inter_frames
 * (same checks, outputs, reference updates; synchronous) with frame i of the batch at src + i*stride in device memory
 * of the engine's device, any byte alignment, stride at least one frame of the layout.  producer_stream: the
 * cudaStream_t src was written on.  NULL or the engine's own stream: nothing extra; otherwise the engine's stream waits,
 * before it reads src, for the work submitted to producer_stream so far (without blocking the host).  src may be reused
 * once the call returns.  VP8R_ERR_INVALID_ARG: null engine / streams / src / out, n <= 0, an unknown layout, a stride
 * smaller than a frame, src not device memory of the engine's device (pinned, pageable and managed memory are refused),
 * and the host calls' argument checks; the checks that need no device come first. */
VP8R_API int vp8r_encode_key_frames_device(vp8r_engine *e, int n, vp8r_stream *const *streams, const void *src, size_t stride,
                                           int layout, void *producer_stream, int width, int height, int q_index,
                                           int loop_filter_level, int sharpness, unsigned flags, vp8r_frame *const *out);
VP8R_API int vp8r_encode_inter_frames_device(vp8r_engine *e, int n, vp8r_stream *const *streams, const void *src, size_t stride,
                                             int layout, void *producer_stream, int width, int height, int q_index,
                                             int loop_filter_level, int sharpness, int search_range, vp8r_frame *const *out);
/* The cropped I420 image (w*h + 2*ceil(w/2)*ceil(h/2) bytes) the encoder codes for each of n frames at src + i*src_stride
 * in `layout`, written to dst + i*dst_stride; src and dst device memory of the engine's device.  For PSNR against the
 * reconstruction of an RGB / NV12 source.  Asynchronous on the engine's stream, ordered against `stream` (the caller's
 * cudaStream_t, e.g. torch's current stream; NULL or the engine's own: nothing extra) as vp8r_read_batch_device orders
 * against its consumer stream: the conversion waits for the work submitted to `stream` so far, and work submitted there
 * afterwards sees dst.  VP8R_ERR_INVALID_ARG as for the encoder calls, and dst_stride smaller than an I420 frame. */
VP8R_API int vp8r_convert_to_i420_device(vp8r_engine *e, int n, const void *src, size_t src_stride, int layout, int width,
                                         int height, void *dst, size_t dst_stride, void *stream);
/* The inverse of vp8r_parser_parse: serialises f into a VP8 frame with one DCT partition and the default token, mode and
 * motion-vector probabilities (see vp8r_frame_write_bitstream_in for inter frames of a stream that was decoded).  Key frames: intra macroblocks.  Inter frames: the frame header's refresh, copy,
 * sign-bias and show_frame fields from f's header, intra macroblocks, and inter macroblocks of any reference coded
 * NEAREST / NEAR / ZERO / NEW.  Both: no segmentation, no loop-filter deltas, the five quantiser deltas that reproduce
 * hdr.dq[0] from q_index.  SPLIT macroblocks and a vector that contradicts its mode are refused.  *size receives the
 * number of bytes needed; VP8R_ERR_INVALID_ARG when cap is too small (call again) or the frame cannot be written. */
VP8R_API int vp8r_frame_write_bitstream(const vp8r_frame *f, uint8_t *dst, size_t cap, size_t *size);
/* The same, with the token, motion-vector and 16x16 / chroma mode probabilities of `context`: the parser that parsed
 * the stream so far, whose state a decoder holds when it reaches this frame.  Write with it when the stream's LAST
 * frame came from decoding: the probability updates a stream carries persist until its next key frame, and a frame
 * coded with the defaults does not decode in such a stream.  context == NULL gives vp8r_frame_write_bitstream's bytes;
 * a key frame ignores context (it resets the decoder's probabilities).  The written frame carries no updates and sets
 * refresh_entropy_probs, so the context is the same after it: consecutive frames can all be written against the same
 * parser without feeding them through it.  VP8R_ERR_STATE: for an inter frame, a context that has not parsed a key
 * frame or whose frame size is not f's. */
VP8R_API int vp8r_frame_write_bitstream_in(const vp8r_frame *f, const vp8r_parser *context, uint8_t *dst, size_t cap,
                                           size_t *size);

/* Device-side checksum of the cropped I420 image: low word sum(b_i), high word
 * sum((i+1)*b_i), both mod 2^32, i = byte index in the Y,U,V stream.  For parity checks at sizes
 * where copying every frame back would dominate. */
VP8R_API int vp8r_stream_checksum(vp8r_stream *s, uint64_t *out);
VP8R_API int vp8r_checksum_batch(vp8r_engine *e, int n, vp8r_stream *const *streams, uint64_t *out);
/* Same checksum computed on host memory holding a cropped I420 image. */
VP8R_API uint64_t vp8r_checksum_i420(const uint8_t *i420, int width, int height);

/* One-call convenience = one iteration of the loop in src/decode.cc:50-77:
 * parse `data`, reconstruct, update references.  *shown receives show_frame. */
VP8R_API int vp8r_stream_decode(vp8r_stream *s, const uint8_t *data, size_t size, int *shown);

/* Accumulated device time per kernel class since the last reset (CUDA events on the engine's
 * stream; enabled with vp8r_engine_set_timing). */
typedef struct vp8r_timers {
  double ms_inter;    /* dequant+IWHT+IDCT + motion compensation of inter MBs */
  double ms_intra;    /* dequant+IWHT+IDCT + intra prediction wavefront */
  double ms_filter;   /* loop-filter wavefront */
  double ms_h2d, ms_d2h;
  double ms_tokens;   /* device-side token decode (frames with deferred tokens) */
  uint64_t launches_inter, launches_intra, launches_filter, launches_other;
  uint64_t frames, coef_blocks;
  uint64_t alg_bytes; /* sum over frames of 1.5*Wa*Ha*(1+is_inter) + 32*n_coef_blocks */
  double ms_border;   /* border extension of the finished frames (a kernel of its own behind the loop filter) */
} vp8r_timers;
VP8R_API int vp8r_engine_set_timing(vp8r_engine *e, int enabled);
VP8R_API int vp8r_engine_get_timers(vp8r_engine *e, vp8r_timers *out, int reset);

VP8R_API const char *vp8r_last_error(void);
VP8R_API const char *vp8r_version(void);
/* 1 when the library was built with the CUDA kernels linked in (always, for the product). */
VP8R_API int vp8r_has_cuda(void);

#ifdef __cplusplus
}
#endif
#endif /* VP8R_H_ */
