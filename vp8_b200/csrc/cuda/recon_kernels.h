// Device-side job description and launch entry points of the reconstruction kernels.
#ifndef VP8R_CUDA_RECON_KERNELS_H_
#define VP8R_CUDA_RECON_KERNELS_H_

#include <cuda_runtime.h>
#include <stdint.h>

#include "vp8r.h"

namespace vp8r {

// Replicated border (pixels) around every plane of a surface.  Motion-compensation windows are
// clamped as a whole into the padded plane, which is bit-identical to the reference's per-pixel
// coordinate clamp (src/inter_predict.cc:252-256) once the border is >= the window size.
constexpr int kBorder = 32;

struct DevPlanes {
  uint8_t *y, *u, *v;  // address of pixel (0,0) of each plane
};

// TMA descriptor (CUtensorMap: 128 bytes, 64-byte aligned) kept opaque here so that this header needs no
// driver API.  A surface has three, for its padded Y, U, V planes (element = one byte, x fastest; boxes of
// kTmaLumaBox / kTmaChromaBox): the reference windows of motion compensation come in as bulk tensor loads.
struct alignas(128) DevTensorMap {
  unsigned char opaque[128];
};
// The first (fastest) coordinate of a bulk tensor load must be a multiple of 16 BYTES (measured on B200: any
// other value traps as "illegal instruction", tools/microbench/tma_probe2.cu), so a box starts at the window's
// x rounded down to 16 and is 48 bytes wide: 15 + 21 <= 48, and 48-byte rows keep the lanes' word reads on
// distinct shared-memory banks.
constexpr int kTmaLumaBoxW = 48, kTmaLumaBoxH = 21;     // 21x21 window of a 16x16 block
constexpr int kTmaChromaBoxW = 48, kTmaChromaBoxH = 13;  // 13x13 window of an 8x8 block

// Per-frame results of the device-side macroblock-header pass (frames with deferred modes): what the
// host parser would have put into vp8r_frame_hdr.
struct DevFrameDyn {
  int n_inter, n_intra, n_intra_levels, n_split;
};

// One frame of one stream inside a batched launch.
struct DevFrameJob {
  const vp8r_mb_info *mbs;
  const int16_t *payload;
  DevPlanes cur;
  DevPlanes ref[4];  // indexed by reference frame id 1..3 (last, golden, altref)
  const DevTensorMap *ref_tmap[4];  // per reference frame: descriptors of its Y, U, V planes
  int pitch_y, pitch_c;
  int mb_cols, mb_rows;
  int n_intra, n_inter;
  int n_intra_levels;               // > 0: intra MBs are scheduled by dependency level (flat kernel)
  const uint32_t *intra_levels;     // n_intra_levels+1 offsets, then MB indices sorted by level
  int16_t dq[4][6];
  uint8_t key_frame, version, filter_type, lf_level, sharpness;
  uint8_t pack_layout;           // PackKernel: VP8R_LAYOUT_I420 / _NV12; ConvertRgbKernel: VP8R_LAYOUT_RGB24 / _RGB_PLANAR;
                                 // StageSourceKernel: the layout of stage_src (any of the four)
  uint8_t enc_flags;             // K_encode: VP8R_ENC_*
  // output side (crop / checksum)
  int width, height;
  unsigned long long *checksum;  // optional: receives the I420 checksum
  uint8_t *pack_dst;             // optional: receives the cropped image in pack_layout (device memory)
  // deferred tokens (K_tokens): vp8r_token_hdr + raw DCT partitions inside the frame's payload,
  // and the frame's device coefficient area (first block index relative to `payload`)
  const uint8_t *tok_hdr;
  uint32_t coef_base;
  int *status;                   // error word of this job in DEVICE memory (bit 0: a DCT partition was over-read,
                                 // bit 1: the first partition was): read by every reconstruction kernel
  int *status_host;              // the same word in mapped pinned host memory, for the host (written on failure only)
  // deferred modes: vp8r_mode_hdr inside the payload; `mbs` then points at a device area the parse
  // kernel fills, as are the SPLIT motion vectors (first block index relative to `payload`), the
  // intra level table and `dyn`; the segment map persists per stream
  const uint8_t *mode_hdr;
  uint32_t split_base;
  // staging by LaunchGather: h2d_bytes of the frame's blob at pinned host address h2d_src -> h2d_dst
  uint32_t h2d_bytes;
  const uint8_t *h2d_src;
  uint8_t *h2d_dst;
  uint8_t *segment_map;
  uint32_t *level_table;
  DevFrameDyn *dyn;
  // encoder (K_encode, enc_kernels.cu): macroblock-aligned source planes in device memory; `mbs` and `payload` are
  // then OUTPUTS (25 coefficient blocks reserved per macroblock)
  const uint8_t *enc_src[3];
  int enc_src_pitch_y, enc_src_pitch_c;
  int enc_search_range;          // K_encode_inter: full-pel search range (whole pixels, 4..24)
  // StageSourceKernel: a width x height frame in pack_layout at stage_src (device memory, any alignment) becomes the
  // I420 planes enc_src[0..2] over stage_w x stage_h luma pixels (source coordinates clamped to the frame)
  const uint8_t *stage_src;
  int stage_w, stage_h;
};

// A frame whose device-side parse ran past the end of a partition: its records are not trustworthy, so no
// kernel reconstructs it (the host stops the stream when it collects the word, rt/engine.cu HarvestStatus).
__device__ __forceinline__ bool JobFailed(const DevFrameJob &j) { return j.status && *reinterpret_cast<const volatile int *>(j.status) != 0; }

// Frame fields that come from the host for host-parsed frames and from the device otherwise.
__device__ __forceinline__ int JobInter(const DevFrameJob &j) { return j.dyn ? j.dyn->n_inter : j.n_inter; }
__device__ __forceinline__ int JobIntra(const DevFrameJob &j) { return j.dyn ? j.dyn->n_intra : j.n_intra; }
__device__ __forceinline__ int JobIntraLevels(const DevFrameJob &j) { return j.dyn ? j.dyn->n_intra_levels : j.n_intra_levels; }
__device__ __forceinline__ const uint32_t *JobLevelTable(const DevFrameJob &j) { return j.dyn ? j.level_table : j.intra_levels; }

// Uploads the constant tables (filter taps, B_PRED gather LUT).  Once per device.
cudaError_t InitKernelTables();

// Device-side parse (token_kernel.cu).  K_modes: macroblock headers of every job with mode_hdr != nullptr, one
// single-lane warp per frame; independent of every other frame, so the launches of consecutive batches may run
// concurrently.  K_segments: persistent segment maps + the segment-dependent record fields of those jobs; has to
// run in batch order, after K_modes and before K_tokens of its batch.  K_tokens: DCT token partitions of every
// job with tok_hdr != nullptr.
cudaError_t LaunchModes(const DevFrameJob *jobs, int n_frames, int max_cols, int max_mbs, cudaStream_t st);
cudaError_t LaunchSegments(const DevFrameJob *jobs, int n_frames, int max_mbs, cudaStream_t st);
cudaError_t LaunchTokens(const DevFrameJob *jobs, int n_frames, int max_cols, int max_parts, cudaStream_t st);
cudaError_t InitParseTables();
cudaError_t InitEncodeTables(const unsigned short *bpred_lut);  // enc_kernels.cu: its copy of the B_PRED gather table
// Level-scheduled intra prediction of frames whose level table was built on the device: one CTA per
// frame walks the dependency levels with a block barrier in between.
cudaError_t LaunchIntraLevels(const DevFrameJob *jobs, int n_frames, cudaStream_t st);
// Blocks (32 B) of device coefficient area a frame with deferred tokens needs.
inline size_t TokenCoefBlocks(int mb_cols, int mb_rows) { return size_t(mb_cols) * mb_rows * 25; }
// K_inter: dequant + IWHT/IDCT + motion compensation + residual add for every inter MB.  Reference windows of
// macroblocks with one motion vector are staged in shared memory by bulk tensor loads through the job's ref_tmap.
cudaError_t LaunchInter(const DevFrameJob *jobs, int n_frames, int max_cols, int max_rows, cudaStream_t st);
// K_intra: dequant + IWHT/IDCT + intra prediction as a per-frame macroblock wavefront.
cudaError_t LaunchIntra(const DevFrameJob *jobs, int n_frames, int max_rows, cudaStream_t st);
// Flat intra: every intra MB of dependency level `level` (frames with n_intra_levels > 0).
cudaError_t LaunchIntraFlat(const DevFrameJob *jobs, int n_frames, int level, int max_count, cudaStream_t st);
// K_encode: closed-loop key-frame encoder (mode decision, forward transform, quantisation, reconstruction) of every
// job with enc_src set; the loop filter follows as for a decoded frame.
cudaError_t LaunchEncodeIntra(const DevFrameJob *jobs, int n_frames, int max_rows, cudaStream_t st);
// K_encode_inter: motion search against LAST (ref[1]), residual, forward transform and quantisation of every
// macroblock of every job with enc_src set, one warp per macroblock; writes records (vector, coef_mask, flags
// without mode bits) and coefficient blocks.  K_inter, the loop filter and the border follow as for a decoded frame.
cudaError_t LaunchEncodeInter(const DevFrameJob *jobs, int n_frames, int max_cols, int max_rows, cudaStream_t st);
// Up to eight frames with the same geometry and filter type (and a non-zero frame filter level) that one
// warp of the batch loop filter walks together; unused slots are -1, slot 0 is always used.
struct FilterGroup {
  int frame[8];
};
// K_filter: normal/simple loop filter as a per-frame macroblock wavefront, then border extension.
// `sync`: device scratch of `sync_ints` ints (ticket + one progress word per (frame, band)).
// With `groups` (device pointer, n_groups > 0) the batch form runs (filter_swar.cu: four pixel lines per
// register, eight frames per warp); without, the scalar form (one warp per macroblock row of one frame),
// which has the shorter latency per frame.
cudaError_t LaunchFilter(const DevFrameJob *jobs, int n_frames, int max_rows, int *sync, int sync_ints,
                         cudaStream_t st, const FilterGroup *groups = nullptr, int n_groups = 0);
// Rewrites the 32-pixel border of every job's current frame (after the loop filter; next frame's motion
// compensation reads through it).
cudaError_t LaunchBorder(const DevFrameJob *jobs, int n_frames, cudaStream_t st);
cudaError_t LaunchFilterSwar(const DevFrameJob *jobs, const FilterGroup *groups, int n_groups, int max_rows, int *sync,
                             int sync_ints, cudaStream_t st);
// Ints of `sync` scratch LaunchFilter needs for a batch.
inline int FilterSyncInts(int n_frames) { return 1 + n_frames * 128; }
// Host->device staging without the copy engines (which the packed read-back keeps busy): `src` is
// pinned host memory read by the SMs over PCIe.  LaunchCopy moves one buffer (bytes % 16 == 0, both
// 16-byte aligned); LaunchGather moves every job's blob (h2d_src -> h2d_dst, h2d_bytes).
cudaError_t LaunchCopy(void *dst, const void *src_pinned, size_t bytes, cudaStream_t st);
cudaError_t LaunchGather(const DevFrameJob *jobs, int n_frames, size_t max_bytes, cudaStream_t st);
// Device-side crop + I420 pack of each job's current surface into job.pack_dst.
cudaError_t LaunchPack(const DevFrameJob *jobs, int n_frames, cudaStream_t st);
// Device-side crop + BT.601 YUV -> RGB (VP8R_LAYOUT_RGB24 / _RGB_PLANAR, from job.pack_layout) of each job's current
// surface into job.pack_dst.  max_w, max_h: the largest frame of the batch (sizes the grid).
cudaError_t LaunchConvertRgb(const DevFrameJob *jobs, int n_frames, int max_w, int max_h, cudaStream_t st);
// Device-side layout / BT.601 conversion + edge padding of each job's stage_src into its enc_src planes
// (StageSourceKernel).  layout: the pack_layout of every job; max_w, max_h: the largest stage_w x stage_h of the batch
// (sizes the grid).
cudaError_t LaunchStageSource(const DevFrameJob *jobs, int n_frames, int layout, int max_w, int max_h, cudaStream_t st);
// Device-side checksum of the cropped I420 image of each job's current surface.
cudaError_t LaunchChecksum(const DevFrameJob *jobs, int n_frames, cudaStream_t st);

}  // namespace vp8r

#endif  // VP8R_CUDA_RECON_KERNELS_H_
