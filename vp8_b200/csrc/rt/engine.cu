// Runtime around the kernels: engine (device, CUDA stream, staging), stream contexts (surface
// pool + last/golden/altref bookkeeping, the role of ref_frames[] in src/decode.cc:40 and
// RefreshRefFrames in src/loop.h:19-46), batched submission, read-back, timers, C ABI.
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstdint>
#include <cstring>
#include <initializer_list>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "../cuda/recon_kernels.h"
#include "../host/frame_parser.h"
#include "../host/frame_writer.h"
#include "../host/parsed_frame.h"
#include "error.h"
#include "vp8r.h"

namespace vp8r {

// ------------------------------------------------------------------ host / device memory ----
void *HostAlloc(size_t bytes, bool pinned) {
  if (!pinned) return std::malloc(bytes);
  void *p = nullptr;
  if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return p;
}
void HostFree(void *p, bool pinned) {
  if (!p) return;
  if (pinned) cudaFreeHost(p);
  else std::free(p);
}
void DeviceFree(void *p, int device) {
  if (!p) return;
  int prev = -1;
  cudaGetDevice(&prev);
  if (device >= 0 && device != prev) cudaSetDevice(device);
  cudaFree(p);
  if (device >= 0 && device != prev && prev >= 0) cudaSetDevice(prev);
}

#define CU_TRY(expr)                                                                         \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess) {                                                                 \
      SetError(std::string(#expr) + ": " + cudaGetErrorString(_e));                          \
      return VP8R_ERR_CUDA;                                                                  \
    }                                                                                        \
  } while (0)

struct Surface {
  uint8_t *base = nullptr;
  DevPlanes planes{};
};

}  // namespace vp8r

using vp8r::DevFrameJob;
using vp8r::SetError;

struct vp8r_stream {
  vp8r_engine *eng = nullptr;
  vp8r::FrameParser parser;
  vp8r_frame *own_frame = nullptr;  // scratch for vp8r_stream_decode
  int mb_cols = 0, mb_rows = 0, width = 0, height = 0;
  int pitch_y = 0, pitch_c = 0;
  vp8r::Surface surf[5];
  uint8_t *d_segmap = nullptr;  // persistent segment map (frames with deferred modes), one byte per MB
  vp8r::DevTensorMap *d_tmaps = nullptr;  // 5 surfaces x (Y, U, V) TMA descriptors of the padded planes
  int ref[4] = {-1, -1, -1, -1};  // surface index of CURRENT(latest), LAST, GOLDEN, ALTREF
  bool have_frame = false;
  bool failed = false;  // a device-parsed frame of this stream was truncated: nothing decodes until the next key frame
};

namespace {
// What a timer measures: the vp8r_timers field its time goes to (kNone: not timed).
enum class Timer { kInter, kIntra, kFilter, kH2D, kD2H, kTokens, kBorder, kNone };
struct EventPair {
  cudaEvent_t a, b;
  Timer cls;
};
struct Slot {
  DevFrameJob *h_jobs = nullptr, *d_jobs = nullptr;
  int cap_jobs = 0;
  uint8_t *d_arena = nullptr;
  size_t arena_cap = 0;
  cudaEvent_t done = nullptr;
  cudaEvent_t parsed = nullptr;  // staging + parse kernels of this slot's batch finished (on the slot's parse stream)
  cudaEvent_t modes_done = nullptr, segments_done = nullptr;  // K_modes of the batch (parse stream), K_segments (st_segments)
  bool pending = false;
  // Device-side parse: one error word per job (mapped pinned host memory; bit 0: a DCT partition was read past
  // its end, bit 1: the first partition was) and the streams of the batch, so that a failure names its stream.
  int *h_status = nullptr, *d_status = nullptr;  // mapped pinned host memory and its device alias: the host's copy
  int *d_status_dev = nullptr;                   // device memory: what the kernels poll (never PCIe)
  std::vector<vp8r_stream *> batch_streams;
  bool any_status = false;
};
}  // namespace

struct vp8r_engine {
  int device = 0;
  unsigned long long id = 0;  // process-wide serial number (vp8r_frame::busy_engine)
  cudaStream_t st = nullptr;
  bool own_stream = false;
  // Batches in flight between the host and the last kernel / packed read-backs in flight.  A batch of
  // device-parsed frames is ~100 ms on its way (header chains, token chains, reconstruction, read-back), so the
  // rate is (batches in flight) / latency until something saturates: eight, not four (profiles/r2_summary.md).
  static constexpr int kSlots = 8;
  static constexpr int kPackBufs = 8;
  Slot slots[kSlots];
  int cur_slot = 0;
  // ticket + per-(frame, band) progress words of the wavefront kernels
  int *d_sync = nullptr;
  int sync_cap = 0;
  // device staging of packed I420 frames (vp8r_read_batch_packed): two halves, so that the D2H
  // copy of one time step (on st_copy) overlaps the kernels of the next (on st)
  uint8_t *d_pack = nullptr;
  size_t pack_cap = 0;  // bytes per half
  cudaStream_t st_copy = nullptr;
  // parse streams, one per batch slot: staging, K_modes and K_tokens of the time steps in flight run side by
  // side here while the reconstruction kernels of the oldest run on `st` (the parse kernels are latency-bound
  // single-lane chains: what they need is many of them resident, and they leave the SMs' issue slots to the
  // reconstruction kernels).  K_segments, the only cross-frame dependency of the parse, runs on st_segments in
  // batch order between K_modes and K_tokens of its batch.
  cudaStream_t st_parse[kSlots] = {};
  cudaStream_t st_segments = nullptr;
  cudaEvent_t pack_done[kPackBufs] = {}, copy_done[kPackBufs] = {};
  bool copy_busy[kPackBufs] = {};
  bool kernel_busy[kPackBufs] = {};  // pack_done of the part marks an output kernel (RunOutputJobs) not yet waited for
  cudaEvent_t consumer_ev = nullptr;  // WaitForCaller: the caller's stream, before the engine's work
  cudaEvent_t fence_copy_ev[16] = {};
  bool fence_has_copy[16] = {};
  // checksum scratch
  DevFrameJob *h_cjobs = nullptr, *d_cjobs = nullptr;
  unsigned long long *d_sums = nullptr, *h_sums = nullptr;
  int cap_cjobs = 0;
  int pack_flip = 0;
  // host-visible fences (vp8r_engine_fence / vp8r_engine_wait)
  cudaEvent_t fence_ev[16] = {};
  uint64_t fence_head = 0;
  // first failure of a device-side parse that has been found but not yet reported
  std::string deferred_error;
  // loop filter form: 0 = by batch size (the batch form from kSwarMinFrames filtered frames on), 1 = always the
  // scalar form, 2 = always the batch form.  VP8R_FILTER=scalar|swar forces one, so that tests can run both forms
  // on the same batch.
  int filter_mode = 0;
  static constexpr int kSwarMinFrames = 128;  // measured: 64 frames 1.22 ms (batch) vs 1.06 (scalar); 256: 1.67 vs 2.23; 512: 2.61 vs 4.11
  // timing
  bool timing = false;
  std::vector<EventPair> live;
  std::vector<EventPair> pool;
  vp8r_timers acc{};
};

namespace {

int EnsureDevice(vp8r_engine *e) {
  CU_TRY(cudaSetDevice(e->device));
  return VP8R_OK;
}

cudaError_t SyncParseStreams(vp8r_engine *e) {
  for (auto st : e->st_parse)
    if (st) {
      cudaError_t err = cudaStreamSynchronize(st);
      if (err != cudaSuccess) return err;
    }
  return e->st_segments ? cudaStreamSynchronize(e->st_segments) : cudaSuccess;
}

void FreeSurfaces(vp8r_stream *s) {
  for (auto &sf : s->surf) {
    if (sf.base) cudaFree(sf.base);
    sf = vp8r::Surface{};
  }
  if (s->d_segmap) cudaFree(s->d_segmap);
  s->d_segmap = nullptr;
  if (s->d_tmaps) cudaFree(s->d_tmaps);
  s->d_tmaps = nullptr;
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda).
using EncodeTiledFn = CUresult (*)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                   const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn TensorMapEncoder() {
  static EncodeTiledFn fn = [] {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
      cudaGetLastError();
      p = nullptr;
    }
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  return fn;
}

// One descriptor per padded plane: bytes, x fastest, rows `pitch` apart; box = the motion-compensation window.
bool EncodePlaneMap(vp8r::DevTensorMap *out, uint8_t *padded_origin, int padded_w, int padded_h, int pitch, int box_w, int box_h) {
  static_assert(sizeof(vp8r::DevTensorMap) == sizeof(CUtensorMap), "opaque descriptor size");
  EncodeTiledFn enc = TensorMapEncoder();
  if (!enc) return false;
  const cuuint64_t dims[2] = {cuuint64_t(padded_w), cuuint64_t(padded_h)};
  const cuuint64_t strides[1] = {cuuint64_t(pitch)};
  const cuuint32_t box[2] = {cuuint32_t(box_w), cuuint32_t(box_h)};
  const cuuint32_t estr[2] = {1, 1};
  if (enc(reinterpret_cast<CUtensorMap *>(out), CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, padded_origin, dims, strides, box, estr,
          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
    return false;
  // Drivers up to CUDA 13.1 set a descriptor bit for tensors below 128 KB with which the load traps ("illegal
  // instruction", measured here with tools/microbench/tma_probe.cu); CUTLASS clears the same bit
  // (cute/atom/copy_traits_sm90_tma.hpp).
  static const int driver = [] {
    int v = 0;
    if (cudaDriverGetVersion(&v) != cudaSuccess) cudaGetLastError();
    return v;
  }();
  if (driver <= 13010 && size_t(pitch) * padded_h < 131072) {
    uint64_t w1;
    std::memcpy(&w1, out->opaque + 8, 8);
    w1 &= ~(uint64_t(1) << 21);
    std::memcpy(out->opaque + 8, &w1, 8);
  }
  return true;
}

// Device areas behind a frame's blob that the parse kernel fills (deferred tokens / modes).  All
// offsets are from the start of the device copy of the blob and multiples of 32 bytes.
struct DevExtra {
  size_t mb_off = 0, split_off = 0, coef_off = 0, level_off = 0, dyn_off = 0, total = 0;
};
DevExtra FrameDevExtra(const vp8r_frame *f) {
  DevExtra x;
  const vp8r_frame_hdr &h = f->hdr;
  size_t at = (f->used_bytes() + 255) & ~size_t(255);
  if (!h.tokens_deferred) {
    x.total = at;
    return x;
  }
  const size_t n_mb = size_t(h.mb_cols) * h.mb_rows;
  if (h.modes_deferred) {
    x.mb_off = at;
    at += n_mb * sizeof(vp8r_mb_info);
    x.split_off = at;
    at += n_mb * 64;
  }
  x.coef_off = at;
  at += vp8r::TokenCoefBlocks(h.mb_cols, h.mb_rows) * 32;
  if (h.modes_deferred) {
    x.level_off = at;
    at += ((64 + n_mb) * 4 + 31) & ~size_t(31);
    x.dyn_off = at;
    at += 32;
  }
  x.total = (at + 255) & ~size_t(255);
  return x;
}

// (Re)allocates the stream's surface pool for a new frame size (key frames only; the reference
// allocates a fresh Frame per frame, src/decode.cc:65-71).
int ConfigureStream(vp8r_stream *s, const vp8r_frame_hdr &h) {
  if (s->mb_cols == h.mb_cols && s->mb_rows == h.mb_rows && s->surf[0].base) {
    s->width = h.width;
    s->height = h.height;
    return VP8R_OK;
  }
  CU_TRY(SyncParseStreams(s->eng));
  CU_TRY(cudaStreamSynchronize(s->eng->st));
  FreeSurfaces(s);
  // until the new pool is complete the stream has no geometry and no frame: a failure below leaves nothing to decode
  s->mb_cols = s->mb_rows = 0;
  s->have_frame = false;
  const int B = vp8r::kBorder;
  const int wa = h.mb_cols * 16, ha = h.mb_rows * 16;
  s->pitch_y = wa + 2 * B;
  s->pitch_c = (wa / 2 + 2 * B + 15) & ~15;
  const size_t ysz = (size_t(s->pitch_y) * (ha + 2 * B) + 255) & ~size_t(255);
  const size_t csz = (size_t(s->pitch_c) * (ha / 2 + 2 * B) + 255) & ~size_t(255);
  for (auto &sf : s->surf) {
    void *p = nullptr;
    cudaError_t err = cudaMalloc(&p, ysz + 2 * csz + 256);
    if (err != cudaSuccess) {
      SetError(std::string("cudaMalloc(surface): ") + cudaGetErrorString(err));
      return VP8R_ERR_NOMEM;
    }
    sf.base = static_cast<uint8_t *>(p);
    CU_TRY(cudaMemsetAsync(p, 0, ysz + 2 * csz + 256, s->eng->st));
    sf.planes.y = sf.base + size_t(B) * s->pitch_y + B;
    sf.planes.u = sf.base + ysz + size_t(B) * s->pitch_c + B;
    sf.planes.v = sf.base + ysz + csz + size_t(B) * s->pitch_c + B;
  }
  {  // TMA descriptors of the padded planes: motion compensation fetches its reference windows with them
    vp8r::DevTensorMap h_maps[15];
    for (int k = 0; k < 5; ++k) {
      uint8_t *base = s->surf[k].base;
      if (!EncodePlaneMap(&h_maps[3 * k + 0], base, s->pitch_y, ha + 2 * B, s->pitch_y, vp8r::kTmaLumaBoxW, vp8r::kTmaLumaBoxH) ||
          !EncodePlaneMap(&h_maps[3 * k + 1], base + ysz, s->pitch_c, ha / 2 + 2 * B, s->pitch_c, vp8r::kTmaChromaBoxW, vp8r::kTmaChromaBoxH) ||
          !EncodePlaneMap(&h_maps[3 * k + 2], base + ysz + csz, s->pitch_c, ha / 2 + 2 * B, s->pitch_c, vp8r::kTmaChromaBoxW, vp8r::kTmaChromaBoxH)) {
        SetError("cuTensorMapEncodeTiled failed for a reference plane (no driver entry point, or the descriptor was refused)");
        return VP8R_ERR_CUDA;
      }
    }
    void *p = nullptr;
    if (cudaMalloc(&p, sizeof(h_maps)) != cudaSuccess) {
      SetError("cudaMalloc(tensor maps) failed");
      return VP8R_ERR_NOMEM;
    }
    s->d_tmaps = static_cast<vp8r::DevTensorMap *>(p);
    CU_TRY(cudaMemcpyAsync(p, h_maps, sizeof(h_maps), cudaMemcpyHostToDevice, s->eng->st));
    CU_TRY(cudaStreamSynchronize(s->eng->st));  // h_maps is on the stack
  }
  {
    const size_t n_mb = size_t(h.mb_cols) * h.mb_rows;
    void *p = nullptr;
    if (cudaMalloc(&p, n_mb + 256) != cudaSuccess) {
      SetError("cudaMalloc(segment map) failed");
      return VP8R_ERR_NOMEM;
    }
    s->d_segmap = static_cast<uint8_t *>(p);
    CU_TRY(cudaMemsetAsync(p, 0, n_mb + 256, s->eng->st));
  }
  CU_TRY(cudaStreamSynchronize(s->eng->st));  // the clears must land before the parse stream touches the new buffers
  s->mb_cols = h.mb_cols;
  s->mb_rows = h.mb_rows;
  s->width = h.width;
  s->height = h.height;
  s->ref[0] = s->ref[1] = s->ref[2] = s->ref[3] = -1;
  return VP8R_OK;
}

// A buffer that Regrow replaces: device memory, or pinned host memory (mapped into the device's address space when
// `mapped` receives its device pointer).
struct GrownBuffer {
  void **p;
  size_t bytes;
  bool host;
  void **mapped;
};
template <class T>
GrownBuffer DeviceBuf(T **p, size_t bytes) {
  return {reinterpret_cast<void **>(p), bytes, false, nullptr};
}
template <class T>
GrownBuffer PinnedBuf(T **p, size_t bytes, T **mapped = nullptr) {
  return {reinterpret_cast<void **>(p), bytes, true, reinterpret_cast<void **>(mapped)};
}

// Replaces buffers that share one capacity by larger ones.  *capacity becomes `cap` only once every buffer is in
// place.  A refused allocation leaves it 0 and the refused buffer null, so that the next call allocates again, and
// clears the runtime's last error, which the next launch check would otherwise report as a failure of its own.
template <class Cap>
cudaError_t Regrow(Cap *capacity, Cap cap, std::initializer_list<GrownBuffer> bufs) {
  *capacity = 0;
  for (const GrownBuffer &b : bufs) {
    if (*b.p) b.host ? cudaFreeHost(*b.p) : cudaFree(*b.p);
    *b.p = nullptr;
    if (b.mapped) *b.mapped = nullptr;
  }
  for (const GrownBuffer &b : bufs) {
    cudaError_t err = b.host ? cudaHostAlloc(b.p, b.bytes, b.mapped ? cudaHostAllocMapped : cudaHostAllocDefault)
                             : cudaMalloc(b.p, b.bytes);
    if (err == cudaSuccess && b.mapped) err = cudaHostGetDevicePointer(b.mapped, *b.p, 0);
    if (err != cudaSuccess) {
      cudaGetLastError();
      return err;
    }
  }
  *capacity = cap;
  return cudaSuccess;
}

int GrowSlot(vp8r_engine *e, Slot &sl, int n_jobs, size_t arena_bytes) {
  if (n_jobs > sl.cap_jobs) {
    int cap = std::max(n_jobs, sl.cap_jobs * 2);
    cap = std::max(cap, 16);
    CU_TRY(cudaStreamSynchronize(e->st));
    // the batch's filter groups (at most one per job) follow the jobs in the same table
    const size_t table = (sizeof(DevFrameJob) + sizeof(vp8r::FilterGroup)) * cap + 16;
    CU_TRY(Regrow(&sl.cap_jobs, cap, {PinnedBuf(&sl.h_jobs, table), DeviceBuf(&sl.d_jobs, table),
                                      PinnedBuf(&sl.h_status, sizeof(int) * cap, &sl.d_status),
                                      DeviceBuf(&sl.d_status_dev, sizeof(int) * cap)}));
    std::memset(sl.h_status, 0, sizeof(int) * cap);
  }
  if (arena_bytes > sl.arena_cap) {
    const size_t cap = std::max(arena_bytes + arena_bytes / 4, size_t(1) << 20);
    CU_TRY(cudaStreamSynchronize(e->st));
    CU_TRY(Regrow(&sl.arena_cap, cap, {DeviceBuf(&sl.d_arena, cap)}));
  }
  return VP8R_OK;
}

EventPair GetPair(vp8r_engine *e, Timer cls) {
  EventPair p;
  if (!e->pool.empty()) {
    p = e->pool.back();
    e->pool.pop_back();
  } else {
    cudaEventCreate(&p.a);
    cudaEventCreate(&p.b);
  }
  p.cls = cls;
  return p;
}

struct ScopedTimer {
  vp8r_engine *e;
  EventPair p;
  bool on;
  cudaStream_t stream;
  ScopedTimer(vp8r_engine *eng, Timer cls, cudaStream_t on_stream = nullptr)
      : e(eng), on(eng->timing && cls != Timer::kNone), stream(on_stream ? on_stream : eng->st) {
    if (on) {
      p = GetPair(e, cls);
      cudaEventRecord(p.a, stream);
    }
  }
  ~ScopedTimer() {
    if (on) {
      cudaEventRecord(p.b, stream);
      e->live.push_back(p);
    }
  }
};

void DrainTimers(vp8r_engine *e) {
  for (auto &p : e->live) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) {
      switch (p.cls) {
        case Timer::kInter: e->acc.ms_inter += ms; break;
        case Timer::kIntra: e->acc.ms_intra += ms; break;
        case Timer::kFilter: e->acc.ms_filter += ms; break;
        case Timer::kH2D: e->acc.ms_h2d += ms; break;
        case Timer::kD2H: e->acc.ms_d2h += ms; break;
        case Timer::kTokens: e->acc.ms_tokens += ms; break;
        case Timer::kBorder: e->acc.ms_border += ms; break;
        case Timer::kNone: break;
      }
    } else {
      cudaGetLastError();
    }
    e->pool.push_back(p);
  }
  e->live.clear();
}

// Scratch job tables of the read-back / checksum paths (kPackBufs parts) and the checksum words.
int EnsureScratchJobs(vp8r_engine *e, int n) {
  if (n <= e->cap_cjobs) return VP8R_OK;
  CU_TRY(cudaStreamSynchronize(e->st));
  const int cap = std::max(n, 64);
  const size_t table = sizeof(DevFrameJob) * cap * vp8r_engine::kPackBufs + 16;
  CU_TRY(Regrow(&e->cap_cjobs, cap, {PinnedBuf(&e->h_cjobs, table), DeviceBuf(&e->d_cjobs, table),
                                     PinnedBuf(&e->h_sums, sizeof(uint64_t) * cap), DeviceBuf(&e->d_sums, sizeof(uint64_t) * cap)}));
  return VP8R_OK;
}

// Takes the next of the kPackBufs rotating parts of the scratch job table (and of the packed staging buffer) for a
// read-back.  LaunchCopy reads a part from pinned host memory while its kernel runs, so the host rewrites the part
// only after the work that last read it has finished: the D2H copy of a packed read-back (which follows its pack
// kernel), or the kernel of any other output.
int AcquirePart(vp8r_engine *e, int *part) {
  e->pack_flip = (e->pack_flip + 1) % vp8r_engine::kPackBufs;
  const int k = e->pack_flip;
  if (e->copy_busy[k]) {
    CU_TRY(cudaEventSynchronize(e->copy_done[k]));
    e->copy_busy[k] = false;
  }
  if (e->kernel_busy[k]) {
    CU_TRY(cudaEventSynchronize(e->pack_done[k]));
    e->kernel_busy[k] = false;
  }
  *part = k;
  return VP8R_OK;
}

// Makes the engine's stream wait for the work queued so far on a caller's stream.  A null stream, or the engine's own,
// asks for nothing; torch's default stream arrives as cudaStreamLegacy and is waited for like any other.
int WaitForCaller(vp8r_engine *e, cudaStream_t caller) {
  if (!caller || caller == e->st) return VP8R_OK;
  CU_TRY(cudaEventRecord(e->consumer_ev, caller));
  CU_TRY(cudaStreamWaitEvent(e->st, e->consumer_ev, 0));
  return VP8R_OK;
}

// Makes a caller's stream wait for `ev`, recorded on the engine's stream (the same rules as WaitForCaller).
int CallerWaitsFor(vp8r_engine *e, cudaStream_t caller, cudaEvent_t ev) {
  if (!caller || caller == e->st) return VP8R_OK;
  CU_TRY(cudaStreamWaitEvent(caller, ev, 0));
  return VP8R_OK;
}

// The path of every output that runs one kernel over a scratch job table (packed, device, conversion, checksum): n jobs
// in the next rotating part (*part, set before fill runs), each cleared and then set by fill(i, job).  The part goes to
// the device with LaunchCopy and launch(device jobs) queues the kernel, timed as `cls`, on the engine's stream behind
// the work queued on `caller` so far (nullptr: none).  pack_done[part] marks the part busy until the kernel has
// finished, and the caller's stream waits for it.
template <class Fill, class Launch>
int RunOutputJobs(vp8r_engine *e, int n, Timer cls, cudaStream_t caller, int *part, Fill fill, Launch launch) {
  int rc = EnsureScratchJobs(e, n);
  if (!rc) rc = AcquirePart(e, part);
  if (rc) return rc;
  DevFrameJob *hj = e->h_cjobs + size_t(*part) * e->cap_cjobs, *dj = e->d_cjobs + size_t(*part) * e->cap_cjobs;
  for (int i = 0; i < n; ++i) {
    std::memset(&hj[i], 0, sizeof(DevFrameJob));
    fill(i, hj[i]);
  }
  rc = WaitForCaller(e, caller);
  if (rc) return rc;
  {
    ScopedTimer t(e, cls);
    CU_TRY(vp8r::LaunchCopy(dj, hj, sizeof(DevFrameJob) * n, e->st));
    CU_TRY(launch(dj));
    e->acc.launches_other++;
  }
  CU_TRY(cudaEventRecord(e->pack_done[*part], e->st));
  e->kernel_busy[*part] = true;
  return CallerWaitsFor(e, caller, e->pack_done[*part]);
}

// Error words of a batch whose kernels have finished: a stream with a truncated frame stops decoding (its frame
// was not reconstructed, see JobFailed in the kernels) until its next key frame.  The first failure found is kept
// in e->deferred_error unless an earlier one is still unreported there.  Returns the number of failures and, in
// *what (optional), describes the first one of this batch.
int HarvestStatus(vp8r_engine *e, Slot &sl, std::string *what) {
  int failures = 0;
  if (!sl.any_status) return 0;
  std::string first;
  for (size_t i = 0; i < sl.batch_streams.size(); ++i) {
    const int w = static_cast<volatile int *>(sl.h_status)[i];
    if (w == 0) continue;
    sl.h_status[i] = 0;
    vp8r_stream *s = sl.batch_streams[i];
    if (s) {
      s->failed = true;
      s->have_frame = false;
      s->ref[0] = s->ref[1] = s->ref[2] = s->ref[3] = -1;
    }
    if (failures++ == 0)
      first = "stream " + std::to_string(i) + " of the batch: " + ((w & 2) ? "the first partition" : "a DCT partition") +
              " was read past its end (device-side parse); the stream is stopped until its next key frame";
  }
  sl.any_status = false;
  sl.batch_streams.clear();
  if (failures && e->deferred_error.empty()) e->deferred_error = first;
  if (failures && what) *what = first;
  return failures;
}

void FillJobSurfaces(const vp8r_stream *s, int cur, DevFrameJob *j) {
  j->cur = s->surf[cur].planes;
  for (int k = 1; k < 4; ++k) {
    j->ref[k] = s->ref[k] >= 0 ? s->surf[s->ref[k]].planes : vp8r::DevPlanes{};
    j->ref_tmap[k] = s->ref[k] >= 0 ? s->d_tmaps + 3 * s->ref[k] : nullptr;
  }
  j->ref[0] = vp8r::DevPlanes{};
  j->ref_tmap[0] = nullptr;
  j->pitch_y = s->pitch_y;
  j->pitch_c = s->pitch_c;
  j->mb_cols = s->mb_cols;
  j->mb_rows = s->mb_rows;
  j->width = s->width;
  j->height = s->height;
}

// Encoder input: a cropped I420 image padded to whole macroblocks by replicating the last row / column (what an
// encoder does with the invisible part is its own business; replication keeps its residual small).  dst: Y plane of
// pitch cols*16, then U and V of pitch cols*8, each rows*16 / rows*8 lines.
void PadToMacroblocks(const uint8_t *i420, int width, int height, int cols, int rows, uint8_t *dst) {
  const int sp_y = cols * 16, sp_c = cols * 8;
  const int cw = (width + 1) / 2, ch = (height + 1) / 2;
  const uint8_t *py = i420, *pu = py + size_t(width) * height, *pv = pu + size_t(cw) * ch;
  uint8_t *dy = dst, *du = dy + size_t(sp_y) * rows * 16, *dv = du + size_t(sp_c) * rows * 8;
  auto pad = [](uint8_t *d, int dp, int dw, int dh, const uint8_t *src, int sw, int sh) {
    for (int y = 0; y < dh; ++y) {
      const uint8_t *srow = src + size_t(std::min(y, sh - 1)) * sw;
      uint8_t *drow = d + size_t(y) * dp;
      std::memcpy(drow, srow, size_t(sw));
      std::memset(drow + sw, srow[sw - 1], size_t(dw - sw));
    }
  };
  pad(dy, sp_y, sp_y, rows * 16, py, width, height);
  pad(du, sp_c, sp_c, rows * 8, pu, cw, ch);
  pad(dv, sp_c, sp_c, rows * 8, pv, cw, ch);
}

// ------------------------------------------------------------- steps of a batch submission ----
// The streams of a batch: each of this engine and in the batch once.
int CheckBatchStreams(const vp8r_engine *e, int n, vp8r_stream *const *streams) {
  std::vector<const vp8r_stream *> seen(streams, streams + n);
  std::sort(seen.begin(), seen.end());
  if (std::adjacent_find(seen.begin(), seen.end()) != seen.end()) {
    SetError("a stream appears twice in one batch (frames of one stream are a dependency chain: one per batch)");
    return VP8R_ERR_INVALID_ARG;
  }
  for (int i = 0; i < n; ++i)
    if (!streams[i] || streams[i]->eng != e) {
      SetError("null stream or stream of another engine");
      return VP8R_ERR_INVALID_ARG;
    }
  return VP8R_OK;
}

// Takes the next slot: waits for the batch that last used it, harvests its error words and sizes the slot for n_jobs
// jobs and arena_bytes of staging.  *failure (optional) describes the first failure harvested, if any.
int TakeSlot(vp8r_engine *e, int n_jobs, size_t arena_bytes, int *slot_index, std::string *failure) {
  const int k = e->cur_slot;
  Slot &sl = e->slots[k];
  e->cur_slot = (k + 1) % vp8r_engine::kSlots;
  if (sl.pending) {
    CU_TRY(cudaEventSynchronize(sl.done));
    sl.pending = false;
  }
  HarvestStatus(e, sl, failure);
  *slot_index = k;
  return GrowSlot(e, sl, n_jobs, arena_bytes);
}

// CURRENT = a surface no reference points at, and not the previous output.
int PickCurrent(const vp8r_stream *s) {
  for (int k = 0; k < 5; ++k)
    if (k != s->ref[0] && k != s->ref[1] && k != s->ref[2] && k != s->ref[3]) return k;
  return -1;
}

// Filter groups for FilterSwarKernel, behind the batch's n jobs in the slot's table: the filtered jobs with the same
// geometry and filter type, eight to a warp, in batch order within a group (filter_swar.cu).  There are none when the
// scalar FilterKernel runs (fewer than kSwarMinFrames filtered frames, or VP8R_FILTER=scalar).  Returns their number.
int BuildFilterGroups(const vp8r_engine *e, Slot &sl, int n) {
  const DevFrameJob *jobs = sl.h_jobs;
  std::vector<int> order;
  for (int i = 0; i < n; ++i)
    if (jobs[i].lf_level != 0) order.push_back(i);
  const bool swar = e->filter_mode == 2 || (e->filter_mode == 0 && int(order.size()) >= vp8r_engine::kSwarMinFrames);
  if (!swar || order.empty()) return 0;
  auto key = [&](int i) {
    return (uint64_t(jobs[i].mb_cols) << 32) | (uint64_t(jobs[i].mb_rows) << 8) | uint64_t(jobs[i].filter_type != 0);
  };
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return key(a) < key(b); });
  vp8r::FilterGroup *hg = reinterpret_cast<vp8r::FilterGroup *>(sl.h_jobs + n);
  int n_groups = 0;
  for (size_t at = 0; at < order.size();) {
    vp8r::FilterGroup g;
    int k = 0;
    const uint64_t kk = key(order[at]);
    for (; k < 8 && at < order.size() && key(order[at]) == kk; ++k, ++at) g.frame[k] = order[at];
    for (; k < 8; ++k) g.frame[k] = -1;
    hg[n_groups++] = g;
  }
  return n_groups;
}

// Loop filter and border extension of a batch whose jobs and filter groups are on the device.
int LaunchFilterAndBorder(vp8r_engine *e, const Slot &sl, int n, int max_rows, int n_groups) {
  {
    ScopedTimer t(e, Timer::kFilter);
    const int need_sync = vp8r::FilterSyncInts(n);
    if (need_sync > e->sync_cap) {
      CU_TRY(cudaStreamSynchronize(e->st));
      CU_TRY(Regrow(&e->sync_cap, need_sync * 2, {DeviceBuf(&e->d_sync, sizeof(int) * size_t(need_sync) * 2)}));
    }
    CU_TRY(vp8r::LaunchFilter(sl.d_jobs, n, max_rows, e->d_sync, e->sync_cap, e->st,
                              reinterpret_cast<const vp8r::FilterGroup *>(sl.d_jobs + n), n_groups));
    e->acc.launches_filter++;
  }
  ScopedTimer t(e, Timer::kBorder);
  CU_TRY(vp8r::LaunchBorder(sl.d_jobs, n, e->st));
  e->acc.launches_other++;
  return VP8R_OK;
}

// RefreshRefFrames (src/loop.h:19-46) on surface indices, after a frame with header h was reconstructed into cur.
void RefreshRefs(vp8r_stream *s, const vp8r_frame_hdr &h, int cur) {
  const bool g2a = !h.refresh_altref && h.copy_to_altref == 2;
  const bool a2g = !h.refresh_golden && h.copy_to_golden == 2;
  if (g2a && a2g) std::swap(s->ref[2], s->ref[3]);
  else if (g2a) s->ref[3] = s->ref[2];
  else if (a2g) s->ref[2] = s->ref[3];
  if (h.refresh_golden) s->ref[2] = cur;
  else if (h.copy_to_golden == 1) s->ref[2] = s->ref[1];
  if (h.refresh_altref) s->ref[3] = cur;
  else if (h.copy_to_altref == 1) s->ref[3] = s->ref[1];
  if (h.refresh_last) s->ref[1] = cur;
  s->ref[0] = cur;
  s->have_frame = true;
}

// Where an encoder batch's pictures come from: cropped I420 images in host memory, one per frame (host), or n frames
// in device memory of the engine's device, frame i at dev + i*stride in `layout` (StageSourceKernel converts them).
struct EncoderSource {
  const uint8_t *const *host = nullptr;
  const uint8_t *dev = nullptr;
  size_t stride = 0;
  int layout = VP8R_LAYOUT_I420;
  cudaStream_t producer = nullptr;  // the stream dev was written on (nullptr: nothing to wait for)
};

// Bytes of one width x height frame in a source / device layout.
size_t LayoutBytes(int layout, int width, int height) {
  if (layout == VP8R_LAYOUT_RGB24 || layout == VP8R_LAYOUT_RGB_PLANAR) return 3 * size_t(width) * height;
  return size_t(width) * height + 2 * size_t((width + 1) / 2) * ((height + 1) / 2);
}

// A pointer into device memory of the engine's device (pinned, pageable and managed memory are not).
bool IsEngineDeviceMemory(const vp8r_engine *e, const void *p) {
  cudaPointerAttributes attr{};
  if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return attr.type == cudaMemoryTypeDevice && attr.device == e->device;
}

// A layout of include/vp8r.h and a frame size VP8 can code.  `call` names the refused call.
int CheckLayoutAndSize(const std::string &call, int layout, int width, int height) {
  if (layout < VP8R_LAYOUT_I420 || layout > VP8R_LAYOUT_RGB_PLANAR) {
    SetError(call + ": unknown layout " + std::to_string(layout));
    return VP8R_ERR_INVALID_ARG;
  }
  if (width < 1 || height < 1 || width > 16383 || height > 16383) {
    SetError(call + ": frame size outside 1..16383");
    return VP8R_ERR_INVALID_ARG;
  }
  return VP8R_OK;
}

// The distance of two frames of a batch holds a width x height frame in `layout`.  `what` names the stride.
int CheckStride(const std::string &what, size_t stride, int layout, int width, int height) {
  if (stride >= LayoutBytes(layout, width, height)) return VP8R_OK;
  SetError(what + " smaller than a frame");
  return VP8R_ERR_INVALID_ARG;
}

// The streams of an output: each of this engine with a reconstructed frame, which fits `stride` in `layout`.
int CheckFrameStreams(const vp8r_engine *e, int n, vp8r_stream *const *streams, size_t stride = SIZE_MAX,
                      int layout = VP8R_LAYOUT_I420) {
  for (int i = 0; i < n; ++i) {
    const vp8r_stream *s = streams[i];
    if (!s || s->eng != e || !s->have_frame) {
      SetError("stream has no reconstructed frame");
      return VP8R_ERR_STATE;
    }
    const int rc = CheckStride("stride", stride, layout, s->width, s->height);
    if (rc) return rc;
  }
  return VP8R_OK;
}

// The arguments of the encoder calls, with a message naming the call for each refusal.  search_range < 0: a key-frame
// call, which takes none (and whose flags are not checked).  The checks that need neither the engine nor a stream come
// first.
int CheckEncoderArgs(vp8r_engine *e, int n, vp8r_stream *const *streams, const EncoderSource &src, vp8r_frame *const *out,
                     int width, int height, int q_index, int loop_filter_level, int sharpness, int search_range,
                     unsigned flags) {
  const std::string call = std::string(search_range < 0 ? "vp8r_encode_key_frames" : "vp8r_encode_inter_frames") +
                           (src.dev ? "_device" : "");
  if (!e || !streams || !(src.host || src.dev) || !out) {
    SetError(call + ": null engine, streams, src or out");
    return VP8R_ERR_INVALID_ARG;
  }
  if (n <= 0) {
    SetError(call + ": n <= 0");
    return VP8R_ERR_INVALID_ARG;
  }
  int rc = CheckLayoutAndSize(call, src.layout, width, height);
  if (rc) return rc;
  if (q_index < 0 || q_index > 127 || loop_filter_level < 0 || loop_filter_level > 63 || sharpness < 0 || sharpness > 7) {
    SetError(call + ": q_index, loop_filter_level or sharpness out of range");
    return VP8R_ERR_INVALID_ARG;
  }
  if (src.dev && (rc = CheckStride(call + ": stride", src.stride, src.layout, width, height))) return rc;
  if (search_range >= 0 && (search_range < 4 || search_range > 24)) {
    SetError(call + ": search_range outside 4..24");
    return VP8R_ERR_INVALID_ARG;
  }
  if (search_range >= 0 && (flags & ~(VP8R_ENC_INTRA_MBS | VP8R_ENC_BPRED))) {
    SetError(call + "_ex: unknown flag bits");
    return VP8R_ERR_INVALID_ARG;
  }
  if (search_range >= 0 && (flags & VP8R_ENC_BPRED) && !(flags & VP8R_ENC_INTRA_MBS)) {
    SetError(call + "_ex: VP8R_ENC_BPRED needs VP8R_ENC_INTRA_MBS");
    return VP8R_ERR_INVALID_ARG;
  }
  rc = EnsureDevice(e);
  if (rc) return rc;
  rc = CheckBatchStreams(e, n, streams);
  if (rc) return rc;
  for (int i = 0; i < n; ++i)
    if ((src.host && !src.host[i]) || !out[i]) {
      SetError("null image or frame");
      return VP8R_ERR_INVALID_ARG;
    }
  if (src.dev && !IsEngineDeviceMemory(e, src.dev)) {
    SetError("src is not device memory of the engine's device (pinned, pageable and managed memory are refused)");
    return VP8R_ERR_INVALID_ARG;
  }
  return VP8R_OK;
}

// An encoder batch: the header of its frames (the fields both encoders share; the caller adds its own) and the
// layout of its slot arena.  Per frame the arena holds the source image padded to whole macroblocks (Y of pitch
// cols*16, then U and V of pitch cols*8), the records the kernels write and their blocks (25 per macroblock), and one
// uint32 per macroblock for the inter prediction's error (VP8R_ENC_INTRA_MBS), each part 256-byte aligned.
struct EncodeLayout {
  vp8r_frame_hdr h{};
  size_t n_mb = 0, src_bytes = 0, mb_bytes = 0, pay_bytes = 0, err_at = 0, per_frame = 0;
};
EncodeLayout MakeEncodeLayout(int width, int height, int q_index, int loop_filter_level, int sharpness) {
  EncodeLayout L;
  vp8r_frame_hdr &h = L.h;
  h.width = uint16_t(width);
  h.height = uint16_t(height);
  h.mb_cols = uint16_t((width + 15) / 16);
  h.mb_rows = uint16_t((height + 15) / 16);
  h.show_frame = 1;
  h.loop_filter_level = uint8_t(loop_filter_level);
  h.sharpness_level = uint8_t(sharpness);
  h.refresh_last = 1;
  h.q_index = uint8_t(q_index);
  vp8r::DequantFactorsForIndex(q_index, h.dq[0]);
  const size_t cols = h.mb_cols, rows = h.mb_rows;
  L.n_mb = cols * rows;
  L.src_bytes = (cols * 16 * rows * 16 + 2 * cols * 8 * rows * 8 + 255) & ~size_t(255);
  L.mb_bytes = (L.n_mb * sizeof(vp8r_mb_info) + 255) & ~size_t(255);
  L.pay_bytes = L.n_mb * 25 * 32;
  L.err_at = L.src_bytes + L.mb_bytes + ((L.pay_bytes + 255) & ~size_t(255));
  L.per_frame = L.err_at + ((L.n_mb * sizeof(uint32_t) + 255) & ~size_t(255));
  return L;
}

// Fills the job fields both encoders set and stages each frame's source picture, padded to whole macroblocks, in its
// part of the slot arena: a host image is padded here and uploaded; a device source is converted and padded there by
// StageSourceKernel, which SubmitEncoderJobs launches once the job table is on the device.  cur[i] is the surface
// frame i is reconstructed into.
int StageEncoderSources(vp8r_engine *e, Slot &sl, int n, vp8r_stream *const *streams, const EncoderSource &src,
                        const EncodeLayout &L, std::vector<int> *cur) {
  const vp8r_frame_hdr &h = L.h;
  const int cols = h.mb_cols, rows = h.mb_rows, sp_y = cols * 16, sp_c = cols * 8;
  std::vector<uint8_t> padded(src.host ? L.src_bytes : 0);
  cur->assign(size_t(n), -1);
  for (int i = 0; i < n; ++i) {
    vp8r_stream *s = streams[i];
    uint8_t *base = sl.d_arena + L.per_frame * size_t(i);
    if (src.host) {
      PadToMacroblocks(src.host[i], h.width, h.height, cols, rows, padded.data());
      CU_TRY(cudaMemcpyAsync(base, padded.data(), L.src_bytes, cudaMemcpyHostToDevice, e->st));
      CU_TRY(cudaStreamSynchronize(e->st));  // `padded` is reused for the next image
    }
    (*cur)[size_t(i)] = PickCurrent(s);
    DevFrameJob &j = sl.h_jobs[i];
    std::memset(&j, 0, sizeof(j));
    FillJobSurfaces(s, (*cur)[size_t(i)], &j);
    j.mbs = reinterpret_cast<const vp8r_mb_info *>(base + L.src_bytes);
    j.payload = reinterpret_cast<const int16_t *>(base + L.src_bytes + L.mb_bytes);
    std::memcpy(j.dq, h.dq, sizeof(j.dq));
    j.key_frame = h.key_frame;
    j.lf_level = h.loop_filter_level;
    j.sharpness = h.sharpness_level;
    j.enc_src[0] = base;
    j.enc_src[1] = base + size_t(sp_y) * rows * 16;
    j.enc_src[2] = j.enc_src[1] + size_t(sp_c) * rows * 8;
    j.enc_src_pitch_y = sp_y;
    j.enc_src_pitch_c = sp_c;
    if (src.dev) {
      j.stage_src = src.dev + size_t(i) * src.stride;
      j.pack_layout = uint8_t(src.layout);
      j.stage_w = sp_y;
      j.stage_h = rows * 16;
    }
    e->acc.frames++;
  }
  return VP8R_OK;
}

// Builds the batch's filter groups and puts its job table on the device; for a device source, the engine's stream
// then waits for the producer stream and StageSourceKernel stages the pictures.  *n_groups: the filter groups.
int SubmitEncoderJobs(vp8r_engine *e, Slot &sl, int n, const EncoderSource &src, const EncodeLayout &L, int *n_groups) {
  *n_groups = BuildFilterGroups(e, sl, n);
  CU_TRY(vp8r::LaunchCopy(sl.d_jobs, sl.h_jobs, sizeof(DevFrameJob) * n + sizeof(vp8r::FilterGroup) * *n_groups, e->st));
  if (!src.dev) return VP8R_OK;
  const int rc = WaitForCaller(e, src.producer);
  if (rc) return rc;
  ScopedTimer t(e, Timer::kH2D);
  CU_TRY(vp8r::LaunchStageSource(sl.d_jobs, n, src.layout, L.h.mb_cols * 16, L.h.mb_rows * 16, e->st));
  e->acc.launches_other++;
  return VP8R_OK;
}

// Reads the records and blocks of an encoder batch back into `out` (header L.h) and waits for them; then moves each
// stream's references to its reconstruction and counts each frame's coded blocks.
int FinishEncoderBatch(vp8r_engine *e, const Slot &sl, int n, vp8r_stream *const *streams, const std::vector<int> &cur,
                       const EncodeLayout &L, vp8r_frame *const *out) {
  const size_t rec_bytes = L.n_mb * sizeof(vp8r_mb_info);
  for (int i = 0; i < n; ++i) {
    vp8r_frame *f = out[i];
    f->DropDeviceCopy();
    f->hdr = L.h;
    f->n_mb = L.n_mb;
    f->hdr.n_payload_blocks = uint32_t(L.n_mb * 25);
    if (!f->Reserve(rec_bytes + L.pay_bytes, 0)) {
      SetError("out of host memory for the encoded frame");
      return VP8R_ERR_NOMEM;
    }
    const uint8_t *base = sl.d_arena + L.per_frame * size_t(i);
    CU_TRY(cudaMemcpyAsync(f->blob, base + L.src_bytes, rec_bytes, cudaMemcpyDeviceToHost, e->st));
    CU_TRY(cudaMemcpyAsync(f->blob + rec_bytes, base + L.src_bytes + L.mb_bytes, L.pay_bytes, cudaMemcpyDeviceToHost, e->st));
  }
  CU_TRY(cudaStreamSynchronize(e->st));
  for (int i = 0; i < n; ++i) {
    RefreshRefs(streams[i], L.h, cur[size_t(i)]);
    uint32_t blocks = 0;
    const vp8r_mb_info *mbs = out[i]->mbs();
    for (size_t m = 0; m < L.n_mb; ++m) blocks += uint32_t(__builtin_popcount(mbs[m].coef_mask));
    out[i]->hdr.n_coef_blocks = blocks;
  }
  return VP8R_OK;
}

// Row f4: closed-loop key-frame encoder (vp8r_encode_key_frames, _device).
int EncodeKeyFrames(vp8r_engine *e, int n, vp8r_stream *const *streams, const EncoderSource &src, int width, int height,
                    int q_index, int loop_filter_level, int sharpness, unsigned flags, vp8r_frame *const *out) {
  int rc = CheckEncoderArgs(e, n, streams, src, out, width, height, q_index, loop_filter_level, sharpness, -1, flags);
  if (rc) return rc;
  EncodeLayout L = MakeEncodeLayout(width, height, q_index, loop_filter_level, sharpness);
  L.h.key_frame = 1;
  L.h.refresh_golden = L.h.refresh_altref = 1;
  for (int i = 0; i < n; ++i) {
    rc = ConfigureStream(streams[i], L.h);
    if (rc) return rc;
    streams[i]->failed = false;
  }
  int slot_index;
  rc = TakeSlot(e, n, L.per_frame * size_t(n), &slot_index, nullptr);
  if (rc) return rc;
  Slot &sl = e->slots[slot_index];
  std::vector<int> cur;
  rc = StageEncoderSources(e, sl, n, streams, src, L, &cur);
  if (rc) return rc;
  for (int i = 0; i < n; ++i) {
    sl.h_jobs[i].n_intra = int(L.n_mb);
    sl.h_jobs[i].enc_flags = uint8_t(flags);
  }
  int n_groups = 0;
  rc = SubmitEncoderJobs(e, sl, n, src, L, &n_groups);
  if (rc) return rc;
  {
    ScopedTimer t(e, Timer::kIntra);
    CU_TRY(vp8r::LaunchEncodeIntra(sl.d_jobs, n, L.h.mb_rows, e->st));
    e->acc.launches_intra++;
  }
  rc = LaunchFilterAndBorder(e, sl, n, L.h.mb_rows, n_groups);
  if (rc) return rc;
  return FinishEncoderBatch(e, sl, n, streams, cur, L, out);
}

// Row f4, inter frames: every macroblock predicts from LAST with one vector (K_encode_inter), the decoder's own
// K_inter reconstructs from the records; with VP8R_ENC_INTRA_MBS, K_encode_intra_mbs then recodes as intra the
// macroblocks that LAST predicts badly; then the loop filter and the border as for a decoded frame.
int EncodeInterFrames(vp8r_engine *e, int n, vp8r_stream *const *streams, const EncoderSource &src, int width, int height,
                      int q_index, int loop_filter_level, int sharpness, int search_range, unsigned flags,
                      vp8r_frame *const *out) {
  int rc = CheckEncoderArgs(e, n, streams, src, out, width, height, q_index, loop_filter_level, sharpness, search_range, flags);
  if (rc) return rc;
  for (int i = 0; i < n; ++i) {
    const vp8r_stream *s = streams[i];
    if (!s->have_frame || s->failed || s->ref[1] < 0) {
      SetError("inter frame for a stream without a frame to predict from");
      return VP8R_ERR_STATE;
    }
    if (s->width != width || s->height != height) {
      SetError("inter frame of another size than the stream's frames");
      return VP8R_ERR_STATE;
    }
  }
  const EncodeLayout L = MakeEncodeLayout(width, height, q_index, loop_filter_level, sharpness);
  const int cols = L.h.mb_cols, rows = L.h.mb_rows;
  int slot_index;
  rc = TakeSlot(e, n, L.per_frame * size_t(n), &slot_index, nullptr);
  if (rc) return rc;
  Slot &sl = e->slots[slot_index];
  std::vector<int> cur;
  rc = StageEncoderSources(e, sl, n, streams, src, L, &cur);
  if (rc) return rc;
  for (int i = 0; i < n; ++i) {
    DevFrameJob &j = sl.h_jobs[i];
    j.n_inter = int(L.n_mb);
    j.enc_search_range = search_range;
    j.enc_flags = uint8_t(flags);
    if (flags & VP8R_ENC_INTRA_MBS) j.enc_inter_err = reinterpret_cast<uint32_t *>(sl.d_arena + L.per_frame * size_t(i) + L.err_at);
  }
  int n_groups = 0;
  rc = SubmitEncoderJobs(e, sl, n, src, L, &n_groups);
  if (rc) return rc;
  {
    ScopedTimer t(e, Timer::kInter);
    CU_TRY(vp8r::LaunchEncodeInter(sl.d_jobs, n, cols, rows, e->st));
    CU_TRY(vp8r::LaunchInter(sl.d_jobs, n, cols, rows, e->st));
    e->acc.launches_inter += 2;
  }
  if (flags & VP8R_ENC_INTRA_MBS) {
    ScopedTimer t(e, Timer::kIntra);
    CU_TRY(vp8r::LaunchEncodeIntraMbs(sl.d_jobs, n, rows, e->st));
    e->acc.launches_intra++;
  }
  rc = LaunchFilterAndBorder(e, sl, n, rows, n_groups);
  if (rc) return rc;
  // The references move with the reconstruction (golden and altref stay), even if a mode cannot be assigned below.
  rc = FinishEncoderBatch(e, sl, n, streams, cur, L, out);
  if (rc) return rc;
  for (int i = 0; i < n; ++i) {
    std::string err;
    rc = vp8r::AssignInterModes(out[i]->mbs(), cols, rows, &err);
    if (rc) {
      SetError(err);
      return rc;
    }
    uint32_t n_inter = 0;
    const vp8r_mb_info *mbs = out[i]->mbs();
    for (size_t m = 0; m < L.n_mb; ++m) n_inter += (mbs[m].flags & VP8R_MB_IS_INTER) ? 1u : 0u;
    out[i]->hdr.n_inter_mbs = n_inter;
  }
  return VP8R_OK;
}

}  // namespace

// ================================================================== C ABI ===================
extern "C" {

VP8R_API int vp8r_has_cuda(void) { return 1; }

VP8R_API int vp8r_engine_create(int device, void *cuda_stream, vp8r_engine **out) {
  if (!out) return VP8R_ERR_INVALID_ARG;
  *out = nullptr;
  int count = 0;
  cudaError_t err = cudaGetDeviceCount(&count);
  if (err != cudaSuccess || count == 0) {
    cudaGetLastError();
    SetError("no CUDA device available: the reconstruction path has no CPU fallback");
    return VP8R_ERR_CUDA;
  }
  if (device < 0 || device >= count) {
    SetError("device index out of range");
    return VP8R_ERR_INVALID_ARG;
  }
  CU_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) {
    SetError("libvp8r kernels are built for sm_100a only");
    return VP8R_ERR_CUDA;
  }
  vp8r_engine *e = new (std::nothrow) vp8r_engine();
  if (e) {
    static std::atomic<unsigned long long> serial{0};
    e->id = ++serial;
  }
  if (!e) return VP8R_ERR_NOMEM;
  e->device = device;
  if (const char *v = std::getenv("VP8R_FILTER")) e->filter_mode = std::strcmp(v, "scalar") == 0 ? 1 : (std::strcmp(v, "swar") == 0 ? 2 : 0);
  if (cuda_stream) {
    e->st = static_cast<cudaStream_t>(cuda_stream);
  } else {
    if (cudaStreamCreateWithFlags(&e->st, cudaStreamNonBlocking) != cudaSuccess) {
      delete e;
      SetError("cudaStreamCreate failed");
      return VP8R_ERR_CUDA;
    }
    e->own_stream = true;
  }
  for (auto &sl : e->slots) {
    cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&sl.parsed, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&sl.modes_done, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&sl.segments_done, cudaEventDisableTiming);
  }
  cudaStreamCreateWithFlags(&e->st_copy, cudaStreamNonBlocking);
  // (stream priorities were measured: reconstruction stream above the parse streams changes nothing with the
  // read-back on and costs 12 % without it, the staging copies of the parse streams being held back)
  for (auto &st : e->st_parse) cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
  cudaStreamCreateWithFlags(&e->st_segments, cudaStreamNonBlocking);
  for (int k = 0; k < vp8r_engine::kPackBufs; ++k) {
    cudaEventCreateWithFlags(&e->pack_done[k], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&e->copy_done[k], cudaEventDisableTiming);
  }
  cudaEventCreateWithFlags(&e->consumer_ev, cudaEventDisableTiming);
  err = vp8r::InitKernelTables();
  if (err != cudaSuccess) {
    SetError(std::string("kernel table upload: ") + cudaGetErrorString(err));
    vp8r_engine_destroy(e);
    return VP8R_ERR_CUDA;
  }
  *out = e;
  return VP8R_OK;
}

VP8R_API void vp8r_engine_destroy(vp8r_engine *e) {
  if (!e) return;
  cudaSetDevice(e->device);
  cudaStreamSynchronize(e->st);
  if (e->st_copy) {
    cudaStreamSynchronize(e->st_copy);
    cudaStreamDestroy(e->st_copy);
  }
  SyncParseStreams(e);
  for (auto &st : e->st_parse)
    if (st) cudaStreamDestroy(st);
  if (e->st_segments) cudaStreamDestroy(e->st_segments);
  for (int k = 0; k < vp8r_engine::kPackBufs; ++k) {
    if (e->pack_done[k]) cudaEventDestroy(e->pack_done[k]);
    if (e->copy_done[k]) cudaEventDestroy(e->copy_done[k]);
  }
  if (e->consumer_ev) cudaEventDestroy(e->consumer_ev);
  for (auto &ev : e->fence_copy_ev)
    if (ev) cudaEventDestroy(ev);
  for (auto &sl : e->slots) {
    if (sl.h_jobs) cudaFreeHost(sl.h_jobs);
    if (sl.d_jobs) cudaFree(sl.d_jobs);
    if (sl.d_arena) cudaFree(sl.d_arena);
    if (sl.h_status) cudaFreeHost(sl.h_status);
    if (sl.d_status_dev) cudaFree(sl.d_status_dev);
    if (sl.done) cudaEventDestroy(sl.done);
    if (sl.parsed) cudaEventDestroy(sl.parsed);
    if (sl.modes_done) cudaEventDestroy(sl.modes_done);
    if (sl.segments_done) cudaEventDestroy(sl.segments_done);
  }
  if (e->h_cjobs) cudaFreeHost(e->h_cjobs);
  if (e->d_cjobs) cudaFree(e->d_cjobs);
  if (e->h_sums) cudaFreeHost(e->h_sums);
  if (e->d_sums) cudaFree(e->d_sums);
  if (e->d_sync) cudaFree(e->d_sync);
  if (e->d_pack) cudaFree(e->d_pack);
  for (auto &ev : e->fence_ev)
    if (ev) cudaEventDestroy(ev);
  DrainTimers(e);
  for (auto &p : e->pool) {
    cudaEventDestroy(p.a);
    cudaEventDestroy(p.b);
  }
  if (e->own_stream) cudaStreamDestroy(e->st);
  delete e;
}

VP8R_API int vp8r_engine_sync(vp8r_engine *e) {
  if (!e) return VP8R_ERR_INVALID_ARG;
  CU_TRY(SyncParseStreams(e));
  CU_TRY(cudaStreamSynchronize(e->st));
  CU_TRY(cudaStreamSynchronize(e->st_copy));
  for (bool &b : e->copy_busy) b = false;
  for (bool &b : e->kernel_busy) b = false;
  for (auto &sl : e->slots) {
    sl.pending = false;
    HarvestStatus(e, sl, nullptr);
  }
  if (!e->deferred_error.empty()) {
    SetError(e->deferred_error);
    e->deferred_error.clear();
    return VP8R_ERR_TRUNCATED;
  }
  return VP8R_OK;
}

VP8R_API int vp8r_stream_open(vp8r_engine *e, vp8r_stream **out) {
  if (!e || !out) return VP8R_ERR_INVALID_ARG;
  vp8r_stream *s = new (std::nothrow) vp8r_stream();
  if (!s) return VP8R_ERR_NOMEM;
  s->eng = e;
  *out = s;
  return VP8R_OK;
}

VP8R_API void vp8r_stream_close(vp8r_stream *s) {
  if (!s) return;
  cudaSetDevice(s->eng->device);
  SyncParseStreams(s->eng);  // a parse kernel may still use the stream's segment map
  cudaStreamSynchronize(s->eng->st);
  for (auto &sl : s->eng->slots)
    for (auto &p : sl.batch_streams)
      if (p == s) p = nullptr;
  FreeSurfaces(s);
  delete s->own_frame;
  delete s;
}

VP8R_API int vp8r_frame_upload(vp8r_engine *e, vp8r_frame *f) {
  if (!e || !f || !f->blob) return VP8R_ERR_INVALID_ARG;
  int rc = EnsureDevice(e);
  if (rc) return rc;
  f->DropDeviceCopy();
  size_t bytes = f->used_bytes();
  void *p = nullptr;
  cudaError_t err = cudaMalloc(&p, FrameDevExtra(f).total + 64);
  if (err != cudaSuccess) {
    SetError(std::string("cudaMalloc(frame): ") + cudaGetErrorString(err));
    return VP8R_ERR_NOMEM;
  }
  err = cudaMemcpy(p, f->blob, bytes, cudaMemcpyHostToDevice);
  if (err != cudaSuccess) {
    cudaFree(p);
    SetError(std::string("cudaMemcpy(frame): ") + cudaGetErrorString(err));
    return VP8R_ERR_CUDA;
  }
  f->d_blob = p;
  f->d_bytes = bytes;
  f->d_device = e->device;
  // host-side facts the batched submission needs, so that the host arrays may be released
  f->level_counts.clear();
  if (f->hdr.n_intra_levels) {
    const uint32_t *tab = reinterpret_cast<const uint32_t *>(f->payload() + size_t(f->hdr.intra_levels_at) * 16);
    for (uint32_t L = 0; L < f->hdr.n_intra_levels; ++L) f->level_counts.push_back(tab[L + 1] - tab[L]);
  }
  f->n_token_parts = f->hdr.tokens_deferred
                         ? reinterpret_cast<const vp8r_token_hdr *>(f->payload() + size_t(f->hdr.tokens_at) * 16)->n_parts
                         : 0;
  return VP8R_OK;
}

VP8R_API int vp8r_frame_release_host(vp8r_frame *f) {
  if (!f || !f->d_blob) {
    SetError("vp8r_frame_release_host: the frame has no device copy");
    return VP8R_ERR_STATE;
  }
  if (f->blob) vp8r::HostFree(f->blob, f->pinned);
  f->blob = nullptr;
  f->blob_cap = 0;
  return VP8R_OK;
}

VP8R_API int vp8r_reconstruct_batch(vp8r_engine *e, int n, vp8r_stream *const *streams, vp8r_frame *const *frames) {
  if (!e || n < 0 || (n > 0 && (!streams || !frames))) return VP8R_ERR_INVALID_ARG;
  if (n == 0) return VP8R_OK;
  int rc = EnsureDevice(e);
  if (rc) return rc;

  // Pass 1: validate everything before anything is changed (a rejected batch leaves every stream as it was),
  // then configure surfaces and size the staging arena.
  rc = CheckBatchStreams(e, n, streams);
  if (rc) return rc;
  for (int i = 0; i < n; ++i) {
    vp8r_stream *s = streams[i];
    vp8r_frame *f = frames[i];
    if (!f || !(f->blob || (f->d_blob && f->d_device == e->device))) {
      SetError("null frame or frame without arrays on this engine's device");
      return VP8R_ERR_INVALID_ARG;
    }
    const vp8r_frame_hdr &h = f->hdr;
    if (!h.key_frame && (!s->have_frame || h.mb_cols != s->mb_cols || h.mb_rows != s->mb_rows)) {
      SetError("inter frame without matching reference frames");
      return VP8R_ERR_STATE;
    }
  }
  size_t arena = 0;
  for (int i = 0; i < n; ++i) {
    vp8r_stream *s = streams[i];
    vp8r_frame *f = frames[i];
    if (f->hdr.key_frame) {
      rc = ConfigureStream(s, f->hdr);
      if (rc) return rc;
      s->failed = false;
    }
    if (!(f->d_blob && f->d_device == e->device)) arena += FrameDevExtra(f).total;
  }
  int slot_index;
  std::string failure;
  rc = TakeSlot(e, n, arena, &slot_index, &failure);
  if (rc) return rc;
  if (!failure.empty())
    for (int i = 0; i < n; ++i)
      if (streams[i]->failed && !frames[i]->hdr.key_frame) {
        SetError(failure);
        return VP8R_ERR_TRUNCATED;
      }
  Slot &sl = e->slots[slot_index];
  sl.batch_streams.assign(streams, streams + n);
  sl.any_status = false;

  // Pass 2: jobs + host->device staging.
  int max_mbs = 0, max_rows = 0, max_cols = 0, max_cols_all = 0, max_parts = 1;
  bool any_inter = false, any_intra = false, any_wave = false, any_tokens = false, any_modes = false;
  std::vector<int> level_max;  // per dependency level: most intra MBs of that level in any frame
  size_t at = 0, gather_max = 0;
  int n_groups = 0;
  std::vector<int> cur_idx(n);
  // Staging and the parse kernel go to the parse stream when any frame has deferred tokens, so that
  // they overlap the reconstruction kernels of the previous time step on `st`.
  bool deferred = false;
  for (int i = 0; i < n; ++i) deferred |= frames[i]->hdr.tokens_deferred != 0;
  cudaStream_t front = deferred ? e->st_parse[slot_index] : e->st;
  {
    ScopedTimer t(e, Timer::kH2D, front);
    for (int i = 0; i < n; ++i) {
      vp8r_stream *s = streams[i];
      vp8r_frame *f = frames[i];
      const vp8r_frame_hdr &h = f->hdr;
      cur_idx[i] = PickCurrent(s);
      DevFrameJob &j = sl.h_jobs[i];
      std::memset(&j, 0, sizeof(j));
      FillJobSurfaces(s, cur_idx[i], &j);
      const uint8_t *dev_blob;
      if (f->d_blob && f->d_device == e->device) {
        dev_blob = static_cast<const uint8_t *>(f->d_blob);
        if (h.tokens_deferred && f->busy_event && f->busy_engine == e->id)  // its last reconstruction still reads the records
          CU_TRY(cudaStreamWaitEvent(front, static_cast<cudaEvent_t>(f->busy_event), 0));
      } else {
        uint8_t *dst = sl.d_arena + at;
        if (f->pinned) {  // staged by the gather kernel below (SM reads of pinned memory, no copy engine)
          j.h2d_src = f->blob;
          j.h2d_dst = dst;
          j.h2d_bytes = uint32_t(f->used_bytes());
          gather_max = std::max(gather_max, f->used_bytes());
        } else {
          CU_TRY(cudaMemcpyAsync(dst, f->blob, f->used_bytes(), cudaMemcpyHostToDevice, front));
        }
        dev_blob = dst;
        at += FrameDevExtra(f).total;
      }
      j.mbs = reinterpret_cast<const vp8r_mb_info *>(dev_blob);
      j.payload = reinterpret_cast<const int16_t *>(dev_blob + f->mb_bytes());
      const int n_mb = int(h.mb_cols) * h.mb_rows;
      j.n_inter = int(h.n_inter_mbs);
      j.n_intra = n_mb - j.n_inter;
      j.n_intra_levels = int(h.n_intra_levels);
      if (h.n_intra_levels) {
        j.intra_levels = reinterpret_cast<const uint32_t *>(j.payload + size_t(h.intra_levels_at) * 16);
        if (level_max.size() < h.n_intra_levels) level_max.resize(h.n_intra_levels, 0);
        if (f->blob) {
          const uint32_t *tab = reinterpret_cast<const uint32_t *>(f->payload() + size_t(h.intra_levels_at) * 16);
          for (uint32_t L = 0; L < h.n_intra_levels; ++L) level_max[L] = std::max(level_max[L], int(tab[L + 1] - tab[L]));
        } else {  // host arrays released after upload
          for (uint32_t L = 0; L < h.n_intra_levels && L < f->level_counts.size(); ++L)
            level_max[L] = std::max(level_max[L], int(f->level_counts[L]));
        }
      } else if (j.n_intra > 0) {
        any_wave = true;
      }
      if (h.tokens_deferred) {
        // device areas right behind the (256-byte aligned) blob, same allocation, so that block
        // indices relative to `payload` reach them
        const DevExtra x = FrameDevExtra(f);
        uint8_t *wr = const_cast<uint8_t *>(dev_blob);
        j.tok_hdr = reinterpret_cast<const uint8_t *>(j.payload + size_t(h.tokens_at) * 16);
        j.coef_base = uint32_t((x.coef_off - f->mb_bytes()) / 32);
        j.status = sl.d_status_dev + i;
        j.status_host = sl.d_status + i;
        sl.any_status = true;
        any_tokens = true;
        max_cols = std::max(max_cols, int(h.mb_cols));
        max_parts = std::max(max_parts, f->blob ? int(reinterpret_cast<const vp8r_token_hdr *>(f->payload() + size_t(h.tokens_at) * 16)->n_parts)
                                                : int(f->n_token_parts));
        if (h.modes_deferred) {
          j.mode_hdr = reinterpret_cast<const uint8_t *>(j.payload + size_t(h.modes_at) * 16);
          j.mbs = reinterpret_cast<const vp8r_mb_info *>(wr + x.mb_off);
          j.split_base = uint32_t((x.split_off - f->mb_bytes()) / 32);
          j.segment_map = s->d_segmap;
          j.level_table = reinterpret_cast<uint32_t *>(wr + x.level_off);
          j.dyn = reinterpret_cast<vp8r::DevFrameDyn *>(wr + x.dyn_off);
          j.n_inter = h.key_frame ? 0 : n_mb;  // placeholders: the kernels read `dyn`
          j.n_intra = n_mb;
          any_modes = true;
          any_wave = true;
        }
      }
      std::memcpy(j.dq, h.dq, sizeof(j.dq));
      j.key_frame = h.key_frame;
      j.version = h.version;
      j.filter_type = h.filter_type;
      j.lf_level = h.loop_filter_level;
      j.sharpness = h.sharpness_level;
      max_mbs = std::max(max_mbs, n_mb);
      max_rows = std::max(max_rows, int(h.mb_rows));
      max_cols_all = std::max(max_cols_all, int(h.mb_cols));
      any_inter |= j.n_inter > 0;
      any_intra |= j.n_intra > 0;
      e->acc.frames++;
      e->acc.coef_blocks += h.n_coef_blocks;
      e->acc.alg_bytes += uint64_t(n_mb) * 384 * (h.key_frame ? 1 : 2) + uint64_t(h.n_coef_blocks) * 32;
    }
    static_assert(sizeof(DevFrameJob) % 8 == 0, "job table is copied in 16-byte units");
    n_groups = BuildFilterGroups(e, sl, n);
    CU_TRY(vp8r::LaunchCopy(sl.d_jobs, sl.h_jobs, sizeof(DevFrameJob) * n + sizeof(vp8r::FilterGroup) * n_groups, front));
    CU_TRY(vp8r::LaunchGather(sl.d_jobs, n, gather_max, front));
    e->acc.launches_other += 2;
  }

  if (any_tokens) {
    CU_TRY(cudaMemsetAsync(sl.d_status_dev, 0, sizeof(int) * n, front));
    ScopedTimer t(e, Timer::kTokens, front);
    if (any_modes) {
      // K_modes here, K_segments in batch order on its own stream, then back (see token_kernel.cu)
      CU_TRY(vp8r::LaunchModes(sl.d_jobs, n, max_cols, max_mbs, front));
      CU_TRY(cudaEventRecord(sl.modes_done, front));
      CU_TRY(cudaStreamWaitEvent(e->st_segments, sl.modes_done, 0));
      CU_TRY(vp8r::LaunchSegments(sl.d_jobs, n, max_mbs, e->st_segments));
      CU_TRY(cudaEventRecord(sl.segments_done, e->st_segments));
      CU_TRY(cudaStreamWaitEvent(front, sl.segments_done, 0));
      e->acc.launches_other += 2;
    }
    CU_TRY(vp8r::LaunchTokens(sl.d_jobs, n, max_cols, max_parts, front));
    e->acc.launches_other++;
  }
  if (front != e->st) {
    CU_TRY(cudaEventRecord(sl.parsed, front));
    CU_TRY(cudaStreamWaitEvent(e->st, sl.parsed, 0));
  }
  if (any_inter) {
    ScopedTimer t(e, Timer::kInter);
    CU_TRY(vp8r::LaunchInter(sl.d_jobs, n, max_cols_all, max_rows, e->st));
    e->acc.launches_inter++;
  }
  if (any_intra) {
    ScopedTimer t(e, Timer::kIntra);
    for (size_t L = 0; L < level_max.size(); ++L) {
      CU_TRY(vp8r::LaunchIntraFlat(sl.d_jobs, n, int(L), level_max[L], e->st));
      e->acc.launches_intra++;
    }
    if (any_modes) {
      CU_TRY(vp8r::LaunchIntraLevels(sl.d_jobs, n, e->st));
      e->acc.launches_intra++;
    }
    if (any_wave) {
      CU_TRY(vp8r::LaunchIntra(sl.d_jobs, n, max_rows, e->st));
      e->acc.launches_intra++;
    }
  }
  rc = LaunchFilterAndBorder(e, sl, n, max_rows, n_groups);
  if (rc) return rc;
  CU_TRY(cudaEventRecord(sl.done, e->st));
  sl.pending = true;
  for (int i = 0; i < n; ++i)
    if (frames[i]->d_blob && frames[i]->hdr.tokens_deferred) {
      frames[i]->busy_event = sl.done;
      frames[i]->busy_engine = e->id;
    }
  for (int i = 0; i < n; ++i) RefreshRefs(streams[i], frames[i]->hdr, cur_idx[i]);
  return VP8R_OK;
}

// Row f4: closed-loop key-frame encoder.
VP8R_API int vp8r_encode_key_frames(vp8r_engine *e, int n, vp8r_stream *const *streams, const uint8_t *const *i420, int width,
                                    int height, int q_index, int loop_filter_level, int sharpness, unsigned flags, vp8r_frame *const *out) {
  EncoderSource src;
  src.host = i420;
  return EncodeKeyFrames(e, n, streams, src, width, height, q_index, loop_filter_level, sharpness, flags, out);
}

VP8R_API int vp8r_encode_key_frames_device(vp8r_engine *e, int n, vp8r_stream *const *streams, const void *src, size_t stride,
                                           int layout, void *producer_stream, int width, int height, int q_index,
                                           int loop_filter_level, int sharpness, unsigned flags, vp8r_frame *const *out) {
  EncoderSource s;
  s.dev = static_cast<const uint8_t *>(src);
  s.stride = stride;
  s.layout = layout;
  s.producer = static_cast<cudaStream_t>(producer_stream);
  return EncodeKeyFrames(e, n, streams, s, width, height, q_index, loop_filter_level, sharpness, flags, out);
}

VP8R_API int vp8r_encode_inter_frames(vp8r_engine *e, int n, vp8r_stream *const *streams, const uint8_t *const *i420,
                                      int width, int height, int q_index, int loop_filter_level, int sharpness,
                                      int search_range, vp8r_frame *const *out) {
  EncoderSource src;
  src.host = i420;
  return EncodeInterFrames(e, n, streams, src, width, height, q_index, loop_filter_level, sharpness, search_range, 0u, out);
}

VP8R_API int vp8r_encode_inter_frames_ex(vp8r_engine *e, int n, vp8r_stream *const *streams, const uint8_t *const *i420,
                                         int width, int height, int q_index, int loop_filter_level, int sharpness,
                                         int search_range, unsigned flags, vp8r_frame *const *out) {
  EncoderSource src;
  src.host = i420;
  return EncodeInterFrames(e, n, streams, src, width, height, q_index, loop_filter_level, sharpness, search_range, flags, out);
}

VP8R_API int vp8r_encode_inter_frames_device(vp8r_engine *e, int n, vp8r_stream *const *streams, const void *src, size_t stride,
                                             int layout, void *producer_stream, int width, int height, int q_index,
                                             int loop_filter_level, int sharpness, int search_range, vp8r_frame *const *out) {
  EncoderSource s;
  s.dev = static_cast<const uint8_t *>(src);
  s.stride = stride;
  s.layout = layout;
  s.producer = static_cast<cudaStream_t>(producer_stream);
  return EncodeInterFrames(e, n, streams, s, width, height, q_index, loop_filter_level, sharpness, search_range, 0u, out);
}

VP8R_API int vp8r_encode_inter_frames_device_ex(vp8r_engine *e, int n, vp8r_stream *const *streams, const void *src,
                                                size_t stride, int layout, void *producer_stream, int width, int height,
                                                int q_index, int loop_filter_level, int sharpness, int search_range,
                                                unsigned flags, vp8r_frame *const *out) {
  EncoderSource s;
  s.dev = static_cast<const uint8_t *>(src);
  s.stride = stride;
  s.layout = layout;
  s.producer = static_cast<cudaStream_t>(producer_stream);
  return EncodeInterFrames(e, n, streams, s, width, height, q_index, loop_filter_level, sharpness, search_range, flags, out);
}

VP8R_API int vp8r_convert_to_i420_device(vp8r_engine *e, int n, const void *src, size_t src_stride, int layout, int width,
                                         int height, void *dst, size_t dst_stride, void *stream) {
  // argument checks that need no device come first
  const std::string call = "vp8r_convert_to_i420_device";
  if (!e || !src || !dst) {
    SetError(call + ": null engine, src or dst");
    return VP8R_ERR_INVALID_ARG;
  }
  if (n <= 0) {
    SetError(call + ": n <= 0");
    return VP8R_ERR_INVALID_ARG;
  }
  int rc = CheckLayoutAndSize(call, layout, width, height);
  if (!rc) rc = CheckStride(call + ": stride", src_stride, layout, width, height);
  if (!rc) rc = CheckStride(call + ": dst_stride", dst_stride, VP8R_LAYOUT_I420, width, height);
  if (!rc) rc = EnsureDevice(e);
  if (rc) return rc;
  if (!IsEngineDeviceMemory(e, src) || !IsEngineDeviceMemory(e, dst)) {
    SetError(call + ": src or dst is not device memory of the engine's device (pinned, pageable and managed memory are "
                    "refused)");
    return VP8R_ERR_INVALID_ARG;
  }
  const size_t cw = size_t(width + 1) / 2, ch = size_t(height + 1) / 2;
  int part;
  // the source is written, and earlier work may still read dst, on the caller's stream
  return RunOutputJobs(
      e, n, Timer::kNone, static_cast<cudaStream_t>(stream), &part,
      [&](int i, DevFrameJob &j) {
        uint8_t *d = static_cast<uint8_t *>(dst) + size_t(i) * dst_stride;
        j.stage_src = static_cast<const uint8_t *>(src) + size_t(i) * src_stride;
        j.pack_layout = uint8_t(layout);
        j.width = j.stage_w = width;
        j.height = j.stage_h = height;
        j.enc_src[0] = d;
        j.enc_src[1] = d + size_t(width) * height;
        j.enc_src[2] = j.enc_src[1] + cw * ch;
        j.enc_src_pitch_y = width;
        j.enc_src_pitch_c = int(cw);
      },
      [&](DevFrameJob *dj) { return vp8r::LaunchStageSource(dj, n, layout, width, height, e->st); });
}

VP8R_API size_t vp8r_stream_frame_bytes(const vp8r_stream *s) {
  if (!s || !s->have_frame) return 0;
  return LayoutBytes(VP8R_LAYOUT_I420, s->width, s->height);
}

VP8R_API int vp8r_stream_dims(const vp8r_stream *s, int *width, int *height) {
  if (!s || !s->have_frame) return VP8R_ERR_STATE;
  if (width) *width = s->width;
  if (height) *height = s->height;
  return VP8R_OK;
}

VP8R_API int vp8r_read_batch(vp8r_engine *e, int n, vp8r_stream *const *streams, uint8_t *const *dst,
                             const size_t *cap, int async) {
  if (!e || n < 0 || (n > 0 && (!streams || !dst))) return VP8R_ERR_INVALID_ARG;
  int rc = EnsureDevice(e);
  if (!rc) rc = CheckFrameStreams(e, n, streams);
  if (rc) return rc;
  {
    ScopedTimer t(e, Timer::kD2H);
    for (int i = 0; i < n; ++i) {
      const vp8r_stream *s = streams[i];
      if (!dst[i]) {
        SetError("null destination");
        return VP8R_ERR_STATE;
      }
      const size_t need = vp8r_stream_frame_bytes(s);
      if (cap && cap[i] < need) {
        SetError("destination buffer too small");
        return VP8R_ERR_INVALID_ARG;
      }
      // src/yuv.cc:6-28: crop to width x height, chroma ceil(w/2) x ceil(h/2), planes Y,U,V.
      const vp8r::DevPlanes &p = s->surf[s->ref[0]].planes;
      const size_t w = s->width, h = s->height, cw = (w + 1) / 2, ch = (h + 1) / 2;
      uint8_t *o = dst[i];
      CU_TRY(cudaMemcpy2DAsync(o, w, p.y, s->pitch_y, w, h, cudaMemcpyDeviceToHost, e->st));
      CU_TRY(cudaMemcpy2DAsync(o + w * h, cw, p.u, s->pitch_c, cw, ch, cudaMemcpyDeviceToHost, e->st));
      CU_TRY(cudaMemcpy2DAsync(o + w * h + cw * ch, cw, p.v, s->pitch_c, cw, ch, cudaMemcpyDeviceToHost, e->st));
    }
  }
  if (!async) CU_TRY(cudaStreamSynchronize(e->st));
  return VP8R_OK;
}

VP8R_API int vp8r_read_batch_packed(vp8r_engine *e, int n, vp8r_stream *const *streams, uint8_t *dst, size_t stride,
                                    int async) {
  return vp8r_read_batch_packed_as(e, n, streams, dst, stride, async, VP8R_LAYOUT_I420);
}

VP8R_API int vp8r_read_batch_packed_as(vp8r_engine *e, int n, vp8r_stream *const *streams, uint8_t *dst, size_t stride,
                                       int async, int layout) {
  if (!e || n <= 0 || !streams || !dst || (layout != VP8R_LAYOUT_I420 && layout != VP8R_LAYOUT_NV12)) return VP8R_ERR_INVALID_ARG;
  int rc = EnsureDevice(e);
  if (!rc) rc = CheckFrameStreams(e, n, streams, stride, layout);
  if (rc) return rc;
  const size_t bytes = size_t(n) * stride;
  if (bytes > e->pack_cap) {
    CU_TRY(cudaStreamSynchronize(e->st));
    CU_TRY(cudaStreamSynchronize(e->st_copy));
    for (bool &b : e->copy_busy) b = false;
    for (bool &b : e->kernel_busy) b = false;
    const size_t half = (bytes + 255) & ~size_t(255);
    CU_TRY(Regrow(&e->pack_cap, half, {DeviceBuf(&e->d_pack, vp8r_engine::kPackBufs * half + 256)}));
  }
  // kPackBufs parts of the job table and of the staging buffer rotate: the pack kernel of this call
  // runs on the engine's stream while the D2H copy of the previous call may still be in flight on
  // the copy stream.
  int part = 0;
  rc = RunOutputJobs(
      e, n, Timer::kD2H, nullptr, &part,
      [&](int i, DevFrameJob &j) {
        FillJobSurfaces(streams[i], streams[i]->ref[0], &j);
        j.pack_dst = e->d_pack + size_t(part) * e->pack_cap + size_t(i) * stride;
        j.pack_layout = uint8_t(layout);
      },
      [&](DevFrameJob *dj) { return vp8r::LaunchPack(dj, n, e->st); });
  if (rc) return rc;
  CU_TRY(cudaStreamWaitEvent(e->st_copy, e->pack_done[part], 0));
  CU_TRY(cudaMemcpyAsync(dst, e->d_pack + size_t(part) * e->pack_cap, bytes, cudaMemcpyDeviceToHost, e->st_copy));
  CU_TRY(cudaEventRecord(e->copy_done[part], e->st_copy));
  e->copy_busy[part] = true;
  if (!async) {
    CU_TRY(cudaStreamSynchronize(e->st_copy));
    e->copy_busy[part] = false;
  }
  return VP8R_OK;
}

VP8R_API int vp8r_read_batch_device(vp8r_engine *e, int n, vp8r_stream *const *streams, void *dst, size_t stride,
                                    int layout, void *consumer_stream) {
  // argument checks that need no device come first
  const std::string call = "vp8r_read_batch_device";
  if (!e || !streams || !dst) {
    SetError(call + ": null engine, streams or destination");
    return VP8R_ERR_INVALID_ARG;
  }
  if (n <= 0) {
    SetError(call + ": n <= 0");
    return VP8R_ERR_INVALID_ARG;
  }
  int rc = CheckLayoutAndSize(call, layout, 1, 1);  // the frames' sizes are the streams', checked as they were parsed
  if (!rc) rc = CheckFrameStreams(e, n, streams, stride, layout);
  if (!rc) rc = EnsureDevice(e);
  if (rc) return rc;
  if (!IsEngineDeviceMemory(e, dst)) {
    SetError(call + ": dst is not device memory of the engine's device (pinned, pageable and managed memory are refused)");
    return VP8R_ERR_INVALID_ARG;
  }
  const bool rgb = layout == VP8R_LAYOUT_RGB24 || layout == VP8R_LAYOUT_RGB_PLANAR;
  int max_w = 0, max_h = 0, part;
  // earlier consumer work may still read dst
  return RunOutputJobs(
      e, n, Timer::kNone, static_cast<cudaStream_t>(consumer_stream), &part,
      [&](int i, DevFrameJob &j) {
        FillJobSurfaces(streams[i], streams[i]->ref[0], &j);
        j.pack_dst = static_cast<uint8_t *>(dst) + size_t(i) * stride;
        j.pack_layout = uint8_t(layout);
        max_w = std::max(max_w, j.width);
        max_h = std::max(max_h, j.height);
      },
      [&](DevFrameJob *dj) {
        return rgb ? vp8r::LaunchConvertRgb(dj, n, max_w, max_h, e->st) : vp8r::LaunchPack(dj, n, e->st);
      });
}

VP8R_API int vp8r_stream_read_frame(vp8r_stream *s, uint8_t *dst, size_t cap) {
  if (!s) return VP8R_ERR_INVALID_ARG;
  vp8r_stream *ss[1] = {s};
  uint8_t *dd[1] = {dst};
  size_t cc[1] = {cap};
  return vp8r_read_batch(s->eng, 1, ss, dd, cc, 0);
}

VP8R_API int vp8r_checksum_batch(vp8r_engine *e, int n, vp8r_stream *const *streams, uint64_t *out) {
  if (!e || n <= 0 || !streams || !out) return VP8R_ERR_INVALID_ARG;
  int rc = EnsureDevice(e);
  if (!rc) rc = CheckFrameStreams(e, n, streams);
  int part;
  if (!rc)
    rc = RunOutputJobs(
        e, n, Timer::kNone, nullptr, &part,
        [&](int i, DevFrameJob &j) {
          FillJobSurfaces(streams[i], streams[i]->ref[0], &j);
          j.checksum = e->d_sums + i;
        },
        [&](DevFrameJob *dj) {
          const cudaError_t err = cudaMemsetAsync(e->d_sums, 0, sizeof(uint64_t) * n, e->st);
          return err != cudaSuccess ? err : vp8r::LaunchChecksum(dj, n, e->st);
        });
  if (rc) return rc;
  // the checksum words are the engine's, not a part's: each call waits for its own
  CU_TRY(cudaMemcpyAsync(e->h_sums, e->d_sums, sizeof(uint64_t) * n, cudaMemcpyDeviceToHost, e->st));
  CU_TRY(cudaStreamSynchronize(e->st));
  for (int i = 0; i < n; ++i) out[i] = e->h_sums[i];
  return VP8R_OK;
}

VP8R_API int vp8r_stream_checksum(vp8r_stream *s, uint64_t *out) {
  if (!s) return VP8R_ERR_INVALID_ARG;
  vp8r_stream *ss[1] = {s};
  return vp8r_checksum_batch(s->eng, 1, ss, out);
}

VP8R_API int vp8r_stream_decode(vp8r_stream *s, const uint8_t *data, size_t size, int *shown) {
  if (!s || !data) return VP8R_ERR_INVALID_ARG;
  if (!s->own_frame) {
    s->own_frame = new (std::nothrow) vp8r_frame();
    if (!s->own_frame) return VP8R_ERR_NOMEM;
    s->own_frame->pinned = true;
  }
  // The staging copy of the previous call must have left the pinned blob before it is rewritten.
  int rc = vp8r_engine_sync(s->eng);
  if (rc) return rc;
  rc = s->parser.Parse(data, size, s->own_frame);
  if (rc) {
    SetError(s->parser.error());
    return rc;
  }
  if (shown) *shown = s->own_frame->hdr.show_frame;
  vp8r_stream *ss[1] = {s};
  vp8r_frame *ff[1] = {s->own_frame};
  return vp8r_reconstruct_batch(s->eng, 1, ss, ff);
}

VP8R_API int vp8r_engine_fence(vp8r_engine *e, uint64_t *ticket) {
  if (!e || !ticket) return VP8R_ERR_INVALID_ARG;
  int rc = EnsureDevice(e);
  if (rc) return rc;
  const uint64_t t = e->fence_head++;
  cudaEvent_t &ev = e->fence_ev[t & 15];
  if (!ev) CU_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  CU_TRY(cudaEventRecord(ev, e->st));
  // ... and everything queued on the copy stream (asynchronous packed read-backs)
  e->fence_has_copy[t & 15] = false;
  for (bool b : e->copy_busy) e->fence_has_copy[t & 15] |= b;
  if (e->fence_has_copy[t & 15]) {
    cudaEvent_t &cev = e->fence_copy_ev[t & 15];
    if (!cev) CU_TRY(cudaEventCreateWithFlags(&cev, cudaEventDisableTiming));
    CU_TRY(cudaEventRecord(cev, e->st_copy));
  }
  *ticket = t;
  return VP8R_OK;
}

VP8R_API int vp8r_engine_wait(vp8r_engine *e, uint64_t ticket) {
  if (!e) return VP8R_ERR_INVALID_ARG;
  if (ticket >= e->fence_head) {
    SetError("unknown fence ticket");
    return VP8R_ERR_INVALID_ARG;
  }
  // A recycled slot holds a LATER fence of the same streams: waiting for that one covers the old ticket too.
  CU_TRY(cudaEventSynchronize(e->fence_ev[ticket & 15]));
  if (e->fence_has_copy[ticket & 15]) CU_TRY(cudaEventSynchronize(e->fence_copy_ev[ticket & 15]));
  return VP8R_OK;
}

VP8R_API int vp8r_engine_set_timing(vp8r_engine *e, int enabled) {
  if (!e) return VP8R_ERR_INVALID_ARG;
  e->timing = enabled != 0;
  return VP8R_OK;
}

VP8R_API int vp8r_engine_get_timers(vp8r_engine *e, vp8r_timers *out, int reset) {
  if (!e || !out) return VP8R_ERR_INVALID_ARG;
  int rc = vp8r_engine_sync(e);
  if (rc) return rc;
  DrainTimers(e);
  *out = e->acc;
  if (reset) e->acc = vp8r_timers{};
  return VP8R_OK;
}

}  // extern "C"
