// Host-only part of the C ABI: parser, parsed-frame objects, checksums, error reporting.
// (The engine half lives in rt/engine.cu.)
#include <atomic>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <cstring>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "host/frame_parser.h"
#include "host/frame_writer.h"
#include "host/parsed_frame.h"
#include "rt/error.h"
#include "vp8r.h"

namespace vp8r {
namespace {
thread_local std::string g_error;
}
void SetError(const std::string &msg) { g_error = msg; }
const char *LastError() { return g_error.c_str(); }
}  // namespace vp8r

extern "C" {

VP8R_API const char *vp8r_last_error(void) { return vp8r::LastError(); }
VP8R_API const char *vp8r_version(void) { return "vp8r 0.1 (sm_100a)"; }

VP8R_API vp8r_parser *vp8r_parser_create(void) { return new (std::nothrow) vp8r_parser(); }
VP8R_API void vp8r_parser_destroy(vp8r_parser *p) { delete p; }
VP8R_API void vp8r_parser_reset(vp8r_parser *p) {
  if (p) p->impl.Reset();
}

VP8R_API void vp8r_parser_set_defer_tokens(vp8r_parser *p, int on) {
  if (p) p->impl.set_defer_tokens(on != 0);
}

VP8R_API void vp8r_parser_set_defer_modes(vp8r_parser *p, int on) {
  if (p) p->impl.set_defer_modes(on != 0);
}

VP8R_API vp8r_frame *vp8r_frame_create(int pinned) {
  vp8r_frame *f = new (std::nothrow) vp8r_frame();
  if (f) f->pinned = pinned != 0;
  return f;
}
VP8R_API void vp8r_frame_destroy(vp8r_frame *f) { delete f; }

VP8R_API int vp8r_frame_get_desc(const vp8r_frame *f, vp8r_frame_desc *out) {
  if (!f || !out || !f->blob) return VP8R_ERR_INVALID_ARG;
  out->hdr = f->hdr;
  out->mbs = f->mbs();
  out->payload = f->payload();
  return VP8R_OK;
}

VP8R_API int vp8r_parser_parse(vp8r_parser *p, const uint8_t *data, size_t size, vp8r_frame *out) {
  if (!p || !out) return VP8R_ERR_INVALID_ARG;
  int rc = p->impl.Parse(data, size, out);
  if (rc != VP8R_OK) vp8r::SetError(p->impl.error());
  return rc;
}

namespace {
// Worker threads of vp8r_parse_batch, kept between calls (a batch decoder calls it once per time step; creating
// and joining threads every call showed up in the host time of the end-to-end pass).  One job at a time; the
// calling thread works too.
class ParsePool {
 public:
  static ParsePool &Get() {
    static ParsePool *pool = new ParsePool();  // never destroyed: worker threads may outlive static destructors
    return *pool;
  }
  // Runs work(tid) on `n_threads` threads (tid 0 = the caller) and returns when all are done.
  void Run(int n_threads, const std::function<void(int)> &work) {
    std::lock_guard<std::mutex> serial(run_mutex_);
    {
      std::unique_lock<std::mutex> lk(m_);
      while (int(threads_.size()) < n_threads - 1) {
        const int tid = int(threads_.size()) + 1;
        threads_.emplace_back([this, tid] { Loop(tid); });
        threads_.back().detach();
      }
      work_ = &work;
      want_ = n_threads - 1;
      pending_ = n_threads - 1;
      ++generation_;
    }
    cv_.notify_all();
    work(0);
    std::unique_lock<std::mutex> lk(m_);
    done_cv_.wait(lk, [this] { return pending_ == 0; });
    work_ = nullptr;
  }

 private:
  void Loop(int tid) {
    uint64_t seen = 0;
    for (;;) {
      const std::function<void(int)> *w = nullptr;
      {
        std::unique_lock<std::mutex> lk(m_);
        cv_.wait(lk, [&] { return generation_ != seen; });
        seen = generation_;
        if (tid <= want_) w = work_;
      }
      if (w) {
        (*w)(tid);
        std::unique_lock<std::mutex> lk(m_);
        if (--pending_ == 0) done_cv_.notify_one();
      }
    }
  }
  std::mutex run_mutex_, m_;
  std::condition_variable cv_, done_cv_;
  std::vector<std::thread> threads_;
  const std::function<void(int)> *work_ = nullptr;
  int want_ = 0, pending_ = 0;
  uint64_t generation_ = 0;
};
}  // namespace

// Parses n frames of n DIFFERENT streams concurrently (one parser per stream; the bool decoder is
// serial within a stream, so stream-level parallelism is what the host has).
VP8R_API int vp8r_parse_batch(int n, vp8r_parser *const *parsers, const uint8_t *const *data, const size_t *sizes,
                              vp8r_frame *const *out, int n_threads, int *status) {
  if (n < 0 || (n > 0 && (!parsers || !data || !sizes || !out))) return VP8R_ERR_INVALID_ARG;
  if (n_threads < 1) n_threads = 1;
  if (n_threads > n) n_threads = n;
  std::atomic<int> next(0), first_err(VP8R_OK);
  std::vector<std::string> errs(static_cast<size_t>(n_threads));
  auto work = [&](int tid) {
    for (;;) {
      int i = next.fetch_add(1);
      if (i >= n) break;
      int rc = (parsers[i] && out[i]) ? parsers[i]->impl.Parse(data[i], sizes[i], out[i]) : VP8R_ERR_INVALID_ARG;
      if (status) status[i] = rc;
      if (rc != VP8R_OK) {
        int expected = VP8R_OK;
        if (first_err.compare_exchange_strong(expected, rc)) errs[size_t(tid)] = parsers[i] ? parsers[i]->impl.error() : "null";
      }
    }
  };
  if (n_threads <= 1) work(0);
  else ParsePool::Get().Run(n_threads, work);
  if (first_err.load() != VP8R_OK)
    for (auto &e : errs)
      if (!e.empty()) vp8r::SetError(e);
  return first_err.load();
}

VP8R_API int vp8r_frame_write_bitstream(const vp8r_frame *f, uint8_t *dst, size_t cap, size_t *size) {
  return vp8r_frame_write_bitstream_in(f, nullptr, dst, cap, size);
}

VP8R_API int vp8r_frame_write_bitstream_in(const vp8r_frame *f, const vp8r_parser *context, uint8_t *dst, size_t cap,
                                           size_t *size) {
  if (!f || !size) return VP8R_ERR_INVALID_ARG;
  std::vector<uint8_t> bytes;
  std::string err;
  const int rc = vp8r::WriteFrame(*f, context ? &context->impl : nullptr, &bytes, &err);
  if (rc != VP8R_OK) {
    vp8r::SetError(err);
    return rc;
  }
  *size = bytes.size();
  if (!dst || cap < bytes.size()) {
    vp8r::SetError("vp8r_frame_write_bitstream: destination too small");
    return VP8R_ERR_INVALID_ARG;
  }
  std::memcpy(dst, bytes.data(), bytes.size());
  return VP8R_OK;
}

VP8R_API int vp8r_is_key_frame(const uint8_t *data, size_t size) {
  return (data && size >= 1) ? !(data[0] & 1) : 0;
}

// s1 = sum(b_i), s2 = sum((i+1) * b_i), both mod 2^32, over the cropped Y,U,V byte stream.
VP8R_API uint64_t vp8r_checksum_i420(const uint8_t *i420, int width, int height) {
  if (!i420 || width <= 0 || height <= 0) return 0;
  const size_t cw = size_t(width + 1) / 2, ch = size_t(height + 1) / 2;
  const size_t total = size_t(width) * height + 2 * cw * ch;
  uint32_t s1 = 0, s2 = 0;
  for (size_t i = 0; i < total; ++i) {
    s1 += i420[i];
    s2 += uint32_t(i + 1) * i420[i];
  }
  return (uint64_t(s2) << 32) | s1;
}

}  // extern "C"
