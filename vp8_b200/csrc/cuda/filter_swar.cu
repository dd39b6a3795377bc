// K_filter, batch form: the VP8 loop filter (src/filter.cc:7-340 of the reference) with FOUR pixel lines per
// register (lf_swar.h) and EIGHT frames per warp.
//
// The scalar wavefront kernel in recon_kernels.cu gives every pixel line of a macroblock row a lane and pays
// one instruction per pixel line and tap.  Here a lane owns four lines: a warp is eight frames x four lanes,
// all at the same macroblock (r, c) of their own frame, so the 32 lanes never wait for each other's data
// (frames are independent streams) and the row-to-row hand-over stays one flag per warp as before.
//
//   luma CTA:   lane (slot, u): vertical edges on rows 4u..4u+3 of the macroblock (words = one pixel column
//               of four rows), then horizontal edges on columns 4u..4u+3 (words = one pixel row of four
//               columns).  The 4x4 byte blocks are turned with PRMT (8 per block) and change lanes through
//               a per-slot shared-memory tile (128-bit, bank-conflict free).
//   chroma CTA: lane (slot, plane, h): the same on the two 8x8 blocks, rows / columns 4h..4h+3.
//
// Per macroblock step: rows come in with 128-bit loads (prefetched one macroblock ahead); finished words go
// into a per-warp shared-memory ring and leave it as whole 32-byte units with 128-bit stores every second
// step (SwarRing below); the last four columns of a macroblock travel to the next step in registers (they
// are filtered again by its left edge) and enter the ring from there.
//
// Measured (B200, 512 1080p frames per launch): 2.61 ms against 4.11 ms of the scalar kernel; ~1350 warp
// instructions per step of 8 macroblocks (luma) + ~750 (chroma) = ~260 per macroblock against 796.
#include "lf_swar.h"
#include "recon_kernels.h"

namespace vp8r {

namespace {


struct SwarLimits {
  int interior, hev, edge_mb, edge_sb;
};

// src/filter.cc:119-149
__device__ __forceinline__ swar::EdgeK EdgeKFor(unsigned flags, int sharp, bool key) {
  const int level = (flags >> VP8R_MB_LF_SHIFT) & 63;
  int in = level;
  if (sharp) {
    in >>= (sharp > 4) ? 2 : 1;
    in = min(in, 9 - sharp);
  }
  const int interior = max(in, 1);
  int hev;
  if (key) hev = level >= 40 ? 2 : (level >= 15 ? 1 : 0);
  else hev = level >= 40 ? 3 : (level >= 20 ? 2 : (level >= 15 ? 1 : 0));
  swar::EdgeK k;
  k.k_int = swar::X2((127 - interior) << 8);
  k.k_hev = swar::X2((127 - hev) << 8);
  // 0x7fff - (2E + 1), E = (level + 2) * 2 + interior resp. level * 2 + interior
  k.k_mb = level ? swar::X2(0x7fff - 9 - 4 * level - 2 * interior) : 0x80008000u;
  k.k_sb = (level && (flags & VP8R_MB_LF_INNER)) ? swar::X2(0x7fff - 1 - 4 * level - 2 * interior) : 0x80008000u;
  return k;
}

// All edges of one direction of a macroblock: W[0..3] = the four lines' pixels before the macroblock edge
// (previous macroblock / rows above), W[4..] = the macroblock.
template <int NB>
__device__ __forceinline__ void FilterEdgesSwar(uint32_t (&W)[4 + 4 * NB], const swar::EdgeK &k, bool mb_edge, bool any_inner,
                                                bool simple) {
  if (!simple) {
    if (mb_edge) swar::NormalMbEdge(W[0], W[1], W[2], W[3], W[4], W[5], W[6], W[7], k);
    if (any_inner) {
#pragma unroll
      for (int e = 1; e < NB; ++e)
        swar::NormalInner(W[4 * e], W[4 * e + 1], W[4 * e + 2], W[4 * e + 3], W[4 * e + 4], W[4 * e + 5], W[4 * e + 6],
                          W[4 * e + 7], k);
    }
  } else {
    if (mb_edge) swar::SimpleEdge(W[2], W[3], W[4], W[5], k.k_mb);
    if (any_inner) {
#pragma unroll
      for (int e = 1; e < NB; ++e) swar::SimpleEdge(W[4 * e + 2], W[4 * e + 3], W[4 * e + 4], W[4 * e + 5], k.k_sb);
    }
  }
}

template <int NB>
__device__ __forceinline__ void LoadRowWords(const uint8_t *p, uint32_t (&w)[NB]) {
  if (NB == 4) {
    const uint4 t = *reinterpret_cast<const uint4 *>(p);
    w[0] = t.x; w[1] = t.y; w[2] = t.z; w[3] = t.w;
  } else {
    const uint2 t = *reinterpret_cast<const uint2 *>(p);
    w[0] = t.x; w[1] = t.y;
  }
}

__device__ __forceinline__ int LoadFlagAcquireSwar(const int *p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// A waiting row sleeps kSwarSleepBase + kSwarSleepSlope * (macroblocks still missing - 1) ns, at most kSwarSleepMax;
// the last row of a band publishes its progress device-wide at every kSwarBandStride-th flush.
constexpr int kSwarSleepBase = 400, kSwarSleepSlope = 1500, kSwarSleepMax = 40000;
constexpr int kSwarBandStride = 4;
// CTA shape: kSwarWarps warps = macroblock rows per band, one CTA per SM.  Measured at 512 1080p frames per launch
// (profiles/r2_filter_swar.md): 12 x 1 = 2.61 ms, 10 x 1 = 2.67, 8 x 1 = 2.72, 6 x 2 = 2.77, 16 x 1 = 3.66,
// 17 x 1 = 3.99, 4 x 5 = 4.19 (the scalar kernel: 4.11).  More resident warps lose: 12.5 KB of shared memory
// per warp leave little L1 for the row loads (each 32-byte sector is read in two consecutive steps).
constexpr int kSwarWarps = 12;

// Output staging.  Finished pixel rows do not go to global memory word by word (a warp-wide 32-bit store of
// this kernel touches 8..32 different sectors, and every hand-over fence has to wait for all of them): the
// lanes drop their words into a per-warp shared-memory ring and the warp writes whole flush units (two
// macroblocks of a pixel row: 32 bytes of luma, 16 of chroma) with 128-bit stores every second step.
// Ring rows of a slot: per plane 3 rows above the macroblock row + its own rows; a ring row holds four
// macroblocks; its 16-byte chunks are swizzled by the row so that neither the word writes nor the 128-bit
// flush reads collide on banks.
template <int NB>
struct SwarRing {
  static constexpr int kN = 4 * NB;
  static constexpr int kG = 2;                               // macroblocks per flush unit
  static constexpr int kRingMbs = 2 * kG;                    // macroblocks per ring row
  static constexpr int kRowBytes = kRingMbs * kN;            // 64 / 32
  static constexpr int kPlanes = NB == 4 ? 1 : 2;
  static constexpr int kR = 3 + kN;                          // ring rows per plane
  static constexpr int kSlotBytes = kPlanes * kR * kRowBytes + 16;  // 1232 / 720: slot stride = 20 words (mod 32)
  static constexpr int kUnit = kG * kN;                      // bytes per flush unit
  static constexpr int kHalves = kUnit / 16;                 // 16-byte stores per unit
  static constexpr int kSwzXor = NB == 4 ? 2 : 1;            // chunk index ^= kSwzXor on swizzled rows
  __host__ __device__ static constexpr bool Swz(int k) { return NB == 4 ? ((k & 2) != 0) : (((k >> 2) & 1) != 0); }  // k: row inside the plane
};
constexpr int kSwarRingBytes = 8 * SwarRing<4>::kSlotBytes;  // per warp; the luma ring is the larger one
constexpr int kSwarTileBytes = 8 * 20 * 16;                  // per warp; exchange tiles (luma: 8 slots x 4 regions x 5 chunks)
constexpr int kSwarPtrBytes = 8 * 2 * 8;                     // per warp; plane pointers of the 8 slots

// One band (rows r0..r1-1 of the group's frames) of one plane kind.  NB = 4x4 blocks per macroblock side:
// 4 for luma, 2 for chroma.
template <int NB>
__device__ __forceinline__ void FilterBandSwar(const DevFrameJob *__restrict__ jobs, const FilterGroup &grp, int band, int n_bands,
                                               int *gflag, volatile int *lprog, uint4 *tiles, unsigned char *rings,
                                               unsigned long long *ptrs) {
  using Ring = SwarRing<NB>;
  constexpr int kN = 4 * NB;            // macroblock size in this plane
  constexpr int kRegion = NB + 1;       // 16-byte chunks between the regions of a slot (one pad chunk)
  constexpr int kSlot = 4 * kRegion;    // chunks per slot; = 4 (mod 8) so that two slots never share a bank group
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;  // from lane 0: known to be warp-uniform
  const int slot = lane >> 2, u = lane & 3;
  const int pl = NB == 4 ? 0 : (u >> 1);   // chroma: 0 = U, 1 = V
  const int sub = NB == 4 ? u : (u & 1);   // row group (vertical edges) / column group (horizontal edges)
  const int fidx = grp.frame[slot];
  const bool active = fidx >= 0 && !JobFailed(jobs[fidx]);  // a failed frame rides along like an idle slot
  // idle slots shadow slot 0 (its loads are in range whatever its records say: they only address its own planes) and store nothing
  const DevFrameJob &job = jobs[active ? fidx : grp.frame[0]];
  // geometry and filter type are the same for every frame of a group
  const int rows = job.mb_rows, cols = job.mb_cols;
  const bool simple = job.filter_type != 0;
  const int sharpness = job.sharpness;
  const bool key_frame = job.key_frame != 0;
  const vp8r_mb_info *const mbs = job.mbs;
  uint8_t *const plane = NB == 4 ? job.cur.y : (pl ? job.cur.v : job.cur.u);
  const int pitch = NB == 4 ? job.pitch_y : job.pitch_c;
  const int rpb = (rows + n_bands - 1) / n_bands;
  const int r0 = band * rpb, r1 = min(rows, r0 + rpb);
  if (r0 >= r1) return;

  uint4 *const tslot = tiles + (size_t)warp * (kSwarTileBytes / 16) + slot * kSlot;
  uint4 *const t_h = tslot + (pl * NB + sub) * kRegion;      // as column group: my region (chunk q = rows 4q..4q+3)
  uint4 *const t_carry = tslot + (pl * NB + NB - 1) * kRegion + sub;  // as row group: my rows of the last column group
  // output ring of this warp: my slot, my plane
  unsigned char *const ring_w = rings + (size_t)warp * kSwarRingBytes;
  unsigned char *const ring_me = ring_w + slot * Ring::kSlotBytes + pl * Ring::kR * Ring::kRowBytes;
  unsigned long long *const ptr_w = ptrs + warp * 16;
  if ((NB == 4 && u == 0) || (NB == 2 && (u & 1) == 0)) ptr_w[slot * 2 + pl] = (unsigned long long)(size_t)plane;
  const unsigned active_mask = __ballot_sync(0xffffffffu, active);
  __syncwarp();
  // flush roles of this lane (constant): the macroblock's own rows ...
  constexpr int kMainItems = kN * Ring::kHalves * Ring::kPlanes;  // per slot: 32 / 16
  constexpr int kMainIters = 8 * kMainItems / 32;                 // 8 / 4
  const int f_rem = lane % kMainItems, f_slot0 = lane / kMainItems;
  const int f_pl = NB == 4 ? 0 : (f_rem >> 3), f_row = NB == 4 ? (f_rem >> 1) : (f_rem & 7), f_half = NB == 4 ? (f_rem & 1) : 0;
  const bool f_swz = Ring::Swz(3 + f_row);
  const int f_smem = (f_pl * Ring::kR + 3 + f_row) * Ring::kRowBytes;
  // ... and the three rows above (6 items per slot, 48 in all: lanes 0..31, then 0..15)
  int a_slot[2], a_pl[2], a_k[2], a_half[2];
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const int it = lane + 32 * j, rem = it % 6;
    a_slot[j] = it / 6;
    a_pl[j] = NB == 4 ? 0 : rem / 3;
    a_k[j] = NB == 4 ? (rem >> 1) : rem % 3;
    a_half[j] = NB == 4 ? (rem & 1) : 0;
  }

  const int publish_row = band + 1 < n_bands ? r1 - 1 : -1;  // the band's last row, read by the next band (none after the last)
  for (int lr = warp; lr < r1 - r0; lr += kSwarWarps) {
    const int r = r0 + lr;
    const bool last_of_band = r == publish_row;
    const bool has_above = r > 0;
    const bool above_local = lr > 0;
    const uint8_t *rowp = plane + (ptrdiff_t)(r * kN + 4 * sub) * pitch;         // row group: first of my four rows, x = 0
    const uint8_t *colp = plane + (ptrdiff_t)(r * kN) * pitch + 4 * sub;         // column group: my four columns, row 0
    const vp8r_mb_info *mbrow = mbs + (size_t)r * cols;
    const ptrdiff_t row_top = (ptrdiff_t)(r * kN - 3) * pitch;                   // ring row 0 of a plane = 3 rows above

    uint32_t nxt[4][NB];
#pragma unroll
    for (int y = 0; y < 4; ++y) LoadRowWords<NB>(rowp + (ptrdiff_t)y * pitch, nxt[y]);
    unsigned flags_n = __ldg(&mbrow[0].flags);
    uint32_t carry[4] = {0, 0, 0, 0};
    uint32_t a4n[4] = {0, 0, 0, 0};
    int gseen = 0;
    bool have_above = false;

    // Writes macroblocks [first, first + kG) of this warp's ring rows to the frames (whole flush units).
    auto flush = [&](int first) {
      const int ms0 = first % Ring::kRingMbs;                                   // ring position of the unit: 0 or kG
      const int chunk0 = (ms0 * kN) >> 4;
      const int x0 = first * kN;
      {
        const int soff = f_smem + ((((chunk0 + f_half) ^ (f_swz ? Ring::kSwzXor : 0))) << 4);
        const ptrdiff_t goff = row_top + (ptrdiff_t)(3 + f_row) * pitch + x0 + 16 * f_half;
#pragma unroll
        for (int it = 0; it < kMainIters; ++it) {
          const int sl = it * (32 / kMainItems) + f_slot0;
          const uint4 v = *reinterpret_cast<const uint4 *>(ring_w + sl * Ring::kSlotBytes + soff);
          uint8_t *base = reinterpret_cast<uint8_t *>((size_t)ptr_w[sl * 2 + f_pl]);
          if ((active_mask >> (4 * sl)) & 1) *reinterpret_cast<uint4 *>(base + goff) = v;
        }
      }
      if (has_above) {
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          if (j == 0 || lane < 16) {
            const int soff = (a_pl[j] * Ring::kR + a_k[j]) * Ring::kRowBytes +
                             ((((chunk0 + a_half[j]) ^ (Ring::Swz(a_k[j]) ? Ring::kSwzXor : 0))) << 4);
            const uint4 v = *reinterpret_cast<const uint4 *>(ring_w + a_slot[j] * Ring::kSlotBytes + soff);
            uint8_t *base = reinterpret_cast<uint8_t *>((size_t)ptr_w[a_slot[j] * 2 + a_pl[j]]);
            if ((active_mask >> (4 * a_slot[j])) & 1)
              *reinterpret_cast<uint4 *>(base + row_top + (ptrdiff_t)a_k[j] * pitch + x0 + 16 * a_half[j]) = v;
          }
        }
      }
    };

    for (int c = 0; c < cols; ++c) {
      uint32_t W[4 + 4 * NB];
#pragma unroll
      for (int k = 0; k < NB; ++k)
#pragma unroll
        for (int y = 0; y < 4; ++y) W[4 + 4 * k + y] = nxt[y][k];
      const unsigned flags = flags_n;
      if (c + 1 < cols) {
#pragma unroll
        for (int y = 0; y < 4; ++y) LoadRowWords<NB>(rowp + (ptrdiff_t)y * pitch + (c + 1) * kN, nxt[y]);
        flags_n = __ldg(&mbrow[c + 1].flags);
      }
      int seen = 0;
      if (has_above) seen = above_local ? lprog[lr - 1] : gseen;

      const swar::EdgeK K = EdgeKFor(flags, sharpness, key_frame);
      const bool any_inner = __any_sync(0xffffffffu, K.k_sb != 0x80008000u);
      const int need = min(c + 1, cols);  // macroblocks 0..c of the row above must be in memory

      // ---- vertical edges: words = pixel columns of my four rows ----
#pragma unroll
      for (int i = 0; i < 4; ++i) W[i] = carry[i];
#pragma unroll
      for (int k = 0; k < NB; ++k) swar::Transpose4(W[4 + 4 * k], W[5 + 4 * k], W[6 + 4 * k], W[7 + 4 * k]);
      FilterEdgesSwar<NB>(W, K, c > 0, any_inner, simple);
      if (c > 0) {  // the previous macroblock's last four columns are final for these rows now: into its ring place
        uint32_t t[4] = {W[0], W[1], W[2], W[3]};
        swar::Transpose4(t[0], t[1], t[2], t[3]);
        const int off = ((c - 1) % Ring::kRingMbs) * kN + 4 * (NB - 1);
        const int chunk = off >> 4, low = off & 15;
        // rows 3 + 4 * sub + y: the swizzle of luma rows does not depend on sub, that of chroma rows flips with it
        const bool flip = NB == 2 && (sub & 1);
        unsigned char *a0 = ring_me + (3 + 4 * sub) * Ring::kRowBytes + low + ((chunk ^ (flip ? Ring::kSwzXor : 0)) << 4);
        unsigned char *a1 = ring_me + (3 + 4 * sub) * Ring::kRowBytes + low + ((chunk ^ (flip ? 0 : Ring::kSwzXor)) << 4);
#pragma unroll
        for (int y = 0; y < 4; ++y)
          *reinterpret_cast<uint32_t *>((Ring::Swz(3 + y) ? a1 : a0) + y * Ring::kRowBytes) = t[y];
      }
      // back to pixel rows and over to the lanes that own the columns
#pragma unroll
      for (int k = 0; k < NB; ++k) {
        swar::Transpose4(W[4 + 4 * k], W[5 + 4 * k], W[6 + 4 * k], W[7 + 4 * k]);
        tslot[(pl * NB + k) * kRegion + sub] = make_uint4(W[4 + 4 * k], W[5 + 4 * k], W[6 + 4 * k], W[7 + 4 * k]);
      }
      __syncwarp();

      // ---- horizontal edges: words = pixel rows of my four columns ----
#pragma unroll
      for (int q = 0; q < NB; ++q) {
        const uint4 t = t_h[q];
        W[4 + 4 * q] = t.x; W[5 + 4 * q] = t.y; W[6 + 4 * q] = t.z; W[7 + 4 * q] = t.w;
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) W[i] = a4n[i];
      if (has_above && !have_above) {  // not prefetched: wait for the row above, then fetch
        if (above_local) {
          for (int got = lprog[lr - 1]; got < need; got = lprog[lr - 1])
            __nanosleep(min(kSwarSleepBase + kSwarSleepSlope * (need - got - 1), kSwarSleepMax));
          __threadfence_block();
        } else {
          for (gseen = LoadFlagAcquireSwar(gflag - 1); gseen < need; gseen = LoadFlagAcquireSwar(gflag - 1))
            __nanosleep(min(kSwarSleepBase + kSwarSleepSlope * (need - gseen - 1), kSwarSleepMax));
        }
#pragma unroll
        for (int y = 0; y < 4; ++y) W[y] = __ldcg(reinterpret_cast<const uint32_t *>(colp + c * kN + (ptrdiff_t)(y - 4) * pitch));
      }
      FilterEdgesSwar<NB>(W, K, has_above, any_inner, simple);
      {  // into the ring: rows above (1..3 of W) and the macroblock's rows, my four columns
        const int off = (c % Ring::kRingMbs) * kN + 4 * sub;
        const int chunk = off >> 4, low = off & 15;
        unsigned char *a0 = ring_me + low + (chunk << 4), *a1 = ring_me + low + ((chunk ^ Ring::kSwzXor) << 4);
        if (has_above) {
#pragma unroll
          for (int y = 1; y < 4; ++y)
            *reinterpret_cast<uint32_t *>((Ring::Swz(y - 1) ? a1 : a0) + (y - 1) * Ring::kRowBytes) = W[y];
        }
#pragma unroll
        for (int y = 0; y < kN; ++y)
          *reinterpret_cast<uint32_t *>((Ring::Swz(3 + y) ? a1 : a0) + (3 + y) * Ring::kRowBytes) = W[4 + y];
      }
      if (c + 1 < cols) {
        if (sub == NB - 1) {
#pragma unroll
          for (int q = 0; q < NB; ++q) t_h[q] = make_uint4(W[4 + 4 * q], W[5 + 4 * q], W[6 + 4 * q], W[7 + 4 * q]);
        }
        __syncwarp();
        const uint4 t = *t_carry;
        carry[0] = t.x; carry[1] = t.y; carry[2] = t.z; carry[3] = t.w;
        swar::Transpose4(carry[0], carry[1], carry[2], carry[3]);
      } else {
        __syncwarp();
      }

      // rows above of the next macroblock: fetch now if the row above is far enough already
      have_above = false;
      if (has_above && c + 1 < cols && seen >= min(c + 2, cols)) {
        if (above_local) __threadfence_block();
#pragma unroll
        for (int y = 0; y < 4; ++y)
          a4n[y] = __ldcg(reinterpret_cast<const uint32_t *>(colp + (c + 1) * kN + (ptrdiff_t)(y - 4) * pitch));
        have_above = true;
      }

      // Flush + publish.  After step c the macroblocks < c are final (the last columns of macroblock c still
      // wait for the next left edge); whole units go out at every kG-th step, everything after the last one.
      const bool last = c == cols - 1;
      if (last || (c >= Ring::kG && c % Ring::kG == 0)) {
        if (last) {
          for (int first = (c / Ring::kG) * Ring::kG - ((c % Ring::kG == 0 && c >= Ring::kG) ? Ring::kG : 0); first < cols; first += Ring::kG)
            flush(first);
        } else {
          flush(c - Ring::kG);
        }
        const int stored = last ? cols : c;
        if (last_of_band && (last || ((c / Ring::kG) % kSwarBandStride) == 0)) {
          __threadfence();
          __syncwarp();
          if (lane == 0) atomicExch(gflag, stored);
        } else {
          __threadfence_block();
        }
        __syncwarp();
        if (lane == 0) lprog[lr] = stored;
      }
    }
  }
}

}  // namespace

__global__ void __launch_bounds__(kSwarWarps * 32, 1) FilterSwarKernel(const DevFrameJob *__restrict__ jobs,
                                                        const FilterGroup *__restrict__ groups, int n_groups, int n_bands,
                                                        int *__restrict__ sync) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ int s_ticket;
  if (threadIdx.x == 0) s_ticket = atomicAdd(&sync[0], 1);
  __syncthreads();
  // Tickets are band-major (band b of every group and plane kind before band b+1 of any): a CTA only waits
  // for a smaller ticket, i.e. a CTA that is running or done.
  const int per_band = 2 * n_groups;
  const int band = s_ticket / per_band, rem = s_ticket - band * per_band;
  const int g = rem >> 1, chroma = rem & 1;
  const FilterGroup grp = groups[g];
  const DevFrameJob &job0 = jobs[grp.frame[0]];
  if (chroma && job0.filter_type != 0) return;  // the simple filter leaves chroma alone (src/filter.cc:69-71)
  const int rpb = (job0.mb_rows + n_bands - 1) / n_bands;
  volatile int *lprog = reinterpret_cast<volatile int *>(smem_raw);
  unsigned char *at = smem_raw + ((rpb * 4 + 15) & ~15);
  uint4 *tiles = reinterpret_cast<uint4 *>(at);
  at += kSwarWarps * kSwarTileBytes;
  unsigned char *rings = at;
  at += kSwarWarps * kSwarRingBytes;
  unsigned long long *ptrs = reinterpret_cast<unsigned long long *>(at);
  for (int i = threadIdx.x; i < rpb; i += blockDim.x) lprog[i] = 0;
  __syncthreads();
  int *gflag = sync + 1 + (g * 2 + chroma) * n_bands + band;
  if (chroma) FilterBandSwar<2>(jobs, grp, band, n_bands, gflag, lprog, tiles, rings, ptrs);
  else FilterBandSwar<4>(jobs, grp, band, n_bands, gflag, lprog, tiles, rings, ptrs);
}

cudaError_t LaunchFilterSwar(const DevFrameJob *jobs, const FilterGroup *groups, int n_groups, int max_rows, int *sync,
                             int sync_ints, cudaStream_t st) {
  if (n_groups <= 0) return cudaSuccess;
  int n_bands = (max_rows + kSwarWarps - 1) / kSwarWarps;
  if (n_bands > 64) n_bands = 64;
  const int n_flags = 1 + 2 * n_groups * n_bands;
  if (n_flags > sync_ints) return cudaErrorInvalidValue;
  cudaError_t e = cudaMemsetAsync(sync, 0, sizeof(int) * size_t(n_flags), st);
  if (e != cudaSuccess) return e;
  const int rpb = (max_rows + n_bands - 1) / n_bands;
  const size_t smem = ((size_t(rpb) * 4 + 15) & ~size_t(15)) + size_t(kSwarWarps) * (kSwarTileBytes + kSwarRingBytes + kSwarPtrBytes);
  if (smem > 48 * 1024) {
    e = cudaFuncSetAttribute(FilterSwarKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  FilterSwarKernel<<<2 * n_groups * n_bands, kSwarWarps * 32, smem, st>>>(jobs, groups, n_groups, n_bands, sync);
  return cudaGetLastError();
}

}  // namespace vp8r
