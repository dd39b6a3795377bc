// Hand-written sm_100a kernels of the VP8 reconstruction path.
//
//   K_inter  : one warp per inter macroblock.  Residual: the coded blocks only, four lanes per block
//              (dequant -> IWHT/IDCT), into shared memory.  Prediction: one 21x21 / 13x13 window per
//              plane for a macroblock with one vector, one 9x9 window per lane and 4x4 block for SPLIT;
//              horizontal then vertical 6-tap/bilinear pass on packed bytes with dp4a -> residual
//              add -> store.   Replaces src/inter_predict.cc:246-333, src/residual.cc:42-157,
//              src/dct.cc:67-133, src/quantizer.cc:10-13 of the reference.
//   K_intra  : one CTA per frame, one warp per macroblock row, rows advance as a wavefront
//              (row r may process column c once row r-1 has finished column c+1).  Replaces
//              src/intra_predict.cc:6-428.
//   K_filter : same wavefront shape; lanes = the 16+8+8 pixel lines of a macroblock.  Replaces
//              src/filter.cc:7-340.  Ends with the border extension motion compensation relies on.
//
// All arithmetic is integer and bit-exact with the reference, including its int16 wrap-arounds.
#include "recon_kernels.h"

#include <algorithm>
#include <cstring>

namespace vp8r {

// ------------------------------------------------------------------------------------------
// constant tables
// ------------------------------------------------------------------------------------------
// Sub-pixel filter taps packed as signed bytes: [bilinear][frac][0] = taps 0..3, [..][1] = taps 4,5.
// frac 0 (identity, tap 128) is special-cased and never looked up.
__constant__ int c_taps[2][8][2];
// The same taps as plain integers, for the packed 16x2 vertical pass: [bilinear][frac][tap].
__constant__ int c_taps6[2][8][6];
// B_PRED gather table: [mode][pixel] -> i0 | i1<<4 | i2<<8 | kind<<12 over the 13-entry edge
// array E = {L3,L2,L1,L0,P,A0..A7}.  kind 0: (E[i0]+2E[i1]+E[i2]+2)>>2, 1: (E[i0]+E[i2]+1)>>1,
// 2: DC, 3: TM = clamp(E[i0]+E[i1]-E[i2]).
__constant__ unsigned short c_bpred_lut[10 * 16];

static int PackTaps(int a, int b, int c, int d) {
  return (a & 0xff) | ((b & 0xff) << 8) | ((c & 0xff) << 16) | ((d & 0xff) << 24);
}

static void BuildBpredLut(unsigned short *lut) {
  auto L = [](int k) { return 3 - k; };
  auto A = [](int k) { return 5 + k; };
  const int P = 4;
  auto put3 = [&](int mode, int y, int x, int a, int b, int c) {
    lut[mode * 16 + y * 4 + x] = (unsigned short)(a | (b << 4) | (c << 8) | (0 << 12));
  };
  auto put2 = [&](int mode, int y, int x, int a, int c) {
    lut[mode * 16 + y * 4 + x] = (unsigned short)(a | (a << 4) | (c << 8) | (1 << 12));
  };
  for (int y = 0; y < 4; ++y)
    for (int x = 0; x < 4; ++x) {
      lut[0 * 16 + y * 4 + x] = (unsigned short)(2 << 12);                                   // B_DC
      lut[1 * 16 + y * 4 + x] = (unsigned short)(L(y) | (A(x) << 4) | (P << 8) | (3 << 12)); // B_TM
      put3(2, y, x, 4 + x, 5 + x, 6 + x);                                                    // B_VE
      put3(3, y, x, 4 - y, 3 - y, (2 - y) > 0 ? 2 - y : 0);                                  // B_HE
      int d = x + y;
      put3(4, y, x, 5 + d, 6 + d, (7 + d) < 12 ? 7 + d : 12);                                // B_LD
      int k = 3 - y + x;
      put3(5, y, x, k, k + 1, k + 2);                                                        // B_RD
    }
  // B_VR (E = first nine entries of the edge array)
  put3(6, 3, 0, 1, 2, 3); put3(6, 2, 0, 2, 3, 4); put3(6, 3, 1, 3, 4, 5); put3(6, 1, 0, 3, 4, 5);
  put2(6, 2, 1, 4, 5);    put2(6, 0, 0, 4, 5);    put3(6, 3, 2, 4, 5, 6); put3(6, 1, 1, 4, 5, 6);
  put2(6, 2, 2, 5, 6);    put2(6, 0, 1, 5, 6);    put3(6, 3, 3, 5, 6, 7); put3(6, 1, 2, 5, 6, 7);
  put2(6, 2, 3, 6, 7);    put2(6, 0, 2, 6, 7);    put3(6, 1, 3, 6, 7, 8); put2(6, 0, 3, 7, 8);
  // B_VL
  put2(7, 0, 0, A(0), A(1));       put3(7, 1, 0, A(0), A(1), A(2)); put2(7, 2, 0, A(1), A(2));
  put2(7, 0, 1, A(1), A(2));       put3(7, 1, 1, A(1), A(2), A(3)); put3(7, 3, 0, A(1), A(2), A(3));
  put2(7, 2, 1, A(2), A(3));       put2(7, 0, 2, A(2), A(3));       put3(7, 3, 1, A(2), A(3), A(4));
  put3(7, 1, 2, A(2), A(3), A(4)); put2(7, 2, 2, A(3), A(4));       put2(7, 0, 3, A(3), A(4));
  put3(7, 3, 2, A(3), A(4), A(5)); put3(7, 1, 3, A(3), A(4), A(5)); put3(7, 2, 3, A(4), A(5), A(6));
  put3(7, 3, 3, A(5), A(6), A(7));
  // B_HD
  put2(8, 3, 0, 0, 1);    put3(8, 3, 1, 0, 1, 2); put2(8, 2, 0, 1, 2);    put2(8, 3, 2, 1, 2);
  put3(8, 2, 1, 1, 2, 3); put3(8, 3, 3, 1, 2, 3); put2(8, 2, 2, 2, 3);    put2(8, 1, 0, 2, 3);
  put3(8, 2, 3, 2, 3, 4); put3(8, 1, 1, 2, 3, 4); put2(8, 1, 2, 3, 4);    put2(8, 0, 0, 3, 4);
  put3(8, 1, 3, 3, 4, 5); put3(8, 0, 1, 3, 4, 5); put3(8, 0, 2, 4, 5, 6); put3(8, 0, 3, 5, 6, 7);
  // B_HU
  put2(9, 0, 0, L(0), L(1));       put3(9, 0, 1, L(0), L(1), L(2)); put2(9, 0, 2, L(1), L(2));
  put2(9, 1, 0, L(1), L(2));       put3(9, 0, 3, L(1), L(2), L(3)); put3(9, 1, 1, L(1), L(2), L(3));
  put2(9, 1, 2, L(2), L(3));       put2(9, 2, 0, L(2), L(3));       put3(9, 1, 3, L(2), L(3), L(3));
  put3(9, 2, 1, L(2), L(3), L(3));
  put3(9, 2, 2, L(3), L(3), L(3)); put3(9, 2, 3, L(3), L(3), L(3)); put3(9, 3, 0, L(3), L(3), L(3));
  put3(9, 3, 1, L(3), L(3), L(3)); put3(9, 3, 2, L(3), L(3), L(3)); put3(9, 3, 3, L(3), L(3), L(3));
}

cudaError_t InitKernelTables() {
  // src/inter_predict.h:18-36 (RFC 6386 section 18.3)
  static const int six[8][6] = {{0, 0, 128, 0, 0, 0},  {0, -6, 123, 12, -1, 0},   {2, -11, 108, 36, -8, 1},
                                {0, -9, 93, 50, -6, 0}, {3, -16, 77, 77, -16, 3}, {0, -6, 50, 93, -9, 0},
                                {1, -8, 36, 108, -11, 2}, {0, -1, 12, 123, -6, 0}};
  int taps[2][8][2];
  for (int f = 0; f < 8; ++f) {
    taps[0][f][0] = PackTaps(six[f][0], six[f][1], six[f][2], six[f][3]);
    taps[0][f][1] = PackTaps(six[f][4], six[f][5], 0, 0);
    taps[1][f][0] = PackTaps(0, 0, 128 - 16 * f, 16 * f);
    taps[1][f][1] = 0;
  }
  cudaError_t err = cudaMemcpyToSymbol(c_taps, taps, sizeof(taps));
  if (err != cudaSuccess) return err;
  int taps6[2][8][6];
  for (int f = 0; f < 8; ++f)
    for (int k = 0; k < 6; ++k) {
      taps6[0][f][k] = six[f][k];
      taps6[1][f][k] = k == 2 ? 128 - 16 * f : (k == 3 ? 16 * f : 0);
    }
  err = cudaMemcpyToSymbol(c_taps6, taps6, sizeof(taps6));
  if (err != cudaSuccess) return err;
  err = InitParseTables();
  if (err != cudaSuccess) return err;
  unsigned short lut[160];
  std::memset(lut, 0, sizeof(lut));
  BuildBpredLut(lut);
  err = InitEncodeTables(lut);
  if (err != cudaSuccess) return err;
  return cudaMemcpyToSymbol(c_bpred_lut, lut, sizeof(lut));
}

// ------------------------------------------------------------------------------------------
// small device helpers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ int dp4a_us(unsigned a, int b, int c) {
  int d;
  asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
__device__ __forceinline__ int clamp255(int x) { return min(max(x, 0), 255); }
__device__ __forceinline__ int clamp128(int x) { return min(max(x, -128), 127); }
__device__ __forceinline__ int s16(int x) { return (int)(short)x; }

// One 1-D pass of the inverse DCT (src/dct.cc:67-107) on v[0..3]: the vertical pass (kRow = false) on a
// column, truncated to int16; the horizontal pass on a row, with the rounding shift.
template <bool kRow>
__device__ __forceinline__ void Idct1D(int *v) {
  const int a = v[0] + v[2], b = v[0] - v[2];
  const int c = ((v[1] * 35468) >> 16) - (v[3] + ((v[3] * 20091) >> 16));
  const int d = (v[1] + ((v[1] * 20091) >> 16)) + ((v[3] * 35468) >> 16);
  const int rnd = kRow ? 4 : 0, sh = kRow ? 3 : 0;
  v[0] = s16((a + d + rnd) >> sh);
  v[1] = s16((b + c + rnd) >> sh);
  v[2] = s16((b - c + rnd) >> sh);
  v[3] = s16((a - d + rnd) >> sh);
}

// The same for the inverse Walsh-Hadamard transform of Y2 (src/dct.cc:109-133).
template <bool kRow>
__device__ __forceinline__ void Iwht1D(int *v) {
  const int a = v[0] + v[3], b = v[1] + v[2], c = v[1] - v[2], d = v[0] - v[3];
  const int rnd = kRow ? 3 : 0, sh = kRow ? 3 : 0;
  v[0] = s16((a + b + rnd) >> sh);
  v[1] = s16((c + d + rnd) >> sh);
  v[2] = s16((a - b + rnd) >> sh);
  v[3] = s16((d - c + rnd) >> sh);
}

// Column j of the macroblock's coded block number `at` (payload order), dequantized with the int16
// wrap-around of the reference (src/quantizer.cc:10-13): v[r] = coefficient (r, j).
__device__ __forceinline__ void LoadColumn(const DevFrameJob &job, int at, int j, int dcq, int acq, int *v) {
  const int4 *src = reinterpret_cast<const int4 *>(job.payload + (size_t)at * 16);
  const int4 lo = __ldg(src), hi = __ldg(src + 1);
  // coefficient (r, j) is half (j & 1) of word 2r + (j >> 1)
  const bool odd = (j & 2) != 0;
  const int w[4] = {odd ? lo.y : lo.x, odd ? lo.w : lo.z, odd ? hi.y : hi.x, odd ? hi.w : hi.z};
  const int sh = (j & 1) * 16;
#pragma unroll
  for (int r = 0; r < 4; ++r) v[r] = s16(s16(w[r] >> sh) * (r == 0 && j == 0 ? dcq : acq));
}

// 4x4 inverse transform by the four lanes of a group: on entry lane j holds column j (v[r] = row r).  The
// block's 16 shorts `t` carry the transposition; on return they hold the result, row j written by lane j as
// four packed int16.  Every lane of the warp calls this; only the `active` ones touch `t`.
template <bool kWht>
__device__ __forceinline__ void Transform4Lanes(int *v, short *t, int j, bool active) {
  if (kWht) Iwht1D<false>(v); else Idct1D<false>(v);
  if (active) {
#pragma unroll
    for (int r = 0; r < 4; ++r) t[4 * r + j] = (short)v[r];
  }
  __syncwarp();
  if (active) {
    uint2 *row = reinterpret_cast<uint2 *>(t + 4 * j);
    const uint2 p = *row;
    v[0] = s16(p.x); v[1] = (int)p.x >> 16; v[2] = s16(p.y); v[3] = (int)p.y >> 16;
    if (kWht) Iwht1D<true>(v); else Idct1D<true>(v);
    *row = make_uint2(((unsigned)v[0] & 0xffffu) | ((unsigned)v[1] << 16), ((unsigned)v[2] & 0xffffu) | ((unsigned)v[3] << 16));
  }
}

// Residual of a macroblock with coef_mask != 0 (src/residual.cc:42-120), into the warp's scratch `s`:
// s.res[b] = the 4x4 residual of block b (0..15 Y raster, 16..19 U, 20..23 V) as four rows of four int16, for
// every block, uncoded ones included.  Only the blocks that need it are transformed, each by four lanes
// (one column, then one row each), eight blocks per pass.  A macroblock has ~5 coded blocks of 25 on typical
// streams, so one pass is the rule; any number of blocks is exact.  Y2 goes first, on lanes 0..3, into s.y2:
// its outputs are the DCs of the Y blocks.  A Y block whose only input is that DC is DC-only: every output
// of its IDCT is (dc + 4) >> 3, written without a transform.  Ends without a barrier: callers sync the warp
// before they read s.res.
template <class Scratch>
__device__ __forceinline__ void WarpResidual(const DevFrameJob &job, const vp8r_mb_info &mb, int lane, Scratch &s) {
  const unsigned mask = mb.coef_mask;  // bit 0: Y2, bit 1 + b: block b
  const unsigned coded = (mask >> 1) & 0xffffffu;
  const bool y2 = (mb.flags & VP8R_MB_HAS_Y2) && (mask & 1);
  const int16_t *dq = job.dq[(mb.flags >> VP8R_MB_QSEG_SHIFT) & 3];
  const int g = lane >> 2, j = lane & 3;
  if (y2) {
    int v[4];
    LoadColumn(job, mb.coef_offset, j, dq[VP8R_DQ_Y2_DC], dq[VP8R_DQ_Y2_AC], v);
    Transform4Lanes<true>(v, s.y2, j, lane < 4);
    __syncwarp();
  }
  // coded blocks by rank, for the transform passes
  if (lane < 24 && ((coded >> lane) & 1)) s.order[__popc(coded & ((1u << lane) - 1))] = (unsigned char)lane;
  // blocks without coefficients: zero, or the DC-only IDCT of their Y2 DC; half a block per lane and store
#pragma unroll
  for (int c = lane; c < 48; c += 32) {
    const int b = c >> 1;
    if (!((coded >> b) & 1)) {
      const unsigned v = y2 && b < 16 ? ((unsigned)((s.y2[b] + 4) >> 3) & 0xffffu) * 0x10001u : 0u;
      reinterpret_cast<uint4 *>(s.res[b])[c & 1] = make_uint4(v, v, v, v);
    }
  }
  __syncwarp();
  const int n = __popc(coded);
  for (int base = 0; base < n; base += 8) {  // warp-uniform
    const int b = s.order[min(base + g, n - 1)];  // lanes past the last block redo it and do not store
    const bool luma = b < 16;
    int v[4];
    LoadColumn(job, mb.coef_offset + __popc(mask & ((2u << b) - 1)), j, luma ? dq[VP8R_DQ_Y1_DC] : dq[VP8R_DQ_UV_DC],
               luma ? dq[VP8R_DQ_Y1_AC] : dq[VP8R_DQ_UV_AC], v);
    if (y2 && luma && j == 0) v[0] = s.y2[b];
    Transform4Lanes<false>(v, s.res[b], j, base + g < n);
  }
}

// ------------------------------------------------------------------------------------------
// K_inter
// ------------------------------------------------------------------------------------------
// Saturating pack of four ints to bytes (o0 lowest): two I2IP.  cvt.pack: d = c<<16 | sat(a)<<8 | sat(b).
__device__ __forceinline__ unsigned PackSat4(int o0, int o1, int o2, int o3) {
  unsigned t, d;
  asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(t) : "r"(o3), "r"(o2), "r"(0));
  asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(o1), "r"(o0), "r"(t));
  return d;
}

// Horizontal filter of 4 outputs from 9 packed bytes (`lo` = bytes 0..3, `mid` = bytes 4..7, `hi` = byte 8, upper
// bytes ignored), the clamp+pack done by I2IP.  The TAPS are shifted instead of the data: pixel j of the word needs
// bytes j..j+5 of (lo, mid, hi), i.e. dp4a(lo, t03 << 8j) + dp4a(mid, (t45:t03) >> (32 - 8j)) [+ dp4a(hi, t45 >> (32 - 8j)),
// non-zero for j = 3 only]: nine dp4a per word instead of eight dp4a and six funnel shifts on byte-shifted words.  The
// seven shifted vectors are per-macroblock values.
struct TapsAt {
  int lo1, lo2, lo3, mid1, mid2, mid3, hi3;
};
__device__ __forceinline__ TapsAt MakeTapsAt(int t03, int t45) {
  TapsAt t;
  t.lo1 = t03 << 8; t.lo2 = t03 << 16; t.lo3 = t03 << 24;
  t.mid1 = (int)__funnelshift_l((unsigned)t03, (unsigned)t45, 8);
  t.mid2 = (int)__funnelshift_l((unsigned)t03, (unsigned)t45, 16);
  t.mid3 = (int)__funnelshift_l((unsigned)t03, (unsigned)t45, 24);
  t.hi3 = (int)((unsigned)t45 >> 8);
  return t;
}
__device__ __forceinline__ unsigned Filter4T(unsigned lo, unsigned mid, unsigned hi, int t03, int t45, const TapsAt &t) {
  const int s0 = dp4a_us(mid, t45, dp4a_us(lo, t03, 64)) >> 7;
  const int s1 = dp4a_us(mid, t.mid1, dp4a_us(lo, t.lo1, 64)) >> 7;
  const int s2 = dp4a_us(mid, t.mid2, dp4a_us(lo, t.lo2, 64)) >> 7;
  const int s3 = dp4a_us(hi, t.hi3, dp4a_us(mid, t.mid3, dp4a_us(lo, t.lo3, 64))) >> 7;
  return PackSat4(s0, s1, s2, s3);
}

// Vertical 6-tap on packed pixels: e[k] / o[k] hold pixels (0,2) / (1,3) of row k in 16-bit lanes.
// acc = sum t[k]*row[k] per lane, in one 32-bit multiply-add per two pixels.  Lane sums lie in
// [-8160, 40800]; the bias 8192 + 64 keeps both lanes non-negative (no borrow into the upper lane) and,
// being 64*128 + rounding, comes out of the >>7 as +64, removed by the saturating add.
__device__ __forceinline__ unsigned Vert6(const unsigned *e, const unsigned *o, const int *t) {
  const unsigned bias = (8192u + 64u) * 0x00010001u;
  unsigned ae = bias, ao = bias;
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    ae += (unsigned)t[k] * e[k];
    ao += (unsigned)t[k] * o[k];
  }
  ae = (ae >> 7) & 0x01ff01ffu;
  ao = (ao >> 7) & 0x01ff01ffu;
  ae = __vmins2(__viaddmax_s16x2(ae, 0xffc0ffc0u, 0u), 0x00ff00ffu);  // clamp(x - 64, 0, 255) per lane
  ao = __vmins2(__viaddmax_s16x2(ao, 0xffc0ffc0u, 0u), 0x00ff00ffu);
  return ae | (ao << 8);
}

// clamp255(int16(pred + res)) on 4 packed pixels; r01 / r23 hold the four int16 residuals.
__device__ __forceinline__ unsigned AddResidual4(unsigned pred, unsigned r01, unsigned r23) {
  const unsigned pe = __byte_perm(pred, 0, 0x4240), po = __byte_perm(pred, 0, 0x4341);
  const unsigned re = __byte_perm(r01, r23, 0x5410), ro = __byte_perm(r01, r23, 0x7632);
  const unsigned se = __vmins2(__vmaxs2(__vadd2(pe, re), 0u), 0x00ff00ffu);  // 16-bit wrap-around add, as the reference
  const unsigned so = __vmins2(__vmaxs2(__vadd2(po, ro), 0u), 0x00ff00ffu);
  return se | (so << 8);
}

// Word index of luma row r in InterScratch::hl: rows are 4 words; every 8 rows one row is skipped so
// that the vertical pass (lanes read rows k, k+2, ..., k+14 at once) hits 8 different bank groups.
__device__ __forceinline__ int HlRow(int r) { return (r + (r >> 3)) * 4; }

// ---- TMA plumbing (sm_90+): a bulk tensor load of one box into shared memory, completion on an mbarrier ----
__device__ __forceinline__ unsigned SmemAddr(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void MbarInit(unsigned long long *bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(SmemAddr(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");  // visible to the async proxy (the TMA unit)
}
__device__ __forceinline__ void MbarExpectTx(unsigned long long *bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(SmemAddr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void MbarWait(unsigned long long *bar, unsigned parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "MBAR_WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra MBAR_DONE_%=;\n\t"
      "bra MBAR_WAIT_%=;\n\t"
      "MBAR_DONE_%=:\n\t}" ::"r"(SmemAddr(bar)), "r"(parity)
      : "memory");
}
// Box of `map` whose first element is (x, y) -> dst (128-byte aligned shared memory); bytes land on `bar`.
__device__ __forceinline__ void TmaLoad2D(void *dst, const DevTensorMap *map, int x, int y, unsigned long long *bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                   SmemAddr(dst)),
               "l"(map), "r"(x), "r"(y), "r"(SmemAddr(bar))
               : "memory");
}

// Reference windows of one macroblock as the TMA unit delivers them: dense boxes.
struct __align__(128) InterTile {
  unsigned char luma[kTmaLumaBoxH * kTmaLumaBoxW];            // 21 rows x 48 bytes
  unsigned char pad0[1024 - kTmaLumaBoxH * kTmaLumaBoxW];
  unsigned char cu[kTmaChromaBoxH * kTmaChromaBoxW];          // 13 rows x 48 bytes
  unsigned char pad1[640 - kTmaChromaBoxH * kTmaChromaBoxW];
  unsigned char cv[kTmaChromaBoxH * kTmaChromaBoxW];
  unsigned char pad2[640 - kTmaChromaBoxH * kTmaChromaBoxW - 8];
  unsigned long long bar;                                      // one transaction barrier per warp
};
static_assert(sizeof(InterTile) == 2304, "tile layout");
constexpr unsigned kInterTileTxBytes = kTmaLumaBoxH * kTmaLumaBoxW + 2 * kTmaChromaBoxH * kTmaChromaBoxW;

// Motion vectors and window origins of a macroblock with one vector (src/inter_predict.cc:116-144,246-333).
struct WholeMbGeometry {
  int fr, fc, cfr, cfc;  // eighth-pel fractions, luma and chroma
  int wy, wx, cwy, cwx;  // window origins (row, column) in plane coordinates, clamped as a whole into the border
};
__device__ __forceinline__ WholeMbGeometry WholeGeometry(const DevFrameJob &job, const vp8r_mb_info &mb, int mb_r, int mb_c) {
  WholeMbGeometry g;
  const int mvr = mb.mv[0], mvc = mb.mv[1];
  const int sr = s16(4 * mvr), sc = s16(4 * mvc);
  // (x + sign(x) 4) / 8, truncating: on magnitudes
  const int ar = (abs(sr) + 4) >> 3, ac = (abs(sc) + 4) >> 3;
  int cmr = sr < 0 ? -ar : ar, cmc = sc < 0 ? -ac : ac;
  if (job.version == 3) {
    cmr &= ~7;
    cmc &= ~7;
  }
  g.fr = mvr & 7; g.fc = mvc & 7; g.cfr = cmr & 7; g.cfc = cmc & 7;
  g.wy = min(max(mb_r * 16 + (mvr >> 3) - 2, -kBorder), job.mb_rows * 16 + kBorder - 21);
  g.wx = min(max(mb_c * 16 + (mvc >> 3) - 2, -kBorder), job.mb_cols * 16 + kBorder - 21);
  g.cwy = min(max(mb_r * 8 + (cmr >> 3) - 2, -kBorder), job.mb_rows * 8 + kBorder - 13);
  g.cwx = min(max(mb_c * 8 + (cmc >> 3) - 2, -kBorder), job.mb_cols * 8 + kBorder - 13);
  return g;
}

// Per-warp scratch of the macroblock-level motion compensation.
struct __align__(16) InterScratch {
  unsigned hl[23 * 4];     // luma after the horizontal pass: 21 rows x 16 pixels, row r at word HlRow(r)
  unsigned hc[2][13 * 2];  // U, V after the horizontal pass: 13 rows x 8 pixels
  short res[24][16];       // residual of the 24 blocks (WarpResidual)
  short y2[16];
  unsigned char order[24];
};

// Motion compensation of a non-SPLIT inter macroblock by one warp (src/inter_predict.cc:246-333): the
// 16x16 luma block and the two 8x8 chroma blocks each have ONE vector, so the reference window is
// fetched and filtered once per macroblock (21x21 / 13x13) instead of once per 4x4 block (9x9 each):
// windows staged in shared memory by TMA, horizontal pass (Filter4T) into shared memory, vertical pass on
// packed 16-bit lanes, residual add, store.
__device__ __forceinline__ void InterMacroblockWhole(const DevFrameJob &job, int mb_r, int mb_c, int lane, InterScratch &s,
                                                     bool has_res, const WholeMbGeometry &g, InterTile *tile) {
  const int bil = job.version != 0;
  const int fr = g.fr, fc = g.fc, cfr = g.cfr, cfc = g.cfc;

  // ---- horizontal pass on the boxes the TMA unit put into shared memory: the box starts at the window's
  // first pixel, so every lane reads aligned words; no address arithmetic on the frame, no byte shifting ----
  MbarWait(&tile->bar, 0);
  {
    const int dx = (g.wx + kBorder) & 15;  // the box starts at the window's x rounded down to 16
    const int w = lane & 3, row0 = lane >> 2, base = (dx >> 2) + w;
    const unsigned shift = (dx & 3) * 8;
    const int r_lo = fr ? 0 : 2, r_hi = (fr | fc) ? (fr ? 21 : 18) : 0;  // whole-pel vectors: the rows are read below, in place
    const int t03 = c_taps[bil][fc][0], t45 = c_taps[bil][fc][1];
    const TapsAt ta = MakeTapsAt(t03, t45);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const int row = row0 + 8 * k;
      if (row >= r_lo && row < r_hi) {
        const unsigned *p = reinterpret_cast<const unsigned *>(tile->luma + row * kTmaLumaBoxW) + base;
        const unsigned w0 = p[0], w1 = p[1], w2 = p[2];
        const unsigned lo = __funnelshift_r(w0, w1, shift), mid = __funnelshift_r(w1, w2, shift), hi = w2 >> shift;
        s.hl[HlRow(row) + w] = fc ? Filter4T(lo, mid, hi, t03, t45, ta) : __funnelshift_r(lo, mid, 16);
      }
    }
  }
  {
    const int dx = (g.cwx + kBorder) & 15;
    const int row = lane >> 1, cw_ = lane & 1, base = (dx >> 2) + cw_;
    const unsigned shift = (dx & 3) * 8;
    const int r_lo = cfr ? 0 : 2, r_hi = (cfr | cfc) ? (cfr ? 13 : 10) : 0;
    const int t03 = c_taps[bil][cfc][0], t45 = c_taps[bil][cfc][1];
    const TapsAt ta = MakeTapsAt(t03, t45);
    if (row >= r_lo && row < r_hi) {
#pragma unroll
      for (int pl = 0; pl < 2; ++pl) {
        const unsigned *p = reinterpret_cast<const unsigned *>((pl ? tile->cv : tile->cu) + row * kTmaChromaBoxW) + base;
        const unsigned w0 = p[0], w1 = p[1], w2 = p[2];
        const unsigned lo = __funnelshift_r(w0, w1, shift), mid = __funnelshift_r(w1, w2, shift), hi = w2 >> shift;
        s.hc[pl][row * 2 + cw_] = cfc ? Filter4T(lo, mid, hi, t03, t45, ta) : __funnelshift_r(lo, mid, 16);
      }
    }
  }
  __syncwarp();

  // ---- vertical pass + residual + store, luma: lane = (output word w, row pair yg) ----
  {
    const int w = lane & 3, y0 = (lane >> 2) * 2;
    unsigned out0, out1;
    if (fr) {
      unsigned e[7], o[7];
#pragma unroll
      for (int k = 0; k < 7; ++k) {
        const unsigned r = s.hl[HlRow(y0 + k) + w];
        e[k] = __byte_perm(r, 0, 0x4240);
        o[k] = __byte_perm(r, 0, 0x4341);
      }
      const int *t = c_taps6[bil][fr];
      out0 = Vert6(e, o, t);
      out1 = Vert6(e + 1, o + 1, t);
    } else if (fc == 0) {  // whole-pel: straight from the window the TMA unit delivered
      const int dx2 = ((g.wx + kBorder) & 15) + 2;
      const unsigned *p = reinterpret_cast<const unsigned *>(tile->luma + (y0 + 2) * kTmaLumaBoxW) + (dx2 >> 2) + w;
      const unsigned sh = (dx2 & 3) * 8;
      out0 = __funnelshift_r(p[0], p[1], sh);
      out1 = __funnelshift_r(p[kTmaLumaBoxW / 4], p[kTmaLumaBoxW / 4 + 1], sh);
    } else {
      out0 = s.hl[HlRow(y0 + 2) + w];
      out1 = s.hl[HlRow(y0 + 3) + w];
    }
    if (has_res) {
      const uint2 *rp = reinterpret_cast<const uint2 *>(&s.res[(y0 >> 2) * 4 + w][(y0 & 3) * 4]);
      const uint2 ra = rp[0], rb = rp[1];
      out0 = AddResidual4(out0, ra.x, ra.y);
      out1 = AddResidual4(out1, rb.x, rb.y);
    }
    uint8_t *d = job.cur.y + (ptrdiff_t)(mb_r * 16 + y0) * job.pitch_y + mb_c * 16 + 4 * w;
    *reinterpret_cast<unsigned *>(d) = out0;
    *reinterpret_cast<unsigned *>(d + job.pitch_y) = out1;
  }
  // ---- chroma: lane = (plane, row y, output word w) ----
  {
    const int pl = lane >> 4, y = (lane >> 1) & 7, w = lane & 1;
    const unsigned *h = s.hc[pl];
    unsigned out;
    if (cfr) {
      unsigned e[6], o[6];
#pragma unroll
      for (int k = 0; k < 6; ++k) {
        const unsigned r = h[(y + k) * 2 + w];
        e[k] = __byte_perm(r, 0, 0x4240);
        o[k] = __byte_perm(r, 0, 0x4341);
      }
      out = Vert6(e, o, c_taps6[bil][cfr]);
    } else if (cfc == 0) {
      const int dx2 = ((g.cwx + kBorder) & 15) + 2;
      const unsigned *p = reinterpret_cast<const unsigned *>((pl ? tile->cv : tile->cu) + (y + 2) * kTmaChromaBoxW) + (dx2 >> 2) + w;
      out = __funnelshift_r(p[0], p[1], (dx2 & 3) * 8);
    } else {
      out = h[(y + 2) * 2 + w];
    }
    if (has_res) {
      const uint2 ra = *reinterpret_cast<const uint2 *>(&s.res[16 + pl * 4 + (y >> 2) * 2 + w][(y & 3) * 4]);
      out = AddResidual4(out, ra.x, ra.y);
    }
    uint8_t *d = (pl ? job.cur.v : job.cur.u) + (ptrdiff_t)(mb_r * 8 + y) * job.pitch_c + mb_c * 8 + 4 * w;
    *reinterpret_cast<unsigned *>(d) = out;
  }
}

constexpr int kInterWarps = 4;
constexpr int kInterMinBlocks = 14;  // 32 registers, 20 bytes of spill: 4 % faster than 12 CTAs at 40 registers; 14 x 14.8 KB
                                     // of shared memory is what an SM holds (before the compacted residual: 12 was best)

// One inter macroblock by one warp.
__device__ __forceinline__ void InterOneMacroblock(const DevFrameJob &job, int mb_r, int mb_c, int lane, InterScratch &scratch, InterTile *tile) {
  const int mb_index = mb_r * job.mb_cols + mb_c;
  vp8r_mb_info mb;
  {
    const int4 *p = reinterpret_cast<const int4 *>(job.mbs + mb_index);
    int4 a = __ldg(p), b = __ldg(p + 1);
    mb.flags = a.x; mb.coef_mask = a.y; mb.coef_offset = a.z;
    mb.mv[0] = (short)(a.w & 0xffff); mb.mv[1] = (short)(a.w >> 16);
    mb.aux[0] = b.x; mb.aux[1] = b.y;
  }
  if (!(mb.flags & VP8R_MB_IS_INTER)) return;

  const bool split = ((mb.flags >> VP8R_MB_MODE_SHIFT) & 7) == 4;
  WholeMbGeometry geo{};
  if (!split) {
    geo = WholeGeometry(job, mb, mb_r, mb_c);
    if (lane == 0) {  // the three windows are on their way while the warp computes the residual
      // (all operands are warp-uniform and, the warp index being read from lane 0 in the kernel, known to be: they
      // live in uniform registers and each UTMALDG is issued directly, not through an elect / broadcast loop)
      const DevTensorMap *maps = job.ref_tmap[(mb.flags >> VP8R_MB_REF_SHIFT) & 3];
      MbarExpectTx(&tile->bar, kInterTileTxBytes);
      TmaLoad2D(tile->luma, maps + 0, (geo.wx + kBorder) & ~15, geo.wy + kBorder, &tile->bar);
      TmaLoad2D(tile->cu, maps + 1, (geo.cwx + kBorder) & ~15, geo.cwy + kBorder, &tile->bar);
      TmaLoad2D(tile->cv, maps + 2, (geo.cwx + kBorder) & ~15, geo.cwy + kBorder, &tile->bar);
    }
  }
  const bool has_res = mb.coef_mask != 0;  // then every block of scratch.res is written, uncoded ones as zero
  if (has_res) WarpResidual(job, mb, lane, scratch);
  if (!split) {  // one vector for the whole macroblock: window fetched and filtered once
    InterMacroblockWhole(job, mb_r, mb_c, lane, scratch, has_res, geo, tile);
    return;
  }
  __syncwarp();  // the residual rows were written by other lanes
  if (lane >= 24) return;

  // SPLIT: every 4x4 block can have its own vector, so each lane predicts one block from its own 9x9 window.
  const int ref_id = (mb.flags >> VP8R_MB_REF_SHIFT) & 3;
  const int *split_mv = reinterpret_cast<const int *>(job.payload + (size_t)mb.aux[0] * 16);

  // Block geometry and motion vector (1/8 pel) of this lane.
  int mvr, mvc, bx, by, pitch, plane_w, plane_h;
  const uint8_t *ref;
  uint8_t *dst;
  if (lane < 16) {
    const int m = __ldg(split_mv + lane);
    mvr = (short)(m & 0xffff);
    mvc = m >> 16;
    by = mb_r * 16 + (lane >> 2) * 4;
    bx = mb_c * 16 + (lane & 3) * 4;
    pitch = job.pitch_y;
    plane_w = job.mb_cols * 16;
    plane_h = job.mb_rows * 16;
    ref = job.ref[ref_id].y;
    dst = job.cur.y;
  } else {
    // Chroma MV: sum of the four luma MVs under the block, rounded away from zero, /8
    // (src/inter_predict.cc:116-144; the reference discards its own clamp of the result).
    const int b = lane & 3, i = b >> 1, j = b & 1;
    const int k0 = i * 8 + j * 2;
    const int m0 = __ldg(split_mv + k0), m1 = __ldg(split_mv + k0 + 1), m2 = __ldg(split_mv + k0 + 4),
              m3 = __ldg(split_mv + k0 + 5);
    const int sr = s16((short)(m0 & 0xffff) + (short)(m1 & 0xffff) + (short)(m2 & 0xffff) + (short)(m3 & 0xffff));
    const int sc = s16((m0 >> 16) + (m1 >> 16) + (m2 >> 16) + (m3 >> 16));
    mvr = (sr >= 0 ? (sr + 4) : (sr - 4)) / 8;
    mvc = (sc >= 0 ? (sc + 4) : (sc - 4)) / 8;
    if (job.version == 3) {
      mvr &= ~7;
      mvc &= ~7;
    }
    by = mb_r * 8 + i * 4;
    bx = mb_c * 8 + j * 4;
    pitch = job.pitch_c;
    plane_w = job.mb_cols * 8;
    plane_h = job.mb_rows * 8;
    ref = lane < 20 ? job.ref[ref_id].u : job.ref[ref_id].v;
    dst = lane < 20 ? job.cur.u : job.cur.v;
  }

  const int fr = mvr & 7, fc = mvc & 7;
  // 9x9 window origin, clamped as a whole into the padded plane (see kBorder).
  int wy = by + (mvr >> 3) - 2, wx = bx + (mvc >> 3) - 2;
  wy = min(max(wy, -kBorder), plane_h + kBorder - 9);
  wx = min(max(wx, -kBorder), plane_w + kBorder - 9);
  // A window row is 9 bytes at up to 7 bytes past an 8-byte boundary: two aligned 8-byte loads hold it (plane
  // origins and pitches are multiples of 16).  Words w0..w2 start at the 4-byte boundary below the row.
  const uint8_t *__restrict__ wp = ref + (ptrdiff_t)wy * pitch + wx;
  const uint2 *__restrict__ wrow = reinterpret_cast<const uint2 *>(wp - ((size_t)wp & 7));
  const bool upper = ((size_t)wp & 4) != 0;
  const unsigned shift = ((unsigned)(size_t)wp & 3u) * 8;
  const int wpitch = pitch >> 3;

  // ---- horizontal pass over the window rows the vertical pass needs (all 9, or rows 2..5), as in the
  // whole-macroblock path: Filter4T, or the plain pixels for whole-pel columns ----
  const int bil = job.version != 0;
  const int r_lo = fr ? 0 : 2, r_hi = fr ? 9 : 6;
  const int t03 = c_taps[bil][fc][0], t45 = c_taps[bil][fc][1];
  const TapsAt ta = MakeTapsAt(t03, t45);
  unsigned h[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) {
    if (i >= r_lo && i < r_hi) {
      const uint2 a = __ldg(wrow + i * wpitch), b = __ldg(wrow + i * wpitch + 1);
      const unsigned w0 = upper ? a.y : a.x, w1 = upper ? b.x : a.y, w2 = upper ? b.y : b.x;
      const unsigned lo = __funnelshift_r(w0, w1, shift), mid = __funnelshift_r(w1, w2, shift), hi = w2 >> shift;
      h[i] = fc ? Filter4T(lo, mid, hi, t03, t45, ta) : __funnelshift_r(lo, mid, 16);
    }
  }
  // ---- vertical pass on packed 16-bit lanes (Vert6), residual add, store ----
  unsigned out[4];
  if (fr) {
    const int v03 = c_taps[bil][fr][0], v45 = c_taps[bil][fr][1];
    const int t[6] = {(signed char)v03, (signed char)(v03 >> 8), (signed char)(v03 >> 16), v03 >> 24,
                      (signed char)v45, (signed char)(v45 >> 8)};
    unsigned e[9], o[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      e[k] = __byte_perm(h[k], 0, 0x4240);
      o[k] = __byte_perm(h[k], 0, 0x4341);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) out[i] = Vert6(e + i, o + i, t);
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i) out[i] = h[2 + i];
  }
  uint8_t *d = dst + (ptrdiff_t)by * pitch + bx;
  const uint2 *rp = reinterpret_cast<const uint2 *>(scratch.res[lane]);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    unsigned v = out[i];
    if (has_res) {
      const uint2 r = rp[i];
      v = AddResidual4(v, r.x, r.y);
    }
    *reinterpret_cast<unsigned *>(d + (ptrdiff_t)i * pitch) = v;
  }
}

// One macroblock per warp.  Walking several consecutive macroblocks per warp (shared record lines,
// overlapping reference windows) was measured and is slower: 2 per warp +23 %, 4 per warp +30 % of the
// time of 1 per warp (the loop body spills ~200 bytes per thread and the warp's serial latency chain
// gets longer); letting the compiler unroll that loop blows the instruction cache (4 per warp 3.8x).
// grid = (macroblock columns / warps, macroblock rows, frames): a warp's macroblock coordinates come from the
// block indices (a linear index cost ~24 instructions per macroblock for the division)
__global__ void __launch_bounds__(kInterWarps * 32, kInterMinBlocks) InterKernel(const DevFrameJob *__restrict__ jobs) {
  __shared__ InterScratch s_scratch[kInterWarps];
  __shared__ InterTile s_tile[kInterWarps];
  const DevFrameJob &job = jobs[blockIdx.z];
  // (read from lane 0: tells the compiler that the warp index, and every address derived from it, is warp-uniform)
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int mb_r = blockIdx.y, cols = job.mb_cols;
  const int mb_c = blockIdx.x * kInterWarps + warp;
  if (mb_r >= job.mb_rows || mb_c >= cols) return;
  if (JobFailed(job) || JobInter(job) == 0) return;
  // the warp fetches one macroblock: its barrier completes phase 0 exactly once
  if (lane == 0) MbarInit(&s_tile[warp].bar, 1);
  __syncwarp();
  InterOneMacroblock(job, mb_r, mb_c, lane, s_scratch[warp], &s_tile[warp]);
  // Not needed for correctness; without it ptxas schedules the kernel differently and it measured 0.2 % slower
  // (B200, 1000 W, 512 1080p frames per launch).
  __syncwarp();
}

cudaError_t LaunchInter(const DevFrameJob *jobs, int n_frames, int max_cols, int max_rows, cudaStream_t st) {
  if (max_rows > 65535 || n_frames > 65535) return cudaErrorInvalidValue;
  dim3 grid((max_cols + kInterWarps - 1) / kInterWarps, max_rows, n_frames);
  InterKernel<<<grid, kInterWarps * 32, 0, st>>>(jobs);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// wavefront plumbing shared by K_intra and K_filter
// ------------------------------------------------------------------------------------------
constexpr int kWaveWarps = 32;

__device__ __forceinline__ void WaitRow(volatile int *progress, int row, int need) {
  if (row < 0) return;
  while (progress[row] < need) __nanosleep(40);
  __threadfence_block();
}
__device__ __forceinline__ void PublishRow(volatile int *progress, int row, int done, int lane) {
  __syncwarp();
  __threadfence_block();
  if (lane == 0) progress[row] = done;
}

// ------------------------------------------------------------------------------------------
// K_intra
// ------------------------------------------------------------------------------------------
struct __align__(16) IntraScratch {
  short y2[16];
  short res[24][16];
  unsigned char tile[17][24];  // B_PRED working tile: row 0 = row above, column 3 = column left,
                               // macroblock pixel (y,x) at tile[1+y][4+x]; columns 20..23 of row 0
                               // hold the above-right pixels.
  unsigned char order[24];
};

// 16x16 / 8x8 prediction of one 4x4 block by its owning lane (src/intra_predict.cc:6-98).
// Every lane of the warp must call this (it shuffles); only lanes < 24 produce output.
__device__ __forceinline__ void PredictMbBlock(const DevFrameJob &job, int mb_r, int mb_c, int lane, int ymode,
                                               int uvmode, bool do_luma, const short *res, bool has_res) {
  const bool luma = lane < 16;
  const int n4 = luma ? 4 : 2;
  const int first = luma ? 0 : (lane < 20 ? 16 : 20);
  const int b = lane - first, i = luma ? (b >> 2) : (b >> 1), j = luma ? (b & 3) : (b & 1);
  const int pitch = luma ? job.pitch_y : job.pitch_c;
  uint8_t *plane = luma ? job.cur.y : (lane < 20 ? job.cur.u : job.cur.v);
  const int n = luma ? 16 : 8;
  uint8_t *mbp = plane + (ptrdiff_t)(mb_r * n) * pitch + mb_c * n;
  const bool active = lane < 24 && (do_luma || !luma);
  const int mode = luma ? ymode : uvmode;
  const bool have_above = mb_r > 0, have_left = mb_c > 0;

  unsigned aw = 0x7f7f7f7fu;
  int l[4] = {129, 129, 129, 129};
  int P = have_above ? (have_left ? 0 : 129) : 127;
  if (lane < 24) {
    if (have_above) aw = *reinterpret_cast<const unsigned *>(mbp - pitch + 4 * j);
    if (have_left) {
#pragma unroll
      for (int k = 0; k < 4; ++k) l[k] = mbp[(ptrdiff_t)(4 * i + k) * pitch - 1];
    }
    if (have_above && have_left) P = mbp[-pitch - 1];
  }
  // DC needs the sums over the whole edge: gather from the lanes on the first block row / column.
  int sum_a = (int)__dp4a(aw, 0x01010101u, 0u);
  int sum_l = l[0] + l[1] + l[2] + l[3];
  int tot_a = 0, tot_l = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    int va = __shfl_sync(0xffffffffu, sum_a, first + (k < n4 ? k : 0));
    int vl = __shfl_sync(0xffffffffu, sum_l, first + (k < n4 ? k * n4 : 0));
    if (k < n4) {
      tot_a += va;
      tot_l += vl;
    }
  }
  if (!active) return;

  unsigned rows[4];
  if (mode == 1) {  // V_PRED
    rows[0] = rows[1] = rows[2] = rows[3] = aw;
  } else if (mode == 2) {  // H_PRED
#pragma unroll
    for (int k = 0; k < 4; ++k) rows[k] = (unsigned)l[k] * 0x01010101u;
  } else if (mode == 0) {  // DC_PRED
    int v = 128;
    if (have_above || have_left) {
      int shf = (luma ? 3 : 2) + (have_above ? 1 : 0) + (have_left ? 1 : 0);
      int sum = (have_above ? tot_a : 0) + (have_left ? tot_l : 0);
      v = (sum + (1 << (shf - 1))) >> shf;
    }
    rows[0] = rows[1] = rows[2] = rows[3] = (unsigned)v * 0x01010101u;
  } else {  // TM_PRED
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      unsigned o = 0;
#pragma unroll
      for (int x = 0; x < 4; ++x) o |= (unsigned)clamp255(l[k] + (int)((aw >> (8 * x)) & 0xff) - P) << (8 * x);
      rows[k] = o;
    }
  }
  uint8_t *d = mbp + (ptrdiff_t)(4 * i) * pitch + 4 * j;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    unsigned v = rows[k];
    if (has_res) {
      unsigned o = 0;
#pragma unroll
      for (int x = 0; x < 4; ++x) o |= (unsigned)clamp255(s16((int)((v >> (8 * x)) & 0xff) + res[k * 4 + x])) << (8 * x);
      v = o;
    }
    *reinterpret_cast<unsigned *>(d + (ptrdiff_t)k * pitch) = v;
  }
}

// B_PRED luma of one macroblock by one warp (src/intra_predict.cc:100-351).
__device__ __forceinline__ void PredictBpred(const DevFrameJob &job, int mb_r, int mb_c, int lane,
                                             const vp8r_mb_info &mb, IntraScratch &s, unsigned res_mask,
                                             const unsigned short *lut) {
  const int pitch = job.pitch_y;
  uint8_t *mbp = job.cur.y + (ptrdiff_t)(mb_r * 16) * pitch + mb_c * 16;
  // Row above: columns -1..19 -> tile[0][3..23].
  if (lane < 21) {
    int col = lane - 1, v;
    if (mb_r == 0) {
      v = 127;
    } else if (col < 0) {
      v = mb_c == 0 ? 129 : mbp[-pitch - 1];
    } else if (col >= 16 && mb_c + 1 == job.mb_cols) {
      v = mbp[-pitch + 15];  // src/intra_predict.cc:130-132
    } else {
      v = mbp[-pitch + col];
    }
    s.tile[0][4 + col] = (unsigned char)v;
  }
  if (lane < 16) s.tile[1 + lane][3] = (unsigned char)(mb_c == 0 ? 129 : mbp[(ptrdiff_t)lane * pitch - 1]);
  __syncwarp();

  const int py = (lane >> 2) & 3, px = lane & 3;
  for (int b = 0; b < 16; ++b) {
    const int i = b >> 2, j = b & 3;
    const int mode = (int)((mb.aux[b >> 3] >> ((b & 7) * 4)) & 15);
    // Edge array E[0..12] = L3,L2,L1,L0,P,A0..A7, one entry per lane.
    int E = 0;
    if (lane < 4) {
      E = s.tile[1 + 4 * i + (3 - lane)][3 + 4 * j];
    } else if (lane < 9) {
      E = s.tile[4 * i][3 + 4 * j + (lane - 4)];
    } else if (lane < 13) {
      const int row = (j == 3) ? 0 : 4 * i;  // right-most column: always the macroblock row above
      E = s.tile[row][3 + 4 * j + (lane - 4)];
    }
    const unsigned e = lut[mode * 16 + (lane & 15)];
    const int x0 = __shfl_sync(0xffffffffu, E, e & 15);
    const int x1 = __shfl_sync(0xffffffffu, E, (e >> 4) & 15);
    const int x2 = __shfl_sync(0xffffffffu, E, (e >> 8) & 15);
    const int dc_in = (lane < 4 || (lane >= 5 && lane < 9)) ? E : 0;
    const int dc = (__reduce_add_sync(0xffffffffu, dc_in) + 4) >> 3;
    const int kind = e >> 12;
    int v;
    if (kind == 0) v = (x0 + 2 * x1 + x2 + 2) >> 2;
    else if (kind == 1) v = (x0 + x2 + 1) >> 1;
    else if (kind == 2) v = dc;
    else v = clamp255(x0 + x1 - x2);
    if (lane < 16) {
      if ((res_mask >> b) & 1) v = clamp255(s16(v + s.res[b][lane]));
      s.tile[1 + 4 * i + py][4 + 4 * j + px] = (unsigned char)v;
    }
    __syncwarp();
  }
  if (lane < 16) {
    const unsigned *t = reinterpret_cast<const unsigned *>(&s.tile[1 + lane][4]);
    uint4 v = make_uint4(t[0], t[1], t[2], t[3]);
    *reinterpret_cast<uint4 *>(mbp + (ptrdiff_t)lane * pitch) = v;
  }
}

// One intra macroblock by one warp: residual, then chroma / 16x16 luma per 4x4 block, then B_PRED.
__device__ __forceinline__ void IntraMacroblock(const DevFrameJob &job, int r, int c, int lane, IntraScratch &s,
                                                const unsigned short *lut, volatile int *progress) {
  vp8r_mb_info mb;
  {
    const int4 *p = reinterpret_cast<const int4 *>(job.mbs + r * job.mb_cols + c);
    int4 a = __ldg(p), b = __ldg(p + 1);
    // every lane holds the same record; reading it from lane 0 makes that known to the compiler where the index came
    // out of a table (uniform branches, uniform-datapath address arithmetic: IntraLevelsKernel 2800 -> 2168 instructions)
    a.x = __shfl_sync(0xffffffffu, a.x, 0); a.y = __shfl_sync(0xffffffffu, a.y, 0);
    a.z = __shfl_sync(0xffffffffu, a.z, 0); a.w = __shfl_sync(0xffffffffu, a.w, 0);
    b.x = __shfl_sync(0xffffffffu, b.x, 0); b.y = __shfl_sync(0xffffffffu, b.y, 0);
    mb.flags = a.x; mb.coef_mask = a.y; mb.coef_offset = a.z;
    mb.aux[0] = b.x; mb.aux[1] = b.y;
  }
  const bool has_res = mb.coef_mask != 0;  // then every block of s.res is written, uncoded ones as zero
  if (has_res) WarpResidual(job, mb, lane, s);
  // Everything above and to the left must be final (unfiltered) pixels of this frame.
  if (progress) WaitRow(progress, r - 1, min(c + 2, job.mb_cols));
  __syncwarp();
  const int ymode = (mb.flags >> VP8R_MB_MODE_SHIFT) & 7, uvmode = (mb.flags >> VP8R_MB_UVMODE_SHIFT) & 3;
  PredictMbBlock(job, r, c, lane, ymode, uvmode, ymode != 4, lane < 24 ? s.res[lane] : s.res[0], has_res);
  if (ymode == 4) PredictBpred(job, r, c, lane, mb, s, mb.coef_mask >> 1, lut);  // no Y2: only coded blocks have a residual
}

// Wavefront variant: frames whose intra macroblocks form long dependency chains (key frames).
__global__ void __launch_bounds__(kWaveWarps * 32) IntraKernel(const DevFrameJob *__restrict__ jobs) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const DevFrameJob &job = jobs[blockIdx.x];
  if (JobFailed(job) || JobIntra(job) == 0 || JobIntraLevels(job) != 0) return;
  const int rows = job.mb_rows, cols = job.mb_cols;
  volatile int *progress = reinterpret_cast<volatile int *>(smem_raw);
  unsigned short *lut = reinterpret_cast<unsigned short *>(smem_raw + ((rows * 4 + 15) & ~15));
  IntraScratch *scratch = reinterpret_cast<IntraScratch *>(reinterpret_cast<unsigned char *>(lut) + 320);
  for (int i = threadIdx.x; i < rows; i += blockDim.x) progress[i] = 0;
  for (int i = threadIdx.x; i < 160; i += blockDim.x) lut[i] = c_bpred_lut[i];
  __syncthreads();

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;  // from lane 0: known to be warp-uniform
  IntraScratch &s = scratch[warp];
  for (int r = warp; r < rows; r += kWaveWarps) {
    for (int c0 = 0; c0 < cols; c0 += 32) {
      // Which of the next 32 macroblocks of this row are intra coded?
      unsigned flags = 0;
      if (c0 + lane < cols) flags = __ldg(&job.mbs[r * cols + c0 + lane].flags);
      unsigned intra_mask = __ballot_sync(0xffffffffu, (c0 + lane < cols) && !(flags & VP8R_MB_IS_INTER));
      while (intra_mask) {
        const int k = __ffs(intra_mask) - 1;
        intra_mask &= intra_mask - 1;
        const int c = c0 + k;
        IntraMacroblock(job, r, c, lane, s, lut, progress);
        PublishRow(progress, r, c + 1, lane);
      }
      PublishRow(progress, r, min(c0 + 32, cols), lane);
    }
  }
}

// Flat variant: all intra macroblocks of dependency level `level` of every frame, one warp each.
// Levels are launched in increasing order; macroblocks of one level never neighbour each other.
constexpr int kFlatWarps = 8;
// 8 CTAs per SM: 32 registers and 12 bytes of spill; measured faster than 6 CTAs at the 39 registers the compiler picks
__global__ void __launch_bounds__(kFlatWarps * 32, 8) IntraFlatKernel(const DevFrameJob *__restrict__ jobs, int level) {
  __shared__ __align__(16) unsigned short lut[160];
  __shared__ IntraScratch scratch[kFlatWarps];
  const DevFrameJob &job = jobs[blockIdx.y];
  if (JobFailed(job) || job.dyn || level >= job.n_intra_levels) return;  // job.dyn: handled by IntraLevelsKernel
  const unsigned first = __ldg(job.intra_levels + level), end = __ldg(job.intra_levels + level + 1);
  if (first + blockIdx.x * kFlatWarps >= end) return;  // the grid is sized by the frame with most macroblocks on this level
  for (int i = threadIdx.x; i < 160; i += blockDim.x) lut[i] = c_bpred_lut[i];
  __syncthreads();
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;  // from lane 0: known to be warp-uniform
  const unsigned slot = first + blockIdx.x * kFlatWarps + warp;
  if (slot >= end) return;
  const unsigned mb_index = __ldg(job.intra_levels + job.n_intra_levels + 1 + slot);
  const int r = mb_index / job.mb_cols, c = mb_index - r * job.mb_cols;
  IntraMacroblock(job, r, c, lane, scratch[warp], lut, nullptr);
}

// Frames whose level table was built on the device (deferred modes): the host does not know how many
// levels or macroblocks per level there are, so one CTA per frame walks all levels, its warps sharing
// the macroblocks of a level, with a block barrier between levels.
constexpr int kLevelWarps = 16;
__global__ void __launch_bounds__(kLevelWarps * 32) IntraLevelsKernel(const DevFrameJob *__restrict__ jobs) {
  __shared__ __align__(16) unsigned short lut[160];
  __shared__ IntraScratch scratch[kLevelWarps];
  const DevFrameJob &job = jobs[blockIdx.x];
  if (JobFailed(job) || !job.dyn) return;
  const int n_levels = JobIntraLevels(job);
  if (n_levels == 0) return;
  for (int i = threadIdx.x; i < 160; i += blockDim.x) lut[i] = c_bpred_lut[i];
  __syncthreads();
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;  // from lane 0: known to be warp-uniform
  const uint32_t *tab = JobLevelTable(job);
  const uint32_t *order = tab + n_levels + 1;
  for (int level = 0; level < n_levels; ++level) {
    const unsigned first = tab[level], end = tab[level + 1];
    for (unsigned slot = first + warp; slot < end; slot += kLevelWarps) {
      const unsigned mb_index = order[slot];
      const int r = mb_index / job.mb_cols, c = mb_index - r * job.mb_cols;
      IntraMacroblock(job, r, c, lane, scratch[warp], lut, nullptr);
    }
    __syncthreads();  // pixels of this level are visible to the whole CTA before the next starts
  }
}

cudaError_t LaunchIntraLevels(const DevFrameJob *jobs, int n_frames, cudaStream_t st) {
  IntraLevelsKernel<<<n_frames, kLevelWarps * 32, 0, st>>>(jobs);
  return cudaGetLastError();
}

cudaError_t LaunchIntraFlat(const DevFrameJob *jobs, int n_frames, int level, int max_count, cudaStream_t st) {
  if (max_count <= 0) return cudaSuccess;
  dim3 grid((max_count + kFlatWarps - 1) / kFlatWarps, n_frames);
  IntraFlatKernel<<<grid, kFlatWarps * 32, 0, st>>>(jobs, level);
  return cudaGetLastError();
}

static size_t IntraSmemBytes(int max_rows) {
  return ((size_t(max_rows) * 4 + 15) & ~size_t(15)) + 320 + sizeof(IntraScratch) * kWaveWarps;
}

cudaError_t LaunchIntra(const DevFrameJob *jobs, int n_frames, int max_rows, cudaStream_t st) {
  size_t smem = IntraSmemBytes(max_rows);
  static size_t configured[64] = {};  // per device: the attribute belongs to the (function, device) pair
  int dev = 0;
  cudaGetDevice(&dev);
  size_t &mark = configured[dev & 63];
  if (smem > 48 * 1024 && smem > mark) {
    cudaError_t e = cudaFuncSetAttribute(IntraKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    mark = smem;
  }
  IntraKernel<<<n_frames, kWaveWarps * 32, smem, st>>>(jobs);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// K_filter
// ------------------------------------------------------------------------------------------
struct LfLimits {
  int interior, hev, edge_mb, edge_sb;
};

// src/filter.cc:119-149
__device__ __forceinline__ LfLimits MakeLimits(int level, int sharp, bool key) {
  LfLimits l;
  int in = level;
  if (sharp) {
    in >>= (sharp > 4) ? 2 : 1;
    in = min(in, 9 - sharp);
  }
  l.interior = max(in, 1);
  if (key) l.hev = level >= 40 ? 2 : (level >= 15 ? 1 : 0);
  else l.hev = level >= 40 ? 3 : (level >= 20 ? 2 : (level >= 15 ? 1 : 0));
  l.edge_mb = (level + 2) * 2 + l.interior;
  l.edge_sb = level * 2 + l.interior;
  return l;
}

// One edge on 8 pixels v[0..7] = p3 p2 p1 p0 | q0 q1 q2 q3, branch-free: every lane evaluates the
// mask, the high-variance test and both filter variants and selects per-pixel deltas (a warp's 32
// lines almost always disagree on the tests, so branching would execute every path anyway).
//   mask / hev:      src/filter.cc:7-20      Adjust:            src/filter.cc:22-35
//   sub-block edge:  src/filter.cc:37-44     macroblock edge:   src/filter.cc:46-67
//   simple filter:   src/filter.cc:14-16,69-71 (luma only)
__device__ __forceinline__ int AddClamp255(int p, int d) { return min(max(p + d, 0), 255); }

template <bool kMbEdge>
__device__ __forceinline__ void LfEdge(int *v, const LfLimits &lim, bool simple) {
  const int edge = kMbEdge ? lim.edge_mb : lim.edge_sb;
  const int p3 = v[0], p2 = v[1], p1 = v[2], p0 = v[3], q0 = v[4], q1 = v[5], q2 = v[6], q3 = v[7];
  const int d_p1q1 = p1 - q1, d_q0p0 = q0 - p0;
  const bool edge_ok = abs(d_q0p0) * 2 + (abs(d_p1q1) >> 1) <= edge;
  const int s = clamp128(d_p1q1);
  if (simple) {
    const int a = clamp128(s + 3 * d_q0p0);
    const int f1 = min(a + 4, 127) >> 3, f2 = min(a + 3, 127) >> 3;
    v[3] = AddClamp255(p0, edge_ok ? f2 : 0);
    v[4] = AddClamp255(q0, edge_ok ? -f1 : 0);
    return;
  }
  const int a_p1p0 = abs(p1 - p0), a_q1q0 = abs(q1 - q0);
  const int interior = max(max(max(abs(p3 - p2), abs(p2 - p1)), a_p1p0), max(max(a_q1q0, abs(q1 - q2)), abs(q2 - q3)));
  const bool on = edge_ok && interior <= lim.interior;
  const bool hev = max(a_p1p0, a_q1q0) > lim.hev;
  if (kMbEdge) {
    const int w = clamp128(s + 3 * d_q0p0);
    const int f1 = min(w + 4, 127) >> 3, f2 = min(w + 3, 127) >> 3;  // hev: Adjust(true)
    const int a27 = (27 * w + 63) >> 7, a18 = (18 * w + 63) >> 7, a9 = (9 * w + 63) >> 7;
    const int dp0 = on ? (hev ? f2 : a27) : 0, dq0 = on ? (hev ? f1 : a27) : 0;
    const int d1 = (on && !hev) ? a18 : 0, d2 = (on && !hev) ? a9 : 0;
    v[1] = AddClamp255(p2, d2);
    v[2] = AddClamp255(p1, d1);
    v[3] = AddClamp255(p0, dp0);
    v[4] = AddClamp255(q0, -dq0);
    v[5] = AddClamp255(q1, -d1);
    v[6] = AddClamp255(q2, -d2);
  } else {
    const int a = clamp128((hev ? s : 0) + 3 * d_q0p0);  // Adjust(hev)
    const int f1 = min(a + 4, 127) >> 3, f2 = min(a + 3, 127) >> 3;
    const int a2 = (on && !hev) ? ((f1 + 1) >> 1) : 0;
    v[2] = AddClamp255(p1, a2);
    v[3] = AddClamp255(p0, on ? f2 : 0);
    v[4] = AddClamp255(q0, on ? -f1 : 0);
    v[5] = AddClamp255(q1, -a2);
  }
}

// Border extension: every plane of the finished frame gets kBorder replicated pixels on each side
// (value = plane[clamp(y)][clamp(x)]), 8 bytes per thread-item, all items independent.
__global__ void __launch_bounds__(256) BorderKernel(const DevFrameJob *__restrict__ jobs) {
  const DevFrameJob &job = jobs[blockIdx.y];
  for (int pl = 0; pl < 3; ++pl) {
    uint8_t *base = pl == 0 ? job.cur.y : (pl == 1 ? job.cur.u : job.cur.v);
    const int pitch = pl == 0 ? job.pitch_y : job.pitch_c;
    const int w = job.mb_cols * (pl == 0 ? 16 : 8), h = job.mb_rows * (pl == 0 ? 16 : 8);
    const int side_items = h * 8;                     // rows x (4 left + 4 right) granules
    const int vecs = (w + 2 * kBorder) / 8;           // granules per full padded row
    const int total = side_items + vecs * 2 * kBorder;
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < total; t += gridDim.x * blockDim.x) {
      if (t < side_items) {
        const int row = t >> 3, part = t & 7;
        uint8_t *rowp = base + (ptrdiff_t)row * pitch;
        const unsigned v = (part < 4 ? rowp[0] : rowp[w - 1]) * 0x01010101u;
        uint8_t *d = part < 4 ? rowp - kBorder + 8 * part : rowp + w + 8 * (part - 4);
        *reinterpret_cast<uint2 *>(d) = make_uint2(v, v);
      } else {
        const int u = t - side_items;
        const int k = u / vecs, x8 = (u - k * vecs) * 8 - kBorder;  // destination x of the granule
        const int src_row = k < kBorder ? 0 : h - 1;
        const int dst_row = k < kBorder ? k - kBorder : h + (k - kBorder);
        const uint8_t *srow = base + (ptrdiff_t)src_row * pitch;
        uint2 v;
        if (x8 < 0) {
          const unsigned e = srow[0] * 0x01010101u;
          v = make_uint2(e, e);
        } else if (x8 >= w) {
          const unsigned e = srow[w - 1] * 0x01010101u;
          v = make_uint2(e, e);
        } else {
          v = *reinterpret_cast<const uint2 *>(srow + x8);
        }
        *reinterpret_cast<uint2 *>(base + (ptrdiff_t)dst_row * pitch + x8) = v;
      }
    }
  }
}

// ---- loop-filter wavefront -------------------------------------------------------------------
// A frame is cut into G horizontal bands of macroblock rows; one CTA per (frame, band), one warp
// per macroblock row.  CTAs take a ticket at start (atomic counter) and tickets map to
// (band, frame) band-major, so a CTA only ever waits for a CTA holding a SMALLER ticket (the band
// above it in the same frame), i.e. one that is already running or done: no co-residency assumption.
// Inside a band rows synchronise through shared-memory progress counters; the last row of a band
// also publishes to global memory for the first row of the next band (another SM, so that row's
// "above" pixels are read with ld.cg, past the non-coherent L1).
constexpr int kFiltWarps = 4;
constexpr int kMaxBands = 64;
constexpr int kBandStride = 8;
constexpr int kFiltCtasPerSm = 8;  // 72 registers: measured best trade of occupancy (28 warps/SM) against spills

// Streaming multiprocessors of the current device (148 on a B200).
static int SmCount() {
  static int count[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  int &c = count[dev & 63];
  if (c == 0 && cudaDeviceGetAttribute(&c, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) c = 148;
  return c;
}

constexpr int kTilePitch = 20;  // bytes between tile rows, the same for luma and chroma so that
                                // every row/column offset below is a compile-time immediate
struct __align__(16) FiltTile {
  unsigned char bytes[(16 + 8 + 8) * kTilePitch];  // 16 luma rows, 8 U rows, 8 V rows (16 or 8 B
                                                   // used per row; the pad makes row stores
                                                   // conflict-free)
};

__device__ __forceinline__ int LoadFlagAcquire(const int *p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

__global__ void __launch_bounds__(kFiltWarps * 32, kFiltCtasPerSm) FilterKernel(const DevFrameJob *__restrict__ jobs, int n_frames,
                                                                   int n_bands, int *__restrict__ sync, int resident_ctas) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ int s_ticket;
  if (threadIdx.x == 0) s_ticket = atomicAdd(&sync[0], 1);
  __syncthreads();
  // Band-major ticket order: band b of every frame before band b+1 of any.  When the grid exceeds
  // what is resident, the CTAs that hold SM slots are then the bands that can actually run (band
  // b+1 becomes runnable ~1.5 macroblock steps per row after band b), not bands parked on a flag.
  // (When everything is resident at once the order is irrelevant for progress; frame-major then
  // keeps the bands of a frame on neighbouring SMs, which measured ~12 % faster.)
  const bool band_major = n_frames * n_bands > resident_ctas;
  const int band = band_major ? s_ticket / n_frames : s_ticket % n_bands;
  const int frame = band_major ? s_ticket - band * n_frames : s_ticket / n_bands;
  const DevFrameJob &job = jobs[frame];
  const int rows = job.mb_rows, cols = job.mb_cols;
  const int rpb = (rows + n_bands - 1) / n_bands;
  const int r0 = band * rpb, r1 = min(rows, r0 + rpb);
  if (job.lf_level == 0 || r0 >= r1 || JobFailed(job)) return;
  int *gflag = sync + 1 + frame * n_bands;  // gflag[b]: macroblocks < gflag[b] of band b's last row are final
  volatile int *lprog = reinterpret_cast<volatile int *>(smem_raw);
  FiltTile *tiles = reinterpret_cast<FiltTile *>(smem_raw + ((rpb * 4 + 15) & ~15));
  for (int i = threadIdx.x; i < rpb; i += blockDim.x) lprog[i] = 0;
  __syncthreads();

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;  // from lane 0: known to be warp-uniform
  // Everything read from the job is copied to registers here: the pixel stores below are char-typed
  // and would otherwise force the compiler to reload job fields from global memory after each one.
  const bool simple = job.filter_type != 0;
  const int sharpness = job.sharpness;
  const bool key_frame = job.key_frame != 0;
  const vp8r_mb_info *const mbs = job.mbs;
  const bool luma = lane < 16;
  const int n = luma ? 16 : 8;
  const int line = luma ? lane : (lane & 7);
  uint8_t *plane = luma ? job.cur.y : (lane < 24 ? job.cur.u : job.cur.v);
  const int pitch = luma ? job.pitch_y : job.pitch_c;
  const bool lane_on = luma || !simple;
  const int n_words = n / 4;  // own-macroblock words per pixel row
  // Transposition tile of this warp, addressed by integer offsets from the dynamic shared-memory
  // base so that every access stays an LDS/STS (no generic addressing).
  unsigned char *const tb = reinterpret_cast<unsigned char *>(tiles + warp);
  const int tbase = luma ? 0 : (lane < 24 ? 16 : 24) * kTilePitch;
  const int trow_off = tbase + line * kTilePitch;  // this lane's pixel row
  const int tcol_off = tbase + line;               // this lane's pixel column

  for (int lr = warp; lr < r1 - r0; lr += kFiltWarps) {
    const int r = r0 + lr;
    const bool last_of_band = (r == r1 - 1) && (band + 1 < n_bands);
    const bool has_above = r > 0;
    const bool above_local = lr > 0;  // the row above is in this CTA (shared flag) or on another SM
    uint8_t *rowp = plane + (ptrdiff_t)(r * n + line) * pitch;  // this lane's pixel row, x = 0
    const uint8_t *abovep = plane + (ptrdiff_t)(r * n - 4) * pitch + line;  // column `line`, 4 rows up
    const vp8r_mb_info *mbrow = mbs + (size_t)r * cols;
    // software pipeline: words and flags of macroblock c+1 are loaded while c is being filtered
    unsigned nxt[4] = {0, 0, 0, 0};
    // flags of 32 macroblocks at a time, one per lane, handed out by shuffle (a per-macroblock
    // prefetch register was spilled and made the warp wait for the load right away)
    unsigned flags32 = lane < cols ? __ldg(&mbrow[lane].flags) : 0u;
    if (lane_on) {
      if (luma) {
        const uint4 t = *reinterpret_cast<const uint4 *>(rowp);
        nxt[0] = t.x; nxt[1] = t.y; nxt[2] = t.z; nxt[3] = t.w;
      } else {
        const uint2 t = *reinterpret_cast<const uint2 *>(rowp);
        nxt[0] = t.x; nxt[1] = t.y;
      }
    }
    unsigned carry = 0;    // columns n-4..n-1 of the previous macroblock of this pixel row
    int a4n[4] = {0, 0, 0, 0};  // rows above of macroblock c, prefetched during c-1 when allowed
    int gseen = 0;              // last value read from the band above's global progress word
    bool have_above = false;

    for (int c = 0; c < cols; ++c) {
      unsigned cur[4] = {nxt[0], nxt[1], nxt[2], nxt[3]};
      if (c && (c & 31) == 0) flags32 = c + lane < cols ? __ldg(&mbrow[c + lane].flags) : 0u;
      const unsigned flags = __shfl_sync(0xffffffffu, flags32, c & 31);
      if (c + 1 < cols) {
        if (lane_on) {
          const uint8_t *np = rowp + (c + 1) * n;
          if (luma) {
            const uint4 t = *reinterpret_cast<const uint4 *>(np);
            nxt[0] = t.x; nxt[1] = t.y; nxt[2] = t.z; nxt[3] = t.w;
          } else {
            const uint2 t = *reinterpret_cast<const uint2 *>(np);
            nxt[0] = t.x; nxt[1] = t.y;
          }
        }
      }
      // Non-blocking sample of the progress of the row above; consumed at the end of the
      // iteration to decide whether the next macroblock's rows above can be fetched early.
      int seen = 0;
      if (has_above) seen = above_local ? lprog[lr - 1] : gseen;  // cross-SM progress: cached, see below

      const int level = (flags >> VP8R_MB_LF_SHIFT) & 63;
      if (level != 0) {
        const bool inner = (flags & VP8R_MB_LF_INNER) != 0;
        const LfLimits lim = MakeLimits(level, sharpness, key_frame);
        const int need = min(c + 2, cols);
        uint8_t *mbp = plane + (ptrdiff_t)(r * n) * pitch + c * n;

        if (lane_on) {
          // ---- vertical edges: lane = pixel row; v[0..3] = carry (previous MB), v[4..] = own ----
          int v[20];
          v[0] = carry & 0xff; v[1] = (carry >> 8) & 0xff; v[2] = (carry >> 16) & 0xff; v[3] = carry >> 24;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            if (k < n_words) {
              v[4 + 4 * k] = cur[k] & 0xff; v[5 + 4 * k] = (cur[k] >> 8) & 0xff;
              v[6 + 4 * k] = (cur[k] >> 16) & 0xff; v[7 + 4 * k] = cur[k] >> 24;
            }
          }
          if (c > 0) LfEdge<true>(v, lim, simple);
          if (inner) {
#pragma unroll
            for (int e = 1; e < 4; ++e)
              if (e < n_words) LfEdge<false>(v + 4 * e, lim, simple);
          }
          if (c > 0)  // columns n-4..n-1 of the previous macroblock are final for this row now
            *reinterpret_cast<unsigned *>(rowp + c * n - 4) =
                (unsigned)v[0] | ((unsigned)v[1] << 8) | ((unsigned)v[2] << 16) | ((unsigned)v[3] << 24);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            if (k < n_words)
              *reinterpret_cast<unsigned *>(tb + trow_off + 4 * k) =
                  (unsigned)v[4 + 4 * k] | ((unsigned)v[5 + 4 * k] << 8) | ((unsigned)v[6 + 4 * k] << 16) |
                  ((unsigned)v[7 + 4 * k] << 24);
        }
        __syncwarp();

        int a4[4] = {a4n[0], a4n[1], a4n[2], a4n[3]};
        if (has_above && !have_above) {  // not prefetched: wait for the row above, then fetch
          // back off in proportion to how far behind the row above still is (>= ~1 us per
          // macroblock), so rows that cannot start yet do not eat issue slots polling
          if (above_local) {
            for (int got = lprog[lr - 1]; got < need; got = lprog[lr - 1]) __nanosleep(min(250 + 700 * (need - got - 1), 20000));
            __threadfence_block();
          } else {
            // The band above publishes in strides of kBandStride macroblocks, so one successful
            // poll usually covers the next several macroblocks (and their prefetches).
            for (gseen = LoadFlagAcquire(&gflag[band - 1]); gseen < need; gseen = LoadFlagAcquire(&gflag[band - 1]))
              __nanosleep(min(200 + 600 * (need - gseen - 1), 20000));
          }
          if (lane_on) {
#pragma unroll
            for (int y = 0; y < 4; ++y) a4[y] = __ldcg(abovep + c * n + (ptrdiff_t)y * pitch);
          }
        }
        if (lane_on) {
          // ---- horizontal edges: lane = pixel column; v[0..3] = rows above, v[4..] = own rows ----
          int v[20];
          v[0] = a4[0]; v[1] = a4[1]; v[2] = a4[2]; v[3] = a4[3];
#pragma unroll
          for (int y = 0; y < 16; ++y)
            if (y < n) v[4 + y] = tb[tcol_off + y * kTilePitch];
          if (has_above) LfEdge<true>(v, lim, simple);
          if (inner) {
#pragma unroll
            for (int e = 1; e < 4; ++e)
              if (e < n_words) LfEdge<false>(v + 4 * e, lim, simple);
          }
          if (has_above) {
#pragma unroll
            for (int y = 1; y < 4; ++y) mbp[line + (ptrdiff_t)(y - 4) * pitch] = (uint8_t)v[y];
          }
#pragma unroll
          for (int y = 0; y < 16; ++y)
            if (y < n) tb[tcol_off + y * kTilePitch] = (unsigned char)v[4 + y];
        }
        __syncwarp();
        if (lane_on) {
          // back to lane = pixel row: write the macroblock row out, keep its last word as carry
          unsigned *outp = reinterpret_cast<unsigned *>(rowp + c * n);
          const unsigned *tr = reinterpret_cast<const unsigned *>(tb + trow_off);
          if (luma) {
            uint4 o = make_uint4(tr[0], tr[1], tr[2], tr[3]);
            *reinterpret_cast<uint4 *>(outp) = o;
            carry = o.w;
          } else {
            uint2 o = make_uint2(tr[0], tr[1]);
            *reinterpret_cast<uint2 *>(outp) = o;
            carry = o.y;
          }
        }
      } else {
        carry = luma ? cur[3] : cur[1];  // untouched macroblock: just hand its last columns on
      }

      // Rows above of the next macroblock: fetch now if the row above is already far enough, so
      // the loads overlap the next vertical phase (a row that runs too close behind its
      // predecessor waits above, drops back, and from then on always finds them ready).
      have_above = false;
      if (has_above && c + 1 < cols && seen >= min(c + 3, cols)) {
        if (above_local) __threadfence_block();
        if (lane_on) {
#pragma unroll
          for (int y = 0; y < 4; ++y) a4n[y] = __ldcg(abovep + (c + 1) * n + (ptrdiff_t)y * pitch);
        }
        have_above = true;
      }

      // Publish.  Same-CTA consumers: block-scope fence, shared flag, every macroblock.  The next
      // band (another SM) needs a device-scope fence, which costs ~2.5k cycles when stores are in
      // flight: it is paid once per kBandStride macroblocks, otherwise the last row of every band
      // would run at less than half the speed of the others and throttle all rows below it.
      if (last_of_band && (c % kBandStride) == kBandStride - 1) {
        __threadfence();
        __syncwarp();
        if (lane == 0) atomicExch(&gflag[band], c + 1);  // macroblocks <= c are final
      } else {
        __threadfence_block();
      }
      __syncwarp();
      if (lane == 0) lprog[lr] = c + 1;
    }
    if (last_of_band) {
      __threadfence();
      __syncwarp();
      if (lane == 0) atomicExch(&gflag[band], cols);
    }
  }
}

cudaError_t LaunchFilter(const DevFrameJob *jobs, int n_frames, int max_rows, int *sync, int sync_ints,
                         cudaStream_t st, const FilterGroup *groups, int n_groups) {
  if (groups && n_groups > 0) {
    cudaError_t e = LaunchFilterSwar(jobs, groups, n_groups, max_rows, sync, sync_ints, st);
    return e;
  }
  // Bands: one warp per macroblock row (8-warp CTAs pack 4 per SM at 64 registers); with few frames
  // in the batch, thinner bands put more SMs to work.
  int n_bands = (max_rows + kFiltWarps - 1) / kFiltWarps;
  while (n_bands < kMaxBands && n_frames * n_bands < SmCount() * 2 && (max_rows + n_bands) / (n_bands + 1) >= 3) ++n_bands;
  if (n_bands > kMaxBands) n_bands = kMaxBands;
  if (1 + n_frames * n_bands > sync_ints) return cudaErrorInvalidValue;
  cudaError_t e = cudaMemsetAsync(sync, 0, sizeof(int) * (1 + (size_t)n_frames * n_bands), st);
  if (e != cudaSuccess) return e;
  const int rpb = (max_rows + n_bands - 1) / n_bands;
  size_t smem = ((size_t(rpb) * 4 + 15) & ~size_t(15)) + sizeof(FiltTile) * kFiltWarps;
  FilterKernel<<<n_frames * n_bands, kFiltWarps * 32, smem, st>>>(jobs, n_frames, n_bands, sync, SmCount() * kFiltCtasPerSm);
  e = cudaGetLastError();
  return e;
}

cudaError_t LaunchBorder(const DevFrameJob *jobs, int n_frames, cudaStream_t st) {
  BorderKernel<<<dim3(8, n_frames), 256, 0, st>>>(jobs);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// checksum of the cropped I420 image: s1 = sum(b_i), s2 = sum((i+1) * b_i), both mod 2^32,
// with i the byte index in the cropped Y,U,V stream (src/yuv.cc:6-28 order).
// ------------------------------------------------------------------------------------------
__global__ void ChecksumKernel(const DevFrameJob *__restrict__ jobs) {
  const DevFrameJob &job = jobs[blockIdx.y];
  if (!job.checksum) return;
  const int w = job.width, h = job.height, cw = (w + 1) / 2, ch = (h + 1) / 2;
  const unsigned ny = (unsigned)w * h, nc = (unsigned)cw * ch, total = ny + 2 * nc;
  unsigned s1 = 0, s2 = 0;
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    unsigned b;
    if (i < ny) {
      unsigned y = i / w, x = i - y * w;
      b = job.cur.y[(size_t)y * job.pitch_y + x];
    } else {
      unsigned k = i - ny;
      const uint8_t *pl = job.cur.u;
      if (k >= nc) {
        k -= nc;
        pl = job.cur.v;
      }
      unsigned y = k / cw, x = k - y * cw;
      b = pl[(size_t)y * job.pitch_c + x];
    }
    s1 += b;
    s2 += (i + 1) * b;
  }
  for (int o = 16; o; o >>= 1) {
    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    s2 += __shfl_xor_sync(0xffffffffu, s2, o);
  }
  if ((threadIdx.x & 31) == 0) {
    // low and high words are accumulated independently (mod 2^32 each) with two 32-bit atomics
    unsigned *out = reinterpret_cast<unsigned *>(job.checksum);
    atomicAdd(out, s1);
    atomicAdd(out + 1, s2);
  }
}

// ------------------------------------------------------------------------------------------
// crop + pack: YUV<WRITE>::WriteFrame (src/yuv.cc:6-28) on the device.  Each job's cropped Y, U, V
// planes are written back to back at job.pack_dst, so one contiguous copy moves any number of frames.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) PackKernel(const DevFrameJob *__restrict__ jobs) {
  const DevFrameJob &job = jobs[blockIdx.y];
  uint8_t *dst = job.pack_dst;
  if (!dst) return;
  const int w = job.width, h = job.height, cw = (w + 1) / 2, ch = (h + 1) / 2;
  const uint8_t *py = job.cur.y, *pu = job.cur.u, *pv = job.cur.v;
  const int pitch_y = job.pitch_y, pitch_c = job.pitch_c;
  // 4 pixels per thread-item where the row allows it (source rows are 16-byte aligned; the
  // destination is byte-packed, so it is written bytewise unless w % 4 == 0).
  const int wy4 = (w + 3) / 4, wc4 = (cw + 3) / 4;
  const int items_y = wy4 * h, items_c = wc4 * ch;
  const int total = items_y + 2 * items_c;
  const bool nv12 = job.pack_layout == VP8R_LAYOUT_NV12;
  const bool y_vec = (w & 3) == 0, c_vec = !nv12 && (cw & 3) == 0 && ((size_t)w * h & 3) == 0 && ((size_t)cw * ch & 3) == 0;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < total; t += gridDim.x * blockDim.x) {
    const uint8_t *src;
    uint8_t *d;
    int x, n;
    bool vec;
    if (t < items_y) {
      const int row = t / wy4;
      x = (t - row * wy4) * 4;
      src = py + (size_t)row * pitch_y + x;
      d = dst + (size_t)row * w + x;
      n = min(4, w - x);
      vec = y_vec;
    } else {
      int u = t - items_y;
      const int plane = u >= items_c;
      if (plane) u -= items_c;
      const int row = u / wc4;
      x = (u - row * wc4) * 4;
      src = (plane ? pv : pu) + (size_t)row * pitch_c + x;
      d = dst + (size_t)w * h + (size_t)plane * cw * ch + (size_t)row * cw + x;
      n = min(4, cw - x);
      vec = c_vec;
      if (nv12) {  // U and V samples alternate: this item's bytes go to every second byte of the UV plane
        const unsigned v = *reinterpret_cast<const unsigned *>(src);
        uint8_t *uv = dst + (size_t)w * h + ((size_t)row * cw + x) * 2 + plane;
        for (int k = 0; k < n; ++k) uv[2 * k] = (uint8_t)(v >> (8 * k));
        continue;
      }
    }
    const unsigned v = *reinterpret_cast<const unsigned *>(src);
    if (vec && (((size_t)d & 3) == 0)) {
      *reinterpret_cast<unsigned *>(d) = v;
    } else {
      for (int k = 0; k < n; ++k) d[k] = (uint8_t)(v >> (8 * k));
    }
  }
}

// ------------------------------------------------------------------------------------------
// crop + BT.601 limited-range YUV -> RGB (vp8r_read_batch_device, VP8R_LAYOUT_RGB24 / _RGB_PLANAR).
// Memory-bound (1.5 B read, 3 B written per pixel): one thread converts a strip of 16 x 2 pixels, which share 8
// chroma samples, so the chroma terms are computed once per sample and every source row is one 128-bit load
// (surface rows are 16-byte aligned and padded to whole macroblocks, so the loads never leave the surface).
// ------------------------------------------------------------------------------------------
constexpr int kRgbStripW = 16;

// Stores the first n of the 4*NW bytes of w[] at d: 128-bit stores for a whole strip at a 16-byte aligned address
// (every strip of a frame whose width is a multiple of 16, at an aligned destination), 32-bit stores at a 4-byte
// aligned one, bytes otherwise (odd widths, the last strip of a row).
// A strip of two words (StageSourceKernel's chroma) takes one 64-bit store at an 8-byte aligned address instead.
template <int NW>
__device__ __forceinline__ void StoreStrip(uint8_t *d, const unsigned (&w)[NW], int n) {
  if (NW % 4 == 0 && n == 4 * NW && ((size_t)d & 15) == 0) {
#pragma unroll
    for (int k = 0; k + 3 < NW; k += 4) *reinterpret_cast<uint4 *>(d + 4 * k) = make_uint4(w[k], w[k + 1], w[k + 2], w[k + 3]);
  } else if (NW == 2 && n == 8 && ((size_t)d & 7) == 0) {
    *reinterpret_cast<uint2 *>(d) = make_uint2(w[0], w[NW - 1]);
  } else if (n == 4 * NW && ((size_t)d & 3) == 0) {
#pragma unroll
    for (int k = 0; k < NW; ++k) *reinterpret_cast<unsigned *>(d + 4 * k) = w[k];
  } else {
#pragma unroll
    for (int k = 0; k < 4 * NW; ++k)
      if (k < n) d[k] = (uint8_t)(w[k >> 2] >> (8 * (k & 3)));
  }
}

__global__ void __launch_bounds__(256) ConvertRgbKernel(const DevFrameJob *__restrict__ jobs) {
  const DevFrameJob &job = jobs[blockIdx.y];
  uint8_t *dst = job.pack_dst;
  if (!dst) return;
  const bool planar = job.pack_layout == VP8R_LAYOUT_RGB_PLANAR;
  const int w = job.width, h = job.height;
  const int strips = (w + kRgbStripW - 1) / kRgbStripW, items = strips * ((h + 1) / 2);
  const size_t plane = (size_t)w * h;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < items; t += gridDim.x * blockDim.x) {
    const int pair = t / strips;
    const int x = (t - pair * strips) * kRgbStripW, y = 2 * pair;
    const int n = min(kRgbStripW, w - x);
    const uint2 u8 = *reinterpret_cast<const uint2 *>(job.cur.u + (size_t)pair * job.pitch_c + x / 2);
    const uint2 v8 = *reinterpret_cast<const uint2 *>(job.cur.v + (size_t)pair * job.pitch_c + x / 2);
    // per chroma sample: the rounding constant and the U / V terms of each channel
    int rc[8], gc[8], bc[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int d = (int)(((k < 4 ? u8.x : u8.y) >> (8 * (k & 3))) & 255) - 128;
      const int e = (int)(((k < 4 ? v8.x : v8.y) >> (8 * (k & 3))) & 255) - 128;
      rc[k] = 409 * e + 128;
      gc[k] = 128 - 100 * d - 208 * e;
      bc[k] = 516 * d + 128;
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      if (y + r >= h) break;
      const uint4 yv = *reinterpret_cast<const uint4 *>(job.cur.y + (size_t)(y + r) * job.pitch_y + x);
      const unsigned yw[4] = {yv.x, yv.y, yv.z, yv.w};
      int R[16], G[16], B[16];
#pragma unroll
      for (int p = 0; p < 16; ++p) {
        const int c = 298 * ((int)((yw[p >> 2] >> (8 * (p & 3))) & 255) - 16);
        R[p] = (c + rc[p >> 1]) >> 8;
        G[p] = (c + gc[p >> 1]) >> 8;
        B[p] = (c + bc[p >> 1]) >> 8;
      }
      const size_t row = (size_t)(y + r) * w + x;
      if (planar) {
        unsigned wr[4], wg[4], wb[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          wr[q] = PackSat4(R[4 * q], R[4 * q + 1], R[4 * q + 2], R[4 * q + 3]);
          wg[q] = PackSat4(G[4 * q], G[4 * q + 1], G[4 * q + 2], G[4 * q + 3]);
          wb[q] = PackSat4(B[4 * q], B[4 * q + 1], B[4 * q + 2], B[4 * q + 3]);
        }
        StoreStrip(dst + row, wr, n);
        StoreStrip(dst + plane + row, wg, n);
        StoreStrip(dst + 2 * plane + row, wb, n);
      } else {
        unsigned o[12];  // four pixels R,G,B,R G,B,R,G B,R,G,B per three words
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          o[3 * q] = PackSat4(R[4 * q], G[4 * q], B[4 * q], R[4 * q + 1]);
          o[3 * q + 1] = PackSat4(G[4 * q + 1], B[4 * q + 1], R[4 * q + 2], G[4 * q + 2]);
          o[3 * q + 2] = PackSat4(B[4 * q + 2], R[4 * q + 3], G[4 * q + 3], B[4 * q + 3]);
        }
        StoreStrip(dst + 3 * row, o, 3 * n);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// Encoder input from device memory (vp8r_encode_*_device, vp8r_convert_to_i420_device): each job's source frame
// (job.stage_src: width x height in job.pack_layout, any byte alignment) becomes I420 by the BT.601 formula of
// include/vp8r.h, written to the planes enc_src[0..2] (pitches enc_src_pitch_y / _c) over stage_w x stage_h luma
// pixels.  Source coordinates are clamped to the picture: with stage_w x stage_h the macroblock-aligned size this is
// PadToMacroblocks (rt/engine.cu) of the cropped I420 image, with the cropped size it is that image.  Same mapping as
// ConvertRgbKernel: one thread per 16 x 2 luma strip and its 8 chroma samples.  Memory-bound (I420 / NV12: about
// 1.5 B read and written per pixel; RGB: 3 B read, 1.5 B written).
// ------------------------------------------------------------------------------------------
// 4*NW bytes at p, any alignment: 128-bit loads at a 16-byte aligned address, 32-bit loads at a 4-byte aligned one,
// otherwise NW+1 aligned words joined by funnel shifts.  Every word read holds at least one of the 4*NW bytes, so the
// loads stay inside the pages of the buffer that holds them.
template <int NW>
__device__ __forceinline__ void LoadBytes(const uint8_t *p, unsigned (&w)[NW]) {
  const unsigned r = (unsigned)(size_t)p & 3;
  if (NW % 4 == 0 && ((size_t)p & 15) == 0) {
#pragma unroll
    for (int k = 0; k + 3 < NW; k += 4) {
      const uint4 v = *reinterpret_cast<const uint4 *>(p + 4 * k);
      w[k] = v.x, w[k + 1] = v.y, w[k + 2] = v.z, w[k + 3] = v.w;
    }
  } else if (r == 0) {
#pragma unroll
    for (int k = 0; k < NW; ++k) w[k] = reinterpret_cast<const unsigned *>(p)[k];
  } else {
    const unsigned *a = reinterpret_cast<const unsigned *>(p - r);
    unsigned lo = a[0];
#pragma unroll
    for (int k = 0; k < NW; ++k) {
      const unsigned hi = a[k + 1];
      w[k] = __funnelshift_r(lo, hi, 8 * r);
      lo = hi;
    }
  }
}

__device__ __forceinline__ int ByteOf(const unsigned *w, int i) { return (int)((w[i >> 2] >> (8 * (i & 3))) & 255); }

// BT.601 limited range (include/vp8r.h): luma of one pixel, chroma of the sums of a 2x2 block's channels.
__device__ __forceinline__ int LumaOf(int r, int g, int b) { return ((66 * r + 129 * g + 25 * b + 128) >> 8) + 16; }
__device__ __forceinline__ int ChromaU(int sr, int sg, int sb) {
  return ((-38 * ((sr + 2) >> 2) - 74 * ((sg + 2) >> 2) + 112 * ((sb + 2) >> 2) + 128) >> 8) + 128;
}
__device__ __forceinline__ int ChromaV(int sr, int sg, int sb) {
  return ((112 * ((sr + 2) >> 2) - 94 * ((sg + 2) >> 2) - 18 * ((sb + 2) >> 2) + 128) >> 8) + 128;
}

__device__ __forceinline__ void RgbAt(const uint8_t *src, bool planar, int w, int h, int x, int y, int &r, int &g, int &b) {
  const size_t o = (size_t)y * w + x;
  if (planar) {
    const size_t plane = (size_t)w * h;
    r = src[o], g = src[plane + o], b = src[2 * plane + o];
  } else {
    r = src[3 * o], g = src[3 * o + 1], b = src[3 * o + 2];
  }
}

// One instance per layout (a batch has one): each path gets the registers it needs.
template <int kLayout>
__global__ void __launch_bounds__(256) StageSourceKernel(const DevFrameJob *__restrict__ jobs) {
  const DevFrameJob &job = jobs[blockIdx.y];
  const uint8_t *src = job.stage_src;
  if (!src) return;
  constexpr int layout = kLayout;
  const int w = job.width, h = job.height, cw = (w + 1) / 2, ch = (h + 1) / 2;
  const int dw = job.stage_w, dh = job.stage_h, dcw = (dw + 1) / 2;
  uint8_t *dy = const_cast<uint8_t *>(job.enc_src[0]), *du = const_cast<uint8_t *>(job.enc_src[1]),
          *dv = const_cast<uint8_t *>(job.enc_src[2]);
  const int py = job.enc_src_pitch_y, pc = job.enc_src_pitch_c;
  const size_t plane = (size_t)w * h, cplane = (size_t)cw * ch;
  const int strips = (dw + 15) / 16, items = strips * ((dh + 1) / 2);
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < items; t += gridDim.x * blockDim.x) {
    const int pair = t / strips;
    const int x = (t - pair * strips) * 16, y = 2 * pair, cx = x / 2;
    // no coordinate of the strip, its 2x2 blocks or its chroma samples needs a clamp
    const bool inside = x + 16 <= w && y + 1 < h;
    const int cy = min(pair, ch - 1);
    unsigned yw[2][4], uw[2], vw[2];
    if constexpr (layout == VP8R_LAYOUT_I420 || layout == VP8R_LAYOUT_NV12) {
      if (inside) {
        LoadBytes(src + (size_t)y * w + x, yw[0]);
        LoadBytes(src + (size_t)(y + 1) * w + x, yw[1]);
        if constexpr (layout == VP8R_LAYOUT_I420) {
          LoadBytes(src + plane + (size_t)cy * cw + cx, uw);
          LoadBytes(src + plane + cplane + (size_t)cy * cw + cx, vw);
        } else {
          unsigned uv[4];
          LoadBytes(src + plane + 2 * ((size_t)cy * cw + cx), uv);
          uw[0] = __byte_perm(uv[0], uv[1], 0x6420), vw[0] = __byte_perm(uv[0], uv[1], 0x7531);
          uw[1] = __byte_perm(uv[2], uv[3], 0x6420), vw[1] = __byte_perm(uv[2], uv[3], 0x7531);
        }
      } else {
#pragma unroll
        for (int r = 0; r < 2; ++r) {
          const uint8_t *row = src + (size_t)min(y + r, h - 1) * w;
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            unsigned v = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k) v |= (unsigned)row[min(x + 4 * q + k, w - 1)] << (8 * k);
            yw[r][q] = v;
          }
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          unsigned u = 0, v = 0;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const size_t o = (size_t)cy * cw + min(cx + 4 * q + k, cw - 1);
            const size_t ou = layout == VP8R_LAYOUT_I420 ? plane + o : plane + 2 * o;
            const size_t ov = layout == VP8R_LAYOUT_I420 ? plane + cplane + o : plane + 2 * o + 1;
            u |= (unsigned)src[ou] << (8 * k);
            v |= (unsigned)src[ov] << (8 * k);
          }
          uw[q] = u, vw[q] = v;
        }
      }
    } else {
      constexpr bool planar = layout == VP8R_LAYOUT_RGB_PLANAR;
      int sr[8], sg[8], sb[8];  // channel sums of the strip's 2x2 blocks (inside only)
#pragma unroll
      for (int k = 0; k < 8; ++k) sr[k] = sg[k] = sb[k] = 0;
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        int Y[16];
        if (inside) {
          const size_t o = (size_t)(y + r) * w + x;
          unsigned a[12];  // RGB24: the strip's 48 bytes; planar: its 16 R, then 16 G, then 16 B bytes
          if (planar) {
            unsigned t[4];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
              LoadBytes(src + c * plane + o, t);
#pragma unroll
              for (int k = 0; k < 4; ++k) a[4 * c + k] = t[k];
            }
          } else {
            LoadBytes(src + 3 * o, a);
          }
#pragma unroll
          for (int p = 0; p < 16; ++p) {
            const int R = ByteOf(a, planar ? p : 3 * p), G = ByteOf(a, planar ? 16 + p : 3 * p + 1),
                      B = ByteOf(a, planar ? 32 + p : 3 * p + 2);
            sr[p >> 1] += R, sg[p >> 1] += G, sb[p >> 1] += B;
            Y[p] = LumaOf(R, G, B);
          }
        } else {
#pragma unroll
          for (int p = 0; p < 16; ++p) {
            int R, G, B;
            RgbAt(src, planar, w, h, min(x + p, w - 1), min(y + r, h - 1), R, G, B);
            Y[p] = LumaOf(R, G, B);
          }
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) yw[r][q] = PackSat4(Y[4 * q], Y[4 * q + 1], Y[4 * q + 2], Y[4 * q + 3]);
      }
      if (!inside) {  // chroma sample (i, j) averages pixels (2i+a, 2j+b), i and j clamped first, then the pixels
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int i = min(cx + k, cw - 1);
          sr[k] = sg[k] = sb[k] = 0;
#pragma unroll
          for (int a = 0; a < 4; ++a) {
            int r, g, b;
            RgbAt(src, planar, w, h, min(2 * i + (a & 1), w - 1), min(2 * cy + (a >> 1), h - 1), r, g, b);
            sr[k] += r, sg[k] += g, sb[k] += b;
          }
        }
      }
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        uw[q] = PackSat4(ChromaU(sr[4 * q], sg[4 * q], sb[4 * q]), ChromaU(sr[4 * q + 1], sg[4 * q + 1], sb[4 * q + 1]),
                         ChromaU(sr[4 * q + 2], sg[4 * q + 2], sb[4 * q + 2]), ChromaU(sr[4 * q + 3], sg[4 * q + 3], sb[4 * q + 3]));
        vw[q] = PackSat4(ChromaV(sr[4 * q], sg[4 * q], sb[4 * q]), ChromaV(sr[4 * q + 1], sg[4 * q + 1], sb[4 * q + 1]),
                         ChromaV(sr[4 * q + 2], sg[4 * q + 2], sb[4 * q + 2]), ChromaV(sr[4 * q + 3], sg[4 * q + 3], sb[4 * q + 3]));
      }
    }
    const int n = min(16, dw - x), nc = min(8, dcw - cx);
    StoreStrip(dy + (size_t)y * py + x, yw[0], n);
    if (y + 1 < dh) StoreStrip(dy + (size_t)(y + 1) * py + x, yw[1], n);
    StoreStrip(du + (size_t)pair * pc + cx, uw, nc);
    StoreStrip(dv + (size_t)pair * pc + cx, vw, nc);
  }
}

// ------------------------------------------------------------------------------------------
// host -> device staging by the SMs (zero-copy reads of pinned host memory)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) CopyKernel(uint4 *__restrict__ dst, const uint4 *__restrict__ src, size_t n16) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) dst[i] = src[i];
}

constexpr int kGatherChunk = 16 * 1024;  // bytes per CTA
__global__ void __launch_bounds__(256) GatherKernel(const DevFrameJob *__restrict__ jobs) {
  const DevFrameJob &job = jobs[blockIdx.y];
  const size_t bytes = job.h2d_bytes;
  const size_t begin = (size_t)blockIdx.x * kGatherChunk;
  if (begin >= bytes) return;
  const size_t end = min(bytes, begin + (size_t)kGatherChunk);
  const uint4 *src = reinterpret_cast<const uint4 *>(job.h2d_src);
  uint4 *dst = reinterpret_cast<uint4 *>(job.h2d_dst);
  // 4 loads in flight per thread: PCIe reads need depth, not width
  for (size_t i = begin / 16 + threadIdx.x; i < (end + 15) / 16; i += 256) dst[i] = src[i];
}

cudaError_t LaunchCopy(void *dst, const void *src_pinned, size_t bytes, cudaStream_t st) {
  const size_t n16 = (bytes + 15) / 16;
  if (n16 == 0) return cudaSuccess;
  const int grid = (int)std::min<size_t>((n16 + 255) / 256, size_t(SmCount()) * 4);
  CopyKernel<<<grid, 256, 0, st>>>(static_cast<uint4 *>(dst), static_cast<const uint4 *>(src_pinned), n16);
  return cudaGetLastError();
}

cudaError_t LaunchGather(const DevFrameJob *jobs, int n_frames, size_t max_bytes, cudaStream_t st) {
  if (max_bytes == 0 || n_frames == 0) return cudaSuccess;
  dim3 grid((unsigned)((max_bytes + kGatherChunk - 1) / kGatherChunk), n_frames);
  GatherKernel<<<grid, 256, 0, st>>>(jobs);
  return cudaGetLastError();
}

cudaError_t LaunchPack(const DevFrameJob *jobs, int n_frames, cudaStream_t st) {
  dim3 grid(48, n_frames);
  PackKernel<<<grid, 256, 0, st>>>(jobs);
  return cudaGetLastError();
}

cudaError_t LaunchConvertRgb(const DevFrameJob *jobs, int n_frames, int max_w, int max_h, cudaStream_t st) {
  const int items = (max_w + kRgbStripW - 1) / kRgbStripW * ((max_h + 1) / 2);
  dim3 grid((unsigned)std::max(1, std::min(48, (items + 255) / 256)), n_frames);
  ConvertRgbKernel<<<grid, 256, 0, st>>>(jobs);
  return cudaGetLastError();
}

cudaError_t LaunchStageSource(const DevFrameJob *jobs, int n_frames, int layout, int max_w, int max_h, cudaStream_t st) {
  const int items = (max_w + 15) / 16 * ((max_h + 1) / 2);
  dim3 grid((unsigned)std::max(1, std::min(48, (items + 255) / 256)), n_frames);
  switch (layout) {
    case VP8R_LAYOUT_I420: StageSourceKernel<VP8R_LAYOUT_I420><<<grid, 256, 0, st>>>(jobs); break;
    case VP8R_LAYOUT_NV12: StageSourceKernel<VP8R_LAYOUT_NV12><<<grid, 256, 0, st>>>(jobs); break;
    case VP8R_LAYOUT_RGB24: StageSourceKernel<VP8R_LAYOUT_RGB24><<<grid, 256, 0, st>>>(jobs); break;
    case VP8R_LAYOUT_RGB_PLANAR: StageSourceKernel<VP8R_LAYOUT_RGB_PLANAR><<<grid, 256, 0, st>>>(jobs); break;
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

cudaError_t LaunchChecksum(const DevFrameJob *jobs, int n_frames, cudaStream_t st) {
  dim3 grid(64, n_frames);
  ChecksumKernel<<<grid, 256, 0, st>>>(jobs);
  return cudaGetLastError();
}

}  // namespace vp8r
