// VP8 loop-filter edge arithmetic on FOUR pixel lines per 32-bit register.
//
// A "line" is the run of eight pixels p3 p2 p1 p0 | q0 q1 q2 q3 across an edge (src/filter.cc:7-67 of the
// reference).  Every argument word below carries the same pixel position of four neighbouring lines, one
// per byte.  Decisions (interior limit, high edge variance, edge limit) are taken on bytes with
// VABSDIFF4 and unsigned 16x2 maxima (the upper byte of a 16-bit lane orders the lane); the filter taps
// run on two 16x2 registers per word ("even" = lines 0 and 2, "odd" = lines 1 and 3) with every
// intermediate biased to be non-negative, so plain 32-bit adds and multiplies never carry between lanes.
// Results are bit-exact with the scalar formulation, including the reference's clamps.
//
// The header compiles for the device (native SIMD instructions of sm_100a) and for the host (emulated
// primitives), so that tests/native/lf_swar_test.cc can compare it exhaustively with the scalar filter
// without a GPU.
#ifndef VP8R_CUDA_LF_SWAR_H_
#define VP8R_CUDA_LF_SWAR_H_

#include <stdint.h>

#if defined(__CUDACC__)
#define VP8R_HD __host__ __device__ __forceinline__
#else
#define VP8R_HD inline
#endif

namespace vp8r {
namespace swar {

// ---- primitives -------------------------------------------------------------------------------------
#if defined(__CUDA_ARCH__)
VP8R_HD uint32_t Absd4(uint32_t a, uint32_t b) { return __vabsdiffu4(a, b); }
VP8R_HD uint32_t Prmt(uint32_t a, uint32_t b, uint32_t sel) {
  uint32_t d;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
  return d;
}
VP8R_HD uint32_t UMax2(uint32_t a, uint32_t b) { return __vmaxu2(a, b); }
VP8R_HD uint32_t UMin2(uint32_t a, uint32_t b) { return __vminu2(a, b); }
VP8R_HD uint32_t UMax3(uint32_t a, uint32_t b, uint32_t c) { return __vimax3_u16x2(a, b, c); }
// clamp(a + b, 0, c) per signed 16-bit lane, the add wrapping inside the lane: one VIADDMNMX.S16x2.RELU
VP8R_HD uint32_t AddClamp2(uint32_t a, uint32_t b, uint32_t c) { return __viaddmin_s16x2_relu(a, b, c); }
VP8R_HD uint32_t Add2(uint32_t a, uint32_t b) { return __vadd2(a, b); }  // per lane, wrapping inside the lane
#else
VP8R_HD uint32_t Absd4(uint32_t a, uint32_t b) {
  uint32_t r = 0;
  for (int i = 0; i < 4; ++i) {
    int x = (a >> (8 * i)) & 0xff, y = (b >> (8 * i)) & 0xff;
    r |= uint32_t(x > y ? x - y : y - x) << (8 * i);
  }
  return r;
}
VP8R_HD uint32_t Prmt(uint32_t a, uint32_t b, uint32_t sel) {
  const uint64_t src = (uint64_t(b) << 32) | a;
  uint32_t r = 0;
  for (int i = 0; i < 4; ++i) {
    const uint32_t s = (sel >> (4 * i)) & 15;
    uint32_t byte = uint32_t(src >> (8 * (s & 7))) & 0xff;
    if (s & 8) byte = (byte & 0x80) ? 0xff : 0x00;
    r |= byte << (8 * i);
  }
  return r;
}
VP8R_HD uint32_t Lanes(uint32_t lo, uint32_t hi) { return (lo & 0xffff) | (hi << 16); }
VP8R_HD uint32_t UMax2(uint32_t a, uint32_t b) {
  uint32_t l = (a & 0xffff) > (b & 0xffff) ? (a & 0xffff) : (b & 0xffff), h = (a >> 16) > (b >> 16) ? (a >> 16) : (b >> 16);
  return Lanes(l, h);
}
VP8R_HD uint32_t UMin2(uint32_t a, uint32_t b) {
  uint32_t l = (a & 0xffff) < (b & 0xffff) ? (a & 0xffff) : (b & 0xffff), h = (a >> 16) < (b >> 16) ? (a >> 16) : (b >> 16);
  return Lanes(l, h);
}
VP8R_HD uint32_t UMax3(uint32_t a, uint32_t b, uint32_t c) { return UMax2(UMax2(a, b), c); }
VP8R_HD uint32_t Add2(uint32_t a, uint32_t b) { return Lanes(uint16_t(a + b), uint16_t((a >> 16) + (b >> 16))); }
VP8R_HD uint32_t AddClamp2(uint32_t a, uint32_t b, uint32_t c) {
  int16_t l = int16_t(uint16_t(a) + uint16_t(b)), h = int16_t(uint16_t(a >> 16) + uint16_t(b >> 16));
  const int16_t cl = int16_t(uint16_t(c)), ch = int16_t(uint16_t(c >> 16));
  if (l > cl) l = cl;
  if (h > ch) h = ch;
  if (l < 0) l = 0;
  if (h < 0) h = 0;
  return Lanes(uint16_t(l), uint16_t(h));
}
#endif

VP8R_HD constexpr uint32_t X2(int v) { return (uint32_t(v) & 0xffffu) * 0x00010001u; }  // both 16-bit lanes = v

// Lines 0,2 / 1,3 of a byte word as 16-bit lanes, and back.
VP8R_HD uint32_t Even(uint32_t w) { return w & 0x00ff00ffu; }
VP8R_HD uint32_t Odd(uint32_t w) { return Prmt(w, 0u, 0x4341u); }
VP8R_HD uint32_t Pack(uint32_t e, uint32_t o) { return Prmt(e, o, 0x6240u); }
// Byte mask (0xff per line) from the sign bits (bit 15 of each lane) of an even / odd flag pair.
VP8R_HD uint32_t ByteMask(uint32_t fe, uint32_t fo) { return Prmt(fe, fo, 0xfbd9u); }
// 16-bit lane mask from bit 15 of each lane.
VP8R_HD uint32_t LaneMask(uint32_t f) { return Prmt(f, 0u, 0xbb99u); }
VP8R_HD uint32_t Select(uint32_t mask, uint32_t a, uint32_t b) { return (a & mask) | (b & ~mask); }  // one LOP3

// Per-macroblock constants, both 16-bit lanes equal (src/filter.cc:119-149 gives the limits).
struct EdgeK {
  uint32_t k_int;  // (127 - interior_limit) << 8
  uint32_t k_hev;  // (127 - hev_threshold) << 8
  uint32_t k_mb;   // 0x7fff - (2 * edge_limit_mb + 1); 0x8000 switches the filter off
  uint32_t k_sb;   // the same for sub-block edges
};
VP8R_HD EdgeK MakeEdgeK(int interior, int hev, int edge_mb, int edge_sb, bool enabled) {
  EdgeK k;
  k.k_int = X2((127 - interior) << 8);
  k.k_hev = X2((127 - hev) << 8);
  k.k_mb = enabled ? X2(0x7fff - (2 * edge_mb + 1)) : 0x80008000u;
  k.k_sb = enabled ? X2(0x7fff - (2 * edge_sb + 1)) : 0x80008000u;
  return k;
}

struct Flags {
  uint32_t off_e, off_o;  // bit 15 of a lane set: this line is NOT filtered
  uint32_t hev_e, hev_o;  // bit 15 set: high edge variance
};

// |q0-p0|*2 + |p1-q1|/2 <= E  <=>  4|q0-p0| + |p1-q1| <= 2E+1.  Returns lanes whose bit 15 says "exceeded".
VP8R_HD void EdgeTest(uint32_t P1, uint32_t P0, uint32_t Q0, uint32_t Q1, uint32_t k_e, uint32_t &se, uint32_t &so) {
  const uint32_t dA = Absd4(P0, Q0), dB = Absd4(P1, Q1);
  se = Even(dA) * 4u + Even(dB) + k_e;
  so = Odd(dA) * 4u + Odd(dB) + k_e;
}

// "upper byte of the lane > limit" as bit 15: m + k has it when the upper byte is below 128 (no wrap then),
// m itself has it otherwise.  The add must not carry from lane 0 into lane 1 (a difference of 255 in the
// junk byte of lane 1 would pass it on into the byte that decides): VIADD.16x2 + LOP3.
VP8R_HD uint32_t Above(uint32_t m, uint32_t k, uint32_t also) { return Add2(m, k) | m | also; }

// src/filter.cc:7-20: interior limit over the six neighbour differences, edge limit, high edge variance.
VP8R_HD Flags NormalFlags(uint32_t P3, uint32_t P2, uint32_t P1, uint32_t P0, uint32_t Q0, uint32_t Q1, uint32_t Q2,
                          uint32_t Q3, uint32_t k_int, uint32_t k_hev, uint32_t k_e) {
  const uint32_t d1 = Absd4(P3, P2), d2 = Absd4(P2, P1), d3 = Absd4(P1, P0);
  const uint32_t d4 = Absd4(Q1, Q0), d5 = Absd4(Q2, Q1), d6 = Absd4(Q3, Q2);
  // odd lines sit in the upper byte of each 16-bit lane already; even lines are shifted there.  The
  // lower byte of a lane is junk that never decides a maximum of upper bytes.
  const uint32_t m34o = UMax2(d3, d4);
  const uint32_t mo = UMax3(UMax3(d1, d2, m34o), d5, d6);
  const uint32_t m34e = UMax2(d3 << 8, d4 << 8);
  const uint32_t me = UMax3(UMax3(d1 << 8, d2 << 8, m34e), d5 << 8, d6 << 8);
  uint32_t se, so;
  EdgeTest(P1, P0, Q0, Q1, k_e, se, so);
  Flags f;
  f.off_e = Above(me, k_int, se);
  f.off_o = Above(mo, k_int, so);
  f.hev_e = Above(m34e, k_hev, 0u);
  f.hev_o = Above(m34o, k_hev, 0u);
  return f;
}

// Common part of every variant on one parity: x = a + 896 with a = s + 3 * (q0 - p0) (not yet clamped),
// s = clamp128(p1 - q1), or 0 where `s_mask` lanes are clear.  0 <= x <= 1791.
VP8R_HD uint32_t TapSum(uint32_t p1, uint32_t p0, uint32_t q0, uint32_t q1, uint32_t s_mask, bool masked) {
  uint32_t s = AddClamp2(p1 + X2(384) - q1, X2(-256), X2(255));  // clamp128(p1 - q1) + 128
  if (masked) s = Select(s_mask, s, X2(128));
  return (q0 + X2(256) - p0) * 3u + s;
}
// h = min(a' + k, 127) + 128 - k with a' = clamp128(a): the argument of the ">> 3" taps, made non-negative
// (the "+ k" is folded into the constants of its users).  k = 0 gives w + 128 of the macroblock edge.
VP8R_HD uint32_t TapArg(uint32_t x, int k) { return AddClamp2(x, X2(128 - 896), X2(255 - k)); }
// clamp255(pixel + delta) where `biased` = delta + bias >= 0: IADD + VIADDMNMX.RELU
VP8R_HD uint32_t Apply(uint32_t pixel, uint32_t biased, int bias) { return AddClamp2(pixel + biased, X2(-bias), X2(255)); }
VP8R_HD uint32_t Hi(uint32_t lanes) { return Prmt(lanes, 0u, 0x4341u); }  // upper byte of each lane

// Sub-block (inner) edge of the normal filter, src/filter.cc:37-44.  P3/P2/Q2/Q3 only enter the decision.
VP8R_HD void NormalInner(uint32_t P3, uint32_t P2, uint32_t &P1, uint32_t &P0, uint32_t &Q0, uint32_t &Q1, uint32_t Q2,
                         uint32_t Q3, const EdgeK &k) {
  const Flags f = NormalFlags(P3, P2, P1, P0, Q0, Q1, Q2, Q3, k.k_int, k.k_hev, k.k_sb);
  const uint32_t m_off = ByteMask(f.off_e, f.off_o);
  const uint32_t m_off1 = m_off | ByteMask(f.hev_e, f.hev_o);  // p1 / q1 move only without high edge variance
  uint32_t n[4][2];
#pragma unroll
  for (int par = 0; par < 2; ++par) {
    const uint32_t p1 = par ? Odd(P1) : Even(P1), p0 = par ? Odd(P0) : Even(P0);
    const uint32_t q0 = par ? Odd(Q0) : Even(Q0), q1 = par ? Odd(Q1) : Even(Q1);
    const uint32_t x = TapSum(p1, p0, q0, q1, LaneMask(par ? f.hev_o : f.hev_e), true);
    // with g = h + k:  f1 = (g1 >> 3) - 16 (k = 4),  f2 = (g2 >> 3) - 16 (k = 3)
    const uint32_t h1 = TapArg(x, 4), h2 = TapArg(x, 3);
    const uint32_t nf1 = Hi(X2(8160 - 32 * 4) - h1 * 32u);        // 15 - f1
    const uint32_t pf2 = Hi(h2 * 32u + X2(32 * 3));               // 16 + f2
    const uint32_t pa2 = Hi(h1 * 16u + X2(128 + 16 * 4));         // 8 + ((f1 + 1) >> 1)
    const uint32_t na2 = Hi(X2(4208 - 16 * 4) - h1 * 16u);        // 8 - ((f1 + 1) >> 1)
    n[0][par] = Apply(p1, pa2, 8);
    n[1][par] = Apply(p0, pf2, 16);
    n[2][par] = Apply(q0, nf1, 15);
    n[3][par] = Apply(q1, na2, 8);
  }
  P1 = Select(m_off1, P1, Pack(n[0][0], n[0][1]));
  P0 = Select(m_off, P0, Pack(n[1][0], n[1][1]));
  Q0 = Select(m_off, Q0, Pack(n[2][0], n[2][1]));
  Q1 = Select(m_off1, Q1, Pack(n[3][0], n[3][1]));
}

// Macroblock edge of the normal filter, src/filter.cc:46-67.
VP8R_HD void NormalMbEdge(uint32_t P3, uint32_t &P2, uint32_t &P1, uint32_t &P0, uint32_t &Q0, uint32_t &Q1, uint32_t &Q2,
                          uint32_t Q3, const EdgeK &k) {
  const Flags f = NormalFlags(P3, P2, P1, P0, Q0, Q1, Q2, Q3, k.k_int, k.k_hev, k.k_mb);
  const uint32_t m_off = ByteMask(f.off_e, f.off_o);
  const uint32_t m_off1 = m_off | ByteMask(f.hev_e, f.hev_o);
  uint32_t n[6][2];
#pragma unroll
  for (int par = 0; par < 2; ++par) {
    const uint32_t p2 = par ? Odd(P2) : Even(P2), p1 = par ? Odd(P1) : Even(P1), p0 = par ? Odd(P0) : Even(P0);
    const uint32_t q0 = par ? Odd(Q0) : Even(Q0), q1 = par ? Odd(Q1) : Even(Q1), q2 = par ? Odd(Q2) : Even(Q2);
    const uint32_t hev = LaneMask(par ? f.hev_o : f.hev_e);
    const uint32_t x = TapSum(p1, p0, q0, q1, 0u, false);
    // high edge variance: only p0 / q0 move, by the ">> 3" taps.  Biased to 27 like the taps below.
    const uint32_t h1 = TapArg(x, 4), h2 = TapArg(x, 3);
    const uint32_t h_q0 = Hi(X2(8160 - 32 * 4 + 12 * 256) - h1 * 32u);  // 27 - f1
    const uint32_t h_p0 = Hi(h2 * 32u + X2(32 * 3 + 11 * 256));         // 27 + f2
    // otherwise (27w+63)>>7, (18w+63)>>7, (9w+63)>>7 with w = clamp128(a); wb = w + 128 makes them
    // ((2k*wb + 126) >> 8) - k, read from the upper byte of the lane.
    const uint32_t wb = TapArg(x, 0);
    const uint32_t a27 = Hi(wb * 54u + X2(126)), n27 = Hi(X2(54 * 256 + 129) - wb * 54u);
    const uint32_t a18 = Hi(wb * 36u + X2(126)), n18 = Hi(X2(36 * 256 + 129) - wb * 36u);
    const uint32_t a9 = Hi(wb * 18u + X2(126)), n9 = Hi(X2(18 * 256 + 129) - wb * 18u);
    n[0][par] = Apply(p2, a9, 9);
    n[1][par] = Apply(p1, a18, 18);
    n[2][par] = Apply(p0, Select(hev, h_p0, a27), 27);
    n[3][par] = Apply(q0, Select(hev, h_q0, n27), 27);
    n[4][par] = Apply(q1, n18, 18);
    n[5][par] = Apply(q2, n9, 9);
  }
  P2 = Select(m_off1, P2, Pack(n[0][0], n[0][1]));
  P1 = Select(m_off1, P1, Pack(n[1][0], n[1][1]));
  P0 = Select(m_off, P0, Pack(n[2][0], n[2][1]));
  Q0 = Select(m_off, Q0, Pack(n[3][0], n[3][1]));
  Q1 = Select(m_off1, Q1, Pack(n[4][0], n[4][1]));
  Q2 = Select(m_off1, Q2, Pack(n[5][0], n[5][1]));
}

// Simple filter (luma only), src/filter.cc:14-16,69-71: the edge limit alone decides, p0 / q0 move.
VP8R_HD void SimpleEdge(uint32_t P1, uint32_t &P0, uint32_t &Q0, uint32_t Q1, uint32_t k_e) {
  uint32_t se, so;
  EdgeTest(P1, P0, Q0, Q1, k_e, se, so);
  const uint32_t m_off = ByteMask(se, so);
  uint32_t n[2][2];
#pragma unroll
  for (int par = 0; par < 2; ++par) {
    const uint32_t p1 = par ? Odd(P1) : Even(P1), p0 = par ? Odd(P0) : Even(P0);
    const uint32_t q0 = par ? Odd(Q0) : Even(Q0), q1 = par ? Odd(Q1) : Even(Q1);
    const uint32_t x = TapSum(p1, p0, q0, q1, 0u, false);
    const uint32_t h1 = TapArg(x, 4), h2 = TapArg(x, 3);
    n[0][par] = Apply(p0, Hi(h2 * 32u + X2(32 * 3)), 16);
    n[1][par] = Apply(q0, Hi(X2(8160 - 32 * 4) - h1 * 32u), 15);
  }
  P0 = Select(m_off, P0, Pack(n[0][0], n[0][1]));
  Q0 = Select(m_off, Q0, Pack(n[1][0], n[1][1]));
}

// Transposition of a 4x4 byte block held as four words (8 PRMT).
VP8R_HD void Transpose4(uint32_t &r0, uint32_t &r1, uint32_t &r2, uint32_t &r3) {
  const uint32_t t0 = Prmt(r0, r1, 0x5140u), t1 = Prmt(r2, r3, 0x5140u);
  const uint32_t t2 = Prmt(r0, r1, 0x7362u), t3 = Prmt(r2, r3, 0x7362u);
  r0 = Prmt(t0, t1, 0x5410u);
  r1 = Prmt(t0, t1, 0x7632u);
  r2 = Prmt(t2, t3, 0x5410u);
  r3 = Prmt(t2, t3, 0x7632u);
}

}  // namespace swar
}  // namespace vp8r

#endif  // VP8R_CUDA_LF_SWAR_H_
