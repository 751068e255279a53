// kernels_mc8.cuh — packed-integer helpers of the 8-bit inter prediction (k_inter_pred_tma, kernels_mct.cuh; tests/mct_emul.cu
// runs the same code on the CPU): the HEVC interpolation taps packed for dp4a / dp2a (Mc8Tables, built on the host by engine.cu
// init_tables into constant memory), the PTX forms of the integer steps, and all four weighting modes through one branch-free
// multiply-add-shift-offset form (Mc8Weight).
#pragma once
#include "dev_common.cuh"

struct Mc8Tables {
  uint32_t qh[5][4][3];  // [frac 0..3, 4 = integer position with gain 64][output j][word]
  uint32_t qv[4][5];     // [frac][A,B (even rows), C,D,E (odd rows)]
  uint32_t eh[9][4][2];  // [frac 0..7, 8 = integer with gain 64][output j][word]
  uint32_t ev[8][3];     // [frac][A (even), C,D (odd)]
};
__constant__ Mc8Tables c_mc8;

// Builds the packed tap tables from the HEVC interpolation taps (host; engine.cu uploads them to c_mc8).
//   qh/eh[f][j][k]: the taps of phase f shifted right by j bytes across k words: dp4a operands for output j of a group of 4
//                   (f = 4 resp. 8: the full-sample position with gain 64); qv/ev: the taps packed for dp2a on int16 pairs,
//                   A,B for outputs on an even pair boundary, C,D,E (C,D for 4 taps) for the odd ones.
inline void mc8_build_tables(Mc8Tables& tb)
{
  static const int8_t q[4][8] = {{0, 0, 0, 1, 0, 0, 0, 0}, {-1, 4, -10, 58, 17, -5, 1, 0}, {-1, 4, -11, 40, 40, -11, 4, -1}, {0, 1, -5, 17, 58, -10, 4, -1}};
  static const int8_t ep[8][4] = {{0, 1, 0, 0},     {-2, 58, 10, -2}, {-4, 54, 16, -2}, {-6, 46, 28, -4},
                                  {-4, 36, 36, -4}, {-4, 28, 46, -6}, {-2, 16, 54, -4}, {-2, 10, 58, -2}};
  auto pack = [](int b0, int b1, int b2, int b3) { return (uint32_t)(uint8_t)b0 | ((uint32_t)(uint8_t)b1 << 8) | ((uint32_t)(uint8_t)b2 << 16) | ((uint32_t)(uint8_t)b3 << 24); };
  auto& qh = tb.qh; auto& qv = tb.qv; auto& eh = tb.eh; auto& ev = tb.ev;
  for (int f = 0; f < 5; f++) {
    int8_t t[8];
    for (int i = 0; i < 8; i++) t[i] = (f == 4) ? (int8_t)(i == 3 ? 64 : 0) : q[f][i];
    for (int j = 0; j < 4; j++)
      for (int k = 0; k < 3; k++) {
        int b[4];
        for (int i = 0; i < 4; i++) { const int idx = 4 * k + i - j; b[i] = (idx >= 0 && idx < 8) ? t[idx] : 0; }
        qh[f][j][k] = pack(b[0], b[1], b[2], b[3]);
      }
    if (f < 4) {
      qv[f][0] = pack(t[0], t[1], t[2], t[3]); qv[f][1] = pack(t[4], t[5], t[6], t[7]);
      qv[f][2] = pack(0, t[0], t[1], t[2]);    qv[f][3] = pack(t[3], t[4], t[5], t[6]); qv[f][4] = pack(t[7], 0, 0, 0);
    }
  }
  for (int f = 0; f < 9; f++) {
    int8_t t[4];
    for (int i = 0; i < 4; i++) t[i] = (f == 8) ? (int8_t)(i == 1 ? 64 : 0) : ep[f][i];
    for (int j = 0; j < 4; j++)
      for (int k = 0; k < 2; k++) {
        int b[4];
        for (int i = 0; i < 4; i++) { const int idx = 4 * k + i - j; b[i] = (idx >= 0 && idx < 4) ? t[idx] : 0; }
        eh[f][j][k] = pack(b[0], b[1], b[2], b[3]);
      }
    if (f < 8) { ev[f][0] = pack(t[0], t[1], t[2], t[3]); ev[f][1] = pack(0, t[0], t[1], t[2]); ev[f][2] = pack(t[3], 0, 0, 0); }
  }
}

__device__ __forceinline__ int dp4a_us(uint32_t a, uint32_t b, int c)
{
  int d;
  asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
__device__ __forceinline__ int dp2a_lo_ss(uint32_t a, uint32_t b, int c)
{
  int d;
  asm("dp2a.lo.s32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
__device__ __forceinline__ int dp2a_hi_ss(uint32_t a, uint32_t b, int c)
{
  int d;
  asm("dp2a.hi.s32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
// (v >> shift) wrapped to int16: one signed bit-field extract of 16 bits at `shift`
__device__ __forceinline__ int shr_wrap16(int v, int shift)
{
  int d;
  asm("bfe.s32 %0, %1, %2, 16;" : "=r"(d) : "r"(v), "r"(shift));
  return d;
}
__device__ __forceinline__ int sat_u8(int v)
{
  int d;
  asm("cvt.sat.u8.s32 %0, %1;" : "=r"(d) : "r"(v));
  return d;
}

// Branch-free weighting: out = sat_u8(((a*w0 + b*w1 + rnd) >> shift) + off) covers fallback-motion.cc:33-256:
//   uni          (a + 32) >> 6                                   w0=1 w1=0 rnd=32            shift=6        off=0
//   bi average   (a + b + 64) >> 7                               w0=1 w1=1 rnd=64            shift=7        off=0
//   uni explicit ((a*w + 2^(wd-1)) >> wd) + o                    w0=w w1=0 rnd=2^(wd-1)      shift=wd       off=o
//   bi explicit  (a*w0 + b*w1 + ((o0+o1+1) << wd)) >> (wd+1)     w0,w1     rnd=(o0+o1+1)<<wd shift=wd+1     off=0
struct Mc8Weight {
  int w0, w1, rnd, shift, off;
};
__host__ __device__ __forceinline__ Mc8Weight mc8_weight(bool bi, bool wgt, int lu, const b200_weight_entry* __restrict__ wp_, int c)
{
  Mc8Weight r;
  if (!wgt) {
    r.w0 = 1; r.w1 = bi ? 1 : 0; r.rnd = bi ? 64 : 32; r.shift = bi ? 7 : 6; r.off = 0;
  } else {
    const int wd = c ? wp_->log2wd_chroma : wp_->log2wd_luma;
    if (bi) { r.w0 = wp_->w[0][c]; r.w1 = wp_->w[1][c]; r.rnd = (int)((unsigned)(wp_->o[0][c] + wp_->o[1][c] + 1) << wd); r.shift = wd + 1; r.off = 0; }
    else { r.w0 = wp_->w[lu][c]; r.w1 = 0; r.rnd = 1 << (wd - 1); r.shift = wd; r.off = wp_->o[lu][c]; }
  }
  return r;
}
