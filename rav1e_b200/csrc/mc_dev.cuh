// mc_dev.cuh — the separable 8-tap prediction of one W x H block by ONE warp, on packed data:
//   put_8tap   src/mc.rs:250-353
// The reference distinguishes four cases (no fraction / V only / H only with a double rounding / H into
// an i16 intermediate, then V).  All four are the fourth one with the identity filter {0,0,0,128,0,0,0,0}
// (row 0 of every filter bank) in the missing direction, bit for bit: an identity H pass leaves
// inter = px << ib exactly (128 px is a multiple of 2^(7-ib)), after which the V rounding
// (sum + 2^(6+ib)) >> (7+ib) equals the V-only (sum + 64) >> 7; an identity V pass turns
// round(128 * inter, 7+ib) into round(inter, ib), the H-only case's second rounding; and the i16
// intermediate never truncates: over the filter table it lies in [-1785, 5865] at 8 bit, [-7161, 23529]
// at 10 and [-7166, 23546] at 12 (tests/test_full_scale_pred.py computes and pins these bounds).  So one
// code path serves all.
//
// Arithmetic on packed words instead of one multiply per tap and pixel:
//   H pass, 8-bit pixels : IDP.4A - four u8 pixels x four s8 taps per instruction (every tap fits s8:
//                          -24..126), the unaligned windows of the 4 outputs of a task by funnel shifts;
//   H pass, 16-bit pixels: IDP.2A - two u16 pixels x two s8 taps per instruction;
//   V pass               : IDP.2A on the i16 intermediate, which the H pass stores TRANSPOSED so that a
//                          column's rows are consecutive halfwords.
// A task = 4 adjacent outputs sharing their loaded words (3 words for 8-bit, 6 for 16-bit lanes).
#pragma once
#include "mc_filters.cuh"

namespace {

__device__ __forceinline__ int dp4a_u8s8(uint32_t a, uint32_t b, int c) {
  int d;
  asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
__device__ __forceinline__ int dp2a_u16s8(uint32_t a, uint32_t b, int c) {  // a: 2 x u16, b: s8 in bytes 0, 1
  int d;
  asm("dp2a.lo.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
__device__ __forceinline__ int dp2a_s16s8(uint32_t a, uint32_t b, int c) {  // a: 2 x s16
  int d;
  asm("dp2a.lo.s32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}

struct McTaps {
  uint32_t q4[2];  // taps 0..3 / 4..7 as s8 x 4 (dp4a)
  uint32_t q2[4];  // taps (0,1) (2,3) (4,5) (6,7) as s8 x 2 in the low bytes (dp2a.lo)
};
__device__ __forceinline__ McTaps mc_taps(int bank, int frac) {
  McTaps t;
  const short *f = kSubpel[bank][frac];
#pragma unroll
  for (int m = 0; m < 4; m++) t.q2[m] = ((uint32_t)f[2 * m] & 0xffu) | (((uint32_t)f[2 * m + 1] & 0xffu) << 8);
  t.q4[0] = t.q2[0] | (t.q2[1] << 16);
  t.q4[1] = t.q2[2] | (t.q2[3] << 16);
  return t;
}

template <typename T, int W, int H>
struct McLayout {
  static constexpr int TW = W + 7, TH = H + 7;
  static constexpr int TP = W + 8;    // tile pitch in pixels: rows word aligned, one pixel of slack
  static constexpr int THP = H + 8;   // transposed intermediate: halfwords per image column
  static constexpr size_t TILE_BYTES = (size_t)TH * TP * sizeof(T);
  static constexpr size_t INTER_BYTES = (size_t)W * THP * 2;
};

// 4 sums of 8 taps over 16-bit lanes: element k of the task starts in word k / 2 of w[0..5]
template <bool SIGNED>
__device__ __forceinline__ void filt4_words16(const uint32_t (&w)[6], const McTaps &t, int (&out)[4]) {
#pragma unroll
  for (int j = 0; j < 4; j++) {
    int s = 0;
#pragma unroll
    for (int m = 0; m < 4; m++) {
      const int k = (j >> 1) + m;
      const uint32_t v = (j & 1) ? __funnelshift_r(w[k], w[k + 1], 16) : w[k];
      s = SIGNED ? dp2a_s16s8(v, t.q2[m], s) : dp2a_u16s8(v, t.q2[m], s);
    }
    out[j] = s;
  }
}

// Stage the (W+7) x (H+7) footprint whose pixel (0,0) is `src` (source pixel (-3,-3) of the block)
template <typename T, int W, int H>
__device__ __forceinline__ void mc_stage_tile(T *tile, const T *src, long long stride, int lane) {
  using L = McLayout<T, W, H>;
  for (int r = 0; r < L::TH; r++) {
    const T *srow = src + (long long)r * stride;
    for (int c = lane; c < L::TW; c += 32) tile[r * L::TP + c] = srow[c];
  }
}

// tile -> pred (W x H, packed) through the transposed i16 intermediate.  All lanes of the warp call it;
// the caller brackets it with __syncwarp() (tile ready before, pred consumed after).
template <typename T, int W, int H>
__device__ __forceinline__ void mc_put_warp(const T *tile, short *interT, T *pred, int xbank, int col_frac, int ybank,
                                            int row_frac, int bit_depth, int lane) {
  using L = McLayout<T, W, H>;
  const int ib = 4 - (bit_depth == 12 ? 2 : 0);
  const int maxv = (1 << bit_depth) - 1;
  const McTaps xt = mc_taps(xbank, col_frac), yt = mc_taps(ybank, row_frac);
  // ---- H pass over the H + 7 rows (mc.rs:312-327), 4 outputs per task.  The identity filter's tap (128)
  // does not fit s8: a direction without a fraction takes its closed form (see the header comment).
  for (int task = lane; task < L::TH * (W / 4); task += 32) {
    const int r = task / (W / 4), g = task - r * (W / 4);
    int s[4];
    if (col_frac == 0) {
#pragma unroll
      for (int j = 0; j < 4; j++) interT[(4 * g + j) * L::THP + r] = (short)((int)tile[r * L::TP + 4 * g + j + 3] << ib);
      continue;
    }
    if (sizeof(T) == 1) {
      const uint32_t *wp = (const uint32_t *)(tile + r * L::TP) + g;
      const uint32_t w0 = wp[0], w1 = wp[1], w2 = wp[2];
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const uint32_t u0 = j ? __funnelshift_r(w0, w1, 8 * j) : w0, u1 = j ? __funnelshift_r(w1, w2, 8 * j) : w1;
        s[j] = dp4a_u8s8(u1, xt.q4[1], dp4a_u8s8(u0, xt.q4[0], 0));
      }
    } else {
      const uint32_t *wp = (const uint32_t *)(tile + r * L::TP) + 2 * g;
      const uint32_t w[6] = {wp[0], wp[1], wp[2], wp[3], wp[4], wp[5]};
      filt4_words16<false>(w, xt, s);
    }
#pragma unroll
    for (int j = 0; j < 4; j++) interT[(4 * g + j) * L::THP + r] = (short)rshift_round(s[j], 7 - ib);  // `as i16`, mc.rs:323
  }
  __syncwarp();
  // ---- V pass (mc.rs:328-343): column c, rows 4q .. 4q+3
  for (int task = lane; task < W * (H / 4); task += 32) {
    const int c = task % W, q = task / W;
    if (row_frac == 0) {
#pragma unroll
      for (int j = 0; j < 4; j++)
        pred[(4 * q + j) * W + c] = (T)min(max(rshift_round((int)interT[c * L::THP + 4 * q + j + 3], ib), 0), maxv);
      continue;
    }
    const uint32_t *wp = (const uint32_t *)(interT + c * L::THP) + 2 * q;
    const uint32_t w[6] = {wp[0], wp[1], wp[2], wp[3], wp[4], wp[5]};
    int s[4];
    filt4_words16<true>(w, yt, s);
#pragma unroll
    for (int j = 0; j < 4; j++) pred[(4 * q + j) * W + c] = (T)min(max(rshift_round(s[j], 7 + ib), 0), maxv);
  }
}

}  // namespace
