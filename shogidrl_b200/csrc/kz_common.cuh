// kz_common.cuh -- bitboard helpers and piece tables shared by the engine kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#define FULL 0xffffffffu
#define BITMAP_WORDS 448      // ceil(13527 / 32) = 423, padded to 14 words per lane (k-th set bit selection)
#ifndef WARPS_PER_CTA
#define WARPS_PER_CTA 8
#endif
#ifndef MIN_CTAS_PER_SM
#define MIN_CTAS_PER_SM 3  // 80 registers per thread: 24 warps per SM (measured best: 2 -> 0.423 ms, 3 -> 0.402 ms, 4 spills)
#endif
#ifndef CTAS_PER_SM
#define CTAS_PER_SM 3  // persistent grid = SMs x resident CTAs
#endif

// step-target classes of the STEP table
#define CLS_BP 0
#define CLS_BS 1
#define CLS_BG 2
#define CLS_BN 3
#define CLS_WP 4
#define CLS_WS 5
#define CLS_WG 6
#define CLS_WN 7
#define CLS_PLUS 8   // +B extra steps (shogi_rules_logic.py:135-140)
#define CLS_X 9      // +R extra steps (:129-134)
#define CLS_KING 10
#define CLS_NONE 11
#define NCLS 12

// 81-bit bitboard, bit = row*9 + col.  Lane l of a warp owns bits l, l+32, l+64 ("slot" 0..2).
struct BB {
  uint32_t w0, w1, w2;
};
__device__ __forceinline__ BB operator&(BB a, BB b) { return BB{a.w0 & b.w0, a.w1 & b.w1, a.w2 & b.w2}; }
__device__ __forceinline__ BB operator|(BB a, BB b) { return BB{a.w0 | b.w0, a.w1 | b.w1, a.w2 | b.w2}; }
__device__ __forceinline__ BB bb_andn(BB a, BB b) { return BB{a.w0 & ~b.w0, a.w1 & ~b.w1, a.w2 & ~b.w2}; }
__device__ __forceinline__ bool bb_any(BB a) { return (a.w0 | a.w1 | a.w2) != 0; }
__device__ __forceinline__ int bb_popc(BB a) { return __popc(a.w0) + __popc(a.w1) + __popc(a.w2); }
__device__ __forceinline__ int bb_lsb(BB a) {
  return a.w0 ? __ffs(a.w0) - 1 : (a.w1 ? 31 + __ffs(a.w1) : 63 + __ffs(a.w2));
}
__device__ __forceinline__ int bb_msb(BB a) {
  return a.w2 ? 95 - __clz(a.w2) : (a.w1 ? 63 - __clz(a.w1) : 31 - __clz(a.w0));
}
__device__ __forceinline__ uint32_t lowmask32(int x) {  // bits [0, clamp(x, 0, 32))
  x = x < 0 ? 0 : (x > 32 ? 32 : x);
  return (uint32_t)((1ull << x) - 1ull);
}
__device__ __forceinline__ BB bb_below(int s) { return BB{lowmask32(s), lowmask32(s - 32), lowmask32(s - 64)}; }
__device__ __forceinline__ BB bb_upto(int s) { return bb_below(s + 1); }
__device__ __forceinline__ BB bb_bit(int s) {
  const uint32_t b = 1u << (s & 31);
  const int w = s >> 5;
  return BB{w == 0 ? b : 0u, w == 1 ? b : 0u, w == 2 ? b : 0u};
}
__device__ __forceinline__ bool bb_test(BB a, int s) {
  const uint32_t w = (s >> 5) == 0 ? a.w0 : ((s >> 5) == 1 ? a.w1 : a.w2);
  return (w >> (s & 31)) & 1;
}
__device__ __forceinline__ BB bb_shr1(BB a) {
  return BB{__funnelshift_r(a.w0, a.w1, 1), __funnelshift_r(a.w1, a.w2, 1), a.w2 >> 1};
}
__device__ __forceinline__ uint32_t spread16(uint32_t x) {  // bit i -> bit 2i
  x = (x | (x << 8)) & 0x00FF00FFu;
  x = (x | (x << 4)) & 0x0F0F0F0Fu;
  x = (x | (x << 2)) & 0x33333333u;
  x = (x | (x << 1)) & 0x55555555u;
  return x;
}

// Counter-based per-game random stream: kz_step's next_actions and kz_heuristic_actions draw from it.  The formula is
// part of the interface: a CPU restatement of it replays those draws bit for bit.
__device__ __forceinline__ uint32_t rand32(unsigned long long seed, unsigned long long env, unsigned long long step) {
  unsigned long long x = seed ^ (env * 0x9E3779B97F4A7C15ull) ^ (step * 0xBF58476D1CE4E5B9ull);
  x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull;
  x ^= x >> 27; x *= 0x94D049BB133111EBull;
  x ^= x >> 31;
  return (uint32_t)(x >> 32);
}

__device__ __forceinline__ int sq_row(int s) { return (s * 57) >> 9; }  // floor(s / 9) for s < 96
__device__ __forceinline__ int sq_col(int s) { return s - 9 * sq_row(s); }

// directions 0:N 1:NE 2:E 3:SE 4:S 5:SW 6:W 7:NW as square-index deltas -9,-8,+1,+10,+9,+8,-1,-10
__device__ __forceinline__ int dir_delta(int d) {
  // (delta + 10) packed 5 bits per direction
  const unsigned long long pack = (1ull) | (2ull << 5) | (11ull << 10) | (20ull << 15) | (19ull << 20) | (18ull << 25) |
                                  (9ull << 30) | (0ull << 35);
  return (int)((pack >> (5 * d)) & 31) - 10;
}
__device__ __forceinline__ bool dir_positive(int d) { return (0x3C >> d) & 1; }  // E, SE, S, SW increase the index

__device__ __forceinline__ int code_color(int code) { return code >= 15; }
__device__ __forceinline__ int code_type(int code) { return code >= 15 ? code - 15 : code - 1; }
__device__ __forceinline__ int promo_delta(int type) { return type <= 3 ? 8 : 7; }           // P,L,N,S +8; B,R +7
__device__ __forceinline__ int base_of_promoted(int type) { return type <= 11 ? type - 8 : type - 7; }

// Per-code properties, held in lane `code` of every warp and fetched with one shuffle:
//   bits 0-7 step directions, 8-15 slide directions (direction sets of shogi_rules_logic.py:103-206),
//   16-19 STEP class, 20 promotable, 21-22 forced-promotion kind (1: last rank, 2: last two ranks), 23 king.
__device__ __forceinline__ uint32_t code_info(int code) {
  if (code < 1 || code > 28) return (uint32_t)CLS_NONE << 16;
  const int color = code_color(code), t = code_type(code);
  uint32_t step = 0, slide = 0, cls = CLS_NONE, prom = 0, must = 0, king = 0;
  const uint32_t P_ = 0x01, S_ = 0x01 | 0x02 | 0x80 | 0x08 | 0x20, G_ = 0x01 | 0x02 | 0x80 | 0x04 | 0x40 | 0x10;
  switch (t) {
    case 0: step = P_; cls = CLS_BP; prom = 1; must = 1; break;
    case 1: slide = 0x01; prom = 1; must = 1; break;
    case 2: cls = CLS_BN; prom = 1; must = 2; break;
    case 3: step = S_; cls = CLS_BS; prom = 1; break;
    case 4: case 8: case 9: case 10: case 11: step = G_; cls = CLS_BG; break;
    case 5: slide = 0xAA; prom = 1; break;
    case 6: slide = 0x55; prom = 1; break;
    case 7: step = 0xFF; cls = CLS_KING; king = 1; break;
    case 12: slide = 0xAA; step = 0x55; cls = CLS_PLUS; break;
    case 13: slide = 0x55; step = 0xAA; cls = CLS_X; break;
  }
  if (color) {  // WHITE: 180-degree rotation of the direction sets
    step = ((step << 4) | (step >> 4)) & 0xFF;
    slide = ((slide << 4) | (slide >> 4)) & 0xFF;
    if (cls <= CLS_BN) cls += 4;
  }
  return step | (slide << 8) | (cls << 16) | (prom << 20) | (must << 21) | (king << 23);
}
