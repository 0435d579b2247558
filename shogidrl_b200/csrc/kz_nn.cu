// kz_nn.cu -- the observation input layer of the policy/value network on sm_100a tensor cores:
//   kz_obs_conv_fwd   : y = [relu](conv3x3(obs, W) + b), obs fp32 [n][46][9][9] -> y bf16 [n][16][9][9]
//   kz_obs_conv_wgrad : dW, db of the same layer from dy (the input needs no gradient)
// (keisei/core/neural_network.py:14-28: nn.Conv2d(46, 16, 3, padding=1) + ReLU under bf16 autocast,
//  keisei/core/ppo_agent.py:323.)
//
// Why a kernel: with 16 output channels the layer is a [16 x 414] x [414 x 81] product per board.  The library's
// implicit-GEMM weight gradient serialises its K = 81 n reduction over a handful of CTAs (2.6 ms per 16,384
// boards on B200, 35 % of a PPO minibatch update; profiles/ppo_update_probe.py); the work itself is 290 MB of
// HBM traffic.  Here every CTA walks its own slab of boards: a board is converted to bf16 once into shared
// memory as a zero-bordered 11 x 11 x 48 channel-last tile, so each 3 x 3 tap is the same tile at a row offset
// (implicit GEMM without an im2col copy), operands come from ldmatrix, products from mma.sync m16n8k16 bf16 with
// fp32 accumulation.  Channel 46 of the tile is constant 1, which folds the bias into the forward GEMM and makes
// the bias gradient one column of the weight gradient.  N = 16 is far below any tcgen05 tile (M >= 64, operands
// through TMA descriptors), and the layer is HBM-bound, so the warp-level MMA is the right instrument here.
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/keisei_b200.h"

int kz_cuda_fail(cudaError_t e);  // kz_engine.cu: records the message for kz_last_cuda_error

namespace {

inline int fail(cudaError_t e) { return kz_cuda_fail(e); }

constexpr int CIN = 46;        // observation planes
constexpr int COUT = 16;       // output channels of the layer (one m16 tile)
constexpr int CPAD = 48;       // 46 planes + the constant-one channel + one zero channel
constexpr int XS_STRIDE = 56;  // bf16 per tile row (112 B): eight consecutive rows hit distinct banks for ldmatrix
constexpr int ZROW = 121;      // an all-zero row for the out-of-range columns of the last tile
constexpr int XS_ROWS = 122;
constexpr int KTOT = 9 * CPAD;  // 432: k = tap * 48 + channel
constexpr int WS_STRIDE = 440;  // bf16 per weight row (880 B): conflict-free
constexpr int DS_STRIDE = 104;  // bf16 per dy row (96 positions + pad; 208 B): conflict-free

__device__ __forceinline__ int tile_row(int xy) { return (xy / 9 + 1) * 11 + (xy % 9 + 1); }
__device__ __forceinline__ int tap_offset(int tap) { return (tap / 3 - 1) * 11 + (tap % 3 - 1); }

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldmatrix_x2(uint32_t (&r)[2], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(addr));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void mma_bf16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// borders, the zero row and the two constant channels of the board tile; written once per CTA
__device__ __forceinline__ void init_tile(__nv_bfloat16* xs, int tid, int nthreads) {
  for (int i = tid; i < XS_ROWS * XS_STRIDE; i += nthreads) xs[i] = __float2bfloat16(0.f);
  __syncthreads();
  for (int xy = tid; xy < 81; xy += nthreads) xs[tile_row(xy) * XS_STRIDE + CIN] = __float2bfloat16(1.f);
}

// One board fp32 [46][81] -> bf16 tile [row][channel], in two halves so that the global loads of the next board are
// in flight while the current one is multiplied: load_board fills registers (two channels of one square per
// slot), store_board converts and writes them as 4-byte bf16 pairs.
template <int NT>
struct BoardRegs {
  static constexpr int SLOTS = ((CIN / 2) * 81 + NT - 1) / NT;
  float a[SLOTS], b[SLOTS];
};
template <int NT>
__device__ __forceinline__ void load_board(BoardRegs<NT>& r, const float* __restrict__ x, int tid) {
#pragma unroll
  for (int k = 0; k < BoardRegs<NT>::SLOTS; k++) {
    const int i = tid + k * NT;
    if (i < (CIN / 2) * 81) {
      const int cp = i / 81, xy = i - cp * 81;
      r.a[k] = __ldg(x + (2 * cp) * 81 + xy);
      r.b[k] = __ldg(x + (2 * cp + 1) * 81 + xy);
    }
  }
}
template <int NT>
__device__ __forceinline__ void store_board(__nv_bfloat16* xs, const BoardRegs<NT>& r, int tid) {
#pragma unroll
  for (int k = 0; k < BoardRegs<NT>::SLOTS; k++) {
    const int i = tid + k * NT;
    if (i < (CIN / 2) * 81) {
      const int cp = i / 81, xy = i - cp * 81;
      *reinterpret_cast<__nv_bfloat162*>(xs + tile_row(xy) * XS_STRIDE + 2 * cp) = __floats2bfloat162_rn(r.a[k], r.b[k]);
    }
  }
}

// ---- forward: 4 warps, warp w owns column tiles w, w + 4, w + 8 (8 board squares each; 11 tiles cover 81) ----
__global__ void __launch_bounds__(128) kz_obs_conv_fwd_kernel(const float* __restrict__ obs,
                                                              const long long* __restrict__ rows,
                                                              const float* __restrict__ w,
                                                              const float* __restrict__ bias, int n, int relu,
                                                              __nv_bfloat16* __restrict__ out) {
  __shared__ __align__(16) __nv_bfloat16 ws[COUT * WS_STRIDE];
  __shared__ __align__(16) __nv_bfloat16 xs[XS_ROWS * XS_STRIDE];
  __shared__ __align__(16) __nv_bfloat16 ys[COUT * 81 + 8];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < COUT * WS_STRIDE; i += 128) {
    const int o = i / WS_STRIDE, k = i - o * WS_STRIDE, tap = k / CPAD, c = k - tap * CPAD;
    float v = 0.f;
    if (k < KTOT) {
      if (c < CIN) v = w[(o * CIN + c) * 9 + tap];
      else if (c == CIN && tap == 4 && bias) v = bias[o];
    }
    ws[i] = __float2bfloat16(v);
  }
  init_tile(xs, tid, 128);
  const uint32_t ws_a = smem_u32(ws) + ((lane & 15) * WS_STRIDE + (lane >> 4) * 8) * 2;
  // this lane's row for the B operand of each of the warp's tiles (lanes 0-7: channels +0, lanes 8-15: +8)
  int brow[3];
  bool bval[3];
#pragma unroll
  for (int j = 0; j < 3; j++) {
    const int col = (warp + 4 * j) * 8 + (lane & 7);
    bval[j] = col < 81;
    brow[j] = bval[j] ? tile_row(col) : ZROW;
  }
  const uint32_t xs_b = smem_u32(xs) + ((lane >> 3) & 1) * 16;
  BoardRegs<128> regs;
  auto board = [&](int b) { return obs + (size_t)(rows ? rows[b] : b) * CIN * 81; };  // in-place minibatch gather
  if (blockIdx.x < n) load_board<128>(regs, board(blockIdx.x), tid);
  for (int b = blockIdx.x; b < n; b += gridDim.x) {
    __syncthreads();  // previous board's ys copied out, xs free
    store_board<128>(xs, regs, tid);
    __syncthreads();
    if (b + gridDim.x < n) load_board<128>(regs, board(b + gridDim.x), tid);  // next board in flight
    float acc[3][4];
#pragma unroll
    for (int j = 0; j < 3; j++) acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f;
#pragma unroll 3
    for (int ks = 0; ks < 27; ks++) {
      const int tap = ks / 3, c0 = (ks - tap * 3) * 16;
      uint32_t a[4];
      ldmatrix_x4(a, ws_a + ks * 32);
      const int off = tap_offset(tap);
#pragma unroll
      for (int j = 0; j < 3; j++) {
        if (warp + 4 * j < 11) {  // warp-uniform
          uint32_t bb[2];
          ldmatrix_x2(bb, xs_b + ((bval[j] ? brow[j] + off : ZROW) * XS_STRIDE + c0) * 2);
          mma_bf16(acc[j], a, bb[0], bb[1]);
        }
      }
    }
#pragma unroll
    for (int j = 0; j < 3; j++) {
      const int col = (warp + 4 * j) * 8 + (lane & 3) * 2, o = lane >> 2;
      if (warp + 4 * j < 11) {
#pragma unroll
        for (int e = 0; e < 4; e++) {
          const int c = col + (e & 1), oo = o + (e >> 1) * 8;
          float v = acc[j][e];
          if (relu) v = v != v ? v : fmaxf(v, 0.f);  // torch.relu keeps NaN
          if (c < 81) ys[oo * 81 + c] = __float2bfloat16(v);
        }
      }
    }
    __syncthreads();
    uint4* dst = reinterpret_cast<uint4*>(out + (size_t)b * COUT * 81);  // 2,592 B per board: 16-byte aligned
    for (int i = tid; i < COUT * 81 * 2 / 16; i += 128) dst[i] = reinterpret_cast<const uint4*>(ys)[i];
  }
}

// ---- weight gradient: 9 warps, warp t owns tap t: dW[o][t][c] += sum_xy dy[o][xy] * tile[row(xy) + off(t)][c] ----
// COBS: the board comes as the engine's compact observation (kz_step_rollout: 160 bytes -- one piece-plane index per
// square + the 18 constant-plane values) instead of the 14,904-byte fp32 tensor: the tile is then PATCHED from one board
// to the next (clear the previous board's piece channel of each square, set the new one, rewrite the constant channels)
// instead of being converted from 3,726 floats, and the kernel stops being bound by those loads.
template <bool COBS>
__global__ void __launch_bounds__(288) kz_obs_conv_wgrad_kernel(const float* __restrict__ obs,
                                                                const long long* __restrict__ rows,
                                                                const __nv_bfloat16* __restrict__ y, const void* dout,
                                                                int dout_bf16, int n, float* __restrict__ part) {
  __shared__ __align__(16) __nv_bfloat16 xs[XS_ROWS * XS_STRIDE];
  __shared__ __align__(16) __nv_bfloat16 ds[COUT * DS_STRIDE];
  __shared__ __align__(16) uint32_t cws[KZ_COBS_WORDS];
  const int tid = threadIdx.x, lane = tid & 31, tap = tid >> 5;
  init_tile(xs, tid, 288);
  for (int i = tid; i < COUT * DS_STRIDE; i += 288) ds[i] = __float2bfloat16(0.f);
  const uint32_t ds_a = smem_u32(ds) + ((lane & 15) * DS_STRIDE + (lane >> 4) * 8) * 2;
  const uint32_t xs_b = smem_u32(xs) + (lane >> 4) * 16;  // lanes 16-31 address the next 8 channels
  const int off = tap_offset(tap);
  float acc[6][4];
#pragma unroll
  for (int j = 0; j < 6; j++) acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f;
  BoardRegs<288> regs;
  constexpr int DSLOTS = (COUT * 81 + 287) / 288;
  float dreg[DSLOTS];
  auto load_dy = [&](int b) {  // dy of board b with the ReLU gate of the saved activation applied
#pragma unroll
    for (int k = 0; k < DSLOTS; k++) {
      const int i = tid + k * 288;
      if (i < COUT * 81) {
        const size_t g = (size_t)b * COUT * 81 + i;
        float v = dout_bf16 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(dout)[g])
                            : reinterpret_cast<const float*>(dout)[g];
        if (y && __bfloat162float(y[g]) <= 0.f) v = 0.f;  // torch's threshold_backward: a NaN output passes dy
        dreg[k] = v;
      }
    }
  };
  auto board = [&](int b) { return obs + (size_t)(rows ? rows[b] : b) * CIN * 81; };
  uint32_t cw = 0;      // COBS: this thread's word of the next board's compact observation
  int prev_plane = 0xFF;  // COBS: the piece channel this thread's square holds in the tile
  auto load_cobs = [&](int b) {
    if (tid < KZ_COBS_WORDS) cw = __ldg(reinterpret_cast<const uint32_t*>(obs) + (size_t)(rows ? rows[b] : b) * KZ_COBS_WORDS + tid);
  };
  if (blockIdx.x < n) {
    if (COBS) load_cobs(blockIdx.x);
    else load_board<288>(regs, board(blockIdx.x), tid);
    load_dy(blockIdx.x);
  }
  for (int b = blockIdx.x; b < n; b += gridDim.x) {
    __syncthreads();  // previous board consumed
    if (COBS) {
      if (tid < KZ_COBS_WORDS) cws[tid] = cw;
    } else {
      store_board<288>(xs, regs, tid);
    }
#pragma unroll
    for (int k = 0; k < DSLOTS; k++) {
      const int i = tid + k * 288;
      if (i < COUT * 81) {
        const int o = i / 81;
        ds[o * DS_STRIDE + (i - o * 81)] = __float2bfloat16(dreg[k]);
      }
    }
    __syncthreads();
    if (COBS) {
      if (tid < 81) {  // this square's piece channel: clear the old one, set the new one
        const int np = reinterpret_cast<const uint8_t*>(cws)[tid];
        __nv_bfloat16* row = xs + tile_row(tid) * XS_STRIDE;
        if (prev_plane != np) {
          if (prev_plane < 28) row[prev_plane] = __float2bfloat16(0.f);
          if (np < 28) row[np] = __float2bfloat16(1.f);
          prev_plane = np;
        }
      }
      for (int i = tid; i < 81 * 9; i += 288) {  // constant channels 28..45 = tile words 14..22 of every square
        const int sq = i / 9, k = i - sq * 9;
        const __nv_bfloat162 v = __floats2bfloat162_rn(__uint_as_float(cws[21 + 2 * k]), __uint_as_float(cws[22 + 2 * k]));
        reinterpret_cast<__nv_bfloat162*>(xs + tile_row(sq) * XS_STRIDE)[14 + k] = v;
      }
      __syncthreads();
    }
    if (b + gridDim.x < n) {  // next board in flight during the products
      if (COBS) load_cobs(b + gridDim.x);
      else load_board<288>(regs, board(b + gridDim.x), tid);
      load_dy(b + gridDim.x);
    }
#pragma unroll
    for (int ks = 0; ks < 6; ks++) {
      uint32_t a[4];
      ldmatrix_x4(a, ds_a + ks * 32);
      // B rows: squares ks*16 + (lane & 15); lanes 0-7 / 8-15 are the k 0-7 / 8-15 halves
      const int xy = ks * 16 + (lane & 15);
      const int row = xy < 81 ? tile_row(xy) + off : ZROW;
      const uint32_t baddr = xs_b + row * XS_STRIDE * 2;
#pragma unroll
      for (int jj = 0; jj < 3; jj++) {
        uint32_t bb[4];
        ldmatrix_x4_trans(bb, baddr + jj * 32);
        mma_bf16(acc[2 * jj], a, bb[0], bb[1]);
        mma_bf16(acc[2 * jj + 1], a, bb[2], bb[3]);
      }
    }
  }
  float* p = part + (size_t)blockIdx.x * COUT * KTOT;
#pragma unroll
  for (int j = 0; j < 6; j++)
#pragma unroll
    for (int e = 0; e < 4; e++) {
      const int o = (lane >> 2) + (e >> 1) * 8, c = j * 8 + (lane & 3) * 2 + (e & 1);
      p[(o * 9 + tap) * CPAD + c] = acc[j][e];
    }
}

// ---- forward from the compact observation: no dense product at all.  A square holds at most one piece, so among
// the 28 piece planes at most one input is non-zero per (output square, tap): out[o][xy] = b[o] + sum over the 9 taps of
// W[o][plane_of(xy + tap)][tap] where that neighbour is occupied, + sum over the non-zero constant planes of
// value x (sum of that plane's weights over the taps that fall on the board at xy: 9 position classes).  ~12 k additions
// per board instead of 536 k multiply-adds and 160 bytes read instead of 14,904.  Operands are rounded to bf16 and
// accumulated in fp32 like the tensor-core path (same products; the constant planes' tap sums are formed first).
constexpr int WP_STRIDE = 9 * COUT + 4;  // floats per plane: rows of different planes fall into different bank groups
__global__ void __launch_bounds__(128) kz_cobs_conv_fwd_kernel(const uint32_t* __restrict__ cobs,
                                                               const long long* __restrict__ rows,
                                                               const float* __restrict__ w, const float* __restrict__ bias,
                                                               int n, int relu, __nv_bfloat16* __restrict__ out) {
  __shared__ __align__(16) float Wp[28 * WP_STRIDE];       // [plane][tap][o]
  __shared__ __align__(16) float Rc[18 * 9 * COUT];        // [constant plane][position class][o]
  __shared__ __align__(16) float Bc[COUT];
  __shared__ __align__(16) uint32_t cbs[4][KZ_COBS_WORDS];
  __shared__ __align__(16) __nv_bfloat16 ys[4][COUT * 81 + 8];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  auto r16 = [](float v) { return __bfloat162float(__float2bfloat16(v)); };
  for (int i = tid; i < 28 * 9 * COUT; i += 128) {
    const int p = i / (9 * COUT), r = i - p * 9 * COUT, tap = r / COUT, o = r - tap * COUT;
    Wp[p * WP_STRIDE + tap * COUT + o] = r16(w[(o * CIN + p) * 9 + tap]);
  }
  for (int i = tid; i < 18 * 9 * COUT; i += 128) {
    const int c = i / (9 * COUT), r = i - c * 9 * COUT, cls = r / COUT, o = r - cls * COUT;
    const int rc = cls / 3, cc = cls - rc * 3;  // 0: first row / column, 1: inner, 2: last
    float sum = 0.f;
    for (int tap = 0; tap < 9; tap++) {
      const int dy = tap / 3 - 1, dx = tap % 3 - 1;
      if ((rc == 0 && dy < 0) || (rc == 2 && dy > 0) || (cc == 0 && dx < 0) || (cc == 2 && dx > 0)) continue;
      sum += r16(w[(o * CIN + 28 + c) * 9 + tap]);
    }
    Rc[i] = sum;
  }
  if (tid < COUT) Bc[tid] = bias ? r16(bias[tid]) : 0.f;
  __syncthreads();
  const uint8_t* sqp = reinterpret_cast<const uint8_t*>(cbs[warp]);
  for (int b = blockIdx.x * 4 + warp; b < n; b += gridDim.x * 4) {
    const uint32_t* src = cobs + (size_t)(rows ? rows[b] : b) * KZ_COBS_WORDS;
    __syncwarp();
    cbs[warp][lane] = __ldg(src + lane);
    if (lane < KZ_COBS_WORDS - 32) cbs[warp][32 + lane] = __ldg(src + 32 + lane);
    __syncwarp();
    const float pv = lane < 18 ? r16(__uint_as_float(cbs[warp][21 + lane])) : 0.f;
    const uint32_t nz = __ballot_sync(0xffffffffu, pv != 0.f);
#pragma unroll 1
    for (int j = 0; j < 3; j++) {
      const int xy = lane + 32 * j;
      const bool act = xy < 81;
      const int r = act ? xy / 9 : 0, c = act ? xy - 9 * r : 0;
      float acc[COUT];
#pragma unroll
      for (int o = 0; o < COUT; o++) acc[o] = Bc[o];
      if (act) {
#pragma unroll
        for (int tap = 0; tap < 9; tap++) {
          const int rr = r + tap / 3 - 1, cc = c + tap % 3 - 1;
          if (rr < 0 || rr > 8 || cc < 0 || cc > 8) continue;
          const int p = sqp[rr * 9 + cc];
          if (p < 28) {
            const float4* wv = reinterpret_cast<const float4*>(Wp + p * WP_STRIDE + tap * COUT);
#pragma unroll
            for (int q = 0; q < 4; q++) {
              const float4 t = wv[q];
              acc[4 * q] += t.x; acc[4 * q + 1] += t.y; acc[4 * q + 2] += t.z; acc[4 * q + 3] += t.w;
            }
          }
        }
      }
      const int cls = (r == 0 ? 0 : (r == 8 ? 2 : 1)) * 3 + (c == 0 ? 0 : (c == 8 ? 2 : 1));
      uint32_t m = nz;
      while (m) {  // warp-uniform
        const int i = __ffs(m) - 1;
        m &= m - 1;
        const float v = __shfl_sync(0xffffffffu, pv, i);
        const float4* rv = reinterpret_cast<const float4*>(Rc + (i * 9 + cls) * COUT);
#pragma unroll
        for (int q = 0; q < 4; q++) {
          const float4 t = rv[q];
          acc[4 * q] = fmaf(v, t.x, acc[4 * q]); acc[4 * q + 1] = fmaf(v, t.y, acc[4 * q + 1]);
          acc[4 * q + 2] = fmaf(v, t.z, acc[4 * q + 2]); acc[4 * q + 3] = fmaf(v, t.w, acc[4 * q + 3]);
        }
      }
      if (act) {
#pragma unroll
        for (int o = 0; o < COUT; o++) ys[warp][o * 81 + xy] = __float2bfloat16(relu && acc[o] == acc[o] ? fmaxf(acc[o], 0.f) : acc[o]);
      }
    }
    __syncwarp();
    uint4* dst = reinterpret_cast<uint4*>(out + (size_t)b * COUT * 81);  // 2,592 B per board: 16-byte aligned
    for (int i = lane; i < COUT * 81 * 2 / 16; i += 32) dst[i] = reinterpret_cast<const uint4*>(ys[warp])[i];
  }
}

// sum the per-CTA partials; scatter into the [16][46][3][3] weight layout and the bias gradient
__global__ void kz_obs_conv_wgrad_reduce_kernel(const float* __restrict__ part, int ctas, float* __restrict__ dw,
                                                float* __restrict__ db) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= COUT * KTOT) return;
  float s = 0.f;
  for (int k = 0; k < ctas; k++) s += part[(size_t)k * COUT * KTOT + i];
  const int o = i / KTOT, r = i - o * KTOT, tap = r / CPAD, c = r - tap * CPAD;
  if (c < CIN) dw[(o * CIN + c) * 9 + tap] = s;
  else if (c == CIN && tap == 4 && db) db[o] = s;
}



// persistent grids: exactly the CTAs that are resident at once (a CTA strides over boards by the grid size)
template <class K>
int resident_ctas(K kernel, int threads) {
  int dev = 0, sms = 148, per_sm = 1;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, 0) != cudaSuccess || per_sm < 1) per_sm = 1;
  return sms * per_sm;
}

}  // namespace

extern "C" {

int kz_obs_conv_fwd(const float* obs, const int64_t* obs_rows, const float* weight, const float* bias, int cout, int n,
                    int relu, void* out_bf16, void* stream) {
  if (!obs || !weight || !out_bf16 || n <= 0 || cout != COUT) return KZ_E_ARG;
  static const int resident = resident_ctas(kz_obs_conv_fwd_kernel, 128);
  kz_obs_conv_fwd_kernel<<<n < resident ? n : resident, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      obs, reinterpret_cast<const long long*>(obs_rows), weight, bias, n, relu, reinterpret_cast<__nv_bfloat16*>(out_bf16));
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? KZ_OK : fail(e);
}

int kz_obs_conv_wgrad_ctas(int n) {
  static const int resident = resident_ctas(kz_obs_conv_wgrad_kernel<false>, 288);
  return n < resident ? (n > 0 ? n : 1) : resident;
}

int kz_cobs_conv_wgrad_ctas(int n) {
  static const int resident = resident_ctas(kz_obs_conv_wgrad_kernel<true>, 288);
  return n < resident ? (n > 0 ? n : 1) : resident;
}

int kz_cobs_conv_fwd(const uint32_t* cobs, const int64_t* cobs_rows, const float* weight, const float* bias, int cout, int n,
                     int relu, void* out_bf16, void* stream) {
  if (!cobs || !weight || !out_bf16 || n <= 0 || cout != COUT || ((uintptr_t)cobs & 3)) return KZ_E_ARG;
  static const int resident = resident_ctas(kz_cobs_conv_fwd_kernel, 128);
  const int want = (n + 3) / 4;
  kz_cobs_conv_fwd_kernel<<<want < resident ? want : resident, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      cobs, reinterpret_cast<const long long*>(cobs_rows), weight, bias, n, relu, reinterpret_cast<__nv_bfloat16*>(out_bf16));
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? KZ_OK : fail(e);
}

int kz_cobs_conv_wgrad(const uint32_t* cobs, const int64_t* cobs_rows, const void* y_bf16, const void* dout, int dout_bf16,
                       int cout, int n, float* workspace, int ctas, float* dweight, float* dbias, void* stream) {
  if (!cobs || !dout || !workspace || !dweight || n <= 0 || cout != COUT || ctas <= 0 || ctas > n || ((uintptr_t)cobs & 3))
    return KZ_E_ARG;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  kz_obs_conv_wgrad_kernel<true><<<ctas, 288, 0, st>>>(reinterpret_cast<const float*>(cobs),
                                                       reinterpret_cast<const long long*>(cobs_rows),
                                                       reinterpret_cast<const __nv_bfloat16*>(y_bf16), dout, dout_bf16, n,
                                                       workspace);
  kz_obs_conv_wgrad_reduce_kernel<<<(COUT * KTOT + 127) / 128, 128, 0, st>>>(workspace, ctas, dweight, dbias);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? KZ_OK : fail(e);
}

int kz_obs_conv_wgrad(const float* obs, const int64_t* obs_rows, const void* y_bf16, const void* dout, int dout_bf16,
                      int cout, int n, float* workspace, int ctas, float* dweight, float* dbias, void* stream) {
  if (!obs || !dout || !workspace || !dweight || n <= 0 || cout != COUT || ctas <= 0 || ctas > n) return KZ_E_ARG;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  kz_obs_conv_wgrad_kernel<false><<<ctas, 288, 0, st>>>(obs, reinterpret_cast<const long long*>(obs_rows),
                                                 reinterpret_cast<const __nv_bfloat16*>(y_bf16), dout, dout_bf16, n, workspace);
  kz_obs_conv_wgrad_reduce_kernel<<<(COUT * KTOT + 127) / 128, 128, 0, st>>>(workspace, ctas, dweight, dbias);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? KZ_OK : fail(e);
}

}  // extern "C"
