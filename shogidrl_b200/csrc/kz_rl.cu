// kz_rl.cu -- sm_100a kernels for the agent/buffer side of the rollout hot path:
//   kz_sample_masked : masked softmax -> Categorical sample / argmax -> log_prob (+ entropy)
//                      (keisei/core/base_actor_critic.py:64-116; torch.distributions.Categorical(probs=...))
//   kz_gae           : reverse-time GAE over a [T][N] rollout (keisei/core/experience_buffer.py:99-145)
//   kz_heuristic_actions : the scripted SimpleHeuristicOpponent's move for every game (keisei/utils/opponents.py)
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <float.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/keisei_b200.h"
#include "kz_common.cuh"

int kz_cuda_fail(cudaError_t e);  // kz_engine.cu: records the message for kz_last_cuda_error

namespace {

inline int fail(cudaError_t e) { return kz_cuda_fail(e); }

__device__ __forceinline__ float ld_logit(const void* row, int i, int bf16) {
  return bf16 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(row)[i]) : reinterpret_cast<const float*>(row)[i];
}

__device__ __forceinline__ uint32_t hash_u32(unsigned long long seed, unsigned long long ctr) {
  unsigned long long x = seed ^ (ctr * 0x9E3779B97F4A7C15ull) ^ 0xD1B54A32D192ED03ull;
  x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull;
  x ^= x >> 27; x *= 0x94D049BB133111EBull;
  x ^= x >> 31;
  return (uint32_t)(x >> 32);
}

// The legal mask of a row is ~0.5 % dense, so every kernel below scans it 16 bytes per lane per load and touches
// logits only at legal entries.  A row is cut into 16-byte windows aligned in memory (whatever the row's own
// alignment); the partial windows at both ends are assembled from byte loads, so no access leaves the row.
struct MaskWindows {
  typedef uint4 Raw;
  const uint8_t* row;
  int shift;  // row address minus the aligned address of window 0
  int nw;
  __device__ __forceinline__ explicit MaskWindows(const void* r) : row(reinterpret_cast<const uint8_t*>(r)) {
    shift = (int)(reinterpret_cast<uintptr_t>(r) & 15);
    nw = (KZ_NUM_ACTIONS + shift + 15) >> 4;
  }
  __device__ __forceinline__ int first(int w) const { return (w << 4) - shift; }  // action index of byte 0 of window w
  // the 16 mask bytes of window w (non-zero = legal); bytes outside the row read as 0
  __device__ __forceinline__ uint4 load(int w) const {
    const int lo = first(w);
    uint4 v = make_uint4(0, 0, 0, 0);
    if (w >= nw) return v;
    if (lo >= 0 && lo + 16 <= KZ_NUM_ACTIONS) {
      v = __ldg(reinterpret_cast<const uint4*>(row + lo));
    } else {
      uint32_t q[4] = {0, 0, 0, 0};
#pragma unroll
      for (int b = 0; b < 16; b++) {
        const int i = lo + b;
        if (i >= 0 && i < KZ_NUM_ACTIONS && row[i]) q[b >> 2] |= 1u << ((b & 3) * 8);
      }
      v = make_uint4(q[0], q[1], q[2], q[3]);
    }
    return v;
  }
  // bit b of the result = byte b of the window is non-zero
  static __device__ __forceinline__ uint32_t bits16(const uint4& v) {
    if (!(v.x | v.y | v.z | v.w)) return 0u;
    // one bit per byte (bit 0 of each byte of the compare result), gathered into a nibble by a carry-free multiply
    auto nib = [](uint32_t x) { return ((__vcmpne4(x, 0) & 0x01010101u) * 0x01020408u) >> 24; };
    return nib(v.x) | (nib(v.y) << 4) | (nib(v.z) << 8) | (nib(v.w) << 12);
  }
  __device__ __forceinline__ bool legal(long long a) const { return row[a] != 0; }
};

// The same windows over a row of the engine's legal BITMAP (kz_step_rollout / kz_legal_bitmap: bit i of the 448-word
// row = action i is legal; 1,792 bytes instead of 13,527).  Window w = bits [16w, 16w + 16) = one half of word w >> 1,
// so the compacted list -- and with it every sum, the sampled action and every gradient -- is the one the byte-mask
// scan of a 16-byte aligned row produces, bit for bit.
struct BitmapWindows {
  typedef uint32_t Raw;
  const uint32_t* row;
  int nw;
  __device__ __forceinline__ explicit BitmapWindows(const void* r) : row(reinterpret_cast<const uint32_t*>(r)) {
    nw = (KZ_NUM_ACTIONS + 15) >> 4;
  }
  __device__ __forceinline__ int first(int w) const { return w << 4; }
  __device__ __forceinline__ uint32_t load(int w) const {
    if (w >= nw) return 0u;
    const uint32_t x = __ldg(row + (w >> 1));
    return (w & 1) ? (x >> 16) : (x & 0xFFFFu);
  }
  static __device__ __forceinline__ uint32_t bits16(uint32_t v) { return v; }
  __device__ __forceinline__ bool legal(long long a) const { return (row[a >> 5] >> (a & 31)) & 1u; }
};

// Compacted list of a row's legal actions in the warp's shared-memory slice.  Scanning the mask lane by lane and
// touching the logits inside that scan would serialise one dependent gather per legal action (a handful of
// lanes active each time); compacting first lets all lanes gather at once.  LIST_CAP covers any Shogi position
// (<= 593 legal moves) in one piece; denser masks are processed in several pieces.
#define MASK_MLP 4                      // window loads in flight per lane
#define LIST_CAP (32 * MASK_MLP * 16)   // one group of windows always fits
struct LegalList {
  uint16_t* buf;
  int cnt;
  bool whole;  // buf holds every legal action of the row: later passes replay it instead of rescanning
};

// f(action index) for every legal action of the row, a fixed order, all lanes taking list entries round-robin
// (entry j of a piece goes to lane j % 32)
template <class WIN, class F>
__device__ __forceinline__ void each_legal_of_row(const WIN& W, int lane, LegalList& ll, F&& f) {
  if (!ll.whole) {
    ll.cnt = 0;
    bool flushed = false;
    typename WIN::Raw nx[MASK_MLP];  // next group's windows, loaded one group ahead of their compaction
#pragma unroll
    for (int k = 0; k < MASK_MLP; k++) nx[k] = W.load(lane + 32 * k);
    for (int w0 = lane; w0 - lane < W.nw; w0 += 32 * MASK_MLP) {
      uint32_t v[MASK_MLP];  // 16 legality bits per window
#pragma unroll
      for (int k = 0; k < MASK_MLP; k++) {
        v[k] = WIN::bits16(nx[k]);
        nx[k] = W.load(w0 + 32 * (MASK_MLP + k));
      }
      int c = 0;
#pragma unroll
      for (int k = 0; k < MASK_MLP; k++) c += __popc(v[k]);
      int incl = c;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += t; }
      const int total = __shfl_sync(FULL, incl, 31);
      if (ll.cnt + total > LIST_CAP) {  // piece full: consume it
        __syncwarp();
        for (int j = lane; j < ll.cnt; j += 32) f((int)ll.buf[j]);
        __syncwarp();
        ll.cnt = 0;
        flushed = true;
      }
      int at = ll.cnt + incl - c;
#pragma unroll
      for (int k = 0; k < MASK_MLP; k++) {
        uint32_t z = v[k];
        const int lo = W.first(w0 + 32 * k);
        while (z) {
          const int b = __ffs(z) - 1;
          z &= z - 1;
          ll.buf[at++] = (uint16_t)(lo + b);
        }
      }
      ll.cnt += total;
    }
    ll.whole = !flushed;
    __syncwarp();
  }
  for (int j = lane; j < ll.cnt; j += 32) f((int)ll.buf[j]);
  if (!ll.whole) __syncwarp();  // the next scan overwrites the slice
}

// One warp per row.  Element order for the inverse CDF: lane-major over the mask windows (lane 0's windows
// 0, 32, 64, ... in ascending action order, then lane 1's, ...), a fixed permutation of the action axis, so the
// sampled law is the masked softmax.
template <class WIN>  // MaskWindows: byte mask rows; BitmapWindows: 448-word legal bitmap rows.  ldm in bytes.
__global__ void __launch_bounds__(256, 4) kz_sample_kernel(const void* logits, int bf16, long long ld, const void* mask,
                                                        long long ldm, int n, unsigned long long seed,
                                                        unsigned long long offset, const unsigned long long* offset_dev,
                                                        void* actions, int actions_i64, float* logp, float* entropy,
                                                        int deterministic) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n) return;
  if (offset_dev) offset += *offset_dev;  // draw counter kept on the device: a captured launch draws fresh numbers on replay
  const char* lrow = reinterpret_cast<const char*>(logits) + (size_t)row * ld * (bf16 ? 2 : 4);
  const WIN W(reinterpret_cast<const char*>(mask) + (size_t)row * ldm);
  __shared__ uint16_t s_list[8][LIST_CAP];
  LegalList ll{s_list[threadIdx.x >> 5], 0, false};
  const int A = KZ_NUM_ACTIONS;

  // pass 1: online max / sum of exp over this lane's share of the legal entries; per-lane argmax (lowest index on ties)
  float m = -INFINITY, s = 0.f;
  int amax = 0x7fffffff;
  each_legal_of_row(W, lane, ll, [&](int i) {
    const float x = ld_logit(lrow, i, bf16);
    if (x > m) { s = s * expf(m - x) + 1.f; m = x; amax = i; }
    else { s += expf(x - m); if (x == m && i < amax) amax = i; }
  });
  float M = m;
#pragma unroll
  for (int o = 16; o; o >>= 1) M = fmaxf(M, __shfl_xor_sync(FULL, M, o));
  long long act = -1;
  float lp = 0.f, ent = 0.f;
  if (!(M > -INFINITY)) {
    // no legal entry (or all legal logits are -inf): softmax is NaN -> uniform over all actions
    // (base_actor_critic.py:93-101)
    const float p = 1.0f / (float)A;
    if (deterministic) act = 0;
    else act = (long long)(((unsigned long long)hash_u32(seed, offset + row) * (unsigned long long)A) >> 32);
    lp = logf(p);
    ent = -logf(p);
  } else {
    const float mys = (m > -INFINITY) ? s * expf(m - M) : 0.f;  // this lane's sum rescaled to the row max
    float tot = mys;
#pragma unroll
    for (int o = 16; o; o >>= 1) tot += __shfl_xor_sync(FULL, tot, o);
    const float inv = 1.0f / tot;
    // argmax of probs == argmax of legal logits; lowest index wins ties
    int best = (m == M) ? amax : 0x7fffffff;
#pragma unroll
    for (int o = 16; o; o >>= 1) best = min(best, __shfl_xor_sync(FULL, best, o));
    int pick = best;
    if (!deterministic) {
      // inverse CDF in the order "lane 0's entries, lane 1's entries, ...": find the lane L holding the target,
      // then lane L walks its own entries (1/32 of the legal actions)
      const float u = (float)(hash_u32(seed, offset + row) >> 8) * (1.0f / 16777216.0f);
      const float target = u * tot;
      float incl = mys;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const float t = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += t; }
      const uint32_t hit = __ballot_sync(FULL, incl > target && mys > 0.f);
      int L = hit ? __ffs(hit) - 1 : -1;
      if (L < 0) {  // rounding pushed the target past the total: take the last lane that has mass
        const uint32_t have = __ballot_sync(FULL, mys > 0.f);
        L = 31 - __clz(have);
      }
      float run = incl - mys;
      int found = -1, last = -1;
      each_legal_of_row(W, lane, ll, [&](int i) {
        if (lane != L) return;
        const float e = expf(ld_logit(lrow, i, bf16) - M);
        if (e > 0.f) {
          last = i;
          run += e;
          if (found < 0 && run > target) found = i;
        }
      });
      if (found < 0) found = last;
      found = __shfl_sync(FULL, found, L);
      if (found >= 0) pick = found;  // (< 0: every exp underflowed on the re-read; keep the argmax)
    }
    act = pick;
    // Categorical(probs=p): logits = log(clamp(p, eps, 1 - eps)) with eps = FLT_EPSILON
    const float eps = FLT_EPSILON;
    if (lane == 0) {
      const float p = expf(ld_logit(lrow, pick, bf16) - M) * inv;
      lp = logf(fminf(fmaxf(p, eps), 1.0f - eps));
    }
    if (entropy) {
      float h = 0.f;
      each_legal_of_row(W, lane, ll, [&](int i) {
        const float p = expf(ld_logit(lrow, i, bf16) - M) * inv;
        h -= p * logf(fminf(fmaxf(p, eps), 1.0f - eps));
      });
#pragma unroll
      for (int o = 16; o; o >>= 1) h += __shfl_xor_sync(FULL, h, o);
      ent = h;
    }
  }
  if (lane == 0) {
    if (actions_i64) reinterpret_cast<long long*>(actions)[row] = act;
    else reinterpret_cast<int*>(actions)[row] = (int)act;
    if (logp) logp[row] = lp;
    if (entropy) entropy[row] = ent;
  }
}

// ---- SimpleHeuristicOpponent.select_move (keisei/utils/opponents.py) for n games, one warp per game ----
// The legal moves fall into three tiers: 0 capture (the destination holds a piece of the other colour; legal moves never
// land on own pieces, so "occupied" suffices), 1 non-promoting move of the mover's unpromoted pawn, 2 everything else,
// every drop included.  The pick is uniform over the first non-empty tier: its k-th member in ascending action order,
// k = mulhi(rand32(seed, env, step), tier size) -- kz_step's next_actions convention, so a CPU replay can follow it.
// A board move's index is from*160 + 2*to' + promote, so the 16 actions [16A, 16A + 16) of window A < 810 share the
// source square A / 10 and cover the destinations to' = 8*(A % 10) .. +7 (to = to' + (to' >= from)); windows 810.. are
// drops.  A window's tiers are then its legality bits ANDed with 8 bits of the enemy-occupancy bitboard (spread to bit
// pairs) and, when the source holds an own pawn, with the non-promoting (even) bits.
#define HEUR_WINDOWS ((KZ_NUM_ACTIONS + 15) / 16)  // 846
#define HEUR_ROUNDS ((HEUR_WINDOWS + 31) / 32)      // 27: window A = 32 * round + lane

// legality bits of actions [16A, 16A + 16); MaskWindows' windows follow the row's own 16-byte phase, so two are merged
__device__ __forceinline__ uint32_t legal16(const MaskWindows& W, int A) {
  const uint32_t lo = MaskWindows::bits16(W.load(A));
  if (!W.shift) return lo;
  return ((lo >> W.shift) | (MaskWindows::bits16(W.load(A + 1)) << (16 - W.shift))) & 0xFFFFu;
}
__device__ __forceinline__ uint32_t legal16(const BitmapWindows& W, int A) { return W.load(A); }

// capture (t0) and pawn (t1) bits of window A's legality bits v; the rest of v is tier 2
__device__ __forceinline__ void heur_classify(uint32_t v, int A, const BB& enemy, const BB& pawns, uint32_t& t0, uint32_t& t1) {
  t0 = t1 = 0u;
  if (A >= 810 || !v) return;
  const int from = A / 10, lo = 8 * (A - 10 * from);
  const int wd = lo >> 5;
  const uint32_t a = wd == 0 ? enemy.w0 : (wd == 1 ? enemy.w1 : enemy.w2);
  const uint32_t b = wd == 0 ? enemy.w1 : (wd == 1 ? enemy.w2 : 0u);
  const uint32_t x = __funnelshift_r(a, b, lo & 31) & 0x1FFu;  // enemy bits of squares lo .. lo + 8
  const uint32_t below = lowmask32(from - lo) & 0xFFu;         // to' < from: to = to'; above: to = to' + 1
  const uint32_t e8 = ((x & below) | ((x >> 1) & ~below)) & 0xFFu;
  t0 = v & (spread16(e8) * 3u);
  if (bb_test(pawns, from)) t1 = v & ~t0 & 0x5555u;
}

template <class WIN>  // MaskWindows: byte mask rows; BitmapWindows: 448-word legal bitmap rows.  ldm in bytes.
__global__ void __launch_bounds__(256) kz_heuristic_kernel(const uint8_t* __restrict__ boards, const uint8_t* __restrict__ meta,
                                                           int n, const void* legal, long long ldm, void* actions,
                                                           int actions_i64, uint8_t* tier_out, int32_t* count_out,
                                                           unsigned long long seed, uint32_t rng_step, uint32_t env_offset) {
  __shared__ uint16_t s_bits[8][HEUR_ROUNDS * 32];  // the row's legality bits, window by window, for the selection pass
  const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
  const int g = blockIdx.x * 8 + wi;
  if (g >= n) return;
  const uint8_t* b = boards + (size_t)g * 96;
  const int side = meta[(size_t)g * 32 + 14];
  uint32_t e[3], p[3];
#pragma unroll
  for (int j = 0; j < 3; j++) {
    const int s = lane + 32 * j;
    const int c = s < 81 ? b[s] : 0;
    e[j] = __ballot_sync(FULL, c != 0 && code_color(c) != side);
    p[j] = __ballot_sync(FULL, c == 1 + 14 * side);
  }
  const BB enemy{e[0], e[1], e[2]}, pawns{p[0], p[1], p[2]};
  const WIN W(reinterpret_cast<const char*>(legal) + (size_t)g * ldm);
  uint16_t* bits = s_bits[wi];

  // pass 1: tier sizes (each lane writes and later reads only its own windows: no warp barrier needed)
  int c0 = 0, c1 = 0, c2 = 0;
#pragma unroll 9
  for (int r = 0; r < HEUR_ROUNDS; r++) {
    const int A = 32 * r + lane;
    uint32_t v = A < HEUR_WINDOWS ? legal16(W, A) : 0u;
    if (A == HEUR_WINDOWS - 1) v &= (1u << (KZ_NUM_ACTIONS - 16 * (HEUR_WINDOWS - 1))) - 1u;  // bitmap pad bits
    uint32_t t0, t1;
    heur_classify(v, A, enemy, pawns, t0, t1);
    c0 += __popc(t0); c1 += __popc(t1); c2 += __popc(v & ~(t0 | t1));
    bits[A] = (uint16_t)v;
  }
  const int n0 = (int)__reduce_add_sync(FULL, (unsigned)c0), n1 = (int)__reduce_add_sync(FULL, (unsigned)c1),
            n2 = (int)__reduce_add_sync(FULL, (unsigned)c2);
  const int tier = n0 ? 0 : (n1 ? 1 : (n2 ? 2 : 255));
  const int cnt = n0 ? n0 : (n1 ? n1 : n2);

  // pass 2: the k-th member of the tier, rounds in ascending action order (lane order inside a round)
  long long pick = -1;
  if (cnt > 0) {
    const int k = (int)(((unsigned long long)rand32(seed, (unsigned long long)env_offset + (unsigned long long)g, rng_step) *
                         (unsigned long long)cnt) >> 32);
    int base = 0;
    for (int r = 0; r < HEUR_ROUNDS; r++) {
      const int A = 32 * r + lane;
      const uint32_t v = bits[A];
      uint32_t t0, t1;
      heur_classify(v, A, enemy, pawns, t0, t1);
      uint32_t m = tier == 0 ? t0 : (tier == 1 ? t1 : (v & ~(t0 | t1)));
      const int c = __popc(m);
      const int tot = (int)__reduce_add_sync(FULL, (unsigned)c);
      if (k < base + tot) {  // warp-uniform
        int incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += t; }
        int rem = k - base - (incl - c);
        int found = -1;
        if (rem >= 0 && rem < c) {
          while (rem--) m &= m - 1;
          found = 16 * A + __ffs(m) - 1;
        }
        const uint32_t own = __ballot_sync(FULL, found >= 0);
        pick = __shfl_sync(FULL, found, __ffs(own) - 1);
        break;
      }
      base += tot;
    }
  }
  if (lane == 0) {
    if (actions_i64) reinterpret_cast<long long*>(actions)[g] = pick;
    else reinterpret_cast<int*>(actions)[g] = (int)pick;
    if (tier_out) tier_out[g] = (uint8_t)tier;
    if (count_out) count_out[g] = cnt;
  }
}

// GAE, exact variant: one thread per env column, sequential over time in the reference's op order with
// every operation rounded separately (__fmul_rn/__fadd_rn are never contracted into FMAs).  Loads are
// coalesced across envs.  Used when N offers enough parallelism.
__global__ void kz_gae_columns_kernel(const float* __restrict__ rewards, const float* __restrict__ values,
                                      const uint8_t* __restrict__ dones, const float* __restrict__ last_value, int T,
                                      int N, float gamma, float gl, float* __restrict__ adv, float* __restrict__ ret) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float gae = 0.f;
  float nv = last_value[n];
#pragma unroll 4
  for (int t = T - 1; t >= 0; t--) {
    const size_t i = (size_t)t * N + n;
    const float r = rewards[i], v = values[i];
    const float m = dones[i] ? 0.f : 1.f;
    const float delta = __fsub_rn(__fadd_rn(r, __fmul_rn(__fmul_rn(gamma, nv), m)), v);
    gae = __fadd_rn(delta, __fmul_rn(__fmul_rn(gl, m), gae));
    adv[i] = gae;
    ret[i] = __fadd_rn(gae, v);
    nv = v;
  }
}

// GAE, warp-scan variant for narrow rollouts (small N, e.g. the reference's flat N = 1 buffer): one warp
// per env column, 32 timesteps per round processed as a reverse inclusive scan over the affine maps
// gae_t = delta_t + c_t * gae_{t+1}.  Composition reassociates the fp32 products, so this variant agrees
// with the sequential order to ~1e-6 relative (north-star tolerance 1e-5), not bit-for-bit.
__global__ void kz_gae_warpscan_kernel(const float* __restrict__ rewards, const float* __restrict__ values,
                                       const uint8_t* __restrict__ dones, const float* __restrict__ last_value, int T,
                                       int N, float gamma, float gl, float* __restrict__ adv, float* __restrict__ ret) {
  const int lane = threadIdx.x & 31;
  const int n = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (n >= N) return;
  float carry = 0.f;  // gae_{t+1} entering the current round
  for (int hi = T - 1; hi >= 0; hi -= 32) {
    const int t = hi - lane;  // lane 0 = latest timestep of the round
    float a = 1.f, b = 0.f, v = 0.f;
    if (t >= 0) {
      const size_t i = (size_t)t * N + n;
      v = values[i];
      const float m = dones[i] ? 0.f : 1.f;
      const float nv = (t == T - 1) ? last_value[n] : values[i + N];
      b = __fsub_rn(__fadd_rn(rewards[i], __fmul_rn(__fmul_rn(gamma, nv), m)), v);  // delta_t
      a = __fmul_rn(gl, m);                                                          // c_t
    }
    // inclusive scan in lane order (= reverse time): f_lane o f_{lane-1} o ... o f_0
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const float pa = __shfl_up_sync(FULL, a, o), pb = __shfl_up_sync(FULL, b, o);
      if (lane >= o) { b = fmaf(a, pb, b); a = a * pa; }
    }
    const float g = fmaf(a, carry, b);
    if (t >= 0) {
      const size_t i = (size_t)t * N + n;
      adv[i] = g;
      ret[i] = g + v;
    }
    carry = __shfl_sync(FULL, g, 31);
  }
}


// ------------------------------------------------------------------------------------------------
// Fused evaluation of taken actions for the PPO update (BaseActorCriticModel.evaluate_actions,
// keisei/core/base_actor_critic.py:118-184): masked softmax over 13,527 logits, log-prob of the taken action and
// entropy with torch.distributions.Categorical(probs)'s clamp(p, eps, 1 - eps), one warp per row, and the
// matching backward.  Replaces ~30 elementwise ATen passes over [B, 13527] by two reads (forward) and one
// read + one write (backward).  Forward saves per row: max M, normaliser Z, S = sum_i g_i p_i with
// g_i = dH/dp_i; rows without a legal action fall back to the uniform distribution with zero gradient.
__device__ __forceinline__ float ent_g(float p, float eps) {  // dH/dp for H = -sum p log(clamp(p))
  if (p < eps) return -logf(eps);
  if (p > 1.0f - eps) return -logf(1.0f - eps);
  return -(logf(p) + 1.0f);
}

template <class WIN>
__global__ void __launch_bounds__(256, 4) kz_eval_fwd_kernel(const void* logits, int bf16, long long ld, const void* mask,
                                                          long long ldm, const long long* mask_rows, const long long* actions,
                                                          int n, float* logp, float* entropy, float* saved /*[n][4]*/) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n) return;
  const char* lrow = reinterpret_cast<const char*>(logits) + (size_t)row * ld * (bf16 ? 2 : 4);
  const WIN W(reinterpret_cast<const char*>(mask) + (size_t)(mask_rows ? mask_rows[row] : row) * ldm);
  __shared__ uint16_t s_list[8][LIST_CAP];
  LegalList ll{s_list[threadIdx.x >> 5], 0, false};
  const int A = KZ_NUM_ACTIONS;
  const float eps = FLT_EPSILON;
  float m = -INFINITY, s = 0.f;
  each_legal_of_row(W, lane, ll, [&](int i) {
    const float x = ld_logit(lrow, i, bf16);
    if (x > m) { s = s * expf(m - x) + 1.f; m = x; }
    else s += expf(x - m);
  });
  float M = m;
#pragma unroll
  for (int o = 16; o; o >>= 1) M = fmaxf(M, __shfl_xor_sync(FULL, M, o));
  float lp, ent, Z = 0.f, S = 0.f;
  if (!(M > -INFINITY)) {  // NaN softmax -> uniform (base_actor_critic.py:166-174); constant, so no gradient
    lp = logf(1.0f / (float)A);
    ent = -lp;
    M = INFINITY;  // marks the row for the backward pass
  } else {
    float z = (m > -INFINITY) ? s * expf(m - M) : 0.f;
#pragma unroll
    for (int o = 16; o; o >>= 1) z += __shfl_xor_sync(FULL, z, o);
    Z = z;
    const float inv = 1.0f / Z;
    float h = 0.f, sg = 0.f;
    each_legal_of_row(W, lane, ll, [&](int i) {
      const float p = expf(ld_logit(lrow, i, bf16) - M) * inv;
      h -= p * logf(fminf(fmaxf(p, eps), 1.0f - eps));
      sg += ent_g(p, eps) * p;
    });
#pragma unroll
    for (int o = 16; o; o >>= 1) { h += __shfl_xor_sync(FULL, h, o); sg += __shfl_xor_sync(FULL, sg, o); }
    ent = h; S = sg;
    const long long a = actions[row];
    float pa = 0.f;
    if (a >= 0 && a < A && W.legal(a)) pa = expf(ld_logit(lrow, (int)a, bf16) - M) * inv;
    lp = logf(fminf(fmaxf(pa, eps), 1.0f - eps));
  }
  if (lane == 0) {
    logp[row] = lp; entropy[row] = ent;
    saved[(size_t)row * 4 + 0] = M; saved[(size_t)row * 4 + 1] = Z; saved[(size_t)row * 4 + 2] = S;
  }
}

// zero `bytes` bytes at p (2-byte aligned, even length) with one warp: 16-byte stores between 2-byte edges
__device__ __forceinline__ void zero_row(char* p, size_t bytes, int lane) {
  const size_t head = min((size_t)((16 - (reinterpret_cast<uintptr_t>(p) & 15)) & 15), bytes);
  const size_t body = (bytes - head) & ~(size_t)15;
  if ((size_t)lane * 2 < head) *reinterpret_cast<uint16_t*>(p + lane * 2) = 0;
  uint4* q = reinterpret_cast<uint4*>(p + head);
  for (size_t k = lane; k < body / 16; k += 32) q[k] = make_uint4(0, 0, 0, 0);
  const size_t tail = bytes - head - body;
  if ((size_t)lane * 2 < tail) *reinterpret_cast<uint16_t*>(p + head + body + lane * 2) = 0;
}

template <class WIN>
__global__ void __launch_bounds__(256, 4) kz_eval_bwd_kernel(const void* logits, int bf16, long long ld, const void* mask,
                                                          long long ldm, const long long* mask_rows, const long long* actions,
                                                          int n, const float* dlogp, const float* dent, const float* saved,
                                                          void* dlogits, long long ldg, long long* dbias_q44) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n) return;
  const char* lrow = reinterpret_cast<const char*>(logits) + (size_t)row * ld * (bf16 ? 2 : 4);
  const WIN W(reinterpret_cast<const char*>(mask) + (size_t)(mask_rows ? mask_rows[row] : row) * ldm);
  char* grow = reinterpret_cast<char*>(dlogits) + (size_t)row * ldg * (bf16 ? 2 : 4);
  const int A = KZ_NUM_ACTIONS;
  const float eps = FLT_EPSILON;
  const float M = saved[(size_t)row * 4], Z = saved[(size_t)row * 4 + 1], S = saved[(size_t)row * 4 + 2];
  const float gl = dlogp[row], ge = dent[row];
  const bool dead = !(M < INFINITY);  // uniform-fallback row
  const float inv = dead ? 0.f : 1.0f / Z;
  const long long a = actions[row];
  float pa = 0.f;
  if (!dead && a >= 0 && a < A && W.legal(a)) pa = expf(ld_logit(lrow, (int)a, bf16) - M) * inv;
  const float wl = (pa > eps && pa < 1.0f - eps) ? gl : 0.f;  // clamp passes gradient only inside (eps, 1 - eps)
  // dlogits is zero except at legal actions: clear the row with 16-byte stores, then scatter the legal entries
  const int esz = bf16 ? 2 : 4;
  zero_row(grow, (size_t)A * esz, lane);
  if (dead) return;
  __syncwarp();  // orders the clearing stores before the scattered ones (different lanes, same addresses)
  __shared__ uint16_t s_list[8][LIST_CAP];
  LegalList ll{s_list[threadIdx.x >> 5], 0, false};
  each_legal_of_row(W, lane, ll, [&](int i) {
    const float p = expf(ld_logit(lrow, i, bf16) - M) * inv;
    const float g = ge * p * (ent_g(p, eps) - S) + wl * ((i == a ? 1.f : 0.f) - p);
    if (bf16) reinterpret_cast<__nv_bfloat16*>(grow)[i] = __float2bfloat16(g);
    else reinterpret_cast<float*>(grow)[i] = g;
    // column sum = bias gradient of the policy head, accumulated in Q20.44 fixed point: integer addition is
    // associative, so the result does not depend on the order the rows arrive in (an fp32 atomicAdd does); scaling by
    // 2^44 is exact in fp32 and |g| <= ~2 keeps 2^20 rows away from overflow (result unused: RED in L2)
    if (dbias_q44) atomicAdd(reinterpret_cast<unsigned long long*>(dbias_q44) + i,
                             (unsigned long long)__float2ll_rn(ldexpf(g, 44)));
  });
}

// ------------------------------------------------------------------------------------------------
// PPO clipped-surrogate loss of one minibatch (keisei/core/ppo_agent.py:332-372) with its gradients in closed
// form: ratio = exp(new_lp - old_lp); policy = -mean(min(ratio A, clamp(ratio, 1 - e, 1 + e) A));
// value = mean((v - R)^2); entropy term = -mean(H); loss = policy + c_v value + c_e entropy term.
// One CTA (a minibatch is a few thousand scalars per vector): replaces ~40 elementwise launches and their
// autograd nodes.  out[0] = loss, out[1..5] = policy, value, entropy term, mean(old_lp - new_lp), clip fraction.
// Gradients (already scaled by grad_scale, e.g. 1 / world size): torch.min passes the gradient to the smaller
// argument and ties (ratio inside the clip range: both arguments equal) recombine to the same value, so
// d policy / d new_lp = -(1/n) A ratio unless the clipped branch is the strict minimum.
__global__ void __launch_bounds__(1024) kz_ppo_loss_kernel(const float* __restrict__ new_lp, const float* __restrict__ ent,
                                                           const float* __restrict__ new_v, const float* __restrict__ old_lp,
                                                           const float* __restrict__ adv, const float* __restrict__ ret, int n,
                                                           float clip_eps, float value_coef, float entropy_coef,
                                                           float grad_scale, float* __restrict__ out,
                                                           float* __restrict__ d_lp, float* __restrict__ d_ent,
                                                           float* __restrict__ d_v) {
  __shared__ float red[5][32];
  float acc[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
  const float inv_n = 1.0f / (float)n;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float lp = new_lp[i], olp = old_lp[i], a = adv[i];
    const float ratio = expf(lp - olp);
    const float clamped = fminf(fmaxf(ratio, 1.0f - clip_eps), 1.0f + clip_eps);
    const float s1 = ratio * a, s2 = clamped * a;
    acc[0] -= fminf(s1, s2);
    const float dv = new_v[i] - ret[i];
    acc[1] += dv * dv;
    acc[2] -= ent[i];
    acc[3] += olp - lp;
    acc[4] += fabsf(ratio - 1.0f) > clip_eps ? 1.f : 0.f;
    // d min(s1, s2) / d ratio: a through s1 when s1 <= s2 (ties: half through each, and s2 passes it on inside the
    // range, where the tie happens); through s2 only inside the clip range, i.e. never when s2 is the strict minimum
    const float g_ratio = (s1 <= s2) ? a : 0.f;
    d_lp[i] = -inv_n * g_ratio * ratio * grad_scale;
    d_ent[i] = -inv_n * entropy_coef * grad_scale;
    d_v[i] = 2.0f * inv_n * dv * value_coef * grad_scale;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 5; k++) {
    float v = acc[k];
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    if (lane == 0) red[k][warp] = v;
  }
  __syncthreads();
  if (warp == 0) {
    float tot[5];
#pragma unroll
    for (int k = 0; k < 5; k++) {
      float v = lane < (int)(blockDim.x >> 5) ? red[k][lane] : 0.f;
#pragma unroll
      for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
      tot[k] = v * inv_n;
    }
    if (lane == 0) {
      out[0] = tot[0] + value_coef * tot[1] + entropy_coef * tot[2];
#pragma unroll
      for (int k = 0; k < 5; k++) out[1 + k] = tot[k];
    }
  }
}

}  // namespace


extern "C" {

static int sample_impl(const void* logits, int logits_bf16, int64_t ld, const void* mask, int64_t ldm_bytes, int bitmap, int n,
                       uint64_t seed, uint64_t offset, const uint64_t* offset_dev, void* actions, int actions_i64, float* logp,
                       float* entropy, int deterministic, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const unsigned long long* od = reinterpret_cast<const unsigned long long*>(offset_dev);
  if (bitmap)
    kz_sample_kernel<BitmapWindows><<<(n + 7) / 8, 256, 0, st>>>(logits, logits_bf16, ld, mask, ldm_bytes, n, seed, offset, od,
                                                                  actions, actions_i64, logp, entropy, deterministic);
  else
    kz_sample_kernel<MaskWindows><<<(n + 7) / 8, 256, 0, st>>>(logits, logits_bf16, ld, mask, ldm_bytes, n, seed, offset, od,
                                                                actions, actions_i64, logp, entropy, deterministic);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? KZ_OK : fail(e);
}

int kz_sample_masked(const void* logits, int logits_bf16, int64_t ld, const uint8_t* mask, int64_t ldm, int n,
                     uint64_t seed, uint64_t offset, const uint64_t* offset_dev, void* actions, int actions_i64, float* logp,
                     float* entropy, int deterministic, void* stream) {
  if (!logits || !mask || !actions || n <= 0 || ld < KZ_NUM_ACTIONS || ldm < KZ_NUM_ACTIONS || ((uintptr_t)offset_dev & 7))
    return KZ_E_ARG;
  return sample_impl(logits, logits_bf16, ld, mask, ldm, 0, n, seed, offset, offset_dev, actions, actions_i64, logp, entropy,
                     deterministic, stream);
}

int kz_sample_bitmap(const void* logits, int logits_bf16, int64_t ld, const uint32_t* bitmap, int64_t ldb_words, int n,
                     uint64_t seed, uint64_t offset, const uint64_t* offset_dev, void* actions, int actions_i64, float* logp,
                     float* entropy, int deterministic, void* stream) {
  if (!logits || !bitmap || !actions || n <= 0 || ld < KZ_NUM_ACTIONS || ldb_words < KZ_BITMAP_WORDS_MIN ||
      ((uintptr_t)bitmap & 3) || ((uintptr_t)offset_dev & 7))
    return KZ_E_ARG;
  return sample_impl(logits, logits_bf16, ld, bitmap, ldb_words * 4, 1, n, seed, offset, offset_dev, actions, actions_i64, logp,
                     entropy, deterministic, stream);
}

int kz_heuristic_actions(const void* state, int n, int hist_cap, const uint8_t* mask, int64_t mask_stride,
                         const uint32_t* bitmap, int64_t bitmap_stride_words, void* actions, int actions_i64, uint8_t* tier,
                         int32_t* tier_count, uint64_t seed, uint32_t rng_step, uint32_t env_offset, void* stream) {
  int64_t offs[3], total = 0;
  if (!state || !actions || (mask == nullptr) == (bitmap == nullptr) || kz_state_layout(n, hist_cap, offs, &total) != KZ_OK)
    return KZ_E_ARG;
  if (mask && mask_stride < KZ_NUM_ACTIONS) return KZ_E_ARG;
  if (bitmap && (bitmap_stride_words < KZ_BITMAP_WORDS_MIN || ((uintptr_t)bitmap & 3))) return KZ_E_ARG;
  if (((uintptr_t)actions & (actions_i64 ? 7 : 3)) || ((uintptr_t)tier_count & 3)) return KZ_E_ARG;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const uint8_t* base = reinterpret_cast<const uint8_t*>(state);
  if (bitmap)
    kz_heuristic_kernel<BitmapWindows><<<(n + 7) / 8, 256, 0, st>>>(base + offs[0], base + offs[1], n, bitmap,
                                                                     bitmap_stride_words * 4, actions, actions_i64, tier,
                                                                     tier_count, seed, rng_step, env_offset);
  else
    kz_heuristic_kernel<MaskWindows><<<(n + 7) / 8, 256, 0, st>>>(base + offs[0], base + offs[1], n, mask, mask_stride,
                                                                   actions, actions_i64, tier, tier_count, seed, rng_step,
                                                                   env_offset);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? KZ_OK : fail(e);
}

int kz_gae(const float* rewards, const float* values, const uint8_t* dones, const float* last_value, int T, int N,
           float gamma, float gamma_lambda, float* adv, float* ret, void* stream) {
  if (!rewards || !values || !dones || !last_value || !adv || !ret || T <= 0 || N <= 0) return KZ_E_ARG;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (N >= 2048) {
    kz_gae_columns_kernel<<<(N + 127) / 128, 128, 0, st>>>(rewards, values, dones, last_value, T, N, gamma, gamma_lambda,
                                                           adv, ret);
  } else {
    kz_gae_warpscan_kernel<<<(N + 3) / 4, 128, 0, st>>>(rewards, values, dones, last_value, T, N, gamma, gamma_lambda, adv,
                                                        ret);
  }
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? KZ_OK : fail(e);
}

static int eval_fwd_impl(const void* logits, int logits_bf16, int64_t ld, const void* mask, int64_t ldm_bytes, int bitmap,
                         const int64_t* mask_rows, const int64_t* actions, int n, float* logp, float* entropy,
                         float* saved4, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const long long* mr = reinterpret_cast<const long long*>(mask_rows);
  const long long* ac = reinterpret_cast<const long long*>(actions);
  if (bitmap)
    kz_eval_fwd_kernel<BitmapWindows><<<(n + 7) / 8, 256, 0, st>>>(logits, logits_bf16, ld, mask, ldm_bytes, mr, ac, n, logp,
                                                                    entropy, saved4);
  else
    kz_eval_fwd_kernel<MaskWindows><<<(n + 7) / 8, 256, 0, st>>>(logits, logits_bf16, ld, mask, ldm_bytes, mr, ac, n, logp,
                                                                  entropy, saved4);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? KZ_OK : fail(e);
}

static int eval_bwd_impl(const void* logits, int logits_bf16, int64_t ld, const void* mask, int64_t ldm_bytes, int bitmap,
                         const int64_t* mask_rows, const int64_t* actions, int n, const float* dlogp, const float* dentropy,
                         const float* saved4, void* dlogits, int64_t ldg, int64_t* dbias_q44, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const long long* mr = reinterpret_cast<const long long*>(mask_rows);
  const long long* ac = reinterpret_cast<const long long*>(actions);
  long long* db = reinterpret_cast<long long*>(dbias_q44);
  if (bitmap)
    kz_eval_bwd_kernel<BitmapWindows><<<(n + 7) / 8, 256, 0, st>>>(logits, logits_bf16, ld, mask, ldm_bytes, mr, ac, n, dlogp,
                                                                    dentropy, saved4, dlogits, ldg, db);
  else
    kz_eval_bwd_kernel<MaskWindows><<<(n + 7) / 8, 256, 0, st>>>(logits, logits_bf16, ld, mask, ldm_bytes, mr, ac, n, dlogp,
                                                                  dentropy, saved4, dlogits, ldg, db);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? KZ_OK : fail(e);
}

int kz_eval_masked_fwd(const void* logits, int logits_bf16, int64_t ld, const uint8_t* mask, int64_t ldm,
                       const int64_t* mask_rows, const int64_t* actions, int n, float* logp, float* entropy, float* saved4,
                       void* stream) {
  if (!logits || !mask || !actions || !logp || !entropy || !saved4 || n <= 0 || ld < KZ_NUM_ACTIONS || ldm < KZ_NUM_ACTIONS)
    return KZ_E_ARG;
  return eval_fwd_impl(logits, logits_bf16, ld, mask, ldm, 0, mask_rows, actions, n, logp, entropy, saved4, stream);
}

int kz_eval_bitmap_fwd(const void* logits, int logits_bf16, int64_t ld, const uint32_t* bitmap, int64_t ldb_words,
                       const int64_t* bitmap_rows, const int64_t* actions, int n, float* logp, float* entropy, float* saved4,
                       void* stream) {
  if (!logits || !bitmap || !actions || !logp || !entropy || !saved4 || n <= 0 || ld < KZ_NUM_ACTIONS ||
      ldb_words < KZ_BITMAP_WORDS_MIN || ((uintptr_t)bitmap & 3))
    return KZ_E_ARG;
  return eval_fwd_impl(logits, logits_bf16, ld, bitmap, ldb_words * 4, 1, bitmap_rows, actions, n, logp, entropy, saved4,
                       stream);
}

int kz_eval_masked_bwd(const void* logits, int logits_bf16, int64_t ld, const uint8_t* mask, int64_t ldm,
                       const int64_t* mask_rows, const int64_t* actions, int n, const float* dlogp, const float* dentropy,
                       const float* saved4, void* dlogits, int64_t ldg, void* stream) {
  if (!logits || !mask || !actions || !dlogp || !dentropy || !saved4 || !dlogits || n <= 0 || ld < KZ_NUM_ACTIONS ||
      ldm < KZ_NUM_ACTIONS || ldg < KZ_NUM_ACTIONS)
    return KZ_E_ARG;
  return eval_bwd_impl(logits, logits_bf16, ld, mask, ldm, 0, mask_rows, actions, n, dlogp, dentropy, saved4, dlogits, ldg,
                       nullptr, stream);
}

int kz_eval_masked_bwd_bias(const void* logits, int logits_bf16, int64_t ld, const uint8_t* mask, int64_t ldm,
                            const int64_t* mask_rows, const int64_t* actions, int n, const float* dlogp,
                            const float* dentropy, const float* saved4, void* dlogits, int64_t ldg, int64_t* dbias_q44,
                            void* stream) {
  if (!logits || !mask || !actions || !dlogp || !dentropy || !saved4 || !dlogits || !dbias_q44 || n <= 0 ||
      ld < KZ_NUM_ACTIONS || ldm < KZ_NUM_ACTIONS || ldg < KZ_NUM_ACTIONS || ((uintptr_t)dbias_q44 & 7))
    return KZ_E_ARG;
  return eval_bwd_impl(logits, logits_bf16, ld, mask, ldm, 0, mask_rows, actions, n, dlogp, dentropy, saved4, dlogits, ldg,
                       dbias_q44, stream);
}

int kz_eval_bitmap_bwd(const void* logits, int logits_bf16, int64_t ld, const uint32_t* bitmap, int64_t ldb_words,
                       const int64_t* bitmap_rows, const int64_t* actions, int n, const float* dlogp, const float* dentropy,
                       const float* saved4, void* dlogits, int64_t ldg, int64_t* dbias_q44, void* stream) {
  if (!logits || !bitmap || !actions || !dlogp || !dentropy || !saved4 || !dlogits || n <= 0 || ld < KZ_NUM_ACTIONS ||
      ldb_words < KZ_BITMAP_WORDS_MIN || ldg < KZ_NUM_ACTIONS || ((uintptr_t)bitmap & 3) || ((uintptr_t)dbias_q44 & 7))
    return KZ_E_ARG;
  return eval_bwd_impl(logits, logits_bf16, ld, bitmap, ldb_words * 4, 1, bitmap_rows, actions, n, dlogp, dentropy, saved4,
                       dlogits, ldg, dbias_q44, stream);
}

/* exact column kernel regardless of N (tests / bit-exact comparisons) */
int kz_gae_exact(const float* rewards, const float* values, const uint8_t* dones, const float* last_value, int T, int N,
                 float gamma, float gamma_lambda, float* adv, float* ret, void* stream) {
  if (!rewards || !values || !dones || !last_value || !adv || !ret || T <= 0 || N <= 0) return KZ_E_ARG;
  kz_gae_columns_kernel<<<(N + 127) / 128, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      rewards, values, dones, last_value, T, N, gamma, gamma_lambda, adv, ret);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? KZ_OK : fail(e);
}

int kz_ppo_loss(const float* new_logp, const float* entropy, const float* new_value, const float* old_logp,
                const float* advantages, const float* returns, int n, float clip_epsilon, float value_coef,
                float entropy_coef, float grad_scale, float* out6, float* d_logp, float* d_entropy, float* d_value,
                void* stream) {
  if (!new_logp || !entropy || !new_value || !old_logp || !advantages || !returns || !out6 || !d_logp || !d_entropy ||
      !d_value || n <= 0)
    return KZ_E_ARG;
  kz_ppo_loss_kernel<<<1, 1024, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      new_logp, entropy, new_value, old_logp, advantages, returns, n, clip_epsilon, value_coef, entropy_coef, grad_scale, out6,
      d_logp, d_entropy, d_value);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? KZ_OK : fail(e);
}

}  // extern "C"
