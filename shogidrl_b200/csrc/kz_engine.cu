// kz_engine.cu -- sm_100a kernels for the Keisei self-play rollout hot path (engine part):
// make_move + legal-move generation + termination + 13,527-byte legal mask + 46x9x9 observation,
// one warp per game.
//
// Reference semantics implemented (paths relative to the reference checkout):
//   keisei/shogi/shogi_rules_logic.py:82-208   pseudo-legal targets (steps, slides)
//   keisei/shogi/shogi_rules_logic.py:486-635  legal moves = candidates whose mover's king is safe afterwards
//   keisei/shogi/shogi_rules_logic.py:275-359  uchifuzume, :211-231 nifu, :382-483 promotion / drop rules
//   keisei/shogi/shogi_game.py:408-450, 574-660 make_move, termination order, rewards
//   keisei/shogi/shogi_game_io.py:434-539      observation planes
//   keisei/utils/utils.py:208-266, 310-336     action enumeration and legal mask
// The reference filters candidates by simulate-and-test; here the same set is computed from
// checker / pin / king-danger bitboards built with warp ballots (lane l owns squares l, l+32, l+64, so
// a ballot over slot j IS word j of an 81-bit bitboard).  tests/ check the two against each other.
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>
#include "../../include/keisei_b200.h"
#include "kz_common.cuh"

namespace {

// ------------------------------------------------------------------------------------------------
// tables (filled by kz_init_tables): RAY[sq][dir] and STEP[class][sq] as 3-word bitboards
__device__ uint32_t g_ray[81 * 8 * 3];
__device__ uint32_t g_step[NCLS * 81 * 3];
__device__ uint32_t g_init_bitmap[BITMAP_WORDS];  // legal bitmap of the start position (30 moves)

__constant__ uint8_t c_init_board[96];  // start position; bytes 84..95 = words x, y, z of its position key
__constant__ uint32_t c_init_key_w;     // word w of that key

struct __align__(16) WarpScratch {
  uint32_t bitmap[BITMAP_WORDS];  // 13,527 legal bits in action-index order (+pad)
  uint8_t board[96];
  uint8_t meta[32];
  uint8_t pind[2][96];    // [main/sub] pin direction per square, 0xFF = not pinned
  uint32_t pinl[2][8 * 3];  // pin line per direction
  uint8_t plist[2][40];   // squares of the mover's pieces
  uint8_t dropv[96];      // 7 drop bits per square
  uint32_t oimg[72];      // compose-once observation writer: bit plane * 81 + square of planes 0..27 (+ one pad word)
  float opv[20];          // ... and the values of the constant planes 28..45
  uint32_t onz;           // ... bit i: constant plane 28 + i is non-zero
  uint32_t pad_[3];
};

// Shared memory of the step kernel, declared at file scope so that every device function addresses it
// with shared-space loads/stores (LDS/STS) instead of generic ones.
__shared__ uint32_t s_ray[81 * 8 * 3];
__shared__ uint32_t s_step[NCLS * 81 * 3];
extern __shared__ __align__(16) unsigned char s_dyn[];  // per-warp scratch: WARPS_PER_CTA x WarpScratch (dynamic)
#define s_ws (reinterpret_cast<WarpScratch*>(s_dyn))

struct Tables {};  // the tables live in s_ray / s_step

// Tuning knobs of the output writers; the defaults are the fastest combination measured on B200
// (profiles/run_variants.sh builds and times alternatives, profiles/README.md has the table).
#ifndef KZ_FILL_UNROLL
#define KZ_FILL_UNROLL 1  // unroll factor of the zero-fill loops
#endif
#ifndef KZ_FILL_AFTER_COMPACT
#define KZ_FILL_AFTER_COMPACT 1  // issue the mask row's zero fill after the from-square compaction (shared-memory reads first)
#endif
#ifndef KZ_ST256
#define KZ_ST256 3  // 256-bit zero-fill stores: bit 0 mask row, bit 1 observation row
#endif
#ifndef KZ_ROWS_ONCE
#define KZ_ROWS_ONCE 1  // per-warp writers compose every 32-byte piece once (bit 0 mask row, bit 1 observation row) instead of zero fill + patch
#endif
#ifndef KZ_BULK_ZERO
#define KZ_BULK_ZERO 0  // 1: the mask row's zero runs are written by the bulk-copy engine from a shared page of zeros
#endif
constexpr int kFillUnroll = KZ_FILL_UNROLL;

#if KZ_BULK_ZERO
// Asynchronous zero writes (experiment, off by default): the all-zero stretches of the mask row (runs of from-squares
// without a legal move) are handed to the bulk-copy engine (cp.async.bulk shared -> global from a page of zeros that
// never changes), everything else is stored directly.  The two kinds of stores never touch the same bytes, so nothing
// waits for a copy before the kernel ends.  Parity-green; measured 0.3489 vs 0.3499 ms per 65,536-game launch: the LSU
// store burst it removes (13 KB per game) is not what bounds the kernel.  The same idea on the observation row (zero
// planes in bulk, planes with pieces stored directly, 3 x STG.32 per plane) was 10 % slower and is not kept.
constexpr int kZeroPage = 16384;  // >= the longest run: 81 squares x 160 bytes
__shared__ __align__(128) unsigned char s_zero[kZeroPage];
__device__ __forceinline__ void bulk_zero(void* dst, uint32_t bytes) {  // dst 16-byte aligned, bytes a multiple of 16
  const uint32_t src = (uint32_t)__cvta_generic_to_shared(s_zero);
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(bytes) : "memory");
}
#endif

// 32 bytes of zeros with one 256-bit store (STG.E.ENL2.256, sm_100+): half the store instructions of a 128-bit fill
__device__ __forceinline__ void st_zero256(void* p) {
  const uint32_t z = 0;
  asm volatile("st.global.v8.b32 [%0], {%1,%1,%1,%1,%1,%1,%1,%1};" ::"l"(p), "r"(z) : "memory");
}

__device__ __forceinline__ void st256(void* p, const uint32_t (&v)[8]) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]),
               "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}

__device__ __forceinline__ BB ld_ray(const Tables&, int sq, int d) {
  const uint32_t* p = s_ray + (sq * 8 + d) * 3;
  return BB{p[0], p[1], p[2]};
}
__device__ __forceinline__ BB ld_step(const Tables&, int cls, int sq) {
  const uint32_t* p = s_step + (cls * 81 + sq) * 3;
  return BB{p[0], p[1], p[2]};
}

// Targets of a slide from sq in direction d: up to and including the first occupied square
// (shogi_rules_logic.py:194-206; own-colour blockers are removed by the caller).
__device__ __forceinline__ BB slide_ray(const Tables& T, int sq, int d, BB occ) {
  BB ray = ld_ray(T, sq, d);
  BB bl = ray & occ;
  if (bb_any(bl)) {
    if (dir_positive(d)) ray = ray & bb_upto(bb_lsb(bl));
    else ray = bb_andn(ray, bb_below(bb_msb(bl)));
  }
  return ray;
}

// Squares next to the king of `me` (on K) that an enemy piece attacks, computed on occupancy `occk`
// (the caller removes the king itself so that sliders x-ray through its square).  64 (neighbour, direction)
// ray probes in two warp rounds + 16 knight probes.
#ifndef KD_ATTR
#define KD_ATTR __forceinline__  // inlined into the generator and into ufz_fast: 0.4025 -> 0.3979 ms
#endif
__device__ KD_ATTR BB king_danger(const uint32_t tab, const int K, const int me, const BB occk) {
  const int lane = threadIdx.x & 31;
  const WarpScratch& ws = s_ws[threadIdx.x >> 5];
  const Tables T{};
  const int fwd = me == 0 ? -1 : 1;
  const BB kingsteps = ld_step(T, CLS_KING, K);
  uint32_t attacked8 = 0;
#pragma unroll
  for (int round = 0; round < 2; round++) {
    const int item = lane + 32 * round;
    const int n = item >> 3, d = item & 7, od = (d + 4) & 7;
    const int Tq = K + dir_delta(n);
    const bool valid = Tq >= 0 && Tq < 81 && bb_test(kingsteps, Tq);
    int code = 0, b = -1;
    if (valid) {
      BB bl = ld_ray(T, Tq, d) & occk;
      if (bb_any(bl)) {
        b = dir_positive(d) ? bb_lsb(bl) : bb_msb(bl);
        code = ws.board[b];
      }
    }
    const uint32_t inf = __shfl_sync(FULL, tab, code);
    const bool att = code && code_color(code) != me &&
                     (((inf >> (8 + od)) & 1) || (b == Tq + dir_delta(d) && ((inf >> od) & 1)));
    const uint32_t bal = __ballot_sync(FULL, att);
#pragma unroll
    for (int q = 0; q < 4; q++)
      if ((bal >> (8 * q)) & 0xFF) attacked8 |= 1u << (round * 4 + q);
  }
  {
    const int n = (lane >> 1) & 7;
    const int Tq = K + dir_delta(n);
    bool att = false;
    if (lane < 16 && Tq >= 0 && Tq < 81 && bb_test(kingsteps, Tq)) {
      const int tr = sq_row(Tq), tc = Tq - 9 * tr;
      const int r = tr + 2 * fwd, cc = tc + ((lane & 1) ? 1 : -1);
      if (r >= 0 && r < 9 && cc >= 0 && cc < 9) att = ws.board[r * 9 + cc] == 3 + 14 * (1 - me);
    }
    const uint32_t bal = __ballot_sync(FULL, att);
#pragma unroll
    for (int q = 0; q < 8; q++)
      if ((bal >> (2 * q)) & 3) attacked8 |= 1u << q;
  }
  BB dg = BB{0, 0, 0};
  if (lane < 8 && ((attacked8 >> lane) & 1)) dg = bb_bit(K + dir_delta(lane));
  return BB{__reduce_or_sync(FULL, dg.w0), __reduce_or_sync(FULL, dg.w1), __reduce_or_sync(FULL, dg.w2)};
}

// Uchifuzume test for the one square a dropped pawn can give check from (D, directly in front of the enemy
// king on KE), valid when that king is not attacked before the drop (always true after a legal move).  The
// caller has already placed the pawn on ws.board[D].  With a single adjacent, non-sliding checker the enemy's
// only replies are (a) a king move to a square the dropper does not attack -- taking the pawn included -- and
// (b) taking the pawn with a piece that is not pinned; blocks and drops cannot answer an adjacent check, and a
// pinned piece can never reach D because D lies on a king ray whose first piece is the pawn itself.
// Equivalent to "generate_all_legal_moves(enemy) is empty" (shogi_rules_logic.py:343-357).
#ifndef UFZ_ATTR
#define UFZ_ATTR __forceinline__  // 0.3978 -> 0.3934 ms
#endif
__device__ UFZ_ATTR bool ufz_fast(const uint32_t tab, const int me, const int KE, const int D, const BB occ,
                                      const BB own) {
  const int lane = threadIdx.x & 31;
  const WarpScratch& ws = s_ws[threadIdx.x >> 5];
  const Tables T{};
  const int en = 1 - me;
  const BB occp = occ | bb_bit(D);
  // (a) king moves
  const BB danger = king_danger(tab, KE, en, bb_andn(occp, bb_bit(KE)));
  const BB enemy_pieces = bb_andn(occ, own);
  const BB kmoves = bb_andn(bb_andn(ld_step(T, CLS_KING, KE), enemy_pieces), danger);
  if (bb_any(kmoves)) return false;
  // (b) captures of the pawn by a non-king enemy piece
  const int kr = sq_row(KE), kc = KE - 9 * kr;
  int b = -1;
  {
    const int d = lane & 7, od = (d + 4) & 7;
    int code = 0, bb = -1;
    if (lane < 8) {
      BB bl = ld_ray(T, D, d) & occp;
      if (bb_any(bl)) {
        bb = dir_positive(d) ? bb_lsb(bl) : bb_msb(bl);
        code = ws.board[bb];
      }
    } else if (lane < 10) {  // enemy knights jumping onto D
      const int dr = sq_row(D), dc = D - 9 * dr;
      const int r = dr - 2 * (en == 0 ? -1 : 1), cc = dc + (lane == 8 ? -1 : 1);
      if (r >= 0 && r < 9 && cc >= 0 && cc < 9 && ws.board[r * 9 + cc] == 3 + 14 * en) { bb = r * 9 + cc; code = 3 + 14 * en; }
    }
    const uint32_t inf = __shfl_sync(FULL, tab, code);
    if (code && code_color(code) == en && !((inf >> 23) & 1)) {
      if (lane >= 8) b = bb;
      else if (((inf >> (8 + od)) & 1) || (bb == D + dir_delta(d) && ((inf >> od) & 1))) b = bb;
    }
  }
  // pinned?  b must be the first piece on a king ray with a dropper's slider right behind it
  bool pinned = false;
  int code3 = 0, d2 = -1;
  if (b >= 0) {
    const int br = sq_row(b), bc = b - 9 * br;
    const int dr = br - kr, dc = bc - kc;
    if (dr == 0) d2 = dc > 0 ? 2 : 6;
    else if (dc == 0) d2 = dr > 0 ? 4 : 0;
    else if (dr == dc) d2 = dr > 0 ? 3 : 7;
    else if (dr == -dc) d2 = dr > 0 ? 5 : 1;
    if (d2 >= 0) {
      const BB ray = ld_ray(T, KE, d2);
      const BB between = dir_positive(d2) ? (ray & bb_below(b)) : bb_andn(ray, bb_upto(b));
      if (!bb_any(between & occp)) {
        const BB beyond = ld_ray(T, b, d2) & occp;
        if (bb_any(beyond)) code3 = ws.board[dir_positive(d2) ? bb_lsb(beyond) : bb_msb(beyond)];
      }
    }
  }
  const uint32_t inf3 = __shfl_sync(FULL, tab, code3);
  if (code3 && code_color(code3) == me && ((inf3 >> (8 + ((d2 + 4) & 7))) & 1)) pinned = true;
  return !__any_sync(FULL, b >= 0 && !pinned);
}

struct GenResult {
  int count;
  bool in_check;
};

// ------------------------------------------------------------------------------------------------
// Legal-move generation for side `me` on ws.board / hands.  EMIT: write the 13,527-bit legal bitmap;
// otherwise count only (early exit as soon as one move is known).  skip_ufz: the is_escape_check mode
// of can_drop_specific_piece (shogi_rules_logic.py:461-467).  ufz_all: test every pawn-drop square
// for uchifuzume instead of only the square in front of the enemy king (needed only for loaded
// positions in which the side NOT to move is already in check).
#define UFZ_SKIP 0     // is_escape_check mode
#define UFZ_FAST 1     // specialised evasion test on the square in front of the enemy king (step mode)
#define UFZ_GENERIC 2  // nested move generation on that square (loaded positions)
#define UFZ_ALL 3      // nested move generation on every pawn-drop square (enemy king already attacked)
template <bool EMIT>
__device__ __noinline__ GenResult gen_moves(const uint32_t tab, const int me, const int ufz_mode);

template <bool EMIT, int UFZ_STATIC = -1>  // UFZ_STATIC >= 0: the uchifuzume mode is known at compile time
__device__ __forceinline__ GenResult gen_moves_impl(const uint32_t tab, const int me, const int ufz_mode_rt) {
  const int ufz_mode = UFZ_STATIC >= 0 ? UFZ_STATIC : ufz_mode_rt;
  constexpr int SCR = EMIT ? 0 : 1;  // scratch set: the count-only instance runs inside the emitting one
  const int lane = threadIdx.x & 31;
  WarpScratch& ws = s_ws[threadIdx.x >> 5];
  const uint8_t* hands = ws.meta;
  const Tables T{};
  GenResult res;
  res.count = 0;
  res.in_check = false;

  // ---- phase A: per-square view -> occupancy bitboards (ballots)
  int c[3];
  c[0] = ws.board[lane];
  c[1] = ws.board[lane + 32];
  c[2] = (lane < 17) ? ws.board[lane + 64] : 0;
  BB occ, own;
  int kcode = 8 + 14 * me, ekcode = 8 + 14 * (1 - me), pcode = 1 + 14 * me;
  uint32_t kb[3], ekb[3];
  uint32_t colbits = 0;
  {
    uint32_t o[3], w[3];
#pragma unroll
    for (int j = 0; j < 3; j++) {
      o[j] = __ballot_sync(FULL, c[j] != 0);
      w[j] = __ballot_sync(FULL, c[j] != 0 && code_color(c[j]) == me);
      kb[j] = __ballot_sync(FULL, c[j] == kcode);
      ekb[j] = __ballot_sync(FULL, c[j] == ekcode);
      if (c[j] == pcode) colbits |= 1u << sq_col(lane + 32 * j);
    }
    occ = BB{o[0], o[1], o[2]};
    own = BB{w[0], w[1], w[2]};
  }
  const uint32_t pawn_cols = __reduce_or_sync(FULL, colbits);  // nifu files (shogi_rules_logic.py:211-231)
  const int K = (kb[0] | kb[1] | kb[2]) ? bb_lsb(BB{kb[0], kb[1], kb[2]}) : -1;   // find_king: first in row-major order
  const int KE = (ekb[0] | ekb[1] | ekb[2]) ? bb_lsb(BB{ekb[0], ekb[1], ekb[2]}) : -1;

  if (EMIT) {
    uint4* bm = reinterpret_cast<uint4*>(ws.bitmap);
    for (int i = lane; i < BITMAP_WORDS / 4; i += 32) bm[i] = make_uint4(0, 0, 0, 0);
  }
  ws.pind[SCR][lane] = 0xFF;
  ws.pind[SCR][lane + 32] = 0xFF;
  ws.pind[SCR][lane + 64] = 0xFF;
  __syncwarp();

  if (K < 0) {  // a missing king counts as "in check" and every candidate fails (shogi_rules_logic.py:370-373)
    res.in_check = true;
    return res;
  }

  // ---- phase B: checkers, pins (8 rays + 2 knight squares from the king), king-danger squares
  const int fwd = me == 0 ? -1 : 1;
  const int kr = sq_row(K), kc = K - 9 * kr;
  int nchk;
  BB CM;  // squares where a non-king move resolves a single check (checker square + squares between)
  {
    const int d = lane & 7;
    const int od = (d + 4) & 7;
    BB ray = ld_ray(T, K, d);
    BB bl = ray & occ;
    int b1 = -1, b2 = -1;
    const bool pos = dir_positive(d);
    if (bb_any(bl)) {
      b1 = pos ? bb_lsb(bl) : bb_msb(bl);
      BB bl2 = bb_andn(bl, bb_bit(b1));
      if (bb_any(bl2)) b2 = pos ? bb_lsb(bl2) : bb_msb(bl2);
    }
    const int code1 = b1 >= 0 ? ws.board[b1] : 0;
    const int code2 = b2 >= 0 ? ws.board[b2] : 0;
    const uint32_t inf1 = __shfl_sync(FULL, tab, code1);
    const uint32_t inf2 = __shfl_sync(FULL, tab, code2);
    const bool adj = (b1 == K + dir_delta(d));
    bool chk = false;
    BB cm = BB{0, 0, 0};
    if (lane < 8 && code1) {
      if (code_color(code1) != me) {
        if (((inf1 >> (8 + od)) & 1) || (adj && ((inf1 >> od) & 1))) {
          chk = true;
          BB between = pos ? (ray & bb_below(b1)) : bb_andn(ray, bb_upto(b1));
          cm = between | bb_bit(b1);
        }
      } else if (code2 && code_color(code2) != me && ((inf2 >> (8 + od)) & 1)) {
        // own piece b1 is pinned against the king by the slider on b2: it may only move along the ray up to b2
        ws.pind[SCR][b1] = (uint8_t)d;
        BB line = pos ? (ray & bb_upto(b2)) : bb_andn(ray, bb_below(b2));
        ws.pinl[SCR][d * 3 + 0] = line.w0;
        ws.pinl[SCR][d * 3 + 1] = line.w1;
        ws.pinl[SCR][d * 3 + 2] = line.w2;
      }
    }
    if (lane == 8 || lane == 9) {  // enemy knights: a knight on (r + 2*fwd, c +- 1) jumps onto the king
      const int r = kr + 2 * fwd, cc = kc + (lane == 8 ? -1 : 1);
      if (r >= 0 && r < 9 && cc >= 0 && cc < 9) {
        const int s = r * 9 + cc;
        if (ws.board[s] == 3 + 14 * (1 - me)) {
          chk = true;
          cm = bb_bit(s);
        }
      }
    }
    nchk = __popc(__ballot_sync(FULL, chk));
    CM = BB{__reduce_or_sync(FULL, cm.w0), __reduce_or_sync(FULL, cm.w1), __reduce_or_sync(FULL, cm.w2)};
  }
  res.in_check = nchk > 0;

  // king targets attacked by the enemy once the king has left its square
  const BB DANGER = king_danger(tab, K, me, bb_andn(occ, bb_bit(K)));
  __syncwarp();

  // ---- uchifuzume squares (shogi_rules_logic.py:275-359).  A dropped pawn gives check only from the
  // square in front of the enemy king, unless that king is already attacked (loaded positions only).
  BB UFZ = BB{0, 0, 0};
  if constexpr (EMIT) {
  if (ufz_mode != UFZ_SKIP && hands[me * 7 + 0] > 0 && KE >= 0 && nchk < 2) {
    const int last = me == 0 ? 0 : 8;
    const bool all = ufz_mode == UFZ_ALL;
    const int lo = all ? 0 : KE - 9 * fwd;
    const int hi = all ? 80 : KE - 9 * fwd;
    for (int D = lo; D <= hi; D++) {  // warp-uniform loop
      if (D < 0 || D > 80) continue;
      const int dr = sq_row(D), dc = D - 9 * dr;
      if (ws.board[D] != 0 || dr == last || ((pawn_cols >> dc) & 1)) continue;
      if (nchk == 1 && !bb_test(CM, D)) continue;  // the drop is illegal anyway: it does not answer the check
      __syncwarp();
      if (lane == 0) ws.board[D] = (uint8_t)pcode;
      __syncwarp();
      bool mate;
      if (UFZ_STATIC == UFZ_FAST || ufz_mode == UFZ_FAST) {
        mate = ufz_fast(tab, me, KE, D, occ, own);
      } else if constexpr (UFZ_STATIC != UFZ_FAST) {
        GenResult sub = gen_moves<false>(tab, 1 - me, UFZ_SKIP);
        mate = sub.in_check && sub.count == 0;
      } else {
        mate = false;
      }
      __syncwarp();
      if (lane == 0) ws.board[D] = 0;
      __syncwarp();
      if (mate) UFZ = UFZ | bb_bit(D);
    }
  }
  }

  // ---- phase C: board moves, one lane per own piece
  int cnt = 0;
  {
    int nown = 0;
#pragma unroll
    for (int j = 0; j < 3; j++) {
      const uint32_t w = j == 0 ? own.w0 : (j == 1 ? own.w1 : own.w2);
      if ((w >> lane) & 1) ws.plist[SCR][nown + __popc(w & ((1u << lane) - 1))] = (uint8_t)(lane + 32 * j);
      nown += __popc(w);
    }
    __syncwarp();
    const BB zone = me == 0 ? BB{0x07FFFFFFu, 0, 0} : BB{0, 0xFFC00000u, 0x0001FFFFu};       // rows 0-2 / rows 6-8
    const BB last1 = me == 0 ? BB{0x000001FFu, 0, 0} : BB{0, 0, 0x0001FF00u};                 // row 0 / row 8
    const BB last2 = me == 0 ? BB{0x0003FFFFu, 0, 0} : BB{0, 0x80000000u, 0x0001FFFFu};       // rows 0-1 / rows 7-8
    for (int base = 0; base < nown; base += 32) {
      const int i = base + lane;
      const bool act = i < nown;
      const int sq = act ? ws.plist[SCR][i] : 0;
      const int code = act ? ws.board[sq] : 0;
      const uint32_t inf = __shfl_sync(FULL, tab, code);
      if (act) {
        BB t = ld_step(T, (inf >> 16) & 15, sq);
        uint32_t sl = (inf >> 8) & 0xFF;
        while (sl) {
          const int d = __ffs(sl) - 1;
          sl &= sl - 1;
          t = t | slide_ray(T, sq, d, occ);
        }
        t = bb_andn(t, own);
        if ((inf >> 23) & 1) {
          t = bb_andn(t, DANGER);
        } else {
          if (nchk >= 2) t = BB{0, 0, 0};
          else if (nchk == 1) t = t & CM;
          const int pd = ws.pind[SCR][sq];
          if (pd != 0xFF) t = t & BB{ws.pinl[SCR][pd * 3], ws.pinl[SCR][pd * 3 + 1], ws.pinl[SCR][pd * 3 + 2]};
        }
        // promotion options (shogi_rules_logic.py:382-421, 509-519)
        BB p = BB{0, 0, 0};
        if ((inf >> 20) & 1) p = (me == 0 ? sq < 27 : sq >= 54) ? t : (t & zone);
        const int mk = (inf >> 21) & 3;
        BB np = t;
        if (mk == 1) np = bb_andn(t, last1);
        else if (mk == 2) np = bb_andn(t, last2);
        cnt += bb_popc(np) + bb_popc(p);
        if (EMIT) {
          // drop the (always clear) self bit so that bit k is target k + (k >= from), then interleave
          // no-promotion (even) and promotion (odd) bits: 160 bits = words [5*sq, 5*sq+5) of the bitmap
          const BB lowm = bb_below(sq);
          const BB npc = (np & lowm) | bb_andn(bb_shr1(np), lowm);
          const BB pc = (p & lowm) | bb_andn(bb_shr1(p), lowm);
          uint32_t* o = ws.bitmap + 5 * sq;
          o[0] = spread16(npc.w0 & 0xFFFF) | (spread16(pc.w0 & 0xFFFF) << 1);
          o[1] = spread16(npc.w0 >> 16) | (spread16(pc.w0 >> 16) << 1);
          o[2] = spread16(npc.w1 & 0xFFFF) | (spread16(pc.w1 & 0xFFFF) << 1);
          o[3] = spread16(npc.w1 >> 16) | (spread16(pc.w1 >> 16) << 1);
          o[4] = spread16(npc.w2 & 0xFFFF) | (spread16(pc.w2 & 0xFFFF) << 1);
        }
      }
    }
  }
  if (!EMIT) {  // count-only: a board move already settles "has a legal move"
    if (__any_sync(FULL, cnt > 0)) {
      res.count = 1;
      return res;
    }
  }

  // ---- phase D: drops, one lane per square (shogi_rules_logic.py:424-483, 561-629)
  const uint8_t* h = hands + me * 7;
  const int hP = h[0], hL = h[1], hN = h[2], hS = h[3], hG = h[4], hB = h[5], hR = h[6];
  const bool anyhand = (hP | hL | hN | hS | hG | hB | hR) != 0 && nchk < 2;  // warp-uniform
  if (anyhand) {
    const int last = me == 0 ? 0 : 8, second = me == 0 ? 1 : 7;
#pragma unroll
    for (int j = 0; j < 3; j++) {
      const int sq = lane + 32 * j;
      const uint32_t cmw = j == 0 ? CM.w0 : (j == 1 ? CM.w1 : CM.w2);
      const uint32_t ufw = j == 0 ? UFZ.w0 : (j == 1 ? UFZ.w1 : UFZ.w2);
      uint32_t v = 0;
      if (sq < 81 && c[j] == 0 && (nchk == 0 || ((cmw >> lane) & 1))) {
        const int r = sq_row(sq), col = sq - 9 * r;
        if (hP > 0 && r != last && !((pawn_cols >> col) & 1) && !((ufw >> lane) & 1)) v |= 1;
        if (hL > 0 && r != last) v |= 2;
        if (hN > 0 && r != last && r != second) v |= 4;
        if (hS > 0) v |= 8;
        if (hG > 0) v |= 16;
        if (hB > 0) v |= 32;
        if (hR > 0) v |= 64;
      }
      cnt += __popc(v);
      if (EMIT && sq < 96) ws.dropv[sq] = (uint8_t)v;
    }
  }
  res.count = __reduce_add_sync(FULL, cnt);
  if (EMIT && anyhand) {  // without pieces in hand the drop words keep the zeros written above
    __syncwarp();
    if (lane < 18) {  // bits 12960 + to*7 + type: word 405 + lane holds drop-stream bits [32*lane, 32*lane+32)
      const int to0 = (32 * lane * 293) >> 11;  // floor(32*lane / 7)
      int pos = 7 * to0 - 32 * lane;            // <= 0
      uint32_t w = 0;
#pragma unroll
      for (int i = 0; i < 6; i++) {
        const int to = to0 + i;
        const uint32_t v = to < 81 ? ws.dropv[to] : 0;
        if (pos >= 0) { if (pos < 32) w |= v << pos; }
        else w |= v >> (-pos);
        pos += 7;
      }
      ws.bitmap[405 + lane] = w;
    }
    __syncwarp();
  }
  return res;
}

template <bool EMIT>
__device__ __noinline__ GenResult gen_moves(const uint32_t tab, const int me, const int ufz_mode) {
  return gen_moves_impl<EMIT>(tab, me, ufz_mode);
}

// ------------------------------------------------------------------------------------------------
// 128-bit Zobrist-style key of (board, hands, side to move): four independent 32-bit tables realised as
// hash functions of (square, code) / (hand slot, count).  Replaces the tuple of shogi_game.py:347-372.
__device__ __forceinline__ uint32_t fmix32(uint32_t h) {
  h ^= h >> 16; h *= 0x85ebca6bu; h ^= h >> 13; h *= 0xc2b2ae35u; h ^= h >> 16;
  return h;
}
__device__ __forceinline__ uint4 zkey_item(uint32_t id) {
  uint4 k;
  k.x = fmix32(id * 0x9E3779B1u + 0x7F4A7C15u);
  k.y = fmix32(id * 0x85EBCA77u + 0x165667B1u);
  k.z = fmix32(id * 0xC2B2AE3Du + 0x27D4EB2Fu);
  k.w = fmix32(id * 0x27D4EB2Fu + 0x9E3779B9u);
  return k;
}
__device__ __forceinline__ uint4 position_key(const WarpScratch& ws, int lane, int side) {
  uint4 k = make_uint4(0, 0, 0, 0);
#pragma unroll
  for (int j = 0; j < 3; j++) {
    const int sq = lane + 32 * j;
    const int code = sq < 81 ? ws.board[sq] : 0;
    if (code) { uint4 t = zkey_item(sq * 32 + code); k.x ^= t.x; k.y ^= t.y; k.z ^= t.z; k.w ^= t.w; }
  }
  if (lane < 14) {
    const int cnt = ws.meta[lane];
    if (cnt) { uint4 t = zkey_item(4096 + lane * 256 + cnt); k.x ^= t.x; k.y ^= t.y; k.z ^= t.z; k.w ^= t.w; }
  }
  if (lane == 31 && side) { uint4 t = zkey_item(8191); k.x ^= t.x; k.y ^= t.y; k.z ^= t.z; k.w ^= t.w; }
  k.x = __reduce_xor_sync(FULL, k.x);
  k.y = __reduce_xor_sync(FULL, k.y);
  k.z = __reduce_xor_sync(FULL, k.z);
  k.w = __reduce_xor_sync(FULL, k.w);
  return k;
}

struct StepParams {
  uint8_t* boards;
  uint8_t* meta;
  uint4* hist;    // repetition tables: rep_slots 16-byte slots per game
  int rep_slots;  // power of two >= 2 * hist_cap (>= 64)
  int hist_cap;
  int n;        // games stepped by this launch ...
  int g_first;  // ... starting at this game of the batch (kz_step_range; 0 otherwise)
  const void* actions;
  int actions_i64;
  float* obs;
  long long obs_stride;
  uint8_t* mask;
  long long mask_stride;
  int mask_vec;  // 16-byte aligned rows: vector stores
  float* reward;
  uint8_t* done;
  uint8_t* reason;
  int8_t* winner;
  int32_t* ep_len;
  int32_t* legal_count;
  uint8_t* in_check;  // optional: side to move is in check (ShogiGame.is_in_check)
  void* next_actions;
  unsigned long long seed;
  uint32_t rng_step;
  uint32_t env_offset;
  int auto_reset;
  int mode;  // 0 = refresh, 1 = step
  int eval_term;
  int* tile_counter;  // zeroed per launch: tiles (8 games, one per warp) beyond the first are claimed dynamically
  uint32_t* bitmap_out;  // the legal bitmap [n][bitmap_stride] (modes 0-2; mode 2 writes it instead of the mask row)
  long long bitmap_stride;  // words per bitmap row (>= BITMAP_WORDS, a multiple of 4)
  uint32_t* cobs_out;  // optional compact observation [n][KZ_COBS_WORDS] (kz_step_rollout / kz_legal_bitmap)
  // start-position pool (kz_step_pool; read by the POOL instantiations only)
  const uint32_t* pool;          // [pool_size][KZ_POOL_RECORD_WORDS] records (kz_pool_records)
  int pool_size;
  const int32_t* pool_pick;      // optional: record of each game that restarts in this launch
  unsigned long long pool_seed;  // otherwise drawn from rand32(pool_seed, env_offset + g, finished episodes)
  int32_t* start_ids;            // optional: receives the record index of each game that restarts
  // move expansion (kz_expand; read by the MODE 3 instantiation only): item g applies actions[g] to a copy of source game
  // parent[g]; boards / meta / hist above are the source batch, which is only read
  const int32_t* parent;  // [n] source game of each item
  int src_n;              // games in the source batch
  uint8_t* err_out;       // optional: error bits of each item
  uint8_t* child_boards;  // optional: child batch of n games (kz_state_layout(n, child_hist_cap)) ...
  uint8_t* child_meta;
  uint4* child_hist;      // ... whose repetition tables the kernel empties
  int child_rep_slots;
};

__device__ __forceinline__ uint16_t ld_u16(const uint8_t* p) { return (uint16_t)(p[0] | (p[1] << 8)); }
__device__ __forceinline__ void st_u16(uint8_t* p, int v) { p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); }

// MODE 2 = step in the rollout form (kz_step_rollout): as MODE 1, but the 13,527-bit legal bitmap is written out instead
// of the mask row.
// MODE 1 = step (the hot kernel: only the fast paths are compiled in, the generator is inlined), MODE 0 = refresh
// (loaded positions: nested-generation uchifuzume, full key, optional termination evaluation).
// POOL (modes 1 and 2, kz_step_pool): a finished game restarts from a record of the start-position pool instead of the
// start position; nothing else differs.
// MODE 3 = move expansion (kz_expand): as MODE 2 without auto-reset, for items instead of games -- item g reads the state
// of source game parent[g] (an item whose parent lies outside the batch reads an empty running game and its action is
// rejected), probes that game's repetition table without inserting, writes its rows and scalars at g, and stores the
// successor in the child batch (if any) as a game with no history.  Nothing of the source batch is written.
template <int MODE, bool POOL = false>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, MIN_CTAS_PER_SM) kz_step_kernel(const StepParams P) {
  for (int i = threadIdx.x; i < 81 * 8 * 3; i += blockDim.x) s_ray[i] = g_ray[i];
  for (int i = threadIdx.x; i < NCLS * 81 * 3; i += blockDim.x) s_step[i] = g_step[i];
#if KZ_BULK_ZERO
  for (int i = threadIdx.x; i < kZeroPage / 16; i += blockDim.x) reinterpret_cast<uint4*>(s_zero)[i] = make_uint4(0, 0, 0, 0);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // the page is read by the async proxy from here on
#endif
  __syncthreads();
  const Tables T{};
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  WarpScratch& ws = s_ws[warp];
  const uint32_t tab = code_info(lane);
  const int g_end = P.g_first + P.n;  // this launch steps games [g_first, g_end) of the batch

  // One 32-bit word of game state per lane (lanes 0-23: board, 24-31: meta) and the action are fetched one
  // game ahead, so that their DRAM latency overlaps the previous game's work.
  // (One load with a per-lane address, not one load per branch: the two branches of a divergent `lane < 24 ? board :
  // meta` write the same destination register, and the register scoreboard is per warp -- the second branch's use of the
  // OLD value then waits for the first branch's just-issued load, a full DRAM round trip per game: 5.6 % of all samples in
  // the round-2 line attribution.)
  auto fetch_state = [&](int g) -> uint32_t {
    if (g >= g_end) return 0u;
    int sg = g;  // the game whose state item g starts from
    if constexpr (MODE == 3) {
      sg = P.parent[g];
      if (sg < 0 || sg >= P.src_n) return lane == 28 ? 0xFFu : 0u;  // empty board, status 0, winner none
    }
    const uint8_t* src = lane < 24 ? P.boards + (size_t)sg * 96 + 4 * lane : P.meta + (size_t)sg * 32 + 4 * (lane - 24);
    return *reinterpret_cast<const uint32_t*>(src);
  };
  auto fetch_action = [&](int g) -> long long {
    if (g >= g_end || MODE == 0) return 0;
    if constexpr (MODE == 3) {
      const int sg = P.parent[g];
      if (sg < 0 || sg >= P.src_n) return -1;  // rejected: KZ_ERR_BAD_ACTION
    }
    return P.actions_i64 ? reinterpret_cast<const long long*>(P.actions)[g]
                         : (long long)reinterpret_cast<const int*>(P.actions)[g];
  };
  // When every warp of the CTA runs the same number of games (n a multiple of the CTA's warp count), the CTA works
  // in lockstep on "tiles" of 8 games: (1) the warps are re-aligned once per game -- warps that run the same code
  // at the same time share instruction-cache lines (the kernel is close to the GPC instruction-fetch limit;
  // measured 0.387 -> 0.375 ms; barriers at more points cost more in waiting than they save); (2) tiles after the
  // first are claimed from a global counter instead of a fixed stride, so CTAs that drew cheap positions take more
  // tiles and the grid drains together (a static split leaves 200 of 444 CTAs one game longer than the rest, and
  // the kernel as slow as its unluckiest CTA).  The id for game i + 1 is needed at the top of game i for the prefetch,
  // so claims run ahead of the games (see s_tile below).
  const bool lockstep = (P.n % WARPS_PER_CTA) == 0 && P.tile_counter != nullptr;
  const int ntiles = P.n / WARPS_PER_CTA;
  // Claims are pipelined three tiles deep: the atomic for the tile of iteration it + 3 is issued at the END of iteration
  // it, its result is stored to s_tile at the top of iteration it + 1 (behind the barrier, whose wait hides the round
  // trip) and read by every warp at the top of iteration it + 2.  (Issued at the loop top and kept until the loop end, the
  // result was spilled to local memory under the 80-register cap: the claiming warp stalled on the atomic at the spill and
  // again on the reload behind the row stores -- 10 % of its samples -- and the whole CTA waited for it at the barrier.)
  __shared__ int s_tile[4];
  int tile = blockIdx.x, pending = 0;
  if (lockstep && threadIdx.x == 0) {
    s_tile[1] = gridDim.x + atomicAdd(P.tile_counter, 1);
    pending = gridDim.x + atomicAdd(P.tile_counter, 1);  // the tile of iteration 2
  }
  const int g_stride = gridDim.x * WARPS_PER_CTA;
  int g = P.g_first + blockIdx.x * WARPS_PER_CTA + warp;
  uint32_t next_word = fetch_state(g);
  long long next_action = fetch_action(g);
  __syncthreads();

  for (int it = 0; lockstep ? tile < ntiles : g < g_end; it++) {
    int g_next = g + g_stride;
    if (lockstep) {
      __syncthreads();
      tile = s_tile[(it + 1) & 3];  // the tile after this one
      g_next = P.g_first + tile * WARPS_PER_CTA + warp;
      if (threadIdx.x == 0) s_tile[(it + 2) & 3] = pending;  // claimed at the end of the previous iteration
    }
    // ---- state of this game (prefetched), start fetching the next one
    __syncwarp();
    static_assert(offsetof(WarpScratch, meta) == offsetof(WarpScratch, board) + 96, "meta must follow board: one store for all 32 lanes");
    reinterpret_cast<uint32_t*>(ws.board)[lane] = next_word;  // lanes 0-23: board words, 24-31: the meta row right behind it
    const long long a = next_action;
    next_word = fetch_state(g_next);
    next_action = fetch_action(g_next);
    __syncwarp();
    int side = ws.meta[14];
    int status = ws.meta[15];
    int winner = ws.meta[16] == 0xFF ? -1 : ws.meta[16];
    int err = ws.meta[17];
    int move_count = ld_u16(ws.meta + 18);
    int hist_len = ld_u16(ws.meta + 20);
    const int max_moves = ld_u16(ws.meta + 22);
    uint32_t episodes = ws.meta[24] | (ws.meta[25] << 8) | (ws.meta[26] << 16) | (ws.meta[27] << 24);



    float reward = 0.f;
    int done_out = 0, reason_out = 0, winner_out = -1, ep_len_out = 0;
    bool fresh_senn = false;
    int mover = 1 - side;
    bool moved = false;
    // position key carried in the padding of the state rows (board bytes 84..95, meta bytes 28..31)
    uint4 key = make_uint4(reinterpret_cast<const uint32_t*>(ws.board)[21], reinterpret_cast<const uint32_t*>(ws.board)[22],
                           reinterpret_cast<const uint32_t*>(ws.board)[23], reinterpret_cast<const uint32_t*>(ws.meta)[7]);
    uint32_t kid = 0;  // id of the key item this lane toggles for the move (0 = none)
    bool probe = false;  // a repetition-table probe is in flight (first window of 32 slots in probe_e)
    uint4 probe_e = make_uint4(0, 0, 0, 0);

    if (MODE != 0) {
      if (status != 0) {
        // make_move on a finished game returns the terminal tuple again (shogi_game.py:589-593)
      } else if (a < 0 || a >= KZ_NUM_ACTIONS) {
        err |= KZ_ERR_BAD_ACTION;
      } else {
        mover = side;
        const int ai = (int)a;
        bool ok = true;
        if (ai < 12960) {
          const int promo = ai & 1, pair = ai >> 1;
          const int from = pair / 80, t80 = pair - from * 80, to = t80 + (t80 >= from);
          const int code = ws.board[from], tcode = ws.board[to];
          const uint32_t inf = __shfl_sync(FULL, tab, code);
          if (!code || code_color(code) != side) { err |= KZ_ERR_BAD_ACTION; ok = false; }
          else {
            // movement-pattern validation only, as _validate_and_populate_board_move_details does
            // (shogi_game.py:518-546): `to` must be in the piece's pseudo-legal set.  Decided from the geometry of
            // (from, to): a knight jump, a single step in a step direction, or a slide along a clear ray.
            const int fr = sq_row(from), fc = from - 9 * fr, tr = sq_row(to), tc = to - 9 * tr;
            const int dr = tr - fr, dc = tc - fc;
            bool pat;
            if (code_type(code) == 2) {
              pat = dr == (side == 0 ? -2 : 2) && (dc == 1 || dc == -1);
            } else {
              int d = -1;
              if (dc == 0) d = dr < 0 ? 0 : 4;
              else if (dr == 0) d = dc > 0 ? 2 : 6;
              else if (dr == dc) d = dr > 0 ? 3 : 7;
              else if (dr == -dc) d = dr > 0 ? 5 : 1;
              pat = false;
              if (d >= 0) {
                const int dist = max(abs(dr), abs(dc));
                if (dist == 1 && ((inf >> d) & 1)) pat = true;
                else if ((inf >> (8 + d)) & 1) {
                  const uint32_t o0 = __ballot_sync(FULL, ws.board[lane] != 0), o1 = __ballot_sync(FULL, ws.board[lane + 32] != 0),
                                 o2 = __ballot_sync(FULL, lane < 17 && ws.board[lane + 64] != 0);
                  const BB ray = ld_ray(T, from, d);
                  const BB between = dir_positive(d) ? (ray & bb_below(to)) : bb_andn(ray, bb_upto(to));
                  pat = !bb_any(between & BB{o0, o1, o2});
                }
              }
            }
            if (!pat || (tcode && code_color(tcode) == side) || (promo && !((inf >> 20) & 1))) {
              err |= KZ_ERR_BAD_PATTERN; ok = false;
            }
          }
          if (ok) {  // apply_move_to_board_state (shogi_move_execution.py:90-132)
            const int newcode = promo ? code + promo_delta(code_type(code)) : code;
            int slot = -1, c_old = 0;
            if (tcode) {
              const int tt = code_type(tcode);
              if (tt == 7) err |= KZ_ERR_KING_CAPTURE;
              else { slot = side * 7 + (tt >= 8 ? base_of_promoted(tt) : tt); c_old = ws.meta[slot]; }
            }
            // key items toggled by this move: piece leaves `from`, piece lands on `to`, captured piece, hand count
            if (lane == 0) kid = from * 32 + code;
            else if (lane == 1) kid = to * 32 + newcode;
            else if (lane == 2) kid = tcode ? to * 32 + tcode : 0;
            else if (lane == 3) kid = (slot >= 0 && c_old > 0) ? 4096 + slot * 256 + c_old : 0;
            else if (lane == 4) kid = slot >= 0 ? 4096 + slot * 256 + c_old + 1 : 0;
            __syncwarp();
            if (lane == 0) {
              if (slot >= 0) ws.meta[slot] = (uint8_t)(c_old + 1);
              ws.board[to] = (uint8_t)newcode;
              ws.board[from] = 0;
            }
          }
        } else {
          const int k = ai - 12960;
          const int to = (k * 293) >> 11, pt = k - to * 7;
          if (ws.board[to] != 0 || ws.meta[side * 7 + pt] == 0) { err |= KZ_ERR_BAD_ACTION; ok = false; }
          if (ok) {  // drop (shogi_move_execution.py:55-71)
            const int slot = side * 7 + pt, c_old = ws.meta[slot];
            if (lane == 1) kid = to * 32 + (1 + pt + 14 * side);
            else if (lane == 3) kid = 4096 + slot * 256 + c_old;
            else if (lane == 4) kid = c_old > 1 ? 4096 + slot * 256 + c_old - 1 : 0;
            __syncwarp();
            if (lane == 0) {
              ws.board[to] = (uint8_t)(1 + pt + 14 * side);
              ws.meta[slot] = (uint8_t)(c_old - 1);
            }
          }
        }
        __syncwarp();
        if (ok) {
          moved = true;
          move_count += 1;  // apply_move_to_game (shogi_move_execution.py:141-156)
          side = 1 - side;
          // history append + repetition count (shogi_game.py:651-654, shogi_rules_logic.py:680-695)
          // The reference counts equal (board, hands, side) entries of move_history; here every game owns an
          // open-addressing table keyed by the 124-bit position key whose low 4 bits of w hold the occurrence
          // count.  One cooperative probe reads 32 consecutive slots (512 B) instead of scanning every earlier ply.
          // the key is updated incrementally: XOR of the (at most six) items the move toggles, one per lane
          {
            if (lane == 5) kid = 8191;  // side to move flips on every move
            uint4 dk = make_uint4(0, 0, 0, 0);
            if (kid) dk = zkey_item(kid);
            key.x ^= __reduce_xor_sync(FULL, dk.x);
            key.y ^= __reduce_xor_sync(FULL, dk.y);
            key.z ^= __reduce_xor_sync(FULL, dk.z);
            key.w ^= __reduce_xor_sync(FULL, dk.w);
          }
          if (hist_len < P.hist_cap) {
            // issue the probe's loads now; they are consumed after the move generation, which hides the DRAM trip
            probe = true;
            const int hg = MODE == 3 ? P.parent[g] : g;  // whose repetition table (MODE 3: only a valid parent moves)
            probe_e = (P.hist + (size_t)hg * P.rep_slots)[(key.y + lane) & ((uint32_t)P.rep_slots - 1u)];
            hist_len += 1;
          } else {
            err |= KZ_ERR_HISTORY_FULL;
          }
        }
      }
    }

    // ---- zero fills of this game's output rows (content-independent; the non-zero entries are overwritten later,
    // behind a __syncwarp()).  (Issuing them here, ahead of the move generation, was measured slower: +5 % for the mask
    // row, +15 % for the observation row.)
    auto fill_mask_zero = [&]() {
      if (!P.mask || !P.mask_vec) return;
      uint8_t* mrow = P.mask + (size_t)g * P.mask_stride;
#if (KZ_ST256 & 1)
      if ((((uintptr_t)mrow) & 31) == 0) {
#pragma unroll kFillUnroll
        for (int q = lane; q < 405; q += 32) st_zero256(mrow + 32 * q);
        return;
      }
#endif
      uint4* m4 = reinterpret_cast<uint4*>(mrow);
      const uint4 z4 = make_uint4(0, 0, 0, 0);
#pragma unroll kFillUnroll
      for (int q = lane; q < 810; q += 32) m4[q] = z4;
    };
    auto fill_obs_zero = [&]() {
      if (!P.obs) return;
      float* orow = P.obs + (size_t)g * P.obs_stride;
#if (KZ_ST256 & 2)
      // rows are 8-byte aligned: up to three float2 to reach a 32-byte line, 256-bit stores, up to three float2 of tail
      float2* o2 = reinterpret_cast<float2*>(orow);
      const int head = (int)(((32u - (unsigned)((uintptr_t)orow & 31)) & 31u) >> 3);
      const int nb = (KZ_OBS_FLOATS * 4 - head * 8) >> 5;
      char* body = reinterpret_cast<char*>(orow) + head * 8;
      if (lane < head) o2[lane] = make_float2(0.f, 0.f);
#pragma unroll kFillUnroll
      for (int q = lane; q < nb; q += 32) st_zero256(body + 32 * q);
      const int tail0 = head + 4 * nb;
      if (lane < KZ_OBS_FLOATS / 2 - tail0) o2[tail0 + lane] = make_float2(0.f, 0.f);
#else
      // float4 chunk q covers floats [mis + 4q, mis + 4q + 4); odd rows start 8 bytes past a 16-byte line
      const int mis = ((uintptr_t)orow & 15) ? 2 : 0;
      float4* o4 = reinterpret_cast<float4*>(orow + mis);
      const float4 zf = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll kFillUnroll
      for (int q = lane; q < 931; q += 32) o4[q] = zf;
      if (lane == 0) {  // the 2 floats the float4 grid does not cover: plane 0 head or plane 45 tail, both 0 here
        float2* o2 = reinterpret_cast<float2*>(orow + (mis ? 0 : 3724));
        *o2 = make_float2(0.f, 0.f);
      }
#endif
    };
    // image of this game's observation (generate_neural_network_observation, shogi_game_io.py:434-539): one bit per
    // non-zero float of the 28 piece planes (bit plane * 81 + square, squares rotated 180 degrees for White to move) and
    // the values of the 18 constant planes -- what the compose-once row writers read
    auto build_obs_image = [&]() {
      __syncwarp();
      ws.oimg[lane] = 0; ws.oimg[lane + 32] = 0;
      if (lane < 8) ws.oimg[lane + 64] = 0;
      float pv = 0.f;
      if (lane < 14) {
        const int cnt = ws.meta[lane < 7 ? side * 7 + lane : (1 - side) * 7 + (lane - 7)];
        if (cnt > 0) pv = __fdiv_rn((float)cnt, 18.0f);  // see write_obs for why one fp32 division is exact here
      } else if (lane == 14) pv = side == 0 ? 1.f : 0.f;
      else if (lane == 15) pv = max_moves > 0 ? __fdiv_rn((float)move_count, (float)max_moves) : 0.f;
      if (lane < 20) ws.opv[lane] = pv;
      const uint32_t nz = __ballot_sync(FULL, pv != 0.f);
      if (lane == 0) ws.onz = nz;
      __syncwarp();
#pragma unroll
      for (int j = 0; j < 3; j++) {
        const int sq = lane + 32 * j;
        const int code = sq < 81 ? ws.board[sq] : 0;
        if (code) {
          const int t = code_type(code), mine = code_color(code) == side;
          const int plane = t < 8 ? (mine ? 0 : 14) + t : (mine ? 8 : 22) + (t - 8);
          const int f = plane * 81 + (side == 0 ? sq : 80 - sq);
          atomicOr(&ws.oimg[f >> 5], 1u << (f & 31));
        }
      }
      __syncwarp();
    };
    auto write_obs = [&]() {
      if (!P.obs) return;
      // generate_neural_network_observation (shogi_game_io.py:434-539)
      float* orow = P.obs + (size_t)g * P.obs_stride;
#if (KZ_ROWS_ONCE & 2)
      {
        // compose-once writer: every 32-byte piece of the row gets its final content in one store (no zero fill that is
        // patched afterwards: profiles/row_store_probe.cu -- patching freshly zeroed sectors costs 7 % of the row
        // bandwidth at 24 warps per SM).  Rows are 8-byte aligned: float2 head / tail around the 32-byte body.
        build_obs_image();
        float2* o2 = reinterpret_cast<float2*>(orow);
        const int head = (int)(((32u - (unsigned)((uintptr_t)orow & 31)) & 31u) >> 3);
        const int nb = (KZ_OBS_FLOATS * 4 - head * 8) >> 5;
        char* body = reinterpret_cast<char*>(orow) + head * 8;
        if (lane < head) {  // floats 0..5: plane 0
          const uint32_t b2 = ws.oimg[0] >> (2 * lane);
          o2[lane] = make_float2((b2 & 1) ? 1.0f : 0.f, (b2 & 2) ? 1.0f : 0.f);
        }
#pragma unroll 1
        for (int q = lane; q < nb; q += 32) {
          const int r0 = 2 * head + 8 * q;
          char* dst = body + 32 * q;
          if (r0 + 8 <= 28 * 81) {  // inside the piece planes: 8 bits of the image
            const uint32_t bits = __funnelshift_r(ws.oimg[r0 >> 5], ws.oimg[(r0 >> 5) + 1], r0 & 31) & 0xFFu;
            if (bits == 0) st_zero256(dst);
            else {
              uint32_t v[8];
#pragma unroll
              for (int k = 0; k < 8; k++) v[k] = ((bits >> k) & 1) ? 0x3F800000u : 0u;
              st256(dst, v);
            }
          } else {
            // constant planes: the piece lies in plane 28 + pl0, its floats from index nb0 on in the next plane
            // (pl0 = -1: the seam piece, whose first nb0 floats are still piece-plane bits)
            const int x = r0 - 28 * 81;
            const int pl0 = x >= 0 ? (x * 1619) >> 17 : -1;  // floor(x / 81), x < 1700
            const int nb0 = (pl0 + 1) * 81 - x;
            const uint32_t a = pl0 >= 0 ? __float_as_uint(ws.opv[pl0]) : 0u, b = __float_as_uint(ws.opv[pl0 + 1]);
            uint32_t bits = 0;
            if (pl0 < 0) bits = __funnelshift_r(ws.oimg[r0 >> 5], ws.oimg[(r0 >> 5) + 1], r0 & 31) & ((1u << nb0) - 1u);
            if (a == 0 && bits == 0 && (nb0 >= 8 || b == 0)) st_zero256(dst);
            else {
              uint32_t v[8];
#pragma unroll
              for (int k = 0; k < 8; k++) v[k] = k < nb0 ? (pl0 >= 0 ? a : (((bits >> k) & 1) ? 0x3F800000u : 0u)) : b;
              st256(dst, v);
            }
          }
        }
        // the last floats of the row lie in plane 45, which is always zero (reserved; shogi_game_io.py:434-539)
        const int tail0 = head + 4 * nb;
        if (lane < KZ_OBS_FLOATS / 2 - tail0) o2[tail0 + lane] = make_float2(0.f, 0.f);
        return;
      }
#endif
      // constant planes 28..45: value of plane 28+i lives in lane i
      float pv = 0.f;
      if (lane < 14) {
        const int cnt = ws.meta[lane < 7 ? side * 7 + lane : (1 - side) * 7 + (lane - 7)];
        // The reference divides in Python doubles and stores fp32.  For integer operands below 2^16 the exact
        // quotient is never within 2^-41 (relative) of an fp32 rounding tie, so rounding once (IEEE fp32 division)
        // and rounding twice (double, then fp32) give the same bits.
        if (cnt > 0) pv = __fdiv_rn((float)cnt, 18.0f);
      } else if (lane == 14) pv = side == 0 ? 1.f : 0.f;
      else if (lane == 15) pv = max_moves > 0 ? __fdiv_rn((float)move_count, (float)max_moves) : 0.f;
      // Zero-fill the whole row with wide stores, then overwrite what is not zero: the constant planes with a non-zero
      // value (a few of the 18) and one float per piece.  Both overwrites follow the zero fill in program order behind a
      // __syncwarp().  (Measured alternatives that were NOT faster: handing the fill to the bulk-copy engine, cp.async.bulk
      // from a shared zero page; streaming __stcs stores.)
      fill_obs_zero();
      __syncwarp();
      uint32_t nzp = __ballot_sync(FULL, pv != 0.f);  // constant planes 28 + i with a non-zero value
      while (nzp) {
        const int i = __ffs(nzp) - 1;
        nzp &= nzp - 1;
        const float v = __shfl_sync(FULL, pv, i);
        float* pl = orow + (28 + i) * 81;
        pl[lane] = v;
        pl[lane + 32] = v;
        if (lane < 17) pl[lane + 64] = v;
      }
#pragma unroll
      for (int j = 0; j < 3; j++) {
        const int sq = lane + 32 * j;
        const int code = sq < 81 ? ws.board[sq] : 0;
        if (code) {
          const int t = code_type(code), mine = code_color(code) == side;
          const int plane = t < 8 ? (mine ? 0 : 14) + t : (mine ? 8 : 22) + (t - 8);
          orow[plane * 81 + (side == 0 ? sq : 80 - sq)] = 1.0f;
        }
      }
    };
    // ---- legal moves of the position now on the board
    // After a legal move the side that just moved is never in check, so a dropped pawn can only give check from
    // the square in front of the enemy king and the specialised test applies.  Loaded positions (refresh mode)
    // may have the side NOT to move in check: they take the nested-generation path, on every pawn-drop square
    // when that king is attacked.
    if (MODE == 0) key = position_key(ws, lane, side);  // loaded positions: full key
    GenResult gr;
    if constexpr (MODE != 0) {
      gr = gen_moves_impl<true, UFZ_FAST>(tab, side, UFZ_FAST);  // inlined, fast uchifuzume path only
    } else {
      int mode = UFZ_GENERIC;
      if (ws.meta[side * 7] > 0) {
        GenResult opp = gen_moves<false>(tab, 1 - side, UFZ_SKIP);
        if (opp.in_check) mode = UFZ_ALL;
      }
      gr = gen_moves<true>(tab, side, mode);
    }

    if (probe) {  // repetition count of the new position: match / insert in the first window, further windows if needed
      uint4* tb = P.hist + (size_t)(MODE == 3 ? P.parent[g] : g) * P.rep_slots;  // MODE 3: the parent's, read only
      const uint32_t smask = (uint32_t)P.rep_slots - 1u;
      uint32_t start = key.y & smask;
      int count = 0;
      uint4 e = probe_e;
      for (int round = 0; round * 32 < P.rep_slots; round++) {
        const uint32_t slot = (start + lane) & smask;
        if (round > 0) e = tb[slot];
        const bool occupied = (e.w & 15u) != 0;
        const bool match = occupied && e.x == key.x && e.y == key.y && e.z == key.z && ((e.w ^ key.w) >> 4) == 0;
        const uint32_t stop = __ballot_sync(FULL, match || !occupied);
        if (stop) {
          const int f = __ffs(stop) - 1;
          const uint32_t oldw = __shfl_sync(FULL, e.w, f);
          const bool was_match = (__ballot_sync(FULL, match) >> f) & 1;
          count = was_match ? min(15, (int)(oldw & 15u) + 1) : 1;
          if (MODE != 3 && lane == f) tb[slot] = make_uint4(key.x, key.y, key.z, (key.w & ~15u) | (uint32_t)count);
          break;
        }
        start += 32;
      }
      if (count == 0) err |= KZ_ERR_HISTORY_FULL;
      fresh_senn = count >= 4;
    }
    if ((moved || (MODE == 0 && P.eval_term)) && status == 0) {
      // _check_and_update_termination_status (shogi_game.py:408-450), in the reference's order
      if (gr.count == 0) {
        if (gr.in_check) { status = KZ_TSUMI; winner = mover; }
        else { status = KZ_STALEMATE; winner = -1; }
      } else if (move_count >= max_moves) { status = KZ_MAX_MOVES; winner = -1; }
      else if (fresh_senn) { status = KZ_SENNICHITE; winner = -1; }
    }
    if (MODE != 0 && status != 0) {  // _handle_real_move_return (shogi_game.py:553-572)
      done_out = 1;
      reason_out = status;
      winner_out = winner;
      ep_len_out = move_count;
      if (winner >= 0) reward = winner == mover ? 1.f : -1.f;
    }

    if (MODE != 0 && MODE != 3 && status != 0 && P.auto_reset) {
      // StepManager.handle_episode_end -> game.reset() (step_manager.py:437-440; shogi_game.py:113-130)
      if constexpr (POOL) {
        // the same reset from record k of the start-position pool: state rows, position key, legal bitmap, count and
        // in-check flag as kz_pool_records packed them from kz_refresh / kz_legal_bitmap (DESIGN.md section 4.9)
        episodes += 1;
        uint32_t k = P.pool_pick ? (uint32_t)P.pool_pick[g]
                                 : (uint32_t)(((unsigned long long)rand32(P.pool_seed, (unsigned long long)P.env_offset + g,
                                                                          episodes) * (unsigned long long)P.pool_size) >> 32);
        if (k >= (uint32_t)P.pool_size) k %= (uint32_t)P.pool_size;
        const uint32_t* rec = P.pool + (size_t)k * KZ_POOL_RECORD_WORDS;
        const uint8_t* rmeta = reinterpret_cast<const uint8_t*>(rec + 24);
        __syncwarp();
        if (lane < 24) reinterpret_cast<uint32_t*>(ws.board)[lane] = rec[lane];
        if (lane < 14) ws.meta[lane] = rmeta[lane];
        side = rmeta[14]; status = 0; winner = -1; move_count = ld_u16(rmeta + 18); hist_len = 0;
        key = make_uint4(rec[21], rec[22], rec[23], rec[31]);
        {
          uint4* tb = P.hist + (size_t)g * P.rep_slots;
          for (int i = lane; i < P.rep_slots; i += 32) tb[i] = make_uint4(0, 0, 0, 0);
        }
        for (int i = lane; i < BITMAP_WORDS; i += 32) ws.bitmap[i] = rec[KZ_POOL_BITMAP_OFFSET + i];
        gr.count = (int)rec[32];
        gr.in_check = rec[33] != 0;
        if (lane == 0 && P.start_ids) P.start_ids[g] = (int32_t)k;
        __syncwarp();
      } else {
        __syncwarp();
        if (lane < 24) reinterpret_cast<uint32_t*>(ws.board)[lane] = reinterpret_cast<const uint32_t*>(c_init_board)[lane];
        if (lane < 14) ws.meta[lane] = 0;
        side = 0; status = 0; winner = -1; move_count = 0; hist_len = 0;
        episodes += 1;
        key = make_uint4(reinterpret_cast<const uint32_t*>(c_init_board)[21], reinterpret_cast<const uint32_t*>(c_init_board)[22],
                         reinterpret_cast<const uint32_t*>(c_init_board)[23], c_init_key_w);
        {
          uint4* tb = P.hist + (size_t)g * P.rep_slots;
          for (int i = lane; i < P.rep_slots; i += 32) tb[i] = make_uint4(0, 0, 0, 0);
        }
        for (int i = lane; i < BITMAP_WORDS; i += 32) ws.bitmap[i] = g_init_bitmap[i];
        gr.count = 30;
        gr.in_check = false;
        __syncwarp();
      }
    }

    // ---- outputs
    if (lane == 0) {
      if (P.reward) P.reward[g] = reward;
      if (P.done) P.done[g] = (uint8_t)done_out;
      if (P.reason) P.reason[g] = (uint8_t)reason_out;
      if (P.winner) P.winner[g] = (int8_t)winner_out;
      if (P.ep_len) P.ep_len[g] = ep_len_out;
      if (P.legal_count) P.legal_count[g] = gr.count;
      if (P.in_check) P.in_check[g] = (uint8_t)gr.in_check;
      if constexpr (MODE == 3) {
        if (P.err_out) P.err_out[g] = (uint8_t)err;
      }
    }

    auto write_mask = [&]() {
      if (!P.mask) return;
      uint8_t* mrow = P.mask + (size_t)g * P.mask_stride;
      if (P.mask_vec) {
        // 16-byte chunk q of the row = bits [16q, 16q+16) of the bitmap; a from-square owns chunks 10f..10f+9.
        // Pass 1 zero-fills the 810 board-move chunks (256-bit stores on 32-byte aligned rows); pass 2 expands only the chunks
        // of from-squares that have a legal move (3 squares x 10 chunks per warp round) and the 36 drop chunks.
#if (KZ_ROWS_ONCE & 1)
        if ((((uintptr_t)mrow) & 31) == 0 && P.mask_stride >= 13536) {
          // compose-once writer: 32-byte piece q of the row = the 32 actions of bitmap word q (pad bytes 13527..13535
          // are written as zeros: the bitmap is zero-padded)
          __syncwarp();
          auto piece = [&](int q, uint32_t w) {
            if (w == 0) st_zero256(mrow + 32 * q);
            else {
              uint32_t v[8];
#pragma unroll
              for (int k = 0; k < 8; k++) v[k] = (((w >> (4 * k)) & 0xF) * 0x00204081u) & 0x01010101u;
              st256(mrow + 32 * q, v);
            }
          };
          // (two pieces per round, both bitmap words loaded before either is tested: measured 0.3494 vs 0.3473 ms, not kept)
#pragma unroll 1
          for (int q = lane; q < 423; q += 32) piece(q, ws.bitmap[q]);
          return;
        }
#endif
        uint4* m4 = reinterpret_cast<uint4*>(mrow);
        if (!KZ_FILL_AFTER_COMPACT && !(KZ_BULK_ZERO & 1)) fill_mask_zero();
        uint32_t act[3];
#pragma unroll
        for (int j = 0; j < 3; j++) {
          const int f = lane + 32 * j;
          bool nz = false;
          if (f < 81) {
            const uint32_t* w = ws.bitmap + 5 * f;
            nz = (w[0] | w[1] | w[2] | w[3] | w[4]) != 0;
          }
          act[j] = __ballot_sync(FULL, nz);
        }
        int nact = 0;
#pragma unroll
        for (int j = 0; j < 3; j++) {
          if ((act[j] >> lane) & 1) ws.plist[0][nact + __popc(act[j] & ((1u << lane) - 1))] = (uint8_t)(lane + 32 * j);
          nact += __popc(act[j]);
        }
#if (KZ_BULK_ZERO & 1)
        {
          // every maximal run of from-squares without a legal move is one bulk copy of 160 zero bytes per square; the
          // squares with moves are written in full (all 10 chunks) by pass 2 below
          const unsigned long long lo = (unsigned long long)act[0] | ((unsigned long long)act[1] << 32);
          const uint32_t hi = act[2];  // squares 64..80
#pragma unroll
          for (int j = 0; j < 3; j++) {
            const int f = lane + 32 * j;
            if (f < 81 && !((act[j] >> lane) & 1)) {
              bool prev_zero = false;
              if (lane > 0) prev_zero = !((act[j] >> (lane - 1)) & 1);
              else if (j > 0) prev_zero = !((act[j > 0 ? j - 1 : 0] >> 31) & 1);
              if (!prev_zero) {
                int end;
                if (f < 64) {
                  const unsigned long long t = lo >> f;
                  end = t ? f + __ffsll((long long)t) - 1 : (hi ? 64 + __ffs(hi) - 1 : 81);
                } else {
                  const uint32_t t = hi >> (f - 64);
                  end = t ? f + __ffs(t) - 1 : 81;
                }
                bulk_zero(mrow + 160 * f, (uint32_t)(160 * (end - f)));
              }
            }
          }
        }
#else
        if (KZ_FILL_AFTER_COMPACT) fill_mask_zero();  // after the shared-memory reads above
#endif
        __syncwarp();  // orders the zero fill before the overwrites below and publishes plist
        auto expand = [](uint32_t b16) {
          uint4 v;
          v.x = ((b16 & 0xF) * 0x00204081u) & 0x01010101u;
          v.y = (((b16 >> 4) & 0xF) * 0x00204081u) & 0x01010101u;
          v.z = (((b16 >> 8) & 0xF) * 0x00204081u) & 0x01010101u;
          v.w = (((b16 >> 12) & 0xF) * 0x00204081u) & 0x01010101u;
          return v;
        };
        const int sub = lane / 10, jj = lane - 10 * sub;  // lanes 30, 31 idle in pass 2
        // (software-pipelining the plist load one round ahead, unrolled by two: measured 0.8 % slower)
#pragma unroll 1
        for (int base = 0; base < nact; base += 3) {
          const int i = base + sub;
          if (sub < 3 && i < nact) {
            const int f = ws.plist[0][i];
            const uint32_t w = ws.bitmap[5 * f + (jj >> 1)];
            m4[10 * f + jj] = expand((jj & 1) ? (w >> 16) : (w & 0xFFFF));
          }
        }
        for (int q = 810 + lane; q < 846; q += 32) {
          const uint32_t w = ws.bitmap[q >> 1];
          const uint4 v = expand((q & 1) ? (w >> 16) : (w & 0xFFFF));
          if (q < 845 || P.mask_stride >= 13536) m4[q] = v;
          else {  // last 7 bytes of an exactly-13,527-byte aligned row
            const uint32_t parts[2] = {v.x, v.y};
            for (int b = 0; b < 7; b++) mrow[13520 + b] = (uint8_t)(parts[b >> 2] >> (8 * (b & 3)));
          }
        }
      } else {
        for (int i = lane; i < KZ_NUM_ACTIONS; i += 32) mrow[i] = (uint8_t)((ws.bitmap[i >> 5] >> (i & 31)) & 1);
      }
    };
    auto pick_next = [&]() {
      if (!P.next_actions) return;
      long long pick = -1;
      if (gr.count > 0) {
        const uint32_t r = rand32(P.seed, (unsigned long long)P.env_offset + (unsigned long long)g, P.rng_step);
        const int k = (int)(((unsigned long long)r * (unsigned long long)gr.count) >> 32);
        // k-th set bit of the bitmap: lane owns words [14*lane, 14*lane+14) (the bitmap is zero-padded to 448 words).
        // All 14 loads are issued together and their popcounts kept in registers, so locating the word is a
        // branch-free walk without further shared-memory round trips.
        const int w0 = lane * 14;
        int pcs[14];
        int mycnt = 0;
#pragma unroll
        for (int i = 0; i < 14; i++) { pcs[i] = __popc(ws.bitmap[w0 + i]); mycnt += pcs[i]; }
        int incl = mycnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += t; }
        const int excl = incl - mycnt;
        int found = -1;
        if (k >= excl && k < incl) {
          int rem = k - excl, widx = 0;
          bool open_ = true;
#pragma unroll
          for (int i = 0; i < 14; i++) {
            if (open_) {
              if (rem < pcs[i]) { widx = i; open_ = false; }
              else rem -= pcs[i];
            }
          }
          // rem < popc(wv) and words hold few bits: clear the rem lowest set bits, the next one is the pick (__fns is a
          // ~50-instruction software routine)
          uint32_t wv = ws.bitmap[w0 + widx];
          for (int r = rem; r > 0; r--) wv &= wv - 1;
          found = (w0 + widx) * 32 + __ffs(wv) - 1;
        }
        const uint32_t who = __ballot_sync(FULL, found >= 0);
        pick = __shfl_sync(FULL, found, __ffs(who) - 1);
      }
      if (lane == 0) {
        if (P.actions_i64) reinterpret_cast<long long*>(P.next_actions)[g] = pick;
        else reinterpret_cast<int*>(P.next_actions)[g] = (int)pick;
      }
    };
    // (Measured and not faster: choosing the next action before the mask row's store burst; writing the observation row
    // ahead of the move generation, +8 %.)
    if (MODE == 2 || P.bitmap_out) {  // rollout form: the legal set leaves as its 1,792-byte bitmap
      __syncwarp();
      uint4* dst = reinterpret_cast<uint4*>(P.bitmap_out + (size_t)g * P.bitmap_stride);
      for (int i = lane; i < BITMAP_WORDS / 4; i += 32) dst[i] = reinterpret_cast<const uint4*>(ws.bitmap)[i];
    }
    if constexpr (MODE != 2 && MODE != 3) write_mask();
    if constexpr (MODE != 3) pick_next();
    write_obs();
    if (P.cobs_out) {
      // compact observation: what the 46 planes are made of -- per observation square (already rotated for White to move)
      // the index of the one piece plane that holds a 1 there (0xFF: none), and the 18 constant-plane values.  160 bytes
      // instead of 14,904: the input layer of the policy network reads this form (kz_cobs_conv_*, csrc/kz_nn.cu).
      __syncwarp();
      uint8_t* cb = reinterpret_cast<uint8_t*>(ws.oimg);
      if (lane < 21) ws.oimg[lane] = 0xFFFFFFFFu;
      float pv = 0.f;
      if (lane < 14) {
        const int cnt = ws.meta[lane < 7 ? side * 7 + lane : (1 - side) * 7 + (lane - 7)];
        if (cnt > 0) pv = __fdiv_rn((float)cnt, 18.0f);
      } else if (lane == 14) pv = side == 0 ? 1.f : 0.f;
      else if (lane == 15) pv = max_moves > 0 ? __fdiv_rn((float)move_count, (float)max_moves) : 0.f;
      if (lane < 19) ws.oimg[21 + lane] = lane < 18 ? __float_as_uint(pv) : 0u;
      __syncwarp();
#pragma unroll
      for (int j = 0; j < 3; j++) {
        const int sq = lane + 32 * j;
        const int code = sq < 81 ? ws.board[sq] : 0;
        if (code) {
          const int t = code_type(code), mine = code_color(code) == side;
          cb[side == 0 ? sq : 80 - sq] = (uint8_t)(t < 8 ? (mine ? 0 : 14) + t : (mine ? 8 : 22) + (t - 8));
        }
      }
      __syncwarp();
      uint32_t* dst = P.cobs_out + (size_t)g * KZ_COBS_WORDS;
      for (int i = lane; i < KZ_COBS_WORDS; i += 32) dst[i] = ws.oimg[i];
      __syncwarp();
    }

    // ---- store state (MODE 3: the child, if any, with no history -- error bits, plies since reset and episodes 0, an
    // emptied repetition table)
    if constexpr (MODE == 3) { err = 0; hist_len = 0; episodes = 0; }
    __syncwarp();
    if (lane == 0) {
      ws.meta[14] = (uint8_t)side;
      ws.meta[15] = (uint8_t)status;
      ws.meta[16] = (uint8_t)(winner < 0 ? 0xFF : winner);
      ws.meta[17] = (uint8_t)err;
      st_u16(ws.meta + 18, move_count);
      st_u16(ws.meta + 20, hist_len);
      ws.meta[24] = (uint8_t)episodes; ws.meta[25] = (uint8_t)(episodes >> 8);
      ws.meta[26] = (uint8_t)(episodes >> 16); ws.meta[27] = (uint8_t)(episodes >> 24);
      reinterpret_cast<uint32_t*>(ws.board)[21] = key.x;
      reinterpret_cast<uint32_t*>(ws.board)[22] = key.y;
      reinterpret_cast<uint32_t*>(ws.board)[23] = key.z;
      reinterpret_cast<uint32_t*>(ws.meta)[7] = key.w;
    }
    __syncwarp();
    if constexpr (MODE == 3) {
      if (P.child_boards) {
        uint32_t* bdst = reinterpret_cast<uint32_t*>(P.child_boards + (size_t)g * 96);
        uint32_t* mdst = reinterpret_cast<uint32_t*>(P.child_meta + (size_t)g * 32);
        if (lane < 24) bdst[lane] = reinterpret_cast<uint32_t*>(ws.board)[lane];
        else mdst[lane - 24] = reinterpret_cast<uint32_t*>(ws.meta)[lane - 24];
        uint4* tb = P.child_hist + (size_t)g * P.child_rep_slots;
        for (int i = lane; i < P.child_rep_slots; i += 32) tb[i] = make_uint4(0, 0, 0, 0);
      }
    } else {
      uint32_t* bdst = reinterpret_cast<uint32_t*>(P.boards + (size_t)g * 96);
      uint32_t* mdst = reinterpret_cast<uint32_t*>(P.meta + (size_t)g * 32);
      if (lane < 24) bdst[lane] = reinterpret_cast<uint32_t*>(ws.board)[lane];
      else mdst[lane - 24] = reinterpret_cast<uint32_t*>(ws.meta)[lane - 24];
    }
    __syncwarp();
    if (lockstep && threadIdx.x == 0) pending = gridDim.x + atomicAdd(P.tile_counter, 1);  // the tile of iteration it + 3
    g = g_next;
  }
#if KZ_BULK_ZERO
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // the zero page must outlive the copies that read it
#endif
}

// ------------------------------------------------------------------------------------------------
// Legal bitmap rows -> byte-mask rows (PolicyOutputMapper.get_legal_mask's layout, utils.py:310-336) for callers of the
// reference API; any row stride / alignment (4 mask bytes per store when the row is 4-byte aligned).
__global__ void __launch_bounds__(256) kz_bitmap_expand_kernel(const uint32_t* __restrict__ bitmap, long long ldb,
                                                               const long long* __restrict__ rows, int n,
                                                               uint8_t* __restrict__ mask, long long ldm) {
  const int lane = threadIdx.x & 31;
  const int g = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (g >= n) return;
  const uint32_t* bm = bitmap + (size_t)(rows ? rows[g] : g) * ldb;
  uint8_t* mrow = mask + (size_t)g * ldm;
  if ((((uintptr_t)mrow) & 3) == 0) {
    uint32_t* m32 = reinterpret_cast<uint32_t*>(mrow);
    for (int q = lane; q < KZ_NUM_ACTIONS / 4; q += 32)  // 4 actions per store
      m32[q] = (((__ldg(bm + (q >> 3)) >> ((q & 7) * 4)) & 0xF) * 0x00204081u) & 0x01010101u;
    for (int i = (KZ_NUM_ACTIONS / 4) * 4 + lane; i < KZ_NUM_ACTIONS; i += 32) mrow[i] = (uint8_t)((__ldg(bm + (i >> 5)) >> (i & 31)) & 1);
  } else {
    for (int i = lane; i < KZ_NUM_ACTIONS; i += 32) mrow[i] = (uint8_t)((__ldg(bm + (i >> 5)) >> (i & 31)) & 1);
  }
}

// ------------------------------------------------------------------------------------------------
// Legal bitmap rows -> a CSR list of legal moves (kz_legal_list), one warp per game: the set bits of row g in ascending
// order go to [offsets[g], offsets[g+1]).  The warp walks the row 32 words at a time and visits only the non-zero words
// (ballot); within a word, lane l owns bit l, and its place is the popcount of the bits below it.  Nothing is written
// outside a row's own range, whatever its offsets say.
__global__ void __launch_bounds__(256) kz_legal_list_kernel(const uint32_t* __restrict__ bitmap, long long ldb, int n,
                                                            const long long* __restrict__ offsets, int32_t* parent_out,
                                                            void* actions_out, int actions_i64) {
  const int lane = threadIdx.x & 31;
  const int g = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (g >= n) return;
  const long long lo = offsets[g], hi = offsets[g + 1];
  if (lo < 0) return;
  const uint32_t* bm = bitmap + (size_t)g * ldb;
  long long base = lo;
  for (int w0 = 0; w0 < KZ_BITMAP_WORDS_MIN && base < hi; w0 += 32) {  // warp-uniform
    const int w = w0 + lane;
    uint32_t v = w < KZ_BITMAP_WORDS_MIN ? __ldg(bm + w) : 0u;
    if (w == KZ_BITMAP_WORDS_MIN - 1) v &= (1u << (KZ_NUM_ACTIONS - 32 * (KZ_BITMAP_WORDS_MIN - 1))) - 1u;
    uint32_t nz = __ballot_sync(FULL, v != 0);
    while (nz) {
      const int k = __ffs(nz) - 1;
      nz &= nz - 1;
      const uint32_t word = __shfl_sync(FULL, v, k);
      const long long pos = base + __popc(word & ((1u << lane) - 1u));
      if (((word >> lane) & 1) && pos < hi) {
        const int a = (w0 + k) * 32 + lane;
        if (actions_i64) reinterpret_cast<long long*>(actions_out)[pos] = a;
        else reinterpret_cast<int32_t*>(actions_out)[pos] = a;
        if (parent_out) parent_out[pos] = g;
      }
      base += __popc(word);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Legal moves that give check (kz_check_bitmap), one warp per game, games in a grid-stride loop.  Built per game from the
// enemy king's square KE at the current occupancy:
//   check squares cs[t]: the squares from which a piece of the mover's type t attacks KE -- the targets from KE of the
//     ENEMY's piece of type t (reverse step pattern; sliders up to and including the first blocker), one lane per type;
//   discovered-check lines: lane d walks ray d from KE; an own first piece followed by an own slider that attacks KE along
//     that ray makes the first piece a candidate, and seg[d] is the squares strictly between KE and the slider.
// A board move from -> to checks if `to` is in the check squares of the piece's type after the move (promoted type for the
// odd bits), or if from is a candidate and to leaves seg[d]; a drop of type t on `to` checks if `to` is in cs[t].  The
// check squares are taken at the occupancy before the move; the only square that changes and could lie between `to`
// and KE is `from`, and then the piece moves along that line away from KE, so it already attacked KE from `from` (no
// promotion adds a slide direction) -- the enemy was in check, which is the out-of-contract case below.
// Row = legal row AND that set.  Finished game: empty row.  Enemy king missing, or already attacked (loaded positions
// only): the whole legal row.
struct CheckScratch {
  uint32_t cs[14][3];  // check squares per piece type of the mover (bitboards)
  uint32_t seg[8][3];  // discovered-check line d: squares strictly between KE and the own slider
  uint8_t board[96];
  uint8_t disc[96];    // direction of the line a discovered-check candidate blocks, 0xFF none
  uint8_t dchk[96];    // bit t: a drop of type t on this square gives check
};

__device__ __forceinline__ uint32_t bits17(const uint32_t (&b)[3], int lo) {  // bits lo .. lo + 16 of a bitboard (lo <= 64)
  const int wd = lo >> 5;
  const uint32_t a = wd == 0 ? b[0] : (wd == 1 ? b[1] : b[2]);
  const uint32_t c = wd == 0 ? b[1] : (wd == 1 ? b[2] : 0u);
  return __funnelshift_r(a, c, lo & 31) & 0x1FFFFu;
}

__global__ void __launch_bounds__(256) kz_check_bitmap_kernel(const uint8_t* __restrict__ boards,
                                                              const uint8_t* __restrict__ meta, int n,
                                                              const uint32_t* __restrict__ bitmap, long long ldb,
                                                              uint32_t* __restrict__ out, long long ldo, int32_t* count) {
  __shared__ CheckScratch s_chk[8];
  for (int i = threadIdx.x; i < 81 * 8 * 3; i += blockDim.x) s_ray[i] = g_ray[i];
  for (int i = threadIdx.x; i < NCLS * 81 * 3; i += blockDim.x) s_step[i] = g_step[i];
  __syncthreads();
  const Tables T{};
  const int lane = threadIdx.x & 31;
  CheckScratch& S = s_chk[threadIdx.x >> 5];
  const uint32_t tab = code_info(lane);
  for (int g = blockIdx.x * 8 + (threadIdx.x >> 5); g < n; g += gridDim.x * 8) {  // warp-uniform
    __syncwarp();
    if (lane < 24) reinterpret_cast<uint32_t*>(S.board)[lane] = reinterpret_cast<const uint32_t*>(boards + (size_t)g * 96)[lane];
    const int me = meta[(size_t)g * 32 + 14], status = meta[(size_t)g * 32 + 15];
    __syncwarp();
    int c[3];
    uint32_t o[3], ek[3];
#pragma unroll
    for (int j = 0; j < 3; j++) {
      c[j] = lane + 32 * j < 81 ? S.board[lane + 32 * j] : 0;
      o[j] = __ballot_sync(FULL, c[j] != 0);
      ek[j] = __ballot_sync(FULL, c[j] == 8 + 14 * (1 - me));
      S.disc[lane + 32 * j] = 0xFF;
    }
    __syncwarp();
    const BB occ{o[0], o[1], o[2]};
    const int KE = (ek[0] | ek[1] | ek[2]) ? bb_lsb(BB{ek[0], ek[1], ek[2]}) : -1;  // find_king: first in row-major order
    int mode = status != 0 ? 0 : (KE < 0 ? 1 : 2);  // 0 empty row, 1 every legal move, 2 checking moves
    if (mode == 2) {
      {  // check squares: lane t < 14 = the targets from KE of the enemy's piece of type t
        const uint32_t inf = __shfl_sync(FULL, tab, lane < 14 ? 1 + lane + 14 * (1 - me) : 0);
        if (lane < 14) {
          BB t = ld_step(T, (inf >> 16) & 15, KE);
          uint32_t sl = (inf >> 8) & 0xFF;
          while (sl) {
            const int d = __ffs(sl) - 1;
            sl &= sl - 1;
            t = t | slide_ray(T, KE, d, occ);
          }
          S.cs[lane][0] = t.w0; S.cs[lane][1] = t.w1; S.cs[lane][2] = t.w2;
        }
      }
      {  // discovered-check candidates on the eight rays from KE
        const int d = lane & 7, od = (d + 4) & 7;
        const BB ray = ld_ray(T, KE, d);
        const BB bl = ray & occ;
        const bool pos = dir_positive(d);
        int b1 = -1, b2 = -1;
        if (bb_any(bl)) {
          b1 = pos ? bb_lsb(bl) : bb_msb(bl);
          const BB bl2 = bb_andn(bl, bb_bit(b1));
          if (bb_any(bl2)) b2 = pos ? bb_lsb(bl2) : bb_msb(bl2);
        }
        const int code1 = b1 >= 0 ? S.board[b1] : 0, code2 = b2 >= 0 ? S.board[b2] : 0;
        const uint32_t inf2 = __shfl_sync(FULL, tab, code2);
        if (lane < 8 && code1 && code_color(code1) == me && code2 && code_color(code2) == me && ((inf2 >> (8 + od)) & 1)) {
          const BB seg = pos ? (ray & bb_below(b2)) : bb_andn(ray, bb_upto(b2));
          S.disc[b1] = (uint8_t)d;
          S.seg[d][0] = seg.w0; S.seg[d][1] = seg.w1; S.seg[d][2] = seg.w2;
        }
      }
      __syncwarp();
      bool attacks = false;  // an own piece already attacks KE: the side not to move is in check
#pragma unroll
      for (int j = 0; j < 3; j++) {
        const int sq = lane + 32 * j;
        if (sq < 81 && c[j] && code_color(c[j]) == me) attacks |= (S.cs[code_type(c[j])][j] >> lane) & 1;
        if (sq < 96) {
          uint32_t v = 0;
#pragma unroll
          for (int t = 0; t < 7; t++) v |= (sq < 81 ? (S.cs[t][j] >> lane) & 1 : 0u) << t;
          S.dchk[sq] = (uint8_t)v;
        }
      }
      if (__any_sync(FULL, attacks)) mode = 1;
      __syncwarp();
    }
    const uint32_t* src = bitmap + (size_t)g * ldb;
    uint32_t* dst = out + (size_t)g * ldo;
    int cnt = 0;
    for (int wi = lane; wi < KZ_BITMAP_WORDS_MIN; wi += 32) {
      uint32_t v = mode ? __ldg(src + wi) : 0u;
      if (wi == KZ_BITMAP_WORDS_MIN - 1) v &= (1u << (KZ_NUM_ACTIONS - 32 * (KZ_BITMAP_WORDS_MIN - 1))) - 1u;
      if (mode == 2 && v) {
        uint32_t chk;
        if (wi < 405) {  // board moves: source square wi / 5, targets to' = lo .. lo + 15 (to = to' + (to' >= from))
          const int from = wi / 5, lo = 16 * (wi - 5 * from);
          const int t = code_type(S.board[from]);
          const int tp = (t <= 3 || t == 5 || t == 6) ? t + promo_delta(t) : t;  // odd bits exist only for promotable types
          const uint32_t below = lowmask32(from - lo);
          auto compact = [&](uint32_t x) { return ((x & below) | ((x >> 1) & ~below)) & 0xFFFFu; };
          chk = spread16(compact(bits17(S.cs[t], lo))) | (spread16(compact(bits17(S.cs[tp], lo))) << 1);
          const int dd = S.disc[from];
          if (dd != 0xFF) chk |= spread16(~compact(bits17(S.seg[dd], lo)) & 0xFFFFu) * 3u;
        } else {  // drops: word 405 + q holds drop-stream bits [32q, 32q + 32) (as gen_moves packs them)
          const int q = wi - 405;
          const int to0 = (32 * q * 293) >> 11;  // floor(32q / 7)
          int p = 7 * to0 - 32 * q;             // <= 0
          chk = 0;
#pragma unroll
          for (int i = 0; i < 6; i++) {
            const int to = to0 + i;
            const uint32_t dv = to < 81 ? S.dchk[to] : 0;
            if (p >= 0) { if (p < 32) chk |= dv << p; }
            else chk |= dv >> (-p);
            p += 7;
          }
        }
        v &= chk;
      }
      dst[wi] = v;
      cnt += __popc(v);
    }
    for (long long wi = KZ_BITMAP_WORDS_MIN + lane; wi < ldo; wi += 32) dst[wi] = 0u;
    cnt = (int)__reduce_add_sync(FULL, (unsigned)cnt);
    if (count && lane == 0) count[g] = cnt;
  }
}

// ------------------------------------------------------------------------------------------------
__global__ void kz_reset_kernel(uint8_t* boards, uint8_t* meta, uint4* rep, int rep_slots, int n,
                                const uint8_t* env_mask, int max_moves) {
  const int g = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (g >= n) return;
  if (env_mask && !env_mask[g]) return;
  if (rep) for (int i = lane; i < rep_slots; i += 32) rep[(size_t)g * rep_slots + i] = make_uint4(0, 0, 0, 0);
  uint32_t* b = reinterpret_cast<uint32_t*>(boards + (size_t)g * 96);
  uint32_t* m = reinterpret_cast<uint32_t*>(meta + (size_t)g * 32);
  if (lane < 24) b[lane] = reinterpret_cast<const uint32_t*>(c_init_board)[lane];
  else {
    const int w = lane - 24;
    uint32_t v = 0;
    if (w == 4) v = 0xFFu;                                  // bytes 16..19: winner none, err 0, move_count 0
    if (w == 5) v = ((uint32_t)max_moves & 0xFFFF) << 16;   // bytes 20..23: hist_len 0, max_moves
    if (w == 6) v = m[6];                                   // keep the finished-episode counter
    if (w == 7) v = c_init_key_w;                           // bytes 28..31: word w of the position key
    m[w] = v;
  }
}

// kz_reset_pool: as kz_reset_kernel, from record k of the start-position pool (same selection as kz_step_kernel<.., true>;
// the finished-episode counter is kept and not advanced)
__global__ void kz_reset_pool_kernel(uint8_t* boards, uint8_t* meta, uint4* rep, int rep_slots, int n, const uint8_t* env_mask,
                                     int max_moves, const uint32_t* pool, int pool_size, const int32_t* pick,
                                     unsigned long long pool_seed, uint32_t env_offset, int32_t* start_ids) {
  const int g = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (g >= n) return;
  if (env_mask && !env_mask[g]) return;
  uint32_t* m = reinterpret_cast<uint32_t*>(meta + (size_t)g * 32);
  const uint32_t episodes = m[6];
  __syncwarp();
  uint32_t k = pick ? (uint32_t)pick[g]
                    : (uint32_t)(((unsigned long long)rand32(pool_seed, (unsigned long long)env_offset + g, episodes) *
                                  (unsigned long long)pool_size) >> 32);
  if (k >= (uint32_t)pool_size) k %= (uint32_t)pool_size;
  const uint32_t* rec = pool + (size_t)k * KZ_POOL_RECORD_WORDS;
  for (int i = lane; i < rep_slots; i += 32) rep[(size_t)g * rep_slots + i] = make_uint4(0, 0, 0, 0);
  uint32_t* b = reinterpret_cast<uint32_t*>(boards + (size_t)g * 96);
  if (lane < 24) b[lane] = rec[lane];
  else {
    const int w = lane - 24;
    uint32_t v = rec[24 + w];                                             // hands, side, status 0, winner none, err 0, move_count
    if (w == 5) v = ((uint32_t)max_moves & 0xFFFF) << 16;                 // bytes 20..23: hist_len 0, max_moves
    if (w == 6) v = episodes;                                             // keep the finished-episode counter
    m[w] = v;                                                             // w == 7: word w of the position key
  }
  if (lane == 0 && start_ids) start_ids[g] = (int32_t)k;
}

// kz_pool_records: one start-position record per game of a refreshed scratch batch (layout: keisei_b200.h)
__global__ void kz_pool_records_kernel(const uint8_t* boards, const uint8_t* meta, int n, const uint32_t* bitmap,
                                       long long bitmap_stride, const int32_t* legal_count, const uint8_t* in_check,
                                       uint32_t* records) {
  const int g = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (g >= n) return;
  uint32_t* rec = records + (size_t)g * KZ_POOL_RECORD_WORDS;
  if (lane < 24) rec[lane] = reinterpret_cast<const uint32_t*>(boards + (size_t)g * 96)[lane];
  else {
    const int w = lane - 24;
    uint32_t v = reinterpret_cast<const uint32_t*>(meta + (size_t)g * 32)[w];
    if (w == 3) v &= 0x00FFFFFFu;  // bytes 12..15: hands, side to move, status 0
    if (w == 4) v = (v & 0xFFFF0000u) | 0xFFu;  // bytes 16..19: winner none, err 0, move_count
    if (w == 5 || w == 6) v = 0;  // plies since reset, max_moves (the env's own applies), finished episodes
    rec[24 + w] = v;
  }
  if (lane == 0) rec[32] = (uint32_t)legal_count[g];
  if (lane == 1) rec[33] = in_check[g];
  if (lane >= 2) for (int i = 32 + lane; i < KZ_POOL_BITMAP_OFFSET; i += 30) rec[i] = 0;
  const uint32_t* src = bitmap + (size_t)g * bitmap_stride;
  for (int i = lane; i < BITMAP_WORDS; i += 32) rec[KZ_POOL_BITMAP_OFFSET + i] = src[i];
}

__global__ void kz_load_kernel(uint8_t* boards, uint8_t* meta, uint4* rep, int rep_slots, int n, const int8_t* src_b,
                               const uint8_t* src_h, const uint8_t* src_side, const int32_t* src_mc,
                               const int32_t* src_mm) {
  const int g = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (g >= n) return;
  for (int i = lane; i < rep_slots; i += 32) rep[(size_t)g * rep_slots + i] = make_uint4(0, 0, 0, 0);
  uint8_t* b = boards + (size_t)g * 96;
  uint8_t* m = meta + (size_t)g * 32;
  for (int i = lane; i < 96; i += 32) b[i] = i < 81 ? (uint8_t)src_b[(size_t)g * 81 + i] : 0;
  uint8_t v = 0;
  if (lane < 14) v = src_h[(size_t)g * 14 + lane];
  else if (lane == 14) v = src_side[g];
  else if (lane == 16) v = 0xFF;
  else if (lane == 18) v = (uint8_t)src_mc[g];
  else if (lane == 19) v = (uint8_t)(src_mc[g] >> 8);
  else if (lane == 22) v = (uint8_t)src_mm[g];
  else if (lane == 23) v = (uint8_t)(src_mm[g] >> 8);
  m[lane] = v;
}

__global__ void kz_export_kernel(const uint8_t* boards, const uint8_t* meta, int n, int8_t* dst_b, uint8_t* dst_h,
                                 int32_t* dst_m) {
  const int g = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (g >= n) return;
  const uint8_t* b = boards + (size_t)g * 96;
  const uint8_t* m = meta + (size_t)g * 32;
  if (dst_b) for (int i = lane; i < 81; i += 32) dst_b[(size_t)g * 81 + i] = (int8_t)b[i];
  if (dst_h && lane < 14) dst_h[(size_t)g * 14 + lane] = m[lane];
  if (dst_m && lane < 8) {
    int v = 0;
    switch (lane) {
      case 0: v = m[14]; break;
      case 1: v = m[18] | (m[19] << 8); break;
      case 2: v = m[22] | (m[23] << 8); break;
      case 3: v = m[15]; break;
      case 4: v = m[16] == 0xFF ? -1 : m[16]; break;
      case 5: v = m[17]; break;
      case 6: v = m[20] | (m[21] << 8); break;
      case 7: v = m[24] | (m[25] << 8) | (m[26] << 16) | (m[27] << 24); break;
    }
    dst_m[(size_t)g * 8 + lane] = v;
  }
}

__global__ void kz_errors_kernel(uint8_t* meta, int n, int32_t* out, int clear) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n) return;
  out[g] = meta[(size_t)g * 32 + 17];
  if (clear) meta[(size_t)g * 32 + 17] = 0;
}

// Pseudo-legal targets of the piece standing on squares[g] (generate_piece_potential_moves,
// shogi_rules_logic.py:82-208): steps + slides up to the first blocker, own-colour squares removed.
__global__ void kz_targets_kernel(const uint8_t* boards, int n, const int32_t* squares, uint32_t* out) {
  for (int i = threadIdx.x; i < 81 * 8 * 3; i += blockDim.x) s_ray[i] = g_ray[i];
  for (int i = threadIdx.x; i < NCLS * 81 * 3; i += blockDim.x) s_step[i] = g_step[i];
  __syncthreads();
  const int g = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (g >= n) return;
  const Tables T{};
  const uint8_t* b = boards + (size_t)g * 96;
  const int sq = squares[g];
  const uint32_t tab = code_info(lane);
  const int code = (sq >= 0 && sq < 81) ? b[sq] : 0;
  const uint32_t inf = __shfl_sync(FULL, tab, code);
  const int me = code_color(code);
  uint32_t o[3], w[3];
#pragma unroll
  for (int j = 0; j < 3; j++) {
    const int s = lane + 32 * j;
    const int c = s < 81 ? b[s] : 0;
    o[j] = __ballot_sync(FULL, c != 0);
    w[j] = __ballot_sync(FULL, c != 0 && code_color(c) == me);
  }
  BB t = BB{0, 0, 0};
  if (code) {
    t = ld_step(T, (inf >> 16) & 15, sq);
    uint32_t sl = (inf >> 8) & 0xFF;
    while (sl) { const int d = __ffs(sl) - 1; sl &= sl - 1; t = t | slide_ray(T, sq, d, BB{o[0], o[1], o[2]}); }
    t = bb_andn(t, BB{w[0], w[1], w[2]});
  }
  if (lane == 0) { out[(size_t)g * 3] = t.w0; out[(size_t)g * 3 + 1] = t.w1; out[(size_t)g * 3 + 2] = t.w2; }
}

thread_local char t_cuda_err[256] = "";
int cuda_fail(cudaError_t e) {
  snprintf(t_cuda_err, sizeof t_cuda_err, "%s", cudaGetErrorString(e));
  return KZ_E_CUDA;
}
}  // namespace
int kz_cuda_fail(cudaError_t e) { return cuda_fail(e); }  // shared with kz_rl.cu / kz_nn.cu: one kz_last_cuda_error
namespace {
#define CK(x) do { cudaError_t _e = (x); if (_e != cudaSuccess) return cuda_fail(_e); } while (0)

// per device (kz_init_tables runs once per device: the tables are __device__ symbols of the current device)
constexpr int kMaxDevices = 64;
int g_sm_counts[kMaxDevices] = {0};
bool g_ready[kMaxDevices] = {false};
inline int cur_device() { int d = 0; return cudaGetDevice(&d) == cudaSuccess && d >= 0 && d < kMaxDevices ? d : -1; }
inline bool host_ready() { const int d = cur_device(); return d >= 0 && g_ready[d]; }
inline int sm_count() { const int d = cur_device(); return d >= 0 ? g_sm_counts[d] : 0; }

// The kz_step_kernel instantiations, [pool][mode]: refresh (mode 0) and expansion (mode 3) have no pool form.  launch_step
// launches through this table and kz_init_tables sets the dynamic shared-memory limit of every entry.
using StepKernel = void (*)(const StepParams);
const StepKernel kStepKernels[2][4] = {{kz_step_kernel<0>, kz_step_kernel<1>, kz_step_kernel<2>, kz_step_kernel<3>},
                                       {nullptr, kz_step_kernel<1, true>, kz_step_kernel<2, true>, nullptr}};
StepKernel step_kernel(int mode, bool pool) { return mode >= 0 && mode < 4 ? kStepKernels[pool][mode] : nullptr; }

#ifndef KZ_COMPACT_CTAS_PER_SM
#define KZ_COMPACT_CTAS_PER_SM 2
#endif

int launch_kernel(StepParams P, const StateBlob& src, int hist_cap, int slot, cudaStream_t st);

int launch_step(void* state, int n, int hist_cap, StepParams P, cudaStream_t st, int first = 0, int count = -1, int slot = 0) {
  StateBlob B;
  if (bind_state(state, n, hist_cap, B) != KZ_OK) return KZ_E_ARG;
  if (count < 0) count = n - first;
  if (first < 0 || count <= 0 || first + count > n || slot < 0 || slot >= 64) return KZ_E_ARG;
  if (!host_ready()) return KZ_E_NOT_INIT;
  P.n = count;
  P.g_first = first;
  return launch_kernel(P, B, hist_cap, slot, st);
}

// Row checks, grid, work counter (slot `slot` of the source blob's scheduling block) and the launch of
// kz_step_kernel<P.mode> on the source blob `src` over the P.n games (or kz_expand's items) from P.g_first on.
int launch_kernel(StepParams P, const StateBlob& src, int hist_cap, int slot, cudaStream_t st) {
  P.boards = src.boards; P.meta = src.meta; P.hist = src.hist; P.rep_slots = src.rep_slots; P.hist_cap = hist_cap;
  const int count = P.n;
  if (P.obs) {
    if (((uintptr_t)P.obs & 15) || (P.obs_stride & 1) || P.obs_stride < KZ_OBS_FLOATS) return KZ_E_ARG;
  }
  if (P.bitmap_out) {
    if (((uintptr_t)P.bitmap_out & 15) || P.bitmap_stride < BITMAP_WORDS || (P.bitmap_stride & 3)) return KZ_E_ARG;
  } else if (P.mode == 2) return KZ_E_ARG;
  if (P.cobs_out && ((uintptr_t)P.cobs_out & 3)) return KZ_E_ARG;
  P.mask_vec = 0;
  if (P.mask) {
    if (P.mask_stride < KZ_NUM_ACTIONS) return KZ_E_ARG;
    P.mask_vec = (((uintptr_t)P.mask & 15) == 0 && (P.mask_stride & 15) == 0) ? 1 : 0;
    if (count == 1 && ((uintptr_t)P.mask & 15) == 0) P.mask_vec = 1;
  }
  const int ctas_needed = (count + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
  // rollout-form launches without observation rows run KZ_COMPACT_CTAS_PER_SM CTAs per SM: tuned in round 1 next to an
  // expander kernel (since removed) and not re-measured since
  int grid = sm_count() * ((P.mode == 2 && !P.obs) ? KZ_COMPACT_CTAS_PER_SM : CTAS_PER_SM);
  if (grid > ctas_needed) grid = ctas_needed;
  const size_t dyn = sizeof(WarpScratch) * WARPS_PER_CTA;
  P.tile_counter = nullptr;
#ifndef KZ_STATIC_TILES
  if (grid < ctas_needed && count % WARPS_PER_CTA == 0) {
    // launches on one state buffer are ordered by their data dependence, so the counter can live in it (launches over
    // disjoint game ranges that run concurrently, kz_step_range, name different counter slots)
    P.tile_counter = reinterpret_cast<int*>(src.sched) + slot;
    CK(cudaMemsetAsync(P.tile_counter, 0, sizeof(int), st));
  }
#endif
  const StepKernel kernel = step_kernel(P.mode, P.pool != nullptr);
  if (!kernel) return KZ_E_ARG;
  kernel<<<grid, WARPS_PER_CTA * 32, dyn, st>>>(P);
  CK(cudaGetLastError());
  return KZ_OK;
}

// kz_step, kz_step_rollout, kz_step_range and kz_step_pool: games [first, first + count) of the batch, in the mask form
// (bitmap == NULL) or the rollout form (bitmap != NULL); finished games restart from the pool when pool != NULL.
int step_games(void* state, int n, int hist_cap, int first, int count, int counter_slot, const void* actions,
               int actions_i64, float* obs, int64_t obs_stride, uint8_t* mask, int64_t mask_stride, uint32_t* bitmap,
               int64_t bitmap_stride_words, uint32_t* cobs, float* reward, uint8_t* done, uint8_t* reason, int8_t* winner,
               int32_t* ep_len, int32_t* legal_count, void* next_actions, uint64_t seed, uint32_t rng_step,
               uint32_t env_offset, int auto_reset, const uint32_t* pool, int pool_size, const int32_t* pick,
               uint64_t pool_seed, int32_t* start_ids, void* stream) {
  if (!actions) return KZ_E_ARG;
  StepParams P{};
  P.actions = actions; P.actions_i64 = actions_i64;
  P.obs = obs; P.obs_stride = obs_stride; P.mask = mask; P.mask_stride = mask_stride;
  P.bitmap_out = bitmap; P.bitmap_stride = bitmap_stride_words; P.cobs_out = cobs;
  P.reward = reward; P.done = done; P.reason = reason; P.winner = winner; P.ep_len = ep_len;
  P.legal_count = legal_count; P.next_actions = next_actions;
  P.seed = seed; P.rng_step = rng_step; P.env_offset = env_offset;
  P.auto_reset = auto_reset; P.mode = bitmap ? 2 : 1;
  P.pool = pool; P.pool_size = pool_size; P.pool_pick = pick; P.pool_seed = pool_seed; P.start_ids = start_ids;
  return launch_step(state, n, hist_cap, P, reinterpret_cast<cudaStream_t>(stream), first, count, counter_slot);
}

}  // namespace

extern "C" {

int kz_abi_version(void) { return KZ_ABI_VERSION; }
#ifndef KZ_SRC_SHA
#define KZ_SRC_SHA "unknown"
#endif
const char* kz_build_info(void) { return "src_sha=" KZ_SRC_SHA " built=" __DATE__ " " __TIME__ " arch=sm_100a"; }
const char* kz_last_cuda_error(void) { return t_cuda_err; }

int kz_state_layout(int n, int hist_cap, int64_t* offsets3, int64_t* total_bytes) {
  if (n <= 0 || hist_cap < 0 || hist_cap > 65535) return KZ_E_ARG;
  const Layout L = layout(n, hist_cap);
  if (offsets3) { offsets3[0] = L.off_boards; offsets3[1] = L.off_meta; offsets3[2] = L.off_hist; }
  if (total_bytes) *total_bytes = L.total;
  return KZ_OK;
}

int kz_init_tables(void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  static const int DR[8] = {-1, -1, 0, 1, 1, 1, 0, -1};
  static const int DC[8] = {0, 1, 1, 1, 0, -1, -1, -1};
  static uint32_t ray[81 * 8 * 3];
  static uint32_t step[NCLS * 81 * 3];
  memset(ray, 0, sizeof ray);
  memset(step, 0, sizeof step);
  auto setb = [](uint32_t* bb, int s) { bb[s >> 5] |= 1u << (s & 31); };
  for (int s = 0; s < 81; s++) {
    const int r = s / 9, c = s % 9;
    for (int d = 0; d < 8; d++)
      for (int k = 1; k < 9; k++) {
        const int rr = r + DR[d] * k, cc = c + DC[d] * k;
        if (rr < 0 || rr > 8 || cc < 0 || cc > 8) break;
        setb(ray + (s * 8 + d) * 3, rr * 9 + cc);
      }
    // step classes: direction sets for BLACK (forward = N = dir 0); WHITE is the 180-degree rotation
    const uint32_t P_ = 0x01, S_ = 0x01 | 0x02 | 0x80 | 0x08 | 0x20, G_ = 0x01 | 0x02 | 0x80 | 0x04 | 0x40 | 0x10;
    const uint32_t PLUS_ = 0x55, X_ = 0xAA, K_ = 0xFF;
    auto rot = [](uint32_t m) { return ((m << 4) | (m >> 4)) & 0xFF; };
    const uint32_t dirsets[NCLS] = {P_, S_, G_, 0, rot(P_), rot(S_), rot(G_), 0, PLUS_, X_, K_, 0};
    for (int cls = 0; cls < NCLS; cls++) {
      uint32_t* bb = step + (cls * 81 + s) * 3;
      for (int d = 0; d < 8; d++)
        if ((dirsets[cls] >> d) & 1) {
          const int rr = r + DR[d], cc = c + DC[d];
          if (rr >= 0 && rr <= 8 && cc >= 0 && cc <= 8) setb(bb, rr * 9 + cc);
        }
      if (cls == CLS_BN || cls == CLS_WN) {  // knight: (2*forward, +-1) (shogi_rules_logic.py:121)
        const int f = cls == CLS_BN ? -1 : 1;
        for (int dc = -1; dc <= 1; dc += 2) {
          const int rr = r + 2 * f, cc = c + dc;
          if (rr >= 0 && rr <= 8 && cc >= 0 && cc <= 8) setb(bb, rr * 9 + cc);
        }
      }
    }
  }
  // start position (shogi_game.py:79-111)
  static uint8_t init[96];
  memset(init, 0, sizeof init);
  static const int back[9] = {1, 2, 3, 4, 7, 4, 3, 2, 1};
  for (int c = 0; c < 9; c++) {
    init[0 * 9 + c] = (uint8_t)(1 + back[c] + 14);
    init[8 * 9 + c] = (uint8_t)(1 + back[c]);
    init[2 * 9 + c] = (uint8_t)(1 + 0 + 14);
    init[6 * 9 + c] = (uint8_t)(1 + 0);
  }
  init[1 * 9 + 1] = 1 + 6 + 14; init[1 * 9 + 7] = 1 + 5 + 14;
  init[7 * 9 + 1] = 1 + 5;      init[7 * 9 + 7] = 1 + 6;
  CK(cudaMemcpyToSymbolAsync(g_ray, ray, sizeof ray, 0, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyToSymbolAsync(g_step, step, sizeof step, 0, cudaMemcpyHostToDevice, st));
  {  // position key of the start position (same hash functions as zkey_item / position_key on the device)
    auto fmix = [](uint32_t h) { h ^= h >> 16; h *= 0x85ebca6bu; h ^= h >> 13; h *= 0xc2b2ae35u; h ^= h >> 16; return h; };
    uint32_t k[4] = {0, 0, 0, 0};
    for (int sq = 0; sq < 81; sq++)
      if (init[sq]) {
        const uint32_t id = (uint32_t)sq * 32u + init[sq];
        k[0] ^= fmix(id * 0x9E3779B1u + 0x7F4A7C15u);
        k[1] ^= fmix(id * 0x85EBCA77u + 0x165667B1u);
        k[2] ^= fmix(id * 0xC2B2AE3Du + 0x27D4EB2Fu);
        k[3] ^= fmix(id * 0x27D4EB2Fu + 0x9E3779B9u);
      }
    memcpy(init + 84, k, 12);
    CK(cudaMemcpyToSymbolAsync(c_init_key_w, &k[3], sizeof(uint32_t), 0, cudaMemcpyHostToDevice, st));
  }
  CK(cudaMemcpyToSymbolAsync(c_init_board, init, sizeof init, 0, cudaMemcpyHostToDevice, st));
  int dev = 0;
  CK(cudaGetDevice(&dev));
  if (dev < 0 || dev >= kMaxDevices) return KZ_E_ARG;
  CK(cudaDeviceGetAttribute(&g_sm_counts[dev], cudaDevAttrMultiProcessorCount, dev));
  {  // per-warp scratch lives in dynamic shared memory (more than 48 KB with tables for CTAs above 8 warps)
    const int dyn = (int)(sizeof(WarpScratch) * WARPS_PER_CTA);
    for (const auto& row : kStepKernels)
      for (StepKernel kernel : row)
        if (kernel) CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn));
  }
  g_ready[dev] = true;
  // legal bitmap of the start position, computed once by the engine itself on a scratch game
  {
    int64_t total = 0;
    kz_state_layout(1, 0, nullptr, &total);
    void* scratch = nullptr;
    CK(cudaMalloc(&scratch, total + KZ_MASK_PAD_STRIDE));
    StateBlob B;
    bind_state(scratch, 1, 0, B);
    kz_reset_kernel<<<1, 32, 0, st>>>(B.boards, B.meta, nullptr, 0, 1, nullptr, 500);
    StepParams P{};
    P.mask = reinterpret_cast<uint8_t*>(scratch) + total;  // the mask row follows the blob
    P.mask_stride = KZ_MASK_PAD_STRIDE;
    P.mode = 0;
    int rc = launch_step(scratch, 1, 0, P, st);
    if (rc != KZ_OK) { cudaFree(scratch); return rc; }
    CK(cudaStreamSynchronize(st));
    static uint8_t hm[KZ_MASK_PAD_STRIDE];
    CK(cudaMemcpy(hm, P.mask, KZ_MASK_PAD_STRIDE, cudaMemcpyDeviceToHost));
    static uint32_t bm[BITMAP_WORDS];
    memset(bm, 0, sizeof bm);
    for (int i = 0; i < KZ_NUM_ACTIONS; i++)
      if (hm[i]) bm[i >> 5] |= 1u << (i & 31);
    CK(cudaMemcpyToSymbol(g_init_bitmap, bm, sizeof bm));
    CK(cudaFree(scratch));
  }
  return KZ_OK;
}

int kz_reset(void* state, int n, int hist_cap, const uint8_t* env_mask, int max_moves, void* stream) {
  StateBlob B;
  if (bind_state(state, n, hist_cap, B) != KZ_OK || max_moves < 0 || max_moves > 65535) return KZ_E_ARG;
  if (!host_ready()) return KZ_E_NOT_INIT;
  kz_reset_kernel<<<(n + 7) / 8, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(B.boards, B.meta, B.hist, B.rep_slots, n,
                                                                                  env_mask, max_moves);
  CK(cudaGetLastError());
  return KZ_OK;
}

int kz_reset_pool(void* state, int n, int hist_cap, const uint8_t* env_mask, int max_moves, const uint32_t* pool, int pool_size,
                  const int32_t* pick, uint64_t pool_seed, uint32_t env_offset, int32_t* start_ids, void* stream) {
  StateBlob B;
  if (bind_state(state, n, hist_cap, B) != KZ_OK || max_moves < 0 || max_moves > 65535 || !pool || pool_size <= 0 ||
      ((uintptr_t)pool & 15))
    return KZ_E_ARG;
  if (!host_ready()) return KZ_E_NOT_INIT;
  kz_reset_pool_kernel<<<(n + 7) / 8, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      B.boards, B.meta, B.hist, B.rep_slots, n, env_mask, max_moves, pool, pool_size, pick, pool_seed, env_offset, start_ids);
  CK(cudaGetLastError());
  return KZ_OK;
}

int kz_pool_records(const void* state, int n, int hist_cap, const uint32_t* bitmap, int64_t bitmap_stride_words,
                    const int32_t* legal_count, const uint8_t* in_check, uint32_t* records, void* stream) {
  StateBlob B;
  if (bind_state(state, n, hist_cap, B) != KZ_OK || !bitmap || bitmap_stride_words < BITMAP_WORDS || !legal_count ||
      !in_check || !records || ((uintptr_t)records & 15))
    return KZ_E_ARG;
  kz_pool_records_kernel<<<(n + 7) / 8, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      B.boards, B.meta, n, bitmap, bitmap_stride_words, legal_count, in_check, records);
  CK(cudaGetLastError());
  return KZ_OK;
}

int kz_load_positions(void* state, int n, int hist_cap, const int8_t* boards, const uint8_t* hands,
                      const uint8_t* side, const int32_t* move_count, const int32_t* max_moves, void* stream) {
  StateBlob B;
  if (bind_state(state, n, hist_cap, B) != KZ_OK || !boards || !hands || !side || !move_count || !max_moves) return KZ_E_ARG;
  kz_load_kernel<<<(n + 7) / 8, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      B.boards, B.meta, B.hist, B.rep_slots, n, boards, hands, side, move_count, max_moves);
  CK(cudaGetLastError());
  return KZ_OK;
}

int kz_export_positions(const void* state, int n, int hist_cap, int8_t* boards, uint8_t* hands, int32_t* meta8,
                        void* stream) {
  StateBlob B;
  if (bind_state(state, n, hist_cap, B) != KZ_OK) return KZ_E_ARG;
  kz_export_kernel<<<(n + 7) / 8, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(B.boards, B.meta, n, boards, hands, meta8);
  CK(cudaGetLastError());
  return KZ_OK;
}

int kz_piece_targets(const void* state, int n, int hist_cap, const int32_t* squares, uint32_t* targets3, void* stream) {
  StateBlob B;
  if (bind_state(state, n, hist_cap, B) != KZ_OK || !squares || !targets3) return KZ_E_ARG;
  if (!host_ready()) return KZ_E_NOT_INIT;
  kz_targets_kernel<<<(n + 7) / 8, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(B.boards, n, squares, targets3);
  CK(cudaGetLastError());
  return KZ_OK;
}

int kz_errors(void* state, int n, int hist_cap, int32_t* out, int clear, void* stream) {
  StateBlob B;
  if (bind_state(state, n, hist_cap, B) != KZ_OK || !out) return KZ_E_ARG;
  kz_errors_kernel<<<(n + 255) / 256, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(B.meta, n, out, clear);
  CK(cudaGetLastError());
  return KZ_OK;
}

int kz_refresh(void* state, int n, int hist_cap, float* obs, int64_t obs_stride, uint8_t* mask, int64_t mask_stride,
               int32_t* legal_count, void* next_actions, int actions_i64, uint64_t seed, uint32_t rng_step,
               uint32_t env_offset, int eval_termination, uint8_t* in_check, void* stream) {
  StepParams P{};
  P.in_check = in_check;
  P.obs = obs; P.obs_stride = obs_stride; P.mask = mask; P.mask_stride = mask_stride;
  P.legal_count = legal_count; P.next_actions = next_actions; P.actions_i64 = actions_i64;
  P.seed = seed; P.rng_step = rng_step; P.env_offset = env_offset;
  P.mode = 0; P.eval_term = eval_termination;
  return launch_step(state, n, hist_cap, P, reinterpret_cast<cudaStream_t>(stream));
}

int kz_step(void* state, int n, int hist_cap, const void* actions, int actions_i64, float* obs, int64_t obs_stride,
            uint8_t* mask, int64_t mask_stride, float* reward, uint8_t* done, uint8_t* reason, int8_t* winner,
            int32_t* ep_len, int32_t* legal_count, void* next_actions, uint64_t seed, uint32_t rng_step,
            uint32_t env_offset, int auto_reset, void* stream) {
  return step_games(state, n, hist_cap, 0, n, 0, actions, actions_i64, obs, obs_stride, mask, mask_stride, nullptr, 0,
                    nullptr, reward, done, reason, winner, ep_len, legal_count, next_actions, seed, rng_step, env_offset,
                    auto_reset, nullptr, 0, nullptr, 0, nullptr, stream);
}

int kz_step_range(void* state, int n, int hist_cap, int first, int count, int counter_slot, const void* actions,
                  int actions_i64, float* obs, int64_t obs_stride, uint8_t* mask, int64_t mask_stride, uint32_t* bitmap,
                  int64_t bitmap_stride_words, uint32_t* cobs, float* reward, uint8_t* done, uint8_t* reason, int8_t* winner,
                  int32_t* ep_len, int32_t* legal_count, void* next_actions, uint64_t seed, uint32_t rng_step,
                  uint32_t env_offset, int auto_reset, void* stream) {
  if (mask && bitmap) return KZ_E_ARG;
  return step_games(state, n, hist_cap, first, count, counter_slot, actions, actions_i64, obs, obs_stride, mask, mask_stride,
                    bitmap, bitmap_stride_words, cobs, reward, done, reason, winner, ep_len, legal_count, next_actions, seed,
                    rng_step, env_offset, auto_reset, nullptr, 0, nullptr, 0, nullptr, stream);
}

int kz_step_pool(void* state, int n, int hist_cap, int first, int count, int counter_slot, const void* actions,
                 int actions_i64, float* obs, int64_t obs_stride, uint8_t* mask, int64_t mask_stride, uint32_t* bitmap,
                 int64_t bitmap_stride_words, uint32_t* cobs, float* reward, uint8_t* done, uint8_t* reason, int8_t* winner,
                 int32_t* ep_len, int32_t* legal_count, void* next_actions, uint64_t seed, uint32_t rng_step,
                 uint32_t env_offset, const uint32_t* pool, int pool_size, const int32_t* pick, uint64_t pool_seed,
                 int32_t* start_ids, void* stream) {
  if ((mask && bitmap) || !pool || pool_size <= 0 || ((uintptr_t)pool & 15)) return KZ_E_ARG;
  return step_games(state, n, hist_cap, first, count, counter_slot, actions, actions_i64, obs, obs_stride, mask, mask_stride,
                    bitmap, bitmap_stride_words, cobs, reward, done, reason, winner, ep_len, legal_count, next_actions, seed,
                    rng_step, env_offset, 1, pool, pool_size, pick, pool_seed, start_ids, stream);
}

int kz_step_rollout(void* state, int n, int hist_cap, const void* actions, int actions_i64, float* obs, int64_t obs_stride,
                    uint32_t* bitmap, int64_t bitmap_stride_words, uint32_t* cobs, float* reward, uint8_t* done, uint8_t* reason,
                    int8_t* winner, int32_t* ep_len, int32_t* legal_count, void* next_actions, uint64_t seed,
                    uint32_t rng_step, uint32_t env_offset, int auto_reset, void* stream) {
  if (!bitmap) return KZ_E_ARG;
  return step_games(state, n, hist_cap, 0, n, 0, actions, actions_i64, obs, obs_stride, nullptr, 0, bitmap,
                    bitmap_stride_words, cobs, reward, done, reason, winner, ep_len, legal_count, next_actions, seed, rng_step,
                    env_offset, auto_reset, nullptr, 0, nullptr, 0, nullptr, stream);
}

int kz_legal_bitmap(void* state, int n, int hist_cap, float* obs, int64_t obs_stride, uint32_t* bitmap,
                    int64_t bitmap_stride_words, uint32_t* cobs, int32_t* legal_count, void* stream) {
  if (!bitmap) return KZ_E_ARG;
  StepParams P{};
  P.obs = obs; P.obs_stride = obs_stride;
  P.bitmap_out = bitmap; P.bitmap_stride = bitmap_stride_words; P.cobs_out = cobs;
  P.legal_count = legal_count;
  P.mode = 0;
  return launch_step(state, n, hist_cap, P, reinterpret_cast<cudaStream_t>(stream));
}

int kz_bitmap_expand(const uint32_t* bitmap, int64_t bitmap_stride_words, const int64_t* bitmap_rows, int n, uint8_t* mask,
                     int64_t mask_stride, void* stream) {
  if (!bitmap || !mask || n <= 0 || bitmap_stride_words < 423 || mask_stride < KZ_NUM_ACTIONS || ((uintptr_t)bitmap & 3))
    return KZ_E_ARG;
  kz_bitmap_expand_kernel<<<(n + 7) / 8, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      bitmap, bitmap_stride_words, reinterpret_cast<const long long*>(bitmap_rows), n, mask, mask_stride);
  CK(cudaGetLastError());
  return KZ_OK;
}

int kz_legal_mask(void* state, int n, int hist_cap, uint8_t* mask, int64_t mask_stride, int32_t* legal_count,
                  void* stream) {
  if (!mask && !legal_count) return KZ_E_ARG;
  return kz_refresh(state, n, hist_cap, nullptr, 0, mask, mask_stride, legal_count, nullptr, 0, 0, 0, 0, 0, nullptr, stream);
}

int kz_observe(void* state, int n, int hist_cap, float* obs, int64_t obs_stride, void* stream) {
  if (!obs) return KZ_E_ARG;
  return kz_refresh(state, n, hist_cap, obs, obs_stride, nullptr, 0, nullptr, nullptr, 0, 0, 0, 0, 0, nullptr, stream);
}

int kz_legal_list(const uint32_t* bitmap, int64_t bitmap_stride_words, int n, const int64_t* offsets, int32_t* parent_out,
                  void* actions_out, int actions_i64, void* stream) {
  if (!bitmap || bitmap_stride_words < KZ_BITMAP_WORDS_MIN || n < 0 || !offsets || !actions_out || ((uintptr_t)bitmap & 3))
    return KZ_E_ARG;
  if (n == 0) return KZ_OK;
  kz_legal_list_kernel<<<(n + 7) / 8, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      bitmap, bitmap_stride_words, n, reinterpret_cast<const long long*>(offsets), parent_out, actions_out, actions_i64);
  CK(cudaGetLastError());
  return KZ_OK;
}

int kz_expand(const void* state, int n, int hist_cap, int counter_slot, const int32_t* parent, const void* actions,
              int actions_i64, int m, float* obs, int64_t obs_stride, uint32_t* bitmap, int64_t bitmap_stride_words,
              uint32_t* cobs, float* reward, uint8_t* done, uint8_t* reason, int8_t* winner, int32_t* ep_len,
              int32_t* legal_count, uint8_t* err, void* child_state, int child_hist_cap, void* stream) {
  StateBlob src, child;
  if (bind_state(state, n, hist_cap, src) != KZ_OK || !parent || !actions || m < 0 || counter_slot < 0 || counter_slot >= 64)
    return KZ_E_ARG;
  if (m == 0) return KZ_OK;
  if (child_state && (child_state == state || bind_state(child_state, m, child_hist_cap, child) != KZ_OK)) return KZ_E_ARG;
  if (!host_ready()) return KZ_E_NOT_INIT;
  // the kernel writes nothing of the source batch but its work counter (MODE 3)
  StepParams P{};
  P.n = m;
  P.g_first = 0;
  P.actions = actions; P.actions_i64 = actions_i64;
  P.obs = obs; P.obs_stride = obs_stride;
  P.bitmap_out = bitmap; P.bitmap_stride = bitmap_stride_words; P.cobs_out = cobs;
  P.reward = reward; P.done = done; P.reason = reason; P.winner = winner; P.ep_len = ep_len;
  P.legal_count = legal_count;
  P.mode = 3;
  P.parent = parent; P.src_n = n; P.err_out = err;
  if (child_state) {
    P.child_boards = child.boards; P.child_meta = child.meta; P.child_hist = child.hist; P.child_rep_slots = child.rep_slots;
  }
  return launch_kernel(P, src, hist_cap, counter_slot, reinterpret_cast<cudaStream_t>(stream));
}

int kz_check_bitmap(const void* state, int n, int hist_cap, const uint32_t* bitmap, int64_t bitmap_stride_words, uint32_t* out,
                    int64_t out_stride_words, int32_t* count, void* stream) {
  StateBlob B;
  if (bind_state(state, n, hist_cap, B) != KZ_OK || !bitmap || !out || bitmap_stride_words < KZ_BITMAP_WORDS_MIN ||
      out_stride_words < KZ_BITMAP_WORDS_MIN || ((uintptr_t)bitmap & 15) || ((uintptr_t)out & 15) || ((uintptr_t)count & 3))
    return KZ_E_ARG;
  const uintptr_t b0 = (uintptr_t)bitmap, b1 = b0 + (uintptr_t)n * (uintptr_t)bitmap_stride_words * 4u;
  const uintptr_t o0 = (uintptr_t)out, o1 = o0 + (uintptr_t)n * (uintptr_t)out_stride_words * 4u;
  if (o0 < b1 && b0 < o1) return KZ_E_ARG;  // out overlaps bitmap
  if (!host_ready()) return KZ_E_NOT_INIT;
  int grid = sm_count() * 8;  // 8 CTAs of 8 warps per SM (24 KB of static shared memory each)
  if (grid > (n + 7) / 8) grid = (n + 7) / 8;
  kz_check_bitmap_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      B.boards, B.meta, n, bitmap, bitmap_stride_words, out, out_stride_words, count);
  CK(cudaGetLastError());
  return KZ_OK;
}

}  // extern "C"
