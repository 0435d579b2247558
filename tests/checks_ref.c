/* checks_ref.c -- checking moves and mates in one by the CPU oracle's own rules (test infrastructure).
 *
 * Built by tests/checks_ref.py into a temporary directory.  It includes oracle/keisei_oracle.c unchanged: every legal move
 * (gen_legal, simulate-and-test) is applied to a copy of the position, and it gives check iff king_in_check(copy, opponent)
 * (a missing king counts as in check); it mates iff it gives check and the opponent then has no legal move (Tsumi comes
 * first in the reference's termination order, so history plays no part).  Shares nothing with the CUDA path's check
 * squares and discovered-check lines. */
#include "../oracle/keisei_oracle.c"

#define CLS_DIRECT 1     /* the moved piece attacks the enemy king, no other piece does */
#define CLS_DISCOVERED 2 /* another piece of the mover attacks it, the moved piece does not */
#define CLS_DOUBLE 3     /* both */
#define CLS_DROP 4       /* a dropped piece gives check */
#define CLS_NOKING 5     /* the enemy king is missing: every move "checks" */
#define CLS_PROMO_ONLY 8 /* flag: a promoting move that checks while the same move without promotion would not */
#define MATE_KING_CAPTURE 2 /* mate[a] value of a "mate" that captures the enemy king (out of contract) */

static int attacks(const int8_t *b, int from, int target) {
  int tg[40];
  int n = potential_moves(b, b[from], from / 9, from % 9, tg);
  for (int i = 0; i < n; i++)
    if (tg[i] == target) return 1;
  return 0;
}

/* other pieces of `color` than the one on `skip` that attack `target` */
static int others_attack(const int8_t *b, int target, int color, int skip) {
  for (int s = 0; s < NSQ; s++)
    if (s != skip && b[s] && pcolor(b[s]) == color && attacks(b, s, target)) return 1;
  return 0;
}

static void apply_action(orc_game *c, int a) {
  int me = c->side;
  if (a < 12960) {
    int pair = a >> 1, from = pair / 80, t = pair % 80;
    apply_board_move(c->board, c->hands, from, t + (t >= from), a & 1, me);
  } else {
    apply_drop(c->board, c->hands, (a - 12960) / 7, (a - 12960) % 7, me);
  }
  c->side = 1 - me;
}

/* For the position (board81, hands14, side): cls[a] (NACT bytes) = 0xFF for an illegal action, 0 for a legal one that
 * does not check, else CLS_* (| CLS_PROMO_ONLY); mate[a] = 1 for a mate, MATE_KING_CAPTURE for a "mate" that captures the
 * king.  Returns the number of legal moves; *enemy_in_check = the side not to move is in check already. */
int ref_checks(const int8_t *board81, const uint8_t *hands14, int side, uint8_t *cls, uint8_t *mate, int *enemy_in_check) {
  orc_game *g = orc_new();
  orc_load(g, board81, hands14, side, 0, 65535, 0);
  memset(cls, 0xFF, NACT);
  memset(mate, 0, NACT);
  int me = side, en = 1 - side;
  *enemy_in_check = king_in_check(g->board, en);
  uint16_t moves[1024], tmp[1024];
  int n = gen_legal(g, 0, moves);
  for (int i = 0; i < n; i++) {
    int a = moves[i];
    orc_game c = *g; /* shares g->hist, which nothing below reads */
    int cap_king = 0;
    if (a < 12960) {
      int pair = a >> 1, from = pair / 80, t = pair % 80, to = t + (t >= from);
      cap_king = c.board[to] == mk(T_KING, en);
    }
    apply_action(&c, a);
    cls[a] = 0;
    if (!king_in_check(c.board, en)) continue;
    int k = find_king(c.board, en);
    if (k < 0) cls[a] = CLS_NOKING;
    else if (a >= 12960) cls[a] = CLS_DROP;
    else {
      int pair = a >> 1, from = pair / 80, t = pair % 80, to = t + (t >= from);
      int direct = attacks(c.board, to, k), disc = others_attack(c.board, k, me, to);
      cls[a] = direct && disc ? CLS_DOUBLE : (direct ? CLS_DIRECT : CLS_DISCOVERED);
      if (a & 1) {
        orc_game u = *g;
        apply_action(&u, a - 1);
        if (!king_in_check(u.board, en)) cls[a] |= CLS_PROMO_ONLY;
      }
    }
    if (gen_legal(&c, 0, tmp) == 0) mate[a] = cap_king ? MATE_KING_CAPTURE : 1;
  }
  orc_free(g);
  return n;
}

/* ref_checks over n positions [first, first + count): per position the legal and checking moves as 423-word bitmaps
 * (bit a of word a / 32), the number of mates that do not capture the king and the lowest of them (-1 none), the number of
 * checking moves of each class (class_counts [n][6]: direct, discovered, double, drop, no king, promotion-only) and the
 * enemy-in-check flag. */
void ref_checks_batch(int first, int count, const int8_t *boards, const uint8_t *hands, const uint8_t *sides,
                      uint32_t *legal_bits, uint32_t *check_bits, int32_t *mate_count, int32_t *mate_lowest,
                      int32_t *class_counts, uint8_t *enemy_in_check) {
  uint8_t *cls = (uint8_t *)malloc(NACT), *mate = (uint8_t *)malloc(NACT);
  for (int p = first; p < first + count; p++) {
    int eic = 0;
    ref_checks(boards + (size_t)p * NSQ, hands + (size_t)p * 14, sides[p], cls, mate, &eic);
    uint32_t *lb = legal_bits + (size_t)p * 423, *cb = check_bits + (size_t)p * 423;
    int32_t *cc = class_counts + (size_t)p * 6;
    memset(lb, 0, 423 * 4);
    memset(cb, 0, 423 * 4);
    memset(cc, 0, 6 * 4);
    mate_count[p] = 0;
    mate_lowest[p] = -1;
    enemy_in_check[p] = (uint8_t)eic;
    for (int a = 0; a < NACT; a++) {
      if (cls[a] == 0xFF) continue;
      lb[a >> 5] |= 1u << (a & 31);
      if (cls[a] == 0) continue;
      cb[a >> 5] |= 1u << (a & 31);
      cc[(cls[a] & 7) - 1] += 1;
      if (cls[a] & CLS_PROMO_ONLY) cc[5] += 1;
      if (mate[a] == 1) {
        if (mate_lowest[p] < 0) mate_lowest[p] = a;
        mate_count[p] += 1;
      }
    }
  }
  free(cls);
  free(mate);
}
