/* lookahead_ref.c -- the one-ply look-ahead opponent's scores by the CPU oracle's own rules (test infrastructure).
 *
 * Built by tests/lookahead_ref.py into a temporary directory.  It includes oracle/keisei_oracle.c unchanged.  Every legal
 * move (gen_legal, simulate-and-test) is applied to a copy of the position and the copy is classified: no legal reply and
 * in check is Tsumi, no legal reply otherwise is stalemate; else gen_legal's replies give R (the best reply gain), and a
 * reply that checks is applied in turn and is a mate when the mover has no legal move left.  Positions are loaded without
 * history and with a move limit that is never reached, so Tsumi and stalemate are the only ways a move ends the game.
 * Shares nothing with the CUDA path's windows or value tables. */
#include "../oracle/keisei_oracle.c"

#define LA_MATE 1000000
#define LA_ILLEGAL INT32_MIN
#define LA_MAX_MOVES 1024

/* piece values by type P L N S G B R K +P +L +N +S +B +R */
static const int VALUE[14] = {1, 3, 4, 5, 6, 8, 10, 0, 6, 6, 6, 6, 10, 12};

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

static int dest_of(int a) {
  int pair = a >> 1, from = pair / 80, t = pair % 80;
  return t + (t >= from);
}

/* what action a gains for `side` on board b: a captured piece's value plus its unpromoted type's, and a promotion's
 * difference in value; a drop gains 0 */
static int gain(const int8_t *b, int side, int a) {
  if (a >= 12960) return 0;
  int from = (a >> 1) / 80, to = dest_of(a), g = 0;
  if (b[to] && pcolor(b[to]) != side) g += VALUE[ptype(b[to])] + VALUE[base_of(ptype(b[to]))];
  if (a & 1) g += VALUE[promoted_of(ptype(b[from]))] - VALUE[ptype(b[from])];
  return g;
}

/* score[a] (NACT int32) of every legal action a of the position, LA_ILLEGAL for the others; *best = the maximum score
 * and *ties = the number of legal actions reaching it (0 and 0 without a legal move).  Returns the number of legal moves. */
int ref_lookahead(const int8_t *board81, const uint8_t *hands14, int side, int32_t *score, int32_t *best, int32_t *ties) {
  orc_game *g = orc_new();
  orc_load(g, board81, hands14, side, 0, 65535, 0);
  for (int a = 0; a < NACT; a++) score[a] = LA_ILLEGAL;
  int me = side, en = 1 - side;
  static __thread uint16_t moves[LA_MAX_MOVES], replies[LA_MAX_MOVES], tmp[LA_MAX_MOVES];
  int n = gen_legal(g, 0, moves);
  *best = 0;
  *ties = 0;
  for (int i = 0; i < n; i++) {
    int a = moves[i];
    int x = gain(g->board, me, a);
    int cap_king = a < 12960 && g->board[dest_of(a)] == mk(T_KING, en);
    orc_game c = *g; /* shares g->hist, which nothing below reads */
    apply_action(&c, a);
    int nr = gen_legal(&c, 0, replies);
    int s;
    if (nr == 0) {
      s = (king_in_check(c.board, en) && !cap_king) ? LA_MATE : x; /* Tsumi, or stalemate (a draw) */
    } else {
      int r_best = 0, mate = 0;
      for (int j = 0; j < nr; j++) {
        int r = replies[j];
        int gr = gain(c.board, en, r);
        if (gr > r_best) r_best = gr;
        if (mate) continue;
        int rk = r < 12960 && c.board[dest_of(r)] == mk(T_KING, me);
        orc_game d = c;
        apply_action(&d, r);
        if (!rk && king_in_check(d.board, me) && gen_legal(&d, 0, tmp) == 0) mate = 1;
      }
      s = mate ? -LA_MATE : x - r_best;
    }
    score[a] = s;
    if (i == 0 || s > *best) {
      *best = s;
      *ties = 1;
    } else if (s == *best) {
      *ties += 1;
    }
  }
  orc_free(g);
  return n;
}

/* ref_lookahead over positions [first, first + count): best [n], ties [n] and the tied actions in ascending order,
 * tied [n][LA_MAX_MOVES] (uint16, the first ties[p] entries of row p). */
void ref_lookahead_batch(int first, int count, const int8_t *boards, const uint8_t *hands, const uint8_t *sides,
                         int32_t *best, int32_t *ties, uint16_t *tied) {
  int32_t *score = (int32_t *)malloc(sizeof(int32_t) * NACT);
  for (int p = first; p < first + count; p++) {
    ref_lookahead(boards + (size_t)p * NSQ, hands + (size_t)p * 14, sides[p], score, best + p, ties + p);
    uint16_t *row = tied + (size_t)p * LA_MAX_MOVES;
    int k = 0;
    for (int a = 0; a < NACT && k < ties[p]; a++)
      if (score[a] != LA_ILLEGAL && score[a] == best[p]) row[k++] = (uint16_t)a;
  }
  free(score);
}

/* R of positions [first, first + count): gain[p] = the largest gain over the side to move's legal moves and count[p] =
 * how many moves reach it (0 and 0 without a legal move). */
void ref_capture_gain_batch(int first, int count, const int8_t *boards, const uint8_t *hands, const uint8_t *sides,
                            int32_t *gain_out, int32_t *count_out) {
  uint16_t *moves = (uint16_t *)malloc(sizeof(uint16_t) * LA_MAX_MOVES);
  orc_game *g = orc_new();
  for (int p = first; p < first + count; p++) {
    orc_load(g, boards + (size_t)p * NSQ, hands + (size_t)p * 14, sides[p], 0, 65535, 0);
    int n = gen_legal(g, 0, moves), best = 0, c = 0;
    for (int i = 0; i < n; i++) {
      int x = gain(g->board, sides[p], moves[i]);
      if (x > best) { best = x; c = 1; }
      else if (x == best) c++;
    }
    gain_out[p] = best;
    count_out[p] = c;
  }
  orc_free(g);
  free(moves);
}
