/* perft_ref.c -- move-tree perft on the CPU oracle's own move generator (test infrastructure).
 *
 * Built by tests/perft_ref.py into a temporary directory.  It includes oracle/keisei_oracle.c unchanged, so the count comes
 * from the oracle's simulate-and-test generator (gen_legal) on copies of the position and shares nothing with the CUDA
 * path's bitboard generator.  History, termination and the move limit play no part: a node without legal moves has no
 * children and repetition never ends a line -- what shogidrl_b200.perft counts. */
#include "../oracle/keisei_oracle.c"

static int64_t perft_rec(orc_game *g, int depth, int64_t *divide_out) {
  if (depth <= 0) return 1;
  uint16_t moves[1024];
  int n = gen_legal(g, 0, moves);
  if (depth == 1 && !divide_out) return n;
  int64_t total = 0;
  for (int i = 0; i < n; i++) {
    orc_game c = *g; /* shares g->hist, which nothing below reads */
    int a = moves[i], me = c.side;
    if (a < 12960) {
      int pair = a >> 1, from = pair / 80, t = pair % 80;
      apply_board_move(c.board, c.hands, from, t + (t >= from), a & 1, me);
    } else {
      apply_drop(c.board, c.hands, (a - 12960) / 7, (a - 12960) % 7, me);
    }
    c.side = 1 - me;
    c.move_count += 1;
    int64_t k = perft_rec(&c, depth - 1, NULL);
    if (divide_out) divide_out[a] = k;
    total += k;
  }
  return total;
}

/* perft of the position (board81, hands14, side) to `depth` plies; divide_out (optional, NACT int64) receives for each
 * legal root action the count below it and keeps the caller's value elsewhere. */
int64_t ref_perft(const int8_t *board81, const uint8_t *hands14, int side, int depth, int64_t *divide_out) {
  orc_game *g = orc_new();
  orc_load(g, board81, hands14, side, 0, 65535, 0);
  int64_t r = perft_rec(g, depth, divide_out);
  orc_free(g);
  return r;
}
