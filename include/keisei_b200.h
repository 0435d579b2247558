/*
 * keisei_b200.h -- C ABI of the B200-native Keisei self-play rollout hot path.
 *
 * The reference (tachyon-beep/shogidrl) is pure Python and has no FFI of its own; the
 * boundary it offers is duck typing (StepManager(config, game, agent, policy_mapper,
 * experience_buffer), keisei/training/step_manager.py:61-68).  Each entry point below
 * replaces the Python computation cited beside it (paths relative to the reference
 * checkout).  INTEGRATION.md shows the ctypes binding a maintainer adds.
 *
 * Conventions: every function returns 0 on success or a negative KZ_E_* code, never
 * throws; every data pointer is a DEVICE pointer into caller-owned memory unless marked
 * HOST; `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  No
 * call synchronises the device.  There is no CPU fallback.
 *
 * Piece code: 0 empty, else 1 + type + 14*colour (type: P0 L1 N2 S3 G4 B5 R6 K7 +P8 +L9
 * +N10 +S11 +B12 +R13; colour BLACK=0/WHITE=1 -- shogi_core_definitions.py:50-83).
 * Square = row*9 + col.  Action index = PolicyOutputMapper's enumeration
 * (keisei/utils/utils.py:208-266): board move ((from*80 + to - (to>from))*2 + promote),
 * drop 12960 + to*7 + piece_type; 13,527 actions.
 */
#ifndef KEISEI_B200_H
#define KEISEI_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define KZ_ABI_VERSION 3
#define KZ_NUM_ACTIONS 13527
#define KZ_OBS_FLOATS 3726  /* 46 x 9 x 9 */
#define KZ_MASK_PAD_STRIDE 13536 /* 16-byte multiple >= 13527: fast-path row stride */
#define KZ_BITMAP_WORDS 448     /* row of a legal BITMAP: bit i = action i legal; 423 words used, zero-padded to 14 per lane */
#define KZ_BITMAP_WORDS_MIN 423 /* smallest row stride (in 32-bit words) the bitmap readers accept */
#define KZ_POOL_RECORD_WORDS 512  /* one start-position record (kz_pool_records): 2 KB, layout below */
#define KZ_POOL_BITMAP_OFFSET 64  /* word of a record where its 448-word legal bitmap begins */
#define KZ_COBS_WORDS 40        /* compact observation: 84 bytes of plane indices + 18 fp32 constant-plane values + pad = 160 B */

/* termination reason codes (shogi_core_definitions.py:135-147) */
#define KZ_ONGOING 0
#define KZ_TSUMI 1      /* "Tsumi"             */
#define KZ_STALEMATE 2  /* "stalemate"         */
#define KZ_MAX_MOVES 3  /* "Max moves reached" */
#define KZ_SENNICHITE 4 /* "Sennichite"        */

/* error codes */
#define KZ_OK 0
#define KZ_E_ARG (-1)       /* null / misaligned / out-of-range argument */
#define KZ_E_CUDA (-2)      /* a CUDA runtime call failed (see kz_last_cuda_error) */
#define KZ_E_NOT_INIT (-3)  /* kz_init_tables has not run on this device */

/* per-env error bits (kz_errors): mirror the ValueError cases StepManager turns into a reset
 * (step_manager.py:303-348; shogi_game.py:461-483, 529-544) */
#define KZ_ERR_BAD_ACTION 1    /* index out of range / no own piece on source / drop not in hand or on occupied square */
#define KZ_ERR_BAD_PATTERN 2   /* "Illegal movement pattern" */
#define KZ_ERR_KING_CAPTURE 4  /* a king was captured (out of contract, shogi_move_execution.py:109-114) */
#define KZ_ERR_HISTORY_FULL 8  /* more plies than hist_cap since the last reset */

int kz_abi_version(void);
const char* kz_last_cuda_error(void);
/* "src_sha=<sha256/16 of csrc/*.cu, *.cuh and this header at build time> built=<date time> arch=sm_100a" */
const char* kz_build_info(void);

/* Move/ray lookup tables -> device memory of the current device.  Idempotent. */
int kz_init_tables(void* stream);

/* Device game state is one caller-allocated blob (torch.empty(total, dtype=uint8)), SoA by
 * field group: boards [n][96] u8, meta [n][32] u8, repetition tables [n][slots] of 16-byte
 * slots (124-bit Zobrist-style position key + 4-bit occurrence count, open addressing, slots =
 * power of two >= 2*hist_cap) replacing the tuple history of shogi_game.py:347-372, and a
 * trailing 256-byte scheduling word block (work counter of the launch in flight).
 * offsets3 (HOST) receives the byte offsets of the first three sections. */
int kz_state_layout(int n, int hist_cap, int64_t* offsets3, int64_t* total_bytes);

/* ShogiGame.reset (shogi_game.py:79-130) for the envs whose env_mask byte is non-zero (all
 * if env_mask is NULL).  max_moves = ShogiGame(max_moves_per_game). */
int kz_reset(void* state, int n, int hist_cap, const uint8_t* env_mask, int max_moves, void* stream);

/* ShogiGame.from_sfen after parsing (shogi_game.py:306-329; SFEN text stays host-side):
 * boards [n][81] piece codes, hands [n][14] (black P..R, white P..R), side [n], move_count [n],
 * max_moves [n].  History is emptied.  Termination of the loaded position (shogi_game.py:343)
 * is evaluated by the next kz_refresh(eval_termination=1). */
int kz_load_positions(void* state, int n, int hist_cap, const int8_t* boards, const uint8_t* hands,
                      const uint8_t* side, const int32_t* move_count, const int32_t* max_moves, void* stream);

/* Inverse of kz_load_positions, for the scalar facade and parity dumps.
 * meta8 [n][8] int32 = side, move_count, max_moves, status(reason), winner(-1 none), error bits,
 * plies since reset, finished-episode counter. */
int kz_export_positions(const void* state, int n, int hist_cap, int8_t* boards, uint8_t* hands,
                        int32_t* meta8, void* stream);

/* Outputs for the CURRENT positions without moving (all output pointers optional):
 *   obs   generate_neural_network_observation (shogi_game_io.py:434-539), fp32, row stride
 *         obs_stride floats (even, base 16-byte aligned);
 *   mask  generate_all_legal_moves + PolicyOutputMapper.get_legal_mask
 *         (shogi_rules_logic.py:486-635, utils.py:310-336), one byte per action, row stride
 *         mask_stride bytes (>= 13527; a multiple of 16 with a 16-byte aligned base takes the
 *         vectorised path and may zero the pad bytes);
 *   legal_count int32 per env;
 *   next_actions: uniform-random legal action for each env (k-th legal index in ascending
 *         order, k = mulhi(rand32(seed, env_offset+env, rng_step), count)); int64 if
 *         actions_i64 else int32; -1 when there is no legal move.
 * eval_termination != 0 applies _check_and_update_termination_status to loaded positions
 * (shogi_game.py:343, 408-450: mover := opponent of the side to move).
 * in_check (optional, u8 per env): the side to move is in check (is_in_check,
 * shogi_rules_logic.py:36-67; a missing king counts as in check). */
int kz_refresh(void* state, int n, int hist_cap, float* obs, int64_t obs_stride, uint8_t* mask,
               int64_t mask_stride, int32_t* legal_count, void* next_actions, int actions_i64,
               uint64_t seed, uint32_t rng_step, uint32_t env_offset, int eval_termination,
               uint8_t* in_check, void* stream);

/* One environment step for n games: ShogiGame.make_move (shogi_game.py:574-660) fused with the
 * legal-move generation, termination test, mask and observation of the successor, plus what
 * StepManager does around it on `done` (reset, step_manager.py:437-440) when auto_reset != 0.
 *   actions      [n] int64 (actions_i64) or int32 policy indices drawn from the previous mask
 *   reward       +1 mover won / -1 mover lost / 0 (shogi_game.py:553-572), fp32
 *   done/reason/winner  u8 / u8 (KZ_*) / i8 (0 black, 1 white, -1 none)
 *   ep_len       move_count at termination (int32), 0 while running
 *   obs/mask/legal_count/next_actions: as kz_refresh, for the RETURNED state (after reset when
 *                auto_reset and done); obs of the terminal state is not materialised then.
 * An action that fails the reference's make_move validation sets the env's error bits, leaves
 * the game untouched and reports reward 0 / done 0. */
int kz_step(void* state, int n, int hist_cap, const void* actions, int actions_i64, float* obs,
            int64_t obs_stride, uint8_t* mask, int64_t mask_stride, float* reward, uint8_t* done,
            uint8_t* reason, int8_t* winner, int32_t* ep_len, int32_t* legal_count, void* next_actions,
            uint64_t seed, uint32_t rng_step, uint32_t env_offset, int auto_reset, void* stream);

/* kz_step / kz_step_rollout over the sub-range [first, first + count) of the batch's n games: every array argument is
 * still indexed by the game's position in the whole batch (row g of obs / mask / bitmap, element g of actions, reward,
 * ...), and the per-game random stream is keyed by env_offset + g as before, so stepping a batch as several ranges gives
 * exactly the results of one kz_step.  Ranges of one batch may run CONCURRENTLY on different streams when each names its
 * own counter_slot (0..63, the dynamic work counter of the launch): a caller that consumes each range's results
 * separately can let the ranges run ahead of each other across steps, so that one range's CTAs fill the SMs another
 * range's draining grid leaves idle.
 * mask != NULL: byte-mask form (kz_step); bitmap != NULL: rollout form (kz_step_rollout); not both. */
int kz_step_range(void* state, int n, int hist_cap, int first, int count, int counter_slot, const void* actions,
                  int actions_i64, float* obs, int64_t obs_stride, uint8_t* mask, int64_t mask_stride, uint32_t* bitmap,
                  int64_t bitmap_stride_words, uint32_t* cobs, float* reward, uint8_t* done, uint8_t* reason, int8_t* winner,
                  int32_t* ep_len, int32_t* legal_count, void* next_actions, uint64_t seed, uint32_t rng_step,
                  uint32_t env_offset, int auto_reset, void* stream);

/* ---- start-position pools: finished games restart from a table of precomputed positions instead of the start position.
 * A RECORD (KZ_POOL_RECORD_WORDS uint32, 16-byte aligned) holds everything the auto-reset writes:
 *   words 0..23   the 96-byte board row (81 piece codes; bytes 84..95 = words x, y, z of the 124-bit position key),
 *   words 24..31  the 32-byte meta row: hands (bytes 0..13), side to move (14), move_count (18..19, u16), word w of the
 *                 key (28..31); status 0, winner none, error bits / plies since reset / max_moves / episodes 0,
 *   word 32       legal-move count, word 33 in-check flag (0 / 1), words 34..63 zero,
 *   words 64..511 the legal bitmap (KZ_BITMAP_WORDS words, kz_legal_bitmap's row).
 * kz_pool_records packs one record per game of a batch that kz_load_positions + kz_refresh (in_check) + kz_legal_bitmap
 * have just prepared: state = that batch (n games, hist_cap), bitmap / legal_count / in_check = those calls' outputs.
 * The positions must be non-terminal (kz_refresh(eval_termination=1) status 0, at least one legal move) and must not let
 * the side to move capture the opponent's king; kz_pool_records does not check this. */
int kz_pool_records(const void* state, int n, int hist_cap, const uint32_t* bitmap, int64_t bitmap_stride_words,
                    const int32_t* legal_count, const uint8_t* in_check, uint32_t* records, void* stream);
/* kz_step_range with auto-reset, where a game that finishes in this launch restarts from pool record k:
 *   k = pick[g] when pick (int32 [n], indexed by the game's position in the batch) is given, otherwise
 *   k = mulhi(rand32(pool_seed, env_offset + g, E), pool_size) with E the game's finished-episode counter after this
 *       episode has been counted (export meta8[7]) -- so a replayed CUDA graph, whose rng_step values repeat, still draws
 *       fresh starts; values of pick outside [0, pool_size) are taken modulo pool_size.
 * The game keeps its own max_moves; move_count continues from the record's (so the ep_len a game reports counts the
 * record's move_count too); the repetition table is emptied and the plies
 * since reset set to 0.  start_ids (optional int32 [n]) receives k for every game that restarts.  Every output of the
 * returned state (obs, mask or bitmap, cobs, legal_count, next_actions) comes from the record exactly as kz_step's
 * outputs come from the start position. */
int kz_step_pool(void* state, int n, int hist_cap, int first, int count, int counter_slot, const void* actions,
                 int actions_i64, float* obs, int64_t obs_stride, uint8_t* mask, int64_t mask_stride, uint32_t* bitmap,
                 int64_t bitmap_stride_words, uint32_t* cobs, float* reward, uint8_t* done, uint8_t* reason, int8_t* winner,
                 int32_t* ep_len, int32_t* legal_count, void* next_actions, uint64_t seed, uint32_t rng_step,
                 uint32_t env_offset, const uint32_t* pool, int pool_size, const int32_t* pick, uint64_t pool_seed,
                 int32_t* start_ids, void* stream);
/* kz_reset from the pool: the envs whose env_mask byte is non-zero (all if NULL) restart from record k, chosen as in
 * kz_step_pool with E = the current finished-episode counter (not advanced); start_ids optional as there.  As after
 * kz_reset, the rows of the new positions come from kz_refresh / kz_legal_bitmap. */
int kz_reset_pool(void* state, int n, int hist_cap, const uint8_t* env_mask, int max_moves, const uint32_t* pool, int pool_size,
                  const int32_t* pick, uint64_t pool_seed, uint32_t env_offset, int32_t* start_ids, void* stream);

/* Rollout form of kz_step (the PPO self-play path, StepManager.execute_step step_manager.py:98-348 over n games): as
 * kz_step, but the successor's legal moves are left as the 13,527-bit legal BITMAP -- bitmap [n][bitmap_stride_words]
 * uint32, 16-byte aligned rows, bit i = action i is legal, the same set PolicyOutputMapper.get_legal_mask
 * (utils.py:310-336) marks -- instead of the 13,527-byte mask row: 1,792 B instead of 13,536 B written per game here, and
 * read again by kz_sample_bitmap and by every kz_eval_bitmap_* pass of the update.  obs as in kz_step (optional).
 * kz_legal_bitmap is the kz_refresh counterpart (current positions, no move); kz_bitmap_expand turns bitmap rows into
 * byte-mask rows for callers of the reference API (ExperienceBuffer.legal_masks, experience_buffer.py:52-54).
 * cobs (optional, [n][KZ_COBS_WORDS] uint32): the COMPACT OBSERVATION of the returned state -- the same information as
 * the 46x9x9 tensor of generate_neural_network_observation (shogi_game_io.py:434-539) in 160 bytes: bytes 0..80 = for
 * each observation square (row-major, already rotated 180 degrees when White is to move) the index 0..27 of the one
 * piece plane that is 1.0 there, 0xFF if none; words 21..38 = the fp32 values of the constant planes 28..45 (hands / 18,
 * side to move, move_count / max_moves, two reserved zeros).  kz_cobs_conv_fwd / _wgrad consume it. */
int kz_step_rollout(void* state, int n, int hist_cap, const void* actions, int actions_i64, float* obs,
                    int64_t obs_stride, uint32_t* bitmap, int64_t bitmap_stride_words, uint32_t* cobs, float* reward,
                    uint8_t* done, uint8_t* reason, int8_t* winner, int32_t* ep_len, int32_t* legal_count,
                    void* next_actions, uint64_t seed, uint32_t rng_step, uint32_t env_offset, int auto_reset,
                    void* stream);
int kz_legal_bitmap(void* state, int n, int hist_cap, float* obs, int64_t obs_stride, uint32_t* bitmap,
                    int64_t bitmap_stride_words, uint32_t* cobs, int32_t* legal_count, void* stream);
int kz_bitmap_expand(const uint32_t* bitmap, int64_t bitmap_stride_words, const int64_t* bitmap_rows, int n, uint8_t* mask,
                     int64_t mask_stride, void* stream);

/* ---- move expansion: the outcome of listed moves without moving the games they start from (look-ahead, search, perft).
 * kz_legal_list turns n legal-bitmap rows (bitmap_stride_words >= KZ_BITMAP_WORDS_MIN, 4-byte aligned) into a list of legal
 * moves grouped by game: offsets (int64 [n+1], device) is the exclusive prefix sum of the rows' legal counts, and game g's
 * legal actions go in ascending order to [offsets[g], offsets[g+1]) of actions_out (int64 if actions_i64 else int32), with
 * parent_out[i] = g (int32, optional).  A row whose offsets disagree with its bitmap writes nothing outside its own range. */
int kz_legal_list(const uint32_t* bitmap, int64_t bitmap_stride_words, int n, const int64_t* offsets, int32_t* parent_out,
                  void* actions_out, int actions_i64, void* stream);
/* kz_expand applies actions[i] (int64 if actions_i64 else int32) to a copy of game parent[i] (int32) of the batch `state`
 * (n games, hist_cap), for each of the m items.  Every output of item i is what kz_step(auto_reset = 0) would give for that
 * one move on a clone of the parent with its history: the action checks, err[i] (u8, the parent's error bits with the
 * move's own), the position key, the repetition count in the parent's table (a match gives the stored count + 1, a miss 1,
 * so the 4th occurrence is sennichite as in kz_step), termination in the reference's order, reward / done / reason /
 * winner / ep_len, legal_count, and the rollout-form rows of kz_step_rollout: obs, bitmap, cobs (rows indexed by the item;
 * every output pointer optional).  The source batch is not written, except for its work counter counter_slot (0..63, as in
 * kz_step_range).  An item whose parent lies outside [0, n) gets KZ_ERR_BAD_ACTION, reads nothing, and reports what a
 * rejected action on an empty board reports (reward 0, done 0, legal_count 0).  Items of one parent should be adjacent:
 * the parent's rows are then read from cache.
 * child_state (optional, not the source) is a batch of m games laid out by kz_state_layout(m, child_hist_cap): item i
 * stores its successor there with status and winner as kz_step leaves them, error bits, plies since reset and finished
 * episodes 0, and an emptied repetition table -- the position as kz_load_positions + kz_refresh would hold it, which can be
 * listed, expanded or stepped again.  Children do NOT inherit history: a repetition is counted from the child on, as the
 * reference's ShogiGame.__deepcopy__ forgets the move history (shogi_game.py:165-169).  m == 0 launches nothing. */
int kz_expand(const void* state, int n, int hist_cap, int counter_slot, const int32_t* parent, const void* actions,
              int actions_i64, int m, float* obs, int64_t obs_stride, uint32_t* bitmap, int64_t bitmap_stride_words,
              uint32_t* cobs, float* reward, uint8_t* done, uint8_t* reason, int8_t* winner, int32_t* ep_len,
              int32_t* legal_count, uint8_t* err, void* child_state, int child_hist_cap, void* stream);
/* Legal moves that give check: out row g = the legal-bitmap row g (input, kz_legal_bitmap's row of the current position)
 * ANDed with "after this move the side that did not move is in check" (is_in_check, shogi_rules_logic.py:36-67, with the
 * reference's "a missing king counts as in check": with the enemy king missing every legal move checks).  Reads the
 * board, side to move and status from the state.  The row is exact whenever the side NOT to move is not already in check,
 * which holds for every position reached by play; a loaded position in which it is gets ALL its legal moves (a superset:
 * callers that decide mates by kz_expand stay exact).  Pad bits 13527..13535 and words 423.. of each out row are zero.  A
 * finished game (status != 0) gets an empty row and count 0.  count (int32 [n], popcount of each out row) may be NULL.
 * Strides in 32-bit words, >= KZ_BITMAP_WORDS_MIN; bitmap and out 16-byte aligned; out must not overlap bitmap. */
int kz_check_bitmap(const void* state, int n, int hist_cap, const uint32_t* bitmap, int64_t bitmap_stride_words, uint32_t* out,
                    int64_t out_stride_words, int32_t* count, void* stream);

/* Thin conveniences over kz_refresh. */
int kz_legal_mask(void* state, int n, int hist_cap, uint8_t* mask, int64_t mask_stride,
                  int32_t* legal_count, void* stream);
int kz_observe(void* state, int n, int hist_cap, float* obs, int64_t obs_stride, void* stream);

/* generate_piece_potential_moves (shogi_rules_logic.py:82-208) for the piece on squares[env]:
 * targets3 [n][3] uint32 = 81-bit set of pseudo-legal target squares (bit = row*9 + col). */
int kz_piece_targets(const void* state, int n, int hist_cap, const int32_t* squares, uint32_t* targets3,
                     void* stream);

/* Per-env error bits (KZ_ERR_*) -> out[n] int32; clear != 0 resets them. */
int kz_errors(void* state, int n, int hist_cap, int32_t* out, int clear, void* stream);

/* BaseActorCriticModel.get_action_and_value after forward() (base_actor_critic.py:64-116):
 * masked softmax over 13,527 logits, Categorical sample (or argmax if deterministic) and
 * log_prob with torch.distributions' probs->logits clamp (eps = FLT_EPSILON).
 *   logits [n][ld] fp32 (logits_bf16 == 0) or bf16; mask [n][ldm] bytes; actions int64/int32;
 *   logp fp32; entropy optional fp32.  A legal logit of -inf has probability 0.  Rows whose softmax is NaN -- mask
 *   all zero, every legal logit -inf, or a legal logit NaN or +inf -- fall back to the uniform distribution over all
 *   actions (base_actor_critic.py:93-101): a uniform draw, argmax 0, log_prob log(1/13527).  Sampling is inverse-CDF on a
 *   counter-based uniform keyed (seed, offset + row): statistical, not bitwise, parity with
 *   torch.multinomial.  offset_dev (optional device uint64): added to offset when the kernel runs,
 *   so that a launch captured in a CUDA graph draws fresh numbers on every replay (the caller
 *   advances the device counter between launches). */
int kz_sample_masked(const void* logits, int logits_bf16, int64_t ld, const uint8_t* mask, int64_t ldm,
                     int n, uint64_t seed, uint64_t offset, const uint64_t* offset_dev, void* actions,
                     int actions_i64, float* logp, float* entropy, int deterministic, void* stream);
/* The same with the legal set given as bitmap rows (kz_step_rollout): bitmap [n][ldb_words] uint32; the pad bits
 * 13,527-13,535 of word 422 and words 423.. are ignored.  For a 16-byte aligned byte mask of the same set the two entry
 * points return identical actions, log-probs and entropies. */
int kz_sample_bitmap(const void* logits, int logits_bf16, int64_t ld, const uint32_t* bitmap, int64_t ldb_words,
                     int n, uint64_t seed, uint64_t offset, const uint64_t* offset_dev, void* actions,
                     int actions_i64, float* logp, float* entropy, int deterministic, void* stream);

/* The scripted opponent SimpleHeuristicOpponent.select_move (keisei/utils/opponents.py) for the CURRENT position of each
 * of the n games: the legal moves are split into tiers -- 0 capture (destination holds a piece of the other colour),
 * 1 non-promoting move of the mover's unpromoted pawn, 2 everything else, every drop included -- and the pick is the k-th
 * member of the first non-empty tier in ascending action order, k = mulhi(rand32(seed, env_offset+env, rng_step), tier
 * size): kz_refresh's next_actions convention.  The legal set is read from exactly one of
 *   mask   [n][mask_stride] bytes (non-zero = legal; kz_step / kz_refresh rows), or
 *   bitmap [n][bitmap_stride_words] uint32 (kz_step_rollout / kz_legal_bitmap rows; 4-byte aligned);
 * both forms give identical results.  actions: int64 if actions_i64 else int32, -1 when there is no legal move.
 * Optional: tier (u8: 0 capture, 1 pawn, 2 other, 255 none) and tier_count (int32: size of the chosen tier).
 * Needs no tables. */
int kz_heuristic_actions(const void* state, int n, int hist_cap, const uint8_t* mask, int64_t mask_stride,
                         const uint32_t* bitmap, int64_t bitmap_stride_words, void* actions, int actions_i64, uint8_t* tier,
                         int32_t* tier_count, uint64_t seed, uint32_t rng_step, uint32_t env_offset, void* stream);

/* ExperienceBuffer.compute_advantages_and_returns (experience_buffer.py:99-145) over a [T][N]
 * layout, one reverse scan per env column (N = 1 is the reference's flat buffer):
 *   delta = (r + (gamma * nv) * m) - V ;  gae = delta + (gamma_lambda * m) * gae   (no FMA)
 * rewards/values/adv/ret fp32 [T][N], dones u8 [T][N], last_value fp32 [N]. */
int kz_gae(const float* rewards, const float* values, const uint8_t* dones, const float* last_value,
           int T, int N, float gamma, float gamma_lambda, float* adv, float* ret, void* stream);
/* kz_gae dispatches on N: wide rollouts (N >= 2048) run one thread per env column, sequential in
 * time, bit-exact with the reference's fp32 op order; narrow ones (the reference's N = 1 buffer)
 * run one warp per column as a reverse affine-map warp scan (agrees to ~1e-6 relative).
 * kz_gae_exact always takes the bit-exact column kernel. */
int kz_gae_exact(const float* rewards, const float* values, const uint8_t* dones, const float* last_value,
                 int T, int N, float gamma, float gamma_lambda, float* adv, float* ret, void* stream);

/* BaseActorCriticModel.evaluate_actions after forward() (base_actor_critic.py:118-184) for the PPO update
 * (SURVEY 8f-1): masked softmax, log-prob of the taken action and entropy (Categorical(probs) clamp semantics),
 * forward and backward.  logits [n][ld] fp32/bf16; mask rows are mask[mask_rows[i]] when mask_rows != NULL (lets
 * a minibatch index the rollout's mask storage without gathering it); saved4 [n][4] fp32 scratch handed from
 * forward to backward; dlogits [n][ldg] in the logits dtype (pad columns beyond 13,527 are not written).  Rows whose
 * softmax is NaN (no legal action, every legal logit -inf, a legal logit NaN or +inf) take the uniform distribution,
 * as kz_sample_masked does, with a zero gradient and no bias contribution. */
int kz_eval_masked_fwd(const void* logits, int logits_bf16, int64_t ld, const uint8_t* mask, int64_t ldm,
                       const int64_t* mask_rows, const int64_t* actions, int n, float* logp, float* entropy,
                       float* saved4, void* stream);
int kz_eval_masked_bwd(const void* logits, int logits_bf16, int64_t ld, const uint8_t* mask, int64_t ldm,
                       const int64_t* mask_rows, const int64_t* actions, int n, const float* dlogp,
                       const float* dentropy, const float* saved4, void* dlogits, int64_t ldg, void* stream);
/* The same backward that also accumulates the column sums of dlogits -- the gradient of the policy head's bias
 * (nn.Linear(…, 13527), keisei/core/neural_network.py:20) -- into dbias_q44 int64 [>= 13527], which the caller has
 * zeroed: dlogits is non-zero only at legal actions (~0.5 % of a row), so the bias gradient is a sparse scatter-add
 * (integer reductions in L2, taken before the rounding to the dlogits dtype) instead of a second pass over [n][13536].
 * The sums are Q20.44 fixed point (gradient = value * 2^-44): integer addition is associative, so the result is
 * deterministic run to run, unlike an fp32 atomic accumulation. */
int kz_eval_masked_bwd_bias(const void* logits, int logits_bf16, int64_t ld, const uint8_t* mask, int64_t ldm,
                            const int64_t* mask_rows, const int64_t* actions, int n, const float* dlogp,
                            const float* dentropy, const float* saved4, void* dlogits, int64_t ldg, int64_t* dbias_q44,
                            void* stream);
/* Bitmap forms of the evaluation pair: legal sets as rows bitmap[bitmap_rows[i]] (or bitmap[i]) of kz_step_rollout's
 * output, pad bits ignored as in kz_sample_bitmap; dbias_q44 optional (NULL: no bias gradient).  Results identical to
 * the byte-mask forms on the same sets. */
int kz_eval_bitmap_fwd(const void* logits, int logits_bf16, int64_t ld, const uint32_t* bitmap, int64_t ldb_words,
                       const int64_t* bitmap_rows, const int64_t* actions, int n, float* logp, float* entropy,
                       float* saved4, void* stream);
int kz_eval_bitmap_bwd(const void* logits, int logits_bf16, int64_t ld, const uint32_t* bitmap, int64_t ldb_words,
                       const int64_t* bitmap_rows, const int64_t* actions, int n, const float* dlogp,
                       const float* dentropy, const float* saved4, void* dlogits, int64_t ldg, int64_t* dbias_q44,
                       void* stream);

/* PPO clipped-surrogate loss of one minibatch and its gradients in closed form (keisei/core/ppo_agent.py:332-372;
 * value clipping off): out6 = {loss, policy loss, value loss, entropy loss (= -mean entropy), mean(old_logp -
 * new_logp), clip fraction}; d_* = d loss / d input, multiplied by grad_scale.  All fp32 [n]. */
int kz_ppo_loss(const float* new_logp, const float* entropy, const float* new_value, const float* old_logp,
                const float* advantages, const float* returns, int n, float clip_epsilon, float value_coef,
                float entropy_coef, float grad_scale, float* out6, float* d_logp, float* d_entropy, float* d_value,
                void* stream);

/* ---- observation input layer of the default policy/value network (keisei/core/neural_network.py:14-28:
 * nn.Conv2d(46, 16, kernel_size=3, padding=1) [+ ReLU], run under bf16 autocast by ppo_agent.py:323) ----
 * kz_obs_conv_fwd: out[n][16][9][9] (bf16) = [relu](conv3x3(obs fp32 [n][46][9][9], weight fp32 [16][46][3][3]) + bias),
 * operands rounded to bf16, fp32 accumulation (what autocast computes).  cout must be 16.  obs_rows (int64 [n] or
 * NULL): board b is read from row obs_rows[b] of the observation storage -- the minibatch gather of
 * ppo_agent.py:300-309 done in place.
 * kz_obs_conv_wgrad: dweight [16][46][3][3] / dbias [16] (fp32, overwritten) from dout [n][16][9][9] (bf16 or fp32);
 * y_bf16 = the saved forward output when the forward applied ReLU (its backward is fused), else NULL.
 * workspace: ctas * 16 * 432 floats with ctas = kz_obs_conv_wgrad_ctas(n); deterministic (no atomics). */
int kz_obs_conv_fwd(const float* obs, const int64_t* obs_rows, const float* weight, const float* bias, int cout, int n,
                    int relu, void* out_bf16, void* stream);
int kz_obs_conv_wgrad_ctas(int n);
int kz_obs_conv_wgrad(const float* obs, const int64_t* obs_rows, const void* y_bf16, const void* dout, int dout_bf16,
                      int cout, int n, float* workspace, int ctas, float* dweight, float* dbias, void* stream);

/* The same layer fed with the engine's COMPACT OBSERVATIONS (kz_step_rollout's cobs output, [..][KZ_COBS_WORDS] uint32; row
 * cobs_rows[b] or b) instead of the fp32 tensors they summarise -- 160 bytes per board instead of 14,904.  The forward needs
 * no dense product: at most one of the 28 piece planes is non-zero per square, so an output is the bias + nine weight
 * look-ups + the constant planes' contribution; the weight gradient patches its board tile from one board to the next.
 * Same operand rounding (bf16) and fp32 accumulation as kz_obs_conv_*; valid for observations the engine produced. */
int kz_cobs_conv_fwd(const uint32_t* cobs, const int64_t* cobs_rows, const float* weight, const float* bias, int cout, int n,
                     int relu, void* out_bf16, void* stream);
int kz_cobs_conv_wgrad_ctas(int n); /* workspace = ctas * 16 * 432 floats, as for kz_obs_conv_wgrad */
int kz_cobs_conv_wgrad(const uint32_t* cobs, const int64_t* cobs_rows, const void* y_bf16, const void* dout, int dout_bf16,
                       int cout, int n, float* workspace, int ctas, float* dweight, float* dbias, void* stream);

/* ---- tail of a PPO minibatch update: torch.nn.utils.clip_grad_norm_(parameters, max_norm) followed by
 * torch.optim.Adam.step() (keisei/core/ppo_agent.py:405-413, optimizer built at :66-80), fused: one read of every
 * gradient for the global L2 norm, then one pass that applies the clip coefficient min(1, max_norm / (norm + 1e-6)),
 * optional L2 weight decay (g += wd * p) and the Adam update with bias correction on fp32 tensors, in place.
 *   params / grads / exp_avg / exp_avg_sq / steps: HOST arrays of `count` DEVICE pointers (fp32 tensors of numel[i]
 *   elements; steps[i] = that parameter's step counter as a device fp32 scalar, ALREADY incremented for this step,
 *   which is where torch's capturable Adam keeps it).  workspace: device fp32 [>= kz_adam_clip_workspace(count, numel)].
 *   norm_out2 (device fp32 [2]) receives {total gradient norm before clipping, clip coefficient}.
 * Hyper-parameters are doubles, as Python hands them to torch: 1 - beta is formed in double before rounding to fp32.
 * Deterministic; the gradients themselves are left unscaled. */
long long kz_adam_clip_workspace(int count, const int64_t* numel);
int kz_adam_clip_step(int count, void* const* params, const void* const* grads, void* const* exp_avg,
                      void* const* exp_avg_sq, const void* const* steps, const int64_t* numel, double lr, double beta1,
                      double beta2, double eps, double weight_decay, double max_norm, float* workspace,
                      int64_t workspace_floats, float* norm_out2, void* stream);

#ifdef __cplusplus
}
#endif
#endif
